"""Repack reference-layout state_dicts into the device blobs / pointer structs of the C ABI.

One-off host work at weight-load time (not on the hot path): re-order convolution weights into
K-major GEMM operands, fold adjacency column sums into bias tables, fold the un-pooling into the
to_mot adjacency, concatenate q/k/v projections. Every derived tensor lives in ONE contiguous fp32
device blob (64-float aligned slices) with a bf16 mirror registered for MOCHA_BF16 mode.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib


class PackedBlob:
    """A flat fp32 device buffer + named 256B-aligned slices (+ bf16 mirror)."""

    def __init__(self, tensors: "dict[str, torch.Tensor]", device):
        self.offsets = {}
        self.shapes = {}
        total = 0
        for k, t in tensors.items():
            self.offsets[k] = total
            self.shapes[k] = tuple(t.shape)
            total += (t.numel() + 63) // 64 * 64
        host = torch.zeros(total, dtype=torch.float32)
        for k, t in tensors.items():
            o = self.offsets[k]
            host[o:o + t.numel()] = t.detach().to(torch.float32).reshape(-1).cpu()
        self.blob32 = host.to(device)
        self.blob16 = self.blob32.to(torch.bfloat16)
        _lib.check(_lib.load().mocha_register_bf16_blob(
            C.c_void_p(self.blob32.data_ptr()), C.c_void_p(self.blob16.data_ptr()), self.blob32.numel()),
            "mocha_register_bf16_blob")

    def __del__(self):
        try:
            _lib.load().mocha_register_bf16_blob(C.c_void_p(self.blob32.data_ptr()), None, self.blob32.numel())
        except Exception:
            pass

    def ptr(self, name: str) -> int:
        return self.blob32.data_ptr() + 4 * self.offsets[name]

    def view(self, name: str) -> torch.Tensor:
        o = self.offsets[name]
        n = 1
        for s in self.shapes[name]:
            n *= s
        return self.blob32[o:o + n].view(self.shapes[name])


def _conv_as_gemm(w: torch.Tensor) -> torch.Tensor:
    """Conv2d weight [Cout, Cin, taps, 1] -> [Cout, taps*Cin] (tap-major K)."""
    co, ci, taps, _ = w.shape
    return w[:, :, :, 0].permute(0, 2, 1).reshape(co, taps * ci).contiguous()


def _gcn_first(w: torch.Tensor, b: torch.Tensor, A: torch.Tensor):
    """SpatialConv 1x1 weight [K*Cout, Cin,1,1] applied AFTER graph aggregation.

    Returns W' [Cout, K*Cin] with W'[co, k*Cin+ci] = W[k*Cout+co, ci] and the bias table
    [V, Cout] = sum_k b[k*Cout+co] * sum_v A[k,v,w]  (bias flows through the einsum of blocks.py:64).
    """
    K = A.shape[0]
    kc, ci = w.shape[0], w.shape[1]
    co = kc // K
    w3 = w[:, :, 0, 0].reshape(K, co, ci)
    wp = w3.permute(1, 0, 2).reshape(co, K * ci).contiguous()
    colsum = A.sum(dim=1)                      # [K, V(w)]
    bias2d = torch.einsum("kc,kw->wc", b.reshape(K, co), colsum).contiguous()
    return wp, bias2d


def _gcn_first_aug(w: torch.Tensor, b: torch.Tensor, A: torch.Tensor) -> torch.Tensor:
    """W' of _gcn_first with K extra columns holding the per-partition biases b[k*Cout+co] (they multiply the
    adjacency column sums that the aggregation kernel appends to its rows), zero-padded to a multiple of 16 (one
    tcgen05 K step; the GEMM's 64-wide TMA boxes read past the last column and are zero-filled by the engine, so the
    padding up to 64 costs no HBM traffic)."""
    K = A.shape[0]
    wp, _ = _gcn_first(w, b, A)
    co = wp.shape[0]
    kaug = (wp.shape[1] + K + 15) // 16 * 16
    out = torch.zeros((co, kaug), dtype=torch.float32)
    out[:, :wp.shape[1]] = wp
    out[:, wp.shape[1]:wp.shape[1] + K] = b.reshape(K, co).t()
    return out.contiguous()


def generator_tensors(sd: "dict[str, torch.Tensor]", cfg: dict) -> "dict[str, torch.Tensor]":
    sd = {k: v.detach().to(torch.float32).cpu() for k, v in sd.items()}
    out = {}
    out["emb_w"] = sd["mot_embedding.1.weight"][:, :, 0, 0].contiguous()
    out["emb_b"] = sd["mot_embedding.1.bias"]
    A_j = sd["mot_embedding.2.A_j"]
    out["A_j"] = A_j
    out["jb_gcn_w"], out["jb_gcn_bias2d"] = _gcn_first(
        sd["mot_embedding.2.blk.gcn.conv.weight"], sd["mot_embedding.2.blk.gcn.conv.bias"], A_j)
    # tensor-core path: bias folded into the GEMM (extra K columns x adjacency column sums), K padded to 64
    out["jb_gcn_w_aug"] = _gcn_first_aug(
        sd["mot_embedding.2.blk.gcn.conv.weight"], sd["mot_embedding.2.blk.gcn.conv.bias"], A_j)
    out["jb_tcn_w"] = _conv_as_gemm(sd["mot_embedding.2.blk.tcn.weight"])
    out["jb_tcn_b"] = sd["mot_embedding.2.blk.tcn.bias"]
    out["pool_w"] = sd["mot_embedding.3.weight"]
    A_b = sd["mot_embedding.5.A_b"]
    out["A_b"] = A_b
    out["bb_gcn_w"], out["bb_gcn_bias2d"] = _gcn_first(
        sd["mot_embedding.5.blk.gcn.conv.weight"], sd["mot_embedding.5.blk.gcn.conv.bias"], A_b)
    out["bb_tcn_w"] = _conv_as_gemm(sd["mot_embedding.5.blk.tcn.weight"])
    out["bb_tcn_b"] = sd["mot_embedding.5.blk.tcn.bias"]
    out["pos_emb"] = sd["pos_emb"][0].contiguous()
    out["tok_bias_pos"] = (sd["pos_emb"][0] + sd["mot_embedding.5.blk.tcn.bias"][None, :]).contiguous()
    for l in range(cfg["encoder_depth"]):
        p = f"encoder.layers.{l}"
        out[f"enc{l}.wqkv"] = torch.cat(
            [sd[p + ".1.to_q.1.weight"], sd[p + ".1.to_k.1.weight"], sd[p + ".1.to_v.weight"]], dim=0).contiguous()
        out[f"enc{l}.wo"] = sd[p + ".1.to_out.0.weight"]
        out[f"enc{l}.bo"] = sd[p + ".1.to_out.0.bias"]
        out[f"enc{l}.w1"] = sd[p + ".2.net.0.weight"]
        out[f"enc{l}.b1"] = sd[p + ".2.net.0.bias"]
        out[f"enc{l}.w2"] = sd[p + ".2.net.3.weight"]
        out[f"enc{l}.b2"] = sd[p + ".2.net.3.bias"]
    for l in range(cfg["decoder_depth"]):
        p = f"decoder.layers.{l}"
        out[f"dec{l}.sw1"] = sd[p + ".0.style.2.weight"]
        out[f"dec{l}.sb1"] = sd[p + ".0.style.2.bias"]
        out[f"dec{l}.sw2"] = sd[p + ".0.style.4.weight"]
        out[f"dec{l}.sb2"] = sd[p + ".0.style.4.bias"]
        out[f"dec{l}.wq"] = sd[p + ".1.to_q.1.weight"]
        out[f"dec{l}.wk"] = sd[p + ".1.to_k.1.weight"]
        out[f"dec{l}.wv"] = sd[p + ".1.to_v.weight"]
        out[f"dec{l}.wo"] = sd[p + ".1.to_out.0.weight"]
        out[f"dec{l}.bo"] = sd[p + ".1.to_out.0.bias"]
        out[f"dec{l}.w1"] = sd[p + ".2.net.0.weight"]
        out[f"dec{l}.b1"] = sd[p + ".2.net.0.bias"]
        out[f"dec{l}.w2"] = sd[p + ".2.net.3.weight"]
        out[f"dec{l}.b2"] = sd[p + ".2.net.3.bias"]
    tA_b = sd["to_mot.1.A_b"]
    out["tm_A_b"] = tA_b
    out["tm_bb_gcn_w"], out["tm_bb_gcn_bias2d"] = _gcn_first(
        sd["to_mot.1.blk.gcn.conv.weight"], sd["to_mot.1.blk.gcn.conv.bias"], tA_b)
    out["tm_bb_tcn_w"] = _conv_as_gemm(sd["to_mot.1.blk.tcn.weight"])
    out["tm_bb_tcn_b"] = sd["to_mot.1.blk.tcn.bias"]
    out["tm_jb_gcn_w"] = sd["to_mot.4.blk.gcn.conv.weight"][:, :, 0, 0].contiguous()
    out["tm_jb_gcn_b"] = sd["to_mot.4.blk.gcn.conv.bias"]
    # fold UnpoolBodypartToJoint (graph.py:606-608) into the joint adjacency: A2[k,p,w] = sum_v U[p,v] A[k,v,w]
    out["tm_A2"] = torch.einsum("pv,kvw->kpw", sd["to_mot.3.weight"], sd["to_mot.4.A_j"]).contiguous()
    out["tm_jb_tcn_w"] = _conv_as_gemm(sd["to_mot.4.blk.tcn.weight"])
    out["tm_jb_tcn_b"] = sd["to_mot.4.blk.tcn.bias"]
    out["tm_out_w"] = sd["to_mot.6.weight"][:, :, 0, 0].contiguous()
    out["tm_out_b"] = sd["to_mot.6.bias"]
    return out


def make_dims(cfg: dict, sd: "dict[str, torch.Tensor]") -> _lib.Dims:
    d = _lib.Dims()
    d.T = cfg["nframes"]
    d.V = cfg["njoints"]
    d.Cin = cfg["mot_in_dim"]
    d.tp = cfg["temporal_patch_size"]
    d.D = cfg["encoder_dim"]
    d.C0 = cfg["encoder_dim"] // cfg["temporal_patch_size"]
    d.P = cfg.get("nbody", 6)
    d.Kj = sd["mot_embedding.2.A_j"].shape[0]
    d.Kb = sd["mot_embedding.5.A_b"].shape[0]
    d.taps_j = sd["mot_embedding.2.blk.tcn.weight"].shape[2]
    d.taps_b = sd["mot_embedding.5.blk.tcn.weight"].shape[2]
    d.heads = cfg["encoder_heads"]
    d.enc_dh = cfg["encoder_dim_head"]
    d.dec_dh = cfg["decoder_dim_head"]
    d.mlp = cfg["encoder_mlp_dim"]
    d.enc_depth = cfg["encoder_depth"]
    d.dec_depth = cfg["decoder_depth"]
    if cfg["decoder_dim"] != cfg["encoder_dim"] or cfg["decoder_heads"] != cfg["encoder_heads"] \
            or cfg["decoder_mlp_dim"] != cfg["encoder_mlp_dim"]:
        raise _lib.MochaError("encoder/decoder dim, heads and mlp_dim must match (configs/config.yaml does)")
    return d


class PackedGenerator:
    def __init__(self, sd, cfg, device):
        self.cfg = cfg
        self.blob = PackedBlob(generator_tensors(sd, cfg), device)
        w = _lib.GeneratorWeights()
        w.dims = make_dims(cfg, sd)
        b = self.blob
        for name in ("emb_w", "emb_b", "A_j", "jb_gcn_w", "jb_gcn_bias2d", "jb_tcn_w", "jb_tcn_b", "pool_w", "A_b",
                     "bb_gcn_w", "bb_gcn_bias2d", "bb_tcn_w", "bb_tcn_b", "pos_emb", "tok_bias_pos", "tm_A_b",
                     "tm_bb_gcn_w", "tm_bb_gcn_bias2d", "tm_bb_tcn_w", "tm_bb_tcn_b", "tm_jb_gcn_w", "tm_jb_gcn_b",
                     "tm_A2", "tm_jb_tcn_w", "tm_jb_tcn_b", "tm_out_w", "tm_out_b"):
            setattr(w, name, b.ptr(name))
        w.jb_gcn_w_aug = b.ptr("jb_gcn_w_aug")
        w.jb_gcn_kaug = int(b.shapes["jb_gcn_w_aug"][1])
        for l in range(cfg["encoder_depth"]):
            for f in ("wqkv", "wo", "bo", "w1", "b1", "w2", "b2"):
                setattr(w.enc[l], f, b.ptr(f"enc{l}.{f}"))
        for l in range(cfg["decoder_depth"]):
            for f in ("sw1", "sb1", "sw2", "sb2", "wq", "wk", "wv", "wo", "bo", "w1", "b1", "w2", "b2"):
                setattr(w.dec[l], f, b.ptr(f"dec{l}.{f}"))
        self.struct = w
        self.dims = w.dims
        self.ntok = (w.dims.T // w.dims.tp) * w.dims.P


def cvae_tensors(sd, depth: int, token_net: str = "prior_net") -> "dict[str, torch.Tensor]":
    """token_net = "prior_net" (PriorNet, model_CVAE.py:49-93) or "encoder" (the posterior Encoder, :95-135: the same
    network over [mu, logvar, c, x] with its own weights) fills the `prior` slots of the ABI struct."""
    sd = {k: v.detach().to(torch.float32).cpu() for k, v in sd.items()}
    out = {
        "mu_token": sd[f"{token_net}.mu_token"].reshape(-1),
        "logvar_token": sd[f"{token_net}.logvar_token"].reshape(-1),
        "pe": sd[f"{token_net}.pos_encoder.pe"][0, :512].contiguous(),
    }
    for l in range(depth):
        p = f"{token_net}.encoder.layers.{l}"
        out[f"pr{l}.in_w"] = sd[p + ".self_attn.in_proj_weight"]
        out[f"pr{l}.in_b"] = sd[p + ".self_attn.in_proj_bias"]
        out[f"pr{l}.out_w"] = sd[p + ".self_attn.out_proj.weight"]
        out[f"pr{l}.out_b"] = sd[p + ".self_attn.out_proj.bias"]
        out[f"pr{l}.l1_w"] = sd[p + ".linear1.weight"]
        out[f"pr{l}.l1_b"] = sd[p + ".linear1.bias"]
        out[f"pr{l}.l2_w"] = sd[p + ".linear2.weight"]
        out[f"pr{l}.l2_b"] = sd[p + ".linear2.bias"]
        out[f"pr{l}.n1_g"] = sd[p + ".norm1.weight"]
        out[f"pr{l}.n1_b"] = sd[p + ".norm1.bias"]
        out[f"pr{l}.n2_g"] = sd[p + ".norm2.weight"]
        out[f"pr{l}.n2_b"] = sd[p + ".norm2.bias"]
        q = f"decoder.decoder.layers.{l}"
        out[f"de{l}.sa_in_w"] = sd[q + ".self_attn.in_proj_weight"]
        out[f"de{l}.sa_in_b"] = sd[q + ".self_attn.in_proj_bias"]
        out[f"de{l}.sa_out_w"] = sd[q + ".self_attn.out_proj.weight"]
        out[f"de{l}.sa_out_b"] = sd[q + ".self_attn.out_proj.bias"]
        out[f"de{l}.ca_in_w"] = sd[q + ".multihead_attn.in_proj_weight"]
        out[f"de{l}.ca_in_b"] = sd[q + ".multihead_attn.in_proj_bias"]
        out[f"de{l}.ca_out_w"] = sd[q + ".multihead_attn.out_proj.weight"]
        out[f"de{l}.ca_out_b"] = sd[q + ".multihead_attn.out_proj.bias"]
        out[f"de{l}.l1_w"] = sd[q + ".linear1.weight"]
        out[f"de{l}.l1_b"] = sd[q + ".linear1.bias"]
        out[f"de{l}.l2_w"] = sd[q + ".linear2.weight"]
        out[f"de{l}.l2_b"] = sd[q + ".linear2.bias"]
        for n in ("1", "2", "3"):
            out[f"de{l}.n{n}_g"] = sd[q + f".norm{n}.weight"]
            out[f"de{l}.n{n}_b"] = sd[q + f".norm{n}.bias"]
    return out


class PackedCVAE:
    def __init__(self, sd, output_seq: int, latent_dim: int, depth: int, nheads: int, dff: int, device,
                 token_net: str = "prior_net"):
        self.blob = PackedBlob(cvae_tensors(sd, depth, token_net), device)
        w = _lib.CvaeWeights()
        w.D, w.heads, w.dff, w.depth, w.out_seq = latent_dim, nheads, dff, depth, output_seq
        w.ln_eps = 1e-5
        b = self.blob
        w.mu_token, w.logvar_token, w.pe = b.ptr("mu_token"), b.ptr("logvar_token"), b.ptr("pe")
        for l in range(depth):
            for f in ("in_w", "in_b", "out_w", "out_b", "l1_w", "l1_b", "l2_w", "l2_b", "n1_g", "n1_b", "n2_g", "n2_b"):
                setattr(w.prior[l], f, b.ptr(f"pr{l}.{f}"))
            for f in ("sa_in_w", "sa_in_b", "sa_out_w", "sa_out_b", "ca_in_w", "ca_in_b", "ca_out_w", "ca_out_b",
                      "l1_w", "l1_b", "l2_w", "l2_b", "n1_g", "n1_b", "n2_g", "n2_b", "n3_g", "n3_b"):
                setattr(w.dec[l], f, b.ptr(f"de{l}.{f}"))
        w.dec0_sa = None
        w.dec0_q16 = None
        self.struct = w
        # decoder layer 0's self-attention block acts on the constant positional query: compute it once
        lib = _lib.load()
        self.dec0_sa = torch.empty((output_seq, latent_dim), dtype=torch.float32, device=device)
        ws = torch.empty(16 << 20, dtype=torch.uint8, device=device)
        _lib.check(lib.mocha_cvae_precompute_dec0(C.byref(w), C.c_void_p(self.dec0_sa.data_ptr()),
                                                  C.c_void_p(ws.data_ptr()), ws.numel(),
                                                  C.c_void_p(torch.cuda.current_stream(device).cuda_stream)),
                   "mocha_cvae_precompute_dec0")
        torch.cuda.current_stream(device).synchronize()
        w.dec0_sa = self.dec0_sa.data_ptr()
        # ... and so does the layer-0 cross-attention query projection of that table (bf16 operands, like the per-clip
        # projection it replaces): mocha_linear in bf16 mode on the registered weight blob
        D = latent_dim
        q32 = torch.empty((output_seq, D), dtype=torch.float32, device=device)
        wsb = lib.mocha_linear_workspace_bytes(output_seq, D, D, _lib.MOCHA_BF16)
        ws2 = torch.empty(max(int(wsb), 256), dtype=torch.uint8, device=device)
        _lib.check(lib.mocha_linear(C.c_void_p(self.dec0_sa.data_ptr()), C.c_void_p(b.ptr("de0.ca_in_w")),
                                    C.c_void_p(b.ptr("de0.ca_in_b")), None, C.c_void_p(q32.data_ptr()), output_seq, D, D, 0,
                                    _lib.MOCHA_BF16, C.c_void_p(ws2.data_ptr()), ws2.numel(),
                                    C.c_void_p(torch.cuda.current_stream(device).cuda_stream)), "mocha_linear(dec0 query)")
        torch.cuda.current_stream(device).synchronize()
        self.dec0_q16 = q32.to(torch.bfloat16).contiguous()
        w.dec0_q16 = self.dec0_q16.data_ptr()
