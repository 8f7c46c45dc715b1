"""Model geometries other than the default config, stage by stage, against the NumPy oracle.

The Generator and CVAE dispatchers pick kernel variants from the model geometry (width, head size, MLP width, graph hop
count, clip length) and the batch size. The default config reaches only one side of most of those choices; a checkpoint
with another geometry lands on the other side. Each row below changes the default config so that a named set of variants
runs. Every stage runs on the oracle's input to that stage (errors do not compound) in every precision mode, and one
extra call per stage runs under torch.profiler to prove that the promised kernels ran and the default ones did not.

The CPU part (`-m "not gpu"`) checks that every row's weights build, packing accepts its dims and the oracle runs it.
"""
from __future__ import annotations

import copy
import functools
import re

import numpy as np
import pytest
import torch

from mocha_oracle import nets
from mocha_sigasia2023_b200 import packing, weights

RTOL_FP32 = 1e-4    # fp32 and 3xTF32 modes (north star)
RTOL_BF16 = 2e-2    # the suite's bf16 bound; the rows below are held to a tighter one, calibrated on the default row

# ---------------------------------------------------------------------------------------------------------------------
# Rows: config changes from weights.DEFAULT_MODEL_CFG (Generator) or from CVAE's default arguments
# ---------------------------------------------------------------------------------------------------------------------
GEN_ROWS = {
    "default": {},
    "wide512": {"encoder_dim": 512, "decoder_dim": 512},                        # C0 = 128
    "hop4": {"graph": {"joint": {"layout": "mocha", "strategy": "distance", "max_hop": 4},
                       "bodypart": {"layout": "mocha", "strategy": "distance", "max_hop": 4}}},   # Kj = Kb = 5
    "dh192": {"encoder_heads": 2, "decoder_heads": 2, "encoder_dim_head": 192, "decoder_dim_head": 64},
    "mlp1024": {"encoder_mlp_dim": 1024, "decoder_mlp_dim": 1024, "encoder_depth": 3, "decoder_depth": 1},
    "mlp384": {"encoder_mlp_dim": 384, "decoder_mlp_dim": 384},
    "t120": {"nframes": 120},                                                    # 180 tokens
}
# (row, batch): every row at B = 3; the style MLP and the CTA-pair / halo convolutions switch on the batch size
GEN_CASES = [("default", 3), ("default", 64), ("default", 65), ("wide512", 3), ("hop4", 3), ("dh192", 3),
             ("mlp1024", 3), ("mlp1024", 64), ("mlp1024", 65), ("mlp384", 3), ("t120", 3)]

CVAE_ROWS = {
    "default": dict(latent_dim=256, depth=2, nheads=4, dff=512),
    "cvae512": dict(latent_dim=512, depth=2, nheads=4, dff=512),
    "cvae_ff1024": dict(latent_dim=256, depth=2, nheads=4, dff=1024),
    "cvae_h2_d3": dict(latent_dim=256, depth=3, nheads=2, dff=512),
}
CVAE_B, CVAE_NCOND, CVAE_NX, CVAE_OUT = 3, 180, 90, 90

PRECISIONS = ("fp32", "tf32x3", "bf16")
GEN_STAGES = ("embed", "encoder", "decoder", "to_mot")
CVAE_STAGES = ("sample", "encode")

# ---------------------------------------------------------------------------------------------------------------------
# Kernel variants, matched on the demangled names the profiler reports (symbols of the sm_100a build, `cuobjdump
# -symbols`); the alternations accept both demangler spellings of template arguments ("4" / "(int)4", "true" / "(bool)1").
# ---------------------------------------------------------------------------------------------------------------------
KERNELS = {
    "embed_mma": r"embed_graph_agg_mma_kernel",
    "embed_simt": r"embed_graph_agg_kernel",
    "pool_v4": r"pool_graph_agg_v4_kernel",
    "pool_list": r"pool_graph_agg_kernel",
    "pool_joint_body": r"pool_joint_body_kernel",
    "agg_small": r"graph_agg_small_kernel",
    "agg_first": r"graph_agg_first_kernel",
    "agg_kv": r"graph_agg_kv_kernel",
    "kv_stream": r"graph_agg_kv_pad16_stream_kernel",
    "kv_list": r"graph_agg_kv_pad16_kernel",
    "tail": r"\btail_kernel",
    "attn_fused": r"\battn_kernel",
    "attn_two_launch": r"tc_gemm_kernel<[^>]*SoftmaxEpi",
    "style_mlp": r"style_mlp_kernel",
    "style_mlp_cluster": r"style_mlp_cluster_kernel",
    "token_mean": r"token_mean_kernel",
    "in_v4": r"instance_norm_tokens_v4_kernel",
    "in_reg": r"instance_norm_tokens_reg_kernel",
    "in_general": r"instance_norm_tokens_kernel",
    "tconv_halo": r"tc_gemm_kernel<(\(int\))?64, [^,]*LinearEpiT<(\(int\))?4>, (true|\(bool\)1)>",
    "gemm_pair": r"tc_gemm2_kernel",
    "out_affine_k64": r"out_conv_affine_kernel<(\(int\))?4>",
    "out_affine_k128": r"out_conv_affine_kernel<(\(int\))?8>",
    "prior_last": r"cvae_prior_last_kernel",
    "prior_last_dff1024": r"cvae_prior_last_kernel<(\(int\))?4>",
    "gather_rows": r"gather_token_rows_kernel",
    "broadcast_rows": r"broadcast_rows_kernel",
    "sgemm": r"sgemm_kernel",
    "tc_bf16": r"LinearEpiT<",
    "tc_tf32x3": r"LinearEpiTf<",
    "tensor_core": r"tc_gemm|\battn_kernel|\btail_kernel",
}

# Per precision mode, what every row's stages must (not) run: fp32 never touches the tensor cores, 3xTF32 never the bf16
# kernels.
MODE_EXPECT = {
    "fp32": {"embed": (["sgemm", "agg_first", "pool_joint_body"], ["tensor_core"]),
             "encoder": (["sgemm"], ["tensor_core"]),
             "decoder": (["sgemm", "token_mean"], ["tensor_core"]),
             "to_mot": (["sgemm", "agg_first", "agg_kv"], ["tensor_core"]),
             "sample": (["sgemm"], ["tensor_core"]),
             "encode": (["sgemm"], ["tensor_core"])},
    "tf32x3": {"embed": (["tc_tf32x3", "agg_first", "pool_joint_body"], ["tc_bf16", "attn_fused", "tail"]),
               "encoder": (["tc_tf32x3"], ["tc_bf16", "attn_fused", "tail"]),
               "decoder": (["tc_tf32x3", "token_mean"], ["tc_bf16", "attn_fused", "tail"]),
               "to_mot": (["tc_tf32x3", "agg_first", "agg_kv"], ["tc_bf16", "attn_fused", "tail"]),
               "sample": (["tc_tf32x3"], ["tc_bf16", "attn_fused", "tail"]),
               "encode": (["tc_tf32x3"], ["tc_bf16", "attn_fused", "tail"])},
    "bf16": {s: (["tc_bf16"], ["sgemm"]) for s in GEN_STAGES + ("sample",)},
}
# the CVAE posterior (272 tokens, more than the tensor-core attention takes) runs its attention on the SIMT GEMM
MODE_EXPECT["bf16"]["encode"] = (["tc_bf16", "sgemm"], ["attn_fused", "tail"])

# The variants each row exists for, in bf16 mode: {(row, B) or row: {stage: (present, absent)}}. A later dispatch change
# that moves a row off its variant fails here ("variant X is no longer covered") instead of quietly losing the coverage.
_DEFAULT_BF16 = {
    "embed": (["embed_mma", "pool_v4"], ["embed_simt", "pool_list"]),
    "encoder": (["attn_fused", "tail"], ["attn_two_launch"]),
    "decoder": (["style_mlp", "in_v4", "attn_fused", "tail"], ["token_mean", "in_general", "style_mlp_cluster", "attn_two_launch"]),
    "to_mot": (["agg_small", "kv_stream", "out_affine_k64"], ["agg_first", "kv_list", "out_affine_k128"]),
}
GEN_BF16_EXPECT = {
    ("default", 3): _DEFAULT_BF16,
    # 64 clips: style MLP on CTA pairs (clusters of two), the JointBlock conv on the CTA-pair kernel, to_mot's 64 -> 64
    # conv on the halo kernel (both need a grid of at least ~one wave)
    ("default", 64): {"embed": (["embed_mma", "gemm_pair"], []),
                      "decoder": (["style_mlp_cluster"], ["style_mlp"]),
                      "to_mot": (["tconv_halo", "kv_stream"], [])},
    # an odd batch above 64 keeps the unclustered style MLP
    ("default", 65): {"embed": (["gemm_pair"], []),
                      "decoder": (["style_mlp"], ["style_mlp_cluster"]),
                      "to_mot": (["tconv_halo"], [])},
    # C0 = 128: SIMT embedding aggregation; D = 512: unfused block tails, token mean + per-layer style GEMMs,
    # to_mot's 128 -> 128 conv on the general kernel and the output layer at K = 128
    ("wide512", 3): {"embed": (["embed_simt", "pool_v4"], ["embed_mma"]),
                     "encoder": (["attn_fused"], ["tail"]),
                     "decoder": (["token_mean", "in_v4", "attn_fused"], ["style_mlp", "style_mlp_cluster", "tail"]),
                     "to_mot": (["agg_small", "kv_stream", "out_affine_k128"], ["out_affine_k64", "tconv_halo"])},
    # Kj = Kb = 5: SIMT embedding (K_aug = 325 -> 336), list-based to_mot aggregations (Kb > 4, Kj * P = 30 > 24)
    ("hop4", 3): {"embed": (["embed_simt", "pool_v4"], ["embed_mma"]),
                  "encoder": (["attn_fused", "tail"], []),
                  "to_mot": (["agg_first", "kv_list", "out_affine_k64"], ["agg_small", "kv_stream"])},
    # dh = 192: Q K^T with the softmax epilogue, then P V (the fused kernel takes 64 / 128 / 256); tails at K0 = 384 / 128
    ("dh192", 3): {"encoder": (["attn_two_launch", "tail"], ["attn_fused"]),
                   "decoder": (["attn_fused", "tail", "style_mlp"], ["attn_two_launch"])},
    # hidden width 1024 > the fused tail's 512: unfused tails; one decoder layer in the style MLP
    ("mlp1024", 3): {"encoder": (["attn_fused"], ["tail"]),
                     "decoder": (["style_mlp", "attn_fused"], ["tail", "token_mean"])},
    ("mlp1024", 64): {"embed": (["gemm_pair"], []),
                      "encoder": ([], ["tail"]),
                      "decoder": (["style_mlp_cluster"], ["style_mlp", "tail"]),
                      "to_mot": (["tconv_halo"], [])},
    ("mlp1024", 65): {"encoder": ([], ["tail"]),
                      "decoder": (["style_mlp"], ["style_mlp_cluster", "tail"])},
    # hidden width 384: the fused tail in three 128-column chunks
    ("mlp384", 3): {"encoder": (["tail"], []), "decoder": (["tail"], [])},
    # 180 tokens: general instance norm (n > 128) instead of the AdaIN pass, the encoder's fused attention over two
    # query tiles, the decoder's dh = 256 attention on the two-launch path (its K / V no longer fit the fused kernel)
    ("t120", 3): {"encoder": (["attn_fused", "tail"], ["attn_two_launch"]),
                  "decoder": (["in_general", "attn_two_launch", "tail"], ["in_v4", "attn_fused"]),
                  "to_mot": (["agg_small", "kv_stream", "out_affine_k64"], [])},
}
CVAE_BF16_EXPECT = {
    # the last prior layer on its two read rows in one SIMT kernel; decoder layer 0 on the shared query table
    "default": {"sample": (["prior_last", "attn_fused", "tail"], ["gather_rows", "broadcast_rows"])},
    # D = 512: gathered rows + two-row attention + unfused tail; layer 0 broadcasts the cached self-attention table
    "cvae512": {"sample": (["gather_rows", "broadcast_rows", "attn_fused"], ["prior_last", "tail"])},
    # dff = 1024: unfused FFN tails (only the FFN-less self-attention tails stay fused), prior_last at dff = 1024
    "cvae_ff1024": {"sample": (["prior_last_dff1024", "broadcast_rows", "attn_fused"], ["gather_rows"])},
    # H = 2 (dh = 128), three layers: the K / V of decoder layers 1 and 2 projected ahead on the side stream
    "cvae_h2_d3": {"sample": (["prior_last", "attn_fused", "tail"], ["gather_rows", "broadcast_rows"])},
}
# fp32-side variants of the same geometries (networks.cu)
GEN_FP32_EXPECT = {
    ("t120", 3): {"decoder": (["in_general"], ["in_reg"])},
    ("default", 3): {"decoder": (["in_reg"], ["in_general"])},
}

# bf16: each stage's error on a row is held to BF16_MULT x the default row's error at that stage (B = 3, measured in
# the same run), capped at RTOL_BF16. Default-row errors measured on a B200 (power limit 1000 W): tokens 2.5e-3,
# encoded 1.0e-3, decoded 1.1e-3, Ytil 1.8e-3; CVAE det 1.6e-3, eps_out 1.7e-3, mu 1.3e-3, logvar 1.4e-3, enc_mu 1.2e-3,
# enc_logvar 1.3e-3, fwd 1.7e-3. The largest ratio of another row to these was 1.6 (cvae_h2_d3 enc_mu); no row needed an
# allowance, the longer contractions (hop4's K = 1280 gcn, mlp1024) included.
BF16_MULT = 4.0


def gen_cfg(row: str) -> dict:
    cfg = copy.deepcopy(weights.DEFAULT_MODEL_CFG)
    cfg.update(copy.deepcopy(GEN_ROWS[row]))
    return cfg


def rel_err(a, b) -> float:
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def _ntok(cfg):
    return cfg["nbody"] * (cfg["nframes"] // cfg["temporal_patch_size"])


@functools.lru_cache(maxsize=None)
def gen_oracle(row: str, B: int):
    """Inputs and outputs of every Generator stage, each stage fed the oracle's output of the previous one."""
    cfg = gen_cfg(row)
    sd = {k: v.numpy() for k, v in weights.generator_state_dict(1777, cfg).items()}
    rng = np.random.default_rng(1000 + B + 17 * list(GEN_ROWS).index(row))
    X = rng.standard_normal((B, cfg["nframes"], cfg["njoints"], cfg["mot_in_dim"])).astype(np.float32)
    tp, n = cfg["temporal_patch_size"], _ntok(cfg)
    tokens = nets.mot_embedding(sd, X, tp)
    tok_in = (tokens + sd["pos_emb"][:, :n]).astype(np.float32)
    enc = nets.encoder(sd, tok_in, cfg["encoder_depth"], cfg["encoder_heads"])
    sty = np.ascontiguousarray(enc[::-1])
    dec = nets.decoder(sd, enc, sty, cfg["decoder_depth"], cfg["decoder_heads"])
    y = nets.to_mot(sd, dec, tp, cfg["nbody"])
    return {"X": X, "tokens": tokens, "tok_in": tok_in, "encoded": enc, "style": sty, "decoded": dec, "Ytil": y}


@functools.lru_cache(maxsize=None)
def cvae_oracle(row: str):
    p = CVAE_ROWS[row]
    D, depth, H = p["latent_dim"], p["depth"], p["nheads"]
    sd = {k: v.numpy() for k, v in weights.cvae_state_dict(1778, D, depth, p["dff"]).items()}
    rng = np.random.default_rng(2000 + list(CVAE_ROWS).index(row))
    cond = rng.standard_normal((CVAE_B, CVAE_NCOND, D)).astype(np.float32)
    eps = rng.standard_normal((CVAE_B, D)).astype(np.float32)
    x = rng.standard_normal((CVAE_B, CVAE_NX, D)).astype(np.float32)
    det, mu, logvar = nets.cvae_sample(sd, cond, None, CVAE_OUT, depth, H)
    out_eps, _, _ = nets.cvae_sample(sd, cond, eps, CVAE_OUT, depth, H)
    enc_mu, enc_logvar = nets.cvae_encode(sd, x, cond, depth, H)
    fwd, _, (fwd_mu_pr, fwd_lv_pr) = nets.cvae_forward(sd, x, cond, eps, CVAE_OUT, depth, H)
    return {"cond": cond, "eps": eps, "x": x, "det": det, "mu": mu, "logvar": logvar, "eps_out": out_eps,
            "enc_mu": enc_mu, "enc_logvar": enc_logvar, "fwd": fwd, "fwd_mu_pr": fwd_mu_pr, "fwd_logvar_pr": fwd_lv_pr}


# ---------------------------------------------------------------------------------------------------------------------
# CPU part: the row table stays buildable and the oracle runs every row
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("row", list(GEN_ROWS))
def test_generator_row_builds_and_oracle_runs(row):
    cfg = gen_cfg(row)
    sd = weights.generator_state_dict(1777, cfg)
    d = packing.make_dims(cfg, sd)
    assert (d.D, d.C0, d.T) == (cfg["encoder_dim"], cfg["encoder_dim"] // 4, cfg["nframes"])
    assert (d.Kj, d.Kb) == (cfg["graph"]["joint"]["max_hop"] + 1, cfg["graph"]["bodypart"]["max_hop"] + 1)
    assert (d.heads, d.enc_dh, d.dec_dh, d.mlp) == (cfg["encoder_heads"], cfg["encoder_dim_head"],
                                                    cfg["decoder_dim_head"], cfg["encoder_mlp_dim"])
    assert (d.enc_depth, d.dec_depth) == (cfg["encoder_depth"], cfg["decoder_depth"])
    # the bf16 stages need C0 % 64 == 0 and at most 256 tokens, else the whole stage silently runs the fp32 path
    assert d.C0 % 64 == 0 and _ntok(cfg) <= 256
    o = gen_oracle(row, 2)
    n, D = _ntok(cfg), cfg["encoder_dim"]
    for k in ("tokens", "encoded", "decoded"):
        assert o[k].shape == (2, n, D) and np.isfinite(o[k]).all(), k
    assert o["Ytil"].shape == (2, cfg["nframes"], cfg["njoints"], cfg["mot_in_dim"]) and np.isfinite(o["Ytil"]).all()


@pytest.mark.parametrize("row", list(CVAE_ROWS))
def test_cvae_row_builds_and_oracle_runs(row):
    p = CVAE_ROWS[row]
    D = p["latent_dim"]
    sd = weights.cvae_state_dict(1778, D, p["depth"], p["dff"])
    assert sd["prior_net.encoder.layers.0.linear1.weight"].shape == (p["dff"], D)
    assert f"decoder.decoder.layers.{p['depth'] - 1}.norm3.weight" in sd
    # the tensor-core attention takes head widths that are multiples of 64; a smaller one sends the CVAE to fp32
    assert (D // p["nheads"]) % 64 == 0
    o = cvae_oracle(row)
    for k in ("det", "eps_out", "fwd"):
        assert o[k].shape == (CVAE_B, CVAE_OUT, D) and np.isfinite(o[k]).all(), k
    for k in ("mu", "logvar", "enc_mu", "enc_logvar", "fwd_mu_pr", "fwd_logvar_pr"):
        assert o[k].shape == (CVAE_B, D) and np.isfinite(o[k]).all(), k


# ---------------------------------------------------------------------------------------------------------------------
# GPU part
# ---------------------------------------------------------------------------------------------------------------------
def cu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


@functools.lru_cache(maxsize=None)
def generator(row: str, precision: str):
    from mocha_sigasia2023_b200.model import Generator
    cfg = gen_cfg(row)
    g = Generator(cfg, precision=precision)
    g.load_state_dict(weights.generator_state_dict(1777, cfg), strict=True)
    return g.to("cuda").eval()


@functools.lru_cache(maxsize=None)
def cvae_model(row: str, precision: str):
    from mocha_sigasia2023_b200.model_CVAE import CVAE
    p = CVAE_ROWS[row]
    c = CVAE(output_seq=CVAE_OUT, latent_dim=p["latent_dim"], depth=p["depth"], nheads=p["nheads"],
             feedforward_dim=p["dff"], precision=precision)
    c.load_state_dict(weights.cvae_state_dict(1778, p["latent_dim"], p["depth"], p["dff"]), strict=True)
    return c.to("cuda").eval()


def gen_stage_calls(row, B, precision):
    """{stage: zero-argument call returning the stage output as a CUDA tensor} on the oracle's stage inputs."""
    g, o = generator(row, precision), gen_oracle(row, B)
    X, tok_in, enc, sty, dec = cu(o["X"]), cu(o["tok_in"]), cu(o["encoded"]), cu(o["style"]), cu(o["decoded"])
    return {"embed": lambda: g.mot_embedding(X), "encoder": lambda: g.encoder(tok_in),
            "decoder": lambda: g.decoder(enc, sty), "to_mot": lambda: g.to_mot(dec)}


def cvae_stage_calls(row, precision):
    c, o = cvae_model(row, precision), cvae_oracle(row)
    cond, x = cu(o["cond"]), cu(o["x"])
    return {"sample": lambda: c.sample(cond, deterministic=True), "encode": lambda: c.encode(x, cond)}


@functools.lru_cache(maxsize=None)
def gen_errors(row: str, B: int, precision: str) -> dict:
    o = gen_oracle(row, B)
    calls = gen_stage_calls(row, B, precision)
    errs = {}
    for stage, want in zip(GEN_STAGES, ("tokens", "encoded", "decoded", "Ytil")):
        got = calls[stage]().cpu().numpy()
        assert got.shape == o[want].shape and np.isfinite(got).all(), (row, B, precision, stage)
        errs[want] = rel_err(got, o[want])
    return errs


@functools.lru_cache(maxsize=None)
def cvae_errors(row: str, precision: str) -> dict:
    c, o = cvae_model(row, precision), cvae_oracle(row)
    cond, x = cu(o["cond"]), cu(o["x"])
    got = {"det": c.sample(cond, deterministic=True)}
    got["mu"], got["logvar"] = c.prior(cond)
    c.eps_fn = lambda shape: torch.from_numpy(o["eps"])
    try:
        got["eps_out"] = c.sample(cond, deterministic=False)
    finally:
        c.eps_fn = None
    got["enc_mu"], got["enc_logvar"] = c.encode(x, cond)
    draws = iter([torch.from_numpy(o["eps"]), torch.zeros(o["eps"].shape)])    # posterior draw, then the prior's
    c.eps_fn = lambda shape: next(draws)
    try:
        got["fwd"], (mu_po, lv_po), (got["fwd_mu_pr"], got["fwd_logvar_pr"]) = c(x, cond)
    finally:
        c.eps_fn = None
    errs = {}
    for k, v in got.items():
        v = v.cpu().numpy()
        assert v.shape == o[k].shape and np.isfinite(v).all(), (row, precision, k)
        errs[k] = rel_err(v, o[k])
    # the posterior's mu / logvar inside forward are encode's
    errs["enc_mu"] = max(errs["enc_mu"], rel_err(mu_po.cpu().numpy(), o["enc_mu"]))
    errs["enc_logvar"] = max(errs["enc_logvar"], rel_err(lv_po.cpu().numpy(), o["enc_logvar"]))
    return errs


def _check_errors(errs, base, row, precision):
    bad = []
    for k, e in errs.items():
        if precision != "bf16":
            # forward's output goes through z_po -> eps' -> z (one more rounding step than sample): 2x, as in test_gpu_nets
            bound = 2 * RTOL_FP32 if k == "fwd" else RTOL_FP32
        elif base is None:
            bound = RTOL_BF16
        else:
            bound = min(BF16_MULT * base[k], RTOL_BF16)
        if not e < bound:
            bad.append(f"{k}: {e:.3e} >= {bound:.3e}")
    assert not bad, f"{row} {precision}: " + "; ".join(bad)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("row,B", GEN_CASES, ids=[f"{r}-B{b}" for r, b in GEN_CASES])
def test_generator_stages_match_oracle(row, B, precision):
    errs = gen_errors(row, B, precision)
    base = gen_errors("default", 3, "bf16") if precision == "bf16" and (row, B) != ("default", 3) else None
    _check_errors(errs, base, f"{row}-B{B}", precision)


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("row", list(CVAE_ROWS))
def test_cvae_surfaces_match_oracle(row, precision):
    errs = cvae_errors(row, precision)
    base = cvae_errors("default", "bf16") if precision == "bf16" and row != "default" else None
    _check_errors(errs, base, row, precision)


def kernels_run_by(fn) -> list:
    """Names of the CUDA kernels one call launches (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn()                                 # packing and first-use set-up outside the profiled call
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sorted({ev.key for ev in prof.key_averages() if ev.device_type == torch.autograd.DeviceType.CUDA})


def _check_variants(names, expect, where):
    missing, unexpected = [], []
    for stage, (present, absent) in expect.items():
        ran = names[stage]
        for v in present:
            if not any(re.search(KERNELS[v], n) for n in ran):
                missing.append(f"{stage}: variant {v} is no longer covered")
        for v in absent:
            hits = [n[:100] for n in ran if re.search(KERNELS[v], n)]
            if hits:
                unexpected.append(f"{stage}: {v} ran ({hits[0]})")
    assert not (missing or unexpected), f"{where}: " + "; ".join(missing + unexpected)


def _merge(*tables):
    out = {}
    for t in tables:
        for stage, (present, absent) in t.items():
            p, a = out.get(stage, ([], []))
            out[stage] = (p + list(present), a + list(absent))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("row,B", GEN_CASES, ids=[f"{r}-B{b}" for r, b in GEN_CASES])
def test_generator_variants_ran(row, B, precision):
    calls = gen_stage_calls(row, B, precision)
    names = {stage: kernels_run_by(calls[stage]) for stage in GEN_STAGES}
    mode = {s: MODE_EXPECT[precision][s] for s in GEN_STAGES}
    row_table = {"bf16": GEN_BF16_EXPECT, "fp32": GEN_FP32_EXPECT}.get(precision, {}).get((row, B), {})
    _check_variants(names, _merge(mode, row_table), f"{row}-B{B} {precision}")


@pytest.mark.gpu
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("row", list(CVAE_ROWS))
def test_cvae_variants_ran(row, precision):
    calls = cvae_stage_calls(row, precision)
    names = {stage: kernels_run_by(calls[stage]) for stage in CVAE_STAGES}
    mode = {s: MODE_EXPECT[precision][s] for s in CVAE_STAGES}
    row_table = CVAE_BF16_EXPECT[row] if precision == "bf16" else {}
    _check_variants(names, _merge(mode, row_table), f"{row} {precision}")
