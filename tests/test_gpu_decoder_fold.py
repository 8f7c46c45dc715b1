"""bf16 decoder on the folded attention (to_q / to_k folded into one key projection, to_v into to_out; dh == D).

The decoder stage must match the NumPy oracle within the suite's bf16 bound, and launch what the folded path promises:
one tcgen05 GEMM (the key projection of every layer and head) ahead of the layers, then per layer the AdaIN
normalisation pass straight into the fused attention kernel, with no q / k / v projection in between."""
import copy
import functools
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from mocha_oracle import nets
from mocha_sigasia2023_b200 import weights

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

RTOL_BF16 = 2e-2    # the suite's bf16 bound
ROWS = {
    "default": {},
    # hidden width 1024: the block tails run unfused (out-projection, FFN GEMMs); one decoder layer
    "mlp1024": {"encoder_mlp_dim": 1024, "decoder_mlp_dim": 1024, "encoder_depth": 3, "decoder_depth": 1},
}
GEMM = "tc_gemm"           # tc_gemm_kernel / tc_gemm2_kernel: every tcgen05 GEMM launch
ATTN = "attn_kernel"
TAIL = "tail_kernel"
NORM = "instance_norm_tokens_v4_kernel"


def _cfg(row):
    cfg = copy.deepcopy(weights.DEFAULT_MODEL_CFG)
    cfg.update(copy.deepcopy(ROWS[row]))
    return cfg


@functools.lru_cache(maxsize=None)
def _model(row):
    from mocha_sigasia2023_b200.model import Generator
    cfg = _cfg(row)
    g = Generator(cfg, precision="bf16")
    g.load_state_dict(weights.generator_state_dict(1777, cfg), strict=True)
    return g.to("cuda").eval()


@functools.lru_cache(maxsize=None)
def _oracle(row, B):
    """Encoded tokens of B seeded clips (the decoder's input), the style (clips reversed) and the decoder output."""
    cfg = _cfg(row)
    sd = {k: v.numpy() for k, v in weights.generator_state_dict(1777, cfg).items()}
    rng = np.random.default_rng(4000 + B)
    X = rng.standard_normal((B, cfg["nframes"], cfg["njoints"], cfg["mot_in_dim"])).astype(np.float32)
    n = cfg["nbody"] * (cfg["nframes"] // cfg["temporal_patch_size"])
    tokens = nets.mot_embedding(sd, X, cfg["temporal_patch_size"])
    enc = nets.encoder(sd, (tokens + sd["pos_emb"][:, :n]).astype(np.float32), cfg["encoder_depth"], cfg["encoder_heads"])
    sty = np.ascontiguousarray(enc[::-1])
    return enc, sty, nets.decoder(sd, enc, sty, cfg["decoder_depth"], cfg["decoder_heads"])


def _call(row, B):
    enc, sty, _ = _oracle(row, B)
    g, enc, sty = _model(row), torch.from_numpy(enc).cuda(), torch.from_numpy(sty).cuda()
    return lambda: g.decoder(enc, sty)


def _launch_names(row):
    """Kernel names of one decoder call at B = 3 in launch order (torch.profiler, CUDA activities)."""
    from torch.profiler import ProfilerActivity, profile
    fn = _call(row, 3)
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "emcpy" not in e.name
          and "emset" not in e.name]
    return [e.name for e in sorted(ev, key=lambda e: e.time_range.start)]


def _launches(row):
    """_launch_names in a process of its own: the profiler session then shares no CUPTI state with the sessions that
    other test files open in the pytest process."""
    code = ("import json, sys; sys.path[:0] = [{root!r}, {oracle!r}, {tests!r}]; import test_gpu_decoder_fold as t; "
            "print(json.dumps(t._launch_names({row!r})))").format(root=ROOT, oracle=os.path.join(ROOT, "oracle"),
                                                                 tests=os.path.join(ROOT, "tests"), row=row)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("row,B", [("default", 3), ("default", 128), ("mlp1024", 3)])
def test_folded_decoder_matches_oracle(row, B):
    want = _oracle(row, B)[2]
    got = _call(row, B)().cpu().numpy()
    assert got.shape == want.shape and np.isfinite(got).all()
    err = float(np.abs(got.astype(np.float64) - want).max() / np.abs(want).max())
    print(f"{row} B={B}: bf16 decoder rel err {err:.3e}")
    assert err < RTOL_BF16


@pytest.mark.parametrize("row", list(ROWS))
def test_folded_decoder_launches(row):
    depth = _cfg(row)["decoder_depth"]
    names = _launches(row)
    attn = [i for i, n in enumerate(names) if ATTN in n]
    assert len(attn) == depth, names
    # one key projection for every layer and head, ahead of the first attention ...
    assert sum(GEMM in n for n in names[:attn[0]]) == 1, names
    # ... and nothing but the AdaIN normalisation pass between a layer's residual stream and its attention
    assert all(NORM in names[i - 1] for i in attn), names
    if row == "default":
        assert sum(GEMM in n for n in names) == 1, names
        assert sum(TAIL in n for n in names) == depth, names
