"""Folded decoder attention weights (packing.decoder_folded) checked on CPU against the oracle's attention.

When the decoder's head width equals the model width, to_q / to_k fold into one key weight per head (G_h = Wq_h^T Wk_h)
and to_v into the out-projection (Wo_h Wv_h). Evaluated in float64, the folded formula is the reference attention up to
float64 rounding: a wrong head order, layer order or transpose shows up as an O(1) difference."""
import copy

import numpy as np
import pytest
import torch

from mocha_oracle import nets
from mocha_sigasia2023_b200 import packing, weights

CFGS = {
    "default": {},
    "three_layers_two_heads": {"encoder_heads": 2, "decoder_heads": 2, "decoder_depth": 3},   # dh = D = 256
}
UNFOLDED = {
    "dh192": {"encoder_heads": 2, "decoder_heads": 2, "encoder_dim_head": 192, "decoder_dim_head": 64},
    "wide512": {"encoder_dim": 512, "decoder_dim": 512},
}


def _cfg(change):
    cfg = copy.deepcopy(weights.DEFAULT_MODEL_CFG)
    cfg.update(copy.deepcopy(change))
    return cfg


def _in_tokens(x, eps=1e-5):
    """Instance norm over the tokens of each clip and channel (unbiased std, eps added to the std), as the oracle."""
    m = x.mean(axis=1, keepdims=True)
    return (x - m) / (x.std(axis=1, ddof=1, keepdims=True) + eps)


def _folded_attention(kfold, wvo, bo, l, src, sty, H, D):
    """softmax(IN(src) (IN(sty) G_{l,h}^T)^T / sqrt(D)) sty per head h, then [.. | .. per head] Wvo^T + bo."""
    q, k_in = _in_tokens(src), _in_tokens(sty)
    outs = []
    for h in range(H):
        g = kfold[(l * H + h) * D:(l * H + h + 1) * D]                    # G_{l,h}, [D, D]
        s = q @ (k_in @ g.T).transpose(0, 2, 1) * D ** -0.5
        p = np.exp(s - s.max(axis=-1, keepdims=True))
        p /= p.sum(axis=-1, keepdims=True)
        outs.append(p @ sty)
    return np.concatenate(outs, axis=-1) @ wvo.T + bo


@pytest.mark.parametrize("name", list(CFGS))
def test_folded_weights_reproduce_decoder_attention(name, monkeypatch):
    cfg = _cfg(CFGS[name])
    D, H, depth = cfg["decoder_dim"], cfg["decoder_heads"], cfg["decoder_depth"]
    sd_t = weights.generator_state_dict(1777, cfg)
    folded = packing.decoder_folded(sd_t, cfg)
    assert set(folded) == {"dec_kfold"} | {f"dec{l}.wvo" for l in range(depth)}
    kfold = folded["dec_kfold"].numpy()
    assert kfold.shape == (depth * H * D, D) and kfold.dtype == np.float64
    # the oracle evaluated in float64 (it names its working type once, as a module global)
    monkeypatch.setattr(nets, "F32", np.float64)
    sd = {k: v.numpy().astype(np.float64) for k, v in sd_t.items()}
    rng = np.random.default_rng(7)
    n = cfg["nbody"] * (cfg["nframes"] // cfg["temporal_patch_size"])
    src = rng.standard_normal((2, n, D))
    sty = rng.standard_normal((2, n, D))
    for l in range(depth):
        p = f"decoder.layers.{l}.1"
        want = nets.attention(sd, p, src, sty, H, True)
        assert want.dtype == np.float64
        wvo = folded[f"dec{l}.wvo"].numpy()
        assert wvo.shape == (D, H * D)
        got = _folded_attention(kfold, wvo, sd[p + ".to_out.0.bias"], l, src, sty, H, D)
        err = np.abs(got - want).max() / np.abs(want).max()
        assert err <= 1e-10, f"layer {l}: rel err {err:.3e}"


@pytest.mark.parametrize("name", list(UNFOLDED))
def test_no_folded_weights_when_head_width_differs_from_model_width(name):
    cfg = _cfg(UNFOLDED[name])
    assert cfg["decoder_dim_head"] != cfg["decoder_dim"]
    sd = weights.generator_state_dict(1777, cfg)
    assert packing.decoder_folded(sd, cfg) == {}
    assert not any(k == "dec_kfold" or k.endswith(".wvo") for k in packing.generator_tensors(sd, cfg))


def test_generator_tensors_carry_folded_and_unfolded_weights():
    """generator_tensors hands the folded products to the blob next to the unfolded weights (the fp32 / 3xTF32 paths
    keep reading those)."""
    cfg = _cfg({})
    sd = weights.generator_state_dict(1777, cfg)
    t = packing.generator_tensors(sd, cfg)
    folded = packing.decoder_folded(sd, cfg)
    for k, v in folded.items():
        assert torch.equal(t[k], v), k
    for l in range(cfg["decoder_depth"]):
        for f in ("wq", "wk", "wv", "wo"):
            assert f"dec{l}.{f}" in t
