"""End-to-end parity: this package's CUDA path vs the UNMODIFIED reference `test_fullframework.main()`
(golden recorded by oracle/ref_harness.py) on the same synthetic clips, weights, normalisation tables
and the same reparameterisation noise (the reference's torch.randn_like draws are replayed)."""
import os

import numpy as np
import pytest

from mocha_sigasia2023_b200 import synthetic
from mocha_sigasia2023_b200.characterize import characterize

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def run(golden_dir):
    g = np.load(os.path.join(golden_dir, "e2e.npz"))
    out = characterize(synthetic.make_clip(240, 0), synthetic.make_clip(400, 1), synthetic.make_norm_stats(),
                       eps_seq=g["eps"], precision="fp32")
    return g, out


def _angle_err_deg(a, b):
    d = np.abs(a - b) % 360.0
    return np.minimum(d, 360.0 - d)


def test_shapes_and_db(run):
    g, out = run
    assert out["n_db"] == int(g["db_shape"][0]) and int(g["db_shape"][1]) == 23040
    for k in ("src_rotations", "src_positions", "ours_rotations", "ours_positions"):
        assert out[k].shape == g[k].shape == (225, 24, 3)


def test_matched_indices_bit_exact(run):
    g, out = run
    np.testing.assert_array_equal(out["match"], g["match"])


def test_source_payload(run):
    g, out = run
    np.testing.assert_allclose(out["src_positions"], g["src_positions"], rtol=1e-4, atol=1e-4)
    assert _angle_err_deg(out["src_rotations"], g["src_rotations"]).max() < 0.05


def test_network_outputs_frame_by_frame(run):
    g, out = run
    ref = g["Ytil_last_rows"][0::2]          # the 'trans' decode of each frame (even entries)
    got = out["Ytil_last_rows"]
    rel = np.abs(got - ref).reshape(len(ref), -1).max(axis=1) / np.abs(ref).max()
    assert rel[0] < 1e-4 and rel[1] < 1e-4, rel[:4]
    # autoregressive CVAE feedback over 224 frames: errors may grow but must stay small
    assert rel.max() < 2e-3, (rel.argmax(), rel.max())


def test_characterised_payload(run):
    g, out = run
    np.testing.assert_allclose(out["ours_positions"], g["ours_positions"], rtol=2e-3, atol=2e-3)
    err = _angle_err_deg(out["ours_rotations"], g["ours_rotations"])
    assert np.median(err) < 0.01
    assert (err < 0.5).mean() > 0.995      # Euler angles are ill-conditioned near gimbal lock


# ---------------------------------------------------------------------------------------------------
# the reference loop's second decode of every frame (the matched DB row's, 'cm_trans') and its first CVAE call
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def run_cm(golden_dir):
    g = np.load(os.path.join(golden_dir, "e2e.npz"))
    out = characterize(synthetic.make_clip(240, 0), synthetic.make_clip(400, 1), synthetic.make_norm_stats(),
                       eps_seq=g["eps"], precision="fp32", with_cm_path=True)
    return g, out


def test_first_cvae_call(run_cm):
    g, out = run_cm
    np.testing.assert_allclose(out["cvae_cond0"], g["cvae_cond0"], rtol=1e-4, atol=1e-4)
    err = np.abs(out["cvae_out0"] - g["cvae_out0"]).max() / np.abs(g["cvae_out0"]).max()
    assert err < 1e-4, err


def test_network_outputs_both_decodes(run_cm):
    g, out = run_cm
    ref = g["Ytil_last_rows"]                   # per frame: the 'trans' decode, then the 'cm_trans' decode
    got = np.stack([out["Ytil_last_rows"], out["Ytil_cm_rows"]], axis=1).reshape(ref.shape)
    rel = np.abs(got - ref).reshape(len(ref), -1).max(axis=1) / np.abs(ref).max()
    assert rel[:4].max() < 1e-4, rel[:4]
    assert rel.max() < 2e-3, (rel.argmax(), rel.max())         # 224 autoregressive CVAE steps


# ---------------------------------------------------------------------------------------------------
# the same 225-frame clip in the throughput mode (bf16 operands on tcgen05): 224 autoregressive CVAE steps
# ---------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def run_bf16(golden_dir):
    g = np.load(os.path.join(golden_dir, "e2e.npz"))
    out = characterize(synthetic.make_clip(240, 0), synthetic.make_clip(400, 1), synthetic.make_norm_stats(),
                       eps_seq=g["eps"], precision="bf16")
    return g, out


def test_bf16_network_outputs_drift_bound(run_bf16):
    """bf16 mode over the whole clip. Stated drift bound: every frame's network output stays within 2e-2 of the
    tensor's range of the fp32 reference (the same bound a single bf16 frame gets): the CVAE feedback loop does
    not amplify the rounding error."""
    g, out = run_bf16
    ref = g["Ytil_last_rows"][0::2]
    got = out["Ytil_last_rows"]
    rel = np.abs(got - ref).reshape(len(ref), -1).max(axis=1) / np.abs(ref).max()
    print(f"[e2e bf16] network output error / range: first {rel[0]:.3e}, median {np.median(rel):.3e}, max {rel.max():.3e} "
          f"at frame {rel.argmax()}")
    assert rel[0] < 2e-2 and rel.max() < 2e-2, (rel.argmax(), rel.max())


def test_bf16_matched_indices(run_bf16):
    """Matched DB index per frame in bf16 mode vs the reference's. The query is the bf16 encoder's context feature,
    so equality is not guaranteed where the top-1 / top-2 margin is within the feature's own error (the matcher itself
    is exact for the query it is given: tests/test_gpu_bench_config.py). Measured on B200: 92 % of the 225 frames agree
    (the synthetic character clip is periodic, so a disagreement picks the same pose one period away and the
    characterised pose stays within 2e-4 of the reference: next test). Required: at least 85 %."""
    g, out = run_bf16
    agree = (out["match"] == g["match"])
    off = np.abs(out["match"] - g["match"])
    print(f"[e2e bf16] matched-index agreement {agree.mean():.4f}; max |index difference| {off.max()}")
    assert agree.mean() >= 0.85


def test_bf16_characterised_payload(run_bf16):
    g, out = run_bf16
    dpos = np.abs(out["ours_positions"] - g["ours_positions"])
    err = _angle_err_deg(out["ours_rotations"], g["ours_rotations"])
    print(f"[e2e bf16] position error max {dpos.max():.4f} (range {np.abs(g['ours_positions']).max():.2f}), "
          f"angle error median {np.median(err):.4f} deg, p99 {np.percentile(err, 99):.3f} deg")
    assert dpos.max() < 2e-2 * np.abs(g["ours_positions"]).max()
    assert np.median(err) < 0.5 and np.percentile(err, 99) < 5.0
