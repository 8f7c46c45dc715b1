"""bench.py --dump-outputs: the last timed step's outputs land as float .npy files; the same arguments give the same
outputs (seeded inputs), so two builds can be compared output for output; --steps sets how many steps ran: the dump
equals the last of exactly that many steps of bench.py's sequence, replayed here through the session API."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CLIPS, WARMUP = 4, 3
NAMES = {"pos", "rot", "vel", "ang", "blend_pos", "ik_pos", "ik_rot", "src_root_pos", "src_root_rot", "src_root_vel",
         "src_root_ang", "Y", "match_idx", "match_dist", "clip_index"}


def _bench(tmp_path_factory, steps):
    out = tmp_path_factory.mktemp("dump")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--clips", str(CLIPS), "--steps", str(steps),
                        "--warmup", str(WARMUP), "--no-extras", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       capture_output=True, text=True, timeout=900, cwd=str(out.parent))
    assert r.returncode == 0, f"bench.py failed:\n{r.stdout[-2000:]}\n{r.stderr[-4000:]}"
    line = json.loads(r.stdout.strip().splitlines()[-1])
    return line, {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}


@pytest.fixture(scope="module")
def runs(tmp_path_factory):
    return [_bench(tmp_path_factory, k) for k in (3, 3, 4)]


def test_dump_files(runs):
    line, d = runs[0]
    assert line["steps"] == 3
    assert set(d) == NAMES
    for name, a in d.items():
        assert a.dtype in (np.float32, np.float64), name
        assert a.shape[0] == CLIPS and np.isfinite(a).all(), name
    assert d["Y"].shape == (CLIPS, 60, 24, 15)
    np.testing.assert_array_equal(d["clip_index"], np.arange(CLIPS))
    assert sum(a.nbytes for a in d.values()) < 64e6


def test_same_arguments_same_outputs(runs):
    (_, a), (_, b) = runs[0], runs[1]
    np.testing.assert_array_equal(a["match_idx"], b["match_idx"])
    for name in NAMES:
        np.testing.assert_allclose(a[name], b[name], rtol=1e-5, atol=1e-6, err_msg=name)


def _replay(steps):
    """bench.py's sequence at rank 0: init frame on input set 0, one eager frame on set 1, graph capture, WARMUP frames,
    then the timed frames, frame i on input set i % 4. Returns the outputs after each timed frame listed in `steps`."""
    from mocha_sigasia2023_b200 import workload
    sess, *_ = workload.build_session(CLIPS, n_db=385, precision="bf16", seed=0, match_tensor_cores=None, lanes=1)
    pool = [workload.step_inputs(CLIPS, seed=i) for i in range(4)]

    def frame(i):
        h = pool[i % 4]
        sess.step_host(h["X"], h["src_hips_vel"], h["src_rvel"], h["src_rang"], h["contacts"], h["eps"])

    frame(0)
    frame(1)
    sess.capture()
    for i in range(WARMUP):
        frame(i)
    got = {}
    for i in range(max(steps)):
        frame(i)
        if i + 1 in steps:
            got[i + 1] = dict(sess.post.read(), Y=sess.Y.cpu().numpy())
    return got


def test_steps_sets_the_timed_steps(runs):
    (line3, a), (line4, c) = runs[0], runs[2]
    assert line3["steps"] == 3 and line4["steps"] == 4
    want = _replay((3, 4))
    for k, d in ((3, a), (4, c)):
        for name, v in want[k].items():
            np.testing.assert_allclose(d[name], v, rtol=1e-5, atol=1e-6, err_msg=f"{k} steps: {name}")
    assert not np.allclose(a["Y"], c["Y"])       # so the comparison above tells 3 steps from 4
