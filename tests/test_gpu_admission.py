"""Clip admission (CharacterizationSession(admission=True)): a new clip can start in any slot on any frame of a running
session, inside the one captured graph.

- the masked post-process entry point against the init / steady entry points it stands in for, bit for bit;
- the seed copy against torch.where(start, table[idx], dst);
- staggered starts and slot reuse are time-shift invariant: clip c at local frame f equals clip c run from frame 0 of a
  default session of the same batch size, bit for bit (bf16 and fp32), and the CPU oracle (fp32) within DESIGN §2's
  session tolerances (2e-4 on Y, exact match indices, 10x on the pose fields);
- the second decode, sub-batch lanes and the pipelined submit / collect path in admission mode;
- CPU only: the new entry points refuse null / empty arguments before touching a device.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from mocha_sigasia2023_b200 import _lib, kinematics, skeleton, weights, workload

OUT_KEYS = ("pos", "rot", "vel", "ang", "blend_pos", "ik_pos", "ik_rot", "src_root_pos", "src_root_rot", "src_root_vel",
            "src_root_ang")
SS, OS = C.sizeof(_lib.ClipState), C.sizeof(_lib.FrameOut)


# ---------------------------------------------------------------------------------------------------------------------
# kernels
# ---------------------------------------------------------------------------------------------------------------------
def _post_inputs(B, seed):
    inp = workload.step_inputs(B, seed)
    rng = np.random.default_rng(seed + 1)
    Y = (0.5 * rng.standard_normal((B, 60, 24, 15))).astype(np.float32)      # stands in for the de-normalised decoder output
    side = np.concatenate([inp["src_hips_vel"].reshape(B, -1), inp["src_rvel"], inp["src_rang"]], axis=1)
    return (torch.from_numpy(Y).cuda(), torch.from_numpy(np.ascontiguousarray(side)).cuda(),
            torch.from_numpy(inp["contacts"]).cuda())


def _post_unaligned(pp, Y, side, ct, state0, out0, init=0, start=None):
    """One frame on copies of the struct arrays placed 8 bytes off 16-byte alignment: that takes the general kernel."""
    B, T, V, Cin = Y.shape
    st = torch.empty(B * SS + 8, dtype=torch.uint8, device="cuda")
    ot = torch.empty(B * OS + 8, dtype=torch.uint8, device="cuda")
    st[8:].copy_(state0)
    ot[8:].copy_(out0)
    sp, op = C.c_void_p(st.data_ptr() + 8), C.c_void_p(ot.data_ptr() + 8)
    lib = _lib.load()
    if start is None:
        _lib.check(lib.mocha_post_frame_packed(C.byref(pp.params), _lib.ptr(Y), _lib.ptr(side), side.stride(0), _lib.ptr(ct),
                                               B, T, V, Cin, init, sp, op, _lib.stream_ptr()), "mocha_post_frame_packed")
    else:
        _lib.check(lib.mocha_post_frame_packed_masked(C.byref(pp.params), _lib.ptr(Y), _lib.ptr(side), side.stride(0),
                                                      _lib.ptr(ct), _lib.ptr(start), B, T, V, Cin, sp, op,
                                                      _lib.stream_ptr()), "mocha_post_frame_packed_masked")
    return st[8:].view(B, SS).clone(), ot[8:].view(B, OS).clone()


@pytest.mark.gpu
def test_masked_post_matches_init_and_step_entry_points():
    B = 8
    pp = kinematics.PostProcessor(B, "cuda")
    for f in range(4):                                   # a steady state with history in every clip
        pp.step_packed(*_post_inputs(B, 40 + f))
    Y, side, ct = _post_inputs(B, 99)
    state0, out0 = pp.state.clone(), pp.out.clone()

    def run(**kw):
        pp.state.copy_(state0)
        pp.out.copy_(out0)
        pp.step_packed(Y, side, ct, **kw)
        return pp.state.view(B, SS).clone(), pp.out.view(B, OS).clone()

    s_init, o_init = run(init=1)                         # general kernel, frame 0
    s_step, o_step = run(init=0)                         # steady-state kernel
    assert not torch.equal(s_init, s_step)
    # the general kernel's steady step, for the masked launch on unaligned struct arrays
    s_gstep, o_gstep = _post_unaligned(pp, Y, side, ct, state0, out0, init=0)
    for row in ([1, 0, 0, 1, 1, 0, 1, 0], [0] * B, [1] * B):
        start = torch.tensor(row, dtype=torch.uint8, device="cuda")
        m = start.bool()[:, None]
        got_s, got_o = run(start=start)                  # masked step kernel
        assert torch.equal(got_s, torch.where(m, s_init, s_step)), f"state, start row {row}"
        assert torch.equal(got_o, torch.where(m, o_init, o_step)), f"frame outputs, start row {row}"
        got_s, got_o = _post_unaligned(pp, Y, side, ct, state0, out0, start=start)   # general kernel, per-clip flag
        assert torch.equal(got_s, torch.where(m, s_init, s_gstep)), f"state (general kernel), start row {row}"
        assert torch.equal(got_o, torch.where(m, o_init, o_gstep)), f"frame outputs (general kernel), start row {row}"


@pytest.mark.gpu
@pytest.mark.parametrize("idx_stride", [1, 2])
def test_seed_rows_matches_where(idx_stride):
    g = torch.Generator(device="cuda").manual_seed(5)
    N, B, n, D = 37, 16, 90, 256
    table = torch.randn((N, n, D), device="cuda", generator=g)
    dst = torch.randn((B, n, D), device="cuda", generator=g)
    idx = torch.randint(0, N, (B, idx_stride), device="cuda", generator=g, dtype=torch.int64)
    start = (torch.rand((B,), device="cuda", generator=g) < 0.5).to(torch.uint8)
    start[0], start[1] = 1, 0
    want = torch.where(start.bool()[:, None, None], table[idx[:, 0]], dst)
    untouched = dst[~start.bool()].clone()
    _lib.check(_lib.load().mocha_seed_rows(_lib.ptr(start), _lib.ptr(idx), idx_stride, _lib.ptr(table), N, n * D,
                                           _lib.ptr(dst), B, _lib.stream_ptr()), "mocha_seed_rows")
    assert torch.equal(dst, want)
    assert torch.equal(dst[~start.bool()], untouched)


def test_new_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    p = kinematics.make_post_params()
    fake = C.c_void_p(256)                               # never dereferenced: validation comes first
    rc = lib.mocha_post_frame_packed_masked(C.byref(p), fake, fake, 60 * 3 + 6, fake, None, 4, 60, 24, 15, fake, fake, None)
    assert rc == -1 and b"mocha_post_frame_packed_masked" in lib.mocha_last_error()
    rc = lib.mocha_post_frame_packed_masked(C.byref(p), fake, fake, 60 * 3 + 6, fake, fake, 0, 60, 24, 15, fake, fake, None)
    assert rc == -1 and b"mocha_post_frame" in lib.mocha_last_error()
    rc = lib.mocha_post_frame_packed_masked(C.byref(p), fake, fake, 60 * 3, fake, fake, 4, 60, 24, 15, fake, fake, None)
    assert rc == -1 and b"side" in lib.mocha_last_error()
    assert lib.mocha_seed_rows(None, fake, 1, fake, 10, 8, fake, 4, None) == -1
    assert b"mocha_seed_rows" in lib.mocha_last_error()
    assert lib.mocha_seed_rows(fake, fake, 1, fake, 10, 8, fake, 0, None) == -1
    assert lib.mocha_seed_rows(fake, fake, 1, fake, 0, 8, fake, 4, None) == -1
    assert lib.mocha_seed_rows(fake, fake, 1, fake, 10, 6, fake, 4, None) == -1


# ---------------------------------------------------------------------------------------------------------------------
# sessions: a staggered schedule with slot reuse
# ---------------------------------------------------------------------------------------------------------------------
B = 8
FRAMES = 9
FIRST = [0, 0, 1, 3, 3, 4, 6, 6]          # frame on which each slot's first clip starts
SECOND = {0: 4, 3: 6}                     # slot -> frame of a second clip, started while the first is mid-stream


def _clips():
    """(clip id, slot, first frame, frames)"""
    out = [(s, s, f0, SECOND.get(s, FRAMES) - f0) for s, f0 in enumerate(FIRST)]
    out += [(B + k, s, f0, FRAMES - f0) for k, (s, f0) in enumerate(sorted(SECOND.items()))]
    return out


def _clip_input(c, lf):
    return workload.step_inputs(1, seed=10_000 + 100 * c + lf)


def _filler(tag, f, s):
    return workload.step_inputs(1, seed=50_000 + 10_000 * tag + 100 * f + s)    # finite inputs of an idle slot


def _batch(rows):
    return {k: np.concatenate([r[k] for r in rows]) for k in rows[0]}


def _snap(sess, out):
    d = {"Y": sess.Y.cpu().numpy(), "match_idx": sess.match_idx[:, 0].cpu().numpy(), "prev_cha": sess.prev_cha.cpu().numpy(),
         **out}
    if sess.with_cm_path:
        d["cm_Y"] = sess.cm_Y.cpu().numpy()
        d.update({"cm_" + k: v for k, v in sess.cm_post.read().items()})
    return d


def _schedule(f):
    """inputs [B, ...] and start row of admission frame f"""
    rows, start = [], np.zeros(B, dtype=np.uint8)
    for s in range(B):
        act = [(c, f0) for c, cs, f0, n in _clips() if cs == s and f0 <= f < f0 + n]
        if act:
            c, f0 = act[0]
            rows.append(_clip_input(c, f - f0))
            start[s] = f == f0
        else:
            rows.append(_filler(0, f, s))
    return _batch(rows), start


def _args(inp):
    return inp["X"], inp["src_hips_vel"], inp["src_rvel"], inp["src_rang"], inp["contacts"], inp["eps"]


def _run_admission(precision, tc, with_cm_path=False, lanes=1):
    sess, *_ = workload.build_session(B, n_db=48, precision=precision, match_tensor_cores=tc, with_cm_path=with_cm_path,
                                      lanes=lanes, admission=True)
    sess.capture()                                       # before the first frame: no slot has started yet
    frames = []
    for f in range(FRAMES):
        inp, start = _schedule(f)
        out = sess.step_host(*_args(inp), start=start)
        frames.append(_snap(sess, out))
    return sess, frames


def _run_reference(precision, tc, clip_ids, with_cm_path=False):
    """Default session of the same batch size: the listed clips run in their slots from frame 0."""
    sess, *_ = workload.build_session(B, n_db=48, precision=precision, match_tensor_cores=tc, with_cm_path=with_cm_path)
    mine = {s: (c, n) for c, s, f0, n in _clips() if c in clip_ids}
    frames = []
    for lf in range(max(n for _, n in mine.values())):
        rows = [_clip_input(mine[s][0], lf) if s in mine and lf < mine[s][1] else _filler(1, lf, s) for s in range(B)]
        if lf == 1:
            sess.capture()
        out = sess.step_host(*_args(_batch(rows)))
        frames.append(_snap(sess, out))
    return frames


_CACHE = {}


def _admission_frames(precision, tc, **kw):
    key = (precision, tc, tuple(sorted(kw.items())))
    if key not in _CACHE:
        _CACHE[key] = _run_admission(precision, tc, **kw)
    return _CACHE[key]


def _check_time_shift(frames, refs, keys):
    first_ids = set(range(B))
    for c, s, f0, n in _clips():
        ref = refs[0] if c in first_ids else refs[1]
        for lf in range(n):
            got, want = frames[f0 + lf], ref[lf]
            for k in keys:
                np.testing.assert_array_equal(got[k][s], want[k][s], err_msg=f"clip {c} slot {s} local frame {lf}: {k}")


TIME_SHIFT_KEYS = ("Y", "match_idx", "prev_cha") + OUT_KEYS


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tc", [("bf16", True), ("fp32", False)])
def test_staggered_starts_and_slot_reuse_are_time_shift_invariant(precision, tc):
    _, frames = _admission_frames(precision, tc)
    refs = (_run_reference(precision, tc, set(range(B))), _run_reference(precision, tc, {B, B + 1}))
    _check_time_shift(frames, refs, TIME_SHIFT_KEYS)


@pytest.mark.gpu
def test_staggered_starts_against_the_oracle_fp32():
    from mocha_oracle.pipeline import OraclePipeline
    sess, frames = _admission_frames("fp32", False)
    gen_sd, cvae_sd = weights.generator_state_dict(1777), weights.cvae_state_dict(1778)
    np_sd = lambda sd: {k: v.numpy() for k, v in sd.items()}
    stats = workload.stats_as_dict(workload.driver_stats())
    cha, db = sess.cha_encoded.cpu().numpy(), sess.tree.data.cpu().numpy()
    tol = 2e-4
    for c, s, f0, n in _clips():
        ora = OraclePipeline(np_sd(gen_sd), np_sd(cvae_sd), stats, cha, db, 1, skeleton.BONE_PARENTS)
        for lf in range(n):
            want = ora.step(*_args(_clip_input(c, lf)))
            got = frames[f0 + lf]
            where = f"clip {c} slot {s} local frame {lf}"
            assert got["match_idx"][s] == ora.last["match_idx"][0], where
            err = np.abs(got["Y"][s] - ora.last["Y"][0]).max() / np.abs(ora.last["Y"][0]).max()
            assert err < tol, f"{where}: decoder output rel err {err}"
            for k in ("pos", "rot", "vel", "ang", "blend_pos", "ik_pos", "src_root_pos", "src_root_rot"):
                np.testing.assert_allclose(got[k][s], want[k][0], rtol=10 * tol, atol=10 * tol, err_msg=f"{where}: {k}")
            dots = np.abs((got["ik_rot"][s] * want["ik_rot"][0]).sum(-1))
            assert dots.min() > 1 - 100 * tol, f"{where}: ik_rot"


@pytest.mark.gpu
def test_second_decode_of_started_clips_matches_reference():
    _, frames = _run_admission("bf16", False, with_cm_path=True)
    refs = (_run_reference("bf16", False, set(range(B)), with_cm_path=True),
            _run_reference("bf16", False, {B, B + 1}, with_cm_path=True))
    _check_time_shift(frames, refs, TIME_SHIFT_KEYS + ("cm_Y",) + tuple("cm_" + k for k in OUT_KEYS))


@pytest.mark.gpu
def test_admission_lanes_are_bit_identical():
    _, one = _admission_frames("bf16", True)
    _, two = _run_admission("bf16", True, lanes=2)
    for f, (a, b) in enumerate(zip(one, two)):
        for k in TIME_SHIFT_KEYS:
            np.testing.assert_array_equal(a[k], b[k], err_msg=f"frame {f}: {k}")


@pytest.mark.gpu
def test_pipelined_submit_collect_with_start_rows():
    _, want = _admission_frames("bf16", True)
    sess, *_ = workload.build_session(B, n_db=48, precision="bf16", match_tensor_cores=True, admission=True)
    sess.capture()
    pins = []
    for f in range(FRAMES):
        inp, start = _schedule(f)
        pin = sess.pinned_inputs()
        assert set(pin) == {"X", "side", "contacts", "eps", "start"}
        pin["X"].numpy()[...] = inp["X"]
        pin["side"].numpy()[...] = np.concatenate([inp["src_hips_vel"].reshape(B, -1), inp["src_rvel"], inp["src_rang"]], 1)
        pin["contacts"].numpy()[...] = inp["contacts"]
        pin["eps"].numpy()[...] = inp["eps"]
        pin["start"].numpy()[...] = start
        pins.append(pin)
    got, prev = [], None
    for f in range(FRAMES):
        t = sess.submit(pins[f])
        if prev is not None:
            got.append(sess.collect(prev))
        prev = t
    got.append(sess.collect(prev))
    for f in range(FRAMES):
        for k in OUT_KEYS:
            np.testing.assert_array_equal(got[f][k], want[f][k], err_msg=f"frame {f}: {k}")
