"""Result bank (ResultBank + mocha_record_frames + mocha_clip_payload, CharacterizationSession.serve, characterize_many):

- record semantics: an 8-slot bank + result session driven through staggered starts, overriding starts, slot reuse,
  re-runs of finished clips, bad ids, unused entries and clamping after the last window; every clip's record rows equal
  what step_bank() returned for its windows, bit for bit, and done() equals a host model;
- payload: the copied columns equal features.extract / the records bit for bit, the computed ones match the reference's
  final_payload (oracle) on the same sequences;
- serve(): bit-identical payloads whatever the order (slot, start frame) of the clips, in bf16 / fp32 and with two
  lanes and the second decode; a session captured mid-serve gives the payloads of one captured before the first frame;
- characterize_many against the reference recording (e2e.npz) and against characterize();
- CPU only: argument checks and serving_schedule.
"""
import ctypes as C
import os
import types

import numpy as np
import pytest
import torch

from mocha_sigasia2023_b200 import _lib, features, kinematics as kin, preprocess, skeleton, synthetic, workload
from mocha_sigasia2023_b200.result_bank import RECORD_DTYPE, ResultBank, serving_schedule
from mocha_sigasia2023_b200.session import CharacterizationSession
from mocha_sigasia2023_b200.source_bank import SourceBank

T = 60
PAR = np.asarray(skeleton.BONE_PARENTS)


def _norm():
    n = synthetic.make_norm_stats(7)["norm"]
    return n["X_mean"], n["X_std"]


def _angle_err_deg(a, b):                                # test_gpu_e2e's
    d = np.abs(a - b) % 360.0
    return np.minimum(d, 360.0 - d)


def _frames16():
    f = preprocess.process_frames(synthetic.make_clip(40, seed=77))
    return {k: (v[10:26] if isinstance(v, np.ndarray) and k != "parents" else v) for k, v in f.items()}


def _bank(lengths, extra_clips=2, seed=300, with16=True):
    Xm, Xs = _norm()
    frames = [preprocess.process_frames(synthetic.make_clip(n, seed=seed + n)) for n in lengths]
    frames += [_frames16()] if with16 else []
    bank = SourceBank(sum(f["pos"].shape[0] for f in frames) + 7, len(frames) + extra_clips, Xm, Xs)
    for f in frames:
        bank.add(f)
    return bank, frames


class RecordModel:
    """Host model of mocha_record_frames: per slot (clip, count); rows[c][w] = (slot, frame) that wrote the row."""

    def __init__(self, B, nwins):
        self.slot = [(None, 0)] * B
        self.nwins = nwins
        self.rows = {c: {} for c in range(len(nwins))}
        self.done = [0] * len(nwins)

    def step(self, f, start, clip):
        for b in range(len(self.slot)):
            c, n = self.slot[b]
            if start[b]:
                c = int(clip[b]) if 0 <= int(clip[b]) < len(self.nwins) else None
                n = 0
            if c is not None and n < self.nwins[c]:
                self.rows[c][n] = (b, f)
                n += 1
                self.done[c] = n
            self.slot[b] = (c, n)


LENGTHS = (31, 40, 75, 100, 240)          # clip ids 0..4 (16, 25, 60, 85, 225 windows); id 5: 16 frames, 1 window
EVENTS = {                                # frame -> {slot: clip id}; no clip records in two slots at once
    0: {0: 4, 5: 5},
    1: {1: 0},
    3: {2: 3},
    5: {4: 99, 7: 2},                     # 99: out of range -> idle
    10: {4: -1},
    12: {4: 1},
    30: {2: 0},                           # overrides clip 3; clip 0 runs again (it ended in slot 1)
    40: {7: 99, 1: 1},                    # a bad id overrides clip 2; clip 1 runs again in another slot
    50: {6: 3},
    60: {5: 2, 4: 7},                     # 7: an unused table entry -> idle
    100: {3: 5},
    150: {1: 2},                          # clip 2 again after it completed
}
NSLOT, NFRAMES = 8, 240
_CACHE = {}


def _record_run():
    """The 8-slot bank + result session over EVENTS: (bank, results, session, per-frame step_bank outputs + match,
    model, clip 4's record rows right after its last window, the error read() raised for an incomplete clip)."""
    if "record" in _CACHE:
        return _CACHE["record"]
    bank, frames = _bank(LENGTHS)
    rb = ResultBank(bank)
    sess, *_ = workload.build_session(NSLOT, n_db=48, precision="bf16", match_tensor_cores=False, admission=True,
                                      source_bank=bank, result_bank=rb)
    sess.capture()
    model = RecordModel(NSLOT, bank.clip_nwin)
    outs, snap4, err = [], None, None
    for f in range(NFRAMES):
        start = np.zeros(NSLOT, dtype=np.uint8)
        clip = np.full(NSLOT, 12345, dtype=np.int32)
        for s, c in EVENTS.get(f, {}).items():
            start[s], clip[s] = 1, c
        eps = np.random.default_rng(500 + f).standard_normal((NSLOT, 256)).astype(np.float32)
        o = sess.step_bank(start, clip, eps)
        o["match"] = sess.match_idx[:, 0].cpu().numpy()
        outs.append(o)
        model.step(f, start, clip)
        if f == 224:                                       # clip 4's last window
            snap4 = rb.records_of(4).copy()
        if f == 20:
            try:
                rb.read(1)                                 # clip 1: 9 of 25 windows recorded
            except _lib.MochaError as e:
                err = e
    _CACHE["record"] = (bank, frames, rb, sess, outs, model, snap4, err)
    return _CACHE["record"]


@pytest.mark.gpu
def test_record_rows_equal_step_outputs_bit_for_bit():
    bank, frames, rb, sess, outs, model, snap4, err = _record_run()
    assert list(rb.done()) == model.done
    assert model.done == bank.clip_nwin                   # every clip completed at least once
    for c in range(bank.n_clips):
        rec = rb.records_of(c)
        assert sorted(model.rows[c]) == list(range(bank.clip_nwin[c]))
        for w, (b, f) in model.rows[c].items():
            where = f"clip {c} window {w} (slot {b}, frame {f})"
            for k in ("ik_pos", "ik_rot", "src_root_pos", "src_root_rot"):
                np.testing.assert_array_equal(rec[k][w], outs[f][k][b], err_msg=where + ": " + k)
            assert rec["match"][w] == outs[f]["match"][b], where
    # frames served after clip 4's last window (it repeats that window until frame 239) leave its rows alone
    np.testing.assert_array_equal(rb.records_of(4).view(np.uint8), snap4.view(np.uint8))
    assert model.slot[0] == (4, bank.clip_nwin[4])
    assert err is not None and "not complete" in str(err)
    assert sess.slot_count.tolist() == [n for _, n in model.slot]


def _oracle_payload(rot_seq, pos_seq):
    from mocha_oracle import clip as oclip
    return oclip.final_payload(rot_seq, pos_seq, PAR)


@pytest.mark.gpu
def test_payload_columns_and_reference_final_payload():
    bank, frames, rb, sess, outs, model, _, _ = _record_run()
    ids = list(range(bank.n_clips))
    with pytest.raises(_lib.MochaError, match="not built"):
        rb.read(0)                                        # complete, but payload() has not run
    rb.payload(ids)
    Xm, Xs = _norm()
    wins = [preprocess.frame_windows(f) for f in frames]
    cat = {k: np.concatenate([w[k] for w in wins]) for k in ("pos", "vel", "rot", "ang", "contacts")}
    cat["parents"] = wins[0]["parents"]
    assert cat["pos"].shape[0] * T >= 4096                # features.extract takes the fk_rows path
    ref = features.extract(cat, Xm, Xs)
    Ypos, Yrot = ref["Ypos"][:, -1].contiguous(), ref["Yrot"][:, -1].contiguous()
    deg32 = np.float32(180.0 / np.pi)
    eul = (kin.quat_op("to_euler_xyz", Yrot.reshape(-1, 4)).reshape(Yrot.shape[0], 25, 3).cpu().numpy() * deg32)
    Ypos, Yrot = Ypos.cpu().numpy(), Yrot.cpu().numpy()
    off = np.concatenate([[0], np.cumsum(bank.clip_nwin)[:-1]])
    for c in ids:
        p = rb.read(c)
        rec = rb.records_of(c)
        n = bank.clip_nwin[c]
        sl = slice(off[c], off[c] + n)
        assert p["src_positions"].dtype == np.float32 and p["ours_positions"].dtype == np.float64
        assert p["src_rotations"].shape == p["ours_positions"].shape == (n, 24, 3)
        # copies: exact
        np.testing.assert_array_equal(p["src_positions"][:, 1:], Ypos[sl, 2:], err_msg=f"clip {c}")
        np.testing.assert_array_equal(p["src_rotations"][:, 1:], eul[sl, 2:], err_msg=f"clip {c}")
        np.testing.assert_array_equal(p["ours_positions"][:, 1:], rec["ik_pos"][:, 2:], err_msg=f"clip {c}")
        np.testing.assert_array_equal(p["match"], rec["match"])
        # computed columns against the reference's final step on the same sequences
        o_rot, o_pos = _oracle_payload(rec["ik_rot"], rec["ik_pos"])
        np.testing.assert_allclose(p["ours_positions"], o_pos, rtol=1e-12, atol=1e-12)
        assert _angle_err_deg(p["ours_rotations"], o_rot).max() < 1e-9
        sp, sr = Ypos[sl].copy(), Yrot[sl].copy()
        sp[:, 0] = rec["src_root_pos"].astype(np.float32)
        sr[:, 0] = rec["src_root_rot"].astype(np.float32)
        s_rot, s_pos = _oracle_payload(sr, sp)
        np.testing.assert_allclose(p["src_positions"], s_pos, rtol=1e-6, atol=1e-6)
        e = _angle_err_deg(p["src_rotations"].astype(np.float64), s_rot.astype(np.float64))
        assert e.max() < 0.05 and np.median(e) < 1e-4, (c, e.max(), np.median(e))
    # serving a clip again makes its payload stale until payload() runs again
    start, clip = np.zeros(NSLOT, dtype=np.uint8), np.zeros(NSLOT, dtype=np.int32)
    start[6], clip[6] = 1, 5                              # the 1-window clip: complete again after this frame
    sess.step_bank(start, clip, np.zeros((NSLOT, 256), dtype=np.float32))
    with pytest.raises(_lib.MochaError, match="not built"):
        rb.read(5)
    rb.read(4)                                            # untouched clips stay readable
    rb.payload([5])
    assert rb.read(5)["match"].shape == (1,)


# ---------------------------------------------------------------------------------------------------------------------
# serve()
# ---------------------------------------------------------------------------------------------------------------------
SERVE_LENGTHS = (31, 40, 52, 36, 45, 70)                 # 16, 25, 37, 21, 30, 55 windows


def _serve_bank():
    if "serve" not in _CACHE:
        bank, _ = _bank(SERVE_LENGTHS, seed=700, with16=False)
        rng = np.random.default_rng(42)
        eps = {c: rng.standard_normal((bank.clip_nwin[c] - 1, 256)).astype(np.float32) for c in range(bank.n_clips)}
        _CACHE["serve"] = bank, eps
    return _CACHE["serve"]


def _assert_same_payloads(a, b, ids):
    for c in ids:
        for k in a[c]:
            np.testing.assert_array_equal(a[c][k], b[c][k], err_msg=f"clip {c}: {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("precision,kw", [("bf16", {}), ("fp32", {}), ("bf16", {"lanes": 2, "with_cm_path": True})])
def test_serve_payloads_do_not_depend_on_the_schedule(precision, kw):
    bank, eps = _serve_bank()
    rb = ResultBank(bank)
    sess, *_ = workload.build_session(4, n_db=48, precision=precision, match_tensor_cores=False, admission=True,
                                      source_bank=bank, result_bank=rb, **kw)
    sess.capture()
    first = sess.serve([0, 1, 2, 3, 4, 5], eps=eps)
    second = sess.serve([5, 3, 1, 0, 4, 2], eps=eps)
    _, _, p1 = serving_schedule([bank.clip_nwin[c] for c in (0, 1, 2, 3, 4, 5)], 4)
    _, _, p2 = serving_schedule([bank.clip_nwin[c] for c in (5, 3, 1, 0, 4, 2)], 4)
    assert p1[2].tolist() != p2[5].tolist()              # clip 2 runs in another slot or from another frame
    _assert_same_payloads(first, second, range(6))
    for c in range(6):
        assert first[c]["ours_positions"].shape == (bank.clip_nwin[c], 24, 3)
        assert np.isfinite(first[c]["ours_rotations"]).all() and np.abs(first[c]["ours_positions"]).max() > 0
        assert (rb.done()[c] == bank.clip_nwin[c])
    with pytest.raises(_lib.MochaError, match="duplicate"):
        sess.serve([1, 2, 1])


@pytest.mark.gpu
def test_capture_mid_serve_and_serve_give_the_same_payloads():
    bank, eps = _serve_bank()
    ids = [2, 0, 5, 1, 4, 3]
    start_rows, clip_rows, place = serving_schedule([bank.clip_nwin[c] for c in ids], 3)
    ids_np = np.asarray(ids, dtype=np.int32)

    def run(capture_at):
        rb = ResultBank(bank)
        sess, *_ = workload.build_session(3, n_db=48, precision="bf16", match_tensor_cores=False, admission=True,
                                          source_bank=bank, result_bank=rb)
        slot_k, slot_f = [-1] * 3, [0] * 3
        for f in range(len(start_rows)):
            if f == capture_at:
                sess.capture()
            e = np.zeros((3, 256), dtype=np.float32)
            for b in range(3):
                if start_rows[f][b]:
                    slot_k[b], slot_f[b] = int(clip_rows[f][b]), f
                k = slot_k[b]
                if k >= 0 and 1 <= f - slot_f[b] < bank.clip_nwin[ids[k]]:
                    e[b] = eps[ids[k]][f - slot_f[b] - 1]
            sess.step_bank(start_rows[f], ids_np[clip_rows[f]], e)
        rb.payload(ids)
        return {c: rb.read(c) for c in ids}

    want = run(0)
    _assert_same_payloads(want, run(9), ids)
    # serve() on the same schedule and eps tables: the same payloads as the frame-by-frame step_bank route
    rb = ResultBank(bank)
    sess, *_ = workload.build_session(3, n_db=48, precision="bf16", match_tensor_cores=False, admission=True,
                                      source_bank=bank, result_bank=rb)
    sess.capture()
    _assert_same_payloads(want, sess.serve(ids, eps=eps), ids)
    assert all(np.abs(want[c]["ours_positions"]).max() > 0 for c in ids)


# ---------------------------------------------------------------------------------------------------------------------
# characterize_many against the reference recording and characterize()
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_characterize_many_matches_the_reference_recording(golden_dir):
    from mocha_sigasia2023_b200.characterize import characterize, characterize_many
    g = np.load(os.path.join(golden_dir, "e2e.npz"))
    src, cha, stats = synthetic.make_clip(240, 0), synthetic.make_clip(400, 1), synthetic.make_norm_stats()
    outs = characterize_many([synthetic.make_clip(50, seed=5), src, synthetic.make_clip(40, seed=6)], cha, stats,
                             slots=1, eps_seqs={1: g["eps"]}, precision="fp32")
    assert [o["match"].shape[0] for o in outs] == [35, 225, 25]
    out = outs[1]                                         # starts in the reused slot on frame 35
    for k in ("src_rotations", "src_positions", "ours_rotations", "ours_positions"):
        assert out[k].shape == g[k].shape and out[k].dtype == g[k].dtype, k
    np.testing.assert_array_equal(out["match"], g["match"])
    np.testing.assert_allclose(out["src_positions"], g["src_positions"], rtol=1e-4, atol=1e-4)
    assert _angle_err_deg(out["src_rotations"], g["src_rotations"]).max() < 0.05
    np.testing.assert_allclose(out["ours_positions"], g["ours_positions"], rtol=2e-3, atol=2e-3)
    err = _angle_err_deg(out["ours_rotations"], g["ours_rotations"])
    assert np.median(err) < 0.01 and (err < 0.5).mean() > 0.995
    # the batch-1 fp32 session of characterize(): equal except for its fp32 FK of the hips and its fp64 Euler of the
    # fp32 source pose
    one = characterize(src, cha, stats, eps_seq=g["eps"], precision="fp32")
    np.testing.assert_array_equal(out["match"], one["match"])
    np.testing.assert_array_equal(out["src_positions"][:, 1:], one["src_positions"][:, 1:].astype(np.float32))
    np.testing.assert_array_equal(out["ours_positions"][:, 1:], one["ours_positions"][:, 1:])
    np.testing.assert_allclose(out["ours_positions"][:, 0], one["ours_positions"][:, 0], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(out["src_positions"][:, 0], one["src_positions"][:, 0], rtol=1e-5, atol=1e-5)
    assert _angle_err_deg(out["ours_rotations"], one["ours_rotations"]).max() < 1e-3
    assert _angle_err_deg(out["src_rotations"].astype(np.float64), one["src_rotations"]).max() < 1e-3


# ---------------------------------------------------------------------------------------------------------------------
# CPU only
# ---------------------------------------------------------------------------------------------------------------------
def test_result_bank_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    fake = C.c_void_p(256)                               # never dereferenced: validation comes first

    def record(**kw):
        a = dict(out=fake, match=fake, ms=1, start=fake, sc=fake, cnt=fake, B=4, first=fake, frames=fake, nc=4, T=60,
                 rec=fake, nr=100, done=fake, built=fake)
        a.update(kw)
        return lib.mocha_record_frames(*a.values(), None)

    for kw, msg in (({"out": None}, b"null slot"), ({"cnt": None}, b"null slot"), ({"match": None}, b"null slot"),
                    ({"rec": None}, b"null bank"), ({"done": None}, b"null bank"), ({"first": None}, b"null bank"),
                    ({"built": None}, b"null bank"), ({"B": 0}, b"bad sizes"), ({"nc": 0}, b"bad sizes"), ({"nr": 0}, b"bad sizes"),
                    ({"ms": 0}, b"bad sizes"), ({"T": 4}, b"bad sizes")):
        assert record(**kw) == -1, kw
        err = lib.mocha_last_error()
        assert b"mocha_record_frames" in err and msg in err, (kw, err)

    def payload(**kw):
        a = dict(rec=fake, nf=100, rot=fake, pos=fake, first=fake, frames=fake, nc=4, done=fake, built=fake, par=fake,
                 T=60, J=25, ids=fake, n=2, mx=10, sr=fake, sp=fake, orr=fake, op=fake, m=fake)
        a.update(kw)
        return lib.mocha_clip_payload(*a.values(), None)

    for kw, msg in (({"rec": None}, b"null bank"), ({"par": None}, b"null bank"), ({"done": None}, b"null bank"),
                    ({"built": None}, b"null bank"),
                    ({"ids": None}, b"null output"), ({"op": None}, b"null output"), ({"m": None}, b"null output"),
                    ({"n": 0}, b"bad sizes"), ({"n": 65536}, b"bad sizes"), ({"mx": 0}, b"bad sizes"),
                    ({"nf": 0}, b"bad sizes"), ({"J": 24}, b"J=25"), ({"T": 4}, b"J=25")):
        assert payload(**kw) == -1, kw
        err = lib.mocha_last_error()
        assert b"mocha_clip_payload" in err and msg in err, (kw, err)


def test_result_bank_and_session_argument_checks():
    Xm, Xs = _norm()
    bank = SourceBank(200, 3, Xm, Xs, device="cpu")      # CPU tensors: the checks need no device
    other = SourceBank(200, 3, Xm, Xs, device="cpu")
    with pytest.raises(_lib.MochaError, match="needs a SourceBank"):
        ResultBank(None)
    rb = ResultBank(bank)
    assert rb.nbytes() == 200 * (1464 + 2 * 288 + 2 * 576 + 8) + 2 * 3 * 4
    assert RECORD_DTYPE.itemsize == 1464
    with pytest.raises(_lib.MochaError, match="not in the bank"):
        rb.read(0)
    assert bank.add(synthetic.make_clip(100, seed=1)) == (0, 85)
    with pytest.raises(_lib.MochaError, match="not in the bank"):
        rb.payload([0, 1])
    with pytest.raises(_lib.MochaError, match="no clip ids"):
        rb.payload([])
    with pytest.raises(_lib.MochaError, match="not complete"):
        rb.read(0)
    assert rb.done().tolist() == [0]
    # the session refuses a result bank without a source bank, or of another bank, before it touches a device
    with pytest.raises(_lib.MochaError, match="result_bank needs"):
        CharacterizationSession(None, None, None, None, None, None, 4, admission=True, result_bank=rb)
    with pytest.raises(_lib.MochaError, match="another source bank"):
        CharacterizationSession(None, None, None, None, None, None, 4, admission=True, source_bank=other,
                                result_bank=rb)
    # serve(): one clip cannot run in two slots at once; a session without a result bank cannot serve
    with pytest.raises(_lib.MochaError, match="duplicate"):
        CharacterizationSession.serve(types.SimpleNamespace(results=rb), [0, 0])
    with pytest.raises(_lib.MochaError, match="result_bank"):
        CharacterizationSession.serve(types.SimpleNamespace(results=None), [0])


def _schedule_before(nwins, B):
    """tools/source_bank_bench.py's serving rows as that benchmark built them inline."""
    queue, slot_left, start_rows, clip_rows = list(range(len(nwins))), np.zeros(B, dtype=np.int64), [], []
    busy = 0
    while queue or slot_left.any():
        row, crow = np.zeros(B, dtype=np.uint8), np.zeros(B, dtype=np.int32)
        for s in range(B):
            if slot_left[s] == 0 and queue:
                c = queue.pop(0)
                slot_left[s], row[s], crow[s] = nwins[c], 1, c
        busy += int((slot_left > 0).sum())
        start_rows.append(row)
        clip_rows.append(crow)
        slot_left = np.maximum(slot_left - 1, 0)
    assert busy == int(np.sum(nwins))
    return np.stack(start_rows), np.stack(clip_rows)


@pytest.mark.parametrize("n,B,lo,hi", [(1024, 128, 30, 225), (40, 8, 1, 20), (7, 16, 1, 5), (1, 1, 3, 3), (50, 3, 1, 1)])
def test_serving_schedule(n, B, lo, hi):
    nwins = np.random.default_rng(n + B).integers(lo, hi + 1, size=n)
    start, clip, place = serving_schedule(nwins, B)
    ref_start, ref_clip = _schedule_before(nwins, B)
    np.testing.assert_array_equal(start, ref_start)
    np.testing.assert_array_equal(clip, ref_clip)
    assert start.dtype == np.uint8 and clip.dtype == np.int32
    owner = np.full(start.shape, -1)                     # clip running in each (frame, slot)
    for k, (s, f0) in enumerate(place):
        assert start[f0, s] == 1 and clip[f0, s] == k
        assert (owner[f0:f0 + nwins[k], s] == -1).all(), "slot double-booked"
        owner[f0:f0 + nwins[k], s] = k                   # nwin consecutive frames in one slot
        assert f0 + nwins[k] <= start.shape[0]
    assert (owner >= 0).sum() == nwins.sum() and int(start.sum()) == n
    assert (np.diff(place[:, 1]) >= 0).all()             # FIFO: clips start in queue order
    assert place[0][1] == 0
    for k in range(1, n):                                # ... on the first frame a slot is free: none idles before
        for f in range(place[k - 1][1], place[k][1]):
            assert (owner[f] >= 0).all(), (k, f)
    with pytest.raises(_lib.MochaError):
        serving_schedule([3, 0], 2)
