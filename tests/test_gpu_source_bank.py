"""Source clip bank (SourceBank + mocha_source_windows): every slot's X, side and contacts built on the device.

- the kernel against features.extract on all clips' windows (the fk_rows path: > 4096 skeletons), bit for bit, through a
  schedule that visits every window of every clip with staggered starts, slot reuse, overriding starts, cursor clamping
  after the last window, never-started slots and bad ids;
- a bank session against an admission session fed with the same features.extract rows, bit for bit (bf16 and fp32),
  also with two lanes, the second decode and the pipelined submit / collect path;
- CPU only: argument checks of the entry point, the bank and the session, and process_frames + frame_windows against
  process_clip.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from mocha_sigasia2023_b200 import _lib, features, preprocess, synthetic, workload
from mocha_sigasia2023_b200.session import CharacterizationSession
from mocha_sigasia2023_b200.source_bank import SourceBank

OUT_KEYS = ("pos", "rot", "vel", "ang", "blend_pos", "ik_pos", "ik_rot", "src_root_pos", "src_root_rot", "src_root_vel",
            "src_root_ang")
T = 60


def _norm():
    n = synthetic.make_norm_stats(7)["norm"]
    return n["X_mean"], n["X_std"]


def _frames16():
    """A 16-frame clip given as per-frame arrays: its one window is padded on both sides."""
    f = preprocess.process_frames(synthetic.make_clip(40, seed=77))
    return {k: (v[10:26] if isinstance(v, np.ndarray) and k != "parents" else v) for k, v in f.items()}


def _bank_and_reference(lengths, capacity_clips=None):
    """Bank of synthetic clips (plus the 16-frame one) and features.extract over all their windows concatenated.
    Returns (bank, ref rows X [W,...], side [W, T*3+6], contacts [W,2], offsets, nwins)."""
    Xm, Xs = _norm()
    frames = [preprocess.process_frames(synthetic.make_clip(n, seed=300 + n)) for n in lengths] + [_frames16()]
    total = sum(f["pos"].shape[0] for f in frames)
    bank = SourceBank(total + 7, capacity_clips or len(frames) + 2, Xm, Xs)
    wins, nwins = [], []
    for f in frames:
        cid, nwin = bank.add(f)
        assert cid == len(nwins)
        nwins.append(nwin)
        wins.append(preprocess.frame_windows(f))
    cat = {k: np.concatenate([w[k] for w in wins]) for k in ("pos", "vel", "rot", "ang", "contacts")}
    cat["parents"] = wins[0]["parents"]
    assert cat["pos"].shape[0] * T >= 4096                # features.extract takes the fk_rows path
    ref = features.extract(cat, Xm, Xs)
    side = torch.cat([ref["Yvel"][:, :, 1].reshape(-1, T * 3), ref["Yrvel"][:, -1], ref["Yrang"][:, -1]], 1)
    offsets = np.concatenate([[0], np.cumsum(nwins)[:-1]])
    return bank, ref["X"], side.contiguous(), ref["contacts"][:, -1].contiguous(), offsets, nwins


class SlotModel:
    """Host model of the per-slot state: (clip, cursor); clip None = idle."""

    def __init__(self, B, nwins):
        self.state = [None] * B
        self.nwins = nwins

    def step(self, start, clip):
        served = []
        for b in range(len(self.state)):
            if start[b]:
                c = int(clip[b])
                self.state[b] = (c, 0) if 0 <= c < len(self.nwins) else None
            if self.state[b] is None:
                served.append(None)
                continue
            c, cur = self.state[b]
            w = min(cur, self.nwins[c] - 1)
            self.state[b] = (c, w + 1)
            served.append((c, w))
        return served


LENGTHS = (31, 40, 75, 100, 240)       # clip ids 0..4; id 5 is the 16-frame clip
EVENTS = {                             # frame -> {slot: clip id}
    0: {0: 4, 5: 5},
    1: {1: 0},
    3: {2: 3},
    5: {4: 99, 7: 2},                  # 99: out of range -> idle
    7: {5: 2},
    10: {4: -1},
    12: {4: 1},
    20: {1: 1},
    30: {2: 2},                        # overrides the running clip 3
    40: {7: 99},                       # a running slot started with a bad id turns idle
    45: {1: 5},
    50: {6: 3},
    60: {5: 0, 4: 7},                  # 7: an unused table entry -> idle
    100: {2: 3},
    150: {1: 2},
}
NSLOT, NFRAMES = 8, 240


@pytest.mark.gpu
def test_source_windows_match_features_extract_bit_for_bit():
    bank, rX, rside, rct, offsets, nwins = _bank_and_reference(LENGTHS)
    B = NSLOT
    dev = "cuda"
    slot_clip = torch.full((B,), -1, dtype=torch.int32, device=dev)
    slot_cursor = torch.zeros((B,), dtype=torch.int32, device=dev)
    X = torch.full((B, T, 24, 15), float("nan"), device=dev)
    side = torch.full((B, T * 3 + 6), float("nan"), device=dev)
    ct = torch.full((B, 2), 7, dtype=torch.uint8, device=dev)
    model = SlotModel(B, nwins)
    seen = set()
    for f in range(NFRAMES):
        start = np.zeros(B, dtype=np.uint8)
        clip = np.full(B, 12345, dtype=np.int32)           # garbage where start is not set
        for s, c in EVENTS.get(f, {}).items():
            start[s], clip[s] = 1, c
        bank.windows(torch.from_numpy(start).to(dev), torch.from_numpy(clip).to(dev), slot_clip, slot_cursor, X, side, ct)
        served = model.step(start, clip)
        for b, sv in enumerate(served):
            where = f"frame {f} slot {b} serves {sv}"
            if sv is None:
                assert not X[b].any() and not side[b].any() and not ct[b].any(), where
                continue
            r = int(offsets[sv[0]] + sv[1])
            seen.add(sv)
            assert torch.equal(X[b], rX[r]), where + ": X"
            assert torch.equal(side[b], rside[r]), where + ": side"
            assert torch.equal(ct[b], rct[r]), where + ": contacts"
    assert seen == {(c, w) for c in range(len(nwins)) for w in range(nwins[c])}, "every window of every clip"
    want_clip = [-1 if st is None else st[0] for st in model.state]
    want_cur = [0 if st is None else st[1] for st in model.state]
    assert slot_clip.tolist() == want_clip and slot_cursor.tolist() == want_cur
    assert want_cur[0] == nwins[4]                     # clamped after the last window
    assert want_clip[3] == -1 and want_clip[7] == -1


# ---------------------------------------------------------------------------------------------------------------------
# sessions
# ---------------------------------------------------------------------------------------------------------------------
SB = 6
SFRAMES = 12
SEVENTS = {0: {0: 0, 1: 5, 3: 2}, 1: {2: 1}, 4: {0: 3, 4: 0}, 6: {1: 2, 5: 9}, 8: {3: 1}, 9: {2: 4}}
_SESSION_CACHE = {}


def _session_bank():
    if "bank" not in _SESSION_CACHE:
        _SESSION_CACHE["bank"] = _bank_and_reference((31, 40, 75, 36, 33))
    return _SESSION_CACHE["bank"]


def _schedule():
    rows = []
    for f in range(SFRAMES):
        start, clip = np.zeros(SB, dtype=np.uint8), np.zeros(SB, dtype=np.int32)
        for s, c in SEVENTS.get(f, {}).items():
            start[s], clip[s] = 1, c
        eps = np.random.default_rng(900 + f).standard_normal((SB, 256)).astype(np.float32)
        rows.append((start, clip, eps))
    return rows


def _snap(sess, out):
    d = {"Y": sess.Y.cpu().numpy(), "match_idx": sess.match_idx[:, 0].cpu().numpy(), **out}
    if sess.with_cm_path:
        d["cm_Y"] = sess.cm_Y.cpu().numpy()
        d.update({"cm_" + k: v for k, v in sess.cm_post.read().items()})
    return d


def _run_reference(precision, tc, **kw):
    """Admission session fed with the features.extract rows of each slot's clip and cursor."""
    bank, rX, rside, rct, offsets, nwins = _session_bank()
    sess, *_ = workload.build_session(SB, n_db=48, precision=precision, match_tensor_cores=tc, admission=True, **kw)
    sess.capture()
    model = SlotModel(SB, nwins)
    frames = []
    for start, clip, eps in _schedule():
        served = model.step(start, clip)
        sess.X.zero_(); sess.side.zero_(); sess.contacts.zero_()
        for b, sv in enumerate(served):
            if sv is not None:
                r = int(offsets[sv[0]] + sv[1])
                sess.X[b].copy_(rX[r]); sess.side[b].copy_(rside[r]); sess.contacts[b].copy_(rct[r])
        sess.start.copy_(torch.from_numpy(start))
        sess.eps.copy_(torch.from_numpy(eps))
        sess.step_device()
        frames.append(_snap(sess, sess.post.read()))
    return frames


def _run_bank(precision, tc, **kw):
    bank = _session_bank()[0]
    sess, *_ = workload.build_session(SB, n_db=48, precision=precision, match_tensor_cores=tc, admission=True,
                                      source_bank=bank, **kw)
    sess.capture()
    frames = []
    for start, clip, eps in _schedule():
        out = sess.step_bank(start, clip, eps)
        frames.append(_snap(sess, out))
    return sess, frames


def _compare(got, want, keys):
    for f, (a, b) in enumerate(zip(got, want)):
        for k in keys:
            np.testing.assert_array_equal(a[k], b[k], err_msg=f"frame {f}: {k}")


KEYS = ("Y", "match_idx") + OUT_KEYS


@pytest.mark.gpu
@pytest.mark.parametrize("precision,tc", [("bf16", True), ("fp32", False)])
def test_bank_session_matches_admission_session(precision, tc):
    sess, got = _run_bank(precision, tc)
    _compare(got, _run_reference(precision, tc), KEYS)
    assert sess.h2d_bytes() == SB + SB * 4 + SB * 256 * 4


@pytest.mark.gpu
def test_bank_session_lanes_and_second_decode():
    _, got = _run_bank("bf16", False, lanes=2, with_cm_path=True)
    want = _run_reference("bf16", False, with_cm_path=True)
    _compare(got, want, KEYS + ("cm_Y",) + tuple("cm_" + k for k in OUT_KEYS))


@pytest.mark.gpu
def test_bank_session_pipelined_submit_collect():
    _, want = _run_bank("bf16", True)
    bank = _session_bank()[0]
    sess, *_ = workload.build_session(SB, n_db=48, precision="bf16", match_tensor_cores=True, admission=True,
                                      source_bank=bank)
    sess.capture()
    pins = []
    for start, clip, eps in _schedule():
        pin = sess.pinned_inputs()
        assert set(pin) == {"start", "clip", "eps"}
        pin["start"].numpy()[...] = start
        pin["clip"].numpy()[...] = clip
        pin["eps"].numpy()[...] = eps
        pins.append(pin)
    got, prev = [], None
    for f in range(SFRAMES):
        t = sess.submit(pins[f])
        if prev is not None:
            got.append(sess.collect(prev))
        prev = t
    got.append(sess.collect(prev))
    _compare(got, want, OUT_KEYS)


# ---------------------------------------------------------------------------------------------------------------------
# CPU only
# ---------------------------------------------------------------------------------------------------------------------
def test_source_windows_rejects_bad_arguments_without_a_device():
    lib = _lib.load()
    fake = C.c_void_p(256)                               # never dereferenced: validation comes first

    def call(**kw):
        a = dict(rot=fake, pos=fake, vel=fake, ang=fake, bc=fake, nf=100, first=fake, frames=fake, nc=4, par=fake, T=60,
                 J=25, xm=fake, xs=fake, start=fake, clip=fake, sc=fake, scur=fake, B=4, X=fake, side=fake,
                 stride=60 * 3 + 6, ct=fake)
        a.update(kw)
        return lib.mocha_source_windows(*a.values(), None)

    for kw, msg in (({"rot": None}, b"null bank"), ({"par": None}, b"null bank"), ({"xs": None}, b"null bank"),
                    ({"start": None}, b"null slot"), ({"sc": None}, b"null slot"), ({"X": None}, b"null slot"),
                    ({"B": 0}, b"bad sizes"), ({"nc": 0}, b"bad sizes"), ({"nf": 0}, b"bad sizes"),
                    ({"J": 33}, b"J="), ({"J": 1}, b"J="), ({"T": 4}, b"T="),
                    ({"stride": 60 * 3 + 5}, b"side rows"), ({"rot": C.c_void_p(260)}, b"aligned")):
        assert call(**kw) == -1, kw
        err = lib.mocha_last_error()
        assert b"mocha_source_windows" in err and msg in err, (kw, err)


def test_frame_windows_of_process_frames_equal_process_clip():
    for n in range(31, 251):
        c = synthetic.make_clip(n, seed=n)
        want = preprocess.process_clip(c)
        got = preprocess.frame_windows(preprocess.process_frames(c))
        for k in ("pos", "vel", "rot", "ang", "contacts", "parents"):
            assert got[k].dtype == want[k].dtype and np.array_equal(got[k], want[k]), (n, k)
        assert got["names"] == want["names"]
        assert got["pos"].shape[0] == n - T // 4


def test_source_bank_and_session_argument_checks():
    Xm, Xs = _norm()
    bank = SourceBank(200, 2, Xm, Xs, device="cpu")      # CPU tensors: add() and its checks need no device
    with pytest.raises(_lib.MochaError, match="more than 15 frames"):
        bank.add(_frames16() | {k: _frames16()[k][:15] for k in ("pos", "vel", "rot", "ang", "contacts")})
    assert bank.add(synthetic.make_clip(100, seed=1)) == (0, 85)
    with pytest.raises(_lib.MochaError, match="bank full"):
        bank.add(synthetic.make_clip(101, seed=2))       # 201 frames > 200
    assert bank.add(_frames16()) == (1, 1)
    with pytest.raises(_lib.MochaError, match="bank full"):
        bank.add(_frames16())                            # 3 clips > 2
    with pytest.raises(_lib.MochaError, match="rot must be"):
        bank.add(_frames16() | {"rot": np.zeros((16, 25, 3), np.float32)})
    bank.clear()
    assert bank.n_clips == 0 and bank.n_frames == 0 and not bank.clip_frames.any()
    assert bank.add(_frames16()) == (0, 1)
    with pytest.raises(_lib.MochaError, match="X_mean"):
        SourceBank(10, 1, Xm[1:], Xs)
    with pytest.raises(_lib.MochaError, match="max_frames"):
        SourceBank(0, 1, Xm, Xs)
    # the session refuses a bank without admission before it touches a device
    with pytest.raises(_lib.MochaError, match="admission=True"):
        CharacterizationSession(None, None, None, None, None, None, 4, source_bank=bank)
