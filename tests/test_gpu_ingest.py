"""Raw clip ingestion on the device (SourceBank.add_raw + mocha_ingest_frames, DESIGN §5d).

- parity with the host path: every float32 array equals preprocess.process_frames bit for bit, but for at most 1e-6 of
  the elements differing by exactly one float32 ulp (fp64 sin / cos / atan2 and the savgol edge fits may land on the
  other side of a float32 rounding boundary); contacts equal. Synthetic clips of 31 .. 1,000 frames, the six Euler
  orders, a clip that winds past 360 degrees, one without foot contact, one in contact throughout;
- one add_raw of a batch equals one call per clip, and the bank tables equal add()'s; add and add_raw mix;
- rejected batches leave the bank unchanged;
- downstream: mocha_source_windows and serve() payloads over a raw-ingested bank against a host-ingested one;
- CPU only: the entry point's argument checks, the savgol tables against scipy.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from mocha_sigasia2023_b200 import _lib, preprocess, synthetic, workload
from mocha_sigasia2023_b200.result_bank import ResultBank
from mocha_sigasia2023_b200.source_bank import EULER_ORDERS, SourceBank, savgol_tables

KEYS = ("pos", "vel", "rot", "ang")
LENGTHS = (31, 32, 45, 61, 100, 240, 1000)


def _norm():
    n = synthetic.make_norm_stats(7)["norm"]
    return n["X_mean"], n["X_std"]


def _winding_clip(F=120, seed=5):
    """A clip whose spine and arm rotations wind through 720 degrees, stored wrapped to [-180, 180) as a BVH exporter
    writes them: at each wrap the quaternion jumps to the other hemisphere and the host _unroll flips signs."""
    clip = synthetic.make_clip(F, seed=seed)
    t = np.arange(F) / (F - 1)
    for j in (5, 10, 17):
        clip["rotations"][:, j, 0] = np.mod(clip["rotations"][:, j, 0] + 720.0 * t + 180.0, 360.0) - 180.0
    return clip


def _no_contact_clip(F=90, seed=6):
    clip = synthetic.make_clip(F, seed=seed)
    clip["positions"][:, 0, 2] *= 15.0                     # >= 2.4 m/s of root speed: toes never slow down
    return clip


def _contact_clip(F=64, seed=7):
    """Every joint moving, slowly: the toes stay below 0.5 m/s throughout. (A clip whose root stands exactly still is
    not used: its filtered root trajectory is constant in exact arithmetic, so its velocities are the rounding noise
    of the savgol edge fits, which scipy computes with polyfit and the device with the same linear map as a table.)"""
    clip = synthetic.make_clip(F, seed=seed)
    clip["rotations"] *= 0.05
    clip["positions"][:, 0, 0] *= 0.05
    clip["positions"][:, 0, 2] *= 0.05
    return clip


def _parity_clips():
    clips = [synthetic.make_clip(F, seed=900 + F) for F in LENGTHS]
    base = synthetic.make_clip(50, seed=42)
    clips += [dict(base, order=o) for o in EULER_ORDERS]
    clips += [_winding_clip(), _no_contact_clip(), _contact_clip()]
    return clips


def _host_toe_speed(clip):
    """The fp64 toe speeds process_frames thresholds at 0.5: its own steps, stopped before the comparison."""
    P = preprocess
    seen = {}
    fk_vel = P._fk_vel

    def spy(*args):
        out = fk_vel(*args)
        seen["gvel"] = out[2]
        return out

    P._fk_vel = spy
    try:
        frames = P.process_frames(clip)
    finally:
        P._fk_vel = fk_vel
    toes = [frames["names"].index("LeftToeBase"), frames["names"].index("RightToeBase")]
    return np.sqrt((seen["gvel"][:, toes] ** 2).sum(-1))


def _bank_for(clips, extra_frames=0, extra_clips=0):
    Xm, Xs = _norm()
    return SourceBank(sum(c["rotations"].shape[0] for c in clips) + extra_frames, len(clips) + extra_clips, Xm, Xs)


def _rows(bank, cid):
    a, F = bank.clip_start[cid], bank.clip_nwin[cid] + bank.T // 4
    out = {k: getattr(bank, k)[a:a + F].cpu().numpy() for k in KEYS}
    out["contacts"] = bank.contacts[a:a + F].cpu().numpy()
    return out


def _ulp_diff(a, b):
    """Elements whose bits differ, and whether every such element is exactly one float32 ulp away."""
    ia, ib = a.view(np.int32).astype(np.int64), b.view(np.int32).astype(np.int64)
    bad = ia != ib
    one = (np.abs(ia - ib) == 1) & (np.sign(a) == np.sign(b))
    return int(bad.sum()), bool(one[bad].all())


_CACHE = {}


def _ingested():
    if "parity" not in _CACHE:
        clips = _parity_clips()
        bank = _bank_for(clips)
        ids = bank.add_raw(clips)
        torch.cuda.synchronize()
        _CACHE["parity"] = clips, bank, ids
    return _CACHE["parity"]


@pytest.mark.gpu
def test_add_raw_matches_process_frames():
    clips, bank, ids = _ingested()
    # the winding clip really exercises the sign recurrence; the two contact clips are what they claim
    P = preprocess
    wind = clips[len(LENGTHS) + 6]
    q = P._from_euler(np.radians(wind["rotations"]), wind["order"])
    assert (P._unroll(q) != q).any()
    total = differ = 0
    for clip, (cid, nwin) in zip(clips, ids):
        want = P.process_frames(clip)
        F = want["pos"].shape[0]
        assert nwin == F - bank.T // 4
        speed = _host_toe_speed(clip)
        assert np.abs(speed - 0.5).min() > 1e-9            # the threshold decision is not a rounding question
        got = _rows(bank, cid)
        for k in KEYS:
            n, one_ulp = _ulp_diff(got[k], want[k])
            assert one_ulp, f"clip of {F} frames ({clip['order']}): {k} differs by more than one ulp"
            total += want[k].size
            differ += n
        np.testing.assert_array_equal(got["contacts"], want["contacts"])
    assert not _rows(bank, ids[-2][0])["contacts"].any()
    assert _rows(bank, ids[-1][0])["contacts"].all()
    print(f"add_raw vs process_frames: {differ} of {total} float32 elements differ (by one ulp)")
    assert differ <= 1e-6 * total


@pytest.mark.gpu
def test_batch_equals_one_at_a_time_and_add_tables():
    clips, bank, ids = _ingested()
    one = _bank_for(clips)
    for clip in clips:
        one.add_raw([clip])
    host = _bank_for(clips)
    for clip in clips:
        host.add(clip)
    torch.cuda.synchronize()
    for k in KEYS + ("contacts",):
        assert torch.equal(getattr(bank, k), getattr(one, k)), k
    for b in (one, host):
        assert (b.n_clips, b.n_frames, b.clip_nwin, b.clip_start) == (bank.n_clips, bank.n_frames, bank.clip_nwin,
                                                                        bank.clip_start)
        assert torch.equal(b.clip_first, bank.clip_first) and torch.equal(b.clip_frames, bank.clip_frames)
    assert [c for c, _ in ids] == list(range(len(clips)))


@pytest.mark.gpu
def test_add_and_add_raw_mix():
    clips = [synthetic.make_clip(F, seed=60 + F) for F in (40, 33, 75, 52)]
    mixed = _bank_for(clips, extra_frames=11, extra_clips=1)
    assert mixed.add(clips[0]) == (0, 40 - 15)
    assert mixed.add_raw(clips[1:3]) == [(1, 33 - 15), (2, 75 - 15)]
    assert mixed.add(clips[3]) == (3, 52 - 15)
    assert mixed.add_raw([]) == []
    host = _bank_for(clips, extra_frames=11, extra_clips=1)
    for c in clips:
        host.add(c)
    torch.cuda.synchronize()
    assert mixed.clip_start == host.clip_start and torch.equal(mixed.clip_first, host.clip_first)
    for cid in range(4):
        a, b = _rows(mixed, cid), _rows(host, cid)
        for k in KEYS:
            assert _ulp_diff(a[k], b[k])[1], k
        np.testing.assert_array_equal(a["contacts"], b["contacts"])


def _rejections():
    good = synthetic.make_clip(40, seed=1)
    missing = synthetic.make_clip(40, seed=2)
    missing["names"] = ["Chest" if n == "Spine2" else n for n in missing["names"]]
    other = synthetic.make_clip(40, seed=3)
    other["parents"] = np.array(other["parents"])
    other["parents"][10] = 8
    return {
        "short": [good, synthetic.make_clip(30, seed=4)],
        "missing joint": [good, missing],
        "skeleton": [good, other],
        "order": [good, dict(synthetic.make_clip(40, seed=5), order="xxz")],
        "overflow": [good] * 4,
    }


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["short", "missing joint", "skeleton", "order", "overflow"])
def test_rejected_batches_leave_the_bank_unchanged(case):
    Xm, Xs = _norm()
    bank = SourceBank(200, 4, Xm, Xs)
    bank.add_raw([synthetic.make_clip(60, seed=9)])
    torch.cuda.synchronize()
    before = (bank.n_clips, bank.n_frames, list(bank.clip_nwin), list(bank.clip_start), bank.clip_first.clone(),
              bank.clip_frames.clone(), bank.pos.clone(), bank.contacts.clone())
    with pytest.raises(_lib.MochaError):
        bank.add_raw(_rejections()[case])
    torch.cuda.synchronize()
    after = (bank.n_clips, bank.n_frames, list(bank.clip_nwin), list(bank.clip_start), bank.clip_first, bank.clip_frames,
             bank.pos, bank.contacts)
    assert before[:4] == after[:4]
    for x, y in zip(before[4:], after[4:]):
        assert torch.equal(x, y)


def _bit_equal(a, b):
    return all(torch.equal(getattr(a, k).view(torch.int32) if k != "contacts" else getattr(a, k),
                           getattr(b, k).view(torch.int32) if k != "contacts" else getattr(b, k))
               for k in KEYS + ("contacts",))


@pytest.mark.gpu
def test_source_windows_over_a_raw_bank():
    clips = [synthetic.make_clip(F, seed=500 + F) for F in (31, 47, 80, 120, 64, 39)]
    raw, host = _bank_for(clips), _bank_for(clips)
    raw.add_raw(clips)
    for c in clips:
        host.add(c)
    exact = _bit_equal(raw, host)
    B, dev = len(clips), torch.device("cuda")
    state = {}
    for name, bank in (("raw", raw), ("host", host)):
        slot_clip = torch.full((B,), -1, dtype=torch.int32, device=dev)
        slot_cursor = torch.zeros((B,), dtype=torch.int32, device=dev)
        outs = []
        for f in range(70):
            start = torch.tensor([1 if f == 0 else 0] * B, dtype=torch.uint8, device=dev)
            clip = torch.arange(B, dtype=torch.int32, device=dev)
            X = torch.empty((B, bank.T, bank.J - 1, 15), dtype=torch.float32, device=dev)
            side = torch.empty((B, bank.T * 3 + 6), dtype=torch.float32, device=dev)
            ct = torch.empty((B, 2), dtype=torch.uint8, device=dev)
            bank.windows(start, clip, slot_clip, slot_cursor, X, side, ct)
            outs.append((X.cpu(), side.cpu(), ct.cpu()))
        state[name] = outs
    for (xa, sa, ca), (xb, sb, cb) in zip(state["raw"], state["host"]):
        assert torch.equal(ca, cb)
        if exact:
            assert torch.equal(xa, xb) and torch.equal(sa, sb)
        else:
            torch.testing.assert_close(xa, xb, rtol=1e-5, atol=1e-5)
            torch.testing.assert_close(sa, sb, rtol=1e-5, atol=1e-5)


@pytest.mark.gpu
def test_serve_payloads_over_a_raw_bank():
    lengths = (31, 40, 52, 36, 45, 70, 33, 58, 41, 37, 49, 66, 34, 44, 39, 61, 35, 47, 55, 32)
    clips = [synthetic.make_clip(F, seed=800 + i) for i, F in enumerate(lengths)]
    raw, host = _bank_for(clips), _bank_for(clips)
    raw.add_raw(clips)
    for c in clips:
        host.add(c)
    exact = _bit_equal(raw, host)
    rng = np.random.default_rng(3)
    eps = {c: rng.standard_normal((host.clip_nwin[c] - 1, 256)).astype(np.float32) for c in range(len(clips))}
    ids = list(range(len(clips)))
    got = {}
    for name, bank in (("raw", raw), ("host", host)):
        rb = ResultBank(bank)
        sess, *_ = workload.build_session(16, n_db=48, precision="bf16", match_tensor_cores=False, admission=True,
                                          source_bank=bank, result_bank=rb)
        sess.capture()
        got[name] = sess.serve(ids, eps=eps)
    for c in ids:
        for k in got["host"][c]:
            a, b = got["raw"][c][k], got["host"][c][k]
            if exact or k == "match":
                np.testing.assert_array_equal(a, b, err_msg=f"clip {c}: {k}")
            else:
                tol = 1e-4 if k.startswith("src") else 2e-3
                np.testing.assert_allclose(a, b, rtol=tol, atol=tol, err_msg=f"clip {c}: {k}")


# ---------------------------------------------------------------------------------------------------------------------
# CPU only
# ---------------------------------------------------------------------------------------------------------------------
def test_ingest_entry_point_rejects_bad_arguments_without_a_device():
    lib = _lib.load()
    par = (C.c_int32 * 24)(*([-1] + [0] * 23))
    jnt = (C.c_int32 * 7)(7, 9, 16, 1, 20, 4, 23)
    p = C.c_void_p(16)
    good = dict(rot=p, pos=p, n=100, first=p, frames=p, order=p, nc=2, maxf=60, parents=par, joints=jnt, J=25, s15=p,
                s31=p, brot=p, bpos=p, bvel=p, bang=p, bct=p, rows=100, row0=0, ws=p, wsb=1 << 30, stream=None)

    def call(**kw):
        a = dict(good, **kw)
        return lib.mocha_ingest_frames(*a.values())

    for kw in ({"J": 1}, {"J": 40}, {"n": 0}, {"nc": 0}, {"rows": 0}, {"row0": -1}, {"maxf": 30}, {"maxf": 10 ** 7},
               {"rot": None}, {"brot": None}, {"s31": None}, {"ws": None}, {"wsb": 16}, {"parents": None},
               {"parents": (C.c_int32 * 24)(*([0] * 24))}, {"parents": (C.c_int32 * 24)(*([-1] + [5] * 23))},
               {"joints": (C.c_int32 * 7)(7, 9, 16, 1, 20, 4, 24)}):
        assert call(**kw) < 0, kw
        assert b"mocha_ingest_frames" in lib.mocha_last_error()
    assert lib.mocha_ingest_workspace_bytes(0, 25) == 0 and lib.mocha_ingest_workspace_bytes(10, 1) == 0
    assert lib.mocha_ingest_workspace_bytes(100, 25) >= 100 * 24 * 7 * 8


def test_savgol_tables_restate_scipy():
    import scipy.signal as signal
    rng = np.random.default_rng(0)
    for wl in (15, 31):
        tab, h = savgol_tables(wl), wl // 2
        w, left, right = tab[:wl], tab[wl:wl + h * wl].reshape(h, wl), tab[wl + h * wl:].reshape(h, wl)
        x = rng.normal(size=200)
        want = signal.savgol_filter(x, wl, 3, mode="interp")
        got = np.empty_like(x)
        for i in range(h, len(x) - h):                    # ndimage's symmetric correlation, in its order
            t = x[i] * w[h]
            for k in range(h):
                t = t + (x[i - h + k] + x[i + h - k]) * w[k]
            got[i] = t
        got[:h], got[-h:] = left @ x[:wl], right @ x[-wl:]
        np.testing.assert_array_equal(got[h:-h], want[h:-h])
        np.testing.assert_allclose(got, want, rtol=0, atol=1e-13)


def test_add_raw_checks_run_before_the_device():
    Xm, Xs = _norm()
    bank = SourceBank(100, 2, Xm, Xs, device="cpu")
    with pytest.raises(_lib.MochaError, match="order"):
        bank.add_raw([dict(synthetic.make_clip(40), order="abc")])
    with pytest.raises(_lib.MochaError, match="frames"):
        bank.add_raw([synthetic.make_clip(30)])
    with pytest.raises(_lib.MochaError, match="full"):
        bank.add_raw([synthetic.make_clip(60), synthetic.make_clip(60)])
    assert bank.n_clips == 0 and bank.add_raw([]) == []
