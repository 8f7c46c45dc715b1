"""Character bank (CharacterBank, segmented matching, mocha_slot_segments, CharacterizationSession(characters=...)):

- kernel level: random rows where each query's global nearest row is planted in ANOTHER character's segment; the
  exact segmented matcher equals mocha_match_exact over the sliced segment (+ its offset) bit for bit, and the split-K,
  persistent bf16 and TF32 segmented matchers equal a float64 brute force over the segment; short, empty and clipped
  segments;
- mocha_slot_segments against a host model through staggered and overriding starts and out-of-range ids;
- session level: 3 characters of 385 / 200 / 97 rows served by one 16-slot session give every clip the payload of a
  single-character session running the same clips in the same slots (fp64 and tensor-core matchers, bf16 and fp32,
  two lanes + the second decode, a capture taken after an earlier serve against one taken mid-run);
- characterize_many with two character clips against the reference recording (e2e.npz);
- CPU only: argument checks of the new entry points, CharacterBank validation, serve(characters=...) checks.
"""
import os
import types

import numpy as np
import pytest
import torch

from mocha_sigasia2023_b200 import _lib, feature_db, preprocess, synthetic, weights, workload
from mocha_sigasia2023_b200.character_bank import CharacterBank
from mocha_sigasia2023_b200.result_bank import ResultBank, serving_schedule
from mocha_sigasia2023_b200.session import CharacterizationSession
from mocha_sigasia2023_b200.source_bank import SourceBank

P = _lib.ptr


def _planted(sizes, D, nq, seed):
    """DB rows of len(sizes) characters back to back and nq queries; query q belongs to character qc[q]. Its two
    nearest rows of its own segment are planted (squared distances ~0.0025 D and ~0.01 D), and its global nearest row
    (~0.0001 D) is planted in the next character's segment (planted[q]) while that segment has free rows. Random rows
    lie ~2 D away."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    N = int(sum(sizes))
    first = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    X = torch.randn((N, D), generator=g, device="cuda")
    Q = torch.randn((nq, D), generator=g, device="cuda")
    qc = np.arange(nq) % len(sizes)
    rng = np.random.default_rng(seed)
    free = [list(rng.permutation(n) + f) for n, f in zip(sizes, first)]
    planted = np.zeros(nq, dtype=bool)
    for q in range(nq):
        c, o = qc[q], (qc[q] + 1) % len(sizes)
        if len(free[c]) < 2 or not free[o]:
            continue
        planted[q] = True
        for scale, cc in ((0.05, c), (0.1, c), (0.01, o)):
            X[int(free[cc].pop())] = Q[q] + scale * torch.randn((D,), generator=g, device="cuda")
    return X.contiguous(), Q.contiguous(), qc, first, planted


def _segments(qc, first, sizes):
    sf = torch.tensor([int(first[c]) for c in qc], dtype=torch.int64, device="cuda")
    sr = torch.tensor([int(sizes[c]) for c in qc], dtype=torch.int32, device="cuda")
    return sf, sr


def _ws(n):
    return torch.empty(max(int(n), 1) + 4096, dtype=torch.uint8, device="cuda")


def _exact_seg(Q, X, sf, sr, k, offset=0):
    lib = _lib.load()
    nq, D = Q.shape
    idx = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dist = torch.empty((nq, k), dtype=torch.float64, device="cuda")
    ws = _ws(lib.mocha_match_exact_workspace_bytes(nq, X.shape[0], k))
    _lib.check(lib.mocha_match_exact_segmented(P(Q), nq, P(X), X.shape[0], D, k, offset, P(sf), P(sr), P(idx), P(dist),
                                               P(ws), ws.numel(), _lib.stream_ptr()), "exact_segmented")
    return idx.cpu().numpy(), dist.cpu().numpy()


def _exact(Q, X, k, offset):
    lib = _lib.load()
    nq, D = Q.shape
    idx = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dist = torch.empty((nq, k), dtype=torch.float64, device="cuda")
    ws = _ws(lib.mocha_match_exact_workspace_bytes(nq, X.shape[0], k))
    _lib.check(lib.mocha_match_exact(P(Q), nq, P(X), X.shape[0], D, k, offset, P(idx), P(dist), P(ws), ws.numel(),
                                     _lib.stream_ptr()), "exact")
    return idx.cpu().numpy(), dist.cpu().numpy()


def _tc_seg(Q, X, sf, sr, k, storage, kc=8):
    lib = _lib.load()
    nq, D = Q.shape
    N = X.shape[0]
    idx = torch.empty((nq, k), dtype=torch.int64, device="cuda")
    dist = torch.empty((nq, k), dtype=torch.float64, device="cuda")
    ws = _ws(lib.mocha_match_tc_workspace_bytes(nq, N, D, kc))
    if storage == "bf16":
        c = X.mean(dim=0)
        X16 = (X - c).to(torch.bfloat16).contiguous()
        Q16 = (Q - c).to(torch.bfloat16).contiguous()
        norm = (X16.float() ** 2).sum(dim=1).contiguous()
        args = (P(Q), P(Q16), nq, P(X16), P(X), P(norm))
    else:
        norm = (X * X).sum(dim=1).contiguous()
        args = (P(Q), None, nq, None, P(X), P(norm))
    _lib.check(lib.mocha_match_tc_segmented(*args, N, D, k, kc, 0, P(sf), P(sr), P(idx), P(dist), P(ws), ws.numel(),
                                            _lib.stream_ptr()), "tc_segmented")
    return idx.cpu().numpy(), dist.cpu().numpy()


def _brute(Q, X, lo, n):
    """float64 squared distances of the queries to rows lo .. lo + n."""
    return torch.cdist(Q.double(), X[lo:lo + n].double(), compute_mode="donot_use_mm_for_euclid_dist").cpu().numpy() ** 2


SIZES = (385, 200, 97)


@pytest.mark.gpu
@pytest.mark.parametrize("nq,k", [(3, 1), (40, 4), (128, 1)])
def test_exact_segmented_equals_exact_on_the_slice_bit_for_bit(nq, k):
    X, Q, qc, first, planted = _planted(SIZES, 23040, nq, seed=nq)
    sf, sr = _segments(qc, first, SIZES)
    idx, dist = _exact_seg(Q, X, sf, sr, k, offset=1000)
    whole, _ = _exact(Q, X, 1, 0)
    for c, n in enumerate(SIZES):
        qs = np.nonzero(qc == c)[0]
        if qs.size == 0:
            continue
        want_i, want_d = _exact(Q[qs].contiguous(), X[first[c]:first[c] + n].contiguous(), k, 1000 + int(first[c]))
        np.testing.assert_array_equal(idx[qs], want_i)
        np.testing.assert_array_equal(dist[qs].view(np.int64), want_d.view(np.int64))   # bit for bit
        # the unsegmented matcher finds the planted row in the next character's segment
        o, qp = (c + 1) % len(SIZES), qs[planted[qs]]
        assert ((whole[qp, 0] >= first[o]) & (whole[qp, 0] < first[o] + SIZES[o])).all()
    assert planted.sum() >= min(nq, 40) and (idx[planted, 0] - 1000 != whole[planted, 0]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("storage,D,nq", [("bf16", 23040, 128),      # split-K coarse pass (N <= 8192, long rows)
                                          ("bf16", 256, 128),        # persistent coarse pass, bf16
                                          ("fp32", 256, 128),        # persistent coarse pass, TF32
                                          ("bf16", 256, 300)])       # persistent, three m-tiles
def test_tc_segmented_equals_float64_brute_force(storage, D, nq):
    X, Q, qc, first, planted = _planted(SIZES, D, nq, seed=D + nq)
    sf, sr = _segments(qc, first, SIZES)
    idx, dist = _tc_seg(Q, X, sf, sr, 2, storage)
    for c, n in enumerate(SIZES):
        qs = np.nonzero(qc == c)[0]
        d2 = _brute(Q[qs], X, int(first[c]), n)
        order = np.argsort(d2, axis=1, kind="stable")[:, :2]
        np.testing.assert_array_equal(idx[qs], order + first[c], err_msg=f"{storage} D={D} character {c}")
        np.testing.assert_allclose(dist[qs] ** 2, np.take_along_axis(d2, order, 1), rtol=1e-9)
    assert planted.sum() >= 40


@pytest.mark.gpu
@pytest.mark.parametrize("path", ["exact", "bf16", "fp32"])
def test_short_empty_and_clipped_segments(path):
    sizes = (3, 1, 300)
    X, Q, qc, first, _ = _planted(sizes, 256, 8, seed=11)
    N = X.shape[0]
    # per query: a 3-row, a 1-row, an empty, a negative-length, a clipped (past N) and a 0-row-at-N segment
    segs = [(0, 3), (3, 1), (100, 0), (50, -5), (N - 2, 10), (N, 4), (-3, 5), (4, 300)]
    sf = torch.tensor([s[0] for s in segs], dtype=torch.int64, device="cuda")
    sr = torch.tensor([s[1] for s in segs], dtype=torch.int32, device="cuda")
    k = 4
    if path == "exact":
        idx, dist = _exact_seg(Q, X, sf, sr, k)
    else:
        idx, dist = _tc_seg(Q, X, sf, sr, k, path, kc=8)
    for q, (f, n) in enumerate(segs):
        lo, hi = max(f, 0), min(f + n, N)
        m = max(hi - lo, 0)
        if m:
            d2 = _brute(Q[q:q + 1], X, lo, m)[0]
            order = np.argsort(d2, kind="stable")[:min(k, m)]
            got = idx[q, :min(k, m)]
            assert set(got.tolist()) <= set(range(lo, hi)), f"query {q}: {got} outside [{lo}, {hi})"
            if m <= k or path == "exact":
                np.testing.assert_array_equal(got, order + lo, err_msg=f"query {q}")
        assert (idx[q, min(k, m):] == -1).all() and np.isinf(dist[q, min(k, m):]).all(), f"query {q}"


class SegModel:
    def __init__(self, B):
        self.slot = np.full(B, -1, dtype=np.int64)

    def step(self, start, character, first, rows):
        self.slot[start.astype(bool)] = character[start.astype(bool)]
        ok = (self.slot >= 0) & (self.slot < len(rows))
        c = np.where(ok, self.slot, 0)
        return np.where(ok, first[c], 0), np.where(ok, rows[c], 0)


@pytest.mark.gpu
def test_slot_segments_against_a_host_model():
    lib = _lib.load()
    B = 300
    rows = np.array([385, 200, 97, 1, 4000], dtype=np.int32)
    first = np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64)
    cf, cr = torch.from_numpy(first).cuda(), torch.from_numpy(rows).cuda()
    slot_char = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    sf = torch.empty((B,), dtype=torch.int64, device="cuda")
    sr = torch.empty((B,), dtype=torch.int32, device="cuda")
    model = SegModel(B)
    rng = np.random.default_rng(3)
    for f in range(12):
        start = (rng.random(B) < (1.0 if f == 0 else 0.3)).astype(np.uint8)
        if f == 1:
            start[:] = 0                                     # no start: segments stay
        character = rng.integers(-2, 7, size=B).astype(np.int32)   # -2, -1, 5, 6: out of range
        st, ch = torch.from_numpy(start).cuda(), torch.from_numpy(character).cuda()
        _lib.check(lib.mocha_slot_segments(P(st), P(ch), P(slot_char), B, P(cf), P(cr), len(rows), P(sf), P(sr),
                                           _lib.stream_ptr()), "slot_segments")
        wf, wr = model.step(start, character, first, rows)
        np.testing.assert_array_equal(slot_char.cpu().numpy(), model.slot, err_msg=f"frame {f}")
        np.testing.assert_array_equal(sf.cpu().numpy(), wf, err_msg=f"frame {f}")
        np.testing.assert_array_equal(sr.cpu().numpy(), wr, err_msg=f"frame {f}")


# ---------------------------------------------------------------------------------------------------------------------
# session level
# ---------------------------------------------------------------------------------------------------------------------
NSLOT = 16
CLIP_LENGTHS = (31, 40, 52, 36, 45, 70, 33, 48, 31, 60, 38, 41, 55, 34, 47, 66, 31, 44, 39, 50)   # 20 clips
CLIP_CHAR = [i % 3 for i in range(len(CLIP_LENGTHS))]
_CACHE = {}


def _fixture():
    if "fx" not in _CACHE:
        gen_sd, cvae_sd = weights.generator_state_dict(1777), weights.cvae_state_dict(1778)
        stats = workload.driver_stats()
        fdbs = [feature_db.build_feature_db(gen_sd, weights.DEFAULT_MODEL_CFG, stats.cnt_mean, stats.cnt_std,
                                            workload.pose_windows(n, 5000 + 17 * c), batch=64)
                for c, n in enumerate(SIZES)]
        n = synthetic.make_norm_stats(7)["norm"]
        frames = [preprocess.process_frames(synthetic.make_clip(L, seed=900 + i)) for i, L in enumerate(CLIP_LENGTHS)]
        bank = SourceBank(sum(f["pos"].shape[0] for f in frames), len(frames), n["X_mean"], n["X_std"])
        for f in frames:
            bank.add(f)
        rng = np.random.default_rng(5)
        eps = {c: rng.standard_normal((bank.clip_nwin[c] - 1, 256)).astype(np.float32) for c in range(bank.n_clips)}
        _CACHE["fx"] = gen_sd, cvae_sd, stats, fdbs, bank, eps
    return _CACHE["fx"]


def _replay_single(c, ids, chars_of, precision, tc, kw, capture_at=0):
    """The single-character session of character c running the bank session's schedule: the clips of character c in
    the same slots on the same frames, every other slot idle. Returns (payloads, per-(clip, window) float64 brute-force
    match over the character's rows and its top-1 / top-2 margin)."""
    gen_sd, cvae_sd, stats, fdbs, bank, eps = _fixture()
    rb = ResultBank(bank)
    fdb = fdbs[c]
    sess = CharacterizationSession(gen_sd, cvae_sd, weights.DEFAULT_MODEL_CFG, stats, fdb.encoded, fdb.rows32,
                                   batch=NSLOT, precision=precision, match_tensor_cores=tc, admission=True,
                                   source_bank=bank, result_bank=rb, **kw)
    start_rows, clip_rows, _ = serving_schedule([bank.clip_nwin[i] for i in ids], NSLOT)
    slot_k, slot_f = [-1] * NSLOT, [0] * NSLOT
    brute = {}
    rows = fdb.rows32
    sess.start.fill_(1)
    sess.clip.fill_(-1)
    sess.step_device()                                     # serve()'s idle frame
    sess.start.zero_()
    for f in range(len(start_rows)):
        if f == capture_at:
            sess.capture()
        e = np.zeros((NSLOT, 256), dtype=np.float32)
        clip = np.full(NSLOT, -1, dtype=np.int32)
        for b in range(NSLOT):
            if start_rows[f][b]:
                slot_k[b], slot_f[b] = int(clip_rows[f][b]), f
                if chars_of[ids[slot_k[b]]] == c:
                    clip[b] = ids[slot_k[b]]
            k = slot_k[b]
            if k >= 0 and chars_of[ids[k]] == c and 1 <= f - slot_f[b] < bank.clip_nwin[ids[k]]:
                e[b] = eps[ids[k]][f - slot_f[b] - 1]
        sess.step_bank(start_rows[f], clip, e)
        mine = [b for b in range(NSLOT) if slot_k[b] >= 0 and chars_of[ids[slot_k[b]]] == c
                and f - slot_f[b] < bank.clip_nwin[ids[slot_k[b]]]]
        if mine:
            d2 = torch.cdist(sess.cnt_nm[mine].double(), rows.double(),
                             compute_mode="donot_use_mm_for_euclid_dist").cpu().numpy() ** 2
            srt = np.sort(d2, axis=1)
            for j, b in enumerate(mine):
                brute[(ids[slot_k[b]], f - slot_f[b])] = (int(np.argmin(d2[j])), srt[j, 1] - srt[j, 0])
    mine_ids = [i for i in ids if chars_of[i] == c]
    rb.payload(mine_ids)
    return {i: rb.read(i) for i in mine_ids}, brute


def _check_session(precision, tc, kw, capture_at=0):
    gen_sd, cvae_sd, stats, fdbs, bank, eps = _fixture()
    chars = CharacterBank.from_feature_dbs(fdbs)
    assert chars.n_chars == 3 and [chars.rows(c) for c in range(3)] == list(SIZES) and chars.N == sum(SIZES)
    rb = ResultBank(bank)
    sess = CharacterizationSession(gen_sd, cvae_sd, weights.DEFAULT_MODEL_CFG, stats, None, None, batch=NSLOT,
                                   precision=precision, match_tensor_cores=tc, admission=True, source_bank=bank,
                                   result_bank=rb, characters=chars, **kw)
    assert sess._use_tc == bool(tc)
    ids = list(range(bank.n_clips))[::-1]
    chars_of = {i: CLIP_CHAR[i] for i in ids}
    if capture_at:
        # a capture taken mid-serve: frames before it run eagerly (a second serve() then replays the graph)
        sess.serve(ids[:3], eps=eps, characters=chars_of)
    sess.capture()
    got = sess.serve(ids, eps=eps, characters=chars_of)
    for c in range(3):
        want, brute = _replay_single(c, ids, chars_of, precision, tc, kw, capture_at=capture_at)
        for i, p in want.items():
            m = got[i]["match"]
            assert ((m >= 0) & (m < SIZES[c])).all(), f"clip {i}: match outside character {c}'s rows"
            if tc:   # the coarse cut differs between the two sessions: both must find the true segment neighbour
                for w in range(bank.clip_nwin[i]):
                    nn, margin = brute[(i, w)]
                    if margin > 1e-5:
                        assert m[w] == nn and p["match"][w] == nn, f"clip {i} window {w}"
            for key in p:
                np.testing.assert_array_equal(got[i][key], p[key], err_msg=f"clip {i} (character {c}): {key}")
        assert len(want) == sum(1 for i in ids if CLIP_CHAR[i] == c)
    # ResultBank.read() keeps bank rows
    i0 = ids[0]
    rb.payload([i0])
    np.testing.assert_array_equal(rb.read(i0)["match"], got[i0]["match"] + chars.char_first_host[CLIP_CHAR[i0]])


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
@pytest.mark.parametrize("tc", [False, True])
def test_bank_session_serves_each_clip_like_its_single_character_session(precision, tc):
    _check_session(precision, tc, {})


@pytest.mark.gpu
def test_bank_session_two_lanes_second_decode_and_capture_mid_serve():
    _check_session("bf16", False, {"lanes": 2, "with_cm_path": True}, capture_at=0)
    _check_session("bf16", True, {}, capture_at=1)


@pytest.mark.gpu
def test_bank_session_inputs_and_idle_characters():
    gen_sd, cvae_sd, stats, fdbs, bank, eps = _fixture()
    chars = CharacterBank.from_feature_dbs(fdbs)
    rb = ResultBank(bank)
    sess = CharacterizationSession(gen_sd, cvae_sd, weights.DEFAULT_MODEL_CFG, stats, None, None, batch=4,
                                   precision="bf16", match_tensor_cores=False, admission=True, source_bank=bank,
                                   result_bank=rb, characters=chars, with_cm_path=True)
    assert set(sess.pinned_inputs()) == {"start", "clip", "character", "eps"}
    assert sess.h2d_bytes() == 4 + 4 * 4 + 4 * 4 * 256 + 4 * 4
    sess.capture()
    # slots 0..3: characters 2, 0, 7 (unknown: matches nothing), -1
    sess.step_bank(np.ones(4, np.uint8), np.array([0, 1, 2, 3], np.int32), None, character=np.array([2, 0, 7, -1]))
    m = sess.match_idx[:, 0].cpu().numpy()
    assert first_of(chars, 2) <= m[0] < first_of(chars, 2) + SIZES[2] and 0 <= m[1] < SIZES[0]
    assert m[2] == -1 and m[3] == -1
    assert np.isfinite(sess.post.out.cpu().numpy().view(np.float64)).all()
    sess.step_bank(None, None, None)                       # no start: characters stay
    assert sess.slot_char.cpu().tolist() == [2, 0, 7, -1]
    with pytest.raises(_lib.MochaError, match="character"):
        sess.serve([0, 1])


def first_of(chars, c):
    return int(chars.char_first_host[c])


@pytest.mark.gpu
def test_characterize_many_with_two_characters_matches_the_reference_recording(golden_dir):
    from mocha_sigasia2023_b200.characterize import characterize_many
    g = np.load(os.path.join(golden_dir, "e2e.npz"))
    src, cha, stats = synthetic.make_clip(240, 0), synthetic.make_clip(400, 1), synthetic.make_norm_stats()
    other = synthetic.make_clip(300, 9)
    outs = characterize_many([synthetic.make_clip(50, seed=5), src, synthetic.make_clip(40, seed=6)], [other, cha],
                             stats, slots=2, eps_seqs={1: g["eps"]}, precision="fp32", cha_index=[0, 1, 0])
    assert [o["match"].shape[0] for o in outs] == [35, 225, 25]
    out = outs[1]
    np.testing.assert_array_equal(out["match"], g["match"])
    np.testing.assert_allclose(out["src_positions"], g["src_positions"], rtol=1e-4, atol=1e-4)
    d = lambda a, b: np.minimum(np.abs(a - b) % 360.0, 360.0 - np.abs(a - b) % 360.0)   # noqa: E731
    assert d(out["src_rotations"], g["src_rotations"]).max() < 0.05
    np.testing.assert_allclose(out["ours_positions"], g["ours_positions"], rtol=2e-3, atol=2e-3)
    err = d(out["ours_rotations"], g["ours_rotations"])
    assert np.median(err) < 0.01 and (err < 0.5).mean() > 0.995
    assert all((o["match"] >= 0).all() and (o["match"] < 285).all() for o in (outs[0], outs[2]))   # 300 frames: 285 rows


# ---------------------------------------------------------------------------------------------------------------------
# CPU only
# ---------------------------------------------------------------------------------------------------------------------
def test_new_entry_points_reject_bad_arguments_without_a_device():
    lib = _lib.load()
    x = 16
    assert lib.mocha_match_exact_segmented(None, 1, None, 1, 1, 1, 0, None, None, None, None, None, 0, None) == -1
    assert b"mocha_match_exact_segmented" in lib.mocha_last_error()
    assert lib.mocha_match_exact_segmented(x, 1, x, 1, 1, 1, 0, None, x, x, None, None, 0, None) == -1
    assert b"segment" in lib.mocha_last_error()
    assert lib.mocha_match_tc_segmented(x, x, 1, x, x, x, 1, 64, 1, 8, 0, x, None, x, None, None, 0, None) == -1
    assert b"segment" in lib.mocha_last_error()
    assert lib.mocha_match_tc_segmented(x, x, 1, x, x, x, 1, 64, 4, 2, 0, x, x, x, None, None, 0, None) == -1
    assert b"mocha_match_tc_segmented" in lib.mocha_last_error()
    assert lib.mocha_slot_segments(x, x, x, 4, x, x, 3, x, None, None) == -1
    assert b"mocha_slot_segments" in lib.mocha_last_error()
    assert lib.mocha_slot_segments(x, x, x, 0, x, x, 3, x, x, None) == -1
    assert lib.mocha_slot_segments(x, x, x, 4, x, x, 0, x, x, None) == -1


def test_character_bank_validation():
    e, r = torch.zeros((5, 90, 256)), torch.zeros((5, 90 * 256))
    with pytest.raises(_lib.MochaError, match="one"):
        CharacterBank([], [])
    with pytest.raises(_lib.MochaError, match="one"):
        CharacterBank([e, e], [r])
    with pytest.raises(_lib.MochaError, match="no rows"):
        CharacterBank([e, e[:0]], [r, r[:0]])
    with pytest.raises(_lib.MochaError, match="same n"):
        CharacterBank([e], [r[:4]])
    with pytest.raises(_lib.MochaError, match="character 1 has rows"):
        CharacterBank([e, e[:, :, :128]], [r, r[:, :90 * 128]])
    with pytest.raises(_lib.MochaError, match="character 1 has rows"):
        CharacterBank([e, e], [r, r[:, :100]])
    with pytest.raises(_lib.MochaError, match="pair of tensors"):
        CharacterBank([e.numpy()], [r])
    with pytest.raises(_lib.MochaError, match="CUDA"):
        CharacterBank([e], [r])                            # CPU tensors
    with pytest.raises(_lib.MochaError, match="CUDA|devices"):
        CharacterBank([e], [r], device="cuda")
    fdb = types.SimpleNamespace(rows32=None, encoded=e)
    with pytest.raises(_lib.MochaError, match="keep_fp32"):
        CharacterBank.from_feature_dbs([fdb])
    fake = types.SimpleNamespace(n_chars=3)
    assert CharacterBank.check_ids(fake, [0, 2]).tolist() == [0, 2]
    with pytest.raises(_lib.MochaError, match="character id 3"):
        CharacterBank.check_ids(fake, [0, 3])
    with pytest.raises(_lib.MochaError, match="character id -1"):
        CharacterBank.check_ids(fake, [-1])


def test_session_and_serve_reject_bad_characters_before_any_launch():
    fake_bank = types.SimpleNamespace(n_chars=2, check_ids=lambda ids: CharacterBank.check_ids(
        types.SimpleNamespace(n_chars=2), ids))
    results = types.SimpleNamespace(_check_ids=lambda ids: None)
    sess = types.SimpleNamespace(results=results, chars=fake_bank)
    with pytest.raises(_lib.MochaError, match="character id 5"):
        CharacterizationSession.serve(sess, [0, 1], characters={0: 1, 1: 5})
    with pytest.raises(_lib.MochaError, match="no character for clip 1"):
        CharacterizationSession.serve(sess, [0, 1], characters={0: 1})
    with pytest.raises(_lib.MochaError, match="pass characters"):
        CharacterizationSession.serve(sess, [0, 1])
    with pytest.raises(_lib.MochaError, match="needs CharacterizationSession"):
        CharacterizationSession.serve(types.SimpleNamespace(results=results, chars=None), [0], characters={0: 0})
    with pytest.raises(_lib.MochaError, match="admission=True"):
        CharacterizationSession(None, None, None, None, None, None, 4, characters=fake_bank)
    with pytest.raises(_lib.MochaError, match="cha_encoded = cha_cnt_nm = None"):
        CharacterizationSession(None, None, None, None, torch.zeros(1), None, 4, admission=True, characters=fake_bank)
    with pytest.raises(_lib.MochaError, match="a character row needs"):
        CharacterizationSession._stage_character(types.SimpleNamespace(chars=None), [0])
    from mocha_sigasia2023_b200.characterize import characterize_many
    with pytest.raises(_lib.MochaError, match="cha_index"):
        characterize_many([{}], [{}, {}], {})
    with pytest.raises(_lib.MochaError, match="cha_index must index"):
        characterize_many([{}], [{}, {}], {}, cha_index=[2])
    with pytest.raises(_lib.MochaError, match="cha_index goes with"):
        characterize_many([{}], {}, {}, cha_index=[0])
