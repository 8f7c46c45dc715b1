"""End-to-end characterization of one source clip with one target character — what the reference's
`test_fullframework.main()` computes (test_fullframework.py:32-721), driven through this package's
CUDA path: preprocess -> GPU window features -> encoder -> per-frame session loop -> final FK ->
Euler angles. Returns the payloads the reference hands to `bvh.save` plus per-frame intermediates."""
from __future__ import annotations

import numpy as np
import torch

from . import features, kinematics as kin
from . import preprocess, skeleton, weights
from .session import CharacterizationSession, NormStats


def to_euler_xyz(q: np.ndarray) -> np.ndarray:
    """quat.to_euler(order='xyz') (motion/quat.py:346-358): host post-processing before BVH export."""
    q0, q1, q2, q3 = q[..., 0:1], q[..., 1:2], q[..., 2:3], q[..., 3:4]
    return np.concatenate([
        np.arctan2(2 * (q0 * q1 + q2 * q3), 1 - 2 * (q1 * q1 + q2 * q2)),
        np.arcsin((2 * (q0 * q2 - q3 * q1)).clip(-1, 1)),
        np.arctan2(2 * (q0 * q3 + q1 * q2), 1 - 2 * (q2 * q2 + q3 * q3))], axis=-1)


def _stats_from_raw(raw: dict) -> NormStats:
    w = raw["cvae_norm"]["std_weight"]
    return NormStats(
        Y_mean=raw["norm"]["Y_mean"][1:], Y_std=raw["norm"]["Y_std"][1:],
        cnt_mean=raw["cnt_norm"]["mean"], cnt_std=raw["cnt_norm"]["std"] / w,
        src_cnt_mean=raw["cvae_norm"]["src_cnt_mean"], src_cnt_std=raw["cvae_norm"]["src_cnt_std"] / w,
        cha_encoded_mean=raw["cvae_norm"]["cha_encoded_mean"], cha_encoded_std=raw["cvae_norm"]["cha_encoded_std"] / w)


def _final_payload(rot, pos, parents_t):
    """(:672-694): global FK of the whole sequence; the simulation root is dropped and the hips take
    their global transform."""
    r = torch.as_tensor(rot, dtype=torch.float32, device="cuda").contiguous()
    p = torch.as_tensor(pos, dtype=torch.float32, device="cuda").contiguous()
    grot, gpos = kin.fk(r, p, parents_t)
    out_pos = np.array(pos[:, 1:], dtype=np.float64)
    out_rot = np.array(rot[:, 1:], dtype=np.float64)
    out_pos[:, 0] = gpos[:, 1].double().cpu().numpy()
    out_rot[:, 0] = grot[:, 1].double().cpu().numpy()
    return np.degrees(to_euler_xyz(out_rot)), out_pos


def _character_db(cha_clip: dict, raw_stats: dict, gen_sd, cvae_sd, stats: NormStats, precision: str,
                  encode_batch: int):
    """Encode the character clip into the feature DB (:213-279, :293-294): (encoded [N,90,256], cnt_nm [N,23040])."""
    dev = "cuda"
    Xm, Xs = raw_stats["norm"]["X_mean"], raw_stats["norm"]["X_std"]
    cha = features.extract(preprocess.process_clip(cha_clip), Xm, Xs, dev)
    dummy = torch.zeros((1, 90, 256)), torch.zeros((1, 90 * 256))
    enc_sess = CharacterizationSession(gen_sd, cvae_sd, weights.DEFAULT_MODEL_CFG, stats, dummy[0], dummy[1],
                                       batch=encode_batch, device=dev, precision=precision)
    encs, nms = [], []
    n_cha = cha["X"].shape[0]
    for s in range(0, n_cha, encode_batch):
        m = min(encode_batch, n_cha - s)
        enc_sess.X.zero_()
        enc_sess.X[:m].copy_(cha["X"][s:s + m])
        enc_sess.encode(enc_sess.X, enc_sess.tokens, enc_sess.encoded, enc_sess.cnt, enc_sess.cnt_nm)
        encs.append(enc_sess.encoded[:m].clone())
        nms.append(enc_sess.cnt_nm[:m].clone())
    return torch.cat(encs), torch.cat(nms)


def characterize(src_clip: dict, cha_clip: dict, raw_stats: dict, gen_sd=None, cvae_sd=None, eps_seq=None,
                 precision: str = "fp32", encode_batch: int = 32, deterministic: bool = False,
                 with_cm_path: bool = False) -> dict:
    """with_cm_path: also run the reference loop's second decode of every frame, the matched DB row's ("cm_trans",
    :465-472), and return its network output rows (Ytil_cm_rows) and the condition and normalised sample of the first
    CVAE call (cvae_cond0, cvae_out0, frame 1)."""
    dev = "cuda"
    gen_sd = gen_sd or weights.generator_state_dict(1777)
    cvae_sd = cvae_sd or weights.cvae_state_dict(1778)
    stats = _stats_from_raw(raw_stats)
    Xm, Xs = raw_stats["norm"]["X_mean"], raw_stats["norm"]["X_std"]
    src = features.extract(preprocess.process_clip(src_clip), Xm, Xs, dev)
    cha_enc, cha_nm = _character_db(cha_clip, raw_stats, gen_sd, cvae_sd, stats, precision, encode_batch)
    n_cha = cha_enc.shape[0]
    sess = CharacterizationSession(gen_sd, cvae_sd, weights.DEFAULT_MODEL_CFG, stats, cha_enc, cha_nm,
                                   batch=1, device=dev, precision=precision, match_tensor_cores=False,
                                   with_cm_path=with_cm_path)
    sess.deterministic = deterministic
    nwin = src["X"].shape[0]
    T = sess.T
    frames, match, ytil_rows, cm_rows, extra = [], [], [], [], {}
    for i in range(nwin):
        sess.X.copy_(src["X"][i:i + 1])
        sess.side[:, :T * 3].copy_(src["Yvel"][i, :, 1].reshape(1, T * 3))
        sess.side[:, T * 3:T * 3 + 3].copy_(src["Yrvel"][i, -1][None])
        sess.side[:, T * 3 + 3:].copy_(src["Yrang"][i, -1][None])
        sess.contacts.copy_(src["contacts"][i, -1][None])
        if i > 0 and not deterministic:
            if eps_seq is not None:
                sess.eps.copy_(torch.as_tensor(eps_seq[i - 1], dtype=torch.float32, device=dev)[None])
            else:
                sess.eps.normal_()
        if i == 2:
            sess.capture()
        sess.step_device()
        frames.append(sess.post.read())
        match.append(int(sess.match_idx[0, 0]))
        ytil_rows.append(((sess.Y[0, -1] - sess.Y_mean) / sess.Y_std).cpu().numpy())
        if with_cm_path:
            cm_rows.append(((sess.cm_Y[0, -1] - sess.Y_mean) / sess.Y_std).cpu().numpy())
            if i == 1:      # read before capture() at frame 2, whose warm-up frame overwrites these buffers
                extra = {"cvae_cond0": sess.cond.cpu().numpy(), "cvae_out0": sess.cvae_out.cpu().numpy()}
    par = kin.parents_tensor(skeleton.BONE_PARENTS, dev)
    # source pose sequence: local pose of each window's last frame with the integrated root (:480-488)
    src_pos = src["Ypos"][:, -1].cpu().numpy().astype(np.float32)
    src_rot = src["Yrot"][:, -1].cpu().numpy().astype(np.float32)
    src_pos[:, 0] = np.stack([f["src_root_pos"][0] for f in frames]).astype(np.float32)
    src_rot[:, 0] = np.stack([f["src_root_rot"][0] for f in frames]).astype(np.float32)
    ik_pos = np.stack([f["ik_pos"][0] for f in frames])
    ik_rot = np.stack([f["ik_rot"][0] for f in frames])
    src_eul, src_p = _final_payload(src_rot, src_pos, par)
    our_eul, our_p = _final_payload(ik_rot, ik_pos, par)
    if with_cm_path:
        extra["Ytil_cm_rows"] = np.stack(cm_rows)
    return {**extra, "src_rotations": src_eul, "src_positions": src_p, "ours_rotations": our_eul, "ours_positions": our_p,
            "match": np.array(match), "Ytil_last_rows": np.stack(ytil_rows),
            "trans_pos": np.stack([f["blend_pos"][0] for f in frames]),
            "trans_rot": np.stack([f["rot"][0] for f in frames]), "n_db": int(n_cha)}


def characterize_many(src_clips, cha_clip: dict, raw_stats: dict, gen_sd=None, cvae_sd=None, slots: int = 1,
                      eps_seqs=None, precision: str = "fp32", encode_batch: int = 32, lanes: int = 1,
                      with_cm_path: bool = False) -> list:
    """The many-clip counterpart of characterize(): every source clip characterized with one target character through
    a source bank, a result bank and one captured admission session of `slots` slots (CharacterizationSession.serve).
    The character DB is built as characterize() builds it, and the session matches with the same fp64 brute-force
    kernel (match_tensor_cores=False).

    eps_seqs: None (fresh standard-normal draws) or {index into src_clips: array [nwin-1, 256]} in characterize()'s
    eps_seq layout; clips without an entry draw standard-normal rows. Returns one dict per source clip:
    {src_rotations, src_positions, ours_rotations, ours_positions, match}."""
    from .result_bank import ResultBank
    from .source_bank import SourceBank
    src_clips = list(src_clips)
    if not src_clips:
        return []
    dev = "cuda"
    gen_sd = gen_sd or weights.generator_state_dict(1777)
    cvae_sd = cvae_sd or weights.cvae_state_dict(1778)
    stats = _stats_from_raw(raw_stats)
    frames = [preprocess.process_frames(c) for c in src_clips]
    bank = SourceBank(sum(f["pos"].shape[0] for f in frames), len(frames), raw_stats["norm"]["X_mean"],
                      raw_stats["norm"]["X_std"], device=dev)
    ids = [bank.add(f)[0] for f in frames]
    results = ResultBank(bank)
    cha_enc, cha_nm = _character_db(cha_clip, raw_stats, gen_sd, cvae_sd, stats, precision, encode_batch)
    sess = CharacterizationSession(gen_sd, cvae_sd, weights.DEFAULT_MODEL_CFG, stats, cha_enc, cha_nm, batch=slots,
                                   device=dev, precision=precision, match_tensor_cores=False, lanes=lanes,
                                   with_cm_path=with_cm_path, admission=True, source_bank=bank, result_bank=results)
    sess.capture()
    eps = None if eps_seqs is None else {ids[i]: e for i, e in eps_seqs.items()}
    out = sess.serve(ids, eps=eps)
    return [out[c] for c in ids]
