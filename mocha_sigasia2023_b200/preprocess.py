"""Host-side clip ingestion: the reference's `process_data` (preprocess/generate_database.py:86-188)
restated for the inference driver's call (window=60, window_step=1, divide=True, mirror=False).

This is one-off per-clip set-up work with SciPy filters (SURVEY §2 row 12: out of scope for kernels,
"next" row f3); it runs on the host in float64 exactly like the reference and feeds the GPU window
feature extraction in features.py. Euler order and units follow motion/bvh.py (degrees, cm)."""
from __future__ import annotations

import numpy as np
import scipy.ndimage as ndimage
import scipy.signal as signal


# --- minimal float64 quaternion helpers ([w,x,y,z]) used only by this set-up stage ----------------
def _qmul(a, b):
    aw, ax, ay, az = a[..., 0], a[..., 1], a[..., 2], a[..., 3]
    bw, bx, by, bz = b[..., 0], b[..., 1], b[..., 2], b[..., 3]
    return np.stack([bw * aw - bx * ax - by * ay - bz * az,
                     bw * ax + bx * aw - by * az + bz * ay,
                     bw * ay + bx * az + by * aw - bz * ax,
                     bw * az - bx * ay + by * ax + bz * aw], axis=-1)


def _qinv(q):
    return q * np.array([1.0, -1.0, -1.0, -1.0])


def _qrot(q, v):
    u = q[..., 1:]
    t = 2.0 * np.cross(u, v)
    return v + q[..., :1] * t + np.cross(u, t)


def _axis_angle(angle, axis):
    half = angle / 2.0
    return np.concatenate([np.cos(half)[..., None], np.sin(half)[..., None] * axis], axis=-1)


def _from_euler(e, order):
    ax = {"x": np.array([1.0, 0, 0]), "y": np.array([0, 1.0, 0]), "z": np.array([0, 0, 1.0])}
    return _qmul(_axis_angle(e[..., 0], ax[order[0]]),
                 _qmul(_axis_angle(e[..., 1], ax[order[1]]), _axis_angle(e[..., 2], ax[order[2]])))


def _unroll(q):
    out = q.copy()
    for i in range(1, len(q)):
        flip = (out[i] * out[i - 1]).sum(-1) < 0.0
        out[i][flip] = -out[i][flip]
    return out


def _fk(lrot, lpos, parents):
    gr, gp = [lrot[:, 0]], [lpos[:, 0]]
    for j in range(1, len(parents)):
        p = parents[j]
        gp.append(_qrot(gr[p], lpos[:, j]) + gp[p])
        gr.append(_qmul(gr[p], lrot[:, j]))
    return np.stack(gr, axis=1), np.stack(gp, axis=1)


def _fk_vel(lrot, lpos, lvel, lang, parents):
    gr, gp, gv, ga = [lrot[:, 0]], [lpos[:, 0]], [lvel[:, 0]], [lang[:, 0]]
    for j in range(1, len(parents)):
        p = parents[j]
        rp = _qrot(gr[p], lpos[:, j])
        gp.append(rp + gp[p])
        gr.append(_qmul(gr[p], lrot[:, j]))
        gv.append(_qrot(gr[p], lvel[:, j]) + np.cross(ga[p], rp) + gv[p])
        ga.append(_qrot(gr[p], lang[:, j]) + ga[p])
    return np.stack(gr, 1), np.stack(gp, 1), np.stack(gv, 1), np.stack(ga, 1)


def _log(q, eps=1e-5):
    ln = np.sqrt((q[..., 1:] ** 2).sum(-1))[..., None]
    with np.errstate(invalid="ignore", divide="ignore"):
        half = np.where(ln < eps, np.ones_like(ln), np.arctan2(ln, q[..., :1]) / ln)
    return half * q[..., 1:]


def _abs(q):
    return np.where(q[..., :1] > 0.0, q, -q)


def _central_diff(x):
    v = np.empty_like(x)
    v[1:-1] = 0.5 * (x[2:] - x[1:-1]) * 60.0 + 0.5 * (x[1:-1] - x[:-2]) * 60.0
    v[0] = v[1] - (v[3] - v[2])
    v[-1] = v[-2] + (v[-2] - v[-3])
    return v


def _angular_velocity(rot):
    w = np.zeros(rot.shape[:-1] + (3,))
    w[1:-1] = (0.5 * 2.0 * _log(_abs(_qmul(rot[2:], _qinv(rot[1:-1])))) * 60.0 +
               0.5 * 2.0 * _log(_abs(_qmul(rot[1:-1], _qinv(rot[:-2])))) * 60.0)
    w[0] = w[1] - (w[3] - w[2])
    w[-1] = w[-2] + (w[-2] - w[-3])
    return w


def sliding_windows(x, window, step, zero_pad=False):
    """divide_clip(divide=True) (generate_database.py:57-84): edge windows are padded by repeating
    the first / last pose (or zeros for velocities)."""
    out = []
    for j in range(0, len(x) - window // 4, step):
        s = x[j:j + window]
        if len(s) < window:
            short = window - len(s)
            left = s[:1].repeat(short // 2 + short % 2, axis=0)
            right = s[-1:].repeat(short // 2, axis=0)
            if zero_pad:
                left = np.zeros_like(left)
                right = np.zeros_like(right)
            s = np.concatenate([left, s, right], axis=0)
        out.append(s)
    return np.stack(out)


def process_frames(clip: dict) -> dict:
    """The per-frame half of process_clip: float32 pos/vel/rot/ang [F, 25, 3|4], uint8 contacts [F, 2], the bone
    parents and names. Its arrays are 62x smaller than the windows of a 240-frame clip; SourceBank keeps them on the
    device and builds the windows there."""
    names = list(clip["names"])
    parents = np.asarray(clip["parents"])
    positions = np.asarray(clip["positions"], dtype=np.float64) * 0.01            # cm -> m (:91)
    rotations = _unroll(_from_euler(np.radians(np.asarray(clip["rotations"], dtype=np.float64)), clip["order"]))
    grot, gpos = _fk(rotations, positions, parents)
    spine2, hips = names.index("Spine2"), names.index("Hips")
    del hips
    root_pos = np.array([1.0, 0.0, 1.0]) * gpos[:, spine2:spine2 + 1]             # :107-108
    root_pos = signal.savgol_filter(root_pos, 15, 3, axis=0, mode="interp")
    sl, sr = names.index("LeftShoulder"), names.index("RightShoulder")
    hl, hr = names.index("LeftUpLeg"), names.index("RightUpLeg")
    across = (gpos[:, sl:sl + 1] - gpos[:, sr:sr + 1]) + (gpos[:, hl:hl + 1] - gpos[:, hr:hr + 1])
    root_dir = np.array([1.0, 0.0, 1.0]) * np.cross(across, np.array([0, 1, 0]))
    root_dir = root_dir / np.sqrt((root_dir ** 2).sum(-1))[..., None]
    root_dir = signal.savgol_filter(root_dir, 31, 3, axis=0, mode="interp")
    root_dir = root_dir / np.sqrt((root_dir ** 2).sum(-1)[..., None])
    fwd = np.array([0.0, 0.0, 1.0])
    between = np.concatenate([                                                    # quat.between (:143-147)
        np.sqrt((fwd * fwd).sum() * (root_dir * root_dir).sum(-1))[..., None] + (fwd * root_dir).sum(-1)[..., None],
        np.cross(np.broadcast_to(fwd, root_dir.shape), root_dir)], axis=-1)
    root_rot = between / (np.sqrt((between ** 2).sum(-1))[..., None] + 1e-8)      # quat.normalize
    positions[:, 0:1] = _qrot(_qinv(root_rot), positions[:, 0:1] - root_pos)      # :127-128
    rotations[:, 0:1] = _qmul(_qinv(root_rot), rotations[:, 0:1])
    positions = np.concatenate([root_pos, positions], axis=1)
    rotations = np.concatenate([root_rot, rotations], axis=1)
    bone_parents = np.concatenate([[-1], parents + 1])
    bone_names = ["Root"] + names
    velocities = _central_diff(positions)                                         # :138-143
    angular = _angular_velocity(rotations)                                        # :146-151
    _, _, gvel, _ = _fk_vel(rotations, positions, velocities, angular, bone_parents)
    toes = np.array([bone_names.index("LeftToeBase"), bone_names.index("RightToeBase")])
    contacts = np.sqrt((gvel[:, toes] ** 2).sum(-1)) < 0.5                        # :162-171
    for ci in range(contacts.shape[1]):
        contacts[:, ci] = ndimage.median_filter(contacts[:, ci], size=6, mode="nearest")
    return {"pos": positions.astype(np.float32), "vel": velocities.astype(np.float32), "rot": rotations.astype(np.float32),
            "ang": angular.astype(np.float32), "contacts": contacts.astype(np.uint8), "parents": bone_parents,
            "names": bone_names}


def frame_windows(frames: dict, window: int = 60, window_step: int = 1) -> dict:
    """process_frames' arrays cut into process_clip's windows (the float32 cast commutes with the windowing)."""
    return {
        "pos": sliding_windows(frames["pos"], window, window_step),
        "vel": sliding_windows(frames["vel"], window, window_step, zero_pad=True),
        "rot": sliding_windows(frames["rot"], window, window_step),
        "ang": sliding_windows(frames["ang"], window, window_step, zero_pad=True),
        "contacts": sliding_windows(frames["contacts"], window, window_step),
        "parents": frames["parents"],
        "names": frames["names"],
    }


def process_clip(clip: dict, window: int = 60, window_step: int = 1) -> dict:
    """Returns float32 window arrays pos/vel/rot/ang [nwin, window, 25, 3|4] and uint8 contacts
    [nwin, window, 2], exactly what the driver builds at test_fullframework.py:126-139."""
    return frame_windows(process_frames(clip), window, window_step)
