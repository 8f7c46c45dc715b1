"""Source clip bank: the preprocessed per-frame arrays of many source clips, resident on the device, from which
`mocha_source_windows` builds every slot's pose window, `side` row and contacts inside the captured frame (DESIGN §5b).

A 240-frame clip takes 312 KB as per-frame arrays against 19.4 MB as the 225 windows features.extract materialises.
`add()` preprocesses one clip on the host; `add_raw()` preprocesses a batch of raw clips on the device, straight into
the bank (DESIGN §5d)."""
from __future__ import annotations

import ctypes as C

import numpy as np
import scipy.signal as signal
import torch

from . import _lib, preprocess, skeleton

_FRAME_KEYS = ("pos", "vel", "rot", "ang", "contacts")
# Euler order codes of mocha_ingest_frames
EULER_ORDERS = ("xyz", "xzy", "yxz", "yzx", "zxy", "zyx")
# raw joints the ingestion stage reads, in mocha_ingest_frames' `joints` order
INGEST_JOINTS = ("Spine2", "LeftShoulder", "RightShoulder", "LeftUpLeg", "RightUpLeg", "LeftToeBase", "RightToeBase")
INGEST_MIN_FRAMES = 31      # savgol_filter(root_dir, 31, 3, mode='interp') needs a clip at least that long
_SAVGOL_CACHE: dict = {}


def savgol_tables(wl: int, polyorder: int = 3) -> np.ndarray:
    """process_frames' savgol_filter(x, wl, polyorder, axis=0, mode='interp') as a table, built from scipy itself:
    [the correlation weights ndimage applies (wl) | map of the first wl samples to the first wl // 2 outputs
    (wl // 2, wl) | map of the last wl samples to the last wl // 2 outputs (wl // 2, wl)], float64. ndimage takes its
    symmetric path when the weights are equal within DBL_EPSILON, which the device sum mirrors: checked here."""
    w = signal.savgol_coeffs(wl, polyorder)[::-1]
    h = wl // 2
    if wl % 2 != 1 or np.abs(w[h + 1:] - w[:h][::-1]).max() > np.finfo(np.float64).eps:
        raise _lib.MochaError(f"savgol weights of window {wl} are not symmetric within DBL_EPSILON")
    edge = signal.savgol_filter(np.eye(wl), wl, polyorder, axis=0, mode="interp")
    return np.ascontiguousarray(np.concatenate([w, edge[:h].ravel(), edge[wl - h:].ravel()]), dtype=np.float64)


def _savgol_device(dev) -> tuple:
    key = str(dev)
    if key not in _SAVGOL_CACHE:
        _SAVGOL_CACHE[key] = tuple(torch.from_numpy(savgol_tables(wl)).to(dev) for wl in (15, 31))
    return _SAVGOL_CACHE[key]


class SourceBank:
    def __init__(self, max_frames: int, max_clips: int, X_mean, X_std, window: int = 60, parents=None, device="cuda"):
        """Capacity (frames over all clips, clips) and the normalisation tables X_mean / X_std [J,15] (norm.npz) are
        fixed here. The device tensors are never reallocated: a captured graph holds their pointers."""
        if max_frames <= 0 or max_clips <= 0:
            raise _lib.MochaError("SourceBank needs max_frames > 0 and max_clips > 0")
        dev = torch.device(device)
        self.parents = np.asarray(skeleton.BONE_PARENTS if parents is None else parents, dtype=np.int64)
        J = len(self.parents)
        xm, xs = (np.ascontiguousarray(np.asarray(a, dtype=np.float32)) for a in (X_mean, X_std))
        if xm.shape != (J, 15) or xs.shape != (J, 15):
            raise _lib.MochaError(f"X_mean / X_std must be [{J}, 15], got {xm.shape} / {xs.shape}")
        self.dev, self.J, self.T = dev, J, int(window)
        self.max_frames, self.max_clips = int(max_frames), int(max_clips)
        f32 = dict(dtype=torch.float32, device=dev)
        self.rot = torch.zeros((max_frames, J, 4), **f32)
        self.pos = torch.zeros((max_frames, J, 3), **f32)
        self.vel = torch.zeros((max_frames, J, 3), **f32)
        self.ang = torch.zeros((max_frames, J, 3), **f32)
        self.contacts = torch.zeros((max_frames, 2), dtype=torch.uint8, device=dev)
        self.clip_first = torch.zeros((max_clips,), dtype=torch.int64, device=dev)
        self.clip_frames = torch.zeros((max_clips,), dtype=torch.int32, device=dev)   # 0 = unused entry (idle)
        self.parents_dev = torch.as_tensor(self.parents, dtype=torch.int32).to(dev)
        self.X_mean = torch.from_numpy(xm).to(dev)
        self.X_std = torch.from_numpy(xs).to(dev)
        self.n_clips = 0
        self.n_frames = 0
        self.clip_nwin: list[int] = []      # host copy of each clip's window count
        self.clip_start: list[int] = []     # host copy of clip_first

    def add(self, clip: dict) -> tuple[int, int]:
        """Append one clip: a raw clip dict (motion/bvh.py:load layout; preprocessed with preprocess.process_frames) or
        process_frames' output. The upload is stream-ordered on the current stream. Returns (clip_id, nwin), nwin being
        the clip's window count, F - window // 4."""
        frames = preprocess.process_frames(clip) if "positions" in clip else clip
        F = int(np.asarray(frames["pos"]).shape[0])
        J = self.J
        want = {"pos": (F, J, 3), "vel": (F, J, 3), "rot": (F, J, 4), "ang": (F, J, 3), "contacts": (F, 2)}
        for k, shape in want.items():
            if tuple(np.asarray(frames[k]).shape) != shape:
                raise _lib.MochaError(f"SourceBank.add: {k} must be {shape}, got {np.asarray(frames[k]).shape}")
        if "parents" in frames and not np.array_equal(np.asarray(frames["parents"]), self.parents):
            raise _lib.MochaError("SourceBank.add: the clip's skeleton differs from the bank's")
        nwin = F - self.T // 4
        if nwin < 1:
            raise _lib.MochaError(f"SourceBank.add: a clip needs more than {self.T // 4} frames, got {F}")
        if self.n_clips >= self.max_clips or self.n_frames + F > self.max_frames:
            raise _lib.MochaError(f"SourceBank.add: bank full ({self.n_clips}/{self.max_clips} clips, "
                                  f"{self.n_frames}/{self.max_frames} frames; clip of {F} frames)")
        a, c = self.n_frames, self.n_clips
        for k in _FRAME_KEYS:
            dt = np.uint8 if k == "contacts" else np.float32
            getattr(self, k)[a:a + F].copy_(torch.from_numpy(np.ascontiguousarray(np.asarray(frames[k], dtype=dt))))
        self.clip_first[c:c + 1].copy_(torch.tensor([a], dtype=torch.int64))
        self.clip_frames[c:c + 1].copy_(torch.tensor([F], dtype=torch.int32))
        self.n_frames, self.n_clips = a + F, c + 1
        self.clip_nwin.append(nwin)
        self.clip_start.append(a)
        return c, nwin

    def add_raw(self, clips) -> list:
        """Append a batch of raw clip dicts (motion/bvh.py:load layout), preprocessed on the device by
        mocha_ingest_frames: the rows equal process_frames' arrays (DESIGN §5d). Everything is checked on the host
        first; a bad clip or a batch that does not fit raises MochaError and leaves the bank unchanged. Then one
        host-to-device copy of the raw arrays and clip tables, five launches and the bank tables, stream-ordered on the
        current stream. Returns [(clip_id, nwin)] as add() would, in order."""
        meta = self._check_raw(clips)
        if not meta["F"]:
            return []
        return self._ingest_raw(self._upload_raw(self._pack_raw(clips, meta)), meta)

    def _check_raw(self, clips) -> dict:
        J0 = self.J - 1
        want_parents = self.parents
        Fs, orders, joints = [], [], None
        for n, clip in enumerate(clips):
            rot, pos = np.asarray(clip["rotations"]), np.asarray(clip["positions"])
            F = int(rot.shape[0]) if rot.ndim == 3 else -1
            if rot.shape != (F, J0, 3) or pos.shape != (F, J0, 3):
                raise _lib.MochaError(f"SourceBank.add_raw: clip {n}: rotations / positions must be [F, {J0}, 3], got "
                                      f"{rot.shape} / {pos.shape}")
            if clip["order"] not in EULER_ORDERS:
                raise _lib.MochaError(f"SourceBank.add_raw: clip {n}: unknown Euler order {clip['order']!r}")
            names = list(clip["names"])
            missing = [j for j in INGEST_JOINTS + ("Hips",) if j not in names]
            if missing or len(names) != J0:
                raise _lib.MochaError(f"SourceBank.add_raw: clip {n}: needs {J0} joint names including {missing}")
            par = np.asarray(clip["parents"])
            if par.shape != (J0,) or not np.array_equal(np.concatenate([[-1], par + 1]), want_parents):
                raise _lib.MochaError(f"SourceBank.add_raw: clip {n}: the clip's skeleton differs from the bank's")
            idx = [names.index(j) for j in INGEST_JOINTS]
            if joints is not None and idx != joints:
                raise _lib.MochaError(f"SourceBank.add_raw: clip {n}: joint names in another order than clip 0's")
            joints = idx
            if F < INGEST_MIN_FRAMES or F - self.T // 4 < 1:
                raise _lib.MochaError(f"SourceBank.add_raw: clip {n}: needs at least {max(INGEST_MIN_FRAMES, self.T // 4 + 1)} "
                                      f"frames, got {F}")
            Fs.append(F)
            orders.append(EULER_ORDERS.index(clip["order"]))
        total = sum(Fs)
        if self.n_clips + len(Fs) > self.max_clips or self.n_frames + total > self.max_frames:
            raise _lib.MochaError(f"SourceBank.add_raw: bank full ({self.n_clips}/{self.max_clips} clips, "
                                  f"{self.n_frames}/{self.max_frames} frames; batch of {len(Fs)} clips, {total} frames)")
        first = np.concatenate([[0], np.cumsum(Fs)[:-1]]).astype(np.int64) if Fs else np.zeros(0, np.int64)
        return {"F": Fs, "order": orders, "joints": joints, "first": first, "total": total}

    def _pack_raw(self, clips, meta) -> np.ndarray:
        """One host buffer: rotations and positions fp64 [total, J-1, 3] each, then first int64, frames and order
        int32 (8-byte aligned pieces, viewed on the device after one copy)."""
        N, n, J0 = meta["total"], len(meta["F"]), self.J - 1
        raw = N * J0 * 3 * 8
        buf = np.empty(2 * raw + n * 8 + 2 * ((n * 4 + 7) // 8 * 8), dtype=np.uint8)
        rot = buf[:raw].view(np.float64).reshape(N, J0, 3)
        pos = buf[raw:2 * raw].view(np.float64).reshape(N, J0, 3)
        for clip, a, F in zip(clips, meta["first"], meta["F"]):
            rot[a:a + F] = np.asarray(clip["rotations"], dtype=np.float64)
            pos[a:a + F] = np.asarray(clip["positions"], dtype=np.float64)
        o = 2 * raw
        buf[o:o + n * 8].view(np.int64)[:] = meta["first"]
        o += n * 8
        buf[o:o + n * 4].view(np.int32)[:] = meta["F"]
        o += (n * 4 + 7) // 8 * 8
        buf[o:o + n * 4].view(np.int32)[:] = meta["order"]
        return buf

    def _upload_raw(self, buf: np.ndarray) -> torch.Tensor:
        return torch.from_numpy(buf).to(self.dev)

    def _ingest_raw(self, dbuf: torch.Tensor, meta) -> list:
        N, n, J0, J = meta["total"], len(meta["F"]), self.J - 1, self.J
        raw = N * J0 * 3 * 8
        o = 2 * raw
        first = dbuf[o:o + n * 8].view(torch.int64)
        o += n * 8
        frames = dbuf[o:o + n * 4].view(torch.int32)
        o += (n * 4 + 7) // 8 * 8
        order = dbuf[o:o + n * 4].view(torch.int32)
        lib = _lib.load()
        ws = torch.empty(max(1, int(lib.mocha_ingest_workspace_bytes(N, J))), dtype=torch.uint8, device=self.dev)
        sg15, sg31 = _savgol_device(self.dev)
        parents = (C.c_int32 * J0)(*[int(p) - 1 if p >= 0 else -1 for p in self.parents[1:]])
        joints = (C.c_int32 * 7)(*meta["joints"])
        a, c = self.n_frames, self.n_clips
        _lib.check(lib.mocha_ingest_frames(
            _lib.ptr(dbuf), C.c_void_p(dbuf.data_ptr() + raw), N, _lib.ptr(first), _lib.ptr(frames), _lib.ptr(order), n,
            max(meta["F"]), parents, joints, J, _lib.ptr(sg15), _lib.ptr(sg31), _lib.ptr(self.rot), _lib.ptr(self.pos),
            _lib.ptr(self.vel), _lib.ptr(self.ang), _lib.ptr(self.contacts), self.max_frames, a, _lib.ptr(ws),
            ws.numel(), _lib.stream_ptr()), "mocha_ingest_frames")
        ws.record_stream(torch.cuda.current_stream(self.dev))
        self.clip_first[c:c + n].copy_(torch.from_numpy(meta["first"] + a))
        self.clip_frames[c:c + n].copy_(torch.tensor(meta["F"], dtype=torch.int32))
        out = []
        for k, F in enumerate(meta["F"]):
            nwin = F - self.T // 4
            self.clip_nwin.append(nwin)
            self.clip_start.append(a + int(meta["first"][k]))
            out.append((c + k, nwin))
        self.n_frames, self.n_clips = a + N, c + n
        return out

    def clear(self):
        """Forget every clip (stream-ordered). A slot still holding a cleared id turns idle, or serves the clip that is
        given that id next from its old cursor: start the slots anew after clear()."""
        self.clip_frames.zero_()
        self.n_clips = self.n_frames = 0
        self.clip_nwin, self.clip_start = [], []

    def nbytes(self) -> int:
        """Device memory of the bank arrays and clip tables."""
        return sum(t.numel() * t.element_size() for t in (self.rot, self.pos, self.vel, self.ang, self.contacts,
                                                           self.clip_first, self.clip_frames))

    def windows(self, start, clip, slot_clip, slot_cursor, X, side, contacts):
        """One frame of mocha_source_windows for B slots: start uint8 [B], clip int32 [B] (read where start is set),
        per-slot state slot_clip / slot_cursor int32 [B] (slot_clip -1 = idle) advanced in place; writes X [B,T,J-1,15],
        side [B, >= T*3+6] (unit column stride) and contacts uint8 [B,2]."""
        B = start.shape[0]
        for t, dt in ((start, torch.uint8), (clip, torch.int32), (slot_clip, torch.int32), (slot_cursor, torch.int32)):
            _lib.require_cuda(t)
            if t.dtype != dt or t.shape != (B,):
                raise _lib.MochaError(f"source windows: expected {dt} [{B}], got {t.dtype} {tuple(t.shape)}")
        _lib.require_cuda(X, contacts)
        if X.shape != (B, self.T, self.J - 1, 15) or X.dtype != torch.float32:
            raise _lib.MochaError(f"source windows: X must be float32 [{B}, {self.T}, {self.J - 1}, 15]")
        if contacts.shape != (B, 2) or contacts.dtype != torch.uint8:
            raise _lib.MochaError(f"source windows: contacts must be uint8 [{B}, 2]")
        if (not side.is_cuda or side.dtype != torch.float32 or side.dim() != 2 or side.shape[0] != B
                or side.shape[1] < self.T * 3 + 6 or side.stride(1) != 1):
            raise _lib.MochaError(f"source windows: side must be float32 [{B}, >= {self.T * 3 + 6}] with unit column stride")
        _lib.check(_lib.load().mocha_source_windows(
            _lib.ptr(self.rot), _lib.ptr(self.pos), _lib.ptr(self.vel), _lib.ptr(self.ang), _lib.ptr(self.contacts),
            self.max_frames, _lib.ptr(self.clip_first), _lib.ptr(self.clip_frames), self.max_clips,
            _lib.ptr(self.parents_dev), self.T, self.J, _lib.ptr(self.X_mean), _lib.ptr(self.X_std), _lib.ptr(start),
            _lib.ptr(clip), _lib.ptr(slot_clip), _lib.ptr(slot_cursor), B, _lib.ptr(X), _lib.ptr(side), side.stride(0),
            _lib.ptr(contacts), _lib.stream_ptr()), "mocha_source_windows")
