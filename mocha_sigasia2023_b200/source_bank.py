"""Source clip bank: the preprocessed per-frame arrays of many source clips, resident on the device, from which
`mocha_source_windows` builds every slot's pose window, `side` row and contacts inside the captured frame (DESIGN §5b).

A 240-frame clip takes 312 KB as per-frame arrays against 19.4 MB as the 225 windows features.extract materialises."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib, preprocess, skeleton

_FRAME_KEYS = ("pos", "vel", "rot", "ang", "contacts")


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
