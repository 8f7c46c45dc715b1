"""Result bank: each served clip's motion recorded on the device, inside the captured frame, and its bvh.save payload
built on the device per finished clip (DESIGN §5c).

`mocha_record_frames` (the last launch of an admission frame) copies each slot's post-IK pose, integrated source root
and matched DB row into record row clip_first[c] + w of the clip c it serves (1,464 B). `mocha_clip_payload` turns the
rows of finished clips into what test_fullframework.py:672-721 hands to bvh.save, in place at the same rows (1,728 B per
window, plus the 8 B matched row). The host downloads finished clips only."""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib

RECORD_BYTES = 1464                     # sizeof(mocha_frame_record)
RECORD_DTYPE = np.dtype([("ik_pos", "f8", (25, 3)), ("ik_rot", "f8", (25, 4)), ("src_root_pos", "f8", (3,)),
                         ("src_root_rot", "f8", (4,)), ("match", "i8")])
assert RECORD_DTYPE.itemsize == RECORD_BYTES
FRAME_OUT_BYTES = C.sizeof(_lib.FrameOut)               # sizeof(mocha_frame_out), one slot's post-process output
PAYLOAD_KEYS = ("src_rotations", "src_positions", "ours_rotations", "ours_positions", "match")


def serving_schedule(nwins, slots: int):
    """First-free-slot FIFO schedule of clips with `nwins` windows each over `slots` slots: each frame, every slot whose
    clip has ended (or that never held one) takes the next clip of the queue, lowest slot first. A clip then runs its
    nwin windows on consecutive frames of that slot.

    Returns (start [frames, slots] uint8, clip [frames, slots] int32 = index into nwins where start is set, else 0,
    placement [len(nwins), 2] int64 = (slot, first frame) of each clip). Clip k's last window is served on frame
    placement[k, 1] + nwins[k] - 1."""
    nwins = np.asarray(nwins, dtype=np.int64)
    if slots <= 0:
        raise _lib.MochaError("serving_schedule needs slots > 0")
    if nwins.ndim != 1 or (nwins < 1).any():
        raise _lib.MochaError("serving_schedule: every clip needs nwin >= 1")
    queue, nxt = len(nwins), 0
    left = np.zeros(slots, dtype=np.int64)
    place = np.zeros((queue, 2), dtype=np.int64)
    start_rows, clip_rows = [], []
    while nxt < queue or left.any():
        row, crow = np.zeros(slots, dtype=np.uint8), np.zeros(slots, dtype=np.int32)
        for s in range(slots):
            if left[s] == 0 and nxt < queue:
                left[s], row[s], crow[s] = nwins[nxt], 1, nxt
                place[nxt] = (s, len(start_rows))
                nxt += 1
        start_rows.append(row)
        clip_rows.append(crow)
        left = np.maximum(left - 1, 0)
    if not start_rows:
        return np.zeros((0, slots), np.uint8), np.zeros((0, slots), np.int32), place
    return np.stack(start_rows), np.stack(clip_rows), place


class ResultBank:
    def __init__(self, source_bank):
        """Record rows, payload rows and per-clip counts for every frame / clip the source bank can hold. Allocated once:
        a captured graph holds their pointers."""
        b = source_bank
        if b is None or not hasattr(b, "clip_first"):
            raise _lib.MochaError("ResultBank needs a SourceBank")
        if b.J != 25:
            raise _lib.MochaError(f"ResultBank records 25-joint skeletons; the source bank has {b.J} joints")
        self.bank = b
        dev, R = b.dev, b.max_frames
        self.records = torch.zeros((R, RECORD_BYTES), dtype=torch.uint8, device=dev)
        self.src_rot = torch.zeros((R, 24, 3), dtype=torch.float32, device=dev)
        self.src_pos = torch.zeros((R, 24, 3), dtype=torch.float32, device=dev)
        self.ours_rot = torch.zeros((R, 24, 3), dtype=torch.float64, device=dev)
        self.ours_pos = torch.zeros((R, 24, 3), dtype=torch.float64, device=dev)
        self.match = torch.zeros((R,), dtype=torch.int64, device=dev)
        self.clip_done = torch.zeros((b.max_clips,), dtype=torch.int32, device=dev)
        # 1 = the payload rows hold the clip's last complete recording (set by mocha_clip_payload, cleared by a new row)
        self.clip_built = torch.zeros((b.max_clips,), dtype=torch.int32, device=dev)

    def payload_arrays(self):
        """The device payload arrays, in PAYLOAD_KEYS order (rows clip_first[c] .. + nwin of clip c)."""
        return self.src_rot, self.src_pos, self.ours_rot, self.ours_pos, self.match

    def _check_ids(self, ids):
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        if ids.size == 0:
            raise _lib.MochaError("result bank: no clip ids")
        bad = ids[(ids < 0) | (ids >= self.bank.n_clips)]
        if bad.size:
            raise _lib.MochaError(f"result bank: clip id {int(bad[0])} not in the bank ({self.bank.n_clips} clips)")
        return ids

    def record(self, out, match_idx, start, slot_clip, slot_count):
        """One frame of mocha_record_frames for B slots: out = the slots' mocha_frame_out rows (uint8 CUDA tensor of
        B * FRAME_OUT_BYTES bytes), match_idx int64 [B, k] (column 0 is recorded), start uint8 [B], slot_clip / slot_count int32
        [B] (slot_count advanced in place)."""
        B = start.shape[0]
        for t, dt in ((start, torch.uint8), (slot_clip, torch.int32), (slot_count, torch.int32)):
            _lib.require_cuda(t)
            if t.dtype != dt or t.shape != (B,):
                raise _lib.MochaError(f"record frames: expected {dt} [{B}], got {t.dtype} {tuple(t.shape)}")
        nb = B * FRAME_OUT_BYTES
        if not out.is_cuda or out.dtype != torch.uint8 or out.numel() != nb or not out.is_contiguous():
            raise _lib.MochaError(f"record frames: out must be the {B} slots' mocha_frame_out rows ({nb} B)")
        if (not match_idx.is_cuda or match_idx.dtype != torch.int64 or match_idx.dim() != 2 or match_idx.shape[0] != B
                or match_idx.stride(1) != 1):
            raise _lib.MochaError(f"record frames: match_idx must be int64 [{B}, k] with unit column stride")
        b = self.bank
        _lib.check(_lib.load().mocha_record_frames(
            _lib.ptr(out), _lib.ptr(match_idx), match_idx.stride(0), _lib.ptr(start), _lib.ptr(slot_clip),
            _lib.ptr(slot_count), B, _lib.ptr(b.clip_first), _lib.ptr(b.clip_frames), b.max_clips, b.T,
            _lib.ptr(self.records), b.max_frames, _lib.ptr(self.clip_done), _lib.ptr(self.clip_built),
            _lib.stream_ptr()), "mocha_record_frames")

    def payload_device(self, ids_dev, n: int, max_nwin: int):
        """mocha_clip_payload for the first n ids of the int32 CUDA tensor ids_dev, on the current stream."""
        b = self.bank
        _lib.check(_lib.load().mocha_clip_payload(
            _lib.ptr(self.records), b.max_frames, _lib.ptr(b.rot), _lib.ptr(b.pos), _lib.ptr(b.clip_first),
            _lib.ptr(b.clip_frames), b.max_clips, _lib.ptr(self.clip_done), _lib.ptr(self.clip_built),
            _lib.ptr(b.parents_dev), b.T, b.J,
            _lib.ptr(ids_dev), n, max_nwin, *(_lib.ptr(t) for t in self.payload_arrays()), _lib.stream_ptr()),
            "mocha_clip_payload")

    def payload(self, clip_ids):
        """Build the payload rows of these clips on the device (stream-ordered on the current stream). Only recorded
        windows are converted; a clip complete at that point is marked built until its next record row."""
        ids = self._check_ids(clip_ids)
        max_nwin = max(self.bank.clip_nwin[int(c)] for c in ids)
        ids_dev = torch.from_numpy(ids.astype(np.int32)).to(self.bank.dev, non_blocking=False)
        for s in range(0, ids.size, 65535):
            self.payload_device(ids_dev[s:], min(65535, ids.size - s), max_nwin)

    def done(self) -> np.ndarray:
        """Recorded windows per clip id of the bank (int32 [n_clips]); a clip is complete when its count is its nwin."""
        return self.clip_done[:self.bank.n_clips].cpu().numpy()

    def read(self, clip_id: int) -> dict:
        """The payload of a complete clip: {src_rotations, src_positions [nwin,24,3] float32, ours_rotations,
        ours_positions [nwin,24,3] float64, match [nwin] int64}, as characterize() returns them. Raises if the clip is
        not complete, or if payload() has not run since its last record row (a clip served again, or never built)."""
        c = int(self._check_ids([clip_id])[0])
        nwin, first = self.bank.clip_nwin[c], self.bank.clip_start[c]
        got, built = (int(v) for v in torch.stack((self.clip_done[c], self.clip_built[c])).tolist())
        if got != nwin:
            raise _lib.MochaError(f"result bank: clip {c} is not complete ({got} of {nwin} windows recorded)")
        if not built:
            raise _lib.MochaError(f"result bank: the payload of clip {c} is not built: call payload() after its last "
                                  "recorded window")
        sl = slice(first, first + nwin)
        return {k: t[sl].cpu().numpy() for k, t in zip(PAYLOAD_KEYS, self.payload_arrays())}

    def records_of(self, clip_id: int) -> np.ndarray:
        """The raw record rows of a clip (structured numpy array [nwin] of RECORD_DTYPE), complete or not."""
        c = int(self._check_ids([clip_id])[0])
        first = self.bank.clip_start[c]
        return self.records[first:first + self.bank.clip_nwin[c]].cpu().numpy().view(RECORD_DTYPE).reshape(-1)

    def clear(self):
        """Forget every count and payload (stream-ordered). Start the slots anew afterwards, as after
        SourceBank.clear()."""
        self.clip_done.zero_()
        self.clip_built.zero_()

    def nbytes(self) -> int:
        """Device memory of the record rows, payload rows and counts."""
        return sum(t.numel() * t.element_size() for t in (self.records, *self.payload_arrays(), self.clip_done,
                                                           self.clip_built))
