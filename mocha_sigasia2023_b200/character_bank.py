"""Character bank: several target characters' feature DBs in one matcher DB, so that one session serves each clip toward
its own character (DESIGN §5e).

Per character, a frame depends on the character DB only: the matcher searches that character's rows, the seed of a
starting clip is the matched row and the second decode reads `encoded[match]`. The normalisation tables are dataset
statistics (test_fullframework.py:64-99), and the CVAE and decoder see the character only through the slot's prev_cha.
So the bank stores every character's rows back to back, and the session matches each slot only against the rows of
its character (mocha_slot_segments + the segmented matchers)."""
from __future__ import annotations

import numpy as np
import torch

from . import _lib
from .balltree import BallTree


def _indexed(dev: torch.device) -> torch.device:
    """"cuda" -> "cuda:<current device>" (tensors always carry the index)."""
    if dev.type == "cuda" and dev.index is None and torch.cuda.is_available():
        return torch.device("cuda", torch.cuda.current_device())
    return dev


class CharacterBank:
    """An immutable bank of characters, built once. Character c owns the global rows
    char_first[c] .. char_first[c] + char_rows[c] - 1 of `encoded` [N, 90, 256] and of the BallTree `tree` over the
    [N, 23040] matcher rows. The bf16 rows of the tensor-core matcher are packed around the mean of all N rows (the
    tree's `_ensure_bf16`), so one centre serves every query.

    Adding a character means building a new bank and a new session: a session's captured graph, workspaces and matcher
    choice are fixed for the bank it was built with."""

    def __init__(self, encoded_list, cnt_nm_list, device=None, use_tensor_cores=None):
        """encoded_list / cnt_nm_list: one [n_c, 90, 256] / [n_c, 23040] pair per character (what
        characterize._character_db returns, or a FeatureDB's `encoded` / `rows32`), all on one device."""
        enc, nm = list(encoded_list), list(cnt_nm_list)
        if not enc or len(enc) != len(nm):
            raise _lib.MochaError(f"CharacterBank needs one (encoded, cnt_nm) pair per character, got {len(enc)} "
                                  f"encoded and {len(nm)} cnt_nm tables")
        for c, (e, r) in enumerate(zip(enc, nm)):
            if not isinstance(e, torch.Tensor) or not isinstance(r, torch.Tensor):
                raise _lib.MochaError(f"CharacterBank: character {c} is not a pair of tensors")
        shape0, D = tuple(enc[0].shape[1:]), (nm[0].shape[-1] if nm[0].dim() else -1)
        rows = []
        for c, (e, r) in enumerate(zip(enc, nm)):
            if e.dim() != 3 or r.dim() != 2 or e.shape[0] != r.shape[0]:
                raise _lib.MochaError(f"CharacterBank: character {c} needs encoded [n, T, D] and cnt_nm [n, T*D] with the "
                                      f"same n, got {tuple(e.shape)} and {tuple(r.shape)}")
            if e.shape[0] == 0:
                raise _lib.MochaError(f"CharacterBank: character {c} has no rows")
            if tuple(e.shape[1:]) != shape0 or r.shape[1] != D:
                raise _lib.MochaError(f"CharacterBank: character {c} has rows {tuple(e.shape[1:])} / {r.shape[1]}, "
                                      f"character 0 has {shape0} / {D}")
            rows.append(int(e.shape[0]))
        devs = {t.device for t in enc + nm}
        if device is not None:
            devs.add(_indexed(torch.device(device)))
        if len(devs) != 1:
            raise _lib.MochaError(f"CharacterBank: the characters' tables are on several devices {sorted(map(str, devs))}")
        dev = devs.pop()
        if dev.type != "cuda":
            raise _lib.MochaError("CharacterBank holds CUDA tensors (no CPU fallback)")
        self.dev = dev
        self.encoded = torch.cat([e.to(torch.float32) for e in enc]).contiguous()
        self.tree = BallTree(torch.cat([r.to(torch.float32) for r in nm]).contiguous(), device=dev,
                             use_tensor_cores=use_tensor_cores)
        self.N, self.D = self.tree.N, self.tree.D
        self.n_chars = len(rows)
        self.char_rows_host = np.asarray(rows, dtype=np.int32)
        self.char_first_host = np.concatenate([[0], np.cumsum(rows)[:-1]]).astype(np.int64)
        self.char_first = torch.from_numpy(self.char_first_host).to(dev)
        self.char_rows = torch.from_numpy(self.char_rows_host).to(dev)

    @classmethod
    def from_feature_dbs(cls, fdbs, **kwargs):
        """Bank of feature_db.FeatureDBs, one per character (built with keep_fp32=True and keep_encoded=True)."""
        fdbs = list(fdbs)
        for c, f in enumerate(fdbs):
            if f.rows32 is None or f.encoded is None:
                raise _lib.MochaError(f"CharacterBank.from_feature_dbs: FeatureDB {c} needs its fp32 rows and encoded "
                                      "features (keep_fp32=True, keep_encoded=True)")
        return cls([f.encoded for f in fdbs], [f.rows32 for f in fdbs], **kwargs)

    def rows(self, c: int) -> int:
        """Rows of character c."""
        return int(self.char_rows_host[self.check_ids([c])[0]])

    def check_ids(self, ids) -> np.ndarray:
        """The character ids as int64, or MochaError for one outside [0, n_chars)."""
        ids = np.asarray(ids, dtype=np.int64).reshape(-1)
        bad = ids[(ids < 0) | (ids >= self.n_chars)]
        if bad.size:
            raise _lib.MochaError(f"character id {int(bad[0])} not in the bank ({self.n_chars} characters)")
        return ids

    def nbytes(self) -> int:
        """Device memory of the encoded rows, the matcher rows (and their bf16 copy once packed) and the tables."""
        t = self.tree
        parts = [self.encoded, t.data, self.char_first, self.char_rows, t._db16, t._norm, t.center]
        return sum(p.numel() * p.element_size() for p in parts if p is not None)
