"""Synthetic workload assembly shared by bench.py, __graft_entry__.smoke() and the GPU tests:
random-init weights, synthetic normalisation tables, a character feature DB produced by the CUDA
encoder, and per-step host inputs of the shapes the reference driver feeds its hot loop."""
from __future__ import annotations

import numpy as np
import torch

from . import synthetic, weights
from .session import CharacterizationSession, NormStats


def driver_stats(seed: int = 7) -> NormStats:
    """Apply the driver's std /= std_weight (test_fullframework.py:89-92) to the synthetic tables."""
    raw = synthetic.make_norm_stats(seed)
    w = raw["cvae_norm"]["std_weight"]
    return NormStats(
        Y_mean=raw["norm"]["Y_mean"][1:], Y_std=raw["norm"]["Y_std"][1:],
        cnt_mean=raw["cnt_norm"]["mean"], cnt_std=raw["cnt_norm"]["std"] / w,
        src_cnt_mean=raw["cvae_norm"]["src_cnt_mean"], src_cnt_std=raw["cvae_norm"]["src_cnt_std"] / w,
        cha_encoded_mean=raw["cvae_norm"]["cha_encoded_mean"], cha_encoded_std=raw["cvae_norm"]["cha_encoded_std"] / w)


def stats_as_dict(s: NormStats) -> dict:
    return {k: np.asarray(getattr(s, k), dtype=np.float32) for k in (
        "Y_mean", "Y_std", "cnt_mean", "cnt_std", "src_cnt_mean", "src_cnt_std", "cha_encoded_mean", "cha_encoded_std")}


def pose_windows(n: int, seed: int) -> np.ndarray:
    """Normalised pose windows [n,60,24,15] (what the driver feeds mot_embedding, :186-190):
    temporally smooth so consecutive windows of a clip look like a sliding window."""
    rng = np.random.default_rng(seed)
    base = rng.standard_normal((n, 1, 24, 15)).astype(np.float32)
    t = np.linspace(0, 1, 60, dtype=np.float32)[None, :, None, None]
    f = rng.uniform(0.5, 2.0, size=(n, 1, 24, 15)).astype(np.float32)
    ph = rng.uniform(0, 2 * np.pi, size=(n, 1, 24, 15)).astype(np.float32)
    return (0.6 * base + np.sin(2 * np.pi * f * t + ph)).astype(np.float32)


def step_inputs(B: int, seed: int) -> dict:
    rng = np.random.default_rng(seed)
    return {
        "X": pose_windows(B, seed + 1000),
        "src_hips_vel": rng.standard_normal((B, 60, 3)).astype(np.float32),
        "src_rvel": rng.standard_normal((B, 3)).astype(np.float32),
        "src_rang": (0.5 * rng.standard_normal((B, 3))).astype(np.float32),
        "contacts": (rng.random((B, 2)) < 0.5).astype(np.uint8),
        "eps": rng.standard_normal((B, 256)).astype(np.float32),
    }


def build_session(batch: int, n_db: int = 385, precision: str = "fp32", device="cuda", seed: int = 0,
                  with_cm_path: bool = False, match_tensor_cores=None, gen_seed: int = 1777, cvae_seed: int = 1778,
                  db_precision: str = "fp32", db_batch: int = 64, lanes: int = 1, admission: bool = False,
                  source_bank=None, result_bank=None):
    """Session on random-init weights with a character DB of n_db encoded synthetic windows
    (n_db = 385 is what a 400-frame character clip yields, SURVEY §8d config 1). The DB comes from the
    feature-DB builder (feature_db.build_feature_db: same CUDA encoder, matcher layout)."""
    from . import feature_db
    from .balltree import BallTree
    gen_sd = weights.generator_state_dict(gen_seed)
    cvae_sd = weights.cvae_state_dict(cvae_seed)
    stats = driver_stats()
    cha_X = pose_windows(n_db, seed + 5000)
    fdb = feature_db.build_feature_db(gen_sd, weights.DEFAULT_MODEL_CFG, stats.cnt_mean, stats.cnt_std, cha_X,
                                      batch=db_batch, precision=db_precision, device=device)
    sess = CharacterizationSession(gen_sd, cvae_sd, weights.DEFAULT_MODEL_CFG, stats, fdb.encoded,
                                   BallTree.from_feature_db(fdb, device=device, use_tensor_cores=match_tensor_cores),
                                   batch=batch, device=device, precision=precision, with_cm_path=with_cm_path,
                                   match_tensor_cores=match_tensor_cores, lanes=lanes, admission=admission,
                                   source_bank=source_bank, result_bank=result_bank)
    sess.feature_db = fdb
    return sess, gen_sd, cvae_sd, stats
