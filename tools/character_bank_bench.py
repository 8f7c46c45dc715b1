"""Cost and benefit of the character bank (CharacterizationSession(..., characters=CharacterBank)) at the bench
configuration of result_bank_bench.py (128 slots, bf16, automatic matcher choice, one CUDA graph, CUDA-event timing
after warm-up), in one process:

  step  device step of four bank sessions, alternating rounds, medians. Each round starts every slot on one of the
        128 longest clips (untimed), slot b on character b % n_chars:
          A  one character of 385 rows through the existing path (no characters=),
          B  the same character as a one-character CharacterBank,
          C  8 characters x 385 rows (3,080 rows: split-K coarse pass),
          D  32 characters x 385 rows (12,320 rows: persistent coarse pass).
  prof  torch.profiler pass per arm (20 graph frames): device time of the matcher kernels and slot_segments_kernel,
        and from the trace, per frame, how long the join after the match side stream waits on the matcher: the end of
        the frame's last matcher kernel minus the end of the last other kernel before seed_rows_kernel (0 = the
        matcher finished first).
  serve 1,024 mixed-length clips (the seeded set of source_bank_bench.py) spread over 8 characters (clip i: i % 8):
        (i) one session with the 8-character bank, (ii) 8 single-character sessions served one after another.
        Useful frames/s, frames, slot occupancy; 3 alternating runs after a warm-up, medians.
  bench.py's result line from the same process tree, to show the default step is untouched.

    python tools/character_bank_bench.py --out DIR [--steps 150 --rounds 5 --clips 1024]

writes DIR/character_bank_bench.json. Needs an sm_100 GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

MATCH_KERNELS = ("match_exact_tile", "topk_rows", "match_rerank", "splitk_reduce", "MatchEpi", "slot_segments")


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="output directory (character_bank_bench.json)")
    ap.add_argument("--clips", type=int, default=1024, help="clips of the serving runs")
    ap.add_argument("--slots", type=int, default=128)
    ap.add_argument("--db-rows", type=int, default=385, help="rows per character")
    ap.add_argument("--steps", type=int, default=150, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--min-win", type=int, default=30)
    ap.add_argument("--max-win", type=int, default=225)
    ap.add_argument("--serve-chars", type=int, default=8)
    ap.add_argument("--seed", type=int, default=2023)
    ap.add_argument("--no-bench-line", action="store_true", help="skip bench.py's line")
    args = ap.parse_args()

    import torch
    from admission_bench import gpu_info
    from mocha_sigasia2023_b200 import _lib, feature_db, preprocess, synthetic, weights, workload
    from mocha_sigasia2023_b200.balltree import BallTree
    from mocha_sigasia2023_b200.character_bank import CharacterBank
    from mocha_sigasia2023_b200.result_bank import ResultBank, serving_schedule
    from mocha_sigasia2023_b200.session import CharacterizationSession
    from mocha_sigasia2023_b200.source_bank import SourceBank
    if not torch.cuda.is_available():
        raise SystemExit("character_bank_bench needs a CUDA device (there is no CPU measurement)")
    _lib.check(_lib.load().mocha_check_device(), "mocha_check_device")
    os.makedirs(args.out, exist_ok=True)
    B, K, T, R = args.slots, args.steps, 60, args.db_rows
    dev = torch.device("cuda")
    info = gpu_info(torch)
    rng = np.random.default_rng(args.seed)
    norm = synthetic.make_norm_stats(7)["norm"]

    nwins = rng.integers(args.min_win, args.max_win + 1, size=args.clips)
    frames = [preprocess.process_frames(synthetic.make_clip(int(n) + T // 4, seed=10_000 + i)) for i, n in enumerate(nwins)]
    bank = SourceBank(sum(f["pos"].shape[0] for f in frames), args.clips, norm["X_mean"], norm["X_std"])
    for f, n in zip(frames, nwins):
        assert bank.add(f)[1] == n
    rb = ResultBank(bank)

    gen_sd, cvae_sd = weights.generator_state_dict(1777), weights.cvae_state_dict(1778)
    stats = workload.driver_stats()
    cfg = weights.DEFAULT_MODEL_CFG
    # character c: R encoded synthetic windows; character 0 is workload.build_session's DB (seed 0)
    fdbs = [feature_db.build_feature_db(gen_sd, cfg, stats.cnt_mean, stats.cnt_std, workload.pose_windows(R, 5000 + c),
                                        batch=64, device=dev) for c in range(32)]
    common = dict(batch=B, device=dev, precision="bf16", match_tensor_cores=None, admission=True, source_bank=bank)

    def single(c, results=None):
        return CharacterizationSession(gen_sd, cvae_sd, cfg, stats, fdbs[c].encoded,
                                       BallTree.from_feature_db(fdbs[c], device=dev), result_bank=results, **common)

    def banked(n, results=None):
        chars = CharacterBank.from_feature_dbs(fdbs[:n])
        return CharacterizationSession(gen_sd, cvae_sd, cfg, stats, None, None, characters=chars, result_bank=results,
                                       **common)

    arms = {"A_single_existing_path": (single(0), 0), "B_bank_1x385": (banked(1), 1), "C_bank_8x385": (banked(8), 8),
            "D_bank_32x385": (banked(32), 32)}
    P = 4
    eps_pool = [torch.from_numpy(workload.step_inputs(B, seed=i)["eps"]).to(dev) for i in range(P)]
    zeros = torch.zeros((B,), dtype=torch.uint8, device=dev)
    ones = torch.ones((B,), dtype=torch.uint8, device=dev)
    longest = torch.from_numpy(np.argsort(-nwins)[:B].astype(np.int32)).to(dev)

    def restart(sess, n):
        sess.clip.copy_(longest); sess.start.copy_(ones); sess.eps.copy_(eps_pool[0])
        if n:
            sess.character.copy_(torch.arange(B, dtype=torch.int32, device=dev) % n)
        sess.step_device()
        sess.start.copy_(zeros)

    for sess, n in arms.values():
        sess.capture()
        restart(sess, n)
        for i in range(args.warmup):
            sess.eps.copy_(eps_pool[i % P]); sess.step_device()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(sess, n):
        restart(sess, n)
        e0.record()
        for i in range(K):
            sess.eps.copy_(eps_pool[i % P])
            sess.step_device()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / K

    rounds = {k: [] for k in arms}
    for r in range(args.rounds):
        for k, (sess, n) in arms.items():
            rounds[k].append(timed(sess, n))
    med = {k: float(np.median(v)) for k, v in rounds.items()}
    matcher = {k: {"rows": int(s.tree.N), "tensor_cores": bool(s._use_tc),
                   "splitk": bool(s._use_tc and s.tree.N <= 8192)} for k, (s, n) in arms.items()}

    # ---- profiler: matcher kernel times and the join's wait on the match side stream ----
    from torch.profiler import ProfilerActivity, profile
    prof_res = {}
    for k, (sess, n) in arms.items():
        restart(sess, n)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(20):
                sess.eps.copy_(eps_pool[i % P]); sess.step_device()
            torch.cuda.synchronize()
        kern = {}
        for ev in prof.key_averages():
            if ev.device_type == torch.autograd.DeviceType.CUDA and any(m in ev.key for m in MATCH_KERNELS):
                kern[ev.key[:140]] = {"calls": ev.count, "device_us_avg": ev.device_time_total / max(ev.count, 1)}
        evs = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                     key=lambda e: e.time_range.start)
        waits, prev = [], 0.0
        for e in evs:
            if "seed_rows_kernel" not in e.name:
                continue
            s0 = e.time_range.start
            win = [x for x in evs if prev < x.time_range.start and x.time_range.end <= s0 and x is not e]
            m_end = max((x.time_range.end for x in win if any(m in x.name for m in MATCH_KERNELS)), default=None)
            o_end = max((x.time_range.end for x in win if not any(m in x.name for m in MATCH_KERNELS)), default=None)
            if m_end is not None and o_end is not None:
                waits.append(max(0.0, m_end - o_end))
            prev = s0
        prof_res[k] = {"kernels": kern, "join_wait_us_median": float(np.median(waits)) if waits else None,
                       "join_wait_us_max": float(np.max(waits)) if waits else None, "frames_seen": len(waits)}
    del arms
    torch.cuda.empty_cache()

    # ---- serving: one 8-character session against 8 single-character sessions one after another ----
    C = args.serve_chars
    char_of = {i: i % C for i in range(args.clips)}
    ids = list(range(args.clips))
    multi = banked(C, rb)
    multi.capture()
    singles = [single(c, rb) for c in range(C)]
    for s in singles:
        s.capture()
    per_char = [[i for i in ids if char_of[i] == c] for c in range(C)]
    useful = int(nwins.sum())
    frames_multi = len(serving_schedule(nwins, B)[0])
    frames_seq = sum(len(serving_schedule(nwins[ids_c], B)[0]) for ids_c in per_char)

    def route_bank():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = multi.serve(ids, characters=char_of)
        return time.perf_counter() - t0, out

    def route_seq():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = {}
        for c, s in enumerate(singles):
            out.update(s.serve(per_char[c]))
        return time.perf_counter() - t0, out

    _, out_bank = route_bank()                            # warm-up
    _, out_seq = route_seq()
    assert all(out_bank[i]["match"].shape == (nwins[i],) and out_seq[i]["match"].shape == (nwins[i],) for i in ids)
    assert all(((out_bank[i]["match"] >= 0) & (out_bank[i]["match"] < R)).all() for i in ids)
    runs_bank, runs_seq = [], []
    for r in range(3):
        runs_bank.append(route_bank()[0])
        runs_seq.append(route_seq()[0])
    wall_bank, wall_seq = float(np.median(runs_bank)), float(np.median(runs_seq))

    bench_line = None
    if not args.no_bench_line:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "50", "--warmup",
                            "10"], capture_output=True, text=True, cwd=ROOT, timeout=1800)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        bench_line = json.loads(lines[-1]) if lines else {"returncode": r.returncode, "stderr": r.stderr[-2000:]}

    res = {
        "gpu": info,
        "config": {"slots": B, "precision": "bf16", "rows_per_character": R, "cuda_graph": True, "timing": "cuda events",
                   "steps_per_round": K, "rounds": args.rounds, "warmup": args.warmup, "seed": args.seed,
                   "match_tensor_cores": "auto"},
        "step_ms": med,
        "step_ms_rounds": rounds,
        "vs_A": {k: med[k] / med["A_single_existing_path"] - 1.0 for k in med},
        "matcher": matcher,
        "profiler": prof_res,
        "profiler_note": "20 graph frames per arm; the split-K coarse pass's K-slice GEMM images run in a tcgen05 GEMM "
                         "kernel shared with other stages and are not listed by name. join_wait_us: end of the frame's "
                         "last matcher kernel minus the end of the last other kernel before seed_rows_kernel",
        "serving": {"clips": args.clips, "characters": C, "window_range": [args.min_win, args.max_win],
                    "useful_frames": useful,
                    "i_one_bank_session": {"frames": frames_multi, "slot_occupancy": useful / (frames_multi * B),
                                           "wall_s_median": wall_bank, "runs": runs_bank,
                                           "useful_frames_per_s": useful / wall_bank},
                    "ii_8_single_sessions_in_turn": {"frames": frames_seq, "slot_occupancy": useful / (frames_seq * B),
                                                     "wall_s_median": wall_seq, "runs": runs_seq,
                                                     "useful_frames_per_s": useful / wall_seq}},
        "bench_py": bench_line,
    }
    path = os.path.join(args.out, "character_bank_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "step_ms", "vs_A", "matcher")}))
    print(json.dumps({k: {kk: v[kk] for kk in ("join_wait_us_median", "join_wait_us_max")} for k, v in prof_res.items()}))
    print(json.dumps(res["serving"]))
    print(json.dumps(bench_line))
    print(path)


if __name__ == "__main__":
    main()
