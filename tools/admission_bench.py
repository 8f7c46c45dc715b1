"""Cost and benefit of clip admission (CharacterizationSession(admission=True)) at the bench configuration
(128 clips, bf16, 385-row DB, one CUDA graph, CUDA-event timing after warm-up), all in one process:

  A  default session, steady-state step
  B  admission session, all-zero start row
  C  admission session, about one start per frame (each slot starts with probability 1/225 per frame, seeded)

timed in alternating rounds (A, B, C, A, B, C, ...); then a seeded mixed-length serving run (clips of 30..225 frames
through the 128 slots of the admission session, a free slot takes the next clip on the next frame): useful frames/s
(frames of real clips only) and slot occupancy; for comparison the occupancy of a wave schedule of the same clips
(128 at a time, each wave lasting its longest clip), computed on the host: a count, not a time. A torch.profiler pass of
a few A / B replays lists the per-kernel device times of the two additions (seed copy, masked post-process).

    python tools/admission_bench.py --out DIR [--steps 200 --rounds 5 --clips 1024]

writes DIR/admission_bench.json. Needs an sm_100 GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info(torch):
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        pl, clk = (x.strip() for x in r.stdout.strip().split(","))
        info.update(power_limit_w=float(pl), max_sm_clock_mhz=float(clk))
    except Exception as e:             # the numbers are still worth having; say why the card data is missing
        info["power_limit_error"] = repr(e)
    return info


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="output directory (admission_bench.json)")
    ap.add_argument("--clips", type=int, default=1024, help="clips of the serving run")
    ap.add_argument("--slots", type=int, default=128)
    ap.add_argument("--db-rows", type=int, default=385)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--min-len", type=int, default=30)
    ap.add_argument("--max-len", type=int, default=225)
    ap.add_argument("--seed", type=int, default=2023)
    args = ap.parse_args()

    import torch
    from mocha_sigasia2023_b200 import _lib, workload
    if not torch.cuda.is_available():
        raise SystemExit("admission_bench needs a CUDA device (there is no CPU measurement)")
    _lib.check(_lib.load().mocha_check_device(), "mocha_check_device")
    os.makedirs(args.out, exist_ok=True)
    B, K = args.slots, args.steps
    dev = torch.device("cuda")
    rng = np.random.default_rng(args.seed)

    # ---- sessions (same weights / DB / inputs as bench.py) ----
    sess_a, *_ = workload.build_session(B, n_db=args.db_rows, precision="bf16", device=dev, match_tensor_cores=None)
    sess_b, *_ = workload.build_session(B, n_db=args.db_rows, precision="bf16", device=dev, match_tensor_cores=None,
                                        admission=True)
    P = 4
    pool = []
    for i in range(P):
        h = workload.step_inputs(B, seed=i)
        side = np.concatenate([h["src_hips_vel"].reshape(B, -1), h["src_rvel"], h["src_rang"]], axis=1)
        pool.append({"X": torch.from_numpy(h["X"]).to(dev), "side": torch.from_numpy(side).to(dev),
                     "contacts": torch.from_numpy(h["contacts"]).to(dev), "eps": torch.from_numpy(h["eps"]).to(dev)})

    def load(sess, i):
        d = pool[i % P]
        sess.X.copy_(d["X"]); sess.side.copy_(d["side"]); sess.contacts.copy_(d["contacts"]); sess.eps.copy_(d["eps"])

    zeros = torch.zeros((B,), dtype=torch.uint8, device=dev)
    c_rows = torch.from_numpy((rng.random((K, B)) < 1.0 / args.max_len).astype(np.uint8)).to(dev)   # arm C start rows
    ones = torch.ones((B,), dtype=torch.uint8, device=dev)

    # first frames: the default session's init frame, every admission slot started once; then the graphs
    load(sess_a, 0); sess_a.step_device()
    sess_b.capture()
    load(sess_b, 0); sess_b.start.copy_(ones); sess_b.step_device()
    sess_a.capture()
    for i in range(args.warmup):
        load(sess_a, i); sess_a.step_device()
        load(sess_b, i); sess_b.start.copy_(zeros); sess_b.step_device()
    torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(arm):
        sess = sess_a if arm == "A" else sess_b
        e0.record()
        for i in range(K):
            load(sess, i)
            if arm == "B":
                sess.start.copy_(zeros)
            elif arm == "C":
                sess.start.copy_(c_rows[i])
            sess.step_device()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / K

    rounds = {"A": [], "B": [], "C": []}
    for r in range(args.rounds):
        for arm in ("A", "B", "C"):
            rounds[arm].append(timed(arm))
    med = {k: float(np.median(v)) for k, v in rounds.items()}

    # ---- kernel times of the two additions (profiler on, separate from the timed rounds) ----
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for arm in ("A", "B", "C"):
        sess = sess_a if arm == "A" else sess_b
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(20):
                load(sess, i)
                if arm != "A":
                    sess.start.copy_(zeros if arm == "B" else c_rows[i])
                sess.step_device()
            torch.cuda.synchronize()
        per, total = {}, 0.0
        for ev in prof.key_averages():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            total += ev.device_time_total
            if any(s in ev.key for s in ("seed_rows", "post_frame")):
                per[ev.key[:120]] = {"calls": ev.count, "device_us_avg": ev.device_time_total / max(ev.count, 1)}
        kernels[arm] = {"kernel_us_per_step_sum": total / 20, "kernels": per}

    # ---- serving run: mixed-length clips through the admission session's slots ----
    lengths = rng.integers(args.min_len, args.max_len + 1, size=args.clips)
    queue, slot_left, start_rows = list(range(args.clips)), np.zeros(B, dtype=np.int64), []
    busy = 0
    while queue or slot_left.any():
        row = np.zeros(B, dtype=np.uint8)
        for s in range(B):
            if slot_left[s] == 0 and queue:
                slot_left[s] = lengths[queue.pop(0)]
                row[s] = 1
        busy += int((slot_left > 0).sum())
        start_rows.append(row)
        slot_left = np.maximum(slot_left - 1, 0)
    frames = len(start_rows)
    starts_dev = torch.from_numpy(np.stack(start_rows)).to(dev)
    useful = int(lengths.sum())
    assert busy == useful
    torch.cuda.synchronize()
    e0.record()
    for f in range(frames):
        load(sess_b, f)
        sess_b.start.copy_(starts_dev[f])
        sess_b.step_device()
    e1.record()
    torch.cuda.synchronize()
    serve_ms = e0.elapsed_time(e1)
    waves = [lengths[i:i + B] for i in range(0, args.clips, B)]
    wave_frames = int(sum(w.max() for w in waves))

    res = {
        "gpu": gpu_info(torch),
        "config": {"slots": B, "precision": "bf16", "db_rows": args.db_rows, "cuda_graph": True, "timing": "cuda events",
                   "steps_per_round": K, "rounds": args.rounds, "warmup": args.warmup, "seed": args.seed,
                   "arm_C_start_probability_per_slot_frame": 1.0 / args.max_len,
                   "arm_C_mean_starts_per_frame": float(c_rows.float().sum(1).mean().item())},
        "step_ms": {"A_default": med["A"], "B_admission_no_starts": med["B"], "C_admission_starts": med["C"]},
        "step_ms_rounds": rounds,
        "overhead_vs_A": {"B": med["B"] / med["A"] - 1.0, "C": med["C"] / med["A"] - 1.0},
        "profiler_kernels_20_steps": kernels,
        "serving": {"clips": args.clips, "length_range": [args.min_len, args.max_len], "useful_frames": useful,
                    "frames": frames, "ms": serve_ms, "useful_frames_per_s": useful * 1e3 / serve_ms,
                    "slot_occupancy": useful / (frames * B),
                    "wave_schedule_count_not_timed": {"frames": wave_frames, "slot_occupancy": useful / (wave_frames * B)}},
    }
    path = os.path.join(args.out, "admission_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "step_ms", "overhead_vs_A")}))
    print(json.dumps(res["serving"]))
    print(path)


if __name__ == "__main__":
    main()
