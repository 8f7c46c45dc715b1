"""Cost and benefit of the source clip bank (CharacterizationSession(..., admission=True, source_bank=bank)) at the
bench configuration (128 slots, bf16, 385-row DB, one CUDA graph, CUDA-event timing after warm-up), in one process:

  A  admission session whose X / side / contacts are copied device to device from a pool each step (admission_bench.py)
  B  bank session: mocha_source_windows builds every slot's inputs inside the graph; only start / clip are copied
  C  pipelined end to end from pinned host buffers (submit / collect): A's session sending X / side / contacts / eps /
     start against B's sending start / clip / eps; frames/s and the host-to-device bytes per step (computed)

A and B alternate within rounds, then C's two sides alternate. A torch.profiler pass gives the new kernel's device
time. Finally a seeded serving run of mixed-length synthetic clips through the bank: host preprocessing time
(process_frames, reported apart), the bank's device memory against the memory of the clips' X windows, useful frames/s.

    python tools/source_bank_bench.py --out DIR [--steps 200 --rounds 5 --clips 1024]

writes DIR/source_bank_bench.json. Needs an sm_100 GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="output directory (source_bank_bench.json)")
    ap.add_argument("--clips", type=int, default=1024, help="clips of the serving run")
    ap.add_argument("--slots", type=int, default=128)
    ap.add_argument("--db-rows", type=int, default=385)
    ap.add_argument("--steps", type=int, default=200, help="timed steps per arm and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--min-win", type=int, default=30, help="fewest windows of a serving clip")
    ap.add_argument("--max-win", type=int, default=225, help="most windows of a serving clip")
    ap.add_argument("--seed", type=int, default=2023)
    args = ap.parse_args()

    import torch
    from admission_bench import gpu_info
    from mocha_sigasia2023_b200 import _lib, preprocess, synthetic, workload
    from mocha_sigasia2023_b200.result_bank import serving_schedule
    from mocha_sigasia2023_b200.source_bank import SourceBank
    if not torch.cuda.is_available():
        raise SystemExit("source_bank_bench needs a CUDA device (there is no CPU measurement)")
    _lib.check(_lib.load().mocha_check_device(), "mocha_check_device")
    os.makedirs(args.out, exist_ok=True)
    B, K, T = args.slots, args.steps, 60
    dev = torch.device("cuda")
    rng = np.random.default_rng(args.seed)
    norm = synthetic.make_norm_stats(7)["norm"]

    # ---- serving clips: preprocessed on the host (timed apart), all in one bank ----
    nwins = rng.integers(args.min_win, args.max_win + 1, size=args.clips)
    t0 = time.perf_counter()
    frames = [preprocess.process_frames(synthetic.make_clip(int(n) + T // 4, seed=10_000 + i)) for i, n in enumerate(nwins)]
    prep_s = time.perf_counter() - t0
    bank = SourceBank(sum(f["pos"].shape[0] for f in frames), args.clips, norm["X_mean"], norm["X_std"])
    t0 = time.perf_counter()
    for f, n in zip(frames, nwins):
        assert bank.add(f)[1] == n
    torch.cuda.synchronize()
    upload_s = time.perf_counter() - t0

    # ---- sessions (same weights / DB as bench.py) ----
    kw = dict(n_db=args.db_rows, precision="bf16", device=dev, match_tensor_cores=None, admission=True)
    sess_a, *_ = workload.build_session(B, **kw)
    sess_b, *_ = workload.build_session(B, source_bank=bank, **kw)
    P = 4
    pool = []
    for i in range(P):
        h = workload.step_inputs(B, seed=i)
        side = np.concatenate([h["src_hips_vel"].reshape(B, -1), h["src_rvel"], h["src_rang"]], axis=1)
        pool.append({"X": torch.from_numpy(h["X"]).to(dev), "side": torch.from_numpy(side).to(dev),
                     "contacts": torch.from_numpy(h["contacts"]).to(dev), "eps": torch.from_numpy(h["eps"]).to(dev)})
    zeros = torch.zeros((B,), dtype=torch.uint8, device=dev)
    ones = torch.ones((B,), dtype=torch.uint8, device=dev)
    longest = torch.from_numpy(np.argsort(-nwins)[:B].astype(np.int32)).to(dev)   # clips the steady arms run

    def load(sess, i):
        d = pool[i % P]
        if sess is sess_a:
            sess.X.copy_(d["X"]); sess.side.copy_(d["side"]); sess.contacts.copy_(d["contacts"])
        else:
            sess.clip.copy_(longest)
        sess.start.copy_(zeros)
        sess.eps.copy_(d["eps"])

    for sess in (sess_a, sess_b):
        sess.capture()
        load(sess, 0)
        sess.start.copy_(ones)
        sess.step_device()
        for i in range(args.warmup):
            load(sess, i); sess.step_device()
    torch.cuda.synchronize()

    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(sess):
        e0.record()
        for i in range(K):
            load(sess, i)
            sess.step_device()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / K

    rounds = {"A": [], "B": []}
    for r in range(args.rounds):
        rounds["A"].append(timed(sess_a))
        rounds["B"].append(timed(sess_b))
    med = {k: float(np.median(v)) for k, v in rounds.items()}

    # ---- C: pipelined end to end from pinned host buffers ----
    pins_a, pins_b = [], []
    for i in range(P):
        h = workload.step_inputs(B, seed=i)
        pa = sess_a.pinned_inputs()
        pa["X"].numpy()[...] = h["X"]
        pa["side"].numpy()[...] = np.concatenate([h["src_hips_vel"].reshape(B, -1), h["src_rvel"], h["src_rang"]], 1)
        pa["contacts"].numpy()[...] = h["contacts"]
        pa["eps"].numpy()[...] = h["eps"]
        pins_a.append(pa)
        pb = sess_b.pinned_inputs()
        pb["clip"].numpy()[...] = longest.cpu().numpy()
        pb["eps"].numpy()[...] = h["eps"]
        pins_b.append(pb)

    def piped(sess, pins):
        torch.cuda.synchronize()
        t = time.perf_counter()
        prev = None
        for i in range(K):
            tk = sess.submit(pins[i % P])
            if prev is not None:
                sess.collect(prev)
            prev = tk
        sess.collect(prev)
        return (time.perf_counter() - t) * 1e3 / K

    piped(sess_a, pins_a), piped(sess_b, pins_b)             # warm-up (pipeline slots, pinned copies)
    prounds = {"A": [], "B": []}
    for r in range(args.rounds):
        prounds["A"].append(piped(sess_a, pins_a))
        prounds["B"].append(piped(sess_b, pins_b))
    pmed = {k: float(np.median(v)) for k, v in prounds.items()}

    # ---- kernel times (profiler on, separate from the timed rounds) ----
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for arm, sess in (("A", sess_a), ("B", sess_b)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for i in range(20):
                load(sess, i)
                sess.step_device()
            torch.cuda.synchronize()
        per, total = {}, 0.0
        for ev in prof.key_averages():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            total += ev.device_time_total
            if "source_windows" in ev.key:
                per[ev.key[:120]] = {"calls": ev.count, "device_us_avg": ev.device_time_total / max(ev.count, 1)}
        kernels[arm] = {"kernel_us_per_step_sum": total / 20, "kernels": per}

    # ---- serving run: the mixed-length clips through the bank session's slots ----
    start_rows, clip_rows, _ = serving_schedule(nwins, B)
    nframes = len(start_rows)
    starts_dev = torch.from_numpy(start_rows).to(dev)
    clips_dev = torch.from_numpy(clip_rows).to(dev)
    useful = int(nwins.sum())
    torch.cuda.synchronize()
    e0.record()
    for f in range(nframes):
        sess_b.start.copy_(starts_dev[f])
        sess_b.clip.copy_(clips_dev[f])
        sess_b.eps.copy_(pool[f % P]["eps"])
        sess_b.step_device()
    e1.record()
    torch.cuda.synchronize()
    serve_ms = e0.elapsed_time(e1)
    window_x_bytes = int(nwins.sum()) * T * 24 * 15 * 4

    res = {
        "gpu": gpu_info(torch),
        "config": {"slots": B, "precision": "bf16", "db_rows": args.db_rows, "cuda_graph": True, "timing": "cuda events",
                   "steps_per_round": K, "rounds": args.rounds, "warmup": args.warmup, "seed": args.seed},
        "step_ms": {"A_admission_d2d_inputs": med["A"], "B_bank": med["B"]},
        "step_ms_rounds": rounds,
        "B_vs_A": med["B"] / med["A"] - 1.0,
        "pipelined_end_to_end": {
            "step_ms": {"A_admission_host_inputs": pmed["A"], "B_bank_host_start_clip_eps": pmed["B"]},
            "step_ms_rounds": prounds,
            "frames_per_s": {"A": B * 1e3 / pmed["A"], "B": B * 1e3 / pmed["B"]},
            "h2d_bytes_per_step_computed": {"A": sess_a.h2d_bytes(), "B": sess_b.h2d_bytes()}},
        "profiler_kernels_20_steps": kernels,
        "serving": {"clips": args.clips, "window_range": [args.min_win, args.max_win], "useful_frames": useful,
                    "frames": nframes, "ms": serve_ms, "useful_frames_per_s": useful * 1e3 / serve_ms,
                    "slot_occupancy": useful / (nframes * B),
                    "host_preprocess_s": prep_s, "bank_upload_s": upload_s,
                    "bank_device_bytes": bank.nbytes(), "bank_frames": bank.n_frames,
                    "x_windows_bytes_computed": window_x_bytes,
                    "x_windows_over_bank": window_x_bytes / bank.nbytes()},
    }
    path = os.path.join(args.out, "source_bank_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "step_ms", "B_vs_A")}))
    print(json.dumps(res["pipelined_end_to_end"]["frames_per_s"]), json.dumps(kernels["B"]["kernels"]))
    print(json.dumps(res["serving"]))
    print(path)


if __name__ == "__main__":
    main()
