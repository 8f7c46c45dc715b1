"""Raw clip ingestion on the device (SourceBank.add_raw, DESIGN §5d) against the host path (process_frames + add), on
the 1,024-clip serving set of source_bank_bench.py (window counts uniform in 30-225, clip i from seed 10_000 + i;
generating the clips is not timed), in one process:

  (a) process_frames of every clip on the host
  (b) one add_raw of every clip: wall time to a device synchronise, split into host checks and packing, the host-to-
      device copy and the five kernels (CUDA events); the kernels also one by one under torch.profiler
  (c) raw clips to payloads on the host, as useful frames/s: arm A = process_frames + add + serve(), arm B = add_raw +
      serve(), one 128-slot bf16 session over one bank and result bank that both arms clear and refill; the arms
      alternate, 3 runs each, medians
  (d) bench.py's line from the same process tree, to show the default step is untouched

The arrays of both arms are compared (float32 elements that differ, contacts that differ).

    python tools/ingest_bench.py --out DIR [--clips 1024]

writes DIR/ingest_bench.json. Needs an sm_100 GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="output directory (ingest_bench.json)")
    ap.add_argument("--clips", type=int, default=1024)
    ap.add_argument("--slots", type=int, default=128)
    ap.add_argument("--db-rows", type=int, default=385)
    ap.add_argument("--min-win", type=int, default=30)
    ap.add_argument("--max-win", type=int, default=225)
    ap.add_argument("--seed", type=int, default=2023)
    ap.add_argument("--runs", type=int, default=3, help="runs of each arm of (c)")
    ap.add_argument("--no-bench-line", action="store_true", help="skip bench.py's line")
    args = ap.parse_args()

    import torch
    from admission_bench import gpu_info
    from mocha_sigasia2023_b200 import _lib, preprocess, synthetic, workload
    from mocha_sigasia2023_b200.result_bank import ResultBank
    from mocha_sigasia2023_b200.source_bank import SourceBank
    if not torch.cuda.is_available():
        raise SystemExit("ingest_bench needs a CUDA device (there is no CPU measurement)")
    _lib.check(_lib.load().mocha_check_device(), "mocha_check_device")
    os.makedirs(args.out, exist_ok=True)
    T, dev = 60, torch.device("cuda")
    info = gpu_info(torch)
    rng = np.random.default_rng(args.seed)
    norm = synthetic.make_norm_stats(7)["norm"]
    nwins = rng.integers(args.min_win, args.max_win + 1, size=args.clips)
    clips = [synthetic.make_clip(int(n) + T // 4, seed=10_000 + i) for i, n in enumerate(nwins)]
    n_frames = int(sum(c["rotations"].shape[0] for c in clips))
    useful = int(nwins.sum())
    ids = list(range(args.clips))

    # ---- (a) host preprocessing ----
    t0 = time.perf_counter()
    frames = [preprocess.process_frames(c) for c in clips]
    host_s = time.perf_counter() - t0

    bank = SourceBank(n_frames, args.clips, norm["X_mean"], norm["X_std"])
    rb = ResultBank(bank)

    def fill_host(fr):
        bank.clear()
        rb.clear()
        for f in fr:
            bank.add(f)

    # ---- (b) add_raw, split ----
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]

    def add_raw_split():
        bank.clear()
        rb.clear()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        meta = bank._check_raw(clips)
        buf = bank._pack_raw(clips, meta)
        t1 = time.perf_counter()
        ev[0].record()
        dbuf = bank._upload_raw(buf)
        ev[1].record()
        bank._ingest_raw(dbuf, meta)
        ev[2].record()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        return {"wall_s": t2 - t0, "host_check_and_pack_s": t1 - t0, "h2d_ms": ev[0].elapsed_time(ev[1]),
                "kernels_and_tables_ms": ev[1].elapsed_time(ev[2]), "h2d_bytes": int(buf.nbytes)}

    add_raw_split()                                        # warm-up: module load, savgol tables, allocator
    split_runs = [add_raw_split() for _ in range(3)]
    split = {k: float(np.median([r[k] for r in split_runs])) for k in split_runs[0]}

    # kernel times, each launch on its own (profiler run, not used for the wall times)
    from torch.profiler import ProfilerActivity, profile
    bank.clear()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        bank.add_raw(clips)
        torch.cuda.synchronize()
    kernels = {}
    for e in prof.key_averages():
        m = re.search(r"ingest_[a-z]+_kernel", e.key)
        if m:
            kernels[m.group(0)] = {"us": getattr(e, "device_time_total", None) or e.cuda_time_total, "count": e.count}

    # compare the two paths' arrays
    def snapshot():
        return {k: getattr(bank, k)[:n_frames].clone() for k in ("pos", "vel", "rot", "ang", "contacts")}

    raw_arrays = snapshot()
    fill_host(frames)
    host_arrays = snapshot()
    diff = {}
    for k in ("pos", "vel", "rot", "ang"):
        a, b = raw_arrays[k].view(torch.int32).long(), host_arrays[k].view(torch.int32).long()
        d = a != b
        diff[k] = {"elements": int(a.numel()), "differ": int(d.sum()), "max_ulp": int((a - b).abs().max())}
    diff["contacts"] = {"elements": int(raw_arrays["contacts"].numel()),
                        "differ": int((raw_arrays["contacts"] != host_arrays["contacts"]).sum())}

    # ---- (c) raw clips to payloads ----
    sess, *_ = workload.build_session(args.slots, n_db=args.db_rows, precision="bf16", device=dev, match_tensor_cores=None,
                                      admission=True, source_bank=bank, result_bank=rb)
    sess.capture()

    def arm_a():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fill_host([preprocess.process_frames(c) for c in clips])
        torch.cuda.manual_seed(1234)                       # the same eps draws in both arms
        out = sess.serve(ids)
        return time.perf_counter() - t0, out

    def arm_b():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        bank.clear()
        rb.clear()
        bank.add_raw(clips)
        torch.cuda.manual_seed(1234)
        out = sess.serve(ids)
        return time.perf_counter() - t0, out

    fill_host(frames)
    sess.serve(ids)                                        # warm-up (pinned buffers, side stream)
    runs = {"A": [], "B": []}
    out_a = out_b = None
    for _ in range(args.runs):
        w, out_a = arm_a()
        runs["A"].append(w)
        w, out_b = arm_b()
        runs["B"].append(w)
    med = {k: float(np.median(v)) for k, v in runs.items()}
    same = all(np.array_equal(out_a[c][k], out_b[c][k]) for c in ids for k in out_a[c])
    assert len(out_b) == args.clips and all(out_b[c]["match"].shape == (nwins[c],) for c in ids)

    bench_line = None
    if not args.no_bench_line:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "50", "--warmup",
                            "10"], capture_output=True, text=True, cwd=ROOT, timeout=1800)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        bench_line = json.loads(lines[-1]) if lines else {"returncode": r.returncode, "stderr": r.stderr[-2000:]}

    res = {
        "gpu": info,
        "config": {"clips": args.clips, "frames": n_frames, "useful_frames": useful,
                   "window_range": [args.min_win, args.max_win], "clip_seeds": "10_000 + i", "slots": args.slots,
                   "precision": "bf16", "db_rows": args.db_rows, "runs": args.runs},
        "a_process_frames_host_s": host_s,
        "b_add_raw": {"median": split, "runs": split_runs,
                      "note": "wall time from the call to a device synchronise; the H2D copy is from pageable memory"},
        "b_kernels_profiler_us": kernels,
        "raw_vs_host_arrays": diff,
        "c_raw_clips_to_payloads": {
            "A_process_frames_add_serve": {"wall_s_median": med["A"], "runs_s": runs["A"],
                                           "useful_frames_per_s": useful / med["A"]},
            "B_add_raw_serve": {"wall_s_median": med["B"], "runs_s": runs["B"], "useful_frames_per_s": useful / med["B"]},
            "B_speedup": med["A"] / med["B"],
            "payloads_identical": bool(same)},
        "d_bench_py": bench_line,
    }
    path = os.path.join(args.out, "ingest_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "a_process_frames_host_s", "b_add_raw", "b_kernels_profiler_us")}))
    print(json.dumps(res["raw_vs_host_arrays"]))
    print(json.dumps(res["c_raw_clips_to_payloads"]))
    print(json.dumps(bench_line))
    print(path)


if __name__ == "__main__":
    main()
