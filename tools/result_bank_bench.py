"""Cost and benefit of the result bank (CharacterizationSession(..., source_bank=bank, result_bank=rb)) at the bench
configuration of source_bank_bench.py (128 slots, bf16, 385-row DB, one CUDA graph, CUDA-event timing after warm-up),
in one process:

  A/B  device step of a bank session (A) against a bank + result session (B), alternating rounds, medians. Each round
       starts every slot on one of the 128 longest clips (untimed), so that every timed frame records a row.
  prof torch.profiler pass: device time of record_frames_kernel inside the frame. Under programmatic dependent
       launch that span starts while the post-process before it still runs, so CUDA events also time the kernel
       launched back to back on its own (100 launches).
  payload  CUDA-event time of one clip_payload_kernel launch over finished clips (every window recorded): the 128
       longest clips and all 1024, after the serving runs.
  serving 1024 mixed-length clips end to end with the payloads on the host:
       (i)  today's route: submit / collect of A's session with the per-step mocha_frame_out download, host-side
            stitching of each clip's frames and the final step on the host (numpy: fk / re-rooting / ik of each
            window's last frame for the source pose, hips fk, Euler degrees), host time reported apart;
       (ii) B's serve(): start / clip rows in, payloads of finished clips out.
       Both: useful frames/s, D2H bytes per useful frame (computed from the copies each route makes), wall time;
       3 alternating runs of each after a warm-up, medians.
  bench.py's result line, for drift against the committed profiles.

    python tools/result_bank_bench.py --out DIR [--steps 150 --rounds 5 --clips 1024]

writes DIR/result_bank_bench.json. Needs an sm_100 GPU.
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


def _qmul(a, b):
    aw, ax, ay, az = np.moveaxis(a, -1, 0)
    bw, bx, by, bz = np.moveaxis(b, -1, 0)
    return np.stack([bw * aw - bx * ax - by * ay - bz * az, bw * ax + bx * aw - by * az + bz * ay,
                     bw * ay + bx * az + by * aw - bz * ax, bw * az - bx * ay + by * ax + bz * aw], -1)


def _qinv(q):
    return q * np.array([1, -1, -1, -1], dtype=q.dtype)


def _qrot(q, x):
    t = 2 * np.cross(q[..., 1:], x)
    return x + q[..., :1] * t + np.cross(q[..., 1:], t)


def host_payload(frames, ik_rot, ik_pos, root_pos, root_rot, parents, T=60):
    """The final step of test_fullframework.py:672-721 on the host for one clip: the source pose of each window's last
    frame (fk, re-rooting on its root, ik: what features.extract gives as Ypos[w, -1] / Yrot[w, -1]) with the
    integrated root, then hips fk and Euler degrees for both sequences."""
    from mocha_sigasia2023_b200.characterize import to_euler_xyz
    F = frames["pos"].shape[0]
    nwin = F - T // 4
    last = np.minimum(np.arange(nwin) + T - 1, F - 1)
    lr, lp = frames["rot"][last], frames["pos"][last]
    J = len(parents)
    gr, gp = lr.copy(), lp.copy()
    for j in range(1, J):
        p = parents[j]
        gp[:, j] = _qrot(gr[:, p], lp[:, j]) + gp[:, p]
        gr[:, j] = _qmul(gr[:, p], lr[:, j])
    r0i = _qinv(gr[:, :1])
    xr, xp = _qmul(np.broadcast_to(r0i, gr.shape), gr), _qrot(np.broadcast_to(r0i, gr.shape), gp - gp[:, :1])
    sr, sp = xr.copy(), xp.copy()
    for j in range(1, J):
        p = parents[j]
        pi = _qinv(xr[:, p])
        sr[:, j], sp[:, j] = _qmul(pi, xr[:, j]), _qrot(pi, xp[:, j] - xp[:, p])
    sr[:, 0], sp[:, 0] = root_rot, root_pos

    def final(r, p):
        out_p, out_r = p[:, 1:].copy(), r[:, 1:].copy()
        out_p[:, 0] = _qrot(r[:, 0], p[:, 1]) + p[:, 0]
        out_r[:, 0] = _qmul(r[:, 0], r[:, 1])
        return np.degrees(to_euler_xyz(out_r)), out_p

    s_r, s_p = final(sr.astype(np.float32), sp.astype(np.float32))
    o_r, o_p = final(ik_rot, ik_pos)
    return {"src_rotations": s_r, "src_positions": s_p, "ours_rotations": o_r, "ours_positions": o_p}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="output directory (result_bank_bench.json)")
    ap.add_argument("--clips", type=int, default=1024, help="clips of the serving runs")
    ap.add_argument("--slots", type=int, default=128)
    ap.add_argument("--db-rows", type=int, default=385)
    ap.add_argument("--steps", type=int, default=150,
                    help="timed steps per arm and round (fewer than the 128 longest clips' windows)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--min-win", type=int, default=30)
    ap.add_argument("--max-win", type=int, default=225)
    ap.add_argument("--seed", type=int, default=2023)
    ap.add_argument("--no-bench-line", action="store_true", help="skip bench.py's drift line")
    args = ap.parse_args()

    import torch
    from admission_bench import gpu_info
    from mocha_sigasia2023_b200 import _lib, preprocess, skeleton, synthetic, workload
    from mocha_sigasia2023_b200.result_bank import ResultBank, serving_schedule
    from mocha_sigasia2023_b200.source_bank import SourceBank
    if not torch.cuda.is_available():
        raise SystemExit("result_bank_bench needs a CUDA device (there is no CPU measurement)")
    _lib.check(_lib.load().mocha_check_device(), "mocha_check_device")
    os.makedirs(args.out, exist_ok=True)
    B, K, T = args.slots, args.steps, 60
    if K >= args.max_win:
        raise SystemExit("--steps must stay below --max-win so that every timed frame records")
    dev = torch.device("cuda")
    info = gpu_info(torch)
    rng = np.random.default_rng(args.seed)
    norm = synthetic.make_norm_stats(7)["norm"]
    parents = np.asarray(skeleton.BONE_PARENTS)

    nwins = rng.integers(args.min_win, args.max_win + 1, size=args.clips)
    frames = [preprocess.process_frames(synthetic.make_clip(int(n) + T // 4, seed=10_000 + i)) for i, n in enumerate(nwins)]
    bank = SourceBank(sum(f["pos"].shape[0] for f in frames), args.clips, norm["X_mean"], norm["X_std"])
    for f, n in zip(frames, nwins):
        assert bank.add(f)[1] == n
    rb = ResultBank(bank)
    kw = dict(n_db=args.db_rows, precision="bf16", device=dev, match_tensor_cores=None, admission=True, source_bank=bank)
    sess_a, *_ = workload.build_session(B, **kw)
    sess_b, *_ = workload.build_session(B, result_bank=rb, **kw)
    P = 4
    eps_pool = [torch.from_numpy(workload.step_inputs(B, seed=i)["eps"]).to(dev) for i in range(P)]
    zeros = torch.zeros((B,), dtype=torch.uint8, device=dev)
    ones = torch.ones((B,), dtype=torch.uint8, device=dev)
    longest = torch.from_numpy(np.argsort(-nwins)[:B].astype(np.int32)).to(dev)
    assert int(nwins[np.argsort(-nwins)[B - 1]]) > K + 1

    def restart(sess):
        sess.clip.copy_(longest); sess.start.copy_(ones); sess.eps.copy_(eps_pool[0]); sess.step_device()
        sess.start.copy_(zeros)

    for sess in (sess_a, sess_b):
        sess.capture()
        restart(sess)
        for i in range(args.warmup):
            sess.eps.copy_(eps_pool[i % P]); sess.step_device()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(sess):
        restart(sess)
        e0.record()
        for i in range(K):
            sess.eps.copy_(eps_pool[i % P])
            sess.step_device()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / K

    rounds = {"A": [], "B": []}
    for r in range(args.rounds):
        rounds["A"].append(timed(sess_a))
        rounds["B"].append(timed(sess_b))
    med = {k: float(np.median(v)) for k, v in rounds.items()}

    # ---- kernel times (profiler on, separate from the timed rounds) ----
    from torch.profiler import ProfilerActivity, profile
    restart(sess_b)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(20):
            sess_b.eps.copy_(eps_pool[i % P]); sess_b.step_device()
        torch.cuda.synchronize()
    kernels = {}
    for ev in prof.key_averages():
        if ev.device_type == torch.autograd.DeviceType.CUDA and "record_frames" in ev.key:
            kernels[ev.key[:120]] = {"calls": ev.count, "device_us_avg": ev.device_time_total / max(ev.count, 1)}
    # the record kernel on its own: 128 recording slots (the slots hold the longest clips, every launch writes a row)
    count0 = sess_b.slot_count.clone()

    def record_alone(n):
        cnt = count0.clone()
        for _ in range(n):
            rb.record(sess_b.post.out, sess_b.match_idx, zeros, sess_b.slot_clip, cnt)

    record_alone(10)
    torch.cuda.synchronize()
    e0.record()
    record_alone(50)
    e1.record()
    torch.cuda.synchronize()
    record_alone_us = e0.elapsed_time(e1) * 1e3 / 50
    assert int(nwins[np.argsort(-nwins)[B - 1]]) > int(count0.max()) + 50

    # ---- serving 1024 clips with the payloads on the host ----
    start_rows, clip_rows, place = serving_schedule(nwins, B)
    nframes = len(start_rows)
    useful = int(nwins.sum())
    ids = np.arange(args.clips)
    eps_h = [workload.step_inputs(B, seed=i)["eps"] for i in range(P)]

    def route_i():
        """submit / collect with the per-step frame-out download, stitching and the host final step."""
        pins = [sess_a.pinned_inputs() for _ in range(3)]
        for i, p in enumerate(pins):
            p["eps"].numpy()[...] = eps_h[i % P]
        ik_rot = [np.empty((n, 25, 4)) for n in nwins]
        ik_pos = [np.empty((n, 25, 3)) for n in nwins]
        rpos = [np.empty((n, 3)) for n in nwins]
        rrot = [np.empty((n, 4)) for n in nwins]
        slot_k, slot_f = np.full(B, -1), np.zeros(B, dtype=np.int64)
        host_s = 0.0

        def stitch(f, out, sk, sf):
            for b in range(B):
                k = sk[b]
                if k < 0:
                    continue
                w = f - sf[b]
                if w < nwins[k]:
                    ik_rot[k][w], ik_pos[k][w] = out["ik_rot"][b], out["ik_pos"][b]
                    rpos[k][w], rrot[k][w] = out["src_root_pos"][b], out["src_root_rot"][b]

        torch.cuda.synchronize()
        t0 = time.perf_counter()
        prev = None
        for f in range(nframes):
            p = pins[f % 3]
            p["start"].numpy()[...] = start_rows[f]
            p["clip"].numpy()[...] = clip_rows[f]
            tk = sess_a.submit(p)
            if prev is not None:
                out = sess_a.collect(prev[0])
                h = time.perf_counter()
                stitch(prev[1], out, prev[2], prev[3])
                host_s += time.perf_counter() - h
            new = np.nonzero(start_rows[f])[0]
            slot_k[new], slot_f[new] = clip_rows[f][new], f
            prev = (tk, f, slot_k.copy(), slot_f.copy())
        out = sess_a.collect(prev[0])
        h = time.perf_counter()
        stitch(prev[1], out, prev[2], prev[3])
        payloads = [host_payload(frames[k], ik_rot[k], ik_pos[k], rpos[k], rrot[k], parents) for k in range(args.clips)]
        host_s += time.perf_counter() - h
        wall = time.perf_counter() - t0
        return wall, host_s, payloads

    def route_ii():
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        out = sess_b.serve(ids)
        return time.perf_counter() - t0, out

    _, out_ii = route_ii()                                # warm-up (pinned buffers, side stream)
    route_i()
    runs_i, runs_ii = [], []
    for r in range(3):
        w, h, _ = route_i()
        runs_i.append({"wall_s": w, "host_stitch_and_payload_s": h})
        runs_ii.append({"wall_s": route_ii()[0]})
    wall_i = float(np.median([r["wall_s"] for r in runs_i]))
    host_i = float(np.median([r["host_stitch_and_payload_s"] for r in runs_i]))
    wall_ii = float(np.median([r["wall_s"] for r in runs_ii]))

    # ---- clip_payload_kernel over finished clips (every clip is complete after the serving runs) ----
    assert (rb.done() == nwins).all()
    payload_us = {}
    for name, sel in (("longest_128_clips", np.argsort(-nwins)[:B]), ("all_clips", ids)):
        ids_dev = torch.from_numpy(sel.astype(np.int32)).to(dev)
        mx = int(nwins[sel].max())
        for _ in range(3):
            rb.payload_device(ids_dev, len(sel), mx)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            rb.payload_device(ids_dev, len(sel), mx)
        e1.record()
        torch.cuda.synchronize()
        payload_us[name] = {"clips": int(len(sel)), "rows": int(nwins[sel].sum()),
                            "us_per_launch": e0.elapsed_time(e1) * 1e3 / 10}
    d2h_i = nframes * sess_a.d2h_bytes()
    d2h_ii = useful * (24 * 3 * 4 * 2 + 24 * 3 * 8 * 2 + 8)

    bench_line = None
    if not args.no_bench_line:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "50", "--warmup",
                            "10"], capture_output=True, text=True, cwd=ROOT, timeout=1800)
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        bench_line = json.loads(lines[-1]) if lines else {"returncode": r.returncode, "stderr": r.stderr[-2000:]}

    res = {
        "gpu": info,
        "config": {"slots": B, "precision": "bf16", "db_rows": args.db_rows, "cuda_graph": True, "timing": "cuda events",
                   "steps_per_round": K, "rounds": args.rounds, "warmup": args.warmup, "seed": args.seed},
        "step_ms": {"A_bank": med["A"], "B_bank_results": med["B"]},
        "step_ms_rounds": rounds,
        "B_vs_A": med["B"] / med["A"] - 1.0,
        "B_minus_A_us": (med["B"] - med["A"]) * 1e3,
        "profiler_kernels": kernels,
        "profiler_note": "record_frames_kernel inside 20 graph frames of 128 recording slots; launched with programmatic "
                         "dependent launch, its span includes the time it waits in griddepcontrol.wait for the "
                         "post-process before it",
        "record_frames_alone_us_per_launch": record_alone_us,
        "record_frames_alone_note": "CUDA events over 50 back-to-back launches, 128 recording slots",
        "clip_payload_event_timed": payload_us,
        "serving": {"clips": args.clips, "window_range": [args.min_win, args.max_win], "useful_frames": useful,
                    "frames": nframes, "slot_occupancy": useful / (nframes * B),
                    "i_submit_collect_host_payload": {
                        "wall_s_median": wall_i, "host_stitch_and_payload_s_median": host_i, "runs": runs_i,
                        "useful_frames_per_s": useful / wall_i,
                        "d2h_bytes_computed": d2h_i, "d2h_bytes_per_useful_frame": d2h_i / useful},
                    "ii_serve": {"wall_s_median": wall_ii, "runs": runs_ii, "useful_frames_per_s": useful / wall_ii,
                                 "d2h_bytes_computed": d2h_ii, "d2h_bytes_per_useful_frame": d2h_ii / useful},
                    "result_bank_device_bytes": rb.nbytes(), "source_bank_device_bytes": bank.nbytes()},
        "bench_py": bench_line,
    }
    assert len(out_ii) == args.clips and all(out_ii[k]["match"].shape == (nwins[k],) for k in range(args.clips))
    path = os.path.join(args.out, "result_bank_bench.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "step_ms", "B_vs_A", "B_minus_A_us")}))
    print(json.dumps(kernels), record_alone_us, json.dumps(payload_us))
    print(json.dumps(res["serving"]))
    print(json.dumps(bench_line))
    print(path)


if __name__ == "__main__":
    main()
