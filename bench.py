#!/usr/bin/env python
"""bench.py — characterised frames/s of MOCHA's per-frame hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--clips C | --total-clips T] [--precision bf16|fp32|tf32x3]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs as DIR/<name>.npy
    python bench.py --impl reference ...      # the UNMODIFIED reference's per-frame loop on the host cores
    python bench.py --workload match_sweep    # BASELINE config 3 alone (4096 queries x --sweep-rows rows x 23040)
    python -m torch.distributed.run ... bench.py --workload match_sharded --gpus N   # BASELINE config 5 alone

A step = one pass of the hot path over one batch: every clip on this GPU advances one frame
(encode its new 60-frame window -> context feature -> nearest-neighbour match -> CVAE sample ->
AdaIN decode -> to_mot -> root integration / blending / foot-lock IK). Clips are independent, so
N GPUs run N x C clips with no data-path collective (weak scaling; --total-clips T fixes the total instead: strong).
Besides the headline the line carries: `roofline` (largest launch), `roofline_step` (whole step vs the tensor roof),
`roofline_kernels` (the GEMM family and the fused block tail), `hbm_kernels` (achieved GB/s of the bandwidth-bound
kernels), `match_sweep` (config 3), `latency_batch1*` (config 2 at 385 / 10 k / 100 k DB rows), `fp32_mode` / `tf32x3_mode`
(parity-mode throughput on FFMA / on 3xTF32 tcgen05 GEMMs), `torch_eager_gpu` (the reference's own modules with stock PyTorch eager
kernels on the same GPU), `cpu_baseline` (the reference itself with per-stage timings, N = 1) and, for N > 1, `match_sharded` (config 5).
Prints ONE JSON line on rank 0, as the LAST line of stdout.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "characterized_frames_per_s"
UNIT = "frames/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--clips", type=int, default=128, help="clips per GPU (config 4: 1024 clips / 8 GPUs)")
    ap.add_argument("--total-clips", type=int, default=0, help="strong scaling: this many clips in total, split over the GPUs")
    ap.add_argument("--workload", default="characterize", choices=["characterize", "match_sweep", "match_sharded"])
    ap.add_argument("--sweep-rows", type=int, default=131072, help="match_sweep DB rows (config 3 is 1000000)")
    ap.add_argument("--sweep-queries", type=int, default=4096)
    ap.add_argument("--rows-per-gpu", type=int, default=2_000_000, help="match_sharded: bf16 DB rows per GPU (16 M at 8 GPUs)")
    ap.add_argument("--no-extras", action="store_true", help="headline only (skip sweep / hbm / latency / fp32 legs)")
    ap.add_argument("--no-match-sharded", action="store_true")
    ap.add_argument("--db-rows", type=int, default=385, help="character DB rows (400-frame character clip)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "tf32x3"])
    ap.add_argument("--lanes", type=int, default=1, help="sub-batch lanes: the clips of a GPU are cut into this many groups "
                    "whose frames run concurrently on separate streams inside the captured graph (measured on B200 at 128 "
                    "clips: 1.37 / 1.49 / 1.63 / 1.83 ms per step for 1 / 2 / 3 / 4 lanes - one lane is fastest)")
    ap.add_argument("--latency-frames", type=int, default=200)
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last of them computed (every rank's clips) as DIR/<name>.npy "
                    "in float32 / float64, at most 64 MB in all (a fixed, seeded sample of clips beyond that)")
    a = ap.parse_args()
    if a.dump_outputs and (a.impl != "b200" or a.workload != "characterize"):
        ap.error("--dump-outputs needs --impl b200 --workload characterize")
    if a.total_clips:
        a.clips = max(1, a.total_clips // max(1, int(os.environ.get("WORLD_SIZE", "1"))))
    return a


def workload_config(args):
    return {
        "workload": "batched characterization, clips sharded data-parallel (BASELINE config 4 per-GPU share): "
                    f"{args.clips} clips/GPU advance one frame per step, 60x24x15 pose window per clip",
        "clips_per_gpu": args.clips,
        "window": [60, 24, 15],
        "db_rows": args.db_rows,
        "feature_dim": 23040,
        "cvae": "stochastic (eps injected)",
        "second_decode_cm_trans": False,
        "l2": "per-step working set (activations + weights + DB) exceeds the 126 MB L2; no explicit flush",
        "parallelism": f"dp{args.gpus} over clips, no collective on the data path",
        "scaling_mode": "strong (--total-clips %d)" % args.total_clips if args.total_clips else "weak (clips per GPU fixed)",
        "lanes": args.lanes,
    }


# -------------------------------------------------------------------------------------------------
# clocks
# -------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "20", "-i", str(self.index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def wait_first_sample(self, timeout_s=3.0):
        """nvidia-smi needs ~0.1-0.5 s to emit its first line; block until it has, then mark the offset so
        that only samples taken after this point (the timed region) are reported."""
        self.skip = 0
        if self.p is None:
            return
        t0 = time.time()
        while time.time() - t0 < timeout_s:
            try:
                if os.path.getsize(self.f.name) > 0:
                    break
            except OSError:
                pass
            time.sleep(0.02)
        try:
            self.skip = os.path.getsize(self.f.name)
        except OSError:
            self.skip = 0

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.03)  # let the sample in flight land
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(getattr(self, "skip", 0))
        sm, mx, reasons, power = [], [], set(), []
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1])); mx.append(float(c[2])); power.append(float(c[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       power_w_max=max(power))
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        return out


# -------------------------------------------------------------------------------------------------
# CPU arm: the reference's own per-frame loop on the host cores
# -------------------------------------------------------------------------------------------------
def reference_rate(threads=None, timeout_s=900):
    """frames/s of the UNMODIFIED reference `test_fullframework.main()` frame loop (oracle/ref_harness.py --time) on the
    host cores, in a subprocess with the GPU hidden (the reference picks its device from torch.cuda.is_available()).
    Returns None when the reference tree is not staged (oracle/stage_reference.py)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import stage_reference
    if stage_reference.reference_root() is None:
        return None
    threads = threads or os.cpu_count() or 1
    out = tempfile.NamedTemporaryFile("w+", suffix=".json", delete=False)
    out.close()
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS=str(threads), MKL_NUM_THREADS=str(threads))
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_harness.py"), "--time", "--threads", str(threads),
                        "--out", out.name], env=env, capture_output=True, text=True, timeout=timeout_s,
                       cwd=tempfile.gettempdir())
    if r.returncode != 0:
        sys.stderr.write("reference harness failed:\n" + r.stderr[-2000:] + "\n")
        return None
    res = json.load(open(out.name))
    os.unlink(out.name)
    return res


def cpu_port_rate(args, clips, steps, warmup, db_rows=None):
    """Fallback when the reference tree is not staged: frames/s of the oracle's NumPy port for `clips` clips."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import numpy as np
    from mocha_oracle import clip as oclip
    from mocha_oracle.pipeline import OraclePipeline
    from mocha_sigasia2023_b200 import skeleton, weights, workload
    gen_sd = {k: v.numpy() for k, v in weights.generator_state_dict(1777).items()}
    cvae_sd = {k: v.numpy() for k, v in weights.cvae_state_dict(1778).items()}
    stats = workload.stats_as_dict(workload.driver_stats())
    n_db = db_rows or args.db_rows
    enc, cnt = oclip.encode_windows(gen_sd, workload.pose_windows(n_db, 5000))
    nm = ((cnt - stats["cnt_mean"][None]) / stats["cnt_std"][None]).reshape(n_db, -1)
    pipe = OraclePipeline(gen_sd, cvae_sd, stats, enc, nm, clips, skeleton.BONE_PARENTS)
    times = []
    for f in range(warmup + steps):
        inp = workload.step_inputs(clips, seed=f)
        t0 = time.perf_counter()
        pipe.step(inp["X"], inp["src_hips_vel"], inp["src_rvel"], inp["src_rang"], inp["contacts"], inp["eps"])
        if f >= warmup:
            times.append(time.perf_counter() - t0)
    return clips * len(times) / sum(times), sum(times) / len(times)


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return None


def torch_eager_gpu_baseline(args, timeout_s=600):
    """BASELINE.md §3 item 3: the reference's own Generator / CVAE modules, unmodified, on the same B200 with stock PyTorch
    eager (library kernels), batched like the bench step, network portion of the frame only (oracle/ref_eager_gpu.py, run
    in a subprocess). A reported baseline: "hand-written kernels vs library kernels" with the GPU held fixed."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import stage_reference
    if stage_reference.reference_root() is None:
        return {"unavailable": "reference tree not staged (oracle/stage_reference.py)"}
    out = tempfile.NamedTemporaryFile("w+", suffix=".json", delete=False)
    out.close()
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_eager_gpu.py"), "--clips", str(args.clips),
                            "--steps", "20", "--warmup", "5", "--db-rows", str(args.db_rows), "--out", out.name],
                           env=env, capture_output=True, text=True, timeout=timeout_s, cwd=tempfile.gettempdir())
        if r.returncode != 0:
            return {"unavailable": "ref_eager_gpu.py failed: " + r.stderr[-300:]}
        modes = json.load(open(out.name))
    except Exception as e:  # noqa: BLE001
        return {"unavailable": f"{type(e).__name__}: {e}"[:300]}
    finally:
        if os.path.exists(out.name):
            os.unlink(out.name)
    return {"what": "the reference's Generator + CVAE modules (unmodified) on this GPU with stock PyTorch eager kernels, "
                    f"{args.clips} clips per step: encode + cdist/argmin match + CVAE.sample + decoder + to_mot + D2H of Y; the "
                    "reference's NumPy FK / IK / inertialization and its second decode are NOT included (so this is an upper "
                    "bound for an eager-GPU run of the reference), CUDA-event timed",
            "modes": modes}


def host_threads():
    try:
        from threadpoolctl import threadpool_info
        return int(max([p.get("num_threads", 1) for p in threadpool_info()] + [1]))
    except Exception:
        return os.cpu_count() or 1


def cpu_baseline_record(args):
    """(record, frames/s, ms per frame): the reference itself when staged, else the oracle port."""
    ref = reference_rate()
    if ref is not None:
        rec = {"value": ref["frames_per_s"], "unit": UNIT, "cores": ref["threads"], "kind": "reference",
               "sample": f"the unmodified reference test_fullframework.main() frame loop (:438-641), {ref['frames']} frames of "
                         f"one 240-frame clip vs a 385-row character DB on CPU (torch threads = {ref['threads']} of "
                         f"{os.cpu_count()} host cpus), timed between its first and last in-loop BallTree.query call; "
                         f"the reference decodes twice per frame (trans + cm_trans) and runs batch 1",
               "ms_per_frame": ref["ms_per_frame"], "main_s": ref["main_s"],
               "p50_ms_per_frame": ref.get("p50_ms_per_frame"), "p99_ms_per_frame": ref.get("p99_ms_per_frame"),
               "cpu_model": cpu_model(),
               # per-stage perf_counter wrappers around the reference's own calls (BASELINE.md §3 item 1), whole main()
               "stages": ref.get("stages")}
        return rec, ref["frames_per_s"], ref["ms_per_frame"]
    import numpy  # noqa: F401
    rate, sec = cpu_port_rate(args, 2, 3, 1)
    rec = {"value": rate, "unit": UNIT, "cores": host_threads(), "kind": "port",
           "sample": "2 clips x 3 frames of the same per-frame path (NumPy port of the reference, oracle/mocha_oracle); the "
                     "reference tree is not staged on this box (oracle/stage_reference.py)"}
    return rec, rate, sec * 1e3 / 2


def run_reference(args):
    """`--impl reference`: rank 0 alone runs (one process, every host core: a CPU arm does not scale with --gpus N)."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    rec, rate, ms_frame = cpu_baseline_record(args)
    cfg = workload_config(args)
    cfg["reference_arm"] = "1 process on rank 0 with all host cores, regardless of --gpus (the CPU path does not shard)"
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_frame * args.clips, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg, "cpu_baseline": rec,
        "note": "ms_per_step = clips_per_gpu x measured ms per frame (the reference advances clips one after another)",
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# -------------------------------------------------------------------------------------------------
# peaks
# -------------------------------------------------------------------------------------------------
def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


FLOP_PER_FRAME = 3.03e9      # SURVEY §8d: mot_embedding 1.205 + encoder 0.316 + CVAE 0.686 + decoder 0.540 + to_mot 0.281


def timed(torch, fn, reps, warm=2):
    """average milliseconds of fn() over `reps` back-to-back calls on the current stream (CUDA events)."""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


# -------------------------------------------------------------------------------------------------
# config 3: matching sweep
# -------------------------------------------------------------------------------------------------
def match_sweep(args, torch, lib, _lib, dev, rows=None, queries=None):
    """Q queries x N rows x 23040, planted and iid data, bf16 and fp32 (TF32) storage: ms, TFLOP/s (2 Q N D), fraction of
    the measured bf16 burst peak, planted rows found, iid top-1 agreement with a float64 brute force on a query subset."""
    from mocha_sigasia2023_b200.balltree import BallTree
    peaks, src = load_peaks()
    Q, N, D = queries or args.sweep_queries, rows or args.sweep_rows, 23040
    out = {"queries": Q, "rows": N, "dim": D, "k": 2, "kc": 8, "peak_source": src, "cases": []}
    flops = 2.0 * Q * N * D
    for kind in ("planted", "iid"):
        g = torch.Generator(device=dev).manual_seed(77 if kind == "planted" else 78)
        db = torch.empty((N, D), dtype=torch.float32, device=dev)
        for s in range(0, N, 32768):
            db[s:s + 32768] = torch.randn((min(32768, N - s), D), generator=g, device=dev)
        if kind == "planted":
            pick = torch.randint(0, N, (Q,), generator=g, device=dev)
            q = db[pick] + 0.05 * torch.randn((Q, D), generator=g, device=dev)
        else:
            pick = None
            q = torch.randn((Q, D), generator=g, device=dev)
        # float64 brute force for a query subset (every row): the arithmetic of oracle/mocha_oracle/matching.knn_gemm
        sub = torch.arange(0, Q, max(1, Q // 256), device=dev)[:256]
        q64 = q[sub].double()
        best = torch.full((len(sub),), float("inf"), dtype=torch.float64, device=dev)
        besti = torch.zeros((len(sub),), dtype=torch.int64, device=dev)
        for s in range(0, N, 16384):
            x = db[s:s + 16384].double()
            d2 = (x * x).sum(1)[None, :] - 2.0 * (q64 @ x.T)
            m, i = d2.min(dim=1)
            upd = m < best
            best = torch.where(upd, m, best)
            besti = torch.where(upd, i + s, besti)
            del x, d2
        for storage in ("bf16", "fp32"):
            tree = BallTree(db, use_tensor_cores=True, kc=8, tc_storage=storage)
            res = {}

            def run():
                res["d"], res["i"] = tree.query_device(q, k=2)

            ms = timed(torch, run, 3, warm=1)
            idx = res["i"][:, 0]
            rec = {"data": kind, "storage": storage + (" (TF32 MMA)" if storage == "fp32" else ""), "ms": ms,
                   "tflops": flops / ms / 1e9, "frac_of_bf16_burst_peak": flops / ms / 1e9 / peaks["bf16_tflops"],
                   "top1_agreement_vs_f64_bruteforce_256q": float((idx[sub] == besti).double().mean())}
            if pick is not None:
                rec["planted_found"] = float((idx == pick).double().mean())
            out["cases"].append(rec)
            del tree
        del db, q
        torch.cuda.empty_cache()
    return out


# -------------------------------------------------------------------------------------------------
# config 5: DB-sharded matching (rows split over the ranks, queries replicated, top-k exchange + merge)
# -------------------------------------------------------------------------------------------------
def match_sharded(args, torch, dist, lib, _lib, dev, rank, world):
    from mocha_sigasia2023_b200.sharded import ShardedMatcher
    Nl, Q, D = args.rows_per_gpu, args.sweep_queries, 23040
    free, _ = torch.cuda.mem_get_info(dev)
    Nl = int(min(Nl, (free - (6 << 30)) // (D * 2 + 4)))          # bf16 rows + norm; keep 6 GB clear
    N = Nl * world
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    db16 = torch.empty((Nl, D), dtype=torch.bfloat16, device=dev)
    norm = torch.empty((Nl,), dtype=torch.float32, device=dev)
    for s in range(0, Nl, 16384):
        m = min(16384, Nl - s)
        rows = torch.randn((m, D), generator=g, device=dev)
        _lib.check(lib.mocha_db_pack_bf16(_lib.ptr(rows), m, D, _lib.ptr(db16[s:s + m]), _lib.ptr(norm[s:s + m]), _lib.stream_ptr()))
    # planted queries: query j is a noisy copy of row (7919 j mod Nl) of rank (j mod world); built on its owner, then shared
    gq = torch.Generator(device=dev).manual_seed(99)
    owner = torch.arange(Q, device=dev) % world
    row = (torch.arange(Q, device=dev) * 7919) % Nl
    q = torch.zeros((Q, D), device=dev)
    mine = owner == rank
    q[mine] = db16[row[mine]].float() + 0.05 * torch.randn((int(mine.sum()), D), generator=gq, device=dev)
    if world > 1:
        dist.all_reduce(q)
    q16 = q.to(torch.bfloat16)
    ws = torch.empty(lib.mocha_match_tc_workspace_bytes(Q, Nl, D, 8) + 1024, dtype=torch.uint8, device=dev)

    def local_query(qt, k):
        idx = torch.empty((Q, k), dtype=torch.int64, device=dev)
        dd = torch.empty((Q, k), dtype=torch.float64, device=dev)
        _lib.check(lib.mocha_match_tc(_lib.ptr(qt), _lib.ptr(q16), Q, _lib.ptr(db16), None, _lib.ptr(norm), Nl, D, k, 8, 0,
                                      _lib.ptr(idx), _lib.ptr(dd), _lib.ptr(ws), ws.numel(), _lib.stream_ptr()))
        return dd, idx

    def tmax(ms):
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    out = {"queries": Q, "rows_total": N, "rows_per_gpu": Nl, "dim": D, "k": 2, "storage": "bf16", "exchange": {}}
    results = {}
    for mode in (["nccl", "peer"] if world > 1 else ["nccl"]):
        m = ShardedMatcher(N, local_query, exchange=mode)
        res = {}

        def run():
            res["d"], res["i"] = m.query(q, k=2)

        run(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        ms = tmax(timed(torch, run, 3, warm=0))
        rec = {"query_ms": ms, "tflops_total": 2.0 * Q * N * D / ms / 1e9, "tflops_per_gpu": 2.0 * Q * Nl * D / ms / 1e9}
        if world > 1:
            dl, il = local_query(q, 2)
            il = il + m.lo

            def xchg():
                if mode == "peer":
                    m._peer.exchange_merge(dl, il)
                else:
                    all_d = torch.empty((world * Q, 2), dtype=torch.float64, device=dev)
                    all_i = torch.empty((world * Q, 2), dtype=torch.int64, device=dev)
                    dist.all_gather_into_tensor(all_d, dl)
                    dist.all_gather_into_tensor(all_i, il)
                    m.merge(all_d.view(world, Q, 2), all_i.view(world, Q, 2), 2)

            dist.barrier()
            rec["exchange_us"] = tmax(timed(torch, xchg, 20, warm=2)) * 1e3
        results[mode] = (res["d"].clone(), res["i"].clone())
        out["exchange"][mode] = rec
        if getattr(m, "_peer", None) is not None:
            m._peer.close()
    want = owner * Nl + row
    i0 = results["nccl"][1]
    out["planted_found"] = float((i0[:, 0] == want).double().mean())
    if "peer" in results:
        out["peer_equals_nccl"] = bool((results["peer"][1] == i0).all()) and bool((results["peer"][0] == results["nccl"][0]).all())
    # parity of the merged lists with a single-GPU run over the rows that can win: every rank re-ranks its own planted
    # rows' neighbourhood exactly (float64, difference form) and the owners' distances must equal the merged ones
    sel = torch.nonzero(mine)[:64, 0]
    if len(sel):
        x = db16[row[sel]].double()
        d = torch.sqrt(((q[sel].double() - x) ** 2).sum(1))
        out["owner_distance_max_rel_err"] = float(((results["nccl"][0][sel, 0] - d).abs() / d).max())
    del db16, norm, ws
    torch.cuda.empty_cache()
    return out


# -------------------------------------------------------------------------------------------------
# B200 arm
# -------------------------------------------------------------------------------------------------
def run_b200(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    from mocha_sigasia2023_b200 import _lib, workload

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL_DEBUG is left as the driver set it (its INFO lines decide comm_nranks_ok); the JSON line is printed LAST
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()
    _lib.check(lib.mocha_check_device(), "mocha_check_device")
    dev = torch.device("cuda", local)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def finish(line):
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        if rank == 0:
            sys.stdout.flush()
            print(json.dumps(line), flush=True)

    if args.workload == "match_sweep":
        peaks, src = load_peaks()
        sw = match_sweep(args, torch, lib, _lib, dev) if rank == 0 else None
        best = max(c["tflops"] for c in sw["cases"] if c["storage"] == "bf16") if sw else 0.0
        finish({"metric": "match_sweep_tflops", "value": best, "unit": "TFLOP/s", "n_gpus": 1, "higher_is_better": True,
                "dtype": "bf16", "data": "synthetic", "config": {"workload": "BASELINE config 3: context-matching sweep"},
                "match_sweep": sw})
        return
    if args.workload == "match_sharded":
        ms = match_sharded(args, torch, dist, lib, _lib, dev, rank, world)
        finish({"metric": "match_sharded_tflops", "value": ms["exchange"]["nccl"]["tflops_total"], "unit": "TFLOP/s",
                "n_gpus": world, "higher_is_better": True, "scaling": "weak", "dtype": "bf16", "data": "synthetic",
                "config": {"workload": "BASELINE config 5: DB-sharded matching, rows split over the GPUs"}, "match_sharded": ms})
        return

    B, K, W = args.clips, args.steps, max(args.warmup, 3)
    sess, *_ = workload.build_session(B, n_db=args.db_rows, precision=args.precision, device=dev,
                                      seed=rank, match_tensor_cores=None, lanes=args.lanes)
    P = 4  # distinct input sets cycled through
    host_pool = [workload.step_inputs(B, seed=1000 * rank + i) for i in range(P)]
    dev_pool = []
    for h in host_pool:
        side = np.concatenate([h["src_hips_vel"].reshape(B, -1), h["src_rvel"], h["src_rang"]], axis=1)
        dev_pool.append({"X": torch.from_numpy(h["X"]).to(dev), "side": torch.from_numpy(side).to(dev),
                         "contacts": torch.from_numpy(h["contacts"]).to(dev), "eps": torch.from_numpy(h["eps"]).to(dev)})

    def load_dev(i):
        d = dev_pool[i % P]
        sess.X.copy_(d["X"]); sess.side.copy_(d["side"]); sess.contacts.copy_(d["contacts"]); sess.eps.copy_(d["eps"])

    # init frame + one eager steady-state frame to count launches, then capture the CUDA graph
    load_dev(0); sess.step_device()
    lib.mocha_reset_launch_count()
    load_dev(1); sess.step_device()
    launches_per_step = int(lib.mocha_launch_count())
    sess.capture()
    for i in range(W):
        load_dev(i); sess.step_device()

    # ---- device-resident throughput ("value") ----
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_first_sample()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(K):
        load_dev(i); sess.step_device()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if sampler else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    value = world * B * K / (ms_total * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, sess, dist, rank, world)   # before the end-to-end pass below advances the session

    # ---- end to end through the public API with HOST buffers: every step copies its inputs from pinned
    # host memory, runs the frame and copies the pose structs back; the H2D of step i+1 overlaps step i ----
    pinned_pool = []
    for h in host_pool:
        pin = sess.pinned_inputs()
        pin["X"].numpy()[...] = h["X"]
        pin["side"].numpy()[...] = np.concatenate([h["src_hips_vel"].reshape(B, -1), h["src_rvel"], h["src_rang"]], axis=1)
        pin["contacts"].numpy()[...] = h["contacts"]
        pin["eps"].numpy()[...] = h["eps"]
        pinned_pool.append(pin)
    for i in range(3):
        sess.collect(sess.submit(pinned_pool[i % P]))
    barrier()
    checksum = 0.0
    e0.record()
    prev = None
    for i in range(K):
        tk = sess.submit(pinned_pool[i % P])
        if prev is not None:
            checksum += float(sess.collect(prev)["ik_pos"][0, 0, 0])
        prev = tk
    checksum += float(sess.collect(prev)["ik_pos"][0, 0, 0])
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * B * K / (float(t.item()) * 1e-3)
    assert checksum == checksum, "end-to-end outputs contain NaN"

    peaks, peak_src = load_peaks()
    ms_step = ms_total / K
    step_tflops = FLOP_PER_FRAME * B / (ms_step * 1e-3) / 1e12
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong" if args.total_clips else "weak",
        "vs_baseline": None, "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
        "config": workload_config(args),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": sess.h2d_bytes(),
                "d2h_bytes_per_step": sess.d2h_bytes()},
        "gpu_launches": launches_per_step * K,
        "gpu_launches_per_step": launches_per_step,
        "clocks": clocks,
        "roofline_step": {"bound": "tensor", "achieved": step_tflops, "peak": peaks["bf16_tflops_sustained"], "unit": "TFLOP/s",
                          "frac": step_tflops / peaks["bf16_tflops_sustained"],
                          "frac_of_burst_peak": step_tflops / peaks["bf16_tflops"],
                          "flops_per_step": FLOP_PER_FRAME * B, "peak_source": peak_src + " (sustained: the step is a long "
                          "back-to-back kernel sequence)",
                          "note": "algorithmic FLOPs of the whole frame (SURVEY §8d: 3.03 GFLOP per clip-frame) / step time"},
    }

    if rank == 0:
        line["roofline"] = roofline_pass(args, sess, torch, lib, _lib)
        if not args.no_extras:
            line["roofline_kernels"] = kernel_rooflines(sess, torch, lib, _lib)
            line["hbm_kernels"] = hbm_kernels(sess, torch, lib, _lib)
    del dev_pool
    if rank == 0 and not args.no_extras:
        if args.precision == "bf16":
            line["fp32_mode"] = fp32_mode_pass(args, dev, torch, workload, lib)
            line["tf32x3_mode"] = fp32_mode_pass(args, dev, torch, workload, lib, precision="tf32x3")
            line["second_decode"] = second_decode_pass(args, dev, torch, workload)
        if not args.no_latency:
            line["latency_batch1"] = latency_pass(args, dev, torch, workload)
            line["latency_batch1_bf16"] = latency_pass(args, dev, torch, workload, precision="bf16")
            line["latency_batch1_db_sweep"] = [latency_pass(args, dev, torch, workload, precision=pr, db_rows=n, frames=100)
                                               for n in (10_000, 100_000) for pr in ("fp32", "bf16")]
    del sess
    torch.cuda.empty_cache()
    if rank == 0 and not args.no_extras:
        line["match_sweep"] = match_sweep(args, torch, lib, _lib, dev)
    if world > 1 and not args.no_match_sharded and not args.no_extras:
        ms = match_sharded(args, torch, dist, lib, _lib, dev, rank, world)
        if rank == 0:
            line["match_sharded"] = ms
    if rank == 0 and world == 1 and not args.no_extras:
        line["torch_eager_gpu"] = torch_eager_gpu_baseline(args)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"], _, _ = cpu_baseline_record(args)
    finish(line)


DUMP_LIMIT_BYTES = 63_000_000      # array bytes; with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, sess, dist=None, rank=0, world=1):
    """What the timed step hands its caller, as of the step that ran last: the FrameOut fields of every clip (pose,
    blended and IK poses, source root: what CharacterizationSession.collect() returns, float64), the network output Y
    and the matched DB row and its distance. Every rank's clips are gathered (rank r holds clips r*B .. r*B+B-1) and
    rank 0 writes them. Above DUMP_LIMIT_BYTES a fixed, seeded sample of clips is written; clip_index.npy says which
    clips the rows are."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    outs = sess.post.read()
    outs["Y"] = sess.Y.cpu().numpy()
    outs["match_idx"] = sess.match_idx.cpu().numpy().astype(np.float64)
    outs["match_dist"] = sess.match_dist.cpu().numpy()
    if world > 1:
        parts = [None] * world
        dist.all_gather_object(parts, outs)
        if rank != 0:
            return
        outs = {k: np.concatenate([p[k] for p in parts]) for k in outs}
    B = len(outs["Y"])
    per_clip = sum(a.nbytes for a in outs.values()) // B + 8
    keep = np.arange(B)
    if per_clip * B > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(B, DUMP_LIMIT_BYTES // per_clip, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    outs = {k: v[keep] for k, v in outs.items()}
    outs["clip_index"] = keep.astype(np.float64)
    for name, a in outs.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))


def roofline_pass(args, sess, torch, lib, _lib):
    """Largest launch of the step, timed alone with CUDA events on its stream: the reflect-padded temporal convolution of
    mot_embedding's JointBlock (5 taps, 256->256 over B*1440 rows = 78 % of the embedding FLOPs, 31 % of the step's).
    FLOPs are algorithmic: 2 * rows * (5*256) * 256."""
    import ctypes as C
    peaks, src = load_peaks()
    B = sess.B
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=sess.dev)
    fn = getattr(lib, "mocha_bench_tconv", None)
    if fn is None:
        return None
    rows = B * 60 * 24
    flops = 2.0 * rows * 1280 * 256
    x = torch.randn((rows, 256), device=sess.dev)
    out = torch.empty((rows, 256), device=sess.dev)
    wp, wn = _lib.ptr(sess.ws), sess.ws.numel()
    # Operands (x 189 MB fp32 -> 106 MB bf16 padded copy, out 189 MB) exceed the 126 MB L2, so launches
    # run back to back without a flush; R launches between two events amortise the launch gap.
    R = 10
    times = []
    for i in range(5):
        flush.zero_()
        _lib.check(fn(C.byref(sess.gen.struct), _lib.ptr(x), B, _lib.ptr(out), sess.prec, 1, wp, wn, _lib.stream_ptr()),
                   "mocha_bench_tconv")
        torch.cuda.synchronize()
        e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        e0.record()
        _lib.check(fn(C.byref(sess.gen.struct), _lib.ptr(x), B, _lib.ptr(out), sess.prec, 1, wp, wn, _lib.stream_ptr()),
                   "mocha_bench_tconv")
        e1.record()
        _lib.check(fn(C.byref(sess.gen.struct), _lib.ptr(x), B, _lib.ptr(out), sess.prec, 1 + R, wp, wn, _lib.stream_ptr()),
                   "mocha_bench_tconv")
        e2.record()
        torch.cuda.synchronize()
        if i >= 2:
            times.append((e1.elapsed_time(e2) - e0.elapsed_time(e1)) / R)   # (stage + (1+R) gemm) - (stage + 1 gemm)
    ms = sum(times) / len(times)
    achieved = flops / (ms * 1e-3) / 1e12
    if sess.prec == _lib.MOCHA_BF16:
        peak = peaks.get("bf16_tflops", 1590.0)
        return {"kernel": "tc_gemm2_kernel<LinearEpiT<1>> (cta_group::2, 256x256 pair tiles, TMA-store epilogue): mot_embedding "
                          "JointBlock temporal conv (5 taps, 256->256) as a TMA-shifted implicit GEMM on tcgen05 "
                          "(largest launch of the step, 31 % of its FLOPs)",
                "bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                # dram__bytes_read.sum + dram__bytes_write.sum of this launch at 128 clips from the `ncu --set full` capture
                # kept under profiles/ (algorithmic: 106 MB padded bf16 operand + 189 MB fp32 output of this stand-alone entry)
                "traffic": (101463040 + 135415040) * (B / 128.0), "traffic_unit": "B/launch",
                "traffic_source": "profiles/r01_ncu_tconv_pair_tc_gemm2_LinearEpiT1.txt (one ncu --set full capture, not re-measured per run)",
                "peak_source": src + " (burst: kernel timed alone)", "ms_per_launch": ms, "flops_per_launch": flops}
    return {"kernel": "sgemm_kernel<128,128,8,8> (temporal conv as implicit GEMM, fp32 FFMA)", "bound": "fp32-simt",
            "achieved": achieved, "peak": 80.0, "unit": "TFLOP/s", "frac": achieved / 80.0, "traffic": None,
            "peak_source": "nominal fp32 FFMA", "ms_per_launch": ms, "flops_per_launch": flops}


def kernel_rooflines(sess, torch, lib, _lib):
    """Tensor rooflines of the two kernel families that carry the transformer layers, timed alone (CUDA events, 20
    back-to-back launches) at the step's shapes: the generic tcgen05 GEMM (QKV projection, 11520 x 1536 x 256) and the
    fused block tail (out-projection + FFN of an encoder layer; out-projection + LN + FFN + LN of a CVAE prior layer)."""
    peaks, src = load_peaks()
    peak = peaks["bf16_tflops"]
    dev, R = sess.dev, sess.B * 90
    g = torch.Generator(device=dev).manual_seed(5)
    rn = lambda *s: torch.randn(*s, generator=g, device=dev)
    P = _lib.ptr
    out = []
    # generic GEMM through the exposed dense primitive (bf16 mode)
    A, Wt = rn(R, 256), rn(1536, 256) * 0.06
    W16 = Wt.to(torch.bfloat16)
    _lib.check(lib.mocha_register_bf16_blob(P(Wt), P(W16), Wt.numel()), "register")
    C32 = torch.empty((R, 1536), device=dev)
    wsb = lib.mocha_linear_workspace_bytes(R, 1536, 256, _lib.MOCHA_BF16)
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev)
    ms = timed(torch, lambda: _lib.check(lib.mocha_linear(P(A), P(Wt), None, None, P(C32), R, 1536, 256, 0, _lib.MOCHA_BF16, P(ws),
                                                          ws.numel(), _lib.stream_ptr()), "mocha_linear"), 20)
    fl = 2.0 * R * 1536 * 256
    out.append({"kernel": "cast + tc_gemm2_kernel<LinearEpiT<1>> (CTA pairs; QKV projection shape 11520 x 1536 x 256, fp32 in/out "
                          "through mocha_linear: includes the bf16 cast of A)", "bound": "tensor", "ms_per_launch": ms,
                "achieved": fl / ms / 1e9, "peak": peak, "unit": "TFLOP/s", "frac": fl / ms / 1e9 / peak, "flops_per_launch": fl})
    lib.mocha_register_bf16_blob(P(Wt), None, Wt.numel())
    # fused block tail
    for name, rows, K0, ln, act in (("encoder layer tail (out-proj 512->256 + GELU FFN 256-512-256)", R, 512, False, 2),
                                    ("CVAE prior layer tail (out-proj 256->256 + LN + ReLU FFN + LN)", sess.B * 182, 256, True, 1)):
        A0 = rn(rows, K0).to(torch.bfloat16)
        W0 = (rn(256, K0) * K0 ** -0.5).to(torch.bfloat16)
        W1 = (rn(512, 256) / 16).to(torch.bfloat16)
        W2 = (rn(256, 512) / 22).to(torch.bfloat16)
        b0, b1, b2, R0 = rn(256), rn(512), rn(256), rn(rows, 256)
        g1, be1 = rn(256), rn(256)
        O32 = torch.empty((rows, 256), device=dev)
        O16 = torch.empty((rows, 256), device=dev, dtype=torch.bfloat16)
        call = lambda: _lib.check(lib.mocha_block_tail(P(A0), K0, K0, P(W0), P(b0), P(R0), P(g1) if ln else None, P(be1) if ln else None,
                                                       512, act, P(W1), P(b1), P(W2), P(b2), P(g1) if ln else None,
                                                       P(be1) if ln else None, 1e-5, P(O32), P(O16), rows, _lib.stream_ptr()), "tail")
        ms = timed(torch, call, 20)
        fl = 2.0 * rows * 256 * (K0 + 512 + 512)
        out.append({"kernel": "tail_kernel: " + name, "bound": "tensor (latency-bound: one 128-row tile per CTA, weights streamed "
                    "from L2 through a 96 KB ring)", "ms_per_launch": ms, "achieved": fl / ms / 1e9, "peak": peak, "unit": "TFLOP/s",
                    "frac": fl / ms / 1e9 / peak, "flops_per_launch": fl, "ctas": (rows + 127) // 128})
    for o in out:
        o["peak_source"] = src + " (burst)"
    return out


def hbm_kernels(sess, torch, lib, _lib):
    """Achieved HBM GB/s of the bandwidth-bound kernels at the step's shapes (CUDA events over 20 back-to-back launches;
    bytes are algorithmic: every input read once, every output written once)."""
    import ctypes as C
    peaks, src = load_peaks()
    peak = peaks["hbm_gbs"]
    dev, B = sess.dev, sess.B
    out = []
    names = {0: "embed_graph_agg_mma_kernel (1x1 embed conv + LeakyReLU + joint-graph aggregation on mma.sync TF32 fragments, "
                "bulk-copy row stores)", 1: "pool_graph_agg_kernel",
             2: "add_layernorm_reg_kernel (CVAE prior rows, fp32 + bf16 out)", 3: "graph_agg_kv_pad16_stream_kernel (to_mot)",
             6: "out_conv_affine_kernel (to_mot output layer on mma.sync bf16 + de-normalisation)",
             7: "graph_agg_small_kernel (to_mot body-part graph aggregation)",
             4: "adain_norm_tokens (AdaIN + instance norm, fp32 + bf16 out)", 5: "instance_norm_tokens_v4_kernel (bf16 out)"}
    wp, wn = _lib.ptr(sess.ws), sess.ws.numel()
    for which, name in names.items():
        nbytes = C.c_double(0.0)
        call = lambda r: _lib.check(lib.mocha_bench_hbm_kernel(C.byref(sess.gen.struct), which, B, r, wp, wn, C.byref(nbytes),
                                                               _lib.stream_ptr()), "mocha_bench_hbm_kernel")
        call(2); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); call(20); e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 20
        out.append({"kernel": name, "ms_per_launch": ms, "bytes_per_launch": nbytes.value, "achieved": nbytes.value / ms / 1e6,
                    "peak": peak, "unit": "GB/s", "frac": nbytes.value / ms / 1e6 / peak})
    # kinematics: fk / fk_vel over clip-sized batches (set-up path, SURVEY §8 a17) and the per-frame post-process
    from mocha_sigasia2023_b200 import kinematics as kin, skeleton
    F = 225 * 60 * 16
    par = kin.parents_tensor(skeleton.BONE_PARENTS, dev)
    lrot = torch.randn((F, 25, 4), device=dev); lpos = torch.randn((F, 25, 3), device=dev)
    lvel = torch.randn((F, 25, 3), device=dev); lang = torch.randn((F, 25, 3), device=dev)
    for name, fn, per in (("fk_rows_kernel (thread per skeleton, bulk-copy slabs; 16 clips x 225 windows x 60 frames)", lambda: kin.fk(lrot, lpos, par), 25 * 7 * 4 * 2),
                          ("fk_rows_kernel<WITH_VEL> (fk_vel)", lambda: kin.fk_vel(lrot, lpos, lvel, lang, par), 25 * 13 * 4 * 2)):
        ms = timed(torch, fn, 10)
        out.append({"kernel": name, "ms_per_launch": ms, "bytes_per_launch": F * per, "achieved": F * per / ms / 1e6, "peak": peak,
                    "unit": "GB/s", "frac": F * per / ms / 1e6 / peak})
    ms = timed(torch, lambda: sess.post.step_packed(sess.Y, sess.side, sess.contacts, init=False), 20)
    nb = B * (60 * 24 * 15 * 4 + 4344)
    out.append({"kernel": "post_frame_kernel (warp per clip: latency-bound state machine)", "ms_per_launch": ms, "bytes_per_launch": nb,
                "achieved": nb / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": nb / ms / 1e6 / peak})
    for o in out:
        o["peak_source"] = src
    return out


def fp32_mode_pass(args, dev, torch, workload, lib, precision="fp32"):
    """The same step in a parity mode, for the record, so that the bf16 headline has its reference-precision counterpart
    next to it: "fp32" = every contraction in fp32 FFMA, "tf32x3" = linear layers, temporal convolutions and the attention
    products as split-fp32 (3xTF32) tcgen05 GEMMs; exact fp64 matcher in both."""
    B = args.clips
    sess, *_ = workload.build_session(B, n_db=args.db_rows, precision=precision, device=dev, seed=5)
    inp = workload.step_inputs(B, seed=11)
    sess.step_host(inp["X"], inp["src_hips_vel"], inp["src_rvel"], inp["src_rang"], inp["contacts"], inp["eps"])
    sess.step_host(inp["X"], inp["src_hips_vel"], inp["src_rvel"], inp["src_rang"], inp["contacts"], inp["eps"])
    sess.capture()
    ms = timed(torch, sess.step_device, 10, warm=2)
    label = ("fp32 (FFMA GEMMs, fp64 brute-force matcher)" if precision == "fp32" else
             "tf32x3 (3xTF32 tcgen05 GEMMs for linear layers, temporal convolutions and both attention products; fp32 softmax / "
             "norms, fp64 brute-force matcher)")
    return {"precision": label, "clips": B, "ms_per_step": ms, "value": B / ms * 1e3, "unit": UNIT,
            "tolerance": "1e-4 relative vs the reference (tests/test_gpu_session.py, test_gpu_e2e.py)"}


def second_decode_pass(args, dev, torch, workload):
    """Stated variant (SURVEY §8d, test_fullframework.py:465-472): the frame WITH the reference's second decode - the
    nearest-neighbour ("cm_trans") pose decoded and post-processed next to the CVAE one, the matcher on the critical path.
    The headline step leaves it out (its result is not an output of the characterized motion)."""
    B = args.clips
    sess, *_ = workload.build_session(B, n_db=args.db_rows, precision="bf16", device=dev, seed=5, with_cm_path=True)
    inp = workload.step_inputs(B, seed=11)
    sess.step_host(inp["X"], inp["src_hips_vel"], inp["src_rvel"], inp["src_rang"], inp["contacts"], inp["eps"])
    sess.step_host(inp["X"], inp["src_hips_vel"], inp["src_rvel"], inp["src_rang"], inp["contacts"], inp["eps"])
    sess.capture()
    ms = timed(torch, sess.step_device, 50, warm=5)
    return {"what": "bf16 step with the second (cm_trans) decode + post-process of the matched DB row, as the reference's loop does",
            "clips": B, "ms_per_step": ms, "value": B / ms * 1e3, "unit": UNIT}


def latency_pass(args, dev, torch, workload, precision="fp32", db_rows=None, frames=None):
    """BASELINE config 2: batch-1 streaming, one CUDA graph per frame; per-frame latency with CUDA
    events (H2D of the new window + frame + D2H of the pose inside the timed region)."""
    db_rows = db_rows or args.db_rows
    frames = frames or args.latency_frames
    big = db_rows > 2000
    sess, *_ = workload.build_session(1, n_db=db_rows, precision=precision, device=dev, seed=99,
                                      db_precision="bf16" if big else "fp32", db_batch=256 if big else 64)
    pool = [workload.step_inputs(1, seed=7000 + i) for i in range(8)]
    h = pool[0]
    sess.step_host(h["X"], h["src_hips_vel"], h["src_rvel"], h["src_rang"], h["contacts"], h["eps"])
    h = pool[1]
    sess.step_host(h["X"], h["src_hips_vel"], h["src_rvel"], h["src_rang"], h["contacts"], h["eps"])
    sess.capture()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run(n, do_flush):
        ts = []
        for i in range(n + 10):
            h = pool[i % len(pool)]
            if do_flush:
                flush.zero_()
                torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            sess.step_host(h["X"], h["src_hips_vel"], h["src_rvel"], h["src_rang"], h["contacts"], h["eps"])
            e1.record()
            torch.cuda.synchronize()
            if i >= 10:
                ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2], ts[min(len(ts) - 1, int(len(ts) * 0.99))]

    p50, p99 = run(frames, True)
    w50, w99 = run(frames, False)
    peaks, _ = load_peaks()
    db_bytes = db_rows * 23040 * 4
    rec = {"p50_ms": p50, "p99_ms": p99, "p50_ms_l2_warm": w50, "p99_ms_l2_warm": w99, "frames": frames,
           "precision": precision, "db_rows": db_rows, "budget_ms": 33.3,
           "matcher": "tensor-core coarse + fp64 re-rank" if sess._use_tc else "exact fp64 brute force (streams the fp32 DB rows once per frame)",
           "note": "L2 flushed (256 MB write) before every timed frame for p50_ms; *_l2_warm without flush"}
    if not sess._use_tc:
        rec["db_stream_bytes_per_frame"] = db_bytes
        rec["db_stream_gbs_if_whole_frame_were_the_matcher"] = db_bytes / (p50 * 1e-3) / 1e9
        rec["hbm_peak_gbs"] = peaks["hbm_gbs"]
    del sess
    torch.cuda.empty_cache()
    return rec


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
