"""Kernel times of the bf16 decoder stage, launch by launch (torch.profiler, CUDA activities).

    CUDA_LAUNCH_BLOCKING=1 python tools/decoder_launches.py [--clips 128] [--reps 20]

Runs the Generator's decoder on seeded [clips, 90, 256] tokens of this tree's build (synthetic weights, default config)
and prints, for each launch of one call in launch order, the median over `reps` profiled calls in microseconds.
The kernels trigger their dependents' launch early (programmatic dependent launch), so without CUDA_LAUNCH_BLOCKING=1 a
kernel's profiled time includes its wait for the previous one; with it, each launch runs alone.
"""
import argparse
import os
import re
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from mocha_sigasia2023_b200 import weights  # noqa: E402
from mocha_sigasia2023_b200.model import Generator  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--clips", type=int, default=128)
    ap.add_argument("--reps", type=int, default=20)
    a = ap.parse_args()
    cfg = weights.DEFAULT_MODEL_CFG
    g = Generator(cfg, precision="bf16")
    g.load_state_dict(weights.generator_state_dict(1777, cfg), strict=True)
    g = g.to("cuda").eval()
    n = cfg["nbody"] * (cfg["nframes"] // cfg["temporal_patch_size"])
    gen = torch.Generator(device="cpu").manual_seed(5)
    src = torch.randn((a.clips, n, cfg["decoder_dim"]), generator=gen).cuda()
    sty = torch.randn((a.clips, n, cfg["decoder_dim"]), generator=gen).cuda()
    for _ in range(3):
        g.decoder(src, sty)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(a.reps):
            g.decoder(src, sty)
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                 and "emcpy" not in e.name and "emset" not in e.name), key=lambda e: e.time_range.start)
    per = len(ev) // a.reps
    assert per * a.reps == len(ev), f"{len(ev)} kernel events over {a.reps} calls"
    print(f"{torch.cuda.get_device_name()} | {a.clips} clips | {per} launches per decoder call | median of {a.reps} calls")
    total = 0.0
    for i in range(per):
        t = statistics.median(ev[r * per + i].time_range.elapsed_us() for r in range(a.reps))
        total += t
        name = re.sub(r"\(anonymous namespace\)::|mocha::|void ", "", ev[i].name)
        print(f"{i:3d} {t:8.1f} us  {name[:110]}")
    print(f"sum of kernel times {total:.1f} us")


if __name__ == "__main__":
    main()
