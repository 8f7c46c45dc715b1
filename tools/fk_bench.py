"""GB/s of the batched FK kernels at the window-feature-extraction size (16 clips x 225 windows x 60 frames skeletons)."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from mocha_sigasia2023_b200 import kinematics as kin, skeleton  # noqa: E402


def timed(fn, n):
    fn(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    dev = "cuda"
    F = 225 * 60 * 16
    par = kin.parents_tensor(skeleton.BONE_PARENTS, dev)
    lrot = torch.randn((F, 25, 4), device=dev); lpos = torch.randn((F, 25, 3), device=dev)
    lvel = torch.randn((F, 25, 3), device=dev); lang = torch.randn((F, 25, 3), device=dev)
    out = {"skeletons": F}
    for name, fn, per in (("fk", lambda: kin.fk(lrot, lpos, par), 25 * 7 * 4 * 2),
                          ("fk_vel", lambda: kin.fk_vel(lrot, lpos, lvel, lang, par), 25 * 13 * 4 * 2)):
        ms = timed(fn, 20)
        out[name] = {"ms": round(ms, 4), "GB/s": round(F * per / ms / 1e6, 1)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
