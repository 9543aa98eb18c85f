"""A/B timing of kernel options on the cfg2 forward (one process, same clocks): python tools/ab_bench.py"""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "climate-super-resolution_b200"))
from climsr_b200._lib import lib  # noqa: E402
from climsr_b200.models import ESRGANGenerator  # noqa: E402

VARIANTS = {
    "default": {},
    "no_pdl": {1: 0},
    "no_eight_acc": {19: 0},
    "no_narrow_box": {17: 0},
    "no_tall": {18: 0},
}


def run(name, opts, n=64, h=64, w=64, steps=20):
    for k in (1, 17, 18, 19):
        lib.csr_set_option(k, 1)
    for k, v in opts.items():
        lib.csr_set_option(k, v)
    torch.manual_seed(0)
    net = ESRGANGenerator(4, 1, 64, 11, 16).cuda().eval()
    x = torch.rand(n, 4, h, w, device="cuda") * 2 - 1
    e = torch.rand(n, 1, 4 * h, 4 * w, device="cuda")
    m = (torch.rand(n, 1, 4 * h, 4 * w, device="cuda") > 0.3).float()
    with torch.no_grad():
        for _ in range(3):
            net(x, e, m)
        torch.cuda.synchronize()
        best = 1e9
        for rep in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                net(x, e, m)
            e1.record()
            torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1) / steps)
    print(f"{name:14s} {best:8.3f} ms/step", flush=True)


if __name__ == "__main__":
    names = sys.argv[1:] or list(VARIANTS)
    for nm in names:
        run(nm, VARIANTS[nm])
