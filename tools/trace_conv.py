"""Per-role pipeline trace of one conv launch (CTA 0): where does a tile's time go?  Debug tool, run on a B200.
The clock stamps are compiled in only on request (they cost ~2 KB of kernel code): build the library with
`CSR_BUILD_TRACE=1 python climate-super-resolution_b200/build.py --force` first."""
import os
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "climate-super-resolution_b200"))
from climsr_b200 import ops  # noqa: E402
from climsr_b200._lib import lib  # noqa: E402


def run(name, n, h, w, cin, cout, k, in_c, act="lrelu", out_coff=0, res=False, in_coff=0):
    x = torch.zeros((n, h, w, in_c), dtype=torch.bfloat16, device="cuda")
    kw = dict(res1=x, scale1=0.2) if res else {}
    if in_coff:
        kw["in_coff"] = in_coff
    wt = torch.rand((cout, cin, k, k), device="cuda") - 0.5
    b = torch.rand((cout,), device="cuda")
    trace = torch.zeros(3 * 64 * 8, dtype=torch.int64, device="cuda")
    out = torch.zeros((n, h, w, max(in_c, 64)), dtype=torch.bfloat16, device="cuda") if cout > 1 else None
    for rep in range(2):
        lib.csr_debug_set_trace(trace.data_ptr())
        if out is not None:
            ops.conv2d_nhwc(x, wt, b, act=act, out=out, out_coff=out_coff, **kw)
        else:
            ops.conv2d_nhwc(x, wt, b, act=act)
        torch.cuda.synchronize()
    lib.csr_debug_set_trace(None)
    if out is not None:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(50):
            ops.conv2d_nhwc(x, wt, b, act=act, out=out, out_coff=out_coff, **kw)
        e1.record()
        torch.cuda.synchronize()
        print(f"== {name}: {e0.elapsed_time(e1) / 50 * 1e3:.1f} us per launch (50 back-to-back, includes host packing)")
    t = trace.cpu().view(3, 64, 8)
    t0 = int(t[0, 0, 0])
    print(f"== {name}: n{n} {h}x{w} cin{cin} cout{cout} k{k}")
    print(" tile | prod: wait_empty_start wait_done | mma: start accempty_ok afull_ok issued | epi: loop_top prefetched accfull_ok math_done bar1 staged bar2 stored")
    for i in range(0, 10):
        if int(t[0, i, 0]) == 0:
            break
        r = lambda v: int(v) - t0  # noqa: E731
        if os.environ.get("CSR_MMA_DETAIL"):
            print(f" {i:4d} | mma: start {r(t[1,i,0])} accempty_ok {r(t[1,i,1])} afull_ok {r(t[1,i,2])} mmas_issued {r(t[1,i,4])} "
                  f"commits_issued {r(t[1,i,5])} synced {r(t[1,i,3])} loop_end {r(t[1,i,6])}")
            continue
        print(f" {i:4d} | {r(t[0,i,0]):8d} {r(t[0,i,1]):8d} | {r(t[1,i,0]):8d} {r(t[1,i,1]):8d} {r(t[1,i,2]):8d} {r(t[1,i,3]):8d} | "
              f"{r(t[2,i,3]):8d} {r(t[2,i,0]):8d} {r(t[2,i,1]):8d} {r(t[2,i,4]):8d} {r(t[2,i,5]):8d} {r(t[2,i,6]):8d} {r(t[2,i,7]):8d} {r(t[2,i,2]):8d}")


if __name__ == "__main__":
    if os.environ.get("CSR_SLOTS"):
        lib.csr_set_option(3, int(os.environ["CSR_SLOTS"]))
    if os.environ.get("CSR_CONV5"):
        run("rdb.conv5+res", 64, 64, 64, 128, 64, 3, 128, act="none", res=True)
        sys.exit(0)
    if os.environ.get("CSR_DENSE"):
        run("dense x-pass 64->64", 64, 64, 64, 64, 64, 3, 128, out_coff=64)
        run("dense conv2 part 16->16", 64, 64, 64, 16, 16, 3, 128, out_coff=80, in_coff=64)
        run("dense conv4 part 48->16", 64, 64, 64, 48, 16, 3, 128, out_coff=112, in_coff=64)
        sys.exit(0)
    if os.environ.get("CSR_ONLY"):
        run("HRconv", 16, 256, 256, 64, 64, 3, 64)
        sys.exit(0)
    run("rdb.conv1", 64, 64, 64, 64, 16, 3, 128, out_coff=64)
    run("rdb.conv4", 64, 64, 64, 112, 16, 3, 128, out_coff=112)
    if os.environ.get("CSR_THIN"):
        sys.exit(0)
    run("rdb.conv5", 64, 64, 64, 128, 64, 3, 128, act="none")
    run("HRconv", 16, 256, 256, 64, 64, 3, 64)
    run("conv_first", 64, 64, 64, 4, 64, 3, 64, act="none")
