"""Bring-up diagnostics for the tcgen05 conv kernel on a real B200 (run through gpurun, not pytest).

    python tests/gpu_selftest.py            # runs every case in a subprocess (a trapped kernel kills only its case)
    python tests/gpu_selftest.py --case conv_basic --pdl 0

Each case compares the CUDA path with torch CPU fp32 on bf16-rounded operands (oracle side only).
"""
from __future__ import annotations

import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "climate-super-resolution_b200"))


def bf16r(t):
    return t.to(__import__("torch").bfloat16).float()


def ref_conv(x_nchw, w, b, act="none"):
    import torch
    import torch.nn.functional as F
    y = F.conv2d(bf16r(x_nchw).double(), bf16r(w).double(), b.double(), padding=(w.shape[2] // 2, w.shape[3] // 2))
    if act == "lrelu":
        y = F.leaky_relu(y, 0.2)
    elif act == "relu":
        y = F.relu(y)
    return y.float()


def run_conv_case(n, h, w, cin, cout, k, act="none", seed=0, in_c=None, verbose=True, single_tap=None):
    import torch
    from climsr_b200 import ops
    g = torch.Generator().manual_seed(seed)
    in_c = in_c or (cin + 63) // 64 * 64
    x = torch.rand((n, cin, h, w), generator=g) * 2 - 1
    wt = (torch.rand((cout, cin, k, k), generator=g) * 2 - 1) / (cin * k * k) ** 0.5
    if single_tap is not None:
        m = torch.zeros_like(wt)
        dy, dx = single_tap
        m[:, :, dy, dx] = 1
        wt = wt * m
    b = torch.rand((cout,), generator=g) - 0.5
    xin = torch.zeros((n, h, w, in_c), dtype=torch.bfloat16)
    xin[..., :cin] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    # poison unused channels with NaN-free garbage to prove they are never multiplied
    if in_c > cin and cin % 16 == 0:
        xin[..., cin:] = 7.0
    out = ops.conv2d_nhwc(xin.cuda(), wt.cuda(), b.cuda(), act=act)
    torch.cuda.synchronize()
    got = out[..., :cout].float().cpu().permute(0, 3, 1, 2)
    want = ref_conv(x, wt, b, act)
    err = (got - want).abs()
    tol = 2e-2 * max(1.0, float(want.abs().max()))
    ok = bool(err.max() <= tol) and bool(torch.isfinite(got).all())
    if verbose:
        print(f"  conv n{n} {h}x{w} cin{cin} cout{cout} k{k} act={act} tap={single_tap}: max_err {float(err.max()):.4g} "
              f"(ref absmax {float(want.abs().max()):.3g}) finite={bool(torch.isfinite(got).all())} -> {'OK' if ok else 'FAIL'}")
        if not ok:
            bad = (err > tol)
            idx = bad.nonzero()
            print(f"    bad elements: {int(bad.sum())} / {bad.numel()}; first: {idx[:6].tolist()}")
            rows = bad.any(dim=1).any(dim=0)  # (h,w)
            print("    bad pixel map (rows):")
            for r in range(min(h, 24)):
                print("    " + "".join("X" if rows[r, c] else "." for c in range(min(w, 64))))
            ch = bad.any(dim=0).any(dim=1).any(dim=1)
            print("    bad channels:", ch.nonzero().flatten().tolist()[:64])
    return ok


def case_layout():
    import torch
    from climsr_b200 import ops
    x = torch.rand(2, 4, 5, 7) * 2 - 1
    nhwc = ops.nchw_to_nhwc_bf16(x.cuda(), 64)
    back = ops.nhwc_bf16_to_nchw(nhwc, 4).cpu()
    ok = bool((back - bf16r(x)).abs().max() == 0) and bool((nhwc[..., 4:] == 0).all())
    print("  layout roundtrip:", "OK" if ok else "FAIL")
    return ok


def case_conv_basic():
    ok = True
    # one k-step, one tap: the simplest possible MMA (checks instruction/smem descriptors and the epilogue mapping)
    ok &= run_conv_case(1, 8, 14, 16, 16, 1)
    ok &= run_conv_case(1, 8, 14, 64, 64, 1)
    # single taps of a 3x3: exercises the shifted A descriptor start (row shift = dy*SW+dx pixels of 128 B)
    for tap in [(1, 1), (1, 2), (0, 0), (2, 2), (2, 0)]:
        ok &= run_conv_case(1, 8, 14, 16, 16, 3, single_tap=tap)
    ok &= run_conv_case(1, 8, 14, 64, 64, 3)
    return ok


def case_conv_shapes():
    ok = True
    ok &= run_conv_case(2, 16, 16, 64, 16, 3, "lrelu")
    ok &= run_conv_case(2, 16, 16, 80, 16, 3, "lrelu", in_c=128)
    ok &= run_conv_case(2, 16, 16, 128, 64, 3, in_c=128)
    ok &= run_conv_case(1, 33, 45, 64, 64, 3, "lrelu")        # ragged edges, several tiles
    ok &= run_conv_case(1, 64, 64, 64, 64, 3)
    ok &= run_conv_case(1, 20, 40, 4, 64, 3)                   # conv_first (cin padded 4 -> 16)
    ok &= run_conv_case(1, 40, 40, 64, 1, 3)                   # conv_last (ragged cout)
    ok &= run_conv_case(1, 40, 40, 3, 64, 9, "relu")           # srcnn.conv1
    ok &= run_conv_case(1, 40, 40, 64, 32, 1, "relu")          # srcnn.conv2
    ok &= run_conv_case(1, 40, 40, 32, 1, 5)                   # srcnn.conv3 (bf16 out here)
    ok &= run_conv_case(1, 24, 24, 192, 64, 3, in_c=192)       # gc=32 conv5: cout split across two launches
    return ok


def case_conv_epilogues():
    import torch
    from climsr_b200 import ops
    ok = True
    g = torch.Generator().manual_seed(5)
    n, h, w = 1, 12, 20
    x = torch.rand((n, 64, h, w), generator=g) * 2 - 1
    wt = (torch.rand((64, 64, 3, 3), generator=g) * 2 - 1) / 24
    b = torch.rand((64,), generator=g) - 0.5
    r1 = torch.rand((n, 64, h, w), generator=g) * 2 - 1
    r2 = torch.rand((n, 64, h, w), generator=g) * 2 - 1
    to_nhwc = lambda t, c=64: torch.nn.functional.pad(t.permute(0, 2, 3, 1), (0, c - t.shape[1])).to(torch.bfloat16).contiguous().cuda()
    y = ref_conv(x, wt, b)
    want = (y * 0.2 + bf16r(r1)) * 0.2 + bf16r(r2)
    out = ops.conv2d_nhwc(to_nhwc(x), wt.cuda(), b.cuda(), res1=to_nhwc(r1), scale1=0.2, res2=to_nhwc(r2), scale2=0.2)
    got = out.float().cpu().permute(0, 3, 1, 2)
    e = float((got - want).abs().max())
    print(f"  residual epilogue: max_err {e:.4g}", "OK" if e < 3e-2 else "FAIL")
    ok &= e < 3e-2
    # nearest x2 on the input, then conv + lrelu (four sub-pixel phases)
    out = ops.conv2d_nhwc(to_nhwc(x), wt.cuda(), b.cuda(), act="lrelu", in_up2=True)
    got = out.float().cpu().permute(0, 3, 1, 2)
    up = torch.nn.functional.interpolate(bf16r(x), scale_factor=2, mode="nearest")
    want = torch.nn.functional.leaky_relu(torch.nn.functional.conv2d(up, wt, b, padding=1), 0.2)
    e = float((got - want).abs().max())
    print(f"  up2 epilogue: shape {tuple(got.shape)} max_err {e:.4g}", "OK" if e < 3e-2 else "FAIL")
    ok &= e < 3e-2
    # fp32 planar
    w1 = (torch.rand((1, 64, 5, 5), generator=g) * 2 - 1) / 40
    b1 = torch.rand((1,), generator=g)
    out = ops.conv2d_nhwc(to_nhwc(x), w1.cuda(), b1.cuda(), out_mode="f32_planar")
    e = float((out.cpu() - ref_conv(x, w1, b1)).abs().max())
    print(f"  f32 planar epilogue: max_err {e:.4g}", "OK" if e < 1e-3 else "FAIL")
    ok &= e < 1e-3
    # concat-slice store
    buf = torch.zeros((n, h, w, 128), dtype=torch.bfloat16).cuda()
    buf[..., :64] = to_nhwc(x)
    w16 = (torch.rand((16, 64, 3, 3), generator=g) * 2 - 1) / 24
    b16 = torch.rand((16,), generator=g) - 0.5
    ops.conv2d_nhwc(buf, w16.cuda(), b16.cuda(), act="lrelu", out=buf, out_coff=64)
    got = buf[..., 64:80].float().cpu().permute(0, 3, 1, 2)
    e = float((got - ref_conv(x, w16, b16, "lrelu")).abs().max())
    untouched = bool((buf[..., 80:] == 0).all()) and bool((buf[..., :64] == to_nhwc(x)).all())
    print(f"  concat-slice store: max_err {e:.4g} untouched={untouched}", "OK" if e < 3e-2 and untouched else "FAIL")
    ok &= e < 3e-2 and untouched
    return ok


def case_generator(cfg="tiny"):
    import numpy as np
    import torch
    from climsr_b200.models import ESRGANGenerator
    from oracle import generator as og
    from oracle import synth
    if cfg == "tiny":
        in_ch, nb, gc, n, h, w, gain = 4, 1, 16, 2, 16, 24, 1.0
    elif cfg == "hydra":
        in_ch, nb, gc, n, h, w, gain = 4, 11, 16, 2, 16, 16, 1.0
    elif cfg == "hydra_trained":
        in_ch, nb, gc, n, h, w, gain = 4, 11, 16, 2, 16, 16, 1.8
    else:
        in_ch, nb, gc, n, h, w, gain = 4, 23, 32, 1, 12, 12, 1.0
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=0, gain=gain)
    x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=1)
    with torch.no_grad():
        want = og.generator_forward(sd, x, elev, mask)
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc)
    net.load_state_dict(sd)
    net = net.cuda().eval()
    with torch.no_grad():
        got = net(x.cuda(), elev.cuda(), mask.cuda())
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            got = net(x.cuda(), elev.cuda(), mask.cuda())
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / 3
    e = float((got.cpu() - want).abs().max())
    print(f"  generator[{cfg}] out {tuple(got.shape)} ref std {float(want.std()):.4g} max_err {e:.4g} ({dt * 1e3:.2f} ms/fwd)",
          "OK" if e <= 1e-2 else "FAIL")
    return e <= 1e-2


def case_metrics():
    import torch
    from climsr_b200.metrics import masked_val_metrics_raw
    from climsr_b200._lib import METRIC_KEYS
    from oracle import metrics as om
    from oracle import synth
    ok = True
    for (n, H, W) in ((2, 64, 64), (3, 45, 50)):
        g = torch.Generator().manual_seed(0)
        sr = (torch.rand(n, 1, H, W, generator=g) * 2 - 1) * 0.8
        t = synth.make_targets(sr, seed=4)
        mask = (torch.rand(n, 1, H, W, generator=g) > 0.3).float()
        orig = om.denormalized_original(t["hr"], t["min"], t["max"])
        want = om.val_test_step(sr, t["hr"], orig, mask, t["min"], t["max"])
        got = masked_val_metrics_raw(sr.cuda(), t["hr"].cuda(), orig.cuda(), mask.cuda(), t["min"].cuda(), t["max"].cuda()).cpu()
        for i, k in enumerate(METRIC_KEYS):
            ref = float(want["loss"]) if k == "l1_loss" else (float(torch.mean((sr * mask - t["hr"] * mask) ** 2)) if k == "mse_loss" else float(want[k]))
            tol = 0.01 if k == "psnr" else 1e-4 * max(1.0, abs(ref))
            good = abs(float(got[i]) - ref) <= tol
            ok &= good
            if not good:
                print(f"    metric {k}: got {float(got[i]):.6g} want {ref:.6g} FAIL")
        print(f"  metrics n{n} {H}x{W}:", "OK" if ok else "FAIL")
    return ok


CASES = {
    "layout": case_layout,
    "conv_basic": case_conv_basic,
    "conv_shapes": case_conv_shapes,
    "conv_epilogues": case_conv_epilogues,
    "gen_tiny": lambda: case_generator("tiny"),
    "gen_hydra": lambda: case_generator("hydra"),
    "gen_hydra_trained": lambda: case_generator("hydra_trained"),
    "gen_default": lambda: case_generator("default"),
    "metrics": case_metrics,
}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--case", default=None)
    ap.add_argument("--pdl", type=int, default=0, help="programmatic dependent launch (option 1) off / on")
    ap.add_argument("--cases", default=",".join(CASES))
    a = ap.parse_args()
    if a.case:
        from climsr_b200._lib import lib
        lib.csr_set_option(1, a.pdl)
        ok = CASES[a.case]()
        sys.exit(0 if ok else 1)
    summary = []
    for mode in (0, 1):
        for name in a.cases.split(","):
            if mode == 1 and name in ("layout", "metrics"):
                continue
            print(f"== case {name} (PDL {'on' if mode else 'off'})", flush=True)
            try:
                r = subprocess.run([sys.executable, __file__, "--case", name, "--pdl", str(mode)], timeout=300,
                                   capture_output=True, text=True)
                out = (r.stdout + r.stderr).strip().splitlines()
                print("\n".join(out[-60:]))
                summary.append((name, mode, r.returncode))
            except subprocess.TimeoutExpired:
                print("  TIMEOUT")
                summary.append((name, mode, "timeout"))
        if all(rc == 0 for (_, m, rc) in summary if m == mode):
            break   # everything passes with this PDL setting: no need to try the other
    print("== summary")
    for name, mode, rc in summary:
        print(f"  {name:20s} PDL {mode}: {'PASS' if rc == 0 else 'FAIL(' + str(rc) + ')'}")


if __name__ == "__main__":
    main()
