"""Parent-vs-branch check for changes that must not alter what the library computes, how many launches it issues, or how fast it runs.

    python tools/ab_compare.py --base DIR [--head DIR] [--reps 3] [--out FILE]

DIR is a checkout of the commit to compare against (for example ``git worktree add DIR HEAD~1``); --head defaults to this tree.
Both trees are built with their own build.py, then every measurement runs in a fresh process that imports one tree's library:

1. launch counts: csr_plan_num_launches / csr_plan_num_backward_ops of inference and training plans for (in, nb, gc) = (4, 11, 16),
   (3, 23, 32), (2, 1, 16) at the cfg2 / cfg4 / cfg3 shapes of bench.py, and the launch-counter delta of one discriminator
   forward + backward, one RCAN training step and one perceptual-loss call;
2. outputs: cfg2 and cfg4 inference (default options), one cfg3 training step with option 25 = 0 (deterministic weight-gradient
   reduction: output and weight gradients bit for bit, bias gradients to the fp32-atomic tolerance 2e-5 * max|ref|), the
   discriminator's scores and input gradient, the RCAN output, the perceptual loss, and single convs and weight gradients at RCAN
   and discriminator shapes (wide ones merged over gridDim.y, job-mode weight gradients).  The base tree runs twice, so the
   report shows the run-to-run spread of the paths that accumulate with atomics next to the base-vs-head difference;
3. host time of csr_conv2d_nhwc (prepacked weights): enqueue time per call over many calls, for discriminator, RCAN and VGG layer shapes;
4. timing: bench.py --workload cfg2, bench.py --mode train --workload cfg3, tools/bench_rcan_train.py and tools/bench_gan_step.py,
   alternating base and head --reps times, with the GPU name and power limit read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

PLAN_NETS = [((4, 11, 16), "cfg2", (64, 64, 64)), ((3, 23, 32), "cfg4", (1, 113, 113)), ((2, 1, 16), "cfg3", (16, 32, 32))]


# ----------------------------------------------------------------------------------------------------------- probe (one tree)
def probe(tree: str, outdir: str) -> None:
    sys.path[:0] = [os.path.join(tree, "climate-super-resolution_b200"), tree, os.path.join(tree, "tools")]
    import ctypes as C
    import time

    import numpy as np
    import torch
    from climsr_b200 import kernel_launch_count
    from climsr_b200._lib import ConvDesc, lib
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.models.discriminator import Discriminator
    from climsr_b200.models.rcan import RCAN
    from climsr_b200.losses import PerceptualLoss
    from oracle import synth

    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    res = {"counts": {}, "host_us_per_conv_call": {}}
    arrays = {}

    def save(name, t):
        arrays[name] = t.detach().float().cpu().numpy()

    # 1. plan launch counts
    for (in_ch, nb, gc), shape, (n, h, w) in PLAN_NETS:
        net = ESRGANGenerator(in_ch, 1, 64, nb, gc).to(dev)
        key = f"in{in_ch}_nb{nb}_gc{gc}@{shape}"
        res["counts"][key + ".infer.num_launches"] = lib.csr_plan_num_launches(net._plan(n, h, w, dev))
        tp = net._plan(n, h, w, dev, train=True)
        res["counts"][key + ".train.num_launches"] = lib.csr_plan_num_launches(tp)
        res["counts"][key + ".train.num_backward_ops"] = lib.csr_plan_num_backward_ops(tp)
        del net
        torch.cuda.empty_cache()

    # 2a. inference outputs, default options
    for name, (in_ch, nb, gc, n, h, w) in {"cfg2": (4, 11, 16, 8, 64, 64), "cfg4": (3, 11, 16, 1, 113, 113)}.items():
        sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=3)
        x, elev, mask = synth.make_inputs(n, in_ch, h, w, seed=4)
        net = ESRGANGenerator(in_ch, 1, 64, nb, gc)
        net.load_state_dict(sd)
        net = net.to(dev).eval()
        with torch.no_grad():
            save(f"infer_{name}", net(x.to(dev), elev.to(dev), mask.to(dev)))
        del net

    # 2b. one cfg3 training step, deterministic weight-gradient reduction
    lib.csr_set_option(25, 0)
    try:
        sd = synth.make_state_dict(4, 1, 64, 11, 16, seed=5)
        x, elev, mask = synth.make_inputs(16, 4, 32, 32, seed=6)
        net = ESRGANGenerator(4, 1, 64, 11, 16)
        net.load_state_dict(sd)
        net = net.to(dev).train()
        out = net(x.to(dev), elev.to(dev), mask.to(dev))
        gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(7)).to(dev)
        (out * gout).sum().backward()
        save("train_cfg3_out", out)
        for k, p in net.named_parameters():
            save(f"train_cfg3_grad.{k}", p.grad)
        del net
    finally:
        lib.csr_set_option(25, 1)

    # 2c. discriminator forward + backward (the GAN step's batch)
    torch.manual_seed(8)
    disc = Discriminator(1, 64, 4).to(dev).train()
    disc.use_cuda_graphs = False                           # count (and compare) the launches themselves, not a graph replay
    xd = (torch.rand((16, 1, 128, 128), generator=torch.Generator().manual_seed(9)) * 2 - 1).to(dev).requires_grad_(True)
    for _ in range(2):                                     # warm the pack caches
        disc(xd).sum().backward()
    xd.grad = None
    disc.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    l0 = kernel_launch_count()
    score = disc(xd)
    score.sum().backward()
    torch.cuda.synchronize()
    res["counts"]["discriminator.fwd_bwd.launches"] = kernel_launch_count() - l0
    save("disc_score", score)
    save("disc_dx", xd.grad)

    # 2d. RCAN training step (bench_rcan_train's workload at batch 4)
    torch.manual_seed(0)
    rc = RCAN(n_resgroups=10, n_resblocks=20, in_channels=3).to(dev).train()
    g = torch.Generator(device=dev).manual_seed(1)
    xr = torch.rand((4, 3, 32, 32), generator=g, device=dev) * 2 - 1
    er = torch.rand((4, 1, 128, 128), generator=g, device=dev) * 2 - 1
    mr = (torch.rand((4, 1, 128, 128), generator=g, device=dev) > 0.3).float()
    for _ in range(2):
        rc(xr, er, mr).abs().mean().backward()
    rc.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    l0 = kernel_launch_count()
    y = rc(xr, er, mr)
    y.abs().mean().backward()
    torch.cuda.synchronize()
    res["counts"]["rcan.train_step.launches"] = kernel_launch_count() - l0
    save("rcan_out", y)

    # 2e. perceptual loss (bench_perceptual's workload)
    pl = PerceptualLoss(seed=0).to(dev)
    hr = torch.rand((16, 1, 128, 128), generator=torch.Generator().manual_seed(10)).to(dev)
    sr = hr + 0.01 * torch.randn(hr.shape, generator=torch.Generator().manual_seed(11)).to(dev)
    with torch.no_grad():
        pl(hr, sr)
        torch.cuda.synchronize()
        l0 = kernel_launch_count()
        loss = pl(hr, sr)
        torch.cuda.synchronize()
    res["counts"]["perceptual.call.launches"] = kernel_launch_count() - l0
    save("perceptual_loss", loss.reshape(1))

    # 2f. single ops at the model shapes, seeded: conv outputs (deterministic) and job-mode weight / bias gradients (fp32 atomics)
    from climsr_b200 import ops
    gs = torch.Generator().manual_seed(12)
    for name, (n, h, w, cin, cout, act, slope) in {
            "conv_rcan_64x64_32x32": (16, 32, 32, 64, 64, "relu", 0.0),
            "conv_rcan_upsampler_64x256_32x32": (16, 32, 32, 64, 256, "none", 0.0),
            "conv_disc_256x512_18x18": (16, 18, 18, 256, 512, "lrelu_slope", 0.01),
            "conv_disc_512x512_10x10": (16, 10, 10, 512, 512, "lrelu_slope", 0.01)}.items():
        xin = (torch.rand((n, h, w, cin), generator=gs) * 2 - 1).to(torch.bfloat16).to(dev)
        wt = ((torch.rand((cout, cin, 3, 3), generator=gs) * 2 - 1) / (3 * cin ** 0.5)).to(dev)
        bt = (torch.rand((cout,), generator=gs) - 0.5).to(dev)
        save(name, ops.conv2d_nhwc(xin, wt, bt, act=act, act_slope=slope))
        g = (torch.rand((n, h, w, cout), generator=gs) * 2 - 1).to(torch.bfloat16).to(dev)
        dw, db = ops.conv2d_wgrad(xin, g, (cout, cin, 3, 3), scale=0.5)
        save(name.replace("conv_", "wgrad_") + ".dw", dw)
        save(name.replace("conv_", "wgrad_") + ".db", db)

    # 3. host time per csr_conv2d_nhwc call (weights prepacked in scratch, as the three models call it)
    stream = torch.cuda.current_stream().cuda_stream
    for name, (n, h, w, cin, cout, act, mode, slope) in {
            "disc_512x512_10x10": (16, 10, 10, 512, 512, 4, 0, 0.01),
            "disc_64x64_130x130": (16, 130, 130, 64, 64, 4, 0, 0.01),
            "rcan_64x64_32x32": (16, 32, 32, 64, 64, 2, 0, 0.0),
            "rcan_upsampler_64x256_32x32": (16, 32, 32, 64, 256, 0, 0, 0.0),
            "vgg_pair_128x128_32x32": (32, 32, 32, 256, 128, 2, 4, 0.0)}.items():
        in_c = (cin + 63) // 64 * 64
        out_c = 2 * cout if mode == 4 else cout
        d = ConvDesc(n, h, w, cin, cout, 3, 3, in_c, 0, out_c, 0, act, mode, 0, 0, 1.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0.2, slope)
        nbytes = lib.csr_conv2d_scratch_bytes(C.byref(d))
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        wt = torch.randn((cout, cin, 3, 3), device=dev) * 0.05
        bt = torch.zeros((cout,), device=dev)
        xin = torch.randn((n, h, w, in_c), device=dev).to(torch.bfloat16)
        yout = torch.empty((n, h, w, out_c), dtype=torch.bfloat16, device=dev)
        assert lib.csr_conv2d_nhwc(C.byref(d), xin.data_ptr(), wt.data_ptr(), bt.data_ptr(), yout.data_ptr(), None, None, None,
                                   scratch.data_ptr(), nbytes, stream) == 0, lib.csr_last_error()
        torch.cuda.synchronize()
        best = 1e9
        for _ in range(5):
            t0 = time.perf_counter()
            for _ in range(200):
                lib.csr_conv2d_nhwc(C.byref(d), xin.data_ptr(), None, None, yout.data_ptr(), None, None, None, scratch.data_ptr(), nbytes, stream)
            best = min(best, (time.perf_counter() - t0) / 200 * 1e6)
            torch.cuda.synchronize()
        res["host_us_per_conv_call"][name] = best

    np.savez(os.path.join(outdir, "arrays.npz"), **arrays)
    with open(os.path.join(outdir, "probe.json"), "w") as f:
        json.dump(res, f, indent=1)


# ----------------------------------------------------------------------------------------------------------- driver
def run(cmd, cwd, timeout=3600):
    p = subprocess.run(cmd, cwd=cwd, capture_output=True, text=True, timeout=timeout)
    if p.returncode:
        raise RuntimeError(f"{' '.join(cmd)} (in {cwd}) exited {p.returncode}:\n{p.stdout[-3000:]}\n{p.stderr[-3000:]}")
    return p.stdout


def last_json(text):
    for line in reversed(text.strip().splitlines()):
        if line.startswith("{"):
            return json.loads(line)
    raise RuntimeError("no JSON line in output:\n" + text[-2000:])


def compare_arrays(a, b):
    import numpy as np
    rows = []
    for k in sorted(set(a.files) | set(b.files)):
        if k not in a.files or k not in b.files:
            rows.append((k, "missing", None, None))
            continue
        x, y = a[k], b[k]
        diff = float(np.max(np.abs(x.astype(np.float64) - y.astype(np.float64)))) if x.size else 0.0
        scale = float(np.max(np.abs(x))) if x.size else 0.0
        rows.append((k, "bitwise" if np.array_equal(x, y, equal_nan=True) else "differs", diff, scale))
    return rows


def gpu_identity():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown (nvidia-smi failed)"


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--base", help="checkout of the commit to compare against")
    ap.add_argument("--head", default=ROOT)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None, help="report file (default: stdout only)")
    ap.add_argument("--probe", nargs=2, metavar=("TREE", "OUTDIR"), help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.probe:
        probe(*args.probe)
        return
    if not args.base:
        ap.error("--base is required")
    trees = {"base": os.path.abspath(args.base), "head": os.path.abspath(args.head)}
    lines = [f"GPU (name, power limit, max SM clock): {gpu_identity()}", "base: the --base checkout, head: the --head tree", ""]

    def emit(s=""):
        print(s, flush=True)
        lines.append(s)

    for t in lines[:-1]:
        print(t)
    for name, tree in trees.items():
        run([sys.executable, os.path.join(tree, "climate-super-resolution_b200", "build.py")], tree)

    tmp = tempfile.mkdtemp(prefix="ab_compare_")
    probes = {}
    for tag, tree in (("base", trees["base"]), ("head", trees["head"]), ("base_again", trees["base"])):
        d = os.path.join(tmp, tag)
        os.makedirs(d)
        run([sys.executable, os.path.abspath(__file__), "--probe", tree, d], tree)
        import numpy as np
        probes[tag] = (json.load(open(os.path.join(d, "probe.json"))), np.load(os.path.join(d, "arrays.npz")))

    emit("== launch counts (base / head)")
    cb, ch = probes["base"][0]["counts"], probes["head"][0]["counts"]
    for k in cb:
        emit(f"{k:55s} {cb[k]:>8} {ch.get(k):>8}  {'same' if cb[k] == ch.get(k) else 'DIFFERENT'}")
    emit()
    emit("== outputs: head vs base, and base vs base (run-to-run spread)   [status, max |diff|, max |base|]")
    hb = compare_arrays(probes["base"][1], probes["head"][1])
    bb = {r[0]: r for r in compare_arrays(probes["base"][1], probes["base_again"][1])}
    for k, st, diff, scale in hb:
        r = bb[k]
        emit(f"{k:60s} head {st:8s} {diff:.3e}   base-again {r[1]:8s} {r[2]:.3e}   scale {scale:.3e}")
    emit()
    emit("== host time per csr_conv2d_nhwc call, us (best of 5 x 200 calls)   base / head")
    hb_t = probes["base"][0]["host_us_per_conv_call"]
    hh_t = probes["head"][0]["host_us_per_conv_call"]
    hb2_t = probes["base_again"][0]["host_us_per_conv_call"]
    for k in hb_t:
        emit(f"{k:30s} base {hb_t[k]:8.2f} / {hb2_t[k]:8.2f}   head {hh_t[k]:8.2f}")
    emit()

    benches = {
        "bench.py cfg2 infer (ms/step)": (["bench.py", "--gpus", "1", "--steps", "20", "--warmup", "3", "--workload", "cfg2", "--no-extras",
                                           "--no-cpu-baseline"], lambda j: j["ms_per_step"]),
        "bench.py cfg3 train (ms/step)": (["bench.py", "--gpus", "1", "--steps", "20", "--warmup", "3", "--mode", "train", "--workload", "cfg3",
                                           "--no-cpu-baseline"], lambda j: j["ms_per_step"]),
        # the host-bound workloads: longer warm-up and windows, so that their spread can resolve a per-call host-time change
        "bench_rcan_train (ms/step)": (["tools/bench_rcan_train.py", "--steps", "60", "--warmup", "15", "--out", os.path.join(tmp, "rcan.json")],
                                       lambda j: j["ours"]["ms_per_step"]),
        "bench_gan_step (ms/step)": (["tools/bench_gan_step.py", "--steps", "100", "--warmup", "15"], lambda j: j["ms_per_step_max_over_ranks"]),
    }
    times = {k: {"base": [], "head": []} for k in benches}
    for rep in range(args.reps):
        for k, (cmd, pick) in benches.items():
            for tag in (("base", "head") if rep % 2 == 0 else ("head", "base")):
                out = run([sys.executable] + cmd, trees[tag])
                times[k][tag].append(pick(last_json(out)))
                print(f"rep {rep} {k} {tag}: {times[k][tag][-1]:.3f}", flush=True)
    emit(f"== timing, alternating base and head, {args.reps} runs each (lower is better): runs, [min, max], median")
    for k, v in times.items():
        b, h = v["base"], v["head"]
        emit(f"{k:32s} base {' '.join(f'{t:8.3f}' for t in b)}  [{min(b):.3f}, {max(b):.3f}] {statistics.median(b):8.3f}   "
             f"head {' '.join(f'{t:8.3f}' for t in h)}  [{min(h):.3f}, {max(h):.3f}] {statistics.median(h):8.3f}")
    emit()
    emit(f"GPU (name, power limit, max SM clock), read again after the timing: {gpu_identity()}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
