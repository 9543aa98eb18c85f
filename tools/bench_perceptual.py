"""VGG19 perceptual loss (pl_gan.py:28-61, one call per generator step on hr and sr): this project's sm_100a path against cuDNN.

Three arms on the same seeded weights (climsr_b200.losses.PerceptualLoss(seed=0)) and inputs (a smooth hr field, sr = hr + sigma N(0,1)):
  cuda         PerceptualLoss: hi/lo bf16 activations on the tcgen05 conv kernels (one pass over 2N images)
  cudnn_fp32   vgg19.features[:35] as stock PyTorch fp32 with TF32 off (the accuracy-equivalent baseline; TF32 has a noise floor
               of its own), 1-channel inputs repeated to 3, hr and sr as one batch, F.l1_loss of the halves
  cudnn_bf16   the same under bf16 autocast + channels_last (speed reference; its error is reported next to it)
For each: ms per call (CUDA events after warm-up), host enqueue time per call, relative error against the float64 oracle
(oracle/perceptual.py, on the GPU) at sigma = 0.01, algorithmic and executed TFLOP/s, kernels per call (torch.profiler, and
csr_kernel_launch_count for the cuda arm), and the GPU's name and power limit read in the same run.

    python tools/bench_perceptual.py [--pairs 16] [--size 128] [--iters 30] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "climate-super-resolution_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)
from climsr_b200 import kernel_launch_count  # noqa: E402
from climsr_b200.losses import PerceptualLoss  # noqa: E402
from climsr_b200.perceptual import VGG19_CFG, vgg19_features  # noqa: E402


def gpu_identity(dev=0):
    """Name and power limit of the GPU, read now (the power limit is part of every absolute number measured on it)."""
    name = torch.cuda.get_device_name(dev)
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or r.stderr.strip()
    except Exception as e:      # pragma: no cover - reported, not hidden
        power = f"unavailable ({e})"
    return {"gpu": name, "power_limit_and_max_sm_clock": power}


def vgg_macs(h, w, cin0=3, pair=False):
    """Multiply-accumulates of features[:35] on one h x w image.  pair: as executed on hi/lo pairs (every cin doubled; conv1_1 over
    a 1-channel input has cin0 = 1, so 2 executed channels)."""
    macs, cin = 0, cin0
    for v in VGG19_CFG:
        if v == "M":
            h, w = h // 2, w // 2
            continue
        macs += h * w * (2 * cin if pair else cin) * v * 9
        cin = v
    return macs


class TorchPerceptual(torch.nn.Module):
    """The cuDNN arms: the same weights as stock PyTorch modules.  bf16=True: bf16 autocast + channels_last."""

    def __init__(self, src: PerceptualLoss, bf16: bool = False):
        super().__init__()
        self.features = vgg19_features()
        self.features.load_state_dict(src.features.state_dict())
        self.bf16 = bf16
        if bf16:
            self.features = self.features.to(memory_format=torch.channels_last)

    @torch.no_grad()
    def forward(self, hr, sr):
        n = hr.shape[0]
        x = torch.cat([hr, sr], 0)
        if x.shape[1] == 1:
            x = x.repeat(1, 3, 1, 1)
        if self.bf16:
            with torch.autocast("cuda", dtype=torch.bfloat16):
                f = self.features(x.contiguous(memory_format=torch.channels_last)).float()
        else:
            f = self.features(x)
        return F.l1_loss(f[:n], f[n:])


def smooth(n, h, w, seed):
    import math
    g = torch.Generator().manual_seed(seed)
    yy = torch.linspace(0, 1, h).view(1, 1, h, 1)
    xx = torch.linspace(0, 1, w).view(1, 1, 1, w)
    f = torch.zeros((n, 1, h, w))
    for _ in range(6):
        fy, fx, ph = (torch.rand((n, 1, 1, 1), generator=g) * 6 for _ in range(3))
        f = f + torch.sin(2 * math.pi * (fy * yy + fx * xx) + ph)
    return (f / f.abs().amax(dim=(1, 2, 3), keepdim=True)).float()


def kernels_per_call(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA and "memcpy" not in e.name.lower()
               and "memset" not in e.name.lower())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=16)
    ap.add_argument("--size", type=int, default=128)
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--sigma", type=float, default=0.01)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    from oracle import perceptual as op
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    ident = gpu_identity(0)
    n, s = args.pairs, args.size
    hr = smooth(n, s, s, 1).to(dev)
    sr = hr + args.sigma * torch.randn(hr.shape, generator=torch.Generator().manual_seed(2)).to(dev)
    mine = PerceptualLoss(seed=0).to(dev)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    arms = {"cuda": mine, "cudnn_fp32": TorchPerceptual(mine).to(dev), "cudnn_bf16": TorchPerceptual(mine, bf16=True).to(dev)}
    with torch.no_grad():
        ref = float(op.perceptual_loss({k: v.to(dev) for k, v in mine.state_dict().items()}, hr, sr))
    alg = 2 * n * vgg_macs(s, s, 3) * 2                  # FLOP, 2N images
    exe_pair = 2 * n * vgg_macs(s, s, 1, pair=True) * 2
    res = {"workload": f"VGG19 features[:35] perceptual loss, {n} pairs of {s}x{s} (1-channel hr / sr), one call", **ident,
           "sigma": args.sigma, "oracle_float64": ref, "algorithmic_gflop_per_call": alg / 1e9, "arms": {}}
    for name, m in arms.items():
        fn = lambda m=m: m(hr, sr)          # noqa: E731
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = kernel_launch_count()
        host = 0.0
        e0.record()
        for _ in range(args.iters):
            t0 = time.perf_counter()
            out = fn()
            host += time.perf_counter() - t0
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.iters
        lib_launches = (kernel_launch_count() - l0) / args.iters
        val = float(out)
        exe = exe_pair if name == "cuda" else alg
        res["arms"][name] = {"ms_per_call": ms, "host_enqueue_ms_per_call": 1e3 * host / args.iters, "loss": val,
                             "rel_err_vs_float64": abs(val - ref) / ref, "algorithmic_tflops": alg / (ms * 1e-3) / 1e12,
                             "executed_gflop_per_call": exe / 1e9, "executed_tflops": exe / (ms * 1e-3) / 1e12,
                             "kernels_per_call_profiler": kernels_per_call(fn),
                             "csr_kernel_launch_count_per_call": lib_launches if name == "cuda" else None}
        print(name, json.dumps(res["arms"][name]), flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
