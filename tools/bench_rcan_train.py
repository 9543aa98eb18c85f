"""RCAN pre-training step (pl_generator_pre_training.py:18-33 with generator_type="rcan"): sr = G(x, elev, mask), L1(sr, hr),
backward, AdamW step - on this repo's CUDA path and, in the same process, as PyTorch eager (the same parameters through the
functional restatement oracle/rcan.py) under bf16 autocast + channels_last (cuDNN).

Shape: the Hydra depth (conf/generator/rcan.yaml: 10 residual groups x 20 blocks), batch 16 of 32 x 32 LR tiles (128 x 128 HR,
the cfg3 shape).  Reported per step: device-event time, host time to enqueue the step (until the Python loop returns, before
the synchronise), the device-busy time summed from a torch.profiler pass of its own, and the kernel launches this library
made (csr_kernel_launch_count).  The GPU's name and power limit are read in the same run.

    python tools/bench_rcan_train.py [--batch 16] [--steps 20] [--warmup 3] [--out profiles/r03_rcan_train_step.json]
"""
import argparse
import copy
import json
import os
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "climate-super-resolution_b200")):
    sys.path.insert(0, p)
from climsr_b200 import kernel_launch_count, losses  # noqa: E402
from climsr_b200.models.rcan import RCAN  # noqa: E402
from oracle import rcan as orc  # noqa: E402


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001
        out = f"nvidia-smi unavailable ({e})"
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": out}


def forward_flops(net, n, h, w):
    """2 * MACs of every conv of one forward (the CALayer 1x1 convs on pooled vectors included)."""
    total = 0
    for name, m in net.named_modules():
        if isinstance(m, torch.nn.Conv2d):
            kh, kw = m.kernel_size
            if "conv_du" in name:
                hh, ww = 1, 1
            elif name.startswith(("head", "body", "tail.0.0")):
                hh, ww = h, w
            elif name.startswith("tail.0.2"):
                hh, ww = 2 * h, 2 * w
            else:
                hh, ww = 4 * h, 4 * w
            total += 2 * n * hh * ww * m.in_channels * m.out_channels * kh * kw
    return total


def timed(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    l0 = kernel_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    host = (time.perf_counter() - t0) * 1e3 / steps
    torch.cuda.synchronize()
    return {"ms_per_step": e0.elapsed_time(e1) / steps, "host_enqueue_ms_per_step": host,
            "csr_launches_per_step": (kernel_launch_count() - l0) / steps}


def device_busy_ms(step, steps=3):
    from torch.profiler import ProfilerActivity, profile
    step()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step()
        torch.cuda.synchronize()
    us = sum(e.self_device_time_total for e in prof.key_averages() if e.device_type == torch.autograd.DeviceType.CUDA)
    return us / 1e3 / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--lr-size", type=int, default=32)
    ap.add_argument("--groups", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=20)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_rcan_train_step.json"))
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be >= 1")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n, h, w = args.batch, args.lr_size, args.lr_size
    torch.manual_seed(0)
    net = RCAN(n_resgroups=args.groups, n_resblocks=args.blocks, in_channels=3).to(dev).train()
    eager = copy.deepcopy(net).to(memory_format=torch.channels_last)
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.rand((n, 3, h, w), generator=g, device=dev) * 2 - 1
    elev = torch.rand((n, 1, 4 * h, 4 * w), generator=g, device=dev) * 2 - 1
    mask = (torch.rand((n, 1, 4 * h, 4 * w), generator=g, device=dev) > 0.3).float()
    hr = torch.rand((n, 1, 4 * h, 4 * w), generator=g, device=dev) * 2 - 1
    l1 = losses.L1Loss()
    opt = torch.optim.AdamW(net.parameters(), lr=1e-4)
    opt_e = torch.optim.AdamW(eager.parameters(), lr=1e-4)
    sd_e = dict(eager.named_parameters())
    x_cl = x.contiguous(memory_format=torch.channels_last)

    def step_ours():
        loss = l1(net(x, elev, mask), hr)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)

    def step_eager():
        with torch.autocast("cuda", dtype=torch.bfloat16):
            sr = orc.rcan_forward(sd_e, x_cl, elev, mask, args.groups, args.blocks)
        loss = F.l1_loss(sr.float(), hr)
        loss.backward()
        opt_e.step()
        opt_e.zero_grad(set_to_none=True)

    torch.backends.cudnn.benchmark = True
    res = {"workload": f"RCAN {args.groups}x{args.blocks} pre-training step (fwd + L1 + bwd + AdamW), batch {n}, LR {h}x{w}",
           "gpu": gpu_info(), "forward_tflop": forward_flops(net, n, h, w) / 1e12}
    # alternate: ours, eager, ours - the two runs of ours show the spread
    res["ours"] = timed(step_ours, args.steps, args.warmup)
    res["eager_bf16_channels_last"] = timed(step_eager, args.steps, args.warmup)
    res["ours_repeat"] = timed(step_ours, args.steps, 1)
    res["ours"]["device_busy_ms_per_step"] = device_busy_ms(step_ours)
    res["eager_bf16_channels_last"]["device_busy_ms_per_step"] = device_busy_ms(step_eager)
    res["peak_memory_gb"] = torch.cuda.max_memory_allocated() / 1e9
    step_tflop = 3 * res["forward_tflop"]
    for k in ("ours", "ours_repeat", "eager_bf16_channels_last"):
        res[k]["tflops_effective"] = step_tflop / (res[k]["ms_per_step"] / 1e3)
    print(json.dumps(res))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
