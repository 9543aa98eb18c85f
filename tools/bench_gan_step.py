"""cfg3 GAN training step (SURVEY.md section 8d): generator AND discriminator on this repo's CUDA path (--disc cuda, default), or the
discriminator as stock PyTorch / cuDNN (--disc torch: the round-1 configuration, kept as the comparison).

One step follows climsr/task/pl_gan.py:28-108 with its two optimizers: (1) sr = G(x); loss_G = 0.01 * L1(sr, hr) +
0.005 * relativistic-average BCE(D(hr), D(sr)) (+ 1.0 * perceptual, DISABLED here: VGG19 weights need a download,
perceptual.py:15) -> backward -> AdamW step of G; (2) sr = G(x) AGAIN (common_step runs per optimizer, pl_gan.py:66) ->
loss_D on sr.detach() -> backward -> AdamW step of D.  Factors / optimizer from conf/experiment/*gan*.yaml and
conf/optimizers/adamw.yaml.  The discriminator below is a plain-PyTorch module with the layer sequence of
climsr/models/discriminator.py:5-46 (eight reflection-padded 3x3 convs, stride 1 / 2 alternating, BatchNorm after the
stride-1 ones, two valid 3x3 convs, Linear 8192 -> 100 -> 1) run under bf16 autocast + channels_last; per-rank BatchNorm
statistics (sync_batchnorm: False).  Multi-GPU: torchrun, bf16 bucketed all-reduce of both parameter sets.

--perceptual cuda adds the 1.0 * perceptual term on this repo's path (climsr_b200.losses.PerceptualLoss, seeded VGG19 weights: hi/lo
bf16 activations on the tcgen05 convs), --perceptual torch the same term as stock PyTorch fp32 with TF32 off (the accuracy-equivalent
cuDNN arm of tools/bench_perceptual.py); the default, off, leaves it out as before.

    python tools/bench_gan_step.py [--batch 16] [--steps 20] [--perceptual off|cuda|torch]
"""
import argparse
import json
import os
import sys

import torch
import torch.distributed as dist
import torch.nn as nn
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "climate-super-resolution_b200"))
from climsr_b200 import losses  # noqa: E402
from climsr_b200.models import ESRGANGenerator  # noqa: E402
from climsr_b200.models.discriminator import Discriminator  # noqa: E402
from climsr_b200.parallel import GradientBucketer, attach_ddp, configure_nccl_for_overlap  # noqa: E402


def make_discriminator(width=64, stages=4):
    layers, cin, cout = [], 1, width
    for _ in range(stages):
        layers += [nn.ReflectionPad2d(1), nn.Conv2d(cin, cout, 3), nn.LeakyReLU(), nn.BatchNorm2d(cout),
                   nn.ReflectionPad2d(1), nn.Conv2d(cout, cout, 3, stride=2), nn.LeakyReLU()]
        cin, cout = cout, cout * 2
    layers += [nn.Conv2d(cin, cin, 3), nn.LeakyReLU(0.2), nn.Conv2d(cin, cin, 3), nn.Flatten(), nn.Linear(8192, 100), nn.Linear(100, 1)]
    return nn.Sequential(*layers)


def relativistic(score_a, score_b, label):
    return F.binary_cross_entropy_with_logits(score_a - score_b.mean(), label)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--disc", default="cuda", choices=["cuda", "torch"])
    ap.add_argument("--perceptual", default="off", choices=["off", "cuda", "torch"])
    args = ap.parse_args()
    world, rank, local = (int(os.environ.get(k, d)) for k, d in (("WORLD_SIZE", "1"), ("RANK", "0"), ("LOCAL_RANK", "0")))
    torch.cuda.set_device(local)
    if world > 1:
        configure_nccl_for_overlap()
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    dev = torch.device("cuda", local)
    torch.manual_seed(rank)
    n, h = args.batch, 32
    G = ESRGANGenerator(4, 1, 64, 11, 16).to(dev).train()
    D = (Discriminator().to(dev) if args.disc == "cuda" else make_discriminator().to(dev).to(memory_format=torch.channels_last)).train()
    g_sync = attach_ddp(G) if world > 1 else None            # generator gradients: exchanged inside its backward
    opt_g = torch.optim.AdamW(G.parameters(), lr=1e-4, weight_decay=1e-4, fused=True)
    opt_d = torch.optim.AdamW(D.parameters(), lr=1e-4, weight_decay=1e-4, fused=True)
    bg = GradientBucketer(G.parameters(), bucket_mb=4.0)
    bd = GradientBucketer(D.parameters(), bucket_mb=8.0)
    x = torch.rand(n, 4, h, h, device=dev) * 2 - 1
    elev = torch.rand(n, 1, 4 * h, 4 * h, device=dev)
    mask = (torch.rand(n, 1, 4 * h, 4 * h, device=dev) > 0.3).float()
    hr = torch.rand(n, 1, 4 * h, 4 * h, device=dev) * 2 - 1
    real, fake = torch.ones((n, 1), device=dev), torch.zeros((n, 1), device=dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    perc = None
    if args.perceptual != "off":
        sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
        from bench_perceptual import TorchPerceptual
        perc = losses.PerceptualLoss(seed=0).to(dev)
        if args.perceptual == "torch":
            torch.backends.cudnn.allow_tf32 = False
            perc = TorchPerceptual(perc).to(dev)

    def d_scores(a, b):
        if args.disc == "cuda":
            return D(a), D(b)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            return D(a).float(), D(b).float()

    def step(timed):
        if timed:
            ev[0].record()
        # ---- optimizer 0: generator (pl_gan.py:68-82, loss_g :28-49)
        opt_g.zero_grad(set_to_none=True)
        sr = G(x, elev, mask)
        if timed:
            ev[1].record()
        for p_ in D.parameters():                             # Lightning's toggle_optimizer (called BEFORE training_step): only the
            p_.requires_grad_(False)                          # generator's parameters require grad while optimizer 0 is active
        s_real, s_fake = d_scores(hr, sr)
        adv = (relativistic(s_fake, s_real, real) + relativistic(s_real, s_fake, fake)) / 2
        loss_g = 0.01 * losses.l1_loss(sr, hr) + 0.005 * adv
        if perc is not None:
            loss_g = loss_g + 1.0 * perc(hr, sr)
        loss_g.backward()
        for p_ in D.parameters():
            p_.requires_grad_(True)
        if world > 1 and g_sync is None:
            bg.allreduce()
        opt_g.step()
        if timed:
            ev[2].record()
        # ---- optimizer 1: discriminator (pl_gan.py:85-96, loss_d :51-61); common_step runs the generator again
        opt_d.zero_grad(set_to_none=True)
        with torch.no_grad():
            sr2 = G(x, elev, mask)
        if timed:
            ev[3].record()
        s_real, s_fake = d_scores(hr, sr2.detach())
        loss_d = (relativistic(s_real, s_fake, real) + relativistic(s_fake, s_real, fake)) / 2
        loss_d.backward()
        if world > 1:
            bd.allreduce()
        opt_d.step()
        if timed:
            ev[4].record()
        return float(loss_g.detach()) if not timed else None

    for _ in range(args.warmup):
        step(False)
    torch.cuda.synchronize()
    acc = [0.0] * 4
    for _ in range(args.steps):
        step(True)
        torch.cuda.synchronize()
        for i in range(4):
            acc[i] += ev[i].elapsed_time(ev[i + 1])
    ms = [a / args.steps for a in acc]
    t = torch.tensor([sum(ms)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        extra = {}
        if perc is not None:
            from bench_perceptual import gpu_identity
            extra = gpu_identity(local)
        print(json.dumps({"workload": f"cfg3 GAN step, batch {n}/GPU of 128x128 HR, Hydra generator (CUDA path) + " +
                                      ("discriminator on the CUDA path" if args.disc == "cuda" else "stock PyTorch discriminator (bf16 autocast, channels_last)") +
                                      (", perceptual term disabled" if perc is None else
                                       f", perceptual term on the {'CUDA path (hi/lo bf16)' if args.perceptual == 'cuda' else 'cuDNN fp32 (TF32 off)'}"),
                          **extra, "n_gpus": world,
                          "ms_per_step_max_over_ranks": float(t), "hr_mpx_s": world * n * 128 * 128 / float(t) / 1e3,
                          "split_ms_rank0": {"G_forward_train": ms[0], "D(hr),D(sr)_fwd + loss_G backward (through D and G) + allreduce + G step": ms[1],
                                             "G_forward_again (common_step of optimizer 1)": ms[2], "D fwd x2 + D backward + allreduce + D step": ms[3]}}))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
