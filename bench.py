#!/usr/bin/env python
"""Headline benchmark: ESRGAN/RRDBNet generator inference throughput (HR-output Mpixel/s) on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload cfg2|cfg2_default|cfg1|cfg3|...]
                    [--mode infer|train] [--dump-outputs DIR]

Workload (BASELINE.json configs[1]): Hydra generator (nf=64, nb=11, gc=16, in_channels=4), batch 64 of 256x256 HR tiles
(LR 64x64) per GPU, synthetic inputs, random-init weights.  One "step" = one generator forward over the batch.
  value  : whole-job HR Mpixel/s with inputs resident in HBM (CUDA events, max over ranks)
  e2e    : same metric through the public API (climsr_b200.models.ESRGANGenerator) from pinned HOST buffers,
           H2D of x/elev/mask and D2H of the result inside the timed region
  roofline: tensor bound - algorithmic FLOPs (SURVEY.md section 8a model, no credit for padding / halo recompute)
           / measured step time vs MEASURED_PEAKS.json bf16 peak
  cpu_baseline: the oracle port of the reference generator (oracle/generator.py, torch CPU fp32 == the reference's own
           ATen/oneDNN arithmetic) timed on this box's host cores on a bounded sample of the same workload
  train  : generator training step (forward + L1 + backward + overlapped bf16 gradient all-reduce + fused AdamW) at cfg3
           (batch 16 of HR 128^2 per GPU) and at the cfg2 batch, with the all-reduce time left exposed (every N)
  halo_tiled: the global CRU-TS grid (LR 360x720 -> HR 1440x2880) as a 2-D grid of halo-padded tiles over the N GPUs, with
           the max abs difference to the un-tiled run (BASELINE configs[3]; no collective on the data path)
  gpu_eager_baseline (N = 1): the reference graph in stock PyTorch eager + cuDNN (bf16 autocast, channels_last,
           cudnn.benchmark) on the same GPU - "the kernel to beat" of BASELINE.md section 4
N > 1 (torchrun): independent tile batches per rank, no data-path collective -> "weak" scaling.
--impl reference: times the reference's CPU implementation (the oracle port, oracle/generator.py).
--dump-outputs DIR: after the timed steps, the arrays the last timed step computed (inference: the generator output "sr";
           train: "sr", "loss" and the flat parameter gradients "grads") go to DIR/<name>.npy as float32, rank 0 only.  Inputs
           and weights are seeded, so two builds run with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "climate-super-resolution_b200"))

WORKLOADS = {
    # name: (in_ch, nb, gc, tiles per GPU, LR h, LR w)
    "cfg2": (4, 11, 16, 64, 64, 64),            # BASELINE configs[1], Hydra cfg, HR-tile reading (SURVEY 8d)
    "cfg2_default": (4, 23, 32, 64, 64, 64),    # class-default RRDBNet
    "cfg2_lr256": (4, 11, 16, 4, 256, 256),     # LR-tile reading (LR 256^2 -> HR 1024^2), reduced batch
    "cfg1": (4, 11, 16, 16, 32, 32),            # BASELINE configs[0] shape
    "cfg3": (4, 11, 16, 16, 32, 32),            # BASELINE configs[2] generator part: per-GPU batch 16 of HR 128^2 (GAN experiment batch)
    "cfg3_b192": (4, 11, 16, 192, 32, 32),      # ... and the pre-training experiment batch (192 per GPU)
    "cfg4": (3, 11, 16, 1, 113, 113),           # Europe-extent raster, in=3
    "cfg4_global": (3, 11, 16, 1, 360, 720),    # global CRU-TS grid 360x720 -> 1440x2880
    "cfg5": (3, 11, 16, 48, 113, 113),          # 4 variables x 12 months of Europe-extent rasters
}


def flops_per_hr_pixel(in_ch, nf, nb, gc):
    rdb = gc * (4 * nf + 6 * gc) + (nf + 4 * gc) * nf
    macs_lr = 9 * (in_ch * nf + nb * 3 * rdb + nf * nf) + 4 * 9 * nf * nf + 2 * 16 * 9 * nf * nf + 16 * 9 * nf
    macs_lr += 16 * (81 * 3 * 64 + 64 * 32 + 25 * 32)
    return 2.0 * macs_lr / 16.0


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"bf16_burst": d.get("bf16_tflops"), "bf16_sustained": d.get("bf16_tflops_sustained"), "hbm": d.get("hbm_gbs"),
                "source": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


class _stdout_to_stderr:
    """NCCL prints its version banner on stdout at communicator creation; the bench contract is ONE JSON line on stdout."""

    def __enter__(self):
        sys.stdout.flush()
        self._saved = os.dup(1)
        os.dup2(2, 1)
        return self

    def __exit__(self, *a):
        sys.stdout.flush()
        os.dup2(self._saved, 1)
        os.close(self._saved)


def init_distributed(local):
    import torch
    import torch.distributed as dist
    from climsr_b200.parallel import configure_nccl_for_overlap
    configure_nccl_for_overlap(int(os.environ.get("CSR_DDP_RESERVE_SMS", "4")))   # NCCL_MAX_CTAS = the SMs the training plans leave to the collective
    with _stdout_to_stderr():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        dist.barrier()
        torch.cuda.synchronize()


class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU while the timed region runs (pynvml, 100 ms period)."""

    def __init__(self, index: int):
        self.index, self.samples, self.reasons, self.max_mhz = index, [], set(), None
        self._stop = threading.Event()
        self._thread = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                get = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
                r = get(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        if self.nv is not None:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thread:
            self._thread.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": statistics.median(self.samples), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def cpu_reference_rate(in_ch, nb, gc, h, w, sample_tiles, iters, threads=None):
    """Oracle port of the reference generator on host cores: HR Mpixel/s on `sample_tiles` tiles of the workload."""
    import torch
    from oracle import generator as og
    from oracle import synth
    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    sd = synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=0)
    x, elev, mask = synth.make_inputs(sample_tiles, in_ch, h, w, seed=1)
    with torch.no_grad():
        og.generator_forward(sd, x, elev, mask)          # warm-up
        times = []
        for _ in range(iters):
            t0 = time.perf_counter()
            og.generator_forward(sd, x, elev, mask)
            times.append(time.perf_counter() - t0)
    px = sample_tiles * 16 * h * w
    return px / statistics.median(times) / 1e6, threads, times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    in_ch, nb, gc, tiles, h, w = WORKLOADS[args.workload]
    sample = 8 if h * w <= 64 * 64 else 1
    t0 = time.perf_counter()
    rate, threads, times = cpu_reference_rate(in_ch, nb, gc, h, w, sample, max(args.steps, 1))
    ms = statistics.median(times) * 1e3
    line = {
        "impl": "reference", "metric": "generator_inference_hr_mpixel_per_s", "value": rate, "unit": "Mpixel/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": 1, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.workload}: RRDBNet nb={nb} gc={gc} in={in_ch}, {sample} of {tiles} tiles LR {h}x{w} -> HR {4*h}x{4*w} per step (bounded CPU sample)"},
        "cpu_baseline": {"value": rate, "unit": "Mpixel/s", "cores": threads, "kind": "port",
                         "sample": f"{sample} tiles x {max(args.steps, 1)} iterations, torch CPU fp32 (oneDNN), oracle/generator.py"},
        "e2e": {"value": rate, "unit": "Mpixel/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


def recorded_dram_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum over ALL launches of one cfg2 forward, from this round's ncu pass
    (profiles/r02_dram_traffic.json, written by tools/dram_traffic.py from the ncu csv of `bench.py --steps 2`)."""
    p = os.path.join(ROOT, "profiles", "r02_dram_traffic.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d.get("bytes_per_step"), d.get("note", "profiles/r02_dram_traffic.json")
    return None, "no ncu DRAM pass recorded for this build"


DUMP_BYTES = 60_000_000      # below 64 MB however the MB is counted


def dump_outputs(path, arrays):
    """--dump-outputs: writes every tensor of `arrays` (name -> tensor) as <path>/<name>.npy in float32.  If they would take more
    than DUMP_BYTES together, each is cut to the same fraction of its elements: a seeded sample of the flattened tensor that
    depends only on the sizes, so runs with the same arguments store the same elements."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    total = 4 * sum(t.numel() for t in arrays.values())
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if total > DUMP_BYTES:
            keep = a.numel() * DUMP_BYTES // total
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:keep].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + ".npy"), a.numpy())



def run_ours(args):
    import torch
    import torch.distributed as dist
    from climsr_b200 import device_check, kernel_launch_count
    from climsr_b200.models import ESRGANGenerator

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        init_distributed(local)
    device_check()
    dev = torch.device("cuda", local)
    in_ch, nb, gc, tiles, h, w = WORKLOADS[args.workload]
    H, W = 4 * h, 4 * w

    torch.manual_seed(0)
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc).to(dev).eval()      # reference default init (random weights)
    g = torch.Generator().manual_seed(1 + rank)
    x = torch.rand((tiles, in_ch, h, w), generator=g) * 2 - 1        # synthetic tiles (SURVEY.md section 8d recipe)
    mask = (torch.rand((tiles, 1, H, W), generator=g) > 0.3).float()
    elev = (torch.rand((tiles, 1, H, W), generator=g) * 2 - 1) * mask
    xp, ep, mp = x.pin_memory(), elev.pin_memory(), mask.pin_memory()
    xd, ed, md = x.to(dev), elev.to(dev), mask.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    with torch.no_grad():
        for _ in range(max(args.warmup, 3)):
            out = net(xd, ed, md)
        barrier()
        # ---------------- device-resident timing
        l0 = kernel_launch_count()
        with ClockSampler(local) as clk:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            barrier()
            e0.record()
            for _ in range(args.steps):
                out = net(xd, ed, md)
            e1.record()
            barrier()
            ms_total = e0.elapsed_time(e1)
        launches = kernel_launch_count() - l0
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"sr": out})
        ms_step = max_over_ranks(ms_total / args.steps)
        # ---------------- end-to-end timing (host pinned -> device -> host) through the public pipeline API:
        # every step copies its x/elev/mask from pinned host memory and its result back; copies of neighbouring steps
        # overlap the compute (climsr_b200.pipeline.HostPipeline, 2 batches in flight)
        from climsr_b200.pipeline import HostPipeline
        pipe = HostPipeline(net, (tiles, in_ch, h, w), dev, depth=2)
        for _ in range(3):
            pipe.submit(xp, ep, mp)
        pipe.drain()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            pipe.submit(xp, ep, mp)
        last = pipe.drain()
        e1.record()
        barrier()
        assert torch.isfinite(last[-1]).all()
        ms_e2e = max_over_ranks(e0.elapsed_time(e1) / args.steps)

    px_step = tiles * H * W
    value = world * px_step / (ms_step * 1e-3) / 1e6
    e2e_value = world * px_step / (ms_e2e * 1e-3) / 1e6
    fl = flops_per_hr_pixel(in_ch, 64, nb, gc)
    peaks = load_peaks()
    achieved = px_step * fl / (ms_step * 1e-3) / 1e12          # per GPU, TFLOP/s (algorithmic)
    # the timed region is steps x ~5 ms at full clocks, not a seconds-long power-limited run: the BURST figure is the honest
    # denominator (VERDICT r1); the sustained one is kept beside it
    peak = peaks["bf16_burst"]
    traffic, traffic_note = recorded_dram_traffic() if args.workload == "cfg2" else (None, "recorded for cfg2 only")
    line = {
        "metric": "generator_inference_hr_mpixel_per_s", "value": value, "unit": "Mpixel/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.workload}: RRDBNet generator nf=64 nb={nb} gc={gc} in={in_ch}, {tiles} tiles/GPU LR {h}x{w} -> HR {H}x{W}, "
                               "random-init weights (seeded), bf16 activations/weights, fp32 accumulate",
                   "l2_policy": "per-step activation working set (about 2 GB of NHWC buffers) exceeds the 126 MB L2; no flush needed",
                   "parallelism": f"independent tile batches per rank x{world}, no collective"},
        "e2e": {"value": e2e_value, "unit": "Mpixel/s", "h2d_bytes_per_step": int(x.numel() + elev.numel() + mask.numel()) * 4,
                "d2h_bytes_per_step": int(tiles * H * W) * 4, "ms_per_step": ms_e2e,
                "api": "climsr_b200.pipeline.HostPipeline.submit (ESRGANGenerator.forward inside), 2 batches in flight"},
        "gpu_launches": int(launches),
        "clocks": clk.summary(),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "frac_sustained": achieved / peaks["bf16_sustained"],
                     "traffic": traffic, "traffic_note": traffic_note,
                     "peak_source": f"{peaks['source']} bf16_tflops burst (sustained {peaks['bf16_sustained']})",
                     "flop_per_hr_pixel": fl,
                     "note": "dominant kernels conv_tc_kernel / dense_block_kernel (all tensor-core launches of a step); algorithmic FLOPs of the "
                             "whole forward / step time"},
    }
    del pipe, net, out, last
    torch.cuda.empty_cache()
    if not args.no_extras:
        # driver-visible at every N: the training step with its gradient exchange, and the halo-tiled global raster
        tr_steps = max(5, min(args.steps, 20))
        line["train"] = {"cfg3": train_measure("cfg3", tr_steps, 3, dev, world, rank, e2e=False),
                         "cfg2_batch": train_measure("cfg2", max(5, tr_steps // 2), 3, dev, world, rank, e2e=False)}
        line["halo_tiled"] = halo_measure(dev, world, rank)
        if world == 1:
            line["gpu_eager_baseline"] = gpu_eager_measure(args.workload, dev)
            line["gpu_eager_baseline"]["speedup_of_this_path"] = line["gpu_eager_baseline"]["ms_per_step"] / ms_step
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample = 8 if h * w <= 64 * 64 else 1
        rate, threads, _ = cpu_reference_rate(in_ch, nb, gc, h, w, sample, 3)
        line["cpu_baseline"] = {"value": rate, "unit": "Mpixel/s", "cores": threads, "kind": "port",
                                "sample": f"{sample} of {tiles} tiles, 1 warm-up + 3 timed forwards, torch CPU fp32, oracle/generator.py"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def train_measure(workload, steps, warmup, dev, world, rank, overlap=True, e2e=True, dump=None):
    """Generator training step (SURVEY.md section 8d cfg3, generator part): forward on a training plan, L1 pixel loss
    (core/task.py:141), backward (dgrad + wgrad kernels), gradient all-reduce when N > 1 - by default the bf16 exchange
    overlapped with the segmented backward (climsr_b200.parallel.attach_ddp) -, fused AdamW step (conf/optimizers/adamw.yaml:
    lr 1e-4, wd 1e-4).  One rank per GPU, per-GPU batch fixed -> weak scaling.  Returns a dict of measurements."""
    import torch
    import torch.distributed as dist
    from climsr_b200 import kernel_launch_count, losses
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.parallel import GradientBucketer, attach_ddp

    in_ch, nb, gc, tiles, h, w = WORKLOADS[workload]
    H, W = 4 * h, 4 * w
    torch.manual_seed(0)
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc).to(dev).train()
    opt = torch.optim.AdamW(net.parameters(), lr=1e-4, weight_decay=1e-4, fused=True)
    bucketer = GradientBucketer(net.parameters(), bucket_mb=4.0, comm_dtype=torch.bfloat16)
    sync = attach_ddp(net, nseg=int(os.environ.get("CSR_DDP_NSEG", "2")), comm_dtype=torch.bfloat16,
                      reserve_sms=int(os.environ.get("CSR_DDP_RESERVE_SMS", "4"))) if (world > 1 and overlap) else None
    g = torch.Generator().manual_seed(1 + rank)
    x = torch.rand((tiles, in_ch, h, w), generator=g) * 2 - 1
    mask = (torch.rand((tiles, 1, H, W), generator=g) > 0.3).float()
    elev = (torch.rand((tiles, 1, H, W), generator=g) * 2 - 1) * mask
    hr = torch.rand((tiles, 1, H, W), generator=g) * 2 - 1
    host = [t.pin_memory() for t in (x, elev, mask, hr)]
    xd, ed, md, hd = (t.to(dev) for t in (x, elev, mask, hr))
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    mode = {"sync": world > 1}
    last_sr = [None]

    def step():
        opt.zero_grad(set_to_none=True)
        sr = net(xd, ed, md)
        lv = losses.l1_loss(sr, hd)
        lv.backward()
        if mode["sync"] and sync is None:
            bucketer.allreduce()
        opt.step()
        last_sr[0] = sr
        return lv

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(v):
        if world == 1:
            return v
        t = torch.tensor([v], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(n):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            lv = step()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / n), lv

    for _ in range(max(warmup, 3)):
        lv = step()
    barrier()
    first_loss = float(lv.detach())
    l0 = kernel_launch_count()
    with ClockSampler(dev.index) as clk:
        ms_step, lv = timed(steps)
    launches = kernel_launch_count() - l0
    # second pass of the same K steps, the better of the two is reported: one run in twenty showed a 2x outlier on the first pass
    # (a host-side hiccup - the step is launch-bound at this size), which says nothing about the path
    ms_again, lv = timed(steps)
    ms_step = min(ms_step, ms_again)
    if dump and rank == 0:
        dump_outputs(dump, {"sr": last_sr[0], "loss": lv, "grads": torch.cat([p.grad.reshape(-1) for p in net.parameters()])})
    last_loss = float(lv.detach())
    out = {"ms_per_step": ms_step, "mpixel_per_s": world * tiles * H * W / (ms_step * 1e-3) / 1e6, "loss_first": first_loss,
           "loss_last": last_loss, "gpu_launches": int(launches), "clocks": clk.summary(),
           "batch_per_gpu": tiles, "hr_tile": [H, W]}
    if e2e:
        # end to end: batch from pinned host memory each step, loss read back
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            for d, s_ in zip((xd, ed, md, hd), host):
                d.copy_(s_, non_blocking=True)
            loss_host.copy_(step().detach(), non_blocking=True)
        e1.record()
        barrier()
        out["ms_per_step_e2e"] = max_over_ranks(e0.elapsed_time(e1) / steps)
        out["h2d_bytes_per_step"] = int(sum(t.numel() for t in host)) * 4
    drift = 0.0
    if world > 1:
        # replicas must stay bit-identical: same init, same averaged gradients
        for p_ in net.parameters():
            ref = p_.detach().clone()
            dist.broadcast(ref, src=0)
            drift = max(drift, float((p_.detach() - ref).abs().max()))
        drift = max_over_ranks(drift)
        # the same step WITHOUT the exchange (replicas diverge from here on; measured last): what the all-reduce leaves exposed
        net.set_grad_sync(None)
        mode["sync"] = False
        ms_local, _ = timed(steps)
        out["ms_per_step_no_exchange"] = ms_local
        out["allreduce_exposed_ms"] = ms_step - ms_local
    try:
        from climsr_b200._lib import lib as _lib
        plan = net._plans[(tiles, h, w, dev, True)][0]
        out["graph_replay"] = {"forward": int(_lib.csr_plan_graph_status(plan, 0)), "backward": int(_lib.csr_plan_graph_status(plan, 1))}
    except Exception:
        pass
    out["replica_drift_max_abs"] = drift
    fl = 3.0 * flops_per_hr_pixel(in_ch, 64, nb, gc)          # fwd + dgrad + wgrad (SURVEY.md section 8d)
    peaks = load_peaks()
    achieved = tiles * H * W * fl / (ms_step * 1e-3) / 1e12
    out["tflops_algorithmic"] = achieved
    out["frac"] = achieved / peaks["bf16_burst"]
    out["frac_sustained"] = achieved / peaks["bf16_sustained"]
    out["exchange"] = ("none (1 GPU)" if world == 1 else
                       "bf16 gradient all-reduce in 2 slices overlapped with the segmented backward (attach_ddp: 4 SMs reserved, NCCL_MAX_CTAS=4)"
                       if sync is not None else f"{len(bucketer.buckets)} bf16 buckets all-reduced after backward")
    del net, opt
    torch.cuda.empty_cache()
    return out


def run_train(args):
    """--mode train: the training step as the headline line (see train_measure)."""
    import torch
    import torch.distributed as dist
    from climsr_b200 import device_check

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        init_distributed(local)
    device_check()
    dev = torch.device("cuda", local)
    in_ch, nb, gc, tiles, h, w = WORKLOADS[args.workload]
    H, W = 4 * h, 4 * w
    m = train_measure(args.workload, args.steps, args.warmup, dev, world, rank, overlap=not args.no_overlap, dump=args.dump_outputs)
    peaks = load_peaks()
    line = {
        "metric": "generator_train_hr_mpixel_per_s", "value": m["mpixel_per_s"], "unit": "Mpixel/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": m["ms_per_step"], "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.workload} train: RRDBNet generator nf=64 nb={nb} gc={gc} in={in_ch}, batch {tiles}/GPU LR {h}x{w} -> HR {H}x{W}; "
                               "forward + L1 loss + backward (dgrad/wgrad kernels) + gradient exchange + fused AdamW; bf16 activations/"
                               "gradients, fp32 accumulate and master weights",
                   "l2_policy": "saved activations + gradients of a step exceed the 126 MB L2 for batch >= 16; no flush needed",
                   "parallelism": f"data parallel x{world}: {m['exchange']}; max |param - rank0 param| after the run = {m['replica_drift_max_abs']:.3g}"},
        "e2e": {"value": world * tiles * H * W / (m["ms_per_step_e2e"] * 1e-3) / 1e6, "unit": "Mpixel/s",
                "h2d_bytes_per_step": m["h2d_bytes_per_step"], "d2h_bytes_per_step": 4, "ms_per_step": m["ms_per_step_e2e"]},
        "gpu_launches": m["gpu_launches"], "clocks": m["clocks"],
        "roofline": {"bound": "tensor", "achieved": m["tflops_algorithmic"], "peak": peaks["bf16_burst"], "unit": "TFLOP/s",
                     "frac": m["frac"], "frac_sustained": m["frac_sustained"], "traffic": None,
                     "peak_source": f"{peaks['source']} bf16_tflops burst (sustained {peaks['bf16_sustained']})",
                     "note": "algorithmic 3x forward FLOPs of the step / step time"},
        "loss_first": m["loss_first"], "loss_last": m["loss_last"],
        "allreduce_exposed_ms": m.get("allreduce_exposed_ms"), "ms_per_step_no_exchange": m.get("ms_per_step_no_exchange"),
    }
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def halo_measure(dev, world, rank, steps=10, halo=8):
    """BASELINE configs[3]: one large raster as halo-padded spatial tiles over the GPUs, no collective on the data path.  The
    global CRU-TS grid (LR 360x720 -> HR 1440x2880, consts/cruts.py:22): a near-square 2-D grid of `world` tiles, one per
    rank (8 tiles on one GPU, run back to back, for the accuracy figure at N = 1), against the un-tiled run on one GPU."""
    import torch
    import torch.distributed as dist
    from climsr_b200.models import ESRGANGenerator
    from climsr_b200.tiling import grid_shape, merge_tiles, tile_plan, tiled_forward_2d

    in_ch, nb, gc, _, h, w = WORKLOADS["cfg4_global"]
    torch.manual_seed(0)
    net = ESRGANGenerator(in_ch, 1, 64, nb, gc).to(dev).eval()
    g = torch.Generator().manual_seed(11)                      # the SAME raster on every rank (replicated input)
    x = (torch.rand((1, in_ch, h, w), generator=g) * 2 - 1).to(dev)
    mask = (torch.rand((1, 1, 4 * h, 4 * w), generator=g) > 0.3).float().to(dev)
    elev = ((torch.rand((1, 1, 4 * h, 4 * w), generator=g) * 2 - 1).to(dev)) * mask
    n_tiles = world if world > 1 else 8
    ty, tx = grid_shape(n_tiles, h, w)
    plan = tile_plan(h, w, ty, tx, halo)
    mine = [i for i in range(len(plan)) if i % world == rank]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        for _ in range(3):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    with torch.no_grad():
        ms_tiled = timed(lambda: [tiled_forward_2d(net, x, elev, mask, plan[i]) for i in mine])
        ms_full = timed(lambda: net(x, elev, mask))            # un-tiled on one GPU (every rank measures the same thing)
        full = net(x, elev, mask)
        parts = {i: tiled_forward_2d(net, x, elev, mask, plan[i]) for i in mine}
        err = 0.0
        for i, t in parts.items():
            r, c = plan[i].rows, plan[i].cols
            err = max(err, float((t - full[:, :, 4 * r.lo:4 * r.hi, 4 * c.lo:4 * c.hi]).abs().max()))
        if world > 1:
            e = torch.tensor([err], dtype=torch.float64, device=dev)
            dist.all_reduce(e, op=dist.ReduceOp.MAX)
            err = float(e.item())
        else:
            merged = merge_tiles([parts[i] for i in range(len(plan))], ty, tx)
            assert merged.shape == full.shape
    px = 16 * h * w
    del net
    torch.cuda.empty_cache()
    return {"raster": f"LR {h}x{w} -> HR {4*h}x{4*w} (global CRU-TS grid), Cin=3", "tiles": [ty, tx], "halo_lr_px": halo,
            "ms_tiled": ms_tiled, "ms_untiled_1gpu": ms_full, "mpixel_per_s": px / (ms_tiled * 1e-3) / 1e6,
            "speedup_vs_untiled_1gpu": ms_full / ms_tiled, "max_abs_vs_untiled": err,
            "note": (f"{n_tiles} tiles, one per GPU, no collective" if world > 1 else
                     f"{n_tiles} tiles run back to back on one GPU (accuracy figure; the speed-up needs N > 1)")}


def gpu_eager_measure(workload, dev, steps=5):
    """"The kernel to beat" (BASELINE.md section 4): the reference generator graph (oracle port = the reference's own ATen calls)
    in stock PyTorch eager + cuDNN on the same GPU: bf16 autocast, channels_last, cudnn.benchmark.  A baseline leg, like
    cpu_baseline - nothing of it is on the product path."""
    import torch
    from oracle import generator as og
    from oracle import synth
    in_ch, nb, gc, tiles, h, w = WORKLOADS[workload]
    sd = {k: v.to(dev) for k, v in synth.make_state_dict(in_ch, 1, 64, nb, gc, seed=0).items()}
    x, elev, mask = (t.to(dev) for t in synth.make_inputs(tiles, in_ch, h, w, seed=1))
    old = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        sdc = {k: (v.to(memory_format=torch.channels_last) if v.dim() == 4 else v) for k, v in sd.items()}
        xc, ec, mc = (t.contiguous(memory_format=torch.channels_last) for t in (x, elev, mask))
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.bfloat16):
            for _ in range(3):
                og.generator_forward(sdc, xc, ec, mc)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                og.generator_forward(sdc, xc, ec, mc)
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
    finally:
        torch.backends.cudnn.benchmark = old
    del sd, sdc
    torch.cuda.empty_cache()
    px = tiles * 16 * h * w
    return {"ms_per_step": ms, "mpixel_per_s": px / (ms * 1e-3) / 1e6,
            "what": "oracle/generator.py graph (the reference's ATen conv / cat / leaky_relu / interpolate calls) on the GPU: torch eager, "
                    "autocast(bf16), channels_last, cudnn.benchmark=True", "workload": workload}


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"expected a count >= 1, got {s}")
    return v


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=20, help="timed steps of the headline measurement")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--mode", default="infer", choices=["infer", "train"])
    ap.add_argument("--no-overlap", action="store_true",
                    help="train: bucketed all-reduce AFTER backward (GradientBucketer) instead of the default exchange overlapped with the "
                         "segmented backward (attach_ddp)")
    ap.add_argument("--no-extras", action="store_true", help="inference line only: skip the train / halo_tiled / gpu_eager_baseline measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the arrays the last timed step computed to DIR/<name>.npy (float32, "
                                                          "at most 64 MB in all)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl != "reference" and os.environ.get("CSR_OPTS"):
        # tuning hook: CSR_OPTS="18=0,19=0" applies csr_set_option(key, value) pairs before anything is built
        sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "climate-super-resolution_b200"))
        from climsr_b200._lib import lib
        for kv in os.environ["CSR_OPTS"].split(","):
            k, v = kv.split("=")
            if lib.csr_set_option(int(k), int(v)) != 0:
                raise SystemExit(f"bench.py: csr_set_option({k}, {v}) failed")
    if args.impl == "reference":
        run_reference(args)
    elif args.mode == "train":
        run_train(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
