"""Training path of the generator: torch.autograd.Function over csr_plan_forward / csr_plan_backward.

Replaces the autograd graph PyTorch would record for ESRGANGenerator.forward (climsr/models/esrgan.py:89-102) when
Lightning calls loss.backward() (climsr/task/pl_generator_pre_training.py:18-33).  Forward runs on a *training plan*
(every dense block keeps its concat buffer, the HR tail keeps its activations); backward runs the input-gradient convs
(same tcgen05 conv kernel, transposed/flipped weight packs) and the weight-gradient GEMMs and hands fp32 gradients of
all 2*L parameters back to autograd, so optimizers / DDP / gradient clipping see ordinary ``.grad`` tensors.
Gradients w.r.t. x, elev and mask are not produced (they are data in the reference's training loop).
"""
from __future__ import annotations

import ctypes as C

import torch

from ._lib import CsrError, check, current_stream_ptr, lib


class GeneratorFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, x, elev, mask, *params):
        n, _, h, w = x.shape
        dev = x.device
        xs = x.detach().contiguous().float()
        es = elev.detach().to(dev).contiguous().float()
        ms = mask.detach().to(dev).contiguous().float()
        # optimizers (fused AdamW in particular) update parameters without bumping the version counters the inference
        # path keys its pack cache on: training always repacks
        packed = module.packed_weights(force=True)
        plan = module._plan(n, h, w, dev, train=True)
        out = torch.empty((n, 1, 4 * h, 4 * w), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib.csr_plan_forward(plan, packed.data_ptr(), xs.data_ptr(), es.data_ptr(), ms.data_ptr(), out.data_ptr(),
                                       current_stream_ptr()), "csr_plan_forward")
        module._fwd_serial += 1
        module._train_plan = plan
        # an optimizer step normally follows: whatever the version counters say, the next inference forward repacks
        module._invalidate_packs()
        ctx.module, ctx.plan, ctx.serial, ctx.dev = module, plan, module._fwd_serial, dev
        ctx.shapes = [tuple(p.shape) for p in params]
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        module = ctx.module
        n_in = 4 + len(ctx.shapes)
        if grad_out is None:
            return (None,) * n_in
        if ctx.needs_input_grad[1]:
            raise CsrError("climsr_b200: the generator does not produce a gradient for its input x (it is data in the reference's "
                           "training loop, climsr/task/pl_generator_pre_training.py:18-33); detach x or clear requires_grad")
        if ctx.serial != module._fwd_serial:
            raise CsrError("climsr_b200: backward() must follow the forward() that produced this output (the training plan keeps "
                           "the saved activations of the latest forward only)")
        dev = ctx.dev
        go = grad_out.detach().contiguous().float()
        packed_bwd = module.packed_weights_bwd(force=True)
        n = len(ctx.shapes) // 2
        # one flat gradient buffer in the plan's layout (csr_plan_grad_offset): written by a single (graph-replayed) call
        flat = torch.empty(lib.csr_plan_grad_floats(ctx.plan), dtype=torch.float32, device=dev)
        sync = getattr(module, "_grad_sync", None)
        with torch.cuda.device(dev):
            if sync is not None and sync.world > 1:
                # segmented backward: each finished gradient slice is all-reduced on a side stream while the next segment runs
                nseg = module._backward_segments(ctx.plan, sync.nseg)
                lo, hi = C.c_size_t(), C.c_size_t()
                pending = []
                for k in range(nseg):
                    check(lib.csr_plan_backward_flat_seg(ctx.plan, packed_bwd.data_ptr(), go.data_ptr(), flat.data_ptr(), k, C.byref(lo),
                                                         C.byref(hi), current_stream_ptr()), "csr_plan_backward_flat_seg")
                    sync.reduce_slice_async(flat, int(lo.value), int(hi.value), pending)
                sync.finish(flat, pending)
            else:
                check(lib.csr_plan_backward_flat(ctx.plan, packed_bwd.data_ptr(), go.data_ptr(), flat.data_ptr(), current_stream_ptr()),
                      "csr_plan_backward_flat")
        offs = module._grad_offsets(ctx.plan)
        grads = []
        for i in range(n):
            for j in (0, 1):
                shape = ctx.shapes[2 * i + j]
                k = int(torch.Size(shape).numel())
                grads.append(flat[offs[2 * i + j]:offs[2 * i + j] + k].view(shape))
        return (None, None, None, None) + tuple(grads)


def generator_apply(module, x, elev, mask):
    pairs = module._ordered_params()
    flat = [p for wb in pairs for p in wb]
    return GeneratorFunction.apply(module, x, elev, mask, *flat)
