"""Drop-in ``Discriminator`` of the GAN step on the sm_100a kernels (SURVEY.md section 8f row 2).

Mirrors climsr/models/discriminator.py:5-46: same constructor, same sub-module / parameter / buffer names (the containers are
the reference's own nn.Sequential of ReflectionPad2d / Conv2d / LeakyReLU / BatchNorm2d and Linear modules, created in the
same order, so ``load_state_dict`` of a reference checkpoint and ``torch.manual_seed`` initialisation behave as before), same
``forward(x) -> (N, 1)`` on 128 x 128 inputs.  The modules are never *called*: forward and backward run

* every 3x3 convolution (stride 1, stride 2, reflection-padded or valid) on the tcgen05 conv kernel - as a same-conv over an
  explicitly reflection-padded NHWC bf16 buffer whose interior (every second interior pixel for stride 2) is the layer's
  output - with bias + LeakyReLU(0.01 / 0.2) fused in the epilogue; input gradients on the same kernel with transposed
  weights, weight gradients on the tcgen05 weight-gradient GEMM;
* padding / stride selection / BatchNorm (batch statistics, normalise-on-load, running-statistics update, backward) / the
  LeakyReLU-derivative gates / flatten / the two Linear layers in the streaming kernels of csrc/disc.cu.

Driven by climsr/task/pl_gan.py:28-61 (four forwards and two backwards per batch; the generator's adversarial loss needs the
gradient w.r.t. the input through frozen discriminator weights - produced here too).  There is no CPU / cuDNN fallback.

Launch overhead: one forward is ~55 small launches, forward + backward ~190, and composed call by call from Python the step was
bound by the host (~11 us per launch).  From the third call with a given batch size on, forward and backward therefore replay
CUDA graphs (``use_cuda_graphs``, default on): every call leases a *slot* - static input / activation / gradient buffers plus the
graphs captured over them - until its backward has run, so D(hr) and D(sr) of one GAN batch live in two slots.  Weight packs
are refreshed outside the graphs (csr_conv2d_pack) whenever the weights change; results are bit-identical to the eager path.
"""
from __future__ import annotations

import ctypes as C
from typing import List

import torch
import torch.nn as nn
from torch import Tensor

from .. import ops
from .._lib import CsrError, View, check, current_stream_ptr, lib
from ._common import DerivedState, f32, flat_grad_views

SLOPE = 0.01            # nn.LeakyReLU() default, discriminator.py:15,23
SLOPE_TAIL = 0.2        # discriminator.py:33


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _gather(src: Tensor, view: View, n: int, pad: int, scale=None, shift=None) -> Tensor:
    dst = torch.empty((n, view.hl + 2 * pad, view.wl + 2 * pad, view.c), dtype=torch.bfloat16, device=src.device)
    check(lib.csr_disc_gather(src.data_ptr(), C.byref(view), n, dst.data_ptr(), pad, _ptr(scale), _ptr(shift), current_stream_ptr()),
          "csr_disc_gather")
    return dst


def _collect(dpad: Tensor, view: View, n: int, pad: int, act, gate_neg: float) -> Tensor:
    g = torch.empty((n, view.hs, view.ws, view.c), dtype=torch.bfloat16, device=dpad.device)
    check(lib.csr_disc_collect(dpad.data_ptr(), C.byref(view), n, pad, _ptr(act), gate_neg, g.data_ptr(), current_stream_ptr()),
          "csr_disc_collect")
    return g


def _conv(p: Tensor, w: Tensor, b: Tensor, slope: float, cache=None) -> Tensor:
    """One conv layer; ``cache`` = (scratch tensor, prepacked flag) from ``Discriminator._packed``."""
    scratch, pre = cache if cache is not None else (None, False)
    if slope:
        return ops.conv2d_nhwc(p, w, b, act="lrelu_slope", act_slope=slope, scratch=scratch, prepacked=pre)
    return ops.conv2d_nhwc(p, w, b, act="none", scratch=scratch, prepacked=pre)


def _conv_t(g: Tensor, w: Tensor, cache=None) -> Tensor:
    """Input gradient of a conv layer (transposed / flipped weights)."""
    scratch, pre = cache if cache is not None else (None, False)
    return ops.conv2d_nhwc(g, w, None, transposed=True, scratch=scratch, prepacked=pre)


def _wgrad(p: Tensor, g: Tensor, w: Tensor, out):
    """Weight / bias gradient of a conv layer into the zeroed views ``out`` = (dw, db): one GEMM launch per layer (job mode of the
    weight-gradient kernel)."""
    return ops.conv2d_wgrad(p, g, tuple(w.shape), dw=out[0], db=out[1])


class _DiscriminatorFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, x, *params):
        need_params = any(p.requires_grad for p in params)
        out, saved, lease = module._forward_saving(x)
        ctx.module, ctx.saved, ctx.lease = module, saved, lease
        ctx.need_param_grads = [p.requires_grad for p in params]
        ctx.need_params = need_params
        ctx.set_materialize_grads(False)
        return out

    @staticmethod
    def backward(ctx, gy):
        n_in = 2 + len(ctx.need_param_grads)
        if gy is None:
            return (None,) * n_in
        if ctx.saved is None:
            raise CsrError("the discriminator's saved activations were released by its first backward; a second backward through the same "
                           "forward (retain_graph=True) is not supported - run the forward again")
        dx, grads = ctx.module._backward_saved(ctx.saved, ctx.lease, gy, ctx.needs_input_grad[1], ctx.need_params)
        ctx.saved = ctx.lease = None
        out = [None, dx]
        for need, gname in zip(ctx.need_param_grads, grads):
            out.append(gname if need else None)
        return tuple(out)


class _Slot:
    """Static buffers + captured graphs of one in-flight discriminator call (see the module docstring)."""

    def __init__(self):
        self.busy = False
        self.x = None           # static input
        self.out = None         # static scores
        self.saved = None       # static saved activations (save slots only)
        self.fwd = None         # torch.cuda.CUDAGraph
        self.bwd = {}           # (need_dx, need_params) -> (graph, gy_static, dx_static, flat_static, grads views)


class _Lease:
    """Marks a slot free again when the autograd context that holds it goes away (backward ran, or the graph was dropped)."""

    def __init__(self, slot):
        self.slot = slot
        slot.busy = True

    def release(self):
        if self.slot is not None:
            self.slot.busy = False
            self.slot = None

    def __del__(self):
        self.release()


class Discriminator(DerivedState, nn.Module):
    _DERIVED = ("_slots", "_calls")
    use_cuda_graphs = True          # replay forward / backward as CUDA graphs from the third call of a kind on
    _EAGER_CALLS = 2                # calls of a kind that run eagerly first (module load, attribute set-up, both calls of a first GAN batch)

    def __init__(self, in_channels=1, out_channels=64, num_conv_block=4):
        super().__init__()
        if in_channels != 1 or out_channels != 64 or num_conv_block != 4:
            # the reference's classifier hard-wires 8192 = 512 * 4 * 4 features (discriminator.py:40): only this shape ever worked
            raise ValueError("climsr_b200 Discriminator supports the reference configuration only: in_channels=1, out_channels=64, num_conv_block=4")
        block = []
        for _ in range(num_conv_block):                      # creation order of discriminator.py:11-27 -> same RNG stream
            block += [nn.ReflectionPad2d(1), nn.Conv2d(in_channels, out_channels, 3), nn.LeakyReLU(), nn.BatchNorm2d(out_channels)]
            in_channels = out_channels
            block += [nn.ReflectionPad2d(1), nn.Conv2d(in_channels, out_channels, 3, 2), nn.LeakyReLU()]
            out_channels *= 2
        out_channels //= 2
        in_channels = out_channels
        block += [nn.Conv2d(in_channels, out_channels, 3), nn.LeakyReLU(0.2), nn.Conv2d(out_channels, out_channels, 3)]
        self.feature_extraction = nn.Sequential(*block)
        self.avgpool = nn.AdaptiveAvgPool2d((512, 512))      # never called in the reference either (discriminator.py:38,42-46)
        self.classification = nn.Sequential(nn.Linear(8192, 100), nn.Linear(100, 1))

    # ------------------------------------------------------------------ packed-weight cache
    def _packed(self, conv: nn.Conv2d, transposed: bool):
        """(scratch, True): the layer's packed bf16 weight tiles, re-packed (csr_conv2d_pack, outside any graph) only when the
        weights changed - the four forwards and two backwards of a GAN batch (pl_gan.py:28-61) see at most two weight versions.
        Keyed like the generator's pack cache (``weights_key``).  The scratch tensor of a layer is reallocated only when its
        device changes, so captured graphs that read it stay valid across weight updates."""
        scratch, pre, new = self._layer_pack(conv, transposed, pack=True)
        if new:
            self.__dict__["_slots"] = {}                      # new scratch storage: graphs captured over the old one are stale
        return scratch, pre

    def _refresh_packs(self, transposed: bool) -> None:
        stages, conv4, conv5, _, _ = self._layers()
        for conv_a, _, conv_b in stages:
            self._packed(conv_a, transposed)
            self._packed(conv_b, transposed)
        self._packed(conv4, transposed)
        self._packed(conv5, transposed)

    # ------------------------------------------------------------------ layer table
    def _layers(self):
        fe = self.feature_extraction
        stages = [(fe[i + 1], fe[i + 3], fe[i + 5]) for i in range(0, 28, 7)]
        return stages, fe[28], fe[30], self.classification[0], self.classification[1]

    def _param_order(self) -> List[nn.Parameter]:
        return list(self.parameters())

    def forward(self, x: Tensor) -> Tensor:
        if x.dim() != 4 or x.shape[1] != 1 or x.shape[2] != 128 or x.shape[3] != 128:
            raise ValueError(f"Discriminator expects (N, 1, 128, 128) inputs (the classifier takes 8192 features, discriminator.py:40), got {tuple(x.shape)}")
        if not x.is_cuda:
            raise CsrError("climsr_b200 Discriminator runs on CUDA (sm_100a) only; there is no CPU fallback")
        params = self._param_order()
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in params)):
            return _DiscriminatorFunction.apply(self, x, *params)
        return self._forward_saving(x, save=False)[0]

    # ------------------------------------------------------------------ CUDA-graph slots
    def _check_bn_momentum(self) -> None:
        """A training-mode forward updates the running statistics with a fixed ``momentum``, which graph replays bake into their
        launches.  PyTorch's ``momentum=None`` (cumulative average, factor 1 / num_batches_tracked, a new value every call) is
        rejected instead of silently replaced."""
        if not self.training:
            return
        for i, (_, bn, _) in enumerate(self._layers()[0]):
            if bn.track_running_stats and bn.momentum is None:
                raise CsrError(f"BatchNorm of discriminator stage {i + 1} has momentum=None (cumulative moving average): not supported "
                               "by climsr_b200 Discriminator in training mode - set a float momentum (PyTorch's default is 0.1)")

    def _graph_key(self, x: Tensor, save: bool):
        bn_mode = tuple((self.training or not st[1].track_running_stats, st[1].momentum, st[1].eps) for st in self._layers()[0])
        ptrs = tuple(t.data_ptr() for t in self.parameters()) + tuple(t.data_ptr() for t in self.buffers())
        return (x.device, x.shape[0], save, bn_mode, ptrs)

    def _graphs_usable(self, x: Tensor) -> bool:
        return bool(self.use_cuda_graphs) and not torch.cuda.is_current_stream_capturing()

    def _forward_saving(self, x: Tensor, save: bool = True):
        """(scores, saved, lease).  Eager for the first calls of a kind, then a graph replay on a leased slot."""
        self._check_bn_momentum()
        with torch.cuda.device(x.device):
            self._refresh_packs(False)
            if not self._graphs_usable(x):
                out, saved = self._run_forward(x, save)
                return out, saved, None
            key = self._graph_key(x, save)
            calls = self.__dict__.setdefault("_calls", {})
            calls[key] = calls.get(key, 0) + 1
            if calls[key] <= self._EAGER_CALLS:
                out, saved = self._run_forward(x, save)
                return out, saved, None
            all_slots = self.__dict__.setdefault("_slots", {})
            if key not in all_slots and len(all_slots) >= 6:       # many batch sizes / re-allocated parameters: drop the idle graphs
                for k in [k for k, v in all_slots.items() if not any(sl.busy for sl in v)]:
                    del all_slots[k]
                if len(calls) > 64:
                    calls.clear()
                    calls[key] = self._EAGER_CALLS + 1
            slots = all_slots.setdefault(key, [])
            slot = next((sl for sl in slots if not sl.busy), None)
            if slot is None:
                if len(slots) >= 8:                                # leases that never came back (graphs kept alive by the caller)
                    out, saved = self._run_forward(x, save)
                    return out, saved, None
                slot = _Slot()
                slot.x = torch.empty_like(x, dtype=torch.float32, memory_format=torch.contiguous_format)
                slot.x.copy_(x.detach())
                torch.cuda.current_stream().synchronize()
                slot.fwd = torch.cuda.CUDAGraph()
                with torch.cuda.graph(slot.fwd, capture_error_mode="thread_local"):
                    slot.out, slot.saved = self._run_forward(slot.x, save)
                slots.append(slot)
            else:
                slot.x.copy_(x.detach())
            slot.fwd.replay()
            lease = _Lease(slot) if save else None
            return slot.out.clone(), slot.saved, lease

    def _backward_saved(self, saved, lease, gy: Tensor, need_dx: bool, need_params: bool):
        with torch.cuda.device(gy.device):
            if need_dx or need_params:
                self._refresh_packs(True)
            slot = lease.slot if lease is not None else None
            if slot is None or not self._graphs_usable(gy):
                res = self._run_backward(saved, gy, need_dx, need_params)
                if lease is not None:
                    lease.release()
                return res
            variant = (bool(need_dx), bool(need_params))
            calls = self.__dict__.setdefault("_calls", {})
            ckey = ("bwd", gy.device, saved["n"]) + variant
            calls[ckey] = calls.get(ckey, 0) + 1
            if calls[ckey] <= self._EAGER_CALLS:
                res = self._run_backward(saved, gy, need_dx, need_params)
                lease.release()
                return res
            ent = slot.bwd.get(variant)
            if ent is None:
                gys = torch.empty_like(gy, dtype=torch.float32, memory_format=torch.contiguous_format)
                gys.copy_(gy.detach())
                torch.cuda.current_stream().synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    dx, grads, flat = self._run_backward(saved, gys, need_dx, need_params, return_flat=True)
                ent = slot.bwd[variant] = (graph, gys, dx, flat, grads)
            else:
                ent[1].copy_(gy.detach())
            graph, _, dx, flat, grads = ent
            graph.replay()
            # the static buffers are overwritten by the next replay: hand out copies (one for all parameter gradients)
            dx_out = dx.clone() if dx is not None else None
            out = flat_grad_views(grads, gy.device, flat.clone())[1] if flat is not None else grads
            lease.release()
            return dx_out, out

    # ------------------------------------------------------------------ forward
    def _run_forward(self, x: Tensor, save: bool):
        dev = x.device
        n = x.shape[0]
        stages, conv4, conv5, lin0, lin1 = self._layers()
        with torch.cuda.device(dev):
            a0 = ops.nchw_to_nhwc_bf16(x.detach(), 64)                            # (N,128,128,64), channel 0 = the image, the rest zero
            buf, view = a0, View(128, 128, 64, 0, 1, 128, 128)
            scale = shift = None
            saved = {"n": n, "stages": [], "view0": view}
            for conv_a, bn, conv_b in stages:
                c = conv_a.out_channels
                pa = _gather(buf, view, n, 1, scale, shift)
                sa = _conv(pa, f32(conv_a.weight), f32(conv_a.bias), SLOPE, self._packed(conv_a, False))
                va = View(view.hl + 2, view.wl + 2, c, 1, 1, view.hl, view.wl)
                scale = torch.empty(c, dtype=torch.float32, device=dev)
                shift = torch.empty_like(scale)
                mean = torch.empty_like(scale)
                invstd = torch.empty_like(scale)
                nbytes = lib.csr_disc_bn_scratch_bytes(c)
                scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                training = self.training or not bn.track_running_stats
                if training and bn.track_running_stats and bn.momentum is None:
                    self._check_bn_momentum()
                if training and bn.track_running_stats and bn.num_batches_tracked is not None:
                    bn.num_batches_tracked += 1
                check(lib.csr_disc_bn_forward(sa.data_ptr(), C.byref(va), n, f32(bn.weight).data_ptr(), f32(bn.bias).data_ptr(), float(bn.eps),
                                              float(bn.momentum if bn.momentum is not None else 0.0),     # unused without running statistics
                                              _ptr(bn.running_mean if bn.track_running_stats else None),
                                              _ptr(bn.running_var if bn.track_running_stats else None), 1 if training else 0,
                                              scale.data_ptr(), shift.data_ptr(), mean.data_ptr(), invstd.data_ptr(), scratch.data_ptr(), nbytes,
                                              current_stream_ptr()), "csr_disc_bn_forward")
                pb = _gather(sa, va, n, 1, scale, shift)
                sb = _conv(pb, f32(conv_b.weight), f32(conv_b.bias), SLOPE, self._packed(conv_b, False))
                vb = View(va.hl + 2, va.wl + 2, c, 1, 2, va.hl // 2, va.wl // 2)
                if save:
                    saved["stages"].append({"pa": pa, "sa": sa, "va": va, "mean": mean, "invstd": invstd, "pb": pb, "sb": sb, "vb": vb,
                                            "bn_training": training})
                buf, view, scale, shift = sb, vb, None, None
            p4 = _gather(buf, view, n, 0)                                          # valid convs: no padding
            s4 = _conv(p4, f32(conv4.weight), f32(conv4.bias), SLOPE_TAIL, self._packed(conv4, False))
            v4 = View(view.hl, view.wl, 512, 1, 1, view.hl - 2, view.wl - 2)
            p5 = _gather(s4, v4, n, 0)
            s5 = _conv(p5, f32(conv5.weight), f32(conv5.bias), 0.0, self._packed(conv5, False))
            v5 = View(v4.hl, v4.wl, 512, 1, 1, v4.hl - 2, v4.wl - 2)
            k = 512 * v5.hl * v5.wl
            feats = torch.empty((n, k), dtype=torch.float32, device=dev)
            check(lib.csr_disc_flatten(s5.data_ptr(), C.byref(v5), n, feats.data_ptr(), current_stream_ptr()), "csr_disc_flatten")
            y1 = torch.empty((n, lin0.out_features), dtype=torch.float32, device=dev)
            check(lib.csr_linear_forward(feats.data_ptr(), f32(lin0.weight).data_ptr(), f32(lin0.bias).data_ptr(), y1.data_ptr(), n, k,
                                         lin0.out_features, current_stream_ptr()), "csr_linear_forward")
            y2 = torch.empty((n, lin1.out_features), dtype=torch.float32, device=dev)
            check(lib.csr_linear_forward(y1.data_ptr(), f32(lin1.weight).data_ptr(), f32(lin1.bias).data_ptr(), y2.data_ptr(), n, lin0.out_features,
                                         lin1.out_features, current_stream_ptr()), "csr_linear_forward")
        if save:
            saved.update({"p4": p4, "s4": s4, "v4": v4, "p5": p5, "v5": v5, "feats": feats, "y1": y1, "last_view": view})
        return y2, (saved if save else None)

    # ------------------------------------------------------------------ backward
    def _run_backward(self, sv, gy: Tensor, need_dx: bool, need_params: bool, return_flat: bool = False):
        dev = gy.device
        n = sv["n"]
        stages, conv4, conv5, lin0, lin1 = self._layers()
        grads = {}
        # every parameter gradient is a view of ONE zeroed buffer (parameters() order): one memset instead of 24, and one copy when a
        # graph replay hands the gradients out
        mods = self._module_order()
        flat = None
        gviews = {}
        if need_params:
            flat, views = flat_grad_views([t for m in mods for t in (m.weight, m.bias)], dev)
            gviews = {m: (views[2 * i], views[2 * i + 1]) for i, m in enumerate(mods)}
        else:                                                     # frozen parameters: BatchNorm backward still writes its two sums
            for m in mods:
                if isinstance(m, nn.BatchNorm2d):
                    t = torch.zeros(2 * m.num_features, dtype=torch.float32, device=dev)
                    gviews[m] = (t[:m.num_features], t[m.num_features:])
        with torch.cuda.device(dev):
            g2 = gy.detach().contiguous().float()
            k0, j0 = lin0.in_features, lin0.out_features
            w1, w0 = f32(lin1.weight), f32(lin0.weight)
            dy1 = torch.empty((n, j0), dtype=torch.float32, device=dev)
            dw1, db1 = gviews[lin1] if need_params else (None, None)
            check(lib.csr_linear_backward(sv["y1"].data_ptr(), w1.data_ptr(), g2.data_ptr(), dy1.data_ptr(), _ptr(dw1), _ptr(db1), n, j0,
                                          lin1.out_features, current_stream_ptr()), "csr_linear_backward")
            dfeat = torch.empty((n, k0), dtype=torch.float32, device=dev)
            dw0, db0 = gviews[lin0] if need_params else (None, None)
            check(lib.csr_linear_backward(sv["feats"].data_ptr(), w0.data_ptr(), dy1.data_ptr(), dfeat.data_ptr(), _ptr(dw0), _ptr(db0), n, k0, j0,
                                          current_stream_ptr()), "csr_linear_backward")
            grads[lin1] = (dw1, db1)
            grads[lin0] = (dw0, db0)
            v5, v4 = sv["v5"], sv["v4"]
            g5 = torch.empty((n, v5.hs, v5.ws, v5.c), dtype=torch.bfloat16, device=dev)
            check(lib.csr_disc_unflatten(dfeat.data_ptr(), C.byref(v5), n, g5.data_ptr(), current_stream_ptr()), "csr_disc_unflatten")
            w5, w4 = f32(conv5.weight), f32(conv4.weight)
            if need_params:
                grads[conv5] = _wgrad(sv["p5"], g5, w5, gviews[conv5])
            dp5 = _conv_t(g5, w5, self._packed(conv5, True))
            g4 = _collect(dp5, v4, n, 0, sv["s4"], SLOPE_TAIL)
            if need_params:
                grads[conv4] = _wgrad(sv["p4"], g4, w4, gviews[conv4])
            dp = _conv_t(g4, w4, self._packed(conv4, True))
            pad_next = 0
            for (conv_a, bn, conv_b), st in zip(reversed(stages), reversed(sv["stages"])):
                c = conv_a.out_channels
                gb = _collect(dp, st["vb"], n, pad_next, st["sb"], SLOPE)
                wb = f32(conv_b.weight)
                if need_params:
                    grads[conv_b] = _wgrad(st["pb"], gb, wb, gviews[conv_b])
                dpb = _conv_t(gb, wb, self._packed(conv_b, True))
                va = st["va"]
                ga = torch.empty((n, va.hs, va.ws, c), dtype=torch.bfloat16, device=dev)
                dgamma, dbeta = gviews[bn]
                gamma = f32(bn.weight)
                if st["bn_training"]:
                    dy = torch.empty((n, va.hl, va.wl, c), dtype=torch.float32, device=dev)
                    nbytes = lib.csr_disc_bn_scratch_bytes(c)
                    scratch = torch.empty(nbytes, dtype=torch.uint8, device=dev)
                    check(lib.csr_disc_bn_backward(dpb.data_ptr(), C.byref(va), n, 1, st["sa"].data_ptr(), SLOPE, gamma.data_ptr(),
                                                   st["mean"].data_ptr(), st["invstd"].data_ptr(), dy.data_ptr(), scratch.data_ptr(), nbytes,
                                                   ga.data_ptr(), dgamma.data_ptr(), dbeta.data_ptr(), current_stream_ptr()), "csr_disc_bn_backward")
                else:
                    raise CsrError("backward through an eval-mode BatchNorm is not implemented (the reference's GAN step trains in train() mode)")
                grads[bn] = (dgamma, dbeta)
                wa = f32(conv_a.weight)
                if need_params:
                    grads[conv_a] = _wgrad(st["pa"], ga, wa, gviews[conv_a])
                is_first = conv_a is stages[0][0]
                if not is_first or need_dx:
                    dp = _conv_t(ga, wa, self._packed(conv_a, True))
                pad_next = 1
            dx = None
            if need_dx:
                v0 = View(128, 128, dp.shape[-1], 0, 1, 128, 128)
                gx = _collect(dp, v0, n, 1, None, 1.0)
                dx = ops.nhwc_bf16_to_nchw(gx, 1)
        out = []
        for mod in mods:
            gw, gb_ = grads.get(mod, (None, None))
            out += [gw, gb_]
        if return_flat:
            # parameters() order == the flat buffer's order; missing entries (need_params False) stay None
            return dx, out, flat
        return dx, out

    def _module_order(self):
        """Modules owning (weight, bias) pairs, in ``parameters()`` order."""
        mods = [m for m in self.feature_extraction if isinstance(m, (nn.Conv2d, nn.BatchNorm2d))]
        return mods + [self.classification[0], self.classification[1]]
