"""Drop-in ESRGANGenerator backed by the sm_100a kernels of libclimsr_b200.so.

Mirrors climsr/models/esrgan.py:57-102 of the reference: same constructor signature (stray kwargs such as the
Hydra key ``scale_factor`` are swallowed, conf/generator/default.yaml:3), same sub-module / parameter names and
OIHW fp32 shapes (so Lightning checkpoints and ``load_state_dict`` work unchanged), same default initialisation
(the parameter containers are plain nn.Conv2d created in the reference's order, so torch.manual_seed(s) gives
bit-identical initial weights), same ``forward(x, elev, mask) -> (N, 1, 4h, 4w)``.

The nn.Conv2d modules are never *called*: forward() hands the fp32 master weights to csr_pack_weights (bf16 UMMA
tiles, re-packed only when a parameter's version counter changes) and runs the whole generator through
csr_plan_forward on torch's current CUDA stream.  There is no eager / CPU fallback.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn
from torch import Tensor

from .._lib import CsrError, NetDesc, check, current_stream_ptr, lib
from ._common import DerivedState, _reg_post_hook, _SRCNNParams, check_generator_inputs, f32, weights_key


class _RDBParams(nn.Module):
    """Parameter container with the names of ResidualDenseBlock (esrgan.py:17-27)."""

    def __init__(self, nf: int = 64, gc: int = 32, bias: bool = True):
        super().__init__()
        self.conv1 = nn.Conv2d(nf, gc, 3, 1, 1, bias=bias)
        self.conv2 = nn.Conv2d(nf + gc, gc, 3, 1, 1, bias=bias)
        self.conv3 = nn.Conv2d(nf + 2 * gc, gc, 3, 1, 1, bias=bias)
        self.conv4 = nn.Conv2d(nf + 3 * gc, gc, 3, 1, 1, bias=bias)
        self.conv5 = nn.Conv2d(nf + 4 * gc, nf, 3, 1, 1, bias=bias)


class _RRDBParams(nn.Module):
    """Names of ResidualInResidualDenseBlock (esrgan.py:41-48)."""

    def __init__(self, nf: int, gc: int = 32):
        super().__init__()
        self.RDB1 = _RDBParams(nf, gc)
        self.RDB2 = _RDBParams(nf, gc)
        self.RDB3 = _RDBParams(nf, gc)


class ESRGANGenerator(DerivedState, nn.Module):
    _DERIVED = ("_packed", "_packed_key", "_plans", "_packed_bwd", "_packed_bwd_key", "_ordered_cache", "_seg_cache", "_goff_cache",
                "_train_plan", "_grad_sync")

    def __init__(self, in_channels: int = 3, out_channels: int = 3, nf: int = 64, nb: int = 23, gc: int = 32,
                 scaling_factor: int = 4, **kwargs):
        super().__init__()
        self.scale_factor = scaling_factor
        self.in_channels, self.out_channels, self.nf, self.nb, self.gc = in_channels, out_channels, nf, nb, gc
        if out_channels != 1:
            # the reference's own tail hard-wires 1+1+1 channels (esrgan.py:87,100), so only 1 ever worked there too
            raise ValueError("ESRGANGenerator: out_channels must be 1 (SRCNN tail takes cat([out, elev, mask]))")
        if scaling_factor != 4 or nf != 64 or gc not in (16, 32) or not (1 <= in_channels <= 16):
            raise ValueError("climsr_b200 ESRGANGenerator supports scaling_factor=4, nf=64, gc in {16,32}, 1<=in_channels<=16")
        # same creation order as esrgan.py:72-87 -> same RNG stream -> same default init
        self.conv_first = nn.Conv2d(in_channels, nf, 3, 1, 1, bias=True)
        self.RRDB_trunk = nn.Sequential(*[_RRDBParams(nf=nf, gc=gc) for _ in range(nb)])
        self.trunk_conv = nn.Conv2d(nf, nf, 3, 1, 1, bias=True)
        self.upconv1 = nn.Conv2d(nf, nf, 3, 1, 1, bias=True)
        self.upconv2 = nn.Conv2d(nf, nf, 3, 1, 1, bias=True)
        self.HRconv = nn.Conv2d(nf, nf, 3, 1, 1, bias=True)
        self.conv_last = nn.Conv2d(nf, out_channels, 3, 1, 1, bias=True)
        self.srcnn = _SRCNNParams(in_channels=3, out_channels=out_channels)
        self._desc = NetDesc(in_channels, out_channels, nf, nb, gc, scaling_factor)
        self._reset_derived()

    def _reset_derived(self) -> None:
        self._packed = self._packed_key = self._packed_bwd = self._packed_bwd_key = None
        self._plans = {}
        self._ordered_cache = self._seg_cache = self._goff_cache = self._grad_sync = None
        self._train_plan = None       # plan of the latest training forward: its saved activations belong to a live autograd node
        self._fwd_serial = 0
        self._dirty = False

    def mark_weights_dirty(self) -> None:
        """Call after changing parameters behind autograd's back (``p.data`` updates): the next forward repacks."""
        self._dirty = True

    def _invalidate_packs(self) -> None:
        """The next forward and backward pack, whatever the cache keys say."""
        self._packed_key = self._packed_bwd_key = None

    def _apply(self, fn, *args, **kwargs):
        # .cuda() / .to() / .float(): parameter storage moves, cached pointers and plans of the old device are stale
        out = super()._apply(fn, *args, **kwargs)
        self._ordered_cache = None
        self._invalidate_packs()
        return out

    # ------------------------------------------------------------------ weights
    def _ordered_params(self):
        """(weight, bias) pairs in state_dict order == csr layer order."""
        if self._ordered_cache is not None:
            return self._ordered_cache
        n = lib.csr_num_layers(C.byref(self._desc))
        if n < 0:
            check(n, "csr_num_layers")
        sd = dict(self.named_parameters())
        out = []
        shape = (C.c_int32 * 4)()
        name = C.create_string_buffer(128)
        for i in range(n):
            check(lib.csr_layer_shape(C.byref(self._desc), i, C.byref(shape), name, 128), "csr_layer_shape")
            key = name.value.decode()
            w, b = sd[key + ".weight"], sd[key + ".bias"]
            if tuple(w.shape) != tuple(shape):
                raise CsrError(f"parameter {key}.weight has shape {tuple(w.shape)}, expected {tuple(shape)}")
            out.append((w, b))
        self._ordered_cache = out
        return out

    def packed_weights(self, force: bool = False) -> Tensor:
        """bf16 UMMA weight tiles + fp32 biases; rebuilt when any parameter changed (optimizer step, load_state_dict)."""
        pairs = self._ordered_params()
        dev = pairs[0][0].device
        key = weights_key((p for wb in pairs for p in wb), dev)
        # a module in train() mode without the optimizer hook cannot trust version counters at all
        force = force or self._dirty or (_reg_post_hook is None and self.training)
        if self._packed is not None and key == self._packed_key and not force:
            return self._packed
        if dev.type != "cuda":
            raise CsrError("ESRGANGenerator parameters must live on a CUDA (B200) device; there is no CPU path")
        nbytes = lib.csr_packed_weight_bytes(C.byref(self._desc))
        if self._packed is None or self._packed.device != dev:
            self._packed = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        keep = []
        n = len(pairs)
        wp, bp = (C.c_void_p * n)(), (C.c_void_p * n)()
        for i, (w, b) in enumerate(pairs):
            wc, bc = f32(w), f32(b)
            keep += [wc, bc]
            wp[i], bp[i] = wc.data_ptr(), bc.data_ptr()
        with torch.cuda.device(dev):
            check(lib.csr_pack_weights(C.byref(self._desc), wp, bp, self._packed.data_ptr(), nbytes, current_stream_ptr()),
                  "csr_pack_weights")
        self._packed_key = key
        self._dirty = False
        return self._packed

    def packed_weights_bwd(self, force: bool = False) -> Tensor:
        """Transposed / flipped bf16 tiles for the input-gradient convs; rebuilt when any weight changed."""
        pairs = self._ordered_params()
        dev = pairs[0][0].device
        key = weights_key((p for wb in pairs for p in wb), dev)
        if self._packed_bwd is not None and key == self._packed_bwd_key and not force:
            return self._packed_bwd
        nbytes = lib.csr_packed_weight_bytes_bwd(C.byref(self._desc))
        if self._packed_bwd is None or self._packed_bwd.device != dev:
            self._packed_bwd = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        n = len(pairs)
        keep = []
        wp = (C.c_void_p * n)()
        for i, (w, _) in enumerate(pairs):
            wc = f32(w)
            keep.append(wc)
            wp[i] = wc.data_ptr()
        with torch.cuda.device(dev):
            check(lib.csr_pack_weights_bwd(C.byref(self._desc), wp, self._packed_bwd.data_ptr(), nbytes, current_stream_ptr()),
                  "csr_pack_weights_bwd")
        self._packed_bwd_key = key
        return self._packed_bwd

    # ------------------------------------------------------------------ plan cache
    def _plan(self, n: int, h: int, w: int, dev: torch.device, train: bool = False):
        key = (n, h, w, dev, train)
        hit = self._plans.get(key)
        if hit is not None:
            self._plans[key] = self._plans.pop(key)      # most recently used last
            return hit[0]
        nbytes = (lib.csr_train_workspace_bytes if train else lib.csr_workspace_bytes)(C.byref(self._desc), n, h, w)
        ws = torch.empty(nbytes + 1024, dtype=torch.uint8, device=dev)
        base = (ws.data_ptr() + 1023) // 1024 * 1024
        plan = C.c_void_p()
        with torch.cuda.device(dev):
            create = lib.csr_train_plan_create if train else lib.csr_plan_create
            check(create(C.byref(self._desc), n, h, w, base, nbytes, C.byref(plan)), "csr_plan_create")
        if len(self._plans) >= 4:   # bound the cached workspaces: evict the least recently used plan ...
            for old_key in list(self._plans.keys()):
                old_plan = self._plans[old_key][0]
                if old_plan == self._train_plan and len(self._plans) > 1:
                    continue          # ... but never the one a live autograd node may still run its backward on
                self._evict(old_key)
                break
        self._plans[key] = (plan.value, ws)
        return plan.value

    def _evict(self, key) -> None:
        plan, _ws = self._plans.pop(key)
        if plan == self._train_plan:
            self._train_plan = None
            self._fwd_serial += 1     # a backward of the evicted plan's forward now raises instead of touching freed memory
        if self._seg_cache is not None and self._seg_cache[0][0] == plan:
            self._seg_cache = None
        if self._goff_cache is not None and self._goff_cache[0] == plan:
            self._goff_cache = None
        lib.csr_plan_destroy(plan)

    def set_grad_sync(self, sync) -> None:
        """Data-parallel training: a climsr_b200.parallel.BackwardGradSync makes backward() return gradients that are already
        averaged over the process group, their all-reduce overlapped with the backward kernels."""
        self._grad_sync = sync

    def _backward_segments(self, plan, nseg: int) -> int:
        cache = self._seg_cache
        if cache is not None and cache[0] == (plan, nseg):
            return cache[1]
        n = lib.csr_plan_backward_segments(plan, nseg)
        if n < 0:
            check(n, "csr_plan_backward_segments")
        self._seg_cache = ((plan, nseg), n)
        return n

    def _grad_offsets(self, plan):
        cache = self._goff_cache
        if cache is not None and cache[0] == plan:
            return cache[1]
        n = lib.csr_num_layers(C.byref(self._desc))
        offs = []
        v = C.c_size_t()
        for i in range(n):
            for j in (0, 1):
                check(lib.csr_plan_grad_offset(plan, i, j, C.byref(v)), "csr_plan_grad_offset")
                offs.append(int(v.value))
        self._goff_cache = (plan, offs)
        return offs

    def __del__(self):
        try:
            for p, _t in self.__dict__.get("_plans", {}).values():
                lib.csr_plan_destroy(p)
        except Exception:
            pass

    # ------------------------------------------------------------------ forward
    def forward(self, x: Tensor, elev: Tensor, mask: Tensor) -> Tensor:
        check_generator_inputs(x, elev, mask, self.in_channels, "generator", "ESRGANGenerator")
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            from ..autograd import generator_apply
            return generator_apply(self, x, elev, mask)
        return self._forward_impl(x, elev, mask)

    def _forward_impl(self, x: Tensor, elev: Tensor, mask: Tensor) -> Tensor:
        n, _, h, w = x.shape
        dev = x.device
        xs = x.detach().contiguous().float()
        es = elev.detach().to(dev).contiguous().float()
        ms = mask.detach().to(dev).contiguous().float()
        packed = self.packed_weights()
        plan = self._plan(n, h, w, dev)
        out = torch.empty((n, 1, 4 * h, 4 * w), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib.csr_plan_forward(plan, packed.data_ptr(), xs.data_ptr(), es.data_ptr(), ms.data_ptr(), out.data_ptr(),
                                       current_stream_ptr()), "csr_plan_forward")
        return out
