"""Host-side plumbing shared by the native models (ESRGANGenerator, RCAN, Discriminator, the VGG19 of PerceptualLoss): when a weight pack is stale,
the per-layer conv pack cache, derived device state that is never copied or pickled, flat gradient buffers, and the SRCNN tail
the two generators share with their input checks."""
from __future__ import annotations

import copy

import torch
import torch.nn as nn
from torch import Tensor

from .. import ops
from .._lib import CsrError

# Parameter version counters do not see every update: torch.optim.*(fused=True).step() and ``p.data.mul_()`` leave
# ``p._version`` unchanged.  A process-wide optimizer post-step hook therefore bumps this epoch, which is part of every
# pack-cache key: the first forward after ANY optimizer step repacks.  (Direct ``.data`` surgery - EMA, SWA - must call
# ``ESRGANGenerator.mark_weights_dirty()``.)
_WEIGHT_EPOCH = [0]


def _bump_weight_epoch(*_args, **_kwargs) -> None:
    _WEIGHT_EPOCH[0] += 1


try:   # torch >= 2.0
    from torch.optim.optimizer import register_optimizer_step_post_hook as _reg_post_hook
    _reg_post_hook(_bump_weight_epoch)
except Exception:   # pragma: no cover - without the hook every forward of an ESRGANGenerator in train() mode repacks
    _reg_post_hook = None


def weights_key(tensors, device) -> tuple:
    """Cache key of a pack built from ``tensors``: it changes with any tensor's storage or version counter, with every
    optimizer step, and with the device."""
    return (device, _WEIGHT_EPOCH[0], *[(t.data_ptr(), t._version) for t in tensors])


def f32(t: Tensor) -> Tensor:
    """``t`` detached, contiguous and fp32: the layout the C ABI reads."""
    return t.detach().contiguous().float()


class LayerPackCache:
    """Packed bf16 weight tiles of single conv layers: one scratch tensor per (layer module, transposed), valid while its
    ``weights_key`` holds.  A layer's shape is fixed, so its scratch is reallocated only when its device changes."""

    def __init__(self):
        self._entries = {}

    def get(self, conv: nn.Conv2d, transposed: bool = False, force: bool = False, pack: bool = False, weight_fn=None,
            variant=None):
        """(scratch, prepacked, new): the layer's pack scratch, whether it already holds the current weights, and whether the
        scratch was just allocated (graphs captured over an older one are stale).

        force: the caller packs in its conv call (training: fused optimizers update weights without bumping the version
        counters); the entry is left without a key so that the next call that does not force repacks too.
        pack: pack here (csr_conv2d_pack, outside any graph) when the weights changed, so that prepacked is always True.
        weight_fn: the layer executes ``weight_fn(conv.weight)`` (same output channels, any input channels) instead of its own
        weight - the [W | W] weights of a conv over hi/lo activation pairs; ``variant`` names that form in the cache slot.
        The key is still that of conv.weight / conv.bias."""
        w, b = conv.weight, conv.bias
        if weight_fn is not None and transposed:
            raise ValueError("weight_fn applies to forward packs only")
        slot = (conv, transposed) if variant is None else (conv, transposed, variant)
        ent = self._entries.get(slot)
        key = None if force else weights_key((w, b), w.device)
        if key is not None and ent is not None and ent[1] == key:
            return ent[0], True, False
        new = ent is None or ent[0].device != w.device
        ew = weight_fn(w.detach()) if weight_fn is not None and (new or pack) else None
        if new:
            kh, kw = conv.kernel_size
            cin = conv.in_channels if ew is None else ew.shape[1]
            nbytes = ops.conv2d_scratch_bytes(conv.in_channels, conv.out_channels, kh, kw, True) if transposed else \
                ops.conv2d_scratch_bytes(conv.out_channels, cin, kh, kw)
            scratch = torch.empty(max(nbytes, 16), dtype=torch.uint8, device=w.device)
        else:
            scratch = ent[0]
        if pack:
            ops.conv2d_pack(w if ew is None else ew, None if transposed else b, scratch, transposed)
        self._entries[slot] = (scratch, key)
        return scratch, pack, new


class DerivedState:
    """Mixin for modules that hold derived device state (plans, weight packs, captured graphs, pointer caches): the
    attributes named by ``_DERIVED`` and the ``_layer_pack`` cache.  copy.deepcopy (EMA / SWA shadows) and
    torch.save(module) leave them out - copied raw CsrPlan* handles would share workspaces and be freed twice - and the copy
    rebuilds what it needs with ``_reset_derived()``."""

    _DERIVED: tuple = ()

    def _reset_derived(self) -> None:
        pass

    def _layer_pack(self, conv: nn.Conv2d, transposed: bool = False, force: bool = False, pack: bool = False, weight_fn=None,
                    variant=None):
        """``LayerPackCache.get`` on this module's cache, created on first use."""
        cache = self.__dict__.get("_pack_cache")
        if cache is None:
            cache = self.__dict__["_pack_cache"] = LayerPackCache()
        return cache.get(conv, transposed, force, pack, weight_fn, variant)

    def __getstate__(self):
        return {k: v for k, v in self.__dict__.items() if k not in self._DERIVED and k != "_pack_cache"}

    def __setstate__(self, state):
        super().__setstate__(state)
        self._reset_derived()

    def __deepcopy__(self, memo):
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__getstate__().items():
            new.__dict__[k] = copy.deepcopy(v, memo)
        new._reset_derived()
        return new


def flat_grad_views(tensors, device, flat: Tensor = None):
    """(flat, views): one fp32 gradient view per tensor, shaped like it and in the given order, of one flat buffer - a new
    zeroed one (one memset for all gradients), or ``flat`` when given (a copy of a buffer an earlier call laid out)."""
    if flat is None:
        flat = torch.zeros(sum(t.numel() for t in tensors), dtype=torch.float32, device=device)
    views, off = [], 0
    for t in tensors:
        views.append(flat[off:off + t.numel()].view(t.shape))
        off += t.numel()
    return flat, views


class _SRCNNParams(nn.Module):
    """Names of SRCNN (srcnn.py:6-11)."""

    def __init__(self, in_channels: int = 3, out_channels: int = 1):
        super().__init__()
        self.conv1 = nn.Conv2d(in_channels, 64, kernel_size=9, padding=4)
        self.conv2 = nn.Conv2d(64, 32, kernel_size=1, padding=0)
        self.conv3 = nn.Conv2d(32, out_channels, kernel_size=5, padding=2)


def check_generator_inputs(x: Tensor, elev: Tensor, mask: Tensor, in_channels: int, built: str, name: str) -> None:
    """Shapes, channels and device of a generator's ``forward(x, elev, mask)``: ``built`` names the model in the channel
    message, ``name`` in the device message."""
    if x.dim() != 4 or elev.dim() != 4 or mask.dim() != 4:
        raise ValueError("expected x (N,C,h,w), elev (N,1,4h,4w), mask (N,1,4h,4w)")
    n, c, h, w = x.shape
    if c != in_channels:
        raise ValueError(f"x has {c} channels, {built} was built with in_channels={in_channels}")
    hr_shape = (n, 1, 4 * h, 4 * w)
    if tuple(elev.shape) != hr_shape or tuple(mask.shape) != hr_shape:
        raise ValueError(f"elev/mask must have shape {hr_shape}, got {tuple(elev.shape)} / {tuple(mask.shape)}")
    if not x.is_cuda:
        raise CsrError(f"climsr_b200 {name} runs on CUDA (sm_100a) only; there is no CPU fallback")
