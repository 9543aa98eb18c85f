"""VGG19 perceptual loss of the GAN step on the sm_100a kernels (mirror of ``climsr/losses/perceptual.py``, used as
``perceptual_criterion(hr, sr)`` by climsr/task/pl_gan.py:28-61 and in validation).

The loss is ``mean |f(hr) - f(sr)|`` with ``f = vgg19().features[:35]``: sixteen zero-padded 3x3 convs with ReLU, four 2x2
max pools, and conv5_4 without its ReLU.  It runs without gradient (the reference wraps it in ``torch.no_grad()``).

Precision.  Once sr is close to hr, the loss is a small difference of two large feature maps, and independent bf16
rounding of each image's activations is noise of the same size: at ``sr = hr + 0.002 N(0, 1)`` plain bf16 activations are
~100 % off.  Every activation is therefore held as a hi/lo bf16 pair, ``hi = bf16(v)``, ``lo = bf16(v - hi)``, stored as 2C
channels ``[hi | lo]``; the next conv runs over the 2C channels with weights ``[W | W]``, which computes ``W (hi + lo)`` in
fp32 on the unchanged tcgen05 mainloop (twice the tensor work).  The input gets the pair too.  Weights stay bf16: their
rounding is the same for hr and sr.  DESIGN.md section 10 has the numbers.

Assumptions about the reference (its source is not part of this project): a 1-channel input is repeated to three channels
(executed here as conv1_1 with ``W.sum(1)``), and no ImageNet mean / std normalisation is applied.  Three-channel inputs
are used as they are.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Mapping, Optional, Union

import torch
import torch.nn as nn
from torch import Tensor

from . import ops
from ._lib import ConvDesc, CsrError, check, current_stream_ptr, lib
from .models._common import DerivedState

# vgg19().features: channel counts, "M" = max pool; [:35] ends with conv5_4 (index 34) before its ReLU
VGG19_CFG = (64, 64, "M", 128, 128, "M", 256, 256, 256, 256, "M", 512, 512, 512, 512, "M", 512, 512, 512, 512)
N_FEATURES = 35
_IN_C = 16          # channels per pixel of the converted input: [hi_0..hi_{c-1}, lo_0..lo_{c-1}, 0...]


def vgg19_features() -> nn.Sequential:
    """``torchvision.models.vgg19().features[:35]`` (same module indices, so the same state_dict keys), without torchvision."""
    layers, cin = [], 3
    for v in VGG19_CFG:
        if v == "M":
            layers.append(nn.MaxPool2d(kernel_size=2, stride=2))
        else:
            layers += [nn.Conv2d(cin, v, kernel_size=3, padding=1), nn.ReLU(inplace=True)]
            cin = v
    return nn.Sequential(*layers[:N_FEATURES])


def _pair_weight(w: Tensor) -> Tensor:
    """[W | W] along the input channels: a conv over [hi | lo] channels computes W (hi + lo)."""
    return torch.cat([w, w], 1)


def _pair_weight_gray(w: Tensor) -> Tensor:
    """conv1_1 over a 1-channel input repeated to three channels: W summed over its input channels, then paired."""
    s = w.sum(1, keepdim=True)
    return torch.cat([s, s], 1)


def _features_only(state_dict: Mapping[str, Tensor]) -> dict:
    """A torchvision VGG19 state dict without its ``classifier.*`` entries."""
    return {k: v for k, v in state_dict.items() if not k.startswith("classifier.")}


class PerceptualLoss(DerivedState, nn.Module):
    """``PerceptualLoss(weights)(hr, sr)`` = mean |vgg19.features[:35](hr) - vgg19.features[:35](sr)|, a 0-dim fp32 tensor.

    weights: a torchvision VGG19 state dict (``classifier.*`` keys are ignored) or a path to one saved with ``torch.save``;
    None gives seeded weights (kaiming-normal, fan-out, ReLU gain, zero bias - torchvision's own init - from
    ``torch.Generator().manual_seed(seed)``).  Nothing is downloaded.  The parameters are frozen (requires_grad False) and
    live in ``features``, an nn.Sequential with torchvision's indices, so ``features.{i}.weight`` are VGG19 keys and
    ``load_state_dict`` takes a torchvision state dict too.  Move the module to the inputs' device (``.cuda()``).

    forward(hr, sr): both (N, C, H, W), C 1 or 3, H and W >= 16, on the same CUDA device.  hr and sr go through the network
    as one batch of 2N images.  The result never requires grad."""

    def __init__(self, weights: Optional[Union[str, os.PathLike, Mapping[str, Tensor]]] = None, seed: int = 0):
        super().__init__()
        self.features = vgg19_features()
        if weights is None:
            gen = torch.Generator().manual_seed(seed)
            for m in self.features:
                if isinstance(m, nn.Conv2d):
                    nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu", generator=gen)
                    nn.init.zeros_(m.bias)
        else:
            if isinstance(weights, (str, os.PathLike)):
                weights = torch.load(weights, map_location="cpu", weights_only=True)
            self.load_state_dict(weights)
        for p in self.parameters():
            p.requires_grad_(False)

    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):
        return super().load_state_dict(_features_only(state_dict), strict=strict, assign=assign)

    def _convs(self):
        return [m for m in self.features if isinstance(m, nn.Conv2d)]

    @staticmethod
    def _check(hr: Tensor, sr: Tensor) -> None:
        if not isinstance(hr, Tensor) or not isinstance(sr, Tensor) or hr.dim() != 4 or sr.dim() != 4:
            raise ValueError("perceptual loss: expected hr and sr of shape (N, C, H, W)")
        if hr.shape != sr.shape:
            raise ValueError(f"perceptual loss: hr {tuple(hr.shape)} and sr {tuple(sr.shape)} differ")
        n, c, h, w = hr.shape
        if c not in (1, 3):
            raise ValueError(f"perceptual loss: {c} channels (1, repeated to 3, or 3)")
        if n < 1 or h < 16 or w < 16:
            raise ValueError(f"perceptual loss: N >= 1 and H, W >= 16 needed (four 2x2 pools), got {tuple(hr.shape)}")
        if not hr.is_cuda or not sr.is_cuda:
            raise CsrError("climsr_b200 perceptual loss runs on CUDA (sm_100a) only; there is no CPU fallback")
        if hr.device != sr.device:
            raise ValueError(f"perceptual loss: hr on {hr.device}, sr on {sr.device}")

    def forward(self, hr: Tensor, sr: Tensor) -> Tensor:
        self._check(hr, sr)
        dev = hr.device
        if self.features[0].weight.device != dev:
            raise ValueError(f"perceptual loss: weights on {self.features[0].weight.device}, inputs on {dev} (move the module with .to())")
        n, c, h, w = hr.shape
        with torch.no_grad(), torch.cuda.device(dev):
            stream = current_stream_ptr()
            x = torch.empty((2 * n, h, w, _IN_C), dtype=torch.bfloat16, device=dev)
            ops.nchw_to_nhwc_split(hr.detach(), _IN_C, out=x[:n])
            ops.nchw_to_nhwc_split(sr.detach(), _IN_C, out=x[n:])
            cin = 2 * c                                   # executed input channels: the hi/lo pairs
            convs = self._convs()
            li = 0
            for m in self.features:
                if isinstance(m, nn.MaxPool2d):
                    x = ops.maxpool2x2_split(x)
                    h, w = h // 2, w // 2
                    continue
                if not isinstance(m, nn.Conv2d):
                    continue
                first, last = li == 0, li == len(convs) - 1
                fn, variant = (_pair_weight_gray, "pair1") if (first and c == 1) else (_pair_weight, "pair")
                scratch, _, _ = self._layer_pack(m, pack=True, weight_fn=fn, variant=variant)
                cout = m.out_channels
                if last:
                    # conv5_4: no ReLU, fp32 NHWC features; the mean |difference| is layout-independent
                    out = torch.empty((2 * n, h, w, cout), dtype=torch.float32, device=dev)
                    d = ConvDesc(2 * n, h, w, cin, cout, 3, 3, x.shape[-1], 0, cout, 0, ops.ACT["none"], ops.OUT_MODE["f32_nhwc"], 0, 0,
                                 1.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0.2, 0.0)
                else:
                    out = torch.empty((2 * n, h, w, 2 * cout), dtype=torch.bfloat16, device=dev)
                    d = ConvDesc(2 * n, h, w, cin, cout, 3, 3, x.shape[-1], 0, 2 * cout, 0, ops.ACT["relu"], ops.OUT_MODE["split"], 0, 0,
                                 1.0, 1.0, 0, 0, 0, 0, 0, 0, 0, 0.2, 0.0)
                check(lib.csr_conv2d_nhwc(C.byref(d), x.data_ptr(), None, None, out.data_ptr(), None, None, None, scratch.data_ptr(),
                                          scratch.numel(), stream), "csr_conv2d_nhwc (perceptual)")
                x, cin, li = out, 2 * cout, li + 1
            numel = n * h * w * x.shape[-1]
            loss = torch.empty((), dtype=torch.float32, device=dev)
            nbytes = lib.csr_pixel_loss_scratch_bytes(numel)
            red = torch.empty(nbytes, dtype=torch.uint8, device=dev)
            check(lib.csr_l1_loss(x[n:].data_ptr(), x[:n].data_ptr(), None, numel, loss.data_ptr(), red.data_ptr(), nbytes, stream),
                  "csr_l1_loss (perceptual)")
        return loss
