"""float64 restatement of the VGG19 perceptual loss (climsr_b200.losses.PerceptualLoss): ``vgg19().features[:35]`` with
F.conv2d / F.relu / F.max_pool2d on the same state dict, then the mean absolute difference of the hr and sr features.

Assumptions, as in the module: a 1-channel input is repeated to three channels, no ImageNet normalisation.

``emulate`` reproduces the rounding points of a kernel path (for setting test tolerances, DESIGN.md section 10):
  "none"  exact float64;
  "split" the sm_100a path: input and every activation as a hi/lo bf16 pair (hi = bf16(v), lo = bf16(v - hi) of the fp32
          value), bf16 weights (conv1_1 of a 1-channel input: the fp32 sum over its input channels, then bf16), fp32 bias,
          fp32 conv5_4 features;
  "bf16"  the same with plain bf16 activations (what a bf16 path without the pairs would compute).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

VGG19_CFG = (64, 64, "M", 128, 128, "M", 256, 256, 256, 256, "M", 512, 512, 512, 512, "M", 512, 512, 512, 512)


def conv_indices():
    """torchvision module indices of the 16 convs of features[:35]: 0, 2, 5, ..., 34."""
    idx, i = [], 0
    for v in VGG19_CFG:
        if v == "M":
            i += 1
        else:
            idx.append(i)
            i += 2
    return idx


def _pair(v: torch.Tensor) -> torch.Tensor:
    v32 = v.float()
    hi = v32.bfloat16()
    lo = (v32 - hi.float()).bfloat16()
    return hi.double() + lo.double()


def _round_act(v: torch.Tensor, emulate: str) -> torch.Tensor:
    if emulate == "split":
        return _pair(v)
    if emulate == "bf16":
        return v.float().bfloat16().double()
    return v


def features(sd, x: torch.Tensor, emulate: str = "none") -> torch.Tensor:
    """conv5_4 features (float64, NCHW) of x (N, 1 or 3, H, W); sd holds ``features.{i}.weight/bias``."""
    if emulate not in ("none", "split", "bf16"):
        raise ValueError(emulate)
    dev = x.device
    c = x.shape[1]
    h = x.double()
    if c == 1 and emulate == "none":
        h = h.repeat(1, 3, 1, 1)
    h = _round_act(h, emulate)
    convs = conv_indices()
    k = 0
    for v in VGG19_CFG:
        if v == "M":
            h = F.max_pool2d(h, 2)
            continue
        i = convs[k]
        w = sd[f"features.{i}.weight"].to(dev)
        b = sd[f"features.{i}.bias"].to(dev)
        if emulate != "none":
            w32 = w.float()
            if k == 0 and c == 1:
                w32 = w32.sum(1, keepdim=True)
            w, b = w32.bfloat16().double(), b.float().double()
        else:
            w, b = w.double(), b.double()
        h = F.conv2d(h, w, b, padding=1)
        last = k == len(convs) - 1
        if last:
            h = h.float().double() if emulate != "none" else h
        else:
            h = _round_act(F.relu(h), emulate)
        k += 1
    return h


def perceptual_loss(sd, hr: torch.Tensor, sr: torch.Tensor, emulate: str = "none") -> torch.Tensor:
    """mean |features(hr) - features(sr)| in float64 (0-dim); hr and sr pass through the network as one batch."""
    n = hr.shape[0]
    f = features(sd, torch.cat([hr, sr], 0), emulate)
    return (f[:n] - f[n:]).abs().mean()
