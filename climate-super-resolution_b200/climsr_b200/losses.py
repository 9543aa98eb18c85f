"""Pixel losses of the training step (mirror of ``self.loss = L1Loss() / MSELoss()``, climsr/core/task.py:141, used un-masked
over all pixels in climsr/task/pl_generator_pre_training.py:29-30 and climsr/task/pl_gan.py:41).

One CUDA pass produces the loss value and d loss / d sr; backward is a scalar multiply.  No CPU fallback.

The GAN step's VGG19 perceptual term is ``PerceptualLoss`` (climsr_b200/perceptual.py, re-exported here)."""
from __future__ import annotations

import torch
from torch import Tensor

from ._lib import CsrError, check, current_stream_ptr, lib


class _PixelLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, sr: Tensor, hr: Tensor, mode: int):
        if not sr.is_cuda:
            raise CsrError("climsr_b200 losses run on CUDA (sm_100a) only; there is no CPU fallback")
        if sr.shape != hr.shape:
            raise ValueError(f"loss: sr {tuple(sr.shape)} and hr {tuple(hr.shape)} differ")
        a = sr.detach().contiguous().float()
        b = hr.detach().to(sr.device).contiguous().float()
        n = a.numel()
        out = torch.empty((), dtype=torch.float32, device=sr.device)
        need_grad = sr.requires_grad
        grad = torch.empty_like(a) if need_grad else None
        nbytes = lib.csr_pixel_loss_scratch_bytes(n)
        scratch = torch.empty(nbytes, dtype=torch.uint8, device=sr.device)
        fn = lib.csr_l1_loss if mode == 0 else lib.csr_mse_loss
        with torch.cuda.device(sr.device):
            check(fn(a.data_ptr(), b.data_ptr(), grad.data_ptr() if grad is not None else None, n, out.data_ptr(), scratch.data_ptr(),
                     nbytes, current_stream_ptr()), "csr_pixel_loss")
        ctx.grad = grad
        ctx.shape = sr.shape
        return out

    @staticmethod
    def backward(ctx, g):
        if ctx.grad is None:
            return None, None, None
        return (ctx.grad * g).view(ctx.shape), None, None


def l1_loss(sr: Tensor, hr: Tensor) -> Tensor:
    """torch.nn.L1Loss()(sr, hr) (mean reduction)."""
    return _PixelLoss.apply(sr, hr, 0)


def mse_loss(sr: Tensor, hr: Tensor) -> Tensor:
    """torch.nn.MSELoss()(sr, hr) (mean reduction)."""
    return _PixelLoss.apply(sr, hr, 1)


class L1Loss(torch.nn.Module):
    def forward(self, sr: Tensor, hr: Tensor) -> Tensor:
        return l1_loss(sr, hr)


class MSELoss(torch.nn.Module):
    def forward(self, sr: Tensor, hr: Tensor) -> Tensor:
        return mse_loss(sr, hr)


from .perceptual import PerceptualLoss  # noqa: E402,F401  (imports this package's models; kept last)
