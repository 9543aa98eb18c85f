"""Host-side mirror of the reference's task layer around the generator hot path - the call patterns a LightningModule drives.

Reference: ``TaskSuperResolutionModule`` (climsr/core/task.py:104-300), ``SuperResolutionLightningModule``
(climsr/task/pl_generator_pre_training.py:10-69) and ``GANLightningModule`` (climsr/task/pl_gan.py:12-139).  Lightning,
Hydra and torchmetrics are control plane (out of scope, SURVEY.md section 2); what sits ON the path is reproduced here with
the same method names, batch-dict keys (climsr/consts/batch_items.py) and return values:

    forward(x, elevation, mask)                      task.py:235-239
    common_step(batch) -> (hr, sr)                   task.py:241-260
    training_step(batch, batch_idx[, optimizer_idx]) pl_generator_pre_training.py:18-33 / pl_gan.py:63-95
    common_val_test_step(batch, prefix)              task.py:262-300  (one fused CUDA pass instead of ~10 tensor passes)
    loss_g / loss_d                                  pl_gan.py:28-61  (relativistic average GAN, BCE-with-logits)

so a Lightning user can either subclass this next to ``pl.LightningModule`` or call the same methods from their own loop.
Everything numeric runs in the sm_100a kernels (generator, pixel loss, masked metrics, discriminator); there is no CPU path.
"""
from __future__ import annotations

from typing import Any, Dict, Optional, Tuple

import torch
import torch.nn as nn
from torch import Tensor

from . import losses
from .metrics import masked_val_metrics

# climsr/consts/batch_items.py
LR, HR, ELEVATION, MASK, ORIGINAL, MIN, MAX = "lr", "hr", "elevation", "mask", "original_data", "min", "max"


class SuperResolutionTask(nn.Module):
    """Pre-training task (``optimizer_idx`` absent) or GAN task (a discriminator is given), like the reference's two modules."""

    def __init__(self, generator: nn.Module, discriminator: Optional[nn.Module] = None, normalization_method: str = "minmax",
                 normalization_range: Tuple[float, float] = (-1.0, 1.0), zscore: Optional[Tuple[float, float]] = None,
                 generator_type: str = "esrgan", pixel_level_loss_factor: float = 0.01, perceptual_loss_factor: float = 1.0,
                 adversarial_loss_factor: float = 0.005, perceptual_criterion: Optional[nn.Module] = None, scaler_eps: float = 1e-8):
        super().__init__()
        self.generator = generator
        self.discriminator = discriminator
        self.generator_type = generator_type
        self.normalization_method = normalization_method
        self.normalization_range = tuple(normalization_range)
        self.zscore = zscore
        self.scaler_eps = scaler_eps
        if normalization_method == "zscore" and zscore is None:
            raise ValueError("normalization_method='zscore' needs zscore=(mean, std) (task.py:146-166 reads them from the stats file)")
        # task.py:141: MSELoss for srcnn, L1Loss otherwise
        self.loss = losses.MSELoss() if generator_type == "srcnn" else losses.L1Loss()
        self.pixel_level_criterion = losses.L1Loss()                    # pl_gan.py:20
        self.adversarial_criterion = nn.BCEWithLogitsLoss()             # pl_gan.py:21 (a scalar epilogue on N logits)
        self.perceptual_criterion = perceptual_criterion               # pl_gan.py:19 (losses.PerceptualLoss: VGG19 features; None = term off)
        self.pixel_level_loss_factor = pixel_level_loss_factor          # conf/task/gan_training.yaml:6-8
        self.perceptual_loss_factor = perceptual_loss_factor
        self.adversarial_loss_factor = adversarial_loss_factor

    # ---------------------------------------------------------------- task.py:235-260
    def forward(self, x: Tensor, elevation: Tensor = None, mask: Tensor = None) -> Tensor:
        if self.generator_type == "srcnn":
            return self.generator(x)
        return self.generator(x, elevation, mask)

    def common_step(self, batch: Any) -> Tuple[Tensor, Tensor]:
        lr, hr, elev, mask = batch[LR], batch[HR], batch[ELEVATION], batch[MASK]
        sr = self(lr, elev, mask)
        return hr, sr

    # ---------------------------------------------------------------- pl_gan.py:23-61
    def _real_fake(self, size: int, device) -> Tuple[Tensor, Tensor]:
        return torch.ones((size, 1), device=device), torch.zeros((size, 1), device=device)

    def loss_g(self, hr: Tensor, sr: Tensor, real_labels: Tensor, fake_labels: Tensor):
        score_real = self.discriminator(hr)
        score_fake = self.discriminator(sr)
        discriminator_rf = score_real - score_fake.mean()
        discriminator_fr = score_fake - score_real.mean()
        adversarial_loss_rf = self.adversarial_criterion(discriminator_rf, fake_labels)
        adversarial_loss_fr = self.adversarial_criterion(discriminator_fr, real_labels)
        adversarial_loss = (adversarial_loss_fr + adversarial_loss_rf) / 2
        perceptual_loss = self.perceptual_criterion(hr, sr) if self.perceptual_criterion is not None else sr.new_zeros(())
        pixel_level_loss = self.pixel_level_criterion(sr, hr)
        loss_g = (self.pixel_level_loss_factor * pixel_level_loss + self.perceptual_loss_factor * perceptual_loss
                  + self.adversarial_loss_factor * adversarial_loss)
        return perceptual_loss, adversarial_loss, pixel_level_loss, loss_g

    def loss_d(self, hr: Tensor, sr: Tensor, real_labels: Tensor, fake_labels: Tensor) -> Tensor:
        score_real = self.discriminator(hr)
        score_fake = self.discriminator(sr.detach())
        discriminator_rf = score_real - score_fake.mean()
        discriminator_fr = score_fake - score_real.mean()
        adversarial_loss_rf = self.adversarial_criterion(discriminator_rf, real_labels)
        adversarial_loss_fr = self.adversarial_criterion(discriminator_fr, fake_labels)
        return (adversarial_loss_fr + adversarial_loss_rf) / 2

    # ---------------------------------------------------------------- training_step of both reference modules
    def training_step(self, batch: Any, batch_idx: int = 0, optimizer_idx: Optional[int] = None):
        if self.discriminator is None or optimizer_idx is None:
            hr, sr = self.common_step(batch)                            # pl_generator_pre_training.py:28-32
            return self.loss(sr, hr)
        hr = batch[HR]
        real_labels, fake_labels = self._real_fake(hr.shape[0], hr.device)
        hr, sr = self.common_step(batch)                                # pl_gan.py:67 (runs for BOTH optimizers)
        if optimizer_idx == 0:
            perceptual_loss, adversarial_loss, pixel_level_loss, loss_g = self.loss_g(hr, sr, real_labels, fake_labels)
            log = {"train/perceptual_loss": perceptual_loss, "train/adversarial_loss": adversarial_loss,
                   "train/pixel_level_loss": pixel_level_loss, "train/loss_G": loss_g}
            return {"loss": loss_g, "log": log}
        if optimizer_idx == 1:
            loss_d = self.loss_d(hr, sr, real_labels, fake_labels)
            return {"loss": loss_d, "log": {"train/loss_D": loss_d}}
        raise ValueError(f"optimizer_idx {optimizer_idx} (the reference has two optimizers: 0 = generator, 1 = discriminator)")

    # ---------------------------------------------------------------- task.py:262-300
    @torch.no_grad()
    def common_val_test_step(self, batch: Any, prefix: str = "val") -> Dict[str, Tensor]:
        hr, sr = self.common_step(batch)
        zs = self.zscore if self.normalization_method == "zscore" else None
        out = masked_val_metrics(sr, hr, batch[ORIGINAL], batch[MASK],
                                 None if zs is not None else batch[MIN], None if zs is not None else batch[MAX], zscore=zs,
                                 feature_range=self.normalization_range, prefix=prefix,
                                 loss="mse" if self.generator_type == "srcnn" else "l1", eps=self.scaler_eps)
        out["sr"] = sr.detach().clone()                                 # task.py:277,298 (un-masked copy for the image logger)
        return out

    def validation_step(self, batch: Any, batch_idx: int = 0, dataloader_idx: Optional[int] = None) -> Dict[str, Tensor]:
        metric_dict = self.common_val_test_step(batch, prefix="val")
        if self.discriminator is not None:                              # pl_gan.py:97-139
            hr = batch[HR]
            real_labels, fake_labels = self._real_fake(hr.size(0), hr.device)
            with torch.no_grad():
                perceptual_loss, adversarial_loss, _pixel, loss_g = self.loss_g(hr, metric_dict["sr"], real_labels, fake_labels)
            metric_dict.update({"val/perceptual_loss": perceptual_loss, "val/adversarial_loss": adversarial_loss, "val/loss_G": loss_g})
        metric_dict.pop("sr", None)
        return metric_dict

    def test_step(self, batch: Any, batch_idx: int = 0, dataloader_idx: Optional[int] = None) -> Dict[str, Tensor]:
        return self.common_val_test_step(batch, prefix="test")
