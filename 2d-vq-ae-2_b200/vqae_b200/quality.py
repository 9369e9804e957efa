"""Reconstruction quality of uint8 RGB patches on the GPU: exact SSE, MSE, PSNR and SSIM per patch.

The reference reports reconstruction MSE in normalised pixels (README.md:35,40) and validation
MSE / PSNR / SSIM per codebook size (scripts/extract_validation_metrics/results.md:3-6).  Here both
images are the uint8 pixels a user stores and looks at: the original tiles (what ``compress_slide``
encodes) and the 8-bit reconstruction (what ``decode_codes_u8`` / ``decompress_region`` produce).
Per patch of H x W x 3 pixels:

* ``sse``  int64 [3]: sum of (ref - rec)^2 per channel, exact;
* ``mse``  sum_c sse_c / (3 H W), in 8-bit levels^2;
* ``psnr`` 10 log10(255^2 / mse) dB, +inf for an exact reconstruction;
* ``mse_normalised`` sum_c sse_c / (255 std_c)^2 / (3 H W), the MSE in the model's normalised units
  (the fp32 scale ``1 / (255 std_c)`` of the input normalisation; CAMELYON16 ``mean`` / ``std`` by
  default, as in ``Encoder.encode``);
* ``ssim`` float64: the mean over the 3 channels and the (H - 10)(W - 10) valid window positions (no
  padding) of SSIM (Wang et al. 2004) with an 11 x 11 Gaussian window (sigma 1.5, the taps normalised to
  sum 1 in float64 and rounded once to fp32), population moments, C1 = (0.01 * 255)^2 and
  C2 = (0.03 * 255)^2 -- ``skimage.metrics.structural_similarity(gaussian_weights=True, sigma=1.5,
  use_sample_covariance=False, data_range=255, channel_axis=-1)``, which is also torchmetrics' default
  SSIM (reflect padding, then the border cropped).  The reference's eval script is not part of this
  project, so its published numbers are not claimed to be reproduced bit for bit.

SSE and SSIM come from one kernel (csrc/quality.cu) that reads both images once; the rest is derived
from ``sse`` on the device.
"""
from __future__ import annotations

import math
from dataclasses import dataclass
from typing import Dict, Optional, Sequence, Tuple

import numpy as np
import torch

from . import engine as E

Tensor = torch.Tensor
WINDOW = 11


def _inv_scale(std: Optional[Sequence[float]]) -> np.ndarray:
    """1 / (255 std_c) as the input normalisation forms it in fp32, widened to float64."""
    s = np.array(std if std is not None else E.CAMELYON16_STD, dtype=np.float32) * np.float32(255.0)
    return np.reciprocal(s, dtype=np.float32).astype(np.float64)


@dataclass
class ReconstructionQuality:
    """Per-patch metrics: ``sse`` int64 [..., 3] and ``ssim`` float64 [...] on the device, for patches
    of ``patch_hw`` = (H, W) pixels."""
    sse: Tensor
    ssim: Tensor
    patch_hw: Tuple[int, int]

    @property
    def _pixels(self) -> int:
        return 3 * self.patch_hw[0] * self.patch_hw[1]

    @property
    def mse(self) -> Tensor:
        """float64 [...]: mean squared error in 8-bit levels^2."""
        return self.sse.sum(-1).double() / self._pixels

    @property
    def psnr(self) -> Tensor:
        """float64 [...]: 10 log10(255^2 / mse) in dB; +inf where the reconstruction is exact."""
        return 10.0 * torch.log10(255.0 ** 2 / self.mse)

    def mse_normalised(self, mean=None, std=None) -> Tensor:
        """float64 [...]: the MSE of the normalised images, sum_c sse_c / (255 std_c)^2 / (3 H W).
        ``mean`` cancels in the difference; it is accepted so that callers can pass the pair they pass
        to ``Encoder.encode``."""
        d2 = torch.from_numpy(_inv_scale(std) ** 2).to(self.sse.device)
        return (self.sse.double() * d2).sum(-1) / self._pixels

    def summary(self, mean=None, std=None) -> Dict[str, float]:
        """Aggregates over all patches.  ``mse_pooled`` / ``psnr_pooled``: from the summed exact SSE,
        i.e. the MSE / PSNR of all patches taken as one image.  ``psnr_mean``: the mean of the per-patch
        PSNRs (+inf if any patch is reconstructed exactly); it weights every patch alike and differs
        from the pooled value.  ``ssim_mean`` and ``mse_normalised_mean``: means of the per-patch
        values.  ``patches``: the patch count."""
        n = self.ssim.numel()
        total = int(self.sse.sum())
        mse = total / (self._pixels * n) if n else math.nan
        return {
            "patches": n,
            "mse_pooled": mse,
            "psnr_pooled": 10.0 * math.log10(255.0 ** 2 / mse) if mse > 0 else math.inf,
            "psnr_mean": float(self.psnr.mean()),
            "ssim_mean": float(self.ssim.mean()),
            "mse_normalised_mean": float(self.mse_normalised(mean, std).mean()),
        }


def check_u8_patches(x: Tensor, what: str) -> None:
    if not isinstance(x, Tensor) or x.dtype != torch.uint8 or x.dim() != 4 or x.shape[-1] != 3:
        raise ValueError(f"{what} must be a uint8 [B,H,W,3] tensor, got "
                         f"{getattr(x, 'dtype', type(x))} {tuple(getattr(x, 'shape', ()))}")


@torch.no_grad()
def reconstruction_quality(ref_u8: Tensor, rec_u8: Tensor) -> ReconstructionQuality:
    """Score reconstructions ``rec_u8`` against originals ``ref_u8``: two contiguous uint8 [B,H,W,3]
    CUDA tensors of one shape on one device, H and W >= 11.  One kernel pass over both."""
    check_u8_patches(ref_u8, "ref_u8")
    check_u8_patches(rec_u8, "rec_u8")
    if ref_u8.shape != rec_u8.shape:
        raise ValueError(f"shape mismatch: {tuple(ref_u8.shape)} vs {tuple(rec_u8.shape)}")
    if ref_u8.device != rec_u8.device:
        raise ValueError(f"device mismatch: {ref_u8.device} vs {rec_u8.device}")
    if not (ref_u8.is_contiguous() and rec_u8.is_contiguous()):
        raise ValueError("reconstruction_quality needs contiguous inputs")
    b, h, w, _ = ref_u8.shape
    if h < WINDOW or w < WINDOW:
        raise ValueError(f"patches of {h} x {w} are smaller than the {WINDOW} x {WINDOW} SSIM window")
    E.require_cuda(ref_u8, "reconstruction_quality")
    sse, ssim = E.quality_u8(ref_u8.view(b * h, w, 3), (0, 0, 1, 0), rec_u8.view(b * h, w, 3), (0, 0, 1, 0),
                             b, h, w)
    return ReconstructionQuality(sse, ssim, (h, w))
