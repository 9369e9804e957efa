"""TEST INFRASTRUCTURE ONLY -- float64 restatement of the reconstruction metrics of vqae_b200.quality.

SSIM as skimage.metrics.structural_similarity(gaussian_weights=True, sigma=1.5,
use_sample_covariance=False, data_range=255, channel_axis=-1), with the 11 Gaussian taps rounded to fp32
(then widened) exactly as the kernel uses them: a separable correlation with scipy.ndimage.correlate1d,
cropped to the valid window positions.  SSE in numpy int64.
"""
from __future__ import annotations

import numpy as np
from scipy.ndimage import correlate1d

R = 5
C1 = (0.01 * 255) ** 2
C2 = (0.03 * 255) ** 2


def gaussian_taps_f32() -> np.ndarray:
    """The 11 taps: exp(-k^2 / (2 * 1.5^2)), k = -5 .. 5, normalised in float64, rounded once to fp32."""
    k = np.arange(-R, R + 1, dtype=np.float64)
    g = np.exp(-k * k / (2.0 * 1.5 * 1.5))
    return (g / g.sum()).astype(np.float32)


def _filter_valid(img: np.ndarray, w: np.ndarray) -> np.ndarray:
    out = correlate1d(correlate1d(img, w, axis=0, mode="constant"), w, axis=1, mode="constant")
    return out[R:-R, R:-R]


def ssim_map(x: np.ndarray, y: np.ndarray) -> np.ndarray:
    """Per-position SSIM [H-10, W-10] of two 2-D images."""
    w = gaussian_taps_f32().astype(np.float64)
    x = x.astype(np.float64)
    y = y.astype(np.float64)
    mx, my = _filter_valid(x, w), _filter_valid(y, w)
    sxx = _filter_valid(x * x, w) - mx * mx
    syy = _filter_valid(y * y, w) - my * my
    sxy = _filter_valid(x * y, w) - mx * my
    return ((2 * mx * my + C1) * (2 * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2))


def ssim(ref: np.ndarray, rec: np.ndarray) -> float:
    """Mean SSIM of one [H,W,3] patch pair over the channels and the valid positions."""
    return float(np.mean([ssim_map(ref[..., c], rec[..., c]).mean() for c in range(3)]))


def sse(ref: np.ndarray, rec: np.ndarray) -> np.ndarray:
    """int64 [..., 3]: per-channel sum of squared differences of [..., H, W, 3] patches."""
    d = ref.astype(np.int64) - rec.astype(np.int64)
    return (d * d).sum(axis=(-3, -2))
