"""TEST INFRASTRUCTURE ONLY -- CPU restatement of code map -> uint8 RGB decompression.

The reference has no uint8 decode (its images end as normalised fp32 tensors), so this is not part of
oracle/vqae_oracle.py, which restates the reference and is pinned against it.  It composes that
oracle's ``decode_from_codes`` with the inverse of its ``normalize_u8``.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

import vqae_oracle as O


def denormalize_u8(x_chw, mean=O.CAMELYON16_MEAN, std=O.CAMELYON16_STD) -> np.ndarray:
    """The inverse of ``O.normalize_u8``: [3,H,W] / [B,3,H,W] fp32 -> [H,W,3] / [B,H,W,3] uint8,
    ``min(max(rint(fma(v, s_c, o_c)), 0), 255)`` with ``s_c = f32(255) f32(std_c)`` and
    ``o_c = f32(255) f32(mean_c)`` (the products ``normalize_u8`` forms), round half to even, NaN -> 0.
    The fused multiply-add is formed in float64 (the product of two fp32 numbers is exact there) and
    rounded to fp32 before ``rint``."""
    x = np.asarray(x_chw, dtype=np.float32)
    s = (np.array(std, dtype=np.float32) * np.float32(255.0)).astype(np.float64)
    o = (np.array(mean, dtype=np.float32) * np.float32(255.0)).astype(np.float64)
    v = np.moveaxis(x, -3, -1).astype(np.float64)
    y = np.rint((v * s + o).astype(np.float32))
    with np.errstate(invalid="ignore"):
        y = np.where(np.isnan(y), np.float32(0.0), np.clip(y, 0.0, 255.0))
    return y.astype(np.uint8)


def decompress_region(code_map, sd, code_hw: Tuple[int, int],
                      region: Optional[Tuple[int, int, int, int]] = None, mean=O.CAMELYON16_MEAN,
                      std=O.CAMELYON16_STD) -> np.ndarray:
    """A stored code map (or its region (r0, c0, nr, nc), in patches) -> uint8 RGB [nr*H, nc*W, 3]:
    cut the map into code tiles, ``O.decode_from_codes``, ``denormalize_u8``, stitch row-major."""
    cm = np.asarray(code_map).astype(np.int64)
    th, tw = code_hw
    rows, cols = cm.shape[0] // th, cm.shape[1] // tw
    r0, c0, nr, nc = region if region is not None else (0, 0, rows, cols)
    tiles = [cm[(r0 + r) * th:(r0 + r + 1) * th, (c0 + c) * tw:(c0 + c + 1) * tw]
             for r in range(nr) for c in range(nc)]
    with torch.no_grad():
        dec = O.decode_from_codes(torch.from_numpy(np.stack(tiles)), sd)
    return stitch(denormalize_u8(dec.numpy(), mean, std), nc)


def stitch(patches: np.ndarray, nc: int) -> np.ndarray:
    """[P,H,W,3] patches in row-major order, nc per row -> [P/nc*H, nc*W, 3]."""
    p, ph, pw, _ = patches.shape
    nr = p // nc
    return patches.reshape(nr, nc, ph, pw, 3).transpose(0, 2, 1, 3, 4).reshape(nr * ph, nc * pw, 3)
