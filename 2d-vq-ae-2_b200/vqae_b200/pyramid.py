"""Slide pyramids on the GPU: exact box-filtered overview levels of uint8 RGB canvases.

Slide viewers (OpenSlide, DeepZoom / OpenSeadragon, QuPath) and thumbnail or tissue-overview code read a
whole-slide image as a pyramid of downsampled levels.  Level f (a power of two in [2, 512] dividing the
patch height H and width W) is, per channel, the box mean of each f x f block rounded half up:

    out = (S + f^2 / 2) >> log2(f^2),   S = the exact integer sum of the f x f pixels,

rounded once from the original pixels (no level is made from another) -- what ``PIL.Image.reduce(f)``
computes.  Because f divides the patch, every output pixel comes from one patch, and the level of a
region equals ``PIL.Image.fromarray(region).reduce(f)`` byte for byte.  Levels coarser than one patch
are a few KB of work and are left to the caller.

One kernel (csrc/pyramid.cu) reads each pixel once and writes every requested level.  ``slide_pyramid``
works on any uint8 canvas already on the GPU; ``extract.decompress_pyramid`` builds the levels of a
stored code map batch by batch as it decodes, without the full-resolution canvas.
"""
from __future__ import annotations

import operator
from typing import Dict, Iterable, Tuple

import torch

from . import engine as E

Tensor = torch.Tensor
FACTORS = tuple(1 << k for k in range(1, 10))                # 2 .. 512


def check_factors(factors: Iterable[int], patch_hw: Tuple[int, int]) -> Tuple[int, ...]:
    """The factors as a sorted tuple of ints; ValueError unless they are distinct powers of two in
    [2, 512] that divide the patch height and width, and at least one."""
    fs = list(factors)
    if not fs:
        raise ValueError("no pyramid factors given")
    out = []
    for f in fs:
        try:
            f = operator.index(f)
        except TypeError:
            raise ValueError(f"pyramid factor {f!r} is not an integer") from None
        if f not in FACTORS:
            raise ValueError(f"pyramid factor {f} is not a power of two in [2, 512]")
        if patch_hw[0] % f or patch_hw[1] % f:
            raise ValueError(f"pyramid factor {f} does not divide the {patch_hw[0]} x {patch_hw[1]} patch")
        out.append(f)
    if len(set(out)) != len(out):
        raise ValueError(f"duplicate pyramid factors in {fs}")
    return tuple(sorted(out))


def level_canvases(grid: Tuple[int, int], patch_hw: Tuple[int, int], factors: Tuple[int, ...],
                   device: torch.device) -> Dict[int, Tensor]:
    """Empty uint8 [rows*H/f, cols*W/f, 3] canvases, one per factor, for a grid of (rows, cols) patches."""
    (rows, cols), (h, w) = grid, patch_hw
    return {f: torch.empty(rows * (h // f), cols * (w // f), 3, dtype=torch.uint8, device=device)
            for f in factors}


@torch.no_grad()
def slide_pyramid(slide_u8: Tensor, patch_hw: Tuple[int, int], factors: Iterable[int],
                  batch: int = 4096) -> Dict[int, Tensor]:
    """The pyramid levels of a uint8 canvas: ``slide_u8`` contiguous uint8 [rows*H, cols*W, 3] on a CUDA
    device (an original slide, or a ``decompress_region`` output), ``patch_hw`` = (H, W).  Returns
    ``{f: uint8 [rows*H/f, cols*W/f, 3]}`` on the same device for every factor (see ``check_factors``).
    ``batch`` patches per kernel launch (it bounds the scratch levels f >= 128 need)."""
    if not isinstance(slide_u8, Tensor) or slide_u8.dtype != torch.uint8 or slide_u8.dim() != 3 or \
            slide_u8.shape[2] != 3:
        raise ValueError(f"slide_u8 must be a uint8 [rows*H, cols*W, 3] tensor, got "
                         f"{getattr(slide_u8, 'dtype', type(slide_u8))} {tuple(getattr(slide_u8, 'shape', ()))}")
    E.require_cuda(slide_u8, "slide_pyramid")
    if not slide_u8.is_contiguous():
        raise ValueError("slide_pyramid needs a contiguous canvas")
    h, w = (int(v) for v in patch_hw)
    if h <= 0 or w <= 0 or slide_u8.shape[0] % h or slide_u8.shape[1] % w:
        raise ValueError(f"canvas {tuple(slide_u8.shape[:2])} is not a grid of {h} x {w} patches")
    if batch <= 0:
        raise ValueError("batch must be positive")
    fs = check_factors(factors, (h, w))
    rows, cols = slide_u8.shape[0] // h, slide_u8.shape[1] // w
    out = level_canvases((rows, cols), (h, w), fs, slide_u8.device)
    total = rows * cols
    for first in range(0, total, batch):
        n = min(batch, total - first)
        E.pyramid_u8(slide_u8, (0, 0, cols, first), n, h, w, out, (0, 0, cols, first))
    return out
