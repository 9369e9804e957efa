"""DeepZoom JPEG tiles on the GPU: baseline JFIF files byte-identical to libjpeg's.

Slide viewers (OpenSeadragon, QuPath, OpenSlide's DeepZoom server) read a whole-slide image as a DeepZoom
pyramid: a ``.dzi`` descriptor and ``<name>_files/<level>/<col>_<row>.jpeg`` tiles.  ``encode_tiles``
cuts one uint8 RGB canvas level into the DeepZoom tile grid and encodes every tile in one call of the
CUDA encoder (csrc/jpeg.cu, DESIGN.md section 4.16).  Each tile is the baseline sequential file that
``PIL.Image.fromarray(tile).save(buf, "JPEG", quality=q, subsampling=s)`` writes (libjpeg-turbo, standard
Huffman tables, no restart markers), byte for byte, for q in 1 .. 100 and s = 0 (4:4:4) or 2 (4:2:0).

This module is the one place that knows the file format's tables and headers: ``quant_tables`` scales
the Annex K quantisation tables like libjpeg's ``jpeg_set_quality``; ``jpeg_header`` writes SOI, APP0
(JFIF 1.01), DQT x 2, SOF0, DHT x 4 and SOS in libjpeg's order.  The kernel writes the entropy-coded
scan and EOI after it.

DeepZoom geometry: a W x H image has levels 0 .. M, M = ceil(log2 max(W, H)); level L is
ceil(W / 2^(M-L)) x ceil(H / 2^(M-L)).  With tile size T and overlap o (0 <= o < T), tile (c, r) of a
level covers x in [max(0, cT - o), min(W_L, (c+1)T + o)) and likewise y.
"""
from __future__ import annotations

import math
from typing import List, Optional, Tuple

import numpy as np
import torch

from . import engine as E

Tensor = torch.Tensor

# Annex K.1 tables, natural (row-major) order
STD_LUMINANCE = (16, 11, 10, 16, 24, 40, 51, 61, 12, 12, 14, 19, 26, 58, 60, 55, 14, 13, 16, 24, 40, 57, 69, 56,
                 14, 17, 22, 29, 51, 87, 80, 62, 18, 22, 37, 56, 68, 109, 103, 77, 24, 35, 55, 64, 81, 104, 113,
                 92, 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99)
STD_CHROMINANCE = (17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99,
                   47, 66, 99, 99, 99, 99, 99, 99, *([99] * 32))
ZIGZAG = (0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7,
          14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46,
          53, 60, 61, 54, 47, 55, 62, 63)                    # zigzag position -> natural index
# Annex K.3 Huffman tables: (code-length counts 1 .. 16, symbols)
DC_LUMINANCE = ((0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0), tuple(range(12)))
DC_CHROMINANCE = ((0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0), tuple(range(12)))
AC_LUMINANCE = ((0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7D), bytes.fromhex(
    "01020300041105122131410613516107227114328191a1082342b1c11552d1f02433627282090a161718191a25262728292a3435363738"
    "393a434445464748494a535455565758595a636465666768696a737475767778797a838485868788898a92939495969798999aa2a3a4a5"
    "a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae1e2e3e4e5e6e7e8e9eaf1f2f3f4f5f6f7f8f9fa"))
AC_CHROMINANCE = ((0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77), bytes.fromhex(
    "000102031104052131061241510761711322328108144291a1b1c109233352f0156272d10a162434e125f11718191a262728292a353637"
    "38393a434445464748494a535455565758595a636465666768696a737475767778797a82838485868788898a92939495969798999aa2a3"
    "a4a5a6a7a8a9aab2b3b4b5b6b7b8b9bac2c3c4c5c6c7c8c9cad2d3d4d5d6d7d8d9dae2e3e4e5e6e7e8e9eaf2f3f4f5f6f7f8f9fa"))


def check_quality(quality: int, subsampling: int) -> Tuple[int, int]:
    q, s = int(quality), int(subsampling)
    if q != quality or not 1 <= q <= 100:
        raise ValueError(f"JPEG quality must be an integer in 1 .. 100, got {quality!r}")
    if s != subsampling or s not in (0, 2):
        raise ValueError(f"JPEG subsampling must be 0 (4:4:4) or 2 (4:2:0), got {subsampling!r}")
    return q, s


def quant_tables(quality: int) -> np.ndarray:
    """The luminance and chrominance tables of ``quality``, uint16 [2, 64] in zigzag order (the DQT
    order): libjpeg's ``jpeg_quality_scaling`` (5000 / q below 50, 200 - 2q otherwise) applied to the
    Annex K tables as (t * scale + 50) // 100, clamped to [1, 255] (baseline)."""
    q, _ = check_quality(quality, 0)
    scale = 5000 // q if q < 50 else 200 - 2 * q
    out = np.empty((2, 64), np.uint16)
    for i, base in enumerate((STD_LUMINANCE, STD_CHROMINANCE)):
        t = (np.asarray(base, np.int64)[list(ZIGZAG)] * scale + 50) // 100
        out[i] = np.clip(t, 1, 255)
    return out


def _segment(marker: int, body: bytes) -> bytes:
    return bytes((0xFF, marker)) + (len(body) + 2).to_bytes(2, "big") + body


def jpeg_header(height: int, width: int, quality: int, subsampling: int) -> bytes:
    """SOI through SOS of a baseline JFIF file of an RGB ``height`` x ``width`` image, as libjpeg writes
    it for ``quality`` and ``subsampling`` (0: 4:4:4, 2: 4:2:0)."""
    _, s = check_quality(quality, subsampling)
    if not (1 <= height <= 65535 and 1 <= width <= 65535):
        raise ValueError(f"a JPEG image is 1 .. 65535 pixels a side, got {height} x {width}")
    qt = quant_tables(quality)
    out = bytearray(b"\xff\xd8")
    out += _segment(0xE0, b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for i in range(2):
        out += _segment(0xDB, bytes((i,)) + bytes(qt[i].astype(np.uint8)))
    y_samp = 0x22 if s == 2 else 0x11
    out += _segment(0xC0, bytes((8,)) + height.to_bytes(2, "big") + width.to_bytes(2, "big") +
                    bytes((3, 1, y_samp, 0, 2, 0x11, 1, 3, 0x11, 1)))
    for cls_id, (counts, symbols) in ((0x00, DC_LUMINANCE), (0x10, AC_LUMINANCE), (0x01, DC_CHROMINANCE),
                                      (0x11, AC_CHROMINANCE)):
        out += _segment(0xC4, bytes((cls_id, *counts)) + bytes(symbols))
    out += _segment(0xDA, bytes((3, 1, 0x00, 2, 0x11, 3, 0x11, 0, 63, 0)))
    return bytes(out)


# ---- DeepZoom geometry --------------------------------------------------------------------------------------
def dz_levels(width: int, height: int) -> List[Tuple[int, int]]:
    """(width, height) of DeepZoom levels 0 .. M, M = ceil(log2 max(width, height))."""
    if width <= 0 or height <= 0:
        raise ValueError(f"image extent must be positive, got {width} x {height}")
    m = math.ceil(math.log2(max(width, height))) if max(width, height) > 1 else 0
    return [(-(-width // (1 << (m - lv))), -(-height // (1 << (m - lv)))) for lv in range(m + 1)]


def tile_grid(width: int, height: int, tile: int) -> Tuple[int, int]:
    """(columns, rows) of the tile grid of a width x height level."""
    return -(-width // tile), -(-height // tile)


def tile_span(i: int, extent: int, tile: int, overlap: int) -> Tuple[int, int]:
    """[start, stop) of tile i along an axis of ``extent`` pixels."""
    return max(0, i * tile - overlap), min(extent, (i + 1) * tile + overlap)


def tile_rect(c: int, r: int, width: int, height: int, tile: int, overlap: int) -> Tuple[int, int, int, int]:
    """(x0, y0, x1, y1) of tile (c, r) of a width x height level."""
    (x0, x1), (y0, y1) = tile_span(c, width, tile, overlap), tile_span(r, height, tile, overlap)
    return x0, y0, x1, y1


def check_tiling(tile: int, overlap: int) -> None:
    if int(tile) != tile or tile <= 0:
        raise ValueError(f"tile size must be a positive integer, got {tile!r}")
    if int(overlap) != overlap or overlap < 0:
        raise ValueError(f"tile overlap must be a non-negative integer, got {overlap!r}")
    if overlap >= tile:
        raise ValueError(f"tile overlap {overlap} must be smaller than the tile size {tile}")


def dzi_xml(width: int, height: int, tile: int = 254, overlap: int = 1, fmt: str = "jpeg") -> str:
    """The DeepZoom descriptor (``.dzi``) of a width x height image."""
    return ('<?xml version="1.0" encoding="UTF-8"?>\n'
            f'<Image xmlns="http://schemas.microsoft.com/deepzoom/2008" Format="{fmt}" Overlap="{overlap}" '
            f'TileSize="{tile}">\n  <Size Height="{height}" Width="{width}"/>\n</Image>\n')


def tile_class(i: int, n: int) -> int:
    """Class of tile i of an axis of n tiles: 0 the first, 1 a middle one, 2 the second-to-last, 3 the last
    (the lower class of a tile that is several).  Tiles of one class have one size: with overlap < tile,
    only the first tile starts at 0 and only the last two can reach the extent."""
    return 0 if i == 0 else 3 if i == n - 1 else 2 if i == n - 2 else 1


def level_headers(width: int, height: int, tile: int, overlap: int, quality: int, subsampling: int) -> bytes:
    """The 16 headers ``vqae_jpeg_tiles`` reads: header 4 * row class + column class (``tile_class``) for
    that class's tile size; a class the grid does not have repeats the first tile's header."""
    check_tiling(tile, overlap)
    cols, rows = tile_grid(width, height, tile)

    def rep(cls: int, n: int) -> int:
        hit = [i for i in {0, 1, n - 2, n - 1} if 0 <= i < n and tile_class(i, n) == cls]
        return hit[0] if hit else 0

    out = b""
    for rc in range(4):
        for cc in range(4):
            x0, y0, x1, y1 = tile_rect(rep(cc, cols), rep(rc, rows), width, height, tile, overlap)
            out += jpeg_header(y1 - y0, x1 - x0, quality, subsampling)
    return out


class JpegTiles:
    """The encoded tiles of one level: ``payload`` (uint8, device) holds tile i = r * cols + c (rows
    counted from ``row0``) at ``[offsets[i], offsets[i + 1])``; ``offsets`` int64 on the host."""

    def __init__(self, payload: Tensor, offsets: np.ndarray, grid: Tuple[int, int], row0: int, tile: int,
                 overlap: int, quality: int, subsampling: int):
        self.payload, self.offsets, self.grid, self.row0 = payload, offsets, grid, row0
        self.tile, self.overlap, self.quality, self.subsampling = tile, overlap, quality, subsampling

    def nbytes(self) -> int:
        return int(self.offsets[-1])

    def tile_bytes(self, c: int, r: int, host: Optional[np.ndarray] = None) -> bytes:
        """The JPEG file of tile (c, r); ``host`` a host copy of ``payload`` to slice instead."""
        cols, rows = self.grid
        if not (0 <= c < cols and self.row0 <= r < self.row0 + rows):
            raise IndexError(f"tile ({c}, {r}) is outside the encoded grid")
        i = (r - self.row0) * cols + c
        lo, hi = int(self.offsets[i]), int(self.offsets[i + 1])
        if host is not None:
            return host[lo:hi].tobytes()
        return self.payload[lo:hi].cpu().numpy().tobytes()


@torch.no_grad()
def encode_tiles(canvas_u8: Tensor, tile: int = 254, overlap: int = 1, quality: int = 90, subsampling: int = 2,
                 rows: Optional[Tuple[int, int]] = None) -> JpegTiles:
    """JPEG-encode the DeepZoom tiles of one level on the GPU.  ``canvas_u8`` uint8 [H, W, 3] on a CUDA
    device, rows of any pitch (a crop of a larger canvas works) and channels packed.  ``rows`` = (row0,
    nrows) restricts the call to those tile rows (default all): scratch and payload scale with it."""
    q, s = check_quality(quality, subsampling)
    check_tiling(tile, overlap)
    h, w = int(canvas_u8.shape[0]), int(canvas_u8.shape[1])
    cols, nrows_total = tile_grid(w, h, tile)
    row0, nrows = rows if rows is not None else (0, nrows_total)
    if not (0 <= row0 and nrows > 0 and row0 + nrows <= nrows_total):
        raise ValueError(f"tile rows {(row0, nrows)} leave the {nrows_total}-row tile grid")
    headers = level_headers(w, h, tile, overlap, q, s)
    payload, offsets = E.jpeg_tiles(canvas_u8, tile, overlap, row0, nrows, q, s, headers, quant_tables(q))
    return JpegTiles(payload, offsets, (cols, nrows), row0, tile, overlap, q, s)
