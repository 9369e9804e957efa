"""Near-lossless residual layers of stored code maps: a guaranteed per-pixel error bound, down to exact
reconstruction, entropy-coded on the GPU.

The code map is the base layer.  A residual layer stores, per patch, the difference between the original
slide and the base decode, quantised so that no byte is off by more than ``e`` (JPEG-LS near-lossless
quantisation; ``e = 0`` is lossless), rANS-coded with one table per patch and 32 interleaved lanes.  Each
patch is a self-contained chunk, so regions decode at random, and carries two Adler-32 checks: of the base
pixels it was made against (a map decoded by another model, precision mode or kernel is reported by name)
and of the reconstruction.  The format (version 1) is defined in DESIGN.md section 4.15;
tests/residual_oracle.py restates it in numpy.

    layer = encode_residual(model, code_map, (32, 32), slide_u8, max_error=0)
    save_residual("slide.vqrl", layer)
    layer = load_residual("slide.vqrl", device)
    pixels = decompress_region_exact(model, code_map, (32, 32), layer, region=(r0, c0, nr, nc))
"""
from __future__ import annotations

import struct
import zlib
from dataclasses import dataclass, field
from pathlib import Path
from typing import List, Tuple, Union

import numpy as np
import torch

Tensor = torch.Tensor

MAGIC = b"VQRL"
VERSION = 1
SCALE_BITS = 14
LANES = 32
MAX_ERROR = 127
CHUNK_HEADER = 768              # 256 x u16 frequencies, 32 x u32 word counts, 32 x u32 final states
MAX_PATCH_PIXELS = 1 << 20
HEADER = struct.Struct("<4sHHHQQIIHH")     # magic, version, e, mode, rows, cols, H, W, S, J
MODES = ("fp32", "fp16", "fp32tc")
FLAG_STREAM, FLAG_BASE, FLAG_OUTPUT = 1, 2, 4
CAUSES = ((FLAG_STREAM, "stream"), (FLAG_BASE, "base mismatch"), (FLAG_OUTPUT, "output mismatch"))


class ResidualIntegrityError(ValueError):
    """Raised by ``decompress_region_exact`` when patches fail their checks.  ``pixels`` holds the decoded
    region (the other patches are exact within the layer's bound), ``flags`` the per-patch flags [nr, nc]
    (bit 0 stream, bit 1 base mismatch, bit 2 output mismatch), ``patches`` the (row, col) grid positions of
    the failing patches and ``causes`` the cause names of each."""

    def __init__(self, msg: str, pixels: Tensor, flags: Tensor, patches, causes):
        super().__init__(msg)
        self.pixels, self.flags, self.patches, self.causes = pixels, flags, patches, causes


def flag_causes(flag: int) -> List[str]:
    return [name for bit, name in CAUSES if flag & bit]


@dataclass
class ResidualLayer:
    """A residual layer on a device: ``payload`` uint8 (chunk p is ``payload[offsets[p]:offsets[p + 1]]``),
    ``offsets`` int64 [P + 1], ``adler`` int32 [P, 2] (the uint32 Adler-32 bits of the base pixels and of the
    reconstruction); ``max_error`` the bound e, ``precision`` the decoder mode the base was decoded in,
    ``grid`` (rows, cols) in patches, ``patch_hw`` (H, W) in pixels."""
    payload: Tensor
    offsets: Tensor
    adler: Tensor
    max_error: int
    precision: str
    grid: Tuple[int, int]
    patch_hw: Tuple[int, int]
    offsets_host: np.ndarray = field(default=None, repr=False)

    def __post_init__(self):
        if self.offsets_host is None:
            self.offsets_host = self.offsets.cpu().numpy().astype(np.int64)

    @property
    def n_patches(self) -> int:
        return self.grid[0] * self.grid[1]

    @property
    def payload_bytes(self) -> int:
        return int(self.offsets_host[-1])

    def nbytes(self) -> int:
        """Size of the whole container (header, offsets, checksums, CRC, payload)."""
        return HEADER.size + 8 * (self.n_patches + 1) + 8 * self.n_patches + 4 + self.payload_bytes

    def bits_per_pixel(self) -> float:
        """Container bits per slide pixel (an RGB pixel is 24 bits raw)."""
        return 8.0 * self.nbytes() / (self.n_patches * self.patch_hw[0] * self.patch_hw[1])

    def to_bytes(self) -> bytes:
        payload = self.payload.cpu().numpy().tobytes()
        return b"".join((
            HEADER.pack(MAGIC, VERSION, self.max_error, MODES.index(self.precision), self.grid[0], self.grid[1],
                        self.patch_hw[0], self.patch_hw[1], SCALE_BITS, LANES),
            self.offsets_host.astype("<u8").tobytes(),
            self.adler.cpu().numpy().astype("<i4").tobytes(),
            struct.pack("<I", zlib.crc32(payload)),
            payload))

    @classmethod
    def from_bytes(cls, buf: Union[bytes, bytearray, memoryview], device) -> "ResidualLayer":
        """Parse and validate a version-1 container (ValueError on any mismatch) onto ``device``."""
        buf = memoryview(buf).cast("B")
        if len(buf) < HEADER.size:
            raise ValueError(f"residual layer: {len(buf)} bytes is shorter than the header")
        magic, version, e, mode, rows, cols, h, w, s, j = HEADER.unpack_from(buf, 0)
        if magic != MAGIC:
            raise ValueError(f"residual layer: bad magic {bytes(magic)!r}")
        if version != VERSION:
            raise ValueError(f"residual layer: version {version} is not supported (only {VERSION})")
        if mode >= len(MODES):
            raise ValueError(f"residual layer: unknown precision mode code {mode}")
        if e > MAX_ERROR:
            raise ValueError(f"residual layer: error bound {e} exceeds {MAX_ERROR}")
        if s != SCALE_BITS or j != LANES:
            raise ValueError(f"residual layer: S = {s}, J = {j} (version 1 has S = {SCALE_BITS}, J = {LANES})")
        if rows <= 0 or cols <= 0 or h <= 0 or w <= 0 or h * w > MAX_PATCH_PIXELS:
            raise ValueError(f"residual layer: a {rows} x {cols} grid of {h} x {w} patches is not supported")
        p = rows * cols
        pos = HEADER.size
        need = pos + 8 * (p + 1) + 8 * p + 4
        if len(buf) < need:
            raise ValueError(f"residual layer: truncated ({len(buf)} bytes, the tables alone need {need})")
        off_u = np.frombuffer(buf, "<u8", p + 1, pos)
        pos += 8 * (p + 1)
        adler = np.frombuffer(buf, "<i4", 2 * p, pos).reshape(p, 2).astype(np.int32)
        pos += 8 * p
        (crc,) = struct.unpack_from("<I", buf, pos)
        pos += 4
        if (off_u > np.uint64(1 << 62)).any():
            raise ValueError("residual layer: offsets out of range")
        off = off_u.astype(np.int64)
        check_offsets(off, 3 * h * w)
        if len(buf) - pos != off[-1]:
            raise ValueError(f"residual layer: payload is {len(buf) - pos} bytes, the offsets say {off[-1]}")
        payload = bytes(buf[pos:])
        if zlib.crc32(payload) != crc:
            raise ValueError("residual layer: payload CRC32 mismatch")
        dev = torch.device(device)
        return cls(payload=torch.frombuffer(bytearray(payload), dtype=torch.uint8).to(dev),
                   offsets=torch.from_numpy(off).to(dev), adler=torch.from_numpy(adler).to(dev), max_error=e,
                   precision=MODES[mode], grid=(rows, cols), patch_hw=(h, w), offsets_host=off)


def check_offsets(off: np.ndarray, n: int) -> None:
    """Offsets start at 0 and step by an even number of bytes in [768, 768 + 2 n] (ValueError otherwise)."""
    if off[0] != 0:
        raise ValueError("residual layer: the first offset is not 0")
    d = np.diff(off)
    bad = (d < CHUNK_HEADER) | (d > CHUNK_HEADER + 2 * n) | ((d & 1) == 1)
    if bad.any():
        i = int(np.flatnonzero(bad)[0])
        raise ValueError(f"residual layer: patch {i} has a {int(d[i])}-byte chunk "
                         f"(chunks are even, {CHUNK_HEADER} .. {CHUNK_HEADER + 2 * n} bytes)")


def check_max_error(max_error) -> int:
    if isinstance(max_error, bool) or not isinstance(max_error, (int, np.integer)) \
            or not 0 <= int(max_error) <= MAX_ERROR:
        raise ValueError(f"max_error must be an integer in [0, {MAX_ERROR}], got {max_error!r}")
    return int(max_error)


def save_residual(path: Union[str, Path], layer: ResidualLayer) -> Path:
    path = Path(path)
    path.write_bytes(layer.to_bytes())
    return path


def load_residual(path: Union[str, Path], device) -> ResidualLayer:
    return ResidualLayer.from_bytes(Path(path).read_bytes(), device)
