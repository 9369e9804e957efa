"""Packed code maps: lossless per-patch rANS entropy coding of stored code maps on the GPU.

A code map (``compress_slide``'s uint8 map, or an int64 one) spends a full byte or more per code whatever
the codes' distribution.  ``pack_code_map`` codes it with one static frequency table per map and one rANS
stream per code tile (patch), so that a region of patches can be unpacked without touching the rest;
``unpack_code_map(packed, region)`` returns exactly the map window that ``decompress_region`` /
``score_region`` take.  The container format (version 1) is defined in DESIGN.md section 4.13;
tests/codemap_pack_oracle.py restates it in numpy.

    code_map = compress_slide(...)                       # uint8 [rows*th, cols*tw] on the GPU
    packed = pack_code_map(code_map, (32, 32))
    save_packed("slide.vqpk", packed)
    packed = load_packed("slide.vqpk", device)
    window = unpack_code_map(packed, region=(r0, c0, nr, nc))
    pixels = decompress_region(model, window, (32, 32))
"""
from __future__ import annotations

import struct
import zlib
from dataclasses import dataclass, field
from pathlib import Path
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch

from . import engine as E

Tensor = torch.Tensor

MAGIC = b"VQPK"
VERSION = 1
SCALE_BITS = 14                 # frequencies sum to 2^14
MAX_SCALE_BITS = 14
MAX_CODES = 1024                # the quantiser's codebook limit
MAX_TILE_CODES = 16384          # th * tw
HEADER = struct.Struct("<4sHHQQIIII")     # magic, version, dtype, rows, cols, th, tw, K, S
DTYPE_CODES = {torch.uint8: 0, torch.int64: 1}
DTYPES = {v: k for k, v in DTYPE_CODES.items()}


def quantise_frequencies(counts, scale_bits: int = SCALE_BITS) -> np.ndarray:
    """The static table of a map from its exact code counts: f = max(1, floor(n 2^S / N)) for present
    codes, 0 for absent ones; then the difference to 2^S is settled one unit per code, codes ordered by
    count (descending, ties to the lower code): a deficit adds 1 to the first codes of that order, an
    excess takes 1 from each code with f > 1 in that order, pass after pass, until the sum is 2^S."""
    n = np.asarray(counts, dtype=np.int64)
    total, m = int(n.sum()), int((n > 0).sum())
    M = 1 << scale_bits
    if n.ndim != 1 or total <= 0 or (n < 0).any():
        raise ValueError("quantise_frequencies needs a 1-D array of non-negative counts with a positive sum")
    if m > M:
        raise ValueError(f"{m} distinct codes do not fit a table of total 2^{scale_bits}")
    if total >= 1 << 48:
        raise ValueError("more than 2^48 codes")
    present = n > 0
    f = np.zeros(n.shape, np.int64)
    f[present] = np.maximum(1, (n[present] * M) // total)
    order = np.lexsort((np.arange(n.size), -n))
    order = order[present[order]]
    d = M - int(f.sum())
    while d > 0:
        take = min(d, order.size)
        f[order[:take]] += 1
        d -= take
    while d < 0:
        elig = order[f[order] > 1]
        take = min(-d, elig.size)
        f[elig[:take]] -= 1
        d += take
    return f.astype(np.uint32)


class PackedIntegrityError(ValueError):
    """Raised by ``unpack_code_map`` when patches fail the stream check.  ``code_map`` holds the decoded
    region (the other patches are decoded as usual), ``flags`` the per-patch flags, ``patches`` the
    (row, col) map positions of the failing patches."""

    def __init__(self, msg: str, code_map: Tensor, flags: Tensor, patches):
        super().__init__(msg)
        self.code_map, self.flags, self.patches = code_map, flags, patches


@dataclass
class PackedCodeMap:
    """A packed code map on a device: ``freq`` int32 [k] (the quantised table, summing to 2^scale_bits),
    ``offsets`` int64 [P + 1] (stream p is ``payload[offsets[p]:offsets[p + 1]]``), ``payload`` uint8;
    ``grid`` (rows, cols) in patches, ``code_hw`` (th, tw), ``k`` codes, ``counts`` the exact int64 [k]
    code counts it was packed from (None after ``from_bytes``: they are not stored)."""
    freq: Tensor
    offsets: Tensor
    payload: Tensor
    grid: Tuple[int, int]
    code_hw: Tuple[int, int]
    k: int
    counts: Optional[Tensor] = None
    scale_bits: int = SCALE_BITS
    source_dtype: torch.dtype = torch.uint8
    freq_host: np.ndarray = field(default=None, repr=False)
    offsets_host: np.ndarray = field(default=None, repr=False)

    def __post_init__(self):
        if self.freq_host is None:
            self.freq_host = self.freq.cpu().numpy().astype(np.uint32)
        if self.offsets_host is None:
            self.offsets_host = self.offsets.cpu().numpy().astype(np.int64)

    @property
    def n_patches(self) -> int:
        return self.grid[0] * self.grid[1]

    @property
    def n_codes(self) -> int:
        return self.n_patches * self.code_hw[0] * self.code_hw[1]

    @property
    def map_shape(self) -> Tuple[int, int]:
        return self.grid[0] * self.code_hw[0], self.grid[1] * self.code_hw[1]

    @property
    def payload_bytes(self) -> int:
        return int(self.offsets_host[-1])

    def nbytes(self) -> int:
        """Size of the whole container (header, table, offsets, CRC, payload)."""
        return HEADER.size + 4 * self.k + 8 * (self.n_patches + 1) + 4 + self.payload_bytes

    def bits_per_code(self) -> float:
        """Container bits per code (the raw map spends 8 per code as uint8, 64 as int64)."""
        return 8.0 * self.nbytes() / self.n_codes

    def bits_per_pixel(self, patch_hw: Sequence[int]) -> float:
        """Container bits per slide pixel for patches of ``patch_hw`` pixels."""
        return 8.0 * self.nbytes() / (self.n_patches * int(patch_hw[0]) * int(patch_hw[1]))

    def to_bytes(self) -> bytes:
        payload = self.payload.cpu().numpy().tobytes()
        rows, cols = self.map_shape
        return b"".join((
            HEADER.pack(MAGIC, VERSION, DTYPE_CODES[self.source_dtype], rows, cols, self.code_hw[0],
                        self.code_hw[1], self.k, self.scale_bits),
            self.freq_host.astype("<u4").tobytes(),
            self.offsets_host.astype("<u8").tobytes(),
            struct.pack("<I", zlib.crc32(payload)),
            payload))

    @classmethod
    def from_bytes(cls, buf: Union[bytes, bytearray, memoryview], device) -> "PackedCodeMap":
        """Parse and validate a version-1 container (ValueError on any mismatch) onto ``device``."""
        buf = memoryview(buf).cast("B")
        if len(buf) < HEADER.size:
            raise ValueError(f"packed code map: {len(buf)} bytes is shorter than the header")
        magic, version, dtc, rows, cols, th, tw, k, s = HEADER.unpack_from(buf, 0)
        if magic != MAGIC:
            raise ValueError(f"packed code map: bad magic {bytes(magic)!r}")
        if version != VERSION:
            raise ValueError(f"packed code map: version {version} is not supported (only {VERSION})")
        if dtc not in DTYPES:
            raise ValueError(f"packed code map: unknown source dtype code {dtc}")
        if th <= 0 or tw <= 0 or rows <= 0 or cols <= 0 or rows % th or cols % tw or th * tw > MAX_TILE_CODES:
            raise ValueError(f"packed code map: a {rows} x {cols} map is not a grid of {th} x {tw} tiles")
        if not 1 <= k <= MAX_CODES or not 1 <= s <= MAX_SCALE_BITS:
            raise ValueError(f"packed code map: K = {k} or S = {s} out of range")
        grid = (rows // th, cols // tw)
        p = grid[0] * grid[1]
        pos = HEADER.size
        need = pos + 4 * k + 8 * (p + 1) + 4
        if len(buf) < need:
            raise ValueError(f"packed code map: truncated ({len(buf)} bytes, the tables alone need {need})")
        freq = np.frombuffer(buf, "<u4", k, pos).astype(np.uint32)
        pos += 4 * k
        off_u = np.frombuffer(buf, "<u8", p + 1, pos)
        pos += 8 * (p + 1)
        (crc,) = struct.unpack_from("<I", buf, pos)
        pos += 4
        if int(freq.astype(np.int64).sum()) != 1 << s:
            raise ValueError(f"packed code map: frequencies sum to {int(freq.sum())}, not 2^{s}")
        if (off_u > np.uint64(1 << 62)).any():
            raise ValueError("packed code map: offsets out of range")
        off = off_u.astype(np.int64)
        check_offsets(off, th * tw)
        if len(buf) - pos != off[-1]:
            raise ValueError(f"packed code map: payload is {len(buf) - pos} bytes, the offsets say {off[-1]}")
        payload = bytes(buf[pos:])
        if zlib.crc32(payload) != crc:
            raise ValueError("packed code map: payload CRC32 mismatch")
        dev = torch.device(device)
        return cls(freq=torch.from_numpy(freq.astype(np.int32)).to(dev), offsets=torch.from_numpy(off).to(dev),
                   payload=torch.frombuffer(bytearray(payload), dtype=torch.uint8).to(dev) if payload
                   else torch.empty(0, dtype=torch.uint8, device=dev),
                   grid=grid, code_hw=(th, tw), k=k, counts=None, scale_bits=s, source_dtype=DTYPES[dtc],
                   freq_host=freq, offsets_host=off)


def check_offsets(off: np.ndarray, n: int) -> None:
    """Offsets start at 0 and step by an even number of bytes in [4, 4 + 2 n] (ValueError otherwise)."""
    if off[0] != 0:
        raise ValueError("packed code map: the first offset is not 0")
    d = np.diff(off)
    if (d < 0).any():
        raise ValueError("packed code map: offsets are not monotone")
    if (d < 4).any() or (d > 4 + 2 * n).any() or (d & 1).any():
        bad = int(np.flatnonzero((d < 4) | (d > 4 + 2 * n) | ((d & 1) == 1))[0])
        raise ValueError(f"packed code map: patch {bad} has a {int(d[bad])}-byte stream "
                         f"(streams are even, 4 .. {4 + 2 * n} bytes)")


def _check_map(code_map: Tensor, code_hw: Sequence[int]) -> Tuple[Tensor, int, int]:
    E.require_cuda(code_map, "pack_code_map")
    if code_map.dim() != 2:
        raise ValueError(f"code_map must be 2-D, got shape {tuple(code_map.shape)}")
    if code_map.dtype not in (torch.uint8, torch.int64):
        if code_map.dtype.is_floating_point or code_map.dtype.is_complex:
            raise ValueError(f"code_map must hold integer codes, got {code_map.dtype}")
        code_map = code_map.long()
    th, tw = (int(v) for v in code_hw)
    if th <= 0 or tw <= 0 or code_map.shape[0] % th or code_map.shape[1] % tw:
        raise ValueError(f"code map {tuple(code_map.shape)} is not a grid of {th} x {tw} code tiles")
    if th * tw > MAX_TILE_CODES:
        raise ValueError(f"code tiles of {th} x {tw} exceed {MAX_TILE_CODES} codes")
    return code_map.contiguous(), th, tw


@torch.no_grad()
def pack_code_map(code_map: Tensor, code_hw: Sequence[int], k: Optional[int] = None) -> PackedCodeMap:
    """Entropy-code a uint8 / int64 code map [rows*th, cols*tw] of th x tw code tiles on its device.
    ``k`` (default: largest code + 1, at most 1024) is the alphabet of the table; codes must lie in
    [0, k).  The map's exact histogram is taken on the GPU, quantised on the host
    (``quantise_frequencies``), then every patch is coded by the rANS kernels."""
    source = code_map.dtype
    code_map, th, tw = _check_map(code_map, code_hw)
    if k is None:
        lo, hi = int(code_map.min()), int(code_map.max())
        if lo < 0:
            raise ValueError(f"code map holds a negative code ({lo})")
        k = hi + 1
    k = int(k)
    if not 1 <= k <= MAX_CODES:
        raise ValueError(f"k = {k} is outside [1, {MAX_CODES}]")
    counts, invalid = E.codemap_histogram(code_map, k)
    if int(invalid):
        raise ValueError(f"code map holds {int(invalid)} codes outside [0, {k})")
    freq = quantise_frequencies(counts.cpu().numpy(), SCALE_BITS)
    offsets, buf = E.codemap_pack(code_map, (th, tw), freq, SCALE_BITS)
    off = offsets.cpu().numpy()
    check_offsets(off, th * tw)
    grid = (code_map.shape[0] // th, code_map.shape[1] // tw)
    return PackedCodeMap(freq=torch.from_numpy(freq.astype(np.int32)).to(code_map.device), offsets=offsets,
                         payload=buf[:int(off[-1])].clone(), grid=grid, code_hw=(th, tw), k=k, counts=counts,
                         scale_bits=SCALE_BITS, source_dtype=torch.uint8 if source == torch.uint8 else torch.int64,
                         freq_host=freq, offsets_host=off)


@torch.no_grad()
def unpack_code_map(packed: PackedCodeMap, region: Optional[Sequence[int]] = None,
                    dtype: torch.dtype = torch.uint8) -> Tensor:
    """Decode the patches ``region = (r0, c0, nr, nc)`` (default: all) of a packed map into a
    [nr*th, nc*tw] map of ``dtype`` (uint8 for k <= 256, or int64) on the packed map's device -- the map
    window ``decompress_region`` / ``score_region`` take.  Raises ``PackedIntegrityError`` (a
    ValueError) naming the patches whose stream did not decode back to the encoder's initial state with
    its words exactly consumed."""
    rows, cols = packed.grid
    r0, c0, nr, nc = (int(v) for v in (region if region is not None else (0, 0, rows, cols)))
    if r0 < 0 or c0 < 0 or nr <= 0 or nc <= 0 or r0 + nr > rows or c0 + nc > cols:
        raise ValueError(f"region {(r0, c0, nr, nc)} leaves the {rows} x {cols} patch grid")
    if dtype not in (torch.uint8, torch.int64):
        raise ValueError(f"unpack_code_map writes uint8 or int64 maps, not {dtype}")
    if dtype == torch.uint8 and packed.k > 256:
        raise ValueError(f"a uint8 map holds at most 256 codes, this one has k = {packed.k}; use torch.int64")
    out, flags = E.codemap_unpack(packed.payload, packed.offsets, packed.offsets_host, packed.map_shape,
                                  packed.code_hw, packed.freq_host, packed.scale_bits, (r0, c0, nr, nc), dtype)
    bad = torch.nonzero(flags).cpu().tolist()
    if bad:
        patches = [(r0 + i, c0 + j) for i, j in bad]
        shown = ", ".join(str(p) for p in patches[:8]) + (" ..." if len(patches) > 8 else "")
        raise PackedIntegrityError(f"packed code map: {len(patches)} patch stream(s) failed the integrity "
                                   f"check at (row, col) {shown}", out, flags, patches)
    return out


def save_packed(path: Union[str, Path], packed: PackedCodeMap) -> Path:
    path = Path(path)
    path.write_bytes(packed.to_bytes())
    return path


def load_packed(path: Union[str, Path], device) -> PackedCodeMap:
    return PackedCodeMap.from_bytes(Path(path).read_bytes(), device)
