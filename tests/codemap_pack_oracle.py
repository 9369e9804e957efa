"""numpy restatement of the packed code map format, version 1 (DESIGN.md section 4.13): the bytes it
produces are what the GPU packer must produce.  Vectorised over patches, looping over the codes of a tile.

    table    f[s] = max(1, floor(n_s 2^S / N)) for present codes, then the difference to 2^S settled one
             unit per code in (count descending, code ascending) order: +1 for a deficit, -1 on codes with
             f > 1 pass after pass for an excess
    stream   rANS, 32-bit state, L = 2^16, 16-bit words; codes of a tile coded last to first from x = L;
             the final state (4 bytes LE), then the words in decoder order (2 bytes LE)
    container  header "<4sHHQQIIII" (magic "VQPK", version 1, dtype 0 = uint8 / 1 = int64, rows, cols,
             th, tw, K, S), K x <u4 frequencies, (P + 1) x <u8 offsets, <u4 CRC32 of the payload, payload
"""
from __future__ import annotations

import struct
import zlib

import numpy as np

L = 1 << 16
S_DEFAULT = 14


def quantise(counts, S: int = S_DEFAULT) -> np.ndarray:
    counts = [int(v) for v in counts]
    total = sum(counts)
    M = 1 << S
    f = [0 if n == 0 else max(1, n * M // total) for n in counts]
    order = sorted((s for s in range(len(counts)) if counts[s] > 0), key=lambda s: (-counts[s], s))
    d = M - sum(f)
    i = 0
    while d > 0:
        f[order[i % len(order)]] += 1
        d -= 1
        i += 1
    while d < 0:
        changed = False
        for s in order:
            if d == 0:
                break
            if f[s] > 1:
                f[s] -= 1
                d += 1
                changed = True
        assert changed
    return np.array(f, dtype=np.uint32)


def tiles(code_map: np.ndarray, th: int, tw: int) -> np.ndarray:
    """[P, th*tw] int64: patches in row-major patch order, codes in row-major order."""
    rows, cols = code_map.shape[0] // th, code_map.shape[1] // tw
    return code_map.astype(np.int64).reshape(rows, th, cols, tw).transpose(0, 2, 1, 3).reshape(rows * cols, th * tw)


def starts(freq) -> np.ndarray:
    f = np.asarray(freq, dtype=np.uint64)
    return np.concatenate(([0], np.cumsum(f)[:-1])).astype(np.uint64)


def encode(sym: np.ndarray, freq, S: int = S_DEFAULT):
    """Streams (list of bytes) of the patches sym [P, n]."""
    P, n = sym.shape
    f, c = np.asarray(freq, dtype=np.uint64), starts(freq)
    x = np.full(P, L, dtype=np.uint64)
    words = np.zeros((P, max(n, 1)), dtype=np.uint16)
    w = np.zeros(P, dtype=np.int64)
    for i in range(n - 1, -1, -1):
        fs, cs = f[sym[:, i]], c[sym[:, i]]
        assert (fs > 0).all()
        idx = np.flatnonzero(x >= (fs << np.uint64(32 - S)))
        words[idx, w[idx]] = (x[idx] & np.uint64(0xffff)).astype(np.uint16)
        w[idx] += 1
        x[idx] >>= np.uint64(16)
        x = ((x // fs) << np.uint64(S)) + x % fs + cs
    assert (x < (1 << 32)).all()
    return [struct.pack("<I", int(x[p])) + words[p, :w[p]][::-1].astype("<u2").tobytes() for p in range(P)]


def pack(code_map: np.ndarray, th: int, tw: int, k=None, S: int = S_DEFAULT):
    """(freq uint32 [k], offsets int64 [P + 1], payload bytes) of a code map."""
    sym = tiles(code_map, th, tw)
    k = int(sym.max()) + 1 if k is None else k
    freq = quantise(np.bincount(sym.ravel(), minlength=k), S)
    streams = encode(sym, freq, S)
    offsets = np.concatenate(([0], np.cumsum([len(s) for s in streams]))).astype(np.int64)
    return freq, offsets, b"".join(streams)


def decode(payload: bytes, offsets, freq, n: int, patches, S: int = S_DEFAULT):
    """(sym [len(patches), n], flags) decoded from the streams of ``patches`` (flags as the kernel's:
    1 final state != L, 2 words not exactly consumed)."""
    patches = np.asarray(patches, dtype=np.int64)
    f, c = np.asarray(freq, dtype=np.uint64), starts(freq)
    table = np.repeat(np.arange(len(f)), np.asarray(freq, dtype=np.int64))
    M = np.uint64((1 << S) - 1)
    Q = len(patches)
    x = np.zeros(Q, dtype=np.uint64)
    w = np.zeros(Q, dtype=np.int64)
    words = np.zeros((Q, n + 1), dtype=np.uint64)
    for q, p in enumerate(patches):
        b = payload[offsets[p]:offsets[p + 1]]
        x[q] = struct.unpack("<I", b[:4])[0]
        ws = np.frombuffer(b[4:], "<u2")
        w[q] = len(ws)
        words[q, :len(ws)] = ws
    k = np.zeros(Q, dtype=np.int64)
    out = np.zeros((Q, n), dtype=np.int64)
    rows = np.arange(Q)
    for i in range(n):
        slot = x & M
        s = table[slot.astype(np.int64)]
        x = f[s] * (x >> np.uint64(S)) + slot - c[s]
        r = np.flatnonzero(x < L)
        v = np.where(k[r] < w[r], words[rows[r], np.minimum(k[r], n)], 0).astype(np.uint64)
        x[r] = (x[r] << np.uint64(16)) | v
        k[r] += 1
        out[:, i] = s
    flags = (x != L).astype(np.uint8) | ((k != w).astype(np.uint8) << 1)
    return out, flags


def ideal_bytes(code_map: np.ndarray, freq, S: int = S_DEFAULT) -> float:
    """Length in bytes of the ideal code of the map under the table: sum of -log2(f / 2^S) / 8."""
    n = np.bincount(code_map.astype(np.int64).ravel(), minlength=len(freq))
    f = np.asarray(freq, dtype=np.float64)
    used = n > 0
    return float((n[used] * (S - np.log2(f[used]))).sum() / 8)


def container(rows: int, cols: int, th: int, tw: int, freq, offsets, payload: bytes, dtype_code: int = 0,
              S: int = S_DEFAULT) -> bytes:
    return (struct.pack("<4sHHQQIIII", b"VQPK", 1, dtype_code, rows, cols, th, tw, len(freq), S)
            + np.asarray(freq, dtype="<u4").tobytes() + np.asarray(offsets, dtype="<u8").tobytes()
            + struct.pack("<I", zlib.crc32(payload)) + payload)
