"""numpy restatement of the residual layer, version 1 (DESIGN.md section 4.15): the bytes it produces are
what the GPU encoder must produce.  Vectorised over patches and the 32 lanes, looping over the steps.

    symbol   e = 0: s = (x - xh) & 255;  e >= 1: k = sign(d) floor((|d| + e) / (2e + 1)), s = k & 255
    decode   e = 0: x' = (xh + s) & 255; e >= 1: x' = clamp(xh + int8(s) (2e + 1), 0, 255)
    table    packing.quantise_frequencies of the patch's 256 symbol counts, S = 14
    chunk    256 x <u2 freq | 32 x <u4 lane word counts | 32 x <u4 final lane states | lane 0 words, ..., lane 31
             words, each in decoder order; symbol i -> lane i mod 32, coded last to first from x = 2^16
    adler    zlib.adler32 of a patch's bytes in canvas order
    container  "<4sHHHQQIIHH" (b"VQRL", 1, e, mode, rows, cols, H, W, 14, 32), (P + 1) x <u8 offsets,
             P x (<u4 base Adler, <u4 output Adler), <u4 CRC32 of the payload, payload
"""
from __future__ import annotations

import struct
import zlib

import numpy as np

from vqae_b200.packing import quantise_frequencies

L = 1 << 16
S = 14
J = 32
M = 1 << S


def symbols(x, xh, e: int) -> np.ndarray:
    d = np.asarray(x, np.int64) - np.asarray(xh, np.int64)
    if e == 0:
        return (d & 255).astype(np.uint8)
    k = np.sign(d) * ((np.abs(d) + e) // (2 * e + 1))
    return (k & 255).astype(np.uint8)


def reconstruct(xh, s, e: int) -> np.ndarray:
    xh = np.asarray(xh, np.int64)
    s = np.asarray(s, np.uint8)
    if e == 0:
        return ((xh + s) & 255).astype(np.uint8)
    return np.clip(xh + s.view(np.int8).astype(np.int64) * (2 * e + 1), 0, 255).astype(np.uint8)


def adler32(b) -> int:
    """The parallel form: A = 1 + sum b, B = n + sum (n - i) b_i, both mod 65521."""
    b = np.asarray(b, np.int64).ravel()
    n = b.size
    a = (1 + int(b.sum())) % 65521
    bb = (n + int(((n - np.arange(n)) * b).sum())) % 65521
    return (bb << 16) | a


def patches(canvas: np.ndarray, h: int, w: int) -> np.ndarray:
    """[P, 3 h w] uint8: the patches of a [rows h, cols w, 3] canvas in row-major patch order, canvas order."""
    rows, cols = canvas.shape[0] // h, canvas.shape[1] // w
    return canvas.reshape(rows, h, cols, w, 3).transpose(0, 2, 1, 3, 4).reshape(rows * cols, h * w * 3)


def tables(sym: np.ndarray) -> np.ndarray:
    return np.stack([quantise_frequencies(np.bincount(s, minlength=256), S) for s in sym])


def encode(sym: np.ndarray):
    """Chunks (list of bytes) and tables [P, 256] of the symbol rows sym [P, n]."""
    P, n = sym.shape
    freq = tables(sym).astype(np.uint64)
    start = np.concatenate([np.zeros((P, 1), np.uint64), np.cumsum(freq, 1)[:, :-1]], 1)
    steps = -(-n // J)
    pad = np.zeros((P, steps * J), np.int64)
    pad[:, :n] = sym
    x = np.full((P, J), L, np.uint64)
    words = np.zeros((P, J, steps), np.uint16)
    w = np.zeros((P, J), np.int64)
    rows = np.arange(P)[:, None].repeat(J, 1)
    for st in range(steps - 1, -1, -1):
        live = (st * J + np.arange(J))[None, :].repeat(P, 0) < n
        s = pad[:, st * J:(st + 1) * J]
        f = np.take_along_axis(freq, s, 1)
        c = np.take_along_axis(start, s, 1)
        assert (f[live] > 0).all()
        emit = live & (x >= (f << np.uint64(32 - S)))
        pi, li = rows[emit], np.nonzero(emit)[1]
        words[pi, li, w[emit]] = (x[emit] & np.uint64(0xffff)).astype(np.uint16)
        w[emit] += 1
        x[emit] >>= np.uint64(16)
        fl = np.where(live, f, 1)
        nx = ((x // fl) << np.uint64(S)) + x % fl + c
        x = np.where(live, nx, x)
    assert (x < (1 << 32)).all()
    chunks = []
    for p in range(P):
        body = b"".join(words[p, j, :w[p, j]][::-1].astype("<u2").tobytes() for j in range(J))
        chunks.append(freq[p].astype("<u2").tobytes() + w[p].astype("<u4").tobytes()
                      + x[p].astype("<u4").tobytes() + body)
    return chunks, freq.astype(np.uint32)


def decode(chunk: bytes, n: int):
    """(symbols [n], stream_ok) of one chunk."""
    freq = np.frombuffer(chunk, "<u2", 256, 0).astype(np.uint64)
    w = np.frombuffer(chunk, "<u4", J, 512).astype(np.int64)
    x = np.frombuffer(chunk, "<u4", J, 640).astype(np.uint64)
    ok = int(freq.sum()) == M and len(chunk) == 768 + 2 * int(w.sum())
    start = np.concatenate([[0], np.cumsum(freq)[:-1]]).astype(np.uint64)
    table = np.repeat(np.arange(256), freq.astype(np.int64)) if ok else np.zeros(M, np.int64)
    pre = np.concatenate([[0], np.cumsum(w)[:-1]])
    body = np.frombuffer(chunk, "<u2", (len(chunk) - 768) // 2, 768).astype(np.uint64)
    k = np.zeros(J, np.int64)
    out = np.zeros(-(-n // J) * J, np.uint8)
    for st in range(-(-n // J)):
        live = st * J + np.arange(J) < n
        slot = x & np.uint64(M - 1)
        s = table[slot.astype(np.int64)]
        nx = freq[s] * (x >> np.uint64(S)) + slot - start[s]
        renorm = live & (nx < L)
        idx = np.minimum(pre + k, body.size - 1) if body.size else np.zeros(J, np.int64)
        v = np.where(renorm & (k < w), body[idx] if body.size else 0, 0).astype(np.uint64)
        nx = np.where(renorm, (nx << np.uint64(16)) | v, nx)
        k += renorm
        x = np.where(live, nx, x)
        out[st * J:(st + 1) * J] = s
    ok = ok and bool((x == L).all()) and bool((k == w).all())
    return out[:n], ok


def layer(x_canvas: np.ndarray, base_canvas: np.ndarray, h: int, w: int, e: int):
    """(offsets int64 [P + 1], payload bytes, adler uint32 [P, 2], x' canvas) of a whole canvas."""
    xp, bp = patches(x_canvas, h, w), patches(base_canvas, h, w)
    sym = symbols(xp, bp, e)
    chunks, _ = encode(sym)
    out = reconstruct(bp, sym, e)
    adler = np.array([[adler32(b), adler32(o)] for b, o in zip(bp, out)], np.uint32)
    offsets = np.concatenate([[0], np.cumsum([len(c) for c in chunks])]).astype(np.int64)
    rows, cols = x_canvas.shape[0] // h, x_canvas.shape[1] // w
    canvas = out.reshape(rows, cols, h, w, 3).transpose(0, 2, 1, 3, 4).reshape(x_canvas.shape)
    return offsets, b"".join(chunks), adler, canvas


def container(rows: int, cols: int, h: int, w: int, e: int, mode: int, offsets, adler, payload: bytes,
              version: int = 1) -> bytes:
    return (struct.pack("<4sHHHQQIIHH", b"VQRL", version, e, mode, rows, cols, h, w, S, J)
            + np.asarray(offsets, "<u8").tobytes() + np.asarray(adler, np.uint32).astype("<u4").tobytes()
            + struct.pack("<I", zlib.crc32(payload)) + payload)


def entropy_bytes(sym: np.ndarray) -> float:
    """Sum over patches of the empirical (order-0) entropy of each patch's symbols, in bytes."""
    total = 0.0
    for s in sym:
        c = np.bincount(s, minlength=256).astype(np.float64)
        p = c[c > 0] / s.size
        total += float(-(c[c > 0] * np.log2(p)).sum()) / 8
    return total
