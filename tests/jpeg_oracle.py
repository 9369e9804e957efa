"""numpy restatement of the baseline JPEG tile encoder (DESIGN.md section 4.16): the bytes it produces are
what ``PIL.Image.fromarray(img).save(buf, "JPEG", quality=q, subsampling=s)`` writes and what the GPU
encoder must write.  Headers and tables come from vqae_b200.jpeg (checked against Pillow by the CPU
tests); the scan is computed here.

    colour   jccolor.c, FIX(x) = round(x 2^16):  Y = (FIX(.299) r + FIX(.587) g + FIX(.114) b + 2^15) >> 16,
             Cb = (-FIX(.16874) r - FIX(.33126) g + FIX(.5) b + (128 << 16) + 2^15 - 1) >> 16, Cr likewise
    edges    full-resolution planes sample (min(y, H-1), min(x, W-1)) out to whole blocks; 4:2:0 chroma is
             converted with columns clamped out to 16 ceil(ceil(W/2)/8) and rows out to 2 ceil(H/2),
             downsampled 2 x 2 as (sum + 1 | 2) >> 2 (1 on even, 2 on odd output columns), and its last
             row replicated down to 8 ceil(ceil(H/2)/8)
    FDCT     jfdctint islow, CONST_BITS 13, PASS1_BITS 2, samples - 128
    quant    sign(v) floor((|v| + 4Q) / 8Q)
    MCUs     4:2:0: Y00 Y01 Y10 Y11 Cb Cr per 16 x 16, 4:4:4: Y Cb Cr per 8 x 8; a Y block outside the image's
             blocks is a dummy: zero AC, the quantised DC of the block before it
    scan     Annex K Huffman codes, DC predictors per component over the scan, MSB first, 0xFF -> 0xFF 00,
             the last byte padded with 1 bits, then EOI
"""
from __future__ import annotations

import numpy as np

from vqae_b200 import jpeg as J

FIX = {k: int(v * 8192 + 0.5) for k, v in dict(
    a=0.298631336, b=0.390180644, c=0.541196100, d=0.765366865, e=0.899976223, f=1.175875602, g=1.501321110,
    h=1.847759065, i=1.961570560, j=2.053119869, k=2.562915447, l=3.072711026).items()}


def ycc(img: np.ndarray):
    F = lambda x: int(x * 65536 + 0.5)   # noqa: E731
    r, g, b = (img[..., i].astype(np.int64) for i in range(3))
    y = (F(0.299) * r + F(0.587) * g + F(0.114) * b + (1 << 15)) >> 16
    cb = (-F(0.16874) * r - F(0.33126) * g + F(0.5) * b + (128 << 16) + (1 << 15) - 1) >> 16
    cr = (F(0.5) * r - F(0.41869) * g - F(0.08131) * b + (128 << 16) + (1 << 15) - 1) >> 16
    return y, cb, cr


def _descale(x, n):
    return (x + (1 << (n - 1))) >> n


def _fdct_1d(d, pass1: bool):
    """islow on the last axis of d (int64 [..., 8])."""
    sh = 13 - 2 if pass1 else 13 + 2
    t0, t7 = d[..., 0] + d[..., 7], d[..., 0] - d[..., 7]
    t1, t6 = d[..., 1] + d[..., 6], d[..., 1] - d[..., 6]
    t2, t5 = d[..., 2] + d[..., 5], d[..., 2] - d[..., 5]
    t3, t4 = d[..., 3] + d[..., 4], d[..., 3] - d[..., 4]
    t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
    o = np.empty_like(d)
    if pass1:
        o[..., 0], o[..., 4] = (t10 + t11) << 2, (t10 - t11) << 2
    else:
        o[..., 0], o[..., 4] = _descale(t10 + t11, 2), _descale(t10 - t11, 2)
    z1 = (t12 + t13) * FIX["c"]
    o[..., 2] = _descale(z1 + t13 * FIX["d"], sh)
    o[..., 6] = _descale(z1 - t12 * FIX["h"], sh)
    z1, z2, z3, z4 = t4 + t7, t5 + t6, t4 + t6, t5 + t7
    z5 = (z3 + z4) * FIX["f"]
    t4, t5, t6, t7 = t4 * FIX["a"], t5 * FIX["j"], t6 * FIX["l"], t7 * FIX["g"]
    z1, z2 = z1 * -FIX["e"], z2 * -FIX["k"]
    z3, z4 = z3 * -FIX["i"] + z5, z4 * -FIX["b"] + z5
    o[..., 7] = _descale(t4 + z1 + z3, sh)
    o[..., 5] = _descale(t5 + z2 + z4, sh)
    o[..., 3] = _descale(t6 + z2 + z3, sh)
    o[..., 1] = _descale(t7 + z1 + z4, sh)
    return o


def quantised_blocks(plane: np.ndarray, qt_zigzag: np.ndarray) -> np.ndarray:
    """int64 [bh, bw, 64] zigzag-ordered quantised coefficients of a plane of whole 8 x 8 blocks."""
    h, w = plane.shape
    blk = plane.reshape(h // 8, 8, w // 8, 8).transpose(0, 2, 1, 3).astype(np.int64) - 128
    blk = _fdct_1d(blk, True)                                             # rows
    blk = _fdct_1d(blk.swapaxes(-1, -2), False).swapaxes(-1, -2)          # columns
    v = blk.reshape(h // 8, w // 8, 64)[..., list(J.ZIGZAG)]
    d = 8 * qt_zigzag.astype(np.int64)
    a = (np.abs(v) + (d >> 1)) // d
    return np.where(v < 0, -a, a)


def _clamped(img, rows, cols):
    h, w = img.shape[:2]
    return img[np.minimum(np.arange(rows), h - 1)][:, np.minimum(np.arange(cols), w - 1)]


def _huff(counts_symbols):
    counts, symbols = counts_symbols
    table, code, k = {}, 0, 0
    for ln in range(1, 17):
        for _ in range(counts[ln - 1]):
            table[symbols[k]] = (code, ln)
            k += 1
            code += 1
        code <<= 1
    return table


DC = [_huff(J.DC_LUMINANCE), _huff(J.DC_CHROMINANCE)]
AC = [_huff(J.AC_LUMINANCE), _huff(J.AC_CHROMINANCE)]


def _cat(v: int) -> int:
    return abs(v).bit_length()


def scan(img: np.ndarray, quality: int, subsampling: int) -> bytes:
    """The entropy-coded segment (stuffed and padded, without EOI) of an RGB uint8 [H, W, 3] image."""
    h, w = img.shape[:2]
    qt = J.quant_tables(quality)
    cd = lambda a, b: -(-a // b)                                          # noqa: E731
    ybh, ybw = cd(h, 8), cd(w, 8)
    if subsampling == 2:
        y = quantised_blocks(ycc(_clamped(img, ybh * 8, ybw * 8))[0], qt[0])
        ch, cw = cd(h, 2), cd(w, 2)
        cbh, cbw = cd(ch, 8), cd(cw, 8)
        _, cb, cr = ycc(_clamped(img, 2 * ch, 16 * cbw))
        planes = []
        for p in (cb, cr):
            s = p[0::2, 0::2] + p[0::2, 1::2] + p[1::2, 0::2] + p[1::2, 1::2]
            s = (s + np.tile([1, 2], s.shape[1] // 2)[None, :]) >> 2
            planes.append(quantised_blocks(s[np.minimum(np.arange(cbh * 8), ch - 1)], qt[1]))
        mh, mw, order = cd(h, 16), cd(w, 16), ((0, 0, 0), (0, 0, 1), (0, 1, 0), (0, 1, 1), (1, 0, 0), (2, 0, 0))
        comps = [y, *planes]
    else:
        comps = [quantised_blocks(p, qt[min(i, 1)]) for i, p in enumerate(ycc(_clamped(img, ybh * 8, ybw * 8)))]
        mh, mw, order = ybh, ybw, ((0, 0, 0), (1, 0, 0), (2, 0, 0))
    out, pred = [], [0, 0, 0]
    for my in range(mh):
        for mx in range(mw):
            prev = None
            for ci, dy, dx in order:
                t = min(ci, 1)
                sc = 2 if (subsampling == 2 and ci == 0) else 1
                by, bx = my * sc + dy, mx * sc + dx
                if by < comps[ci].shape[0] and bx < comps[ci].shape[1]:
                    q = comps[ci][by, bx]
                else:
                    q = np.zeros(64, np.int64)
                    q[0] = prev[0]
                prev = q
                diff = int(q[0]) - pred[ci]
                pred[ci] = int(q[0])
                s = _cat(diff)
                out.append(DC[t][s])
                if s:
                    out.append(((diff if diff >= 0 else diff - 1) & ((1 << s) - 1), s))
                nz = np.flatnonzero(q[1:]) + 1
                last = 0
                for k in nz:
                    run, v = k - last - 1, int(q[k])
                    while run > 15:
                        out.append(AC[t][0xF0])
                        run -= 16
                    s = _cat(v)
                    out.append(AC[t][(run << 4) | s])
                    out.append(((v if v >= 0 else v - 1) & ((1 << s) - 1), s))
                    last = k
                if last != 63:
                    out.append(AC[t][0x00])
    bits = "".join(format(c, f"0{n}b") for c, n in out if n)
    bits += "1" * (-len(bits) % 8)
    data = int(bits, 2).to_bytes(len(bits) // 8, "big") if bits else b""
    return data.replace(b"\xff", b"\xff\x00")


def encode(img: np.ndarray, quality: int, subsampling: int) -> bytes:
    """The whole JFIF file of an RGB uint8 [H, W, 3] image."""
    h, w = img.shape[:2]
    return J.jpeg_header(h, w, quality, subsampling) + scan(img, quality, subsampling) + b"\xff\xd9"
