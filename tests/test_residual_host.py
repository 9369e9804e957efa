"""CPU: the numpy residual oracle of tests/residual_oracle.py (error bound, round trips, the parallel Adler
form), the VQRL container checks of vqae_b200.residual, and the argument checks of vqae_residual_*, which
return before any CUDA call."""
import ctypes as C
import zlib

import numpy as np
import pytest
import torch

import residual_oracle as RO
from vqae_b200 import _lib as L
from vqae_b200.residual import ResidualLayer, check_max_error


@pytest.mark.parametrize("e", [0, 1, 2, 3, 7, 31, 127])
def test_exhaustive_error_bound(e):
    x, xh = np.meshgrid(np.arange(256), np.arange(256), indexing="ij")
    s = RO.symbols(x, xh, e)
    out = RO.reconstruct(xh, s, e).astype(np.int64)
    if e == 0:
        assert np.array_equal(out, x)
    else:
        assert int(np.abs(out - x).max()) <= e
        k = s.view(np.int8).astype(np.int64)
        assert int(np.abs(k).max()) <= 85


def _roundtrip(x, xh, h, w, e):
    offsets, payload, adler, canvas = RO.layer(x, xh, h, w, e)
    n = 3 * h * w
    sym = RO.symbols(RO.patches(x, h, w), RO.patches(xh, h, w), e)
    for p in range(len(offsets) - 1):
        chunk = payload[offsets[p]:offsets[p + 1]]
        assert len(chunk) % 2 == 0 and 768 <= len(chunk) <= 768 + 2 * n
        got, ok = RO.decode(chunk, n)
        assert ok and np.array_equal(got, sym[p]), p
    assert np.array_equal(adler[:, 0], [zlib.adler32(b.tobytes()) for b in RO.patches(xh, h, w)])
    assert np.array_equal(adler[:, 1], [zlib.adler32(b.tobytes()) for b in RO.patches(canvas, h, w)])
    if e == 0:
        assert np.array_equal(canvas, x)
    else:
        assert int(np.abs(canvas.astype(int) - x.astype(int)).max()) <= e
    return offsets, payload


@pytest.mark.parametrize("e", [0, 1, 4])
@pytest.mark.parametrize("hw", [(16, 16), (8, 12), (5, 7)])
def test_oracle_round_trips(e, hw):
    h, w = hw
    rng = np.random.default_rng(h * 100 + w + e)
    x = rng.integers(0, 256, (2 * h, 3 * w, 3)).astype(np.uint8)
    xh = np.clip(x.astype(int) + rng.laplace(0, 3, x.shape).round().astype(int), 0, 255).astype(np.uint8)
    _roundtrip(x, xh, h, w, e)
    _roundtrip(x, rng.integers(0, 256, x.shape).astype(np.uint8), h, w, e)     # uniform residual


def test_constant_and_extreme_patches():
    h = w = 16
    x = np.full((h, w, 3), 255, np.uint8)
    xh = np.zeros_like(x)
    for e in (0, 1, 4, 127):
        offsets, payload = _roundtrip(x, xh, h, w, e)                          # one-symbol table
        freq = np.frombuffer(payload, "<u2", 256)
        assert (freq == 0).sum() == 255 and freq.max() == 1 << 14
        assert len(payload) == 768 + 2 * 0                                      # f = 2^14: no words at all
    _roundtrip(x, x.copy(), h, w, 0)                                            # all-zero residual


def test_parallel_adler_equals_zlib():
    rng = np.random.default_rng(3)
    for n in (0, 1, 31, 5552, 5553, 3 * 256 * 256, 3 * 1024 * 1024):
        b = rng.integers(0, 256, n).astype(np.uint8)
        assert RO.adler32(b) == zlib.adler32(b.tobytes()), n
    b = np.full(3 * 1024 * 1024, 255, np.uint8)
    assert RO.adler32(b) == zlib.adler32(b.tobytes())


def _container(**kw):
    h = w = 8
    rng = np.random.default_rng(1)
    x = rng.integers(0, 256, (2 * h, 2 * w, 3)).astype(np.uint8)
    xh = rng.integers(0, 256, x.shape).astype(np.uint8)
    offsets, payload, adler, _ = RO.layer(x, xh, h, w, 2)
    args = dict(rows=2, cols=2, h=h, w=w, e=2, mode=1, offsets=offsets, adler=adler, payload=payload)
    args.update(kw)
    return RO.container(**args), args


def test_container_round_trip_and_rejections():
    buf, args = _container()
    layer = ResidualLayer.from_bytes(buf, "cpu")
    assert layer.max_error == 2 and layer.precision == "fp16" and layer.grid == (2, 2) and layer.patch_hw == (8, 8)
    assert layer.to_bytes() == buf
    assert np.array_equal(layer.adler.numpy().view(np.uint32), args["adler"])
    assert layer.nbytes() == len(buf)
    assert layer.bits_per_pixel() == pytest.approx(8 * len(buf) / (4 * 64))
    off, payload = args["offsets"], args["payload"]
    bad = {
        "short": buf[:20], "truncated": buf[:-1], "long": buf + b"\0",
        "magic": b"VQRX" + buf[4:],
        "version": _container(version=2)[0], "mode": _container(mode=3)[0], "e": _container(e=128)[0],
        "first offset": _container(offsets=off + 2)[0],
        "odd step": _container(offsets=np.array([0, off[1] + 1, off[2] + 1, off[3] + 1, off[4] + 1]),
                               payload=payload[:off[1]] + b"\0" + payload[off[1]:])[0],
        "short step": _container(offsets=np.array([0, 766, off[4] - (off[4] - 766) // 3 * 2 - 2, off[4] - 2,
                                                   off[4]]))[0],
        "long step": _container(offsets=np.array([0, 768 + 2 * 192 + 2, off[2], off[3], off[4]]))[0],
        "crc": buf[:-1] + bytes([buf[-1] ^ 1]),
    }
    for name, b in bad.items():
        with pytest.raises(ValueError):
            ResidualLayer.from_bytes(b, "cpu")
        assert name


def test_max_error_validation():
    assert check_max_error(0) == 0 and check_max_error(np.int64(127)) == 127
    for bad in (-1, 128, 1.0, "1", True, None):
        with pytest.raises(ValueError):
            check_max_error(bad)


def test_abi_rejects_bad_arguments_without_cuda():
    lib = L.load()                          # no GPU needed: every case returns before a CUDA call
    fake = C.c_void_p(4096)                 # never dereferenced
    h = w = 16
    n = 3 * h * w
    assert lib.vqae_residual_encode_scratch_bytes(4, h, w) > 0
    for args in ((0, h, w), (4, 0, w), (4, 2048, 1024)):
        assert lib.vqae_residual_encode_scratch_bytes(*args) == 0

    def canvas(p=fake, rows=2 * h, cols=2 * w, r0=0, c0=0, rc=2, first=0):
        return [p, rows, cols, r0, c0, rc, first]

    def stats(x={}, b={}, batch=4, hh=h, ww=w, e=0, hist=fake, adler=fake):
        return lib.vqae_residual_stats(*canvas(**x), *canvas(**b), batch, hh, ww, e, hist, adler, None)

    def encode(x={}, b={}, batch=4, hh=h, ww=w, e=0, freq=fake, cap=4 * (768 + 2 * n), scratch=fake,
               nbytes=None):
        nb = lib.vqae_residual_encode_scratch_bytes(batch, hh, ww) if nbytes is None else nbytes
        return lib.vqae_residual_encode(*canvas(**x), *canvas(**b), batch, hh, ww, e, freq, fake, fake, cap,
                                        scratch, nb, None)

    for call in (stats, encode):
        for kw in ({"x": {"p": None}}, {"b": {"p": None}}, {"batch": 0}, {"hh": 0}, {"ww": -1}, {"e": -1},
                   {"x": {"rows": 2 * h - 1}}, {"b": {"cols": 2 * w - 1}}, {"x": {"first": 1}},
                   {"b": {"r0": 1}}, {"x": {"c0": 1}}, {"b": {"rc": 3}}, {"x": {"rc": 0}},
                   {"b": {"first": -1}}):
            assert call(**kw) == L.ERR_BAD_ARG, (call.__name__, kw)
        assert call(e=128) == L.ERR_UNSUPPORTED
        big = 1 << 31
        assert call(x={"first": big - 1, "rc": big, "cols": big * w}, batch=2) == L.ERR_UNSUPPORTED
    assert stats(hist=None) == L.ERR_BAD_ARG and stats(adler=None) == L.ERR_BAD_ARG
    assert encode(freq=None) == L.ERR_BAD_ARG
    assert encode(cap=4 * (768 + 2 * n) - 1) == L.ERR_BAD_ARG
    assert encode(scratch=None) == L.ERR_SCRATCH
    assert encode(nbytes=lib.vqae_residual_encode_scratch_bytes(4, h, w) - 1) == L.ERR_SCRATCH
    assert lib.vqae_residual_tables(None, 4, fake, None) == L.ERR_BAD_ARG
    assert lib.vqae_residual_tables(fake, 0, fake, None) == L.ERR_BAD_ARG
    assert lib.vqae_residual_tables(fake, 4, None, None) == L.ERR_BAD_ARG

    # apply: a 2 x 2 layer of 16 x 16 patches with 800-byte chunks
    off = np.array([0, 800, 1600, 2400, 3200], np.int64)

    def apply(off=off, pbytes=3200, grid=(2, 2), layer=(0, 0, 2, 0), cv={}, batch=4, e=0, flags=fake):
        oh = np.ascontiguousarray(off)
        return lib.vqae_residual_apply(fake, pbytes, oh.ctypes.data_as(C.c_void_p), fake, fake, grid[0], grid[1],
                                       *layer, *canvas(**cv)[:], batch, h, w, e, flags, None)
    for kw in ({"flags": None}, {"pbytes": 3202}, {"off": off + 2}, {"off": np.array([0, 801, 1600, 2400, 3200])},
               {"off": np.array([0, 700, 1600, 2400, 3200])}, {"off": np.array([0, 800 + 2 * n + 2, 1600, 2400,
                                                                                3200])},
               {"layer": (1, 0, 2, 0)}, {"layer": (0, 1, 2, 0)}, {"layer": (0, 0, 3, 0)}, {"layer": (0, 0, 2, 1)},
               {"layer": (0, 0, 0, 0)}, {"grid": (0, 2)}, {"cv": {"first": 1}}, {"cv": {"p": None}}, {"batch": 0}):
        assert apply(**kw) == L.ERR_BAD_ARG, kw
    assert apply(e=128) == L.ERR_UNSUPPORTED


def test_layer_is_importable_without_a_device():
    layer = ResidualLayer(payload=torch.zeros(768, dtype=torch.uint8), offsets=torch.tensor([0, 768]),
                          adler=torch.zeros(1, 2, dtype=torch.int32), max_error=0, precision="fp32", grid=(1, 1),
                          patch_hw=(8, 8))
    again = ResidualLayer.from_bytes(layer.to_bytes(), "cpu")
    assert again.payload_bytes == 768 and again.precision == "fp32"
