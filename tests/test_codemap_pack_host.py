"""CPU: the packed code map format -- the numpy oracle of tests/codemap_pack_oracle.py round-trips every
map family, its payload stays within the ideal length under its table plus the 4-byte states, the table
quantisation of vqae_b200.packing agrees with the oracle's, the container round-trips and rejects damaged
buffers, and the argument checks of the vqae_codemap_* entry points return before any CUDA call."""
import ctypes as C
import struct
import zlib

import numpy as np
import pytest
import torch

import codemap_pack_oracle as O
from vqae_b200 import _lib as L
from vqae_b200 import packing as PK

TILES = [(32, 32), (16, 16), (8, 12)]


def make_map(kind: str, th: int, tw: int, grid=(5, 7), seed: int = 0) -> np.ndarray:
    rng = np.random.default_rng(seed)
    shape = (grid[0] * th, grid[1] * tw)
    if kind == "single":
        return np.full(shape, 7, dtype=np.uint8)
    if kind == "two":
        return (rng.random(shape) < 0.2).astype(np.uint8) * 200
    if kind == "geometric":
        return np.minimum(rng.geometric(0.3, shape) - 1, 255).astype(np.uint8)
    if kind == "uniform256":
        return rng.integers(0, 256, shape).astype(np.uint8)
    if kind == "k1024":
        return rng.integers(0, 1024, shape).astype(np.int64)
    raise KeyError(kind)


KINDS = ["single", "two", "geometric", "uniform256", "k1024"]


@pytest.mark.parametrize("hw", TILES, ids=lambda t: f"{t[0]}x{t[1]}")
@pytest.mark.parametrize("kind", KINDS)
def test_oracle_round_trip_and_size(kind, hw):
    th, tw = hw
    m = make_map(kind, th, tw)
    k = 1024 if kind == "k1024" else None
    freq, offsets, payload = O.pack(m, th, tw, k=k)
    P = offsets.size - 1
    assert P == m.size // (th * tw) and offsets[-1] == len(payload)
    d = np.diff(offsets)
    assert (d >= 4).all() and (d <= 4 + 2 * th * tw).all() and (d % 2 == 0).all()
    sym, flags = O.decode(payload, offsets, freq, th * tw, np.arange(P))
    assert (flags == 0).all()
    assert np.array_equal(sym, O.tiles(m, th, tw))
    # no larger than the ideal code under the stored table plus the per-patch states
    assert len(payload) <= O.ideal_bytes(m, freq) + 4 * P
    if kind == "single":
        assert len(payload) == 4 * P and all(payload[4 * p:4 * p + 4] == struct.pack("<I", O.L) for p in range(P))
    if kind == "uniform256":
        assert len(payload) > m.size          # slightly larger than raw uint8: reported, not special-cased


@pytest.mark.parametrize("kind", KINDS)
def test_quantised_table(kind):
    m = make_map(kind, 16, 16)
    k = 1024 if kind == "k1024" else int(m.max()) + 1
    counts = np.bincount(m.astype(np.int64).ravel(), minlength=k)
    f = PK.quantise_frequencies(counts)
    assert f.dtype == np.uint32 and f.shape == (k,)
    assert int(f.astype(np.int64).sum()) == 1 << 14
    assert ((f > 0) == (counts > 0)).all()
    assert np.array_equal(f, O.quantise(counts))


def test_quantised_table_edge_cases():
    rng = np.random.default_rng(1)
    for counts in ([5], [0, 0, 3], [1] * 1024, [10 ** 9] + [1] * 1023, [1, 1 << 40],
                   list(rng.integers(0, 50, 1024)), list(rng.geometric(0.01, 300))):
        counts = np.array(counts, dtype=np.int64)
        f = PK.quantise_frequencies(counts)
        assert int(f.astype(np.int64).sum()) == 1 << 14 and ((f > 0) == (counts > 0)).all()
        assert np.array_equal(f, O.quantise(counts))
    with pytest.raises(ValueError):
        PK.quantise_frequencies(np.zeros(4, np.int64))
    with pytest.raises(ValueError):
        PK.quantise_frequencies(np.ones(5, np.int64), scale_bits=2)


def cpu_packed(kind="geometric", th=16, tw=16, grid=(3, 5)) -> PK.PackedCodeMap:
    m = make_map(kind, th, tw, grid)
    freq, offsets, payload = O.pack(m, th, tw)
    return PK.PackedCodeMap(freq=torch.from_numpy(freq.astype(np.int32)), offsets=torch.from_numpy(offsets),
                            payload=torch.frombuffer(bytearray(payload), dtype=torch.uint8), grid=grid,
                            code_hw=(th, tw), k=len(freq), source_dtype=torch.uint8)


def test_container_matches_oracle_and_round_trips():
    p = cpu_packed()
    buf = p.to_bytes()
    assert buf == O.container(p.map_shape[0], p.map_shape[1], 16, 16, p.freq_host, p.offsets_host,
                              p.payload.numpy().tobytes())
    assert len(buf) == p.nbytes()
    q = PK.PackedCodeMap.from_bytes(buf, "cpu")
    assert (q.grid, q.code_hw, q.k, q.scale_bits, q.source_dtype) == (p.grid, p.code_hw, p.k, 14, torch.uint8)
    assert torch.equal(q.freq, p.freq) and torch.equal(q.offsets, p.offsets) and torch.equal(q.payload, p.payload)
    assert q.to_bytes() == buf
    assert p.bits_per_code() == pytest.approx(8 * len(buf) / (15 * 256))
    assert p.bits_per_pixel((128, 128)) == pytest.approx(8 * len(buf) / (15 * 128 * 128))


def _rewrite(buf: bytes, pos: int, fmt: str, value) -> bytes:
    b = bytearray(buf)
    struct.pack_into(fmt, b, pos, value)
    return bytes(b)


def test_container_rejects_damage():
    p = cpu_packed()
    buf = p.to_bytes()
    hs, k, P = PK.HEADER.size, p.k, p.n_patches
    off_pos = hs + 4 * k
    crc_pos = off_pos + 8 * (P + 1)
    bad = {
        "short header": buf[:20],
        "truncated tables": buf[:crc_pos],
        "truncated payload": buf[:-1],
        "extra byte": buf + b"\0",
        "magic": b"XQPK" + buf[4:],
        "version": _rewrite(buf, 4, "<H", 2),
        "dtype": _rewrite(buf, 6, "<H", 9),
        "grid": _rewrite(buf, 8, "<Q", p.map_shape[0] + 1),
        "k": _rewrite(buf, 32, "<I", 1025),
        "crc": _rewrite(buf, crc_pos, "<I", zlib.crc32(b"x")),
        "payload bit": buf[:-1] + bytes([buf[-1] ^ 1]),
        "table sum": _rewrite(buf, hs, "<I", int(p.freq_host[0]) + 1),
        "non-monotone offsets": _rewrite(buf, off_pos + 8 * 2, "<Q", int(p.offsets_host[1]) - 2),
        "odd stream": _rewrite(buf, off_pos + 8, "<Q", int(p.offsets_host[1]) + 1),
        "first offset": _rewrite(buf, off_pos, "<Q", 2),
    }
    for name, b in bad.items():
        with pytest.raises(ValueError):
            PK.PackedCodeMap.from_bytes(b, "cpu")
        assert name


def test_abi_rejects_bad_arguments_without_cuda():
    lib = L.load()                          # no GPU needed: every case returns before a CUDA call
    fake = C.c_void_p(4096)                 # never dereferenced
    th = tw = 4
    rows, cols = 8, 12                      # 2 x 3 patches
    P, n = 6, 16
    worst = lib.vqae_codemap_pack_worst_bytes(P, th, tw)
    need = lib.vqae_codemap_pack_scratch_bytes(P, th, tw)
    assert worst == P * (4 + 2 * n) and need > 0 and lib.vqae_codemap_pack_scratch_bytes(1, 200, 200) == 0
    f_ok = np.array([1 << 13, 1 << 13], dtype=np.uint32)
    f_sum = np.array([1 << 13, 5], dtype=np.uint32)
    f_big = np.zeros(1025, dtype=np.uint32)
    f_big[0] = 1 << 14
    hp = lambda a: a.ctypes.data_as(C.c_void_p)          # noqa: E731

    def hist(m=fake, r0=0, c0=0, nr=rows, nc=cols, k=2, counts=fake):
        return lib.vqae_codemap_histogram(m, 1, rows, cols, r0, c0, nr, nc, k, counts, None)
    for kw in ({"m": None}, {"counts": None}, {"nr": 0}, {"nc": -1}, {"r0": -1}, {"r0": 1}, {"c0": 1},
               {"nc": cols + 1}):
        assert hist(**kw) == L.ERR_BAD_ARG, kw
    assert hist(k=0) == L.ERR_UNSUPPORTED and hist(k=1025) == L.ERR_UNSUPPORTED

    def pack(m=fake, r=rows, c=cols, h=th, w=tw, f=f_ok, k=None, s=14, off=fake, pay=fake, cap=worst,
             scratch=fake, nbytes=need):
        return lib.vqae_codemap_pack(m, 1, r, c, h, w, hp(f) if f is not None else None,
                                     (2 if f is None else len(f)) if k is None else k, s, off, pay, cap, scratch,
                                     nbytes, None)
    for kw in ({"m": None}, {"off": None}, {"pay": None}, {"f": None}, {"r": 0}, {"c": 11}, {"h": 3},
               {"w": 0}, {"f": f_sum}, {"cap": worst - 1}, {"s": 13}):
        assert pack(**kw) == L.ERR_BAD_ARG, kw
    for kw in ({"k": 0}, {"f": f_big}, {"s": 15}, {"s": 0}, {"h": 8, "w": 2049, "r": 8, "c": 2049}):
        assert pack(**kw) == L.ERR_UNSUPPORTED, kw
    assert pack(nbytes=need - 1) == L.ERR_SCRATCH and pack(scratch=None) == L.ERR_SCRATCH

    good = np.arange(P + 1, dtype=np.int64) * 6           # 6-byte streams
    def unpack(pay=fake, nbytes=int(good[-1]), oh=good, od=fake, f=f_ok, k=None, s=14, region=(0, 0, 2, 3),
               out=fake, u8=1, flags=fake):
        return lib.vqae_codemap_unpack(pay, nbytes, hp(oh) if oh is not None else None, od, rows, cols, th, tw,
                                       hp(f), len(f) if k is None else k, s, *region, out, u8, flags, None)
    bad_off = [good.copy() for _ in range(5)]
    bad_off[0][0] = 2                                       # first offset
    bad_off[1][3] = bad_off[1][2] - 2                       # not monotone
    bad_off[2][1:] += 1                                     # an odd stream
    bad_off[3][1:] -= 4                                     # a 2-byte stream
    bad_off[4][1:] += 2 + 2 * n                             # longer than the worst case
    for kw in ({"pay": None}, {"oh": None}, {"od": None}, {"out": None}, {"flags": None}, {"f": f_sum},
               {"region": (0, 0, 3, 3)}, {"region": (0, 1, 2, 3)}, {"region": (-1, 0, 1, 1)},
               {"region": (0, 0, 0, 1)}, {"nbytes": int(good[-1]) + 2}):
        assert unpack(**kw) == L.ERR_BAD_ARG, kw
    for o in bad_off:
        assert unpack(oh=o, nbytes=int(o[-1])) == L.ERR_BAD_ARG
    f1024 = np.full(1024, 16, dtype=np.uint32)
    assert unpack(f=f1024, u8=1) == L.ERR_UNSUPPORTED
    assert unpack(k=1025) == L.ERR_UNSUPPORTED and unpack(s=15) == L.ERR_UNSUPPORTED


def test_pack_code_map_rejects_cpu_tensors():
    with pytest.raises(RuntimeError):
        PK.pack_code_map(torch.zeros(32, 32, dtype=torch.uint8), (32, 32))
