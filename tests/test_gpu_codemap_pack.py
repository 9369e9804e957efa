"""GPU: packed code maps -- the histogram kernel against torch.bincount, the rANS packer against the numpy
oracle of tests/codemap_pack_oracle.py byte for byte (table, offsets, payload, container), region unpack
against slicing the original map, an fp16 slide through compress_slide -> pack -> save / load -> unpack ->
decompress_region, and the per-patch integrity flags on a damaged payload."""
import numpy as np
import pytest
import torch

import codemap_pack_oracle as O
import helpers as H
import vqae_b200
from vqae_b200 import engine as E
from vqae_b200 import synthetic as S
from vqae_b200.extract import compress_slide, decompress_region
from vqae_b200.packing import (PackedCodeMap, PackedIntegrityError, load_packed, pack_code_map, save_packed,
                               unpack_code_map)

from test_codemap_pack_host import KINDS, make_map

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TILES = [(32, 32), (16, 16), (8, 12)]


def _dev_map(m: np.ndarray, dtype) -> torch.Tensor:
    return torch.from_numpy(m.astype(np.int64)).to(DEV).to(dtype)


@pytest.mark.parametrize("dtype", [torch.uint8, torch.int64])
def test_histogram_equals_bincount(dtype):
    k = 256 if dtype == torch.uint8 else 1024
    g = torch.Generator(device=DEV).manual_seed(2)
    m = torch.randint(0, k, (1000, 777), device=DEV, generator=g).to(dtype)
    m[:300] = torch.minimum(m[:300], torch.tensor(3, device=DEV, dtype=dtype))    # a skewed band
    for kk in (k, 200):                                    # 200: codes >= 200 land in the overflow bin
        counts, invalid = E.codemap_histogram(m, kk)
        want = torch.bincount(m.long().ravel(), minlength=k)
        assert torch.equal(counts, want[:kk]) and int(invalid) == int(want[kk:].sum())
    for win in ((0, 0, 1, 777), (5, 9, 1, 1), (290, 13, 20, 700), (999, 776, 1, 1)):
        r0, c0, nr, nc = win
        counts, invalid = E.codemap_histogram(m, k, win)
        assert torch.equal(counts, torch.bincount(m[r0:r0 + nr, c0:c0 + nc].long().ravel(), minlength=k))
        assert int(invalid) == 0
    if dtype == torch.int64:
        m[7, 7] = -5
        assert int(E.codemap_histogram(m, k)[1]) == 1


def _check_against_oracle(m: np.ndarray, dtype, th, tw, k=None):
    freq, offsets, payload = O.pack(m, th, tw, k=k)
    p = pack_code_map(_dev_map(m, dtype), (th, tw), k=k)
    assert np.array_equal(p.freq_host, freq)
    assert np.array_equal(p.offsets.cpu().numpy(), offsets)
    assert p.payload.cpu().numpy().tobytes() == payload
    code = 0 if dtype == torch.uint8 else 1
    assert p.to_bytes() == O.container(m.shape[0], m.shape[1], th, tw, freq, offsets, payload, code)
    return p


@pytest.mark.parametrize("hw", TILES, ids=lambda t: f"{t[0]}x{t[1]}")
@pytest.mark.parametrize("kind", KINDS)
def test_pack_equals_oracle_bytes(kind, hw):
    th, tw = hw
    for grid in ((5, 7), (1, 1), (9, 11)):                 # 35, 1, 99 patches: ragged last CTA
        m = make_map(kind, th, tw, grid, seed=grid[0])
        k = 1024 if kind == "k1024" else None
        dtypes = [torch.int64] if kind == "k1024" else [torch.uint8, torch.int64]
        for dtype in dtypes:
            p = _check_against_oracle(m, dtype, th, tw, k)
            assert p.counts is not None and int(p.counts.sum()) == m.size
            whole = unpack_code_map(p, dtype=dtype)
            assert torch.equal(whole.cpu(), torch.from_numpy(m.astype(np.int64)).to(dtype))


def test_repeated_launches_are_identical():
    m = make_map("geometric", 32, 32, (13, 17), seed=4)
    p = pack_code_map(_dev_map(m, torch.uint8), (32, 32))
    for _ in range(3):
        q = pack_code_map(_dev_map(m, torch.uint8), (32, 32))
        assert q.to_bytes() == p.to_bytes()
        assert torch.equal(unpack_code_map(q), unpack_code_map(p))


@pytest.mark.parametrize("out_dtype", [torch.uint8, torch.int64])
def test_unpack_regions_equal_slices(out_dtype):
    th, tw = 16, 12
    rows, cols = 11, 37
    m = make_map("geometric", th, tw, (rows, cols), seed=9)
    ref = torch.from_numpy(m.astype(np.int64)).to(out_dtype)
    p = pack_code_map(_dev_map(m, torch.uint8), (th, tw))
    for reg in ((0, 0, rows, cols), (0, 0, 1, 1), (rows - 1, cols - 1, 1, 1), (0, cols - 1, rows, 1),
                (rows - 1, 0, 1, cols), (3, 4, 4, 33), (2, 1, 9, 3)):
        r0, c0, nr, nc = reg
        got = unpack_code_map(p, reg, dtype=out_dtype)
        assert got.dtype == out_dtype and tuple(got.shape) == (nr * th, nc * tw)
        assert torch.equal(got.cpu(), ref[r0 * th:(r0 + nr) * th, c0 * tw:(c0 + nc) * tw]), reg


def test_int64_map_with_1024_codes():
    m = make_map("k1024", 32, 32, (6, 7), seed=3)
    p = pack_code_map(_dev_map(m, torch.int64), (32, 32), k=1024)
    assert p.k == 1024 and p.source_dtype == torch.int64
    with pytest.raises(ValueError):
        unpack_code_map(p)                                  # uint8 cannot hold 1024 codes
    assert torch.equal(unpack_code_map(p, (1, 2, 3, 4), dtype=torch.int64).cpu(),
                       torch.from_numpy(m[32:128, 64:192]))
    with pytest.raises(ValueError):
        pack_code_map(_dev_map(m, torch.int64), (32, 32), k=1000)        # codes >= k


def test_slide_round_trip_through_packing(tmp_path):
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = vqae_b200.set_precision(m.to(DEV), "fp16")
    try:
        grid = (3, 5)
        img = S.synthetic_patches_u8(15, 256, 8)
        cmap = compress_slide(m.encoder, [(0, img[:8]), (8, img[8:])], grid, (32, 32), torch.device(DEV))
        packed = pack_code_map(cmap, (32, 32))
        path = save_packed(tmp_path / "slide.vqpk", packed)
        loaded = load_packed(path, DEV)
        assert loaded.to_bytes() == packed.to_bytes()
        for reg in (None, (1, 2, 2, 3), (2, 4, 1, 1)):
            window = unpack_code_map(loaded, reg)
            r0, c0, nr, nc = reg if reg is not None else (0, 0) + grid
            assert torch.equal(window, cmap[r0 * 32:(r0 + nr) * 32, c0 * 32:(c0 + nc) * 32])
            got = decompress_region(m, window, (32, 32))
            want = decompress_region(m, cmap, (32, 32), region=reg)
            assert torch.equal(got, want)
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()


def test_damaged_payload_is_flagged_and_other_patches_decode():
    th = tw = 32
    rows, cols = 4, 6
    m = make_map("geometric", th, tw, (rows, cols), seed=12)
    p = pack_code_map(_dev_map(m, torch.uint8), (th, tw))
    victim = 9                                               # patch (1, 3)
    a, b = int(p.offsets_host[victim]), int(p.offsets_host[victim + 1])
    pos = a + 4 + 2 * ((b - a - 4) // 4)                     # a word in the middle of its stream
    payload = p.payload.clone()
    payload[pos] ^= 0x5a
    # the oracle's decoder flags the same stream
    _, oflags = O.decode(payload.cpu().numpy().tobytes(), p.offsets_host, p.freq_host, th * tw, [victim])
    assert oflags[0] != 0
    bad = PackedCodeMap(freq=p.freq, offsets=p.offsets, payload=payload, grid=p.grid, code_hw=p.code_hw, k=p.k,
                        freq_host=p.freq_host, offsets_host=p.offsets_host)
    with pytest.raises(PackedIntegrityError) as ei:
        unpack_code_map(bad)
    err = ei.value
    assert isinstance(err, ValueError) and err.patches == [(1, 3)] and "(1, 3)" in str(err)
    got = err.code_map.cpu().numpy().reshape(rows, th, cols, tw)
    want = m.reshape(rows, th, cols, tw)
    for r in range(rows):
        for c in range(cols):
            if (r, c) != (1, 3):
                assert np.array_equal(got[r, :, c], want[r, :, c])
    assert int(err.flags[1, 3]) != 0 and int(err.flags.count_nonzero()) == 1
    assert torch.equal(unpack_code_map(bad, (0, 0, 1, cols)).cpu(), torch.from_numpy(m[:32]))   # other rows
    damaged = p.to_bytes()[:-len(payload)] + payload.cpu().numpy().tobytes()
    with pytest.raises(ValueError, match="CRC"):             # in a container, the CRC catches it first
        PackedCodeMap.from_bytes(damaged, DEV)
