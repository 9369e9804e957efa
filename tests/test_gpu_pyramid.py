"""GPU: box-filtered pyramid levels of uint8 RGB canvases (csrc/pyramid.cu, engine.pyramid_u8,
vqae_b200.pyramid.slide_pyramid, extract.decompress_pyramid) against the numpy oracle of
tests/pyramid_oracle.py and PIL.Image.reduce, all with torch.equal."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

import helpers as H
import pyramid_oracle as PO
import ref_shim
import vqae_b200
from vqae_b200 import _lib as L
from vqae_b200 import engine as E
from vqae_b200.extract import decompress_pyramid, decompress_region
from vqae_b200.pyramid import FACTORS, slide_pyramid

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _rand_u8(shape, seed):
    return torch.randint(0, 256, shape, generator=torch.Generator().manual_seed(seed), dtype=torch.uint8)


def _valid(h, w):
    return tuple(f for f in FACTORS if h % f == 0 and w % f == 0)


def _batch_levels(x, factors):
    """x: uint8 [n, h, w, 3] on the device -> {f: [n, h/f, w/f, 3]} through one pyramid launch."""
    n, h, w, _ = x.shape
    dst = {f: torch.empty(n * (h // f), w // f, 3, dtype=torch.uint8, device=x.device) for f in factors}
    E.pyramid_u8(x.reshape(n * h, w, 3), (0, 0, 1, 0), n, h, w, dst, (0, 0, 1, 0))
    return {f: v.view(n, h // f, w // f, 3) for f, v in dst.items()}


def _oracle_batch(x_np, f):
    return np.stack([PO.reduce(p, f) for p in x_np])


def _factor_sets(h, w):
    fs = _valid(h, w)
    return [(f,) for f in fs] + [fs, (fs[0], fs[-1])] + ([(4, 128)] if 128 in fs else [])


@pytest.mark.parametrize("hw", [(256, 256), (512, 512), (192, 320), (16, 16)])
def test_batches_against_oracle(hw):
    h, w = hw
    x = _rand_u8((3, h, w, 3), h * 1000 + w)
    xd = x.to(DEV)
    xn = x.numpy()
    want = {f: _oracle_batch(xn, f) for f in _valid(h, w)}
    for fs in _factor_sets(h, w):
        got = _batch_levels(xd, fs)
        assert sorted(got) == sorted(fs)
        for f in fs:
            assert torch.equal(got[f].cpu(), torch.from_numpy(want[f])), (hw, fs, f)
    # the same batch from a canvas whose base is not 16-byte aligned (byte loads)
    buf = torch.empty(3 * h * w * 3 + 5, dtype=torch.uint8, device=DEV)
    odd = buf[5:].view(3 * h, w, 3)
    odd.copy_(xd.view(3 * h, w, 3))
    dst = {f: torch.empty(3 * (h // f), w // f, 3, dtype=torch.uint8, device=DEV) for f in _valid(h, w)}
    E.pyramid_u8(odd, (0, 0, 1, 0), 3, h, w, dst, (0, 0, 1, 0))
    for f, v in dst.items():
        assert torch.equal(v.view(3, h // f, w // f, 3).cpu(), torch.from_numpy(want[f])), ("unaligned", f)


@pytest.mark.parametrize("extra", [0, 5])
def test_canvas_addressing_and_no_stray_writes(extra):
    """Source: region patches 1 .. 5 of a region at grid (1, 1) with 3 patches per row inside a 4 x 5 grid
    (rows carry `extra` more pixels: not 16-byte multiples when extra = 5).  Destination: patches 1 .. 5 of
    a region at grid (0, 1) with 2 patches per row in level canvases of 3 x 4 patches (+ `extra`).  Every
    byte outside the written patches keeps its sentinel."""
    h, w = 256, 128
    fs = _valid(h, w)
    src = _rand_u8((4 * h, 5 * w + extra, 3), 3 + extra)
    srcd = src.to(DEV)
    sentinel = 77
    dst = {f: torch.full((3 * (h // f), 4 * (w // f) + extra, 3), sentinel, dtype=torch.uint8, device=DEV)
           for f in fs}
    E.pyramid_u8(srcd, (1, 1, 3, 1), 5, h, w, dst, (0, 1, 2, 1))
    patches = PO.gather_patches(src.numpy(), h, w, 1, 1, 3, 1, 5)
    for f in fs:
        want = np.full(tuple(dst[f].shape), sentinel, np.uint8)
        hf, wf = h // f, w // f
        for t in range(5):
            q = 1 + t
            r, c = q // 2, 1 + q % 2
            want[r * hf:(r + 1) * hf, c * wf:(c + 1) * wf] = PO.reduce(patches[t], f)
        assert np.array_equal(dst[f].cpu().numpy(), want), (extra, f)


def test_abi_rejects_bad_placements_before_launching():
    lib = L.load()
    src = torch.zeros(512, 256, 3, dtype=torch.uint8, device=DEV)
    lv = torch.zeros(256, 128, 3, dtype=torch.uint8, device=DEV)          # level 2 of two 256^2 patches
    ptrs, rows, cols = (C.c_void_p * 10)(), (C.c_int64 * 10)(), (C.c_int64 * 10)()
    ptrs[1], rows[1], cols[1] = lv.data_ptr(), 256, 128
    ptrs[8], rows[8], cols[8] = lv.data_ptr(), 2, 1                        # level 8: 1 x 1 per patch
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = E._ptr

    def call(first=0, rc=1, r0=0, dfirst=0, drc=1, dc0=0, mask=2):
        return lib.vqae_pyramid_u8(p(src), 512, 256, r0, 0, rc, first, 2, 256, 256, mask, ptrs, rows, cols, 0,
                                   dc0, drc, dfirst, None, 0, st)
    n0 = E.raw_launch_count()
    assert call(first=1) == L.ERR_BAD_ARG
    assert call(r0=1) == L.ERR_BAD_ARG
    assert call(rc=2) == L.ERR_BAD_ARG
    assert call(dfirst=1) == L.ERR_BAD_ARG
    assert call(dc0=1) == L.ERR_BAD_ARG
    assert call(mask=2 | 4) == L.ERR_BAD_ARG                               # level 2 has no canvas
    assert call(mask=1 << 8) == L.ERR_SCRATCH
    torch.cuda.synchronize()
    assert E.raw_launch_count() == n0
    assert call() == L.OK and E.raw_launch_count() == n0 + 1


# launcher mirror (pyramid.cu pyramid_u8): units of T x T pixels, T = 64 for 256^2 patches;
# grid = min(units, sm_count x PY_MIN_CTAS = 6)
def test_saturated_and_ragged_launches_equal_single_patches():
    h = w = 256
    rows, cols = 10, 20
    n = rows * cols
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    units, cap = n * (h // 64) * (w // 64), 6 * sm
    assert units >= 3 * cap and units % cap != 0                       # >= 3 units per CTA, a partial wave
    slide = _rand_u8((rows * h, cols * w, 3), 12).to(DEV)
    whole = slide_pyramid(slide, (h, w), FACTORS[:8], batch=n)
    ragged = slide_pyramid(slide, (h, w), FACTORS[:8], batch=64)            # 64, 64, 64, 8
    single = slide_pyramid(slide, (h, w), FACTORS[:8], batch=1)
    for f in FACTORS[:8]:
        assert torch.equal(whole[f], ragged[f]) and torch.equal(whole[f], single[f]), f
        assert torch.equal(whole[f].cpu(), torch.from_numpy(PO.reduce(slide.cpu().numpy(), f))), f
    again = slide_pyramid(slide, (h, w), FACTORS[:8], batch=n)
    assert all(torch.equal(again[f], whole[f]) for f in FACTORS[:8])


def test_largest_sums():
    x = torch.full((2, 512, 512, 3), 255, dtype=torch.uint8, device=DEV)
    got = _batch_levels(x, FACTORS)
    for f in FACTORS:
        assert int(got[f].min()) == 255, f
    x[1].zero_()
    x[1, :256, :, 0] = 255                                                  # mean 127.5 in channel 0: a tie
    got = _batch_levels(x, (512,))[512].cpu()
    assert got[0].flatten().tolist() == [255, 255, 255] and got[1].flatten().tolist() == [128, 0, 0]


def test_source_canvas_beyond_2_31_bytes():
    h = w = 256
    grid_rows, grid_cols = 1000, 12
    canvas = torch.zeros(grid_rows * h, grid_cols * w, 3, dtype=torch.uint8, device=DEV)
    assert canvas.numel() > 2 ** 31
    tiles = _rand_u8((4, h, w, 3), 99)
    r = grid_rows - 1
    for t in range(4):
        canvas[r * h:(r + 1) * h, (8 + t) * w:(9 + t) * w] = tiles[t].to(DEV)
    dst = {f: torch.empty(h // f, 4 * (w // f), 3, dtype=torch.uint8, device=DEV) for f in FACTORS[:8]}
    E.pyramid_u8(canvas, (r, 8, 4, 0), 4, h, w, dst, (0, 0, 4, 0))
    del canvas
    for f in FACTORS[:8]:
        want = np.concatenate([PO.reduce(tiles[t].numpy(), f) for t in range(4)], axis=1)
        assert np.array_equal(dst[f].cpu().numpy(), want), f


def test_pil_cross_check():
    Image = pytest.importorskip("PIL.Image")
    slide = _rand_u8((2 * 512, 3 * 512, 3), 41)
    got = slide_pyramid(slide.to(DEV), (512, 512), FACTORS)
    region = slide.numpy()
    for f in FACTORS:
        assert np.array_equal(got[f].cpu().numpy(), np.asarray(Image.fromarray(region).reduce(f))), f


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("kind", ["uint8", "int64"])
def test_decompress_pyramid(precision, kind):
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = vqae_b200.set_precision(m.to(DEV), precision)
    try:
        cm = np.random.default_rng(6).integers(0, 256, (3 * 32, 5 * 32)).astype(np.uint8).astype(kind)
        cmd = torch.from_numpy(cm).to(DEV)
        fs = _valid(256, 256)
        for region, batch in ((None, 4), ((1, 1, 2, 3), 4), ((2, 4, 1, 1), 256)):     # 15 = 4+4+4+3, 6 = 4+2
            full = decompress_region(m, cmd, (32, 32), region, batch)
            got = decompress_pyramid(m, cmd, (32, 32), fs, region, batch)
            assert sorted(got) == list(fs)
            via_slide = slide_pyramid(full, (256, 256), fs)
            full_np = full.cpu().numpy()
            for f in fs:
                assert got[f].dtype == torch.uint8 and tuple(got[f].shape) == (full.shape[0] // f,
                                                                                full.shape[1] // f, 3)
                assert torch.equal(got[f].cpu(), torch.from_numpy(PO.reduce(full_np, f))), (region, f)
                assert torch.equal(got[f], via_slide[f]), (region, f)
        sparse = decompress_pyramid(m, cmd, (32, 32), (256, 2), batch=4)
        assert sorted(sparse) == [2, 256]
        whole = decompress_pyramid(m, cmd, (32, 32), fs, batch=4)
        assert torch.equal(sparse[2], whole[2]) and torch.equal(sparse[256], whole[256])
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()


@pytest.mark.skipif(not ref_shim.reference_available(), reason="no reference copy under oracle/_ref")
def test_decompress_pyramid_on_accelerated_reference_model():
    from vqae_b200.config import compose_vqae_conf
    tag = "model_nd3_perturbed"
    n_down, regime, batch, size, seed = H.MODEL_CASES[tag]
    model_mod, *_ = ref_shim.load_reference()
    conf = compose_vqae_conf(n_down=n_down)
    conf.pop("_target_"), conf.pop("_recursive_")
    ref = model_mod.VQAE(**conf).eval()
    mine, sd, _ = H.model_and_state(tag)
    ref.load_state_dict(mine.state_dict())
    fast = vqae_b200.accelerate(copy.deepcopy(ref)).to(DEV)
    mine = mine.to(DEV)
    try:
        cm = torch.from_numpy(np.random.default_rng(9).integers(0, 256, (64, 96)).astype(np.uint8)).to(DEV)
        fs = (2, 16, 256)
        n0 = E.launch_count()
        got = decompress_pyramid(fast, cm, (32, 32), fs, batch=4)
        assert E.launch_count() > n0
        want = decompress_pyramid(mine, cm, (32, 32), fs, batch=4)
        full = decompress_region(mine, cm, (32, 32), batch=4).cpu().numpy()
        for f in fs:
            assert torch.equal(got[f], want[f]) and torch.equal(got[f].cpu(), torch.from_numpy(PO.reduce(full, f)))
    finally:
        mine.cpu()


def test_errors():
    slide = _rand_u8((512, 768, 3), 1).to(DEV)
    with pytest.raises(RuntimeError):
        slide_pyramid(slide.cpu(), (256, 256), (2,))
    with pytest.raises(ValueError):
        slide_pyramid(slide.transpose(0, 1), (256, 256), (2,))              # not contiguous
    with pytest.raises(ValueError):
        slide_pyramid(slide.float(), (256, 256), (2,))
    with pytest.raises(ValueError):
        slide_pyramid(slide, (256, 200), (2,))                              # not a grid of patches
    for bad in ((), (3,), (1,), (2, 2), (1024,), (512,)):                 # 512 does not divide 256
        with pytest.raises(ValueError):
            slide_pyramid(slide, (256, 256), bad)
    with pytest.raises(ValueError):
        slide_pyramid(slide, (256, 256), (2,), batch=0)
    dst = {2: torch.empty(256, 384, 3, dtype=torch.uint8, device=DEV)}
    with pytest.raises(ValueError):
        E.pyramid_u8(slide, (0, 0, 3, 0), 6, 256, 256, {2: dst[2].transpose(0, 1)}, (0, 0, 3, 0))
    with pytest.raises(ValueError):
        E.pyramid_u8(slide, (0, 0, 3, 0), 6, 256, 256, {3: dst[2]}, (0, 0, 3, 0))
    with pytest.raises(L.VqaeError):
        E.pyramid_u8(slide, (0, 0, 3, 0), 7, 256, 256, dst, (0, 0, 3, 0))  # a 7th patch: outside
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    try:
        cm = torch.zeros(64, 96, dtype=torch.uint8, device=DEV)
        with pytest.raises(ValueError):
            decompress_pyramid(m, cm, (32, 32), (512,))
        with pytest.raises(ValueError):
            decompress_pyramid(m, cm, (32, 32), (6,))
        with pytest.raises(ValueError):
            decompress_pyramid(m, cm, (32, 32), (2,), region=(1, 1, 1, 3))
        with pytest.raises(RuntimeError):
            decompress_pyramid(m, cm.cpu(), (32, 32), (2,))
    finally:
        m.cpu()
