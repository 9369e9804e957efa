"""GPU: code map -> uint8 RGB decompression (out_stem's uint8 epilogue, the code-map window gather,
VQAE.decode_codes_u8, extract.decompress_region)."""
import copy
import ctypes as C

import numpy as np
import pytest
import torch

import decompress_oracle as D
import helpers as H
import ref_shim
import vqae_b200
import vqae_oracle as O
from vqae_b200 import _lib as L
from vqae_b200 import engine as E
from vqae_b200 import synthetic as S
from vqae_b200.extract import compress_slide, decompress_region, encode_patches

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
S255 = (np.array(O.CAMELYON16_STD, np.float32) * np.float32(255)).astype(np.float64)
O255 = (np.array(O.CAMELYON16_MEAN, np.float32) * np.float32(255)).astype(np.float64)


def _copy_stem():
    """out_stem weights that pass input channels 0-2 through the centre tap, zero bias."""
    w = torch.zeros(3, 8, 3, 3)
    for c in range(3):
        w[c, c, 1, 1] = 1.0
    return w.to(DEV), torch.zeros(3, device=DEV)


def _normalised_nhwc8(tiles_u8):
    """normalize_u8 of uint8 [B,H,W,3] tiles, NHWC, zero-padded to 8 channels, on the device."""
    x = np.moveaxis(O.normalize_u8(tiles_u8.numpy()), 1, -1)
    out = torch.zeros(*x.shape[:3], 8)
    out[..., :3] = torch.from_numpy(x)
    return out.to(DEV)


@pytest.mark.parametrize("size", [256, 512])
@pytest.mark.parametrize("precision", ["fp32", "fp16"])          # CUDA-core / tensor-core kernel
def test_u8_epilogue_is_exact_inverse(size, precision):
    w, b = _copy_stem()
    tiles = S.synthetic_patches_u8(5, size, 17)
    x = _normalised_nhwc8(tiles)
    # batch form
    canvas = torch.empty(5 * size, size, 3, dtype=torch.uint8, device=DEV)
    E.stem_out_u8(x, w, b, canvas, 0, 1, precision=precision)
    assert torch.equal(canvas.view(5, size, size, 3).cpu(), tiles)
    # canvas form: patches 7 .. 11 of a 3 x 4 grid (the last row and the last column), and the same on
    # a canvas whose rows are not 16-byte multiples (byte stores)
    for extra in (0, 8):
        canvas = torch.full((3 * size, 4 * size + extra, 3), 77, dtype=torch.uint8, device=DEV)
        E.stem_out_u8(x, w, b, canvas, 7, 4, precision=precision)
        want = torch.full_like(canvas, 77).cpu()
        for t in range(5):
            q = 7 + t
            r, c = q // 4, q % 4
            want[r * size:(r + 1) * size, c * size:(c + 1) * size] = tiles[t]
        assert torch.equal(canvas.cpu(), want), extra
    # values pushed out of range clamp to 0 / 255
    x2 = x.clone()
    x2[1, 5, 7, 0] = 10.0
    x2[3, size - 1, size - 1, 1] = -10.0
    x2[4, 0, 31, 2] = 50.0
    out = torch.empty(5 * size, size, 3, dtype=torch.uint8, device=DEV)
    E.stem_out_u8(x2, w, b, out, precision=precision)
    want = tiles.clone()
    want[1, 5, 7, 0], want[3, size - 1, size - 1, 1], want[4, 0, 31, 2] = 255, 0, 255
    assert torch.equal(out.view(5, size, size, 3).cpu(), want)
    # a NaN bias makes every value NaN: all zero
    E.stem_out_u8(x, w, torch.full((3,), float("nan"), device=DEV), out, precision=precision)
    assert int(out.max()) == 0


def _denorm64(f_nchw):
    """float64 pre-rounding values 255 std_c v + 255 mean_c, NHWC."""
    v = f_nchw.permute(0, 2, 3, 1).double().cpu().numpy()
    return v * S255 + O255


@pytest.mark.parametrize("tag", ["model_nd3_perturbed", "model_nd3_fixup", "model_nd4_perturbed_512"])
@pytest.mark.parametrize("precision", ["fp32", "fp16", "fp32tc"])
def test_decode_codes_u8_equals_float_path(tag, precision):
    """The u8 kernels share the arithmetic of the fp32-output kernels up to the stored value, so the
    uint8 result is the rounded float output of the same mode: equal except where the value lies
    within 1e-3 of a half-integer (fma and float64 may round to different sides), and there by 1."""
    g = H.golden(tag)
    m, sd, _ = H.model_and_state(tag)
    m = vqae_b200.set_precision(m.to(DEV), precision)
    try:
        idx = torch.from_numpy(g["idx"].astype(np.int64)).to(DEV)
        u8 = m.decode_codes_u8(idx)
        f = m.decode_codes(idx)
        u8_from_u8_codes = m.decode_codes_u8(idx.to(torch.uint8))
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()
    assert u8.dtype == torch.uint8 and tuple(u8.shape) == (f.shape[0], f.shape[2], f.shape[3], 3)
    assert torch.equal(u8, u8_from_u8_codes)
    pre = _denorm64(f)
    ref = np.clip(np.rint(pre), 0, 255)
    d = np.abs(u8.cpu().numpy().astype(np.float64) - ref)
    near_half = np.abs(pre - np.floor(pre) - 0.5) < 1e-3
    assert not (d[~near_half] > 0).any(), int((d[~near_half] > 0).sum())
    assert d.max() <= 1


@pytest.mark.parametrize("tag", sorted(H.MODEL_CASES))
@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_decode_codes_u8_vs_reference_golden(tag, precision):
    """The reference's codes decoded to pixels against the reference's own decode, de-normalised by the
    oracle, on the ::8 sub-grid the goldens store.  fp32: within one level.  fp16: the 1e-2 relative
    decoder bar of the float path, in levels."""
    g = H.golden(tag)
    m, sd, _ = H.model_and_state(tag)
    m = vqae_b200.set_precision(m.to(DEV), precision)
    try:
        u8 = m.decode_codes_u8(torch.from_numpy(g["idx"].astype(np.int64)).to(DEV))
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()
    ref_f = g["decode_codes_sub"]
    ref = D.denormalize_u8(ref_f).astype(np.int32)
    got = u8.cpu().numpy()[:, ::8, ::8].astype(np.int32)
    d = int(np.abs(got - ref).max())
    bar = 1.0 if precision == "fp32" else 1 + 0.01 * float(np.abs(ref_f).max()) * 255 * max(O.CAMELYON16_STD)
    print(f"{tag} [{precision}]: max |u8 - reference| = {d} levels (bar {bar:.2f})")
    assert d <= bar


def _gather_tiles(cm, th, tw, region):
    r0, c0, nr, nc = region
    return np.stack([cm[(r0 + r) * th:(r0 + r + 1) * th, (c0 + c) * tw:(c0 + c + 1) * tw]
                     for r in range(nr) for c in range(nc)])


@pytest.mark.parametrize("kind", ["uint8", "int64", "bool"])
def test_decompress_region(kind):
    m, sd, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    try:
        rng = np.random.default_rng(5)
        if kind == "bool":
            cm = rng.integers(0, 2, (3 * 32, 5 * 32)).astype(bool)
        else:
            cm = rng.integers(0, 256, (3 * 32, 5 * 32)).astype(np.uint8).astype(kind)
        cmd = torch.from_numpy(cm).to(DEV)
        for arg, region, batch in ((None, (0, 0, 3, 5), 4), ((0, 0, 3, 5), (0, 0, 3, 5), 256),
                                   ((1, 1, 2, 2), (1, 1, 2, 2), 3), ((2, 4, 1, 1), (2, 4, 1, 1), 4)):
            got = decompress_region(m, cmd, (32, 32), arg, batch)
            tiles = torch.from_numpy(_gather_tiles(cm.astype(np.int64), 32, 32, region)).to(DEV)
            want = D.stitch(m.decode_codes_u8(tiles).cpu().numpy(), region[3])
            assert got.dtype == torch.uint8 and got.device == cmd.device
            assert np.array_equal(got.cpu().numpy(), want), (region, batch)
        out = torch.empty(2 * 256, 2 * 256, 3, dtype=torch.uint8, device=DEV)
        a = decompress_region(m, cmd, (32, 32), (1, 1, 2, 2), 3, out=out)
        first = out.clone()
        b = decompress_region(m, cmd, (32, 32), (1, 1, 2, 2), 3, out=out)
        assert a.data_ptr() == out.data_ptr() == b.data_ptr()
        assert torch.equal(first, out)
    finally:
        m.cpu()


def test_round_trip_through_compress_slide():
    m, sd, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    try:
        grid = (2, 3)
        img = S.synthetic_patches_u8(6, 256, 5)
        cmap = compress_slide(m.encoder, [(0, img[:4]), (4, img[4:])], grid, (32, 32), torch.device(DEV))
        slide = decompress_region(m, cmap, (32, 32), batch=4)
        assert tuple(slide.shape) == (2 * 256, 3 * 256, 3)
        want = D.stitch(m.decode_codes_u8(encode_patches(m.encoder, img.to(DEV))).cpu().numpy(), 3)
        assert np.array_equal(slide.cpu().numpy(), want)
        # the pixels go back into the encoder as they are
        idx = encode_patches(m.encoder, m.decode_codes_u8(cmap[:32, :32][None].long()))
        assert idx.shape == (1, 32, 32)
    finally:
        m.cpu()


def test_errors():
    m, sd, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    try:
        cm = torch.zeros(64, 96, dtype=torch.int64, device=DEV)
        bad = cm.clone()
        bad[40, 70] = 256
        with pytest.raises(ValueError):
            decompress_region(m, bad, (32, 32))
        bad[40, 70] = -1
        with pytest.raises(ValueError):
            decompress_region(m, bad, (32, 32))
        decompress_region(m, bad, (32, 32), region=(0, 0, 1, 3))        # outside the region: fine
        with pytest.raises(ValueError):
            decompress_region(m, cm, (32, 32), region=(1, 1, 1, 3))
        with pytest.raises(ValueError):
            decompress_region(m, cm, (32, 32), region=(0, 0, 0, 1))
        with pytest.raises(ValueError):
            decompress_region(m, cm[:60], (32, 32))
        with pytest.raises(ValueError):
            decompress_region(m, cm.float(), (32, 32))
        with pytest.raises(ValueError):
            decompress_region(m, cm, (32, 32), out=torch.empty(512, 512, 3, dtype=torch.uint8, device=DEV))
        with pytest.raises(ValueError):
            decompress_region(m, cm, (32, 32), out=torch.empty(512, 768, 3, dtype=torch.int32, device=DEV))
        with pytest.raises(RuntimeError):
            decompress_region(m, cm.cpu(), (32, 32))
        with pytest.raises(RuntimeError):
            m.decode_codes_u8(cm[:32, :32][None].cpu())
        m.train()
        try:
            with pytest.raises(RuntimeError):
                m.decode_codes_u8(cm[:32, :32][None])
            with pytest.raises(RuntimeError):
                decompress_region(m, cm, (32, 32))
        finally:
            m.eval()
    finally:
        m.cpu()
    two, _, _ = H.multilevel_model_and_state("flat")
    with pytest.raises(NotImplementedError):
        two.decode_codes_u8(torch.zeros(1, 32, 32, dtype=torch.int64, device=DEV))
    with pytest.raises(NotImplementedError):
        decompress_region(two, torch.zeros(32, 32, dtype=torch.int64, device=DEV), (32, 32))


def test_abi_rejects_bad_placements_before_launching():
    lib = L.load()
    x = torch.zeros(2, 64, 64, 8, device=DEV)
    w, b = _copy_stem()
    canvas = torch.zeros(128, 128, 3, dtype=torch.uint8, device=DEV)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    mean, std = L.f3(O.CAMELYON16_MEAN), L.f3(O.CAMELYON16_STD)
    p = E._ptr
    n0 = E.raw_launch_count()
    for kernel in (L.STEM_OUT_EXACT, L.STEM_OUT_TENSOR_CORE):
        def call(xp=p(x), cp=p(canvas), rows=128, cols=128, first=0, gcols=2, batch=2, mp=mean, sp=std):
            return lib.vqae_stem_out_u8(xp, p(w), p(b), mp, sp, cp, rows, cols, first, gcols, batch, 64,
                                        64, 8, kernel, st)
        assert call(first=3) == L.ERR_BAD_ARG                   # patches 3, 4: row 2 of a 2-row canvas
        assert call(gcols=3) == L.ERR_BAD_ARG                   # 3 columns of 64 on 128
        assert call(first=2, rows=127) == L.ERR_BAD_ARG          # patches 2, 3: rows 64 .. 127
        assert call(first=-1) == L.ERR_BAD_ARG
        assert call(gcols=0) == L.ERR_BAD_ARG
        assert call(batch=0) == L.ERR_BAD_ARG
        assert call(xp=None) == L.ERR_BAD_ARG
        assert call(cp=None) == L.ERR_BAD_ARG
        assert call(mp=None) == L.ERR_BAD_ARG
    table = torch.zeros(256, 64, device=DEV)
    cm = torch.zeros(64, 96, dtype=torch.uint8, device=DEV)
    out = torch.empty(6, 32, 32, 64, device=DEV)

    def gather(mp=p(cm), r0=0, c0=0, rcols=3, first=0, n=6, tp=p(table), op=p(out)):
        return lib.vqae_embed_codemap_f32(mp, 1, 64, 96, 32, 32, r0, c0, rcols, first, n, tp, 256, 64, op, st)
    assert gather(n=7) == L.ERR_BAD_ARG                         # a third patch row
    assert gather(c0=1) == L.ERR_BAD_ARG
    assert gather(r0=-1) == L.ERR_BAD_ARG
    assert gather(mp=None) == L.ERR_BAD_ARG
    assert gather(op=None) == L.ERR_BAD_ARG
    assert gather(tp=None) == L.ERR_BAD_ARG
    torch.cuda.synchronize()
    assert E.raw_launch_count() == n0                           # nothing was launched
    assert gather() == L.OK and E.raw_launch_count() == n0 + 1


@pytest.mark.skipif(not ref_shim.reference_available(), reason="no reference copy under oracle/_ref")
def test_decompress_region_on_accelerated_reference_model():
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
        n0 = E.launch_count()
        got = decompress_region(fast, cm, (32, 32), batch=4)
        assert E.launch_count() > n0
        assert torch.equal(got, decompress_region(mine, cm, (32, 32), batch=4))
    finally:
        mine.cpu()
