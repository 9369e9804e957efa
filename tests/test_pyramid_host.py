"""CPU: the numpy pyramid oracle of tests/pyramid_oracle.py against PIL.Image.reduce, exact ties, the factor
validation of vqae_b200.pyramid, and the argument checks of vqae_pyramid_u8, which return before any CUDA
call."""
import ctypes as C

import numpy as np
import pytest

import pyramid_oracle as PO
from vqae_b200 import _lib as L
from vqae_b200.pyramid import FACTORS, check_factors


def _images():
    rng = np.random.default_rng(4)
    yy, xx = np.mgrid[:512, :1024]
    board = (((yy + xx) % 2) * 255).astype(np.uint8)[..., None].repeat(3, -1)
    return {"random": rng.integers(0, 256, (512, 1024, 3)).astype(np.uint8),
            "zeros": np.zeros((512, 1024, 3), np.uint8), "full": np.full((512, 1024, 3), 255, np.uint8),
            "checkerboard": board, "checkerboard_inv": 255 - board}


@pytest.mark.parametrize("f", FACTORS)
def test_oracle_equals_pil_reduce(f):
    Image = pytest.importorskip("PIL.Image")
    for name, img in _images().items():
        want = np.asarray(Image.fromarray(img).reduce(f))
        got = PO.reduce(img, f)
        assert got.shape == (512 // f, 1024 // f, 3)
        assert np.array_equal(got, want), (name, f)


def test_exact_ties_round_up():
    """Blocks whose sum is q f^2 + f^2 / 2 (a mean of exactly q + 1/2) give q + 1, for every factor and
    for q from 0 to 254."""
    for f in FACTORS:
        qs = np.arange(255)
        img = np.repeat(qs.astype(np.uint8), f)[None, :].repeat(f, 0)           # [f, 255 f]: block q = q
        img = img.copy()
        for b, q in enumerate(qs):
            blk = img[:, b * f:(b + 1) * f].reshape(-1)
            blk[:f * f // 2] = q + 1                                            # half the pixels one higher
            img[:, b * f:(b + 1) * f] = blk.reshape(f, f)
        img3 = np.stack([img, img, img], -1)
        s = img3.astype(np.int64).reshape(1, f, 255, f, 3).sum(axis=(1, 3))
        assert ((s % (f * f)) == f * f // 2).all()
        assert np.array_equal(PO.reduce(img3, f)[0, :, 0], (qs + 1).astype(np.uint8)), f


def test_factor_validation():
    assert check_factors([16, 2, 256], (256, 256)) == (2, 16, 256)
    assert check_factors([np.int64(64)], (192, 320)) == (64,)
    assert check_factors(FACTORS, (512, 512)) == FACTORS
    for bad, hw in (([], (256, 256)), ([1], (256, 256)), ([3], (256, 256)), ([1024], (1024, 1024)),
                    ([2, 2], (256, 256)), ([128], (192, 320)), ([32], (16, 16)), ([2.0], (256, 256)),
                    (["2"], (256, 256)), ([0], (256, 256)), ([-2], (256, 256)), ([True], (256, 256))):
        with pytest.raises(ValueError):
            check_factors(bad, hw)


def test_abi_rejects_bad_arguments_without_cuda():
    lib = L.load()                          # no GPU needed: every case returns before a CUDA call
    fake = C.c_void_p(4096)                 # never dereferenced
    m_all = 0x3fe
    need = lib.vqae_pyramid_u8_scratch_bytes(2, 512, 512, m_all)
    assert need > 0
    assert lib.vqae_pyramid_u8_scratch_bytes(2, 256, 256, 0x7e) == 0              # f <= 64: no scratch
    assert lib.vqae_pyramid_u8_scratch_bytes(2, 64, 64, 1 << 7) == 0              # 128 does not divide 64
    assert lib.vqae_pyramid_u8_scratch_bytes(2, 256, 256, 1 << 10) == 0
    assert lib.vqae_pyramid_u8_scratch_bytes(2, 256, 256, 1) == 0
    assert lib.vqae_pyramid_u8_scratch_bytes(0, 256, 256, 1 << 8) == 0

    def call(src=fake, rows=1024, cols=512, r0=0, c0=0, rc=1, first=0, batch=2, h=512, w=512, mask=m_all,
             dst=None, drows=None, dcols=None, dr0=0, dc0=0, drc=1, dfirst=0, scratch=fake, nbytes=need,
             null_level=None):
        ptrs, rr, cc = (C.c_void_p * 10)(), (C.c_int64 * 10)(), (C.c_int64 * 10)()
        for k in range(1, 10):              # level canvases [2 * 512 / f, 512 / f, 3]
            ptrs[k], rr[k], cc[k] = 4096 * (k + 1), 1024 >> k, 512 >> k
        if null_level is not None:
            ptrs[null_level] = None
        if drows is not None:
            rr[drows[0]] = drows[1]
        if dcols is not None:
            cc[dcols[0]] = dcols[1]
        return lib.vqae_pyramid_u8(src, rows, cols, r0, c0, rc, first, batch, h, w, mask,
                                   ptrs if dst is None else dst, rr, cc, dr0, dc0, drc, dfirst, scratch, nbytes,
                                   None)
    for kw in ({"src": None}, {"batch": 0}, {"h": 0}, {"w": -512}, {"mask": 0}, {"first": -1},
               {"dfirst": -1}, {"null_level": 5}, {"rows": 1023}, {"rows": 0}, {"cols": 511}, {"first": 1},
               {"r0": 1}, {"c0": 1}, {"rc": 2}, {"rc": 0}, {"r0": -1}, {"drows": (3, 127)},
               {"dcols": (9, 0)}, {"dfirst": 1}, {"dc0": 1}, {"drc": 2}, {"dr0": 1}):
        assert call(**kw) == L.ERR_BAD_ARG, kw
    assert lib.vqae_pyramid_u8(fake, 1024, 512, 0, 0, 1, 0, 2, 512, 512, m_all, None, fake, fake, 0, 0, 1, 0,
                               fake, need, None) == L.ERR_BAD_ARG
    for kw in ({"mask": 1}, {"mask": 1 << 10}, {"mask": m_all | 1}, {"mask": -1},
               {"h": 256, "mask": 1 << 9}, {"w": 320, "mask": 1 << 7}, {"h": 192, "w": 320, "mask": 1 << 7}):
        assert call(**kw) == L.ERR_UNSUPPORTED, kw
    big = 1 << 31
    assert call(first=big - 1, rc=big, cols=big * 512, batch=2) == L.ERR_UNSUPPORTED   # patches 2^31 - 1, 2^31
    assert call(dfirst=big - 1, drc=big, batch=2) == L.ERR_UNSUPPORTED
    assert call(nbytes=need - 1) == L.ERR_SCRATCH
    assert call(scratch=None) == L.ERR_SCRATCH
