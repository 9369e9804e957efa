"""CPU: the float64 metric oracle of tests/quality_oracle.py (against a direct 2-D window sum and known
answers), the host-side metrics of vqae_b200.quality, and the argument checks of vqae_quality_u8, which
return before any CUDA call."""
import ctypes as C

import numpy as np
import pytest
import torch

import quality_oracle as Q
import vqae_oracle as O
from vqae_b200 import _lib as L
from vqae_b200.quality import ReconstructionQuality


def _direct_ssim(x, y):
    """SSIM from a direct 11 x 11 window sum (torch float64 conv2d, valid padding)."""
    g = torch.from_numpy(Q.gaussian_taps_f32().astype(np.float64))
    w2 = torch.outer(g, g)[None, None]
    X = torch.from_numpy(x.astype(np.float64))[None, None]
    Y = torch.from_numpy(y.astype(np.float64))[None, None]
    f = lambda t: torch.nn.functional.conv2d(t, w2)[0, 0]      # noqa: E731
    mx, my = f(X), f(Y)
    sxx, syy, sxy = f(X * X) - mx * mx, f(Y * Y) - my * my, f(X * Y) - mx * my
    return (((2 * mx * my + Q.C1) * (2 * sxy + Q.C2)) / ((mx * mx + my * my + Q.C1) * (sxx + syy + Q.C2))).numpy()


@pytest.mark.parametrize("hw", [(11, 11), (40, 23), (64, 64)])
def test_oracle_matches_direct_window_sum(hw):
    rng = np.random.default_rng(hw[0] * 100 + hw[1])
    x = rng.integers(0, 256, hw)
    y = np.clip(x + rng.integers(-40, 41, hw), 0, 255)
    a, b = Q.ssim_map(x, y), _direct_ssim(x, y)
    assert a.shape == (hw[0] - 10, hw[1] - 10)
    assert np.abs(a - b).max() <= 1e-12


def test_known_answers():
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (32, 40, 3)).astype(np.uint8)
    assert Q.ssim(img, img) == pytest.approx(1.0, abs=1e-12)
    assert (Q.sse(img, img) == 0).all()
    q = ReconstructionQuality(torch.zeros(3, dtype=torch.int64), torch.ones((), dtype=torch.float64), (32, 40))
    assert float(q.psnr) == float("inf")
    # constant images a, b: (2ab + C1) / (a^2 + b^2 + C1).  The fp32 taps sum to W = 1 + O(1e-8), so the
    # window's moments are mu = a W^2 and s_xx = a^2 W^2 (1 - W^2): exact with W, to ~1e-6 without
    w2 = float(Q.gaussian_taps_f32().astype(np.float64).sum()) ** 2
    for a, b in ((255, 254), (30, 200), (0, 0)):
        x = np.full((20, 20, 3), a, np.uint8)
        y = np.full((20, 20, 3), b, np.uint8)
        v = w2 * (1 - w2)
        exact = ((2 * a * b * w2 * w2 + Q.C1) * (2 * a * b * v + Q.C2)) / \
            (((a * a + b * b) * w2 * w2 + Q.C1) * ((a * a + b * b) * v + Q.C2))
        assert Q.ssim(x, y) == pytest.approx(exact, rel=1e-12)
        assert Q.ssim(x, y) == pytest.approx((2 * a * b + Q.C1) / (a * a + b * b + Q.C1), rel=1e-5)
    yy, xx = np.mgrid[:24, :24]
    board = (((yy + xx) % 2) * 255).astype(np.uint8)[..., None].repeat(3, -1)
    assert Q.ssim(board, 255 - board) < 0


def test_weight_table():
    w = Q.gaussian_taps_f32()
    assert w.dtype == np.float32 and w.shape == (11,)
    assert abs(float(w.astype(np.float64).sum()) - 1.0) <= 1e-7
    assert np.array_equal(w, w[::-1])


def test_mse_psnr_and_normalised_mse_from_sse():
    rng = np.random.default_rng(11)
    ref = rng.integers(0, 256, (4, 16, 24, 3)).astype(np.uint8)
    rec = np.clip(ref.astype(np.int64) + rng.integers(-9, 10, ref.shape), 0, 255).astype(np.uint8)
    q = ReconstructionQuality(torch.from_numpy(Q.sse(ref, rec)), torch.zeros(4, dtype=torch.float64), (16, 24))
    d = ref.astype(np.float64) - rec.astype(np.float64)
    mse = (d * d).mean(axis=(1, 2, 3))
    assert np.allclose(q.mse.numpy(), mse, rtol=1e-14, atol=0)
    assert np.allclose(q.psnr.numpy(), 10 * np.log10(255.0 ** 2 / mse), rtol=1e-14, atol=0)
    for mean, std in ((None, None), ((0.5, 0.5, 0.5), (0.25, 0.2, 0.1))):
        kw = {} if mean is None else {"mean": mean, "std": std}
        # normalize_u8's formula (u8 - 255 mean) / (255 std) with its fp32 constants, in float64 ...
        m32 = np.array(kw.get("mean", O.CAMELYON16_MEAN), np.float32) * np.float32(255)
        d32 = np.reciprocal(np.array(kw.get("std", O.CAMELYON16_STD), np.float32) * np.float32(255),
                            dtype=np.float32)
        n64 = lambda u: (u.astype(np.float64) - m32) * d32.astype(np.float64)    # noqa: E731
        want = ((n64(ref) - n64(rec)) ** 2).mean(axis=(1, 2, 3))
        got = q.mse_normalised(mean, std).numpy()
        assert np.allclose(got, want, rtol=1e-12, atol=0)
        # ... and normalize_u8 itself (its fp32 rounding)
        f32 = ((O.normalize_u8(ref, **kw).astype(np.float64) - O.normalize_u8(rec, **kw)) ** 2).mean(axis=(1, 2, 3))
        assert np.allclose(got, f32, rtol=1e-5, atol=0)
    s = q.summary()
    assert s["patches"] == 4
    assert s["mse_pooled"] == pytest.approx(mse.mean(), rel=1e-14)
    assert s["psnr_pooled"] == pytest.approx(10 * np.log10(255.0 ** 2 / mse.mean()), rel=1e-14)
    assert s["psnr_mean"] == pytest.approx(float(np.mean(10 * np.log10(255.0 ** 2 / mse))), rel=1e-14)


def test_abi_rejects_bad_arguments_without_cuda():
    lib = L.load()                          # no GPU needed: every case returns before a CUDA call
    fake = C.c_void_p(4096)                 # never dereferenced
    out_sse, out_ssim = C.c_void_p(8192), C.c_void_p(16384)
    need = lib.vqae_quality_u8_scratch_bytes(2, 64, 64)
    assert need > 0 and lib.vqae_quality_u8_scratch_bytes(2, 10, 64) == 0

    def call(ref=fake, rec=fake, rows=128, cols=64, r0=0, c0=0, rc=1, first=0, rec_rows=128, batch=2,
             h=64, w=64, sse=out_sse, ssim=out_ssim, scratch=fake, nbytes=need):
        return lib.vqae_quality_u8(ref, rows, cols, r0, c0, rc, first, rec, rec_rows, 64, 0, 0, 1, 0, batch,
                                   h, w, sse, ssim, scratch, nbytes, None)
    for kw in ({"ref": None}, {"rec": None}, {"sse": None}, {"ssim": None}, {"batch": 0}, {"h": 0},
               {"first": 1}, {"rows": 127}, {"rec_rows": 64}, {"c0": 1}, {"rc": 2}, {"r0": -1}, {"rc": 0}):
        assert call(**kw) == L.ERR_BAD_ARG, kw
    assert call(h=10, w=10, rows=20, rec_rows=20) == L.ERR_UNSUPPORTED
    assert call(h=64, w=10) == L.ERR_UNSUPPORTED
    big = 1 << 31
    assert call(first=big - 1, rc=big, cols=big * 64, batch=2) == L.ERR_UNSUPPORTED     # patches 2^31 - 1, 2^31
    assert call(nbytes=need - 1) == L.ERR_SCRATCH
    assert call(scratch=None) == L.ERR_SCRATCH
