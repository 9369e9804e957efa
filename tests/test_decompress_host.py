"""CPU: the uint8 output convention of out_stem (u8 = rint(fma(v, 255 std_c, 255 mean_c)) clamped to
[0, 255], NaN -> 0) is the exact inverse of the input normalisation, level by level."""
import numpy as np
import pytest

import decompress_oracle as D
import vqae_oracle as O

STATS = {
    "camelyon16": (O.CAMELYON16_MEAN, O.CAMELYON16_STD),
    "imagenet": ((0.485, 0.456, 0.406), (0.229, 0.224, 0.225)),
    "half": ((0.5, 0.5, 0.5), (0.5, 0.5, 0.5)),
}


@pytest.mark.parametrize("name", sorted(STATS))
def test_denormalize_inverts_normalize_at_every_level(name):
    mean, std = STATS[name]
    levels = np.arange(256, dtype=np.uint8)
    img = np.stack([levels, levels[::-1], np.roll(levels, 77)], axis=-1).reshape(16, 16, 3)
    back = D.denormalize_u8(O.normalize_u8(img, mean, std), mean, std)
    assert back.dtype == np.uint8 and back.shape == img.shape
    assert np.array_equal(back, img)
    batch = np.stack([img, img[::-1]])                              # [B,H,W,3] <-> [B,3,H,W]
    assert np.array_equal(D.denormalize_u8(O.normalize_u8(batch, mean, std), mean, std), batch)


def test_denormalize_clamps_rounds_half_even_and_zeroes_nan():
    mean, std = (0.0, 0.0, 0.0), (1 / 255, 1 / 255, 1 / 255)      # s_c = 1 (exactly), o_c = 0
    s = np.float32(255.0) * np.float32(1 / 255)
    assert s == np.float32(1.0)
    v = np.array([-1e6, -0.6, -0.5, 0.5, 1.5, 2.5, 254.5, 255.4, 255.5, 1e9, np.inf, -np.inf, np.nan],
                 dtype=np.float32)
    want = np.array([0, 0, 0, 0, 2, 2, 254, 255, 255, 255, 255, 0, 0], dtype=np.uint8)
    x = np.broadcast_to(v[None, None, :], (3, 1, v.size))
    got = D.denormalize_u8(x, mean, std)
    for c in range(3):
        assert np.array_equal(got[0, :, c], want), (c, got[0, :, c])
    # with the CAMELYON16 constants: far outside the range -> 0 / 255, NaN -> 0
    x = np.array([-100.0, 100.0, np.nan], dtype=np.float32)[None, None, :].repeat(3, 0)
    got = D.denormalize_u8(x)
    assert np.array_equal(got[0], np.array([[0, 0, 0], [255, 255, 255], [0, 0, 0]], dtype=np.uint8))


def test_stitch_is_row_major():
    p = np.arange(6, dtype=np.uint8)[:, None, None, None] * np.ones((6, 2, 3, 3), dtype=np.uint8)
    img = D.stitch(p, 3)
    assert img.shape == (4, 9, 3)
    assert img[0, 0, 0] == 0 and img[0, 3, 0] == 1 and img[0, 8, 0] == 2 and img[2, 0, 0] == 3
    assert img[3, 8, 0] == 5
