"""CPU: the numpy JPEG oracle of tests/jpeg_oracle.py against Pillow byte for byte, the DeepZoom geometry of
vqae_b200.jpeg, and the argument checks of vqae_jpeg_tiles, which return before any CUDA call."""
import ctypes as C
import io
import xml.etree.ElementTree as ET

import numpy as np
import pytest

import jpeg_oracle as JO
from vqae_b200 import _lib as L
from vqae_b200 import jpeg as J

Image = pytest.importorskip("PIL.Image")

SIZES = [(1, 1), (8, 8), (15, 31), (17, 33), (120, 200), (195, 195), (255, 256), (256, 256)]
QUALITIES = [1, 10, 50, 75, 90, 100]


def images(h, w, seed=0):
    rng = np.random.default_rng(seed + 7 * h + w)
    yy, xx = np.mgrid[:h, :w]
    smooth = np.stack([128 + 100 * np.sin(xx / 7 + c) * np.cos(yy / 11) for c in range(3)], -1)
    return {"random": rng.integers(0, 256, (h, w, 3), dtype=np.uint8), "zeros": np.zeros((h, w, 3), np.uint8),
            "full": np.full((h, w, 3), 255, np.uint8), "smooth": smooth.astype(np.uint8),
            "checkerboard": (((yy + xx) % 2) * 255).astype(np.uint8)[..., None].repeat(3, -1)}


def pil_jpeg(img, quality, subsampling):
    buf = io.BytesIO()
    Image.fromarray(img).save(buf, "JPEG", quality=quality, subsampling=subsampling)
    return buf.getvalue()


@pytest.mark.parametrize("subsampling", [0, 2])
@pytest.mark.parametrize("quality", QUALITIES)
def test_oracle_equals_pillow(quality, subsampling):
    for h, w in SIZES:
        for name, img in images(h, w).items():
            assert JO.encode(img, quality, subsampling) == pil_jpeg(img, quality, subsampling), (h, w, name)


def test_header_and_tables_match_pillow():
    for q in range(1, 101):
        got = pil_jpeg(np.zeros((9, 250, 3), np.uint8), q, 2)
        hdr = J.jpeg_header(9, 250, q, 2)
        assert got[:len(hdr)] == hdr, q
    with pytest.raises(ValueError):
        J.jpeg_header(0, 5, 90, 2)
    with pytest.raises(ValueError):
        J.jpeg_header(5, 65536, 90, 2)
    for bad in ((0, 2), (101, 2), (90, 1), (90, 3), (90.5, 2)):
        with pytest.raises(ValueError):
            J.check_quality(*bad)


def test_deepzoom_geometry():
    assert J.dz_levels(1, 1) == [(1, 1)]
    lv = J.dz_levels(768, 512)                                   # M = ceil(log2 768) = 10
    assert len(lv) == 11 and lv[-1] == (768, 512) and lv[0] == (1, 1) and lv[9] == (384, 256)
    assert J.dz_levels(49920, 49920)[-2] == (24960, 24960)
    assert J.dz_levels(1000, 3)[5] == (32, 1)                    # ceil(1000 / 32), ceil(3 / 32)
    for w, t, o in ((768, 254, 1), (1000, 254, 3), (254, 254, 1), (255, 254, 0), (5, 3, 2)):
        cols, _ = J.tile_grid(w, 1, t)
        assert cols == -(-w // t)
        covered = np.zeros(w, bool)
        for c in range(cols):
            x0, x1 = J.tile_span(c, w, t, o)
            assert x0 == max(0, c * t - o) and x1 == min(w, (c + 1) * t + o) and x1 > x0
            covered[x0:x1] = True
        assert covered.all()
    assert J.tile_rect(1, 2, 768, 512, 254, 1) == (253, 507, 509, 512)
    root = ET.fromstring(J.dzi_xml(768, 512, 254, 1))
    assert root.tag.endswith("Image") and root.attrib == {"Format": "jpeg", "Overlap": "1", "TileSize": "254"}
    size = root[0]
    assert size.tag.endswith("Size") and size.attrib == {"Height": "512", "Width": "768"}
    hdrs = J.level_headers(768, 512, 254, 1, 90, 2)
    n = len(J.jpeg_header(1, 1, 90, 2))
    assert len(hdrs) == 16 * n
    assert hdrs[0:n] == J.jpeg_header(255, 255, 90, 2)           # first row, first column
    assert hdrs[9 * n:10 * n] == J.jpeg_header(256, 256, 90, 2)  # row 1 (of 3: class 2), column 1
    assert hdrs[15 * n:16 * n] == J.jpeg_header(512 - 507, 768 - 761, 90, 2)
    for bad in ((254, 254), (8, 16), (0, 0), (5, -1)):
        with pytest.raises(ValueError):
            J.check_tiling(*bad)


@pytest.mark.parametrize("width,height,tile,overlap", [
    (763, 509, 254, 2), (763, 509, 254, 3), (1017, 255, 254, 4), (154, 87, 17, 3), (19, 10, 9, 8), (9, 9, 8, 2),
    (768, 512, 254, 1), (771, 517, 64, 3), (5, 5, 2, 1), (1, 1, 254, 1), (255, 254, 254, 0)])
def test_every_tile_gets_a_header_of_its_size(width, height, tile, overlap):
    """Tiles of one class have one size, including a second-to-last tile that reaches the extent because
    the last one is narrower than the overlap (extent = k tile + 1, overlap >= 2)."""
    hdrs = J.level_headers(width, height, tile, overlap, 75, 2)
    n = len(hdrs) // 16
    cols, rows = J.tile_grid(width, height, tile)
    for r in range(rows):
        for c in range(cols):
            x0, y0, x1, y1 = J.tile_rect(c, r, width, height, tile, overlap)
            k = 4 * J.tile_class(r, rows) + J.tile_class(c, cols)
            assert hdrs[k * n:(k + 1) * n] == J.jpeg_header(y1 - y0, x1 - x0, 75, 2), (c, r)


def test_abi_rejects_bad_arguments_without_cuda():
    lib = L.load()                          # no GPU needed: every case returns before a CUDA call
    hl = len(J.jpeg_header(1, 1, 90, 2))
    hdr = np.frombuffer(J.level_headers(600, 500, 254, 1, 90, 2), np.uint8)
    assert len(hdr) == 16 * hl
    qt = J.quant_tables(90)
    args = (500, 600, 254, 1, 0, 2, 2, hl)
    worst = lib.vqae_jpeg_tiles_worst_bytes(*args)
    need = lib.vqae_jpeg_tiles_scratch_bytes(*args)
    assert worst > 0 and need > 0
    assert lib.vqae_jpeg_tiles_worst_bytes(500, 600, 254, 1, 0, 3, 2, hl) == -1       # only 2 tile rows
    assert lib.vqae_jpeg_tiles_scratch_bytes(500, 600, 254, 1, 0, 2, 1, hl) == 0      # 4:2:2
    assert lib.vqae_jpeg_tiles_scratch_bytes(100, 100, 8, 16, 0, 1, 0, hl) == 0       # overlap >= tile
    assert lib.vqae_jpeg_tiles_worst_bytes(100, 100, 8, 8, 0, 1, 0, hl) == -1
    fake = C.c_void_p(0x1000)

    def call(canvas=fake, pitch=1800, h=500, w=600, t=254, o=1, r0=0, nr=2, q=90, s=2, hdr_p=hdr.ctypes.data,
             hlen=hl, qt_p=qt.ctypes.data, offsets=fake, payload=fake, cap=worst, scratch=fake, sb=need):
        return lib.vqae_jpeg_tiles(canvas, pitch, h, w, t, o, r0, nr, q, s, hdr_p, hlen, qt_p, offsets, payload,
                                   cap, scratch, sb, None)

    bad_arg = [dict(canvas=None), dict(hdr_p=None), dict(qt_p=None), dict(offsets=None), dict(payload=None),
               dict(scratch=None), dict(h=0), dict(w=-1), dict(t=0), dict(o=-1), dict(o=254), dict(t=8, o=16, nr=1),
               dict(r0=-1), dict(nr=0), dict(nr=3), dict(r0=1, nr=2), dict(pitch=1799), dict(hlen=0), dict(cap=worst - 1)]
    for kw in bad_arg:
        assert call(**kw) == L.ERR_BAD_ARG, kw
    for kw in (dict(q=0), dict(q=101), dict(s=1), dict(s=4), dict(h=70000, t=65535, o=1, nr=1, pitch=1800)):
        assert call(**kw) == L.ERR_UNSUPPORTED, kw
    assert call(sb=need - 1) == L.ERR_SCRATCH
    zero_q = qt.copy()
    zero_q[1, 5] = 0
    assert call(qt_p=zero_q.ctypes.data) == L.ERR_BAD_ARG
