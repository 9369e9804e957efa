"""GPU: DeepZoom JPEG tiles (csrc/jpeg.cu, engine.jpeg_tiles, vqae_b200.jpeg.encode_tiles,
extract.export_deepzoom) against Pillow and the numpy oracle of tests/jpeg_oracle.py; every check is byte
equality."""
import io
import xml.etree.ElementTree as ET

import numpy as np
import pytest
import torch

import helpers as H
import jpeg_oracle as JO
import vqae_b200
from test_jpeg_host import QUALITIES, SIZES, images, pil_jpeg
from vqae_b200 import _lib as L
from vqae_b200 import engine as E
from vqae_b200 import jpeg as J
from vqae_b200.extract import decompress_region, export_deepzoom
from vqae_b200.pyramid import slide_pyramid

Image = pytest.importorskip("PIL.Image")
pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def check_level(img, tiles, tile, overlap, quality, subsampling, rows=None):
    """Every tile of ``tiles`` equals Pillow's encode of the matching crop of ``img``."""
    h, w = img.shape[:2]
    cols, n_rows = J.tile_grid(w, h, tile)
    r0, nr = rows if rows is not None else (0, n_rows)
    assert tiles.grid == (cols, nr) and len(tiles.offsets) == cols * nr + 1
    host = tiles.payload.cpu().numpy()
    assert tiles.nbytes() == len(host)
    for r in range(r0, r0 + nr):
        for c in range(cols):
            x0, y0, x1, y1 = J.tile_rect(c, r, w, h, tile, overlap)
            want = pil_jpeg(np.ascontiguousarray(img[y0:y1, x0:x1]), quality, subsampling)
            assert tiles.tile_bytes(c, r, host) == want, (c, r, quality, subsampling)


@pytest.mark.parametrize("subsampling", [0, 2])
@pytest.mark.parametrize("quality", QUALITIES)
def test_single_tiles_equal_pillow(quality, subsampling):
    for h, w in SIZES:
        for name, img in images(h, w).items():
            tiles = J.encode_tiles(torch.from_numpy(img).to(DEV), tile=max(h, w), overlap=0, quality=quality,
                                   subsampling=subsampling)
            want = pil_jpeg(img, quality, subsampling)
            assert tiles.tile_bytes(0, 0) == want, (h, w, name)
            if quality in (1, 100):
                assert want == JO.encode(img, quality, subsampling)


@pytest.mark.parametrize("subsampling", [0, 2])
@pytest.mark.parametrize("tile_overlap", [(254, 1), (64, 3), (100, 0), (17, 2)])
def test_grids(tile_overlap, subsampling):
    tile, overlap = tile_overlap
    rng = np.random.default_rng(tile)
    yy, xx = np.mgrid[:517, :771]
    img = np.clip(np.stack([128 + 90 * np.sin(xx / 13 + c) * np.cos(yy / 29) for c in range(3)], -1)
                  + rng.integers(-25, 26, (517, 771, 3)), 0, 255).astype(np.uint8)
    d = torch.from_numpy(img).to(DEV)
    for q in (10, 90):
        check_level(img, J.encode_tiles(d, tile, overlap, q, subsampling), tile, overlap, q, subsampling)
    rows = J.tile_grid(771, 517, tile)[1]
    for r0, nr in ((0, 1), (1, max(1, rows - 2)), (rows - 1, 1)):
        check_level(img, J.encode_tiles(d, tile, overlap, 75, subsampling, rows=(r0, nr)), tile, overlap, 75,
                    subsampling, (r0, nr))



@pytest.mark.parametrize("subsampling", [0, 2])
@pytest.mark.parametrize("width,height,tile,overlap", [
    (763, 509, 254, 2), (1017, 763, 254, 3), (154, 87, 17, 3), (19, 10, 9, 8), (9, 9, 8, 2), (1, 1, 254, 1)])
def test_grids_whose_last_tile_is_narrower_than_the_overlap(width, height, tile, overlap, subsampling):
    """extent = k tile + 1 (or + 2) with overlap >= 2: the second-to-last tile reaches the extent and is
    smaller than the middle ones, on both axes."""
    rng = np.random.default_rng(width + height)
    img = rng.integers(0, 256, (height, width, 3), dtype=np.uint8)
    img[::3] //= 4
    d = torch.from_numpy(img).to(DEV)
    check_level(img, J.encode_tiles(d, tile, overlap, 70, subsampling), tile, overlap, 70, subsampling)
    rows = J.tile_grid(width, height, tile)[1]
    if rows > 2:
        check_level(img, J.encode_tiles(d, tile, overlap, 70, subsampling, rows=(rows - 2, 2)), tile, overlap, 70,
                    subsampling, (rows - 2, 2))

def test_saturated_grid_against_single_tile_launches():
    """Thousands of tiles in one launch equal each tile encoded by a launch of its own."""
    rng = np.random.default_rng(3)
    img = rng.integers(0, 256, (40 * 33, 60 * 33, 3), dtype=np.uint8)
    img[:, ::7] = 255
    d = torch.from_numpy(img).to(DEV)
    for s in (0, 2):
        grid = J.encode_tiles(d, 32, 1, 80, s)
        host = grid.payload.cpu().numpy()
        assert grid.grid == (62, 42)
        for r in (0, 1, 20, 41):
            for c in (0, 1, 30, 61):
                x0, y0, x1, y1 = J.tile_rect(c, r, d.shape[1], d.shape[0], 32, 1)
                one = J.encode_tiles(d[y0:y1, x0:x1], max(y1 - y0, x1 - x0), 0, 80, s)
                assert grid.tile_bytes(c, r, host) == one.tile_bytes(0, 0), (s, c, r)


def test_subrectangle_with_unaligned_pitch_and_sentinels():
    rng = np.random.default_rng(5)
    big = torch.from_numpy(rng.integers(0, 256, (300, 419, 3), dtype=np.uint8)).to(DEV)
    view = big[13:290, 7:400]                                    # pitch 1257 bytes, offset not aligned
    assert view.stride() == (419 * 3, 3, 1)
    img = view.cpu().numpy()
    for s in (0, 2):
        check_level(img, J.encode_tiles(view, 100, 2, 85, s), 100, 2, 85, s)
    # the raw call writes nothing outside offsets and the files
    hdr = J.level_headers(393, 277, 100, 2, 85, 2)
    n_hdr = len(hdr) // 16
    lib = L.load()
    args = (277, 393, 100, 2, 0, 3, 2, n_hdr)
    worst = lib.vqae_jpeg_tiles_worst_bytes(*args)
    pad = 4096
    payload = torch.full((worst + 2 * pad,), 0xA5, dtype=torch.uint8, device=DEV)
    offsets = torch.full((3 * 4 + 1 + 2,), -7, dtype=torch.int64, device=DEV)
    ws = torch.empty(lib.vqae_jpeg_tiles_scratch_bytes(*args), dtype=torch.uint8, device=DEV)
    qt = J.quant_tables(85)
    hb = np.frombuffer(hdr, np.uint8)
    L.check(lib.vqae_jpeg_tiles(view.data_ptr(), view.stride(0), 277, 393, 100, 2, 0, 3, 85, 2, hb.ctypes.data,
                                n_hdr, qt.ctypes.data, offsets[1:].data_ptr(), payload[pad:].data_ptr(), worst,
                                ws.data_ptr(), ws.numel(), E._stream(torch.device(DEV))), "vqae_jpeg_tiles")
    off = offsets.cpu().numpy()
    assert off[0] == -7 and off[-1] == -7 and off[1] == 0
    total = int(off[-2])
    p = payload.cpu().numpy()
    assert (p[:pad] == 0xA5).all() and (p[pad + total:] == 0xA5).all()
    ref = J.encode_tiles(view, 100, 2, 85, 2)
    assert np.array_equal(off[1:-1], ref.offsets) and np.array_equal(p[pad:pad + total], ref.payload.cpu().numpy())


def test_q100_noise_stays_within_worst_case():
    rng = np.random.default_rng(11)
    img = rng.integers(0, 256, (1000, 1300, 3), dtype=np.uint8)
    d = torch.from_numpy(img).to(DEV)
    lib = L.load()
    n_hdr = len(J.jpeg_header(1, 1, 100, 0))
    for s in (0, 2):
        tiles = J.encode_tiles(d, 254, 1, 100, s)
        check_level(img, tiles, 254, 1, 100, s)
        host = tiles.payload.cpu().numpy()
        assert tiles.nbytes() < lib.vqae_jpeg_tiles_worst_bytes(1000, 1300, 254, 1, 0, 4, s, n_hdr)
        stuffed = sum(tiles.tile_bytes(c, r, host).count(b"\xff\x00") for r in range(4) for c in range(6))
        assert stuffed > 10000


def test_canvas_over_2_31_bytes():
    h, w = 26000, 28000                                          # 2.18e9 bytes
    big = torch.zeros(h, w, 3, dtype=torch.uint8, device=DEV)
    rng = np.random.default_rng(2)
    patch = rng.integers(0, 256, (300, 500, 3), dtype=np.uint8)
    big[h - 300:, w - 500:] = torch.from_numpy(patch).to(DEV)
    rows = J.tile_grid(w, h, 254)[1]
    tiles = J.encode_tiles(big, 254, 1, 90, 2, rows=(rows - 2, 2))
    img = big[h - 600:].cpu().numpy()
    host = tiles.payload.cpu().numpy()
    cols = tiles.grid[0]
    for r in (rows - 2, rows - 1):
        for c in (0, cols - 2, cols - 1):
            x0, y0, x1, y1 = J.tile_rect(c, r, w, h, 254, 1)
            want = pil_jpeg(np.ascontiguousarray(img[y0 - (h - 600):y1 - (h - 600), x0:x1]), 90, 2)
            assert tiles.tile_bytes(c, r, host) == want, (c, r)
    del big


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_export_deepzoom(tmp_path, precision):
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = vqae_b200.set_precision(m.to(DEV), precision)
    try:
        cm = torch.from_numpy(np.random.default_rng(6).integers(0, 256, (2 * 32, 3 * 32)).astype(np.uint8)).to(DEV)
        info = export_deepzoom(m, cm, (32, 32), tmp_path, "slide", tile=254, overlap=1, quality=80, batch=4)
        full = decompress_region(m, cm, (32, 32), batch=4)
        levels = slide_pyramid(full, (256, 256), [2 ** k for k in range(1, 9)])
        levels[1] = full
        root = ET.parse(info["dzi"]).getroot()
        size = root[0].attrib
        assert (int(size["Width"]), int(size["Height"])) == (768, 512)
        assert root.attrib["TileSize"] == "254" and root.attrib["Overlap"] == "1" and root.attrib["Format"] == "jpeg"
        dims = J.dz_levels(768, 512)
        assert info["levels"] == len(dims) == 11
        m_top = len(dims) - 1
        finer = None
        n = 0
        for lv in range(m_top, -1, -1):
            f = 1 << (m_top - lv)
            img = levels[f].cpu().numpy() if f in levels else np.asarray(Image.fromarray(finer).reduce(2))
            finer = img
            w_l, h_l = dims[lv]
            assert img.shape == (h_l, w_l, 3)
            cols, rows = J.tile_grid(w_l, h_l, 254)
            files = sorted(p.name for p in (tmp_path / "slide_files" / str(lv)).iterdir())
            assert files == sorted(f"{c}_{r}.jpeg" for c in range(cols) for r in range(rows))
            for r in range(rows):
                for c in range(cols):
                    x0, y0, x1, y1 = J.tile_rect(c, r, w_l, h_l, 254, 1)
                    data = (tmp_path / "slide_files" / str(lv) / f"{c}_{r}.jpeg").read_bytes()
                    assert data == pil_jpeg(np.ascontiguousarray(img[y0:y1, x0:x1]), 80, 2), (lv, c, r)
                    assert Image.open(io.BytesIO(data)).size == (x1 - x0, y1 - y0)
                    n += 1
        assert info["tiles"] == n
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()


def test_errors(tmp_path):
    d = torch.zeros(64, 64, 3, dtype=torch.uint8, device=DEV)
    with pytest.raises(RuntimeError):
        J.encode_tiles(d.cpu())
    with pytest.raises(ValueError):
        J.encode_tiles(d.float())
    with pytest.raises(ValueError):
        J.encode_tiles(d.transpose(0, 1))                         # pixels not packed
    with pytest.raises(ValueError):
        J.encode_tiles(d[:, :, :2])
    for kw in (dict(quality=0), dict(quality=101), dict(subsampling=1), dict(tile=0), dict(overlap=-1),
               dict(overlap=64), dict(tile=8, overlap=16), dict(rows=(0, 2)), dict(rows=(-1, 1))):
        with pytest.raises(ValueError):
            J.encode_tiles(d, **{"tile": 64, **kw})
    with pytest.raises(ValueError):                              # a 65536-row tile
        J.encode_tiles(torch.zeros(70000, 1, 3, dtype=torch.uint8, device=DEV), tile=65535, overlap=1)
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    try:
        cm = torch.zeros(64, 96, dtype=torch.uint8, device=DEV)
        with pytest.raises(ValueError):
            export_deepzoom(m, cm, (32, 30), tmp_path, "x")        # not a grid of code tiles
        with pytest.raises(ValueError):
            export_deepzoom(m, cm, (32, 32), tmp_path, "x", quality=0)
        with pytest.raises(ValueError):
            export_deepzoom(m, cm, (32, 32), tmp_path, "a/b")
        with pytest.raises(RuntimeError):
            export_deepzoom(m, cm.cpu(), (32, 32), tmp_path, "x")
        assert not any(tmp_path.iterdir())
    finally:
        m.cpu()
    mm, _, _ = H.multilevel_model_and_state("flat")
    with pytest.raises(NotImplementedError):
        export_deepzoom(mm.to(DEV), torch.zeros(64, 64, dtype=torch.uint8, device=DEV), (32, 32), tmp_path, "x")
    mm.cpu()
