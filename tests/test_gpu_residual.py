"""GPU: near-lossless residual layers (csrc/residual.cu, engine.residual_*, vqae_b200.residual,
extract.encode_residual / decompress_region_exact) against the numpy oracle of tests/residual_oracle.py, byte
for byte, and exact round trips with torch.equal."""
import numpy as np
import pytest
import torch

import helpers as H
import residual_oracle as RO
import vqae_b200
from vqae_b200 import engine as E
from vqae_b200.extract import decompress_region, decompress_region_exact, encode_residual
from vqae_b200.packing import quantise_frequencies
from vqae_b200.residual import ResidualIntegrityError, ResidualLayer, load_residual, save_residual

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _laplace_slide(base: torch.Tensor, scale: float, seed: int) -> torch.Tensor:
    rng = np.random.default_rng(seed)
    b = base.cpu().numpy().astype(np.int64)
    return torch.from_numpy(np.clip(b + rng.laplace(0, scale, b.shape).round().astype(np.int64), 0, 255)
                            .astype(np.uint8)).to(base.device)


@pytest.fixture(scope="module")
def model():
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    yield m
    vqae_b200.set_precision(m, None)
    m.cpu()


def _check_layer(layer, slide, base, hw, e):
    h, w = hw
    off, payload, adler, want = RO.layer(slide.cpu().numpy(), base.cpu().numpy(), h, w, e)
    assert np.array_equal(layer.offsets_host, off) and np.array_equal(layer.offsets.cpu().numpy(), off)
    assert layer.payload.cpu().numpy().tobytes() == payload
    assert np.array_equal(layer.adler.cpu().numpy().view(np.uint32), adler)
    return want


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
@pytest.mark.parametrize("e", [0, 1, 4])
def test_layer_equals_oracle_and_round_trips(model, precision, e):
    vqae_b200.set_precision(model, precision)
    cm = torch.from_numpy(np.random.default_rng(5).integers(0, 256, (2 * 32, 3 * 32)).astype(np.uint8)).to(DEV)
    base = decompress_region(model, cm, (32, 32), batch=4)
    slide = _laplace_slide(base, 3.0, 10 + e)
    layer = encode_residual(model, cm, (32, 32), slide, max_error=e, batch=4)              # 6 = 4 + 2
    assert layer.precision == precision and layer.max_error == e and layer.grid == (2, 3)
    want = torch.from_numpy(_check_layer(layer, slide, base, (256, 256), e)).to(DEV)
    assert torch.equal(encode_residual(model, cm, (32, 32), slide, max_error=e, batch=256).payload, layer.payload)
    if e == 0:
        assert torch.equal(want, slide)
    assert int((want.int() - slide.int()).abs().max()) <= e
    for region, batch in ((None, 1), (None, 3), (None, 256), ((1, 1, 1, 2), 1), ((0, 1, 2, 2), 3)):
        got = decompress_region_exact(model, cm, (32, 32), layer, region, batch)
        r0, c0, nr, nc = region or (0, 0, 2, 3)
        assert torch.equal(got, want[r0 * 256:(r0 + nr) * 256, c0 * 256:(c0 + nc) * 256]), (region, batch)
    out = torch.empty(512, 512, 3, dtype=torch.uint8, device=DEV)
    got = decompress_region_exact(model, cm, (32, 32), layer, (0, 1, 2, 2), 3, out=out)
    assert got.data_ptr() == out.data_ptr() and torch.equal(out, want[:, 256:])


def test_non_square_patches(model):
    vqae_b200.set_precision(model, "fp32")
    cm = torch.from_numpy(np.random.default_rng(8).integers(0, 256, (2 * 16, 2 * 32)).astype(np.uint8)).to(DEV)
    base = decompress_region(model, cm, (16, 32), batch=3)
    assert tuple(base.shape) == (256, 512, 3)
    for e in (0, 2):
        slide = _laplace_slide(base, 5.0, 20 + e)
        layer = encode_residual(model, cm, (16, 32), slide, max_error=e, batch=3)        # 4 = 3 + 1
        assert layer.patch_hw == (128, 256)
        want = torch.from_numpy(_check_layer(layer, slide, base, (128, 256), e)).to(DEV)
        assert torch.equal(decompress_region_exact(model, cm, (16, 32), layer, batch=3), want)


def _engine_layer(x, xaddr, base, baddr, n, h, w, e):
    hist, adler = E.residual_stats(x, xaddr, base, baddr, n, h, w, e)
    freq = E.residual_tables(hist)
    off, payload = E.residual_encode(x, xaddr, base, baddr, n, h, w, e, freq)
    off = off.cpu().numpy()
    return hist, freq, adler, off, payload[:int(off[-1])]


def test_saturated_launches_equal_single_patch_launches():
    """3600 patches of 16 x 16: more than the capped grids of every kernel hold, so their CTAs loop."""
    h = w = 16
    rows = cols = 60
    n = rows * cols
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    assert n > 8 * sm * 2 and n > 8 * sm
    g = torch.Generator().manual_seed(3)
    base = torch.randint(0, 256, (rows * h, cols * w, 3), generator=g, dtype=torch.uint8)
    noise = torch.from_numpy(np.random.default_rng(4).laplace(0, 2, tuple(base.shape)).round().astype(np.int64))
    x = (base.long() + noise).clamp(0, 255).to(torch.uint8)
    xd, bd = x.to(DEV), base.to(DEV)
    for e in (0, 3):
        hist, freq, adler, off, payload = _engine_layer(xd, (0, 0, cols, 0), bd, (0, 0, cols, 0), n, h, w, e)
        hn, fn = hist.cpu().numpy(), freq.cpu().numpy()
        for p in range(n):
            assert np.array_equal(fn[p], quantise_frequencies(hn[p])), p
        sym = RO.symbols(RO.patches(x.numpy(), h, w), RO.patches(base.numpy(), h, w), e)
        assert np.array_equal(hn, np.stack([np.bincount(s, minlength=256) for s in sym]))
        ro, rp, ra, want = RO.layer(x.numpy(), base.numpy(), h, w, e)
        assert np.array_equal(off, ro) and payload.cpu().numpy().tobytes() == rp
        assert np.array_equal(adler.cpu().numpy().view(np.uint32), ra)
        for p in (0, 1, 1234, n - 1):                                      # single-patch launches
            _, _, a1, o1, p1 = _engine_layer(xd, (0, 0, cols, p), bd, (0, 0, cols, p), 1, h, w, e)
            assert torch.equal(p1, payload[off[p]:off[p + 1]]) and torch.equal(a1[0], adler[p])
        canvas = bd.clone()
        flags = torch.empty(n, dtype=torch.uint8, device=DEV)
        E.residual_apply(payload, torch.from_numpy(off).to(DEV), off, adler, (rows, cols), (0, 0, cols, 0), canvas,
                         (0, 0, cols, 0), n, h, w, e, flags)
        assert int(flags.max()) == 0 and torch.equal(canvas.cpu(), torch.from_numpy(want))
        one = bd.clone()
        for p in (7, n - 2):
            E.residual_apply(payload, torch.from_numpy(off).to(DEV), off, adler, (rows, cols), (0, 0, cols, p), one,
                             (0, 0, cols, p), 1, h, w, e, flags[:1])
            assert int(flags[0]) == 0
            r, c = divmod(p, cols)
            assert torch.equal(one[r * h:(r + 1) * h, c * w:(c + 1) * w], canvas[r * h:(r + 1) * h, c * w:(c + 1) * w])


def test_all_zero_and_uniform_residuals():
    h, w = 64, 96
    g = torch.Generator().manual_seed(9)
    base = torch.randint(0, 256, (2 * h, 3 * w, 3), generator=g, dtype=torch.uint8)
    for x, e in ((base.clone(), 0), (torch.randint(0, 256, base.shape, generator=g, dtype=torch.uint8), 0),
                 (torch.randint(0, 256, base.shape, generator=g, dtype=torch.uint8), 5)):
        xd, bd = x.to(DEV), base.to(DEV)
        _, _, adler, off, payload = _engine_layer(xd, (0, 0, 3, 0), bd, (0, 0, 3, 0), 6, h, w, e)
        ro, rp, ra, want = RO.layer(x.numpy(), base.numpy(), h, w, e)
        assert np.array_equal(off, ro) and payload.cpu().numpy().tobytes() == rp
        if torch.equal(x, base):
            assert np.array_equal(np.diff(off), [768] * 6)
        flags = torch.empty(6, dtype=torch.uint8, device=DEV)
        E.residual_apply(payload, torch.from_numpy(off).to(DEV), off, adler, (2, 3), (0, 0, 3, 0), bd,
                         (0, 0, 3, 0), 6, h, w, e, flags)
        assert int(flags.max()) == 0 and torch.equal(bd.cpu(), torch.from_numpy(want))
        if e == 0:
            assert torch.equal(bd.cpu(), x)


def test_slide_canvas_beyond_2_31_bytes():
    h = w = 256
    grid_rows, grid_cols = 1000, 12
    canvas = torch.zeros(grid_rows * h, grid_cols * w, 3, dtype=torch.uint8, device=DEV)
    assert canvas.numel() > 2 ** 31
    g = torch.Generator().manual_seed(77)
    x = torch.randint(0, 256, (h, 4 * w, 3), generator=g, dtype=torch.uint8)
    base = torch.randint(0, 256, (h, 4 * w, 3), generator=g, dtype=torch.uint8)
    r = grid_rows - 1
    canvas[r * h:, 8 * w:] = x.to(DEV)
    bd = base.to(DEV)
    _, _, adler, off, payload = _engine_layer(canvas, (r, 8, 4, 0), bd, (0, 0, 4, 0), 4, h, w, 0)
    ro, rp, ra, _ = RO.layer(x.numpy(), base.numpy(), h, w, 0)
    assert np.array_equal(off, ro) and payload.cpu().numpy().tobytes() == rp
    canvas[r * h:, 8 * w:] = bd                                                # the base, in place
    flags = torch.empty(4, dtype=torch.uint8, device=DEV)
    E.residual_apply(payload, torch.from_numpy(off).to(DEV), off, adler, (1, 4), (0, 0, 4, 0), canvas, (r, 8, 4, 0),
                     4, h, w, 0, flags)
    assert int(flags.max()) == 0 and torch.equal(canvas[r * h:, 8 * w:].cpu(), x)
    assert int(canvas[:r * h].max()) == 0 and int(canvas[r * h:, :8 * w].max()) == 0
    del canvas


def test_failure_modes_and_save_load(model, tmp_path):
    vqae_b200.set_precision(model, "fp32")
    cm = torch.from_numpy(np.random.default_rng(12).integers(0, 256, (2 * 32, 3 * 32)).astype(np.uint8)).to(DEV)
    base = decompress_region(model, cm, (32, 32), batch=4)
    slide = _laplace_slide(base, 4.0, 13)
    layer = encode_residual(model, cm, (32, 32), slide, max_error=0, batch=4)

    path = save_residual(tmp_path / "slide.vqrl", layer)
    again = load_residual(path, DEV)
    assert again.to_bytes() == layer.to_bytes() and again.precision == "fp32"
    assert torch.equal(decompress_region_exact(model, cm, (32, 32), again), slide)
    assert layer.bits_per_pixel() == pytest.approx(8 * path.stat().st_size / (6 * 256 * 256))

    vqae_b200.set_precision(model, "fp16")                                      # mode mismatch: no launch
    n0 = E.launch_count()
    with pytest.raises(ValueError, match="fp32"):
        decompress_region_exact(model, cm, (32, 32), layer)
    with pytest.raises(ValueError):
        decompress_region_exact(model, cm[:32], (32, 32), layer)               # another grid
    assert E.launch_count() == n0
    vqae_b200.set_precision(model, "fp32")

    changed = cm.clone()                                                        # one code of patch (1, 2)
    changed[32 + 5, 64 + 7] = (int(changed[32 + 5, 64 + 7]) + 1) % 256
    with pytest.raises(ResidualIntegrityError) as ei:
        decompress_region_exact(model, changed, (32, 32), layer, batch=4)
    err = ei.value
    assert err.patches == [(1, 2)] and "base mismatch" in err.causes[0] and "stream" not in err.causes[0]
    keep = torch.ones(2, 3, dtype=torch.bool)
    keep[1, 2] = False
    for r in range(2):
        for c in range(3):
            if keep[r, c]:
                assert torch.equal(err.pixels[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256],
                                   slide[r * 256:(r + 1) * 256, c * 256:(c + 1) * 256])

    damaged = ResidualLayer(payload=layer.payload.clone(), offsets=layer.offsets, adler=layer.adler,
                            max_error=0, precision="fp32", grid=layer.grid, patch_hw=layer.patch_hw,
                            offsets_host=layer.offsets_host)
    a, b = (int(v) for v in layer.offsets_host[3:5])                            # patch (1, 0)
    damaged.payload[a + 900:b - 50] ^= 0x5a                                     # words, CRC not involved
    damaged.payload[a + 600] ^= 0xff                                            # a lane's word count
    with pytest.raises(ResidualIntegrityError) as ei:
        decompress_region_exact(model, cm, (32, 32), damaged, batch=4)
    err = ei.value
    assert err.patches == [(1, 0)] and "stream" in err.causes[0]
    assert torch.equal(err.pixels[:256], slide[:256]) and torch.equal(err.pixels[256:, 256:], slide[256:, 256:])
    damaged.payload[a:a + 512] = 0                                              # a table that sums to 0
    with pytest.raises(ResidualIntegrityError) as ei:
        decompress_region_exact(model, cm, (32, 32), damaged, region=(1, 0, 1, 2), batch=1)
    assert ei.value.patches == [(1, 0)]
    torch.cuda.synchronize()


def test_rate_against_empirical_entropy(model):
    vqae_b200.set_precision(model, "fp32")
    cm = torch.from_numpy(np.random.default_rng(31).integers(0, 256, (2 * 32, 2 * 32)).astype(np.uint8)).to(DEV)
    base = decompress_region(model, cm, (32, 32))
    slide = _laplace_slide(base, 3.0, 32)
    for e in (0, 2):
        layer = encode_residual(model, cm, (32, 32), slide, max_error=e)
        sym = RO.symbols(RO.patches(slide.cpu().numpy(), 256, 256), RO.patches(base.cpu().numpy(), 256, 256), e)
        bound = 1.01 * RO.entropy_bytes(sym) + 768 * 4
        print(f"e = {e}: payload {layer.payload_bytes} B, entropy + 768 B per chunk {bound / 1.01:.0f} B")
        assert layer.payload_bytes <= bound


def test_argument_errors(model):
    vqae_b200.set_precision(model, "fp32")
    cm = torch.zeros(32, 64, dtype=torch.uint8, device=DEV)
    slide = torch.zeros(256, 512, 3, dtype=torch.uint8, device=DEV)
    for bad in (-1, 128, 0.5):
        with pytest.raises(ValueError):
            encode_residual(model, cm, (32, 32), slide, max_error=bad)
    with pytest.raises(ValueError):
        encode_residual(model, cm, (32, 32), slide[:128])
    with pytest.raises(ValueError):
        encode_residual(model, cm, (32, 32), slide.transpose(0, 1))
    layer = encode_residual(model, cm, (32, 32), slide)
    with pytest.raises(ValueError):
        decompress_region_exact(model, cm, (32, 32), layer, out=torch.empty(256, 256, 3, dtype=torch.uint8,
                                                                            device=DEV))
    with pytest.raises(ValueError):
        decompress_region_exact(model, cm, (32, 32), layer, region=(0, 1, 1, 2))
    assert torch.equal(decompress_region_exact(model, cm, (32, 32), layer), slide)
