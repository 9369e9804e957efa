"""GPU: per-patch SSE / SSIM of uint8 RGB patches (csrc/quality.cu, vqae_b200.quality,
extract.compress_slide_scored / score_region) against torch int64 and the float64 oracle of
tests/quality_oracle.py."""
import ctypes as C

import numpy as np
import pytest
import torch

import decompress_oracle as D
import helpers as H
import quality_oracle as Q
import vqae_b200
from vqae_b200 import _lib as L
from vqae_b200 import engine as E
from vqae_b200 import synthetic as S
from vqae_b200.extract import compress_slide, compress_slide_scored, encode_patches, score_region
from vqae_b200.quality import reconstruction_quality

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _noisy(ref, amp, seed):
    g = torch.Generator().manual_seed(seed)
    d = torch.randint(-amp, amp + 1, ref.shape, generator=g)
    return (ref.long() + d).clamp(0, 255).to(torch.uint8)


def _rand_u8(shape, seed):
    return torch.randint(0, 256, shape, generator=torch.Generator().manual_seed(seed), dtype=torch.uint8)


def _sse_torch(ref, rec):
    d = ref.long() - rec.long()
    return (d * d).sum((1, 2))


@pytest.mark.parametrize("hw", [(256, 256), (512, 512), (200, 328), (11, 11)])
def test_sse_exact_batch_and_canvas(hw):
    h, w = hw
    ref = _rand_u8((5, h, w, 3), h + w)
    rec = _noisy(ref, 40, 7)
    q = reconstruction_quality(ref.to(DEV), rec.to(DEV))
    assert q.sse.dtype == torch.int64 and q.ssim.dtype == torch.float64
    assert torch.equal(q.sse.cpu(), _sse_torch(ref, rec))
    # the same patches read out of canvases: ref as region patches 1 .. 5 of a region at grid (1, 1) with
    # 3 patches per row inside a 4 x 5 grid whose rows carry 5 extra pixels (rows are not 16-byte
    # multiples), rec from a plain canvas of its own with 2 patches per row
    for extra in (0, 5):
        cv = _rand_u8((4 * h, 5 * w + extra, 3), 1)
        for t in range(5):
            p = 1 + t
            r, c = 1 + p // 3, 1 + p % 3
            cv[r * h:(r + 1) * h, c * w:(c + 1) * w] = ref[t]
        rc = torch.zeros(3 * h, 2 * w, 3, dtype=torch.uint8)
        for t in range(5):
            rc[(t // 2) * h:(t // 2 + 1) * h, (t % 2) * w:(t % 2 + 1) * w] = rec[t]
        sse, ssim = E.quality_u8(cv.to(DEV), (1, 1, 3, 1), rc.to(DEV), (0, 0, 2, 0), 5, h, w)
        assert torch.equal(sse, q.sse) and torch.equal(ssim, q.ssim), extra


def _accuracy_cases():
    noise_a, noise_b = _rand_u8((2, 256, 256, 3), 21), _rand_u8((2, 256, 256, 3), 22)
    flat255 = torch.full((1, 256, 256, 3), 255, dtype=torch.uint8)
    half = torch.full((2, 256, 256, 3), 240, dtype=torch.uint8)
    half[:, :, 128:] = _rand_u8((2, 256, 128, 3), 23)            # right half textured
    half[1, :, :, :] = half[1].flip(1)                          # and the flat half on the right
    half_rec = _noisy(half, 6, 24)
    yy, xx = torch.meshgrid(torch.arange(64), torch.arange(96), indexing="ij")
    board = (((yy + xx) % 2) * 255).to(torch.uint8)[None, ..., None].expand(1, 64, 96, 3).contiguous()
    return {"noise": (noise_a, noise_b), "flat_255_254": (flat255, flat255 - 1),
            "half_flat": (half, half_rec), "checkerboard": (board, 255 - board)}


def test_ssim_accuracy():
    """|ssim - float64 oracle| <= 1e-5 per patch.  Measured maximum on an NVIDIA B200: 1.2e-13 (the moments
    are accumulated in fp64, quality.cu)."""
    cases = _accuracy_cases()
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    try:
        tiles = S.synthetic_patches_u8(3, 256, 31)
        for precision in ("fp32", "fp16"):
            vqae_b200.set_precision(m, precision)
            rec = m.decode_codes_u8(encode_patches(m.encoder, tiles.to(DEV))).cpu()
            cases["round_trip_" + precision] = (tiles, rec)
        vqae_b200.set_precision(m, None)
    finally:
        m.cpu()
    worst = 0.0
    for name, (ref, rec) in cases.items():
        q = reconstruction_quality(ref.to(DEV), rec.to(DEV))
        assert torch.equal(q.sse.cpu(), torch.from_numpy(Q.sse(ref.numpy(), rec.numpy())))
        for i in range(ref.shape[0]):
            want = Q.ssim(ref[i].numpy(), rec[i].numpy())
            err = abs(float(q.ssim[i]) - want)
            worst = max(worst, err)
            print(f"{name}[{i}]: ssim {float(q.ssim[i]):.9f} oracle {want:.9f} |d| {err:.2e}")
            assert err <= 1e-5, (name, i)
        if name == "checkerboard":
            assert float(q.ssim[0]) < 0
    print(f"max |ssim - oracle| = {worst:.3e}")


# ---- launcher mirror: quality.cu quality_u8 -- units = batch x tiles, tiles of 16 x 32 window positions
#      (QT_Y, QT_X), grid = min(units, sm_count x QT_MIN_CTAS = 3)
def _quality_units(batch, h, w):
    tiles = -(-(h - 10) // 16) * -(-(w - 10) // 32)
    return batch * tiles, 3 * torch.cuda.get_device_properties(0).multi_processor_count


@pytest.mark.parametrize("hw", [(256, 256), (200, 328)])
def test_saturated_and_ragged_launch_equals_single_patches(hw):
    h, w = hw
    batch = 17
    units, cap = _quality_units(batch, h, w)
    sm = torch.cuda.get_device_properties(0).multi_processor_count
    assert units >= 3 * 4 * sm                                  # >= 3 units per CTA even at 4 CTAs / SM
    assert units % cap != 0                                     # a partial last wave
    ref = _rand_u8((batch, h, w, 3), 5).to(DEV)
    rec = _noisy(ref.cpu(), 30, 6).to(DEV)
    q = reconstruction_quality(ref, rec)
    for i in range(batch):
        one = reconstruction_quality(ref[i:i + 1], rec[i:i + 1])
        assert torch.equal(one.sse[0], q.sse[i]) and torch.equal(one.ssim[0], q.ssim[i]), i
    for s in range(0, batch, 4):
        part = reconstruction_quality(ref[s:s + 4], rec[s:s + 4])
        assert torch.equal(part.sse, q.sse[s:s + 4]) and torch.equal(part.ssim, q.ssim[s:s + 4]), s
    again = reconstruction_quality(ref, rec)                    # determinism: a second launch, once
    assert torch.equal(again.sse, q.sse) and torch.equal(again.ssim, q.ssim)


def test_abi_rejects_bad_placements_before_launching():
    lib = L.load()
    a = torch.zeros(128, 128, 3, dtype=torch.uint8, device=DEV)
    b = torch.zeros(128, 128, 3, dtype=torch.uint8, device=DEV)
    sse = torch.empty(2, 3, dtype=torch.int64, device=DEV)
    ssim = torch.empty(2, dtype=torch.float64, device=DEV)
    ws = E.workspace(a.device, lib.vqae_quality_u8_scratch_bytes(2, 64, 64))
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = E._ptr

    def call(ar0=0, ac0=0, arc=2, afirst=0, br0=0, bc0=0, brc=2, bfirst=0, rows=128, batch=2):
        return lib.vqae_quality_u8(p(a), rows, 128, ar0, ac0, arc, afirst, p(b), 128, 128, br0, bc0, brc,
                                   bfirst, batch, 64, 64, p(sse), p(ssim), p(ws), ws.numel(), st)
    n0 = E.launch_count()
    assert call(afirst=3) == L.ERR_BAD_ARG                      # patches 3, 4: row 2 of a 2-row canvas
    assert call(bfirst=3) == L.ERR_BAD_ARG
    assert call(arc=3) == L.ERR_BAD_ARG                         # 3 columns of 64 on 128
    assert call(bc0=1) == L.ERR_BAD_ARG
    assert call(br0=2) == L.ERR_BAD_ARG
    assert call(ar0=1, afirst=2) == L.ERR_BAD_ARG
    assert call(rows=127, afirst=2) == L.ERR_BAD_ARG
    torch.cuda.synchronize()
    assert E.launch_count() == n0
    assert call() == L.OK and E.launch_count() == n0 + 2


def _stitch(tiles, nc):
    return torch.from_numpy(D.stitch(tiles.numpy(), nc))


@pytest.mark.parametrize("precision", ["fp32", "fp16"])
def test_scored_compression_and_region_scores(precision):
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = vqae_b200.set_precision(m.to(DEV), precision)
    try:
        grid, th = (3, 5), 32
        tiles = S.synthetic_patches_u8(15, 256, 8)
        batches = [(0, tiles[:4]), (4, tiles[4:8]), (8, tiles[8:12]), (12, tiles[12:])]   # last one short
        cmap = compress_slide(m.encoder, batches, grid, (th, th), torch.device(DEV))
        cmap2, q = compress_slide_scored(m, batches, grid, (th, th), torch.device(DEV))
        assert torch.equal(cmap, cmap2)
        assert q.sse.shape == (3, 5, 3) and q.ssim.shape == (3, 5) and q.patch_hw == (256, 256)
        for first, t in batches:
            codes = torch.stack([cmap[(i // 5) * th:(i // 5 + 1) * th, (i % 5) * th:(i % 5 + 1) * th]
                                 for i in range(first, first + len(t))]).long()
            want = reconstruction_quality(t.to(DEV), m.decode_codes_u8(codes))
            assert torch.equal(q.sse.view(15, 3)[first:first + len(t)], want.sse)
            assert torch.equal(q.ssim.view(15)[first:first + len(t)], want.ssim)
        slide = _stitch(tiles, 5).to(DEV)
        whole = score_region(m, cmap, (th, th), slide, batch=4)
        assert torch.equal(whole.sse, q.sse) and torch.equal(whole.ssim, q.ssim)
        part = score_region(m, cmap, (th, th), slide, region=(1, 1, 2, 3), batch=4)
        assert torch.equal(part.sse, q.sse[1:3, 1:4]) and torch.equal(part.ssim, q.ssim[1:3, 1:4])
        assert 0 < float(q.ssim.min()) and float(q.ssim.max()) < 1
        s = q.summary()
        assert s["patches"] == 15 and s["psnr_pooled"] > 0
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()


def test_errors():
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    try:
        tiles = S.synthetic_patches_u8(2, 256, 3)
        with pytest.raises(ValueError):
            compress_slide_scored(m, [(0, tiles.permute(0, 3, 1, 2).float() / 255)], (1, 2), (32, 32),
                                  torch.device(DEV))
        cmap = torch.zeros(32, 64, dtype=torch.uint8, device=DEV)
        slide = torch.zeros(256, 512, 3, dtype=torch.uint8, device=DEV)
        with pytest.raises(ValueError):
            score_region(m, cmap, (32, 32), slide[:, :256])
        with pytest.raises(ValueError):
            score_region(m, cmap, (32, 32), slide, region=(0, 1, 1, 2))
        a = tiles.to(DEV)
        small = a[:, :10, :10].contiguous()
        for ref, rec in ((a, a[:1]), (a, a.float()), (a, a.cpu()), (small, small), (a, a.transpose(1, 2))):
            with pytest.raises(ValueError):
                reconstruction_quality(ref, rec)
    finally:
        m.cpu()
    two, _, _ = H.multilevel_model_and_state("flat")
    with pytest.raises(NotImplementedError):
        score_region(two, torch.zeros(32, 32, dtype=torch.int64, device=DEV), (32, 32),
                     torch.zeros(256, 256, 3, dtype=torch.uint8, device=DEV))
    with pytest.raises(NotImplementedError):
        compress_slide_scored(two, [], (1, 1), (32, 32), torch.device(DEV))
