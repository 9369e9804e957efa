"""GPU: the persistent kernels with their CTAs (or warps) looping over several work units.

Every hot kernel caps its grid at ``sm_count x MIN_CTAS`` and walks ``tile += gridDim.x``; prefetch
buffers, mbarrier phases, weight rings and reused accumulators only matter from a CTA's second unit on.
For each kernel:

* a saturated launch (>= 3 units per CTA or per warp, also if the cap were 4 CTAs per SM, unless the
  kernel's shared memory holds one CTA per SM) and a *ragged* one (the last wave partial) are compared
  image by image, bit for bit, with the same kernel run over chunks small enough for one unit per CTA;
* three images of every saturated run (first, middle, last: the last runs in the partial final wave)
  are held to the float64 reference of tests/f64_bound.py with its per-element error bound, derived
  from the points where the kernel rounds its operands (for the fp16 kernels the reference rounds at
  those points itself, so the bound only covers accumulation order and fp32 elementwise steps);
* the profiler's kernel names confirm which kernel ran (a launch count of 1 would also fit the fp32
  fallback).

The fp32 CUDA-core kernels, which every other test uses as the reference, get the same bound with
operand rounding u = 0 at non-square shapes.  Then the model at the benched shapes, and the decode-side
code-map gather past the 65 535 limit of gridDim.y.
"""
import pytest
import torch

import f64_bound as FB
import helpers as H
import vqae_b200
from vqae_b200 import _lib as L
from vqae_b200 import engine as E
from vqae_b200 import synthetic as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SMEM_PER_CTA_MAX = 227 * 1024


def _sm() -> int:
    return torch.cuda.get_device_properties(0).multi_processor_count


# ---- launcher mirrors: (work units, units of one image, cap in units processed at once, fits 4/SM) ------
# A "slot" is a CTA, or a warp for the m-tile kernels; ``cap`` is the number of slots the launcher starts
# at most.  ``one_per_sm``: the kernel's shared memory leaves room for one CTA per SM only.
def _ms_min_ctas(c, th):
    """MsCfg<C, TH>::MIN_CTAS (mma_same.cu:49-73)."""
    k8 = c == 8
    npad = (th + 2) * 34
    mt1 = (npad + 15) // 16
    up = 16 if k8 else c * 2 + 16
    nxb = 1 if c == 32 else 2
    smem = nxb * mt1 * 16 * c * 4 + mt1 * 16 * up + (0 if k8 else 9 * c * (c * 2 + 16)) + 16
    fit = SMEM_PER_CTA_MAX // (smem + 1024)
    return 4 if fit >= 4 else max(fit, 1)


def units_stem_in(h, w):
    """mma_stem.cu:556-570: 16 x 32 pixel tiles, grid <= 4 sm."""
    return (h // 16) * (w // 32), 4 * _sm(), False


def units_same(c, h, w):
    """mma_same.cu:407-415 and 437-440: 32-pixel-wide tiles of TH rows, grid <= MIN_CTAS sm."""
    th = 16 if c == 8 and h % 16 == 0 else 8
    return (h // th) * (w // 32), _ms_min_ctas(c, th) * _sm(), False


def units_down(c, h, w, split=False):
    """mma_down.cu:330-339: m-tiles of 16 output pixels, 8 warps per CTA, grid <= MIN_CTAS sm
    (SPLIT: md_split_ctas, mma_down.cu:80-82)."""
    ctas = ({8: 2, 16: 1, 32: 1} if split else {8: 4, 16: 2, 32: 1})[c]
    return (h // 2) * (w // 2 // 16), 8 * ctas * _sm(), False


def units_up(c, h, w):
    """mma_up.cu:433-435 (head: m-tiles of 16 low-res pixels, 8 warps per CTA, UhCfg MIN_CTAS) and
    448-456, 500-505 (tail: 32-pixel-wide tiles of TY output rows, U3Cfg MIN_CTAS).  Two kernels:
    returns both."""
    head = ((h * w) // 16, 8 * (2 if c <= 32 else 1) * _sm(), False)
    ty = 16 if c <= 32 and (2 * h) % 16 == 0 else 8
    tail = ((2 * h // ty) * (2 * w // 32), (3 if c <= 32 else (2 if c == 64 else 1)) * _sm(), False)
    return head, tail


def units_down128(h, w):
    """tc_down128.cu:317-330: 8 x 16 output tiles, grid <= sm (DW_SMEM ~226 KB: one CTA per SM)."""
    return (h // 2 // 8) * (w // 2 // 16), _sm(), True


def units_split_same(c, h, w):
    """mma_same_split.cu:356-365 (C = 8, 16: TH = 8, MIN_CTAS 2) and tc_split.cu:415-416, 440
    (C = 32, 64: 8 x 32 tiles, MIN_CTAS 2 / 1; C = 64 needs ~194 KB of shared memory)."""
    if c in E.SPLIT_MMA:
        return (h // 8) * (w // 32), 2 * _sm(), False
    return (h // 8) * (w // 32), {32: 2, 64: 1}[c] * _sm(), c == 64


def _assert_saturated(units_img, cap, one_per_sm, batch, slot):
    units = units_img * batch
    grid = min(units, cap)
    per = units / grid
    assert per >= 3, (units, grid)
    if not one_per_sm:
        four = 4 * _sm() * (8 if slot == "warp" else 1)
        assert units >= 3 * four, (units, four)
    return units, grid


def _ragged_batch(kernels, start):
    """The largest batch <= start that leaves every kernel of the launch (head and tail for 'up') a
    partial last wave of 1 .. grid/4 units and still >= 3 per slot."""
    for b in range(start, 0, -1):
        if all(u * b >= 3 * cap and 1 <= (u * b) % cap <= cap // 4 for u, cap, *_ in kernels):
            return b
    raise AssertionError("no ragged batch")


def _run_profiled(fn, x):
    """fn(x) under torch.profiler: (result, names of the CUDA kernels that ran, spaces removed)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        y = fn(x)
        torch.cuda.synchronize()
    return y, {e.key.replace(" ", "") for e in prof.key_averages()}


def _assert_ran(names, expected):
    for k in expected:
        assert any(k.replace(" ", "") in n for n in names), (k, sorted(names))


def _chunk(units_img, cap):
    return max(1, cap // units_img)


# ---- blocks -----------------------------------------------------------------------------------------------
def _block(mode, c_in, seed):
    from vqae_b200.config import pre_activation_fixup
    from vqae_b200.layers.conv_block import PreActFixupResBlock
    c_out = {"same": c_in, "down": 2 * c_in, "up": c_in // 2}[mode]
    conf = pre_activation_fixup(n_layers=12)
    for k in ("_target_", "_recursive_", "in_channels", "out_channels", "mode"):
        conf.pop(k)
    blk = PreActFixupResBlock(in_channels=c_in, out_channels=c_out, mode=mode, **conf).eval()
    blk.load_state_dict(S.make_state_dict(blk.state_dict(), seed=seed, regime="perturbed", n_layers=12))
    return blk.to(DEV)


def _params(blk):
    return {k: v.detach().cpu() for k, v in blk.state_dict().items()}


def _split_w_abs(pk):
    """absolute error of a split weight whose low half is subnormal: 2^-25 / premul (tc_split.cu:9-13)"""
    return tuple(2.0 ** -25 / float(v) for v in pk.split_premul)


def _bound_images(y, x, p, batch, **kw):
    """f64 bound at the first, middle and last image; returns the largest err/bound."""
    worst = 0.0
    for i in sorted({0, batch // 2, batch - 1}):
        xi = x[i].permute(2, 0, 1)[None].cpu()
        ref = FB.fixup_block(xi, p, **kw)
        ok, ratio, err = FB.check(y[i].permute(2, 0, 1)[None].cpu(), ref)
        assert ok, (i, ratio, err)
        worst = max(worst, ratio)
    return worst


def _run_chunks(fn, x, chunk, launches):
    outs = []
    for i in range(0, x.shape[0], chunk):
        n0 = E.launch_count()
        outs.append(fn(x[i:i + chunk]))
        assert E.launch_count() - n0 == launches
    return torch.cat(outs)


def _equal_per_image(a, b):
    torch.cuda.synchronize()
    bad = [i for i in range(a.shape[0]) if not torch.equal(a[i], b[i])]
    assert not bad, f"images {bad[:8]} differ between the saturated and the chunked launch"


# (mode, c_in, h, w, batch, precision) -- 'up' at 32^2 runs B = 256: at B = 64 its head
# would have < 3 m-tiles per warp at 4 CTAs per SM
BLOCK_CASES = {
    "same8_256": ("same", 8, 256, 256, 256, "fp16"),
    "same8_512": ("same", 8, 512, 512, 64, "fp16"),
    "same16_128": ("same", 16, 128, 128, 256, "fp16"),
    "same8_128x256": ("same", 8, 128, 256, 256, "fp16"),
    "down8_256": ("down", 8, 256, 256, 256, "fp16"),
    "down16_128": ("down", 16, 128, 128, 256, "fp16"),
    "down32_64": ("down", 32, 64, 64, 256, "fp16"),
    "down16_64x192": ("down", 16, 64, 192, 256, "fp16"),
    "up16_128": ("up", 16, 128, 128, 64, "fp16"),
    "up16_256": ("up", 16, 256, 256, 64, "fp16"),
    "up32_32": ("up", 32, 32, 32, 256, "fp16"),
    "up64_32": ("up", 64, 32, 32, 256, "fp16"),
    "up128_32": ("up", 128, 32, 32, 256, "fp16"),
    "up32_16x64": ("up", 32, 16, 64, 256, "fp16"),
    "down128_64": ("down", 64, 64, 64, 64, "fp16"),
    "down128_32x96": ("down", 64, 32, 96, 128, "fp16"),
    "split_same8_256": ("same", 8, 256, 256, 256, "fp32tc"),
    "split_same16_128": ("same", 16, 128, 128, 256, "fp32tc"),
    "split_same32_64": ("same", 32, 64, 64, 256, "fp32tc"),
    "split_same64_32": ("same", 64, 32, 32, 256, "fp32tc"),
    "split_same16_64x96": ("same", 16, 64, 96, 256, "fp32tc"),
    "split_down8_256": ("down", 8, 256, 256, 256, "fp32tc"),
    "split_down16_128": ("down", 16, 128, 128, 256, "fp32tc"),
    "split_down32_64": ("down", 32, 64, 64, 256, "fp32tc"),
}


def _units(mode, c, h, w, precision):
    """[(units per image, cap, one_per_sm, slot, kernel name)] of the kernel(s) this block dispatches to
    (engine.fixup_forward_nhwc with the switches below; names as the profiler shows them)."""
    if precision == "fp32tc":
        if mode == "same":
            name = (f"same_block_mma_split_kernel<{c}, 8>" if c in E.SPLIT_MMA
                    else f"same_block_split_kernel<{c}, {c}>")
            return [units_split_same(c, h, w) + ("cta", name)]
        return [units_down(c, h, w, split=True) + ("warp", f"down_block_mma_kernel<{c}, true>")]
    if mode == "same":
        th = 16 if c == 8 and h % 16 == 0 else 8
        return [units_same(c, h, w) + ("cta", f"same_block_mma_kernel<{c}, {th}>")]
    if mode == "down":
        if c == 64:
            return [units_down128(h, w) + ("cta", "down128_tc_kernel")]
        return [units_down(c, h, w) + ("warp", f"down_block_mma_kernel<{c}, false>")]
    head, tail = units_up(c, h, w)
    ty = 16 if c <= 32 and (2 * h) % 16 == 0 else 8
    return [head + ("warp", f"up_head_mma_kernel<{c}>"), tail + ("cta", f"up_tail3_mma_kernel<{c}, {ty}>")]


def _bound_kw(mode, c, precision, pk):
    if precision == "fp32tc":
        return dict(r=FB.SPLIT, fold_scale=mode == "down", w_abs=_split_w_abs(pk))
    interp = FB.Rounding(FB.U_SPLIT_ACT, FB.ETA_F16, 0.0, FB.U_ACC_TC, 3)    # mma_up.cu:11-15
    # fp16 operands: the reference rounds A1, U, V, the skip operand and the packed weights to fp16
    # where the kernels do (mma_same.cu:19-28, mma_down.cu:6-14, mma_up.cu:6-17, tc_down128.cu:6-13)
    return dict(r=FB.FP16_ROUNDED, interp=interp, fold_scale=mode in ("down", "up"))


@pytest.mark.parametrize("case", sorted(BLOCK_CASES))
def test_block_saturated_vs_chunked_and_f64_bound(case, monkeypatch):
    mode, c, h, w, batch, precision = BLOCK_CASES[case]
    monkeypatch.setattr(E, "LOWC_MMA", {8, 16})
    monkeypatch.setattr(E, "DOWN_MMA", {8, 16, 32})
    monkeypatch.setattr(E, "SPLIT_MMA", {8, 16})
    lib = L.load()
    if precision == "fp32tc":
        if mode == "down":
            assert lib.vqae_down_block_mma_supported(h, w, c)
        elif c in E.SPLIT_MMA:                                   # engine.py:495-497
            assert lib.vqae_same_block_mma_split_supported(h, w, c)
        else:
            assert lib.vqae_same_block_split_supported(h, w, c)
    elif mode == "same":
        assert lib.vqae_same_block_mma_supported(h, w, c)
    elif mode == "up":
        assert lib.vqae_up_block_mma_supported(h, w, c)
    elif c == 64:
        assert h % 32 == 0 and w % 32 == 0                      # down128_tc_supported
    else:
        assert lib.vqae_down_block_mma_supported(h, w, c)
    blk = _block(mode, c, 300 + c)
    pk = blk.packed()
    p = _params(blk)
    launches = 2 if mode == "up" and precision == "fp16" else 1
    kernels = _units(mode, c, h, w, precision)
    # chunks of whole images (a block's borders wrap / clamp per image): one unit per slot, except where
    # one image alone exceeds the grid (up16_256: 1.73 head m-tiles per warp, 1.15 tail tiles per CTA);
    # there the chunked side loops at most twice against ~110 times in the saturated launch
    chunk = min(_chunk(u, cap) for u, cap, *_ in kernels)
    chunk_desc = ", ".join(f"{u * chunk / min(u * chunk, cap):.2f}" for u, cap, *_ in kernels)
    fn = lambda t: E.fixup_forward_nhwc(pk, t, precision=precision)          # noqa: E731
    ragged = _ragged_batch(kernels, batch - 1)
    worst = 0.0
    for b in (batch, ragged):
        desc = []
        for u, cap, one, slot, _ in kernels:
            units, grid = _assert_saturated(u, cap, one, b, slot)
            desc.append(f"{units / grid:.2f} units/{slot} (last wave {units % grid}/{grid})")
        x = torch.randn(b, h, w, c, generator=torch.Generator().manual_seed(b + c + h), device="cpu").to(DEV)
        fn(x[:1])                                              # packs the weights (one more launch)
        n0 = E.launch_count()
        y, names = _run_profiled(fn, x)
        assert E.launch_count() - n0 == launches
        _assert_ran(names, [k[-1] for k in kernels])
        y_chunks = _run_chunks(fn, x, chunk, launches)
        _equal_per_image(y, y_chunks)
        worst = max(worst, _bound_images(y, x, p, b, **_bound_kw(mode, c, precision, pk)))
        print(f"{case} B={b}: " + ", ".join(desc) + f"; chunks of {chunk}: {chunk_desc} units/slot")
        del x, y, y_chunks
    print(f"{case}: max err/bound {worst:.3g}")


# ---- stems --------------------------------------------------------------------------------------------------
def _stem_weights(seed=7):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(8, 3, 3, 3, generator=g) * 0.3).to(DEV), (torch.randn(8, generator=g) * 0.1).to(DEV)


@pytest.mark.parametrize("kind,h,w,batch", [("u8", 256, 256, 256), ("nchw", 256, 256, 256),
                                            ("nhwc", 256, 256, 256), ("u8", 128, 384, 256)])
def test_stem_in_saturated_vs_chunked_and_f64_bound(kind, h, w, batch):
    """stem_in_u8_mma_kernel (u8, 4-byte aligned input) and stem_in_mma_kernel<0/1> (fp32 NCHW / NHWC)."""
    wt, bias = _stem_weights()
    u_img, cap, one = units_stem_in(h, w)
    ragged = _ragged_batch([(u_img, cap)], batch - 1)
    kname = {"u8": "stem_in_u8_mma_kernel", "nchw": "stem_in_mma_kernel<0>", "nhwc": "stem_in_mma_kernel<1>"}[kind]
    wmax = float(wt.abs().max())
    worst = 0.0
    for b in (batch, ragged):
        units, grid = _assert_saturated(u_img, cap, one, b, "cta")
        if kind == "u8":
            x = S.synthetic_patches_u8(b, h, b).to(DEV) if h == w else \
                torch.randint(0, 256, (b, h, w, 3), generator=torch.Generator().manual_seed(b),
                              dtype=torch.uint8).to(DEV)
            assert x.data_ptr() % 4 == 0
        else:
            x = torch.randn(b, 3, h, w, generator=torch.Generator().manual_seed(b)).to(DEV)
            if kind == "nhwc":
                x = x.contiguous(memory_format=torch.channels_last)
        fn = lambda t: E.stem_in(t, wt, bias, precision="fp16")          # noqa: E731
        n0 = E.launch_count()
        y, names = _run_profiled(fn, x)
        assert E.launch_count() - n0 == 1
        _assert_ran(names, [kname])
        chunk = _chunk(u_img, cap)
        for i in range(0, b, chunk):                   # every chunk keeps the input's 4-byte alignment
            assert x[i:i + chunk].data_ptr() % 4 == x.data_ptr() % 4
        _equal_per_image(y, _run_chunks(fn, x, chunk, 1))
        for i in sorted({0, b // 2, b - 1}):
            if kind == "u8":
                xi = FB.normalized_u8(x[i:i + 1].cpu())
                r = FB.Rounding(0.0, 0.0, 0.0, FB.U_ACC_TC, 2)           # exact u8 operands, split weights
            else:
                xi = FB.exact(x[i:i + 1].cpu())
                r = FB.SPLIT
            ref = FB.stem(xi, wt.cpu(), bias.cpu(), r, w_abs=2.0 ** -25 * wmax / 2.0 ** 13)
            ok, ratio, err = FB.check(y[i:i + 1].permute(0, 3, 1, 2).cpu(), ref)
            assert ok, (i, ratio, err)
            worst = max(worst, ratio)
        print(f"stem_in {kind} {h}x{w} B={b}: {units / grid:.2f} units/cta (last wave {units % grid}/{grid})")
    print(f"stem_in {kind} {h}x{w}: max err/bound {worst:.3g}")


# ---- the fp32 CUDA-core kernels (the reference of every other GPU test) ---------------------------------------
@pytest.mark.parametrize("mode,c,h,w", [("same", 16, 48, 96), ("same", 64, 24, 40), ("down", 16, 64, 96),
                                        ("down", 64, 32, 48), ("up", 32, 16, 48), ("up", 64, 12, 20)])
def test_fp32_block_kernels_within_f64_bound(mode, c, h, w):
    """conv_f32.cu / up_head.cu / up_tail.cu ("fp32" precision) at non-square shapes, u = 0."""
    blk = _block(mode, c, 500 + c)
    pk = blk.packed()
    x = torch.randn(3, h, w, c, generator=torch.Generator().manual_seed(h * w)).to(DEV)
    y = E.fixup_forward_nhwc(pk, x, precision="fp32")
    worst = _bound_images(y, x, _params(blk), 3, r=FB.EXACT)
    print(f"fp32 {mode} C{c} {h}x{w}: max err/bound {worst:.3g}")


@pytest.mark.parametrize("h,w", [(48, 80), (64, 96)])
def test_fp32_stems_within_f64_bound(h, w):
    """stems.cu: in_stem from fp32 (NCHW) and u8 input, out_stem (NCHW out), u = 0."""
    wt, bias = _stem_weights(11)
    g = torch.Generator().manual_seed(h + w)
    x = torch.randn(2, 3, h, w, generator=g).to(DEV)
    xu = torch.randint(0, 256, (2, h, w, 3), generator=g, dtype=torch.uint8).to(DEV)
    y = E.stem_in(x, wt, bias, precision="fp32")
    yu = E.stem_in(xu, wt, bias, precision="fp32")
    wo = (torch.randn(3, 8, 3, 3, generator=g) * 0.3).to(DEV)
    bo = (torch.randn(3, generator=g) * 0.1).to(DEV)
    z = E.stem_out(y, wo, bo, channels_last=False, precision="fp32")
    torch.cuda.synchronize()
    ref_y = FB.stem(FB.exact(x.cpu()), wt.cpu(), bias.cpu(), FB.EXACT)
    ref_u = FB.stem(FB.normalized_u8(xu.cpu()), wt.cpu(), bias.cpu(), FB.EXACT)
    ref_z = FB.stem(FB.exact(y.permute(0, 3, 1, 2).cpu()), wo.cpu(), bo.cpu(), FB.EXACT)
    ratios = []
    for got, ref in ((y.permute(0, 3, 1, 2), ref_y), (yu.permute(0, 3, 1, 2), ref_u), (z, ref_z)):
        ok, ratio, err = FB.check(got.cpu(), ref)
        assert ok, (ratio, err)
        ratios.append(ratio)
    print(f"fp32 stems {h}x{w}: max err/bound in {ratios[0]:.3g}, u8 {ratios[1]:.3g}, out {ratios[2]:.3g}")


# ---- the model at the benched shapes ----------------------------------------------------------------------------
def test_encode256_codes_across_precisions():
    """encode256 (batch 256 of 256^2): fp32tc codes equal fp32 codes outside near-ties (the latent-error
    scaled threshold of test_model_vs_reference_golden); fp16 codes agree with fp32 at >= 0.994."""
    m, _, _ = H.model_and_state("model_nd3_perturbed")
    m = m.to(DEV)
    x = S.synthetic_patches(256, 256, 4242).to(DEV)
    out = {}
    try:
        with torch.no_grad():
            for prec in ("fp32", "fp32tc", "fp16"):
                vqae_b200.set_precision(m, prec)
                _, idx, _, _, z = m.encoder.encode(x, want_latents=True)
                out[prec] = (idx.reshape(-1), z.reshape(-1, z.shape[-1]))
            embed = m.encoder.vq_layers[0].embed.detach().double()
            idx32, z32 = out["fp32"]
            d1s, gaps = [], []
            for s in range(0, z32.shape[0], 32768):
                d4 = ((z32[s:s + 32768].double()[:, None, :] - embed[None]) ** 4).sum(-1)
                top = d4.topk(2, dim=1, largest=False).values
                d1s.append(top[:, 0] ** 0.25)
                gaps.append((top[:, 1] - top[:, 0]) / top[:, 0].clamp_min(1e-300))
            d1, gap = torch.cat(d1s), torch.cat(gaps)
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()
    idx_tc, z_tc = out["fp32tc"]
    z_err = float((z_tc - z32).abs().max())
    thresh = torch.clamp(64.0 * z_err / d1.clamp_min(1e-12), min=H.NEAR_TIE_REL_GAP)
    bad = (idx_tc != idx32) & (gap >= thresh)
    assert int(bad.sum()) == 0, (int(bad.sum()), int((idx_tc != idx32).sum()), z_err)
    agree = float((out["fp16"][0] == idx32).double().mean())
    print(f"encode256: fp32tc flips {int((idx_tc != idx32).sum())} (all near-ties, latent err {z_err:.2e}); "
          f"fp16 agreement {agree:.4f}")
    assert agree >= 0.994, agree


def test_decode512_fp16_decoder_on_fp32_codes():
    """roundtrip512 shape (batch 64 of 512^2): the fp16 decoder on the fp32 encoder's codes stays within
    2e-3 of the fp32 decoder (the bar of test_gpu_golden_reduced.py)."""
    m, _, _ = H.model_and_state("model_nd4_perturbed_512")
    m = m.to(DEV)
    x = S.synthetic_patches(64, 512, 4343).to(DEV)
    try:
        with torch.no_grad():
            vqae_b200.set_precision(m, "fp32")
            _, idx, _, _, _ = m.encoder.encode(x, want_quantized=False)
            d32 = m.decode_codes(idx)
            vqae_b200.set_precision(m, "fp16")
            d16 = m.decode_codes(idx)
        err = H.rel_err(d16, d32)
    finally:
        vqae_b200.set_precision(m, None)
        m.cpu()
    print(f"decode512: fp16 vs fp32 decoder {err:.2e}")
    assert err < 2e-3, err


# ---- decode-side gather past gridDim.y = 65 535 ----------------------------------------------------------------
@pytest.mark.parametrize("u8", [True, False])
def test_embed_codemap_beyond_65535_patches(u8):
    """vqae_embed_codemap_f32 strides its patches over gridDim.y <= 65 535 (quantize.cu:315, 486):
    70 001 patches of 2 x 2 codes, first_patch 123, region_cols 257 (does not divide n), codes out of
    range clamped like embed_codes."""
    lib = L.load()
    k, c, th, tw = 200, 8, 2, 2
    n, first, rcols, r0, c0 = 70001, 123, 257, 1, 2
    rows = (r0 + (first + n - 1) // rcols + 1) * th
    cols = (c0 + rcols) * tw + 2
    g = torch.Generator().manual_seed(9)
    if u8:
        cm = torch.randint(0, 256, (rows, cols), generator=g, dtype=torch.uint8).to(DEV)
    else:
        cm = torch.randint(-3, k + 3, (rows, cols), generator=g, dtype=torch.int64).to(DEV)
    table = torch.randn(k, c, generator=g).to(DEV)
    out = torch.full((n, th, tw, c), float("nan"), device=DEV)
    n0 = E.raw_launch_count()
    L.check(lib.vqae_embed_codemap_f32(E._ptr(cm), int(u8), rows, cols, th, tw, r0, c0, rcols, first, n,
                                       E._ptr(table), k, c, E._ptr(out), E._stream(cm.device)),
            "vqae_embed_codemap_f32")
    assert E.raw_launch_count() - n0 == 1
    q = torch.arange(first, first + n, device=DEV)
    pr, pc = q // rcols, q % rcols
    yy = ((r0 + pr) * th)[:, None, None] + torch.arange(th, device=DEV)[None, :, None]
    xx = ((c0 + pc) * tw)[:, None, None] + torch.arange(tw, device=DEV)[None, None, :]
    codes = cm.long()[yy, xx].clamp(0, k - 1)
    assert torch.equal(out, table[codes])
