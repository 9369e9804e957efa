"""CPU: the float64 error bound of tests/f64_bound.py against a 'same' block emulated with the fp16
roundings of mma_same.cu (``.half().float()`` at the points its header lists): the bound holds and is
not vacuous, and a fault confined to the image border that passes the max-normalised bar of the older
tensor-core tests fails the per-element check (with the rounding points emulated; the plain worst-case
fp16 bound is too loose for that)."""
import torch
import torch.nn.functional as F

import f64_bound as B
import helpers as H
import vqae_oracle as O


def _f16(t):
    return t.half().float()


def _emulate_same(x, p, fault=0.0):
    """mma_same.cu in fp32 with fp16 operands: A1, U, V and W1, W2, W3 rounded to fp16 (header
    lines 19-28).  ``fault``: the branch_conv2 weights of tap (ky, kx) = (0, 1) are off by this
    fraction, but only where that tap reads the wrapped halo row above row 0."""
    f = {k: float(v) for k, v in p.items() if v.dim() == 0 or v.numel() == 1}
    w1, w2, w3 = (_f16(p[f"branch_conv{i}.weight"].float()) for i in (1, 2, 3))
    a1 = _f16(O.elu(x + f["bias1a"]) + f["bias1b"])
    u = _f16(O.elu(F.conv2d(a1, w1) + f["bias2a"]) + f["bias2b"])
    d2 = F.conv2d(F.pad(u, (1, 1, 1, 1), mode="circular"), w2)
    if fault:
        d2[:, :, 0, :] += fault * torch.einsum("oc,bcw->bow", w2[:, :, 0, 1], u[:, :, -1, :])
    v = _f16(O.elu(d2 + f["bias3a"]) + f["bias3b"])
    return x + (F.conv2d(v, w3) * f["scale"] + f["bias4"])


def _case():
    blk = H.make_block("same16")
    p = {k: v.detach() for k, v in blk.state_dict().items()}
    x = torch.randn(2, 16, 32, 48, generator=torch.Generator().manual_seed(5))
    return p, x


def test_emulated_fp16_same_block_within_bound():
    p, x = _case()
    y = _emulate_same(x, p)
    ok_w, ratio_w, _ = B.check(y, B.fixup_block(x, p, B.FP16))
    ok, ratio, err = B.check(y, B.fixup_block(x, p, B.FP16_ROUNDED))
    print(f"emulated fp16 'same' C16: max err/bound {ratio:.3g} with the rounding points emulated "
          f"(max err {err:.3g}), {ratio_w:.3g} against the worst-case fp16 bound")
    assert ok_w and ok, (ratio_w, ratio)
    assert ratio >= 1e-2, ratio                        # the bound is not vacuous
    assert ratio_w >= 1e-2, ratio_w


def test_border_fault_passes_old_bar_and_fails_per_element_check():
    """A fault of one tap's weights (a few percent) used only at the wrapped border row, sized so that
    the error stays under the old bar (1e-2 of the branch maximum, here 5e-3): the per-element check
    with the rounding points emulated flags it, on the faulted row only.  The worst-case fp16 bound
    (``B.FP16``: every rounding charged as u |a| and carried through |W2|, whose entries sum to ~15 per
    output channel here) is about 50x above the actual error and does not see a fault this small --
    which is why the fp16 kernels are checked against ``B.FP16_ROUNDED``."""
    p, x = _case()
    ref = B.fixup_block(x, p, B.FP16_ROUNDED)
    clean = _emulate_same(x, p)
    branch = float((ref.v - x.double()).abs().max())
    probe = float((_emulate_same(x, p, fault=1.0) - clean).abs().max())
    delta = 5e-3 * branch / probe
    assert 0.005 < delta < 0.1, delta                  # a few percent of one tap's weights
    y = _emulate_same(x, p, fault=delta)
    old = float((y.double() - ref.v).abs().max()) / branch
    assert old < 1e-2, old                             # the max-normalised bar does not see it
    ok, ratio, _ = B.check(y, ref)
    _, ratio_w, _ = B.check(y, B.fixup_block(x, p, B.FP16))
    print(f"border fault of {delta:.2%}: {old:.2e} of the branch max; max err/bound {ratio:.3g} "
          f"(worst-case fp16 bound: {ratio_w:.3g})")
    assert not ok
    bad = (y.double() - ref.v).abs() > 2.0 * ref.e
    assert bad[:, :, 0, :].any() and not bad[:, :, 1:, :].any()


def test_bound_of_exact_arithmetic_covers_float32_torch():
    """u = 0 (the fp32 CUDA-core kernels' setting): torch's own fp32 block is within the bound."""
    p, x = _case()
    ref = B.fixup_block(x, p, B.EXACT)
    y = O.fixup_block(x, {k: v.float() for k, v in p.items()})
    ok, ratio, _ = B.check(y, ref)
    assert ok, ratio


def test_bicubic_abs_is_the_tap_magnitude_sum():
    x = torch.ones(1, 1, 5, 7, dtype=torch.float64)
    assert torch.allclose(O.bicubic_up2(x), torch.ones(1, 1, 10, 14, dtype=torch.float64))
    inner = B.bicubic_abs(x)[0, 0, 3:7, 3:11]
    assert torch.allclose(inner, torch.full_like(inner, (328 / 256) ** 2))
