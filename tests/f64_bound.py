"""TEST INFRASTRUCTURE ONLY -- float64 references that carry a per-element forward error bound.

Each function restates a layer of ``oracle/vqae_oracle.py`` (``fixup_block``, ``bicubic_up2``, the
zero-padded stems) on CPU float64 tensors and, alongside the value, an upper bound on how far a kernel
that rounds at the given points can be from it.  The bound is the textbook forward analysis:

* a rounded operand adds ``u |a| + eta`` to the error it already carries (``eta``: fp16 numbers below
  2^-14 are subnormal, spacing 2^-24, so rounding there is off by up to 2^-25 absolute) -- or, for the
  fp16 kernels (``FP16_ROUNDED``), the reference rounds the operand to fp16 itself and the bound passes
  through the rounding as the exact image of its interval;
* a conv carries an input error ``e`` as ``|W| conv e``, and adds ``(u_w + gamma_K) |W| conv |a|``
  for rounded weights and K fp32 accumulations, ``gamma_K = K u_acc / (1 - K u_acc)``;
* ELU is 1-Lipschitz, so it passes the error on unchanged; each fp32 elementwise step (bias add, the
  activation, the residual add) adds a few ulps of its operands and result.

Magnitudes ``|a|`` are taken as ``|a_ref| + e`` so that the bound also covers the kernel's own (perturbed)
operands.  A kernel that is right sits well inside the bound; the tests assert ``|y - y64| <= 2 bound``
at every element.  With the rounding points emulated (fp16 kernels) or operand errors near 2^-22
(split and fp32 kernels) the bound is a few times the actual error, so a fault confined to a few
pixels is caught even where a bar normalised to the tensor's maximum would not see it.  The plain
worst-case fp16 bound (``FP16``) is not that tight: tests/test_f64_bound_host.py shows both.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Mapping, Optional, Tuple

import torch
import torch.nn.functional as F

import vqae_oracle as O

Tensor = torch.Tensor

# fp16 operand: round to nearest, 11 significand bits
U_F16 = 2.0 ** -11
ETA_F16 = 2.0 ** -25
# Split operand (tc_split.cu, mma_same_split.cu, mma_down.cu SPLIT, mma_stem.cu): v = hi + lo with
# hi = f16(v), lo = f16(v - hi); |v - hi| <= 2^-11 |v| and |v - hi - lo| <= 2^-11 |lo| <= 2^-22 |v| (lo
# normal) or 2^-25 (lo subnormal).  A product is hi.hi + lo.hi + hi.lo; the dropped lo.lo is <= 2^-22 |a||w|.
# So per product: 2^-22 (activation remainder) + 2^-22 (lo.lo) on the activation side, charged as
# U_SPLIT_ACT, and 2^-22 on the weight side.  The weights are pre-multiplied by a power of two that moves
# max|w| into (2^13, 2^14] (engine.py:302-305, PackedFixup.descs_split): their low halves are normal down to
# 2^-27 of max|w|, below that the absolute error is 2^-25 / premul (``split_w_abs``).
U_SPLIT_ACT = 2.0 * 2.0 ** -22
U_SPLIT_W = 2.0 ** -22
# fp32 accumulation: tensor-core MMAs align and add without a guard digit (one ulp per step, not half);
# the CUDA-core kernels accumulate with IEEE fmaf (half an ulp)
U_ACC_TC = 2.0 ** -23
U_ACC_F32 = 2.0 ** -24
# fp32 elementwise steps: relative, per step, and the absolute error of the SFU exponential in the
# ELUs (ex2.approx: 2^-22 relative on e^x <= 1; elu1_tc: < 2.5e-7, common.cuh:36-41)
U_EW = 2.0 ** -22
EW_ABS = 2.0 ** -21


@dataclass(frozen=True)
class Rounding:
    """Where a kernel rounds the operands of one conv (or interpolation)."""
    act: float = 0.0          # relative error of an activation operand
    act_abs: float = 0.0      # absolute floor of that error
    w: float = 0.0            # relative error of a weight operand
    acc: float = U_ACC_F32    # unit roundoff of one accumulation step
    terms: int = 1            # products summed per weight-activation pair (3 for split operands)
    emulate: bool = False     # the reference itself rounds operand and weights to fp16 (``round_f16``)


# fp16 operands, worst case: the reference is the plain float64 block, every rounding is charged as
# u |a| (+ eta) and carried through the later convs as |W| conv error.  Valid, but with three chained
# convs it is two orders of magnitude above the error fp16 kernels actually make.
FP16 = Rounding(U_F16, ETA_F16, U_F16, U_ACC_TC, 1)
# fp16 operands, rounding points emulated: the reference rounds each operand and weight to fp16 where
# the kernel does, so only the accumulation order and the fp32 elementwise steps are charged; across a
# rounding point the bound is the exact image of its interval (``round_f16``).  The accumulation unit is
# doubled (2^-22) to cover accumulators that two convs share (the skip conv in the 'down' kernels).
FP16_ROUNDED = Rounding(0.0, 0.0, 0.0, 2.0 * U_ACC_TC, 1, emulate=True)
SPLIT = Rounding(U_SPLIT_ACT, ETA_F16, U_SPLIT_W, U_ACC_TC, 3)
# the fp32 CUDA-core kernels: no operand rounding (u = 0); weights may be pre-multiplied in fp32 at
# pack time (scale * W3), one rounding
EXACT = Rounding(0.0, 0.0, 2.0 ** -24, U_ACC_F32, 1)


@dataclass
class Bounded:
    v: Tensor                 # float64 reference value
    e: Tensor                 # float64 bound on |kernel - v|

    def mag(self) -> Tensor:
        return self.v.abs() + self.e


def exact(x: Tensor) -> Bounded:
    x = x.double()
    return Bounded(x, torch.zeros_like(x))


def gamma(k: int, u: float) -> float:
    assert k * u < 0.5
    return k * u / (1.0 - k * u)


def _pad(x: Tensor, pad: Optional[str]) -> Tensor:
    if pad == "circular":
        return F.pad(x, (1, 1, 1, 1), mode="circular")
    if pad == "zero":
        return F.pad(x, (1, 1, 1, 1))
    return x


def _f16(t: Tensor) -> Tensor:
    """fp16 rounding of an fp32 number (what __float2half_rn does to the kernel's fp32 value), in float64."""
    return t.float().half().double()


def round_f16(x: Bounded) -> Bounded:
    """The kernel rounds to fp16 an fp32 value that lies in [v - e, v + e].  Rounding is monotone, so
    the result lies between the roundings of the two ends: where both round to f16(v) the error is
    zero, elsewhere it is at most one fp16 spacing."""
    v = _f16(x.v)
    e = torch.maximum((_f16(x.v + x.e) - v).abs(), (_f16(x.v - x.e) - v).abs())
    return Bounded(v, e)


def conv(x: Bounded, w: Tensor, r: Rounding, stride: int = 1, pad: Optional[str] = None,
         w_abs: float = 0.0, into: Optional[Bounded] = None) -> Bounded:
    """conv2d without bias (``pad``: None, "circular" (the 'same' branch conv) or "zero" (the stems)).
    ``r.emulate``: the operand is rounded to fp16 first, and ``w`` (fp32, as packed) too.
    ``into``: the products accumulate onto this value in the same fp32 accumulator (one more term of
    the sum, whose magnitude joins the accumulation error)."""
    if r.emulate:
        x = round_f16(x)
        w = _f16(w)
    w = w.double()
    aw = w.abs()
    m = x.mag()
    k = r.terms * w.shape[1] * w.shape[2] * w.shape[3] + (into is not None)
    carried = x.e + r.act * m + r.act_abs
    y = F.conv2d(_pad(x.v, pad), w, stride=stride)
    e = F.conv2d(_pad(carried, pad), aw, stride=stride) + \
        F.conv2d(_pad(m, pad), (r.w + gamma(k, r.acc)) * aw + w_abs, stride=stride)
    if into is not None:
        y = y + into.v
        e = e + into.e + gamma(k, r.acc) * into.mag()
    return Bounded(y, e)


def pre_act(x: Bounded, a: float, b: Optional[float], elu: bool = True, a_mag: float = 0.0) -> Bounded:
    """elu(x + a) + b (the Fixup pre-activation; ``elu=False``: x + a, the skip path).  ``a_mag``: the
    kernel folds further terms of this size into ``a`` (the resident kernel's running bias4)."""
    s = x.v + a
    if not elu:
        return Bounded(s, x.e + U_EW * s.abs())
    v = O.elu(s) + (b or 0.0)
    # the fp16 kernels form elu(x + a) + b as x + (a + b) or exp2(x log2e + a log2e) + (b - 1)
    # (mma_common.cuh:33-35): roundings of a few ulps of |a| and |b| as well
    return Bounded(v, x.e + U_EW * (s.abs() + v.abs() + abs(a) + a_mag + abs(b or 0.0)) + EW_ABS)


def affine(x: Bounded, scale: float, bias: float) -> Bounded:
    v = x.v * scale + bias
    return Bounded(v, abs(scale) * x.e + U_EW * (x.v.abs() * abs(scale) + v.abs()))


def add(x: Bounded, y: Bounded) -> Bounded:
    v = x.v + y.v
    return Bounded(v, x.e + y.e + U_EW * v.abs())


def _bicubic_taps(n: int, absolute: bool):
    """O.bicubic_up2's clamped 4-tap table along one axis (optionally |weights|)."""
    o = torch.arange(2 * n, dtype=torch.float64)
    src = (o + 0.5) / 2.0 - 0.5
    fl = torch.floor(src)
    t = src - fl
    idx = torch.stack([(fl.long() + k).clamp(0, n - 1) for k in (-1, 0, 1, 2)], 0)
    w = torch.tensor([O._cubic_weights(float(tj)) for tj in t], dtype=torch.float64).t()
    return idx, (w.abs() if absolute else w)


def bicubic_abs(x: Tensor) -> Tensor:
    """O.bicubic_up2 with every tap weight replaced by its magnitude (carries error bounds)."""
    _, _, h, w = x.shape
    iy, wy = _bicubic_taps(h, True)
    ix, wx = _bicubic_taps(w, True)
    rows = sum(x[:, :, :, ix[k]] * wx[k] for k in range(4))
    return sum(rows[:, :, iy[k], :] * wy[k][:, None] for k in range(4))


def bicubic(x: Bounded, r: Rounding) -> Bounded:
    """nn.Upsample(bicubic, x2): 16 taps, operands rounded as ``r`` says."""
    m = x.mag()
    carried = x.e + r.act * m + r.act_abs
    return Bounded(O.bicubic_up2(x.v), bicubic_abs(carried) + gamma(16 * r.terms, r.acc) * bicubic_abs(m))


def fixup_block(x, p: Mapping[str, Tensor], r: Rounding, interp: Optional[Rounding] = None,
                fold_scale: bool = False, w_abs: Tuple[float, float, float] = (0.0, 0.0, 0.0),
                residual_in_acc: bool = False, cum_mag: float = 0.0) -> Bounded:
    """O.fixup_block in float64 with its bound.  ``x``: a Tensor (exact) or a ``Bounded`` that carries
    an input error in.  ``r``: the rounding of every conv; ``interp``: that of the 'up' interpolation
    (default ``r``); ``fold_scale``: the kernel multiplies branch_conv3 by the Fixup scale at pack time
    (rounded with the weights), otherwise it scales the accumulator.  An 'up' block is evaluated as the
    kernels do: both 1x1 ResizeConv2D convs at low resolution, then the upsample (they commute; |W| and
    the |taps| commute too, so the bound holds for either order).

    ``residual_in_acc`` (tc_resident.cu, a 'same' block with ``fold_scale``): branch_conv3 accumulates
    straight into the fp32 residual, so the residual add is one more accumulation term, charged as
    gamma(C + 1) (|R| + |W3s| conv |V|); bias4 joins a running sum that the kernel folds into the next
    block's bias1a and adds at the store (``cum_mag``: a bound on |that sum| when this block starts)."""
    f = lambda k: float(p[k])                                         # noqa: E731
    w1, w2, w3 = p["branch_conv1.weight"], p["branch_conv2.weight"], p["branch_conv3.weight"]
    k2 = w2.shape[-1]
    interp = interp or r
    x = x if isinstance(x, Bounded) else exact(x)
    h = pre_act(x, f("bias1a"), f("bias1b"), a_mag=cum_mag)
    h = conv(h, w1, r, w_abs=w_abs[0])
    h = pre_act(h, f("bias2a"), f("bias2b"))
    if k2 == 3:
        h = conv(h, w2, r, pad="circular", w_abs=w_abs[1])
    elif k2 == 2:
        h = conv(h, w2, r, stride=2, w_abs=w_abs[1])
    else:
        h = bicubic(conv(h, w2, r, w_abs=w_abs[1]), interp)
    h = pre_act(h, f("bias3a"), f("bias3b"))
    scale = float(p["scale"])
    if fold_scale:
        w3s = w3.float() * torch.tensor(scale, dtype=torch.float32)      # pack.cu: fp32 product
        if residual_in_acc:
            h = conv(h, w3s, r, w_abs=w_abs[2], into=x)
            # the accumulator holds R = y - cum, so |R| <= |y| + |cum| joins the accumulation term
            h = Bounded(h.v, h.e + gamma(r.terms * w3.shape[1] + 1, r.acc) * cum_mag)
            return affine(h, 1.0, f("bias4"))
        h = affine(conv(h, w3s, r, w_abs=w_abs[2]), 1.0, f("bias4"))
    else:
        h = affine(conv(h, w3, r, w_abs=w_abs[2]), scale, f("bias4"))
    if "skip_conv.weight" not in p:
        return add(h, x)
    ws = p["skip_conv.weight"]
    s = pre_act(x, f("bias1c"), None, elu=False)
    if ws.shape[-1] == 2:
        s = conv(s, ws, r, stride=2, w_abs=w_abs[2])
    elif k2 == 1:
        s = bicubic(conv(s, ws, r, w_abs=w_abs[2]), interp)
    else:
        s = conv(s, ws, r, w_abs=w_abs[2])
    return add(h, affine(s, 1.0, f("bias1d")))


def resident_carry(y: Tensor, bias4s) -> Tuple[Bounded, float]:
    """The input of block k + 1 of an image-resident run (tc_resident.cu) as the stored output y_k of
    the k-block run, and a bound on |cum_k|, the running fp32 sum of the bias4 of those k blocks
    (float64 sum plus one rounding per add).  The kernel holds R_k = y_k - cum_k in tensor memory; y_k
    is R_k + cum_k rounded once: carried error 2^-24 (|y_k| + |cum_k|)."""
    cum = abs(sum(bias4s)) + len(bias4s) * 2.0 ** -24 * sum(abs(b) for b in bias4s)
    y = y.double()
    return Bounded(y, 2.0 ** -24 * (y.abs() + cum)), cum


def stem(x: Bounded, w: Tensor, bias: Tensor, r: Rounding, w_abs: float = 0.0) -> Bounded:
    """3x3 conv with zero padding and bias (Encoder.in_stem / Decoder.out_stem)."""
    y = conv(x, w, r, pad="zero", w_abs=w_abs)
    v = y.v + bias.double()[None, :, None, None]
    return Bounded(v, y.e + U_EW * (y.v.abs() + v.abs()))


def normalized_u8(img_u8: Tensor, mean=O.CAMELYON16_MEAN, std=O.CAMELYON16_STD) -> Bounded:
    """u8 [B,H,W,3] -> [B,3,H,W] ``(u8 - 255 mean) / (255 std)`` in float64, with the error of the
    kernels' fp32 form ``(u8 - f32(255 mean)) * f32(1 / (255 std))`` (stems.cu:21-29, mma_stem.cu:563-566),
    or of folding the constants into split weights (mma_stem.cu): both within
    2^-20 (|x_n| + 2 * 255 mean / (255 std))."""
    m = torch.tensor(mean, dtype=torch.float64)[None, :, None, None]
    s = torch.tensor(std, dtype=torch.float64)[None, :, None, None]
    v = (img_u8.permute(0, 3, 1, 2).double() - 255.0 * m) / (255.0 * s)
    return Bounded(v, 2.0 ** -20 * (v.abs() + 2.0 * m / s))


def check(y: Tensor, ref: Bounded, factor: float = 2.0) -> Tuple[bool, float, float]:
    """(every element within ``factor`` x bound, max |y - ref| / bound, max |y - ref|)."""
    err = (y.double() - ref.v).abs()
    ratio = err / ref.e.clamp_min(1e-300)
    return bool((err <= factor * ref.e).all()), float(ratio.max()), float(err.max())
