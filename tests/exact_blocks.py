"""TEST INFRASTRUCTURE ONLY -- integer-valued 'same' blocks on which the tensor-core kernels are exact.

With every weight in {-1, 0, 1}, ``scale`` in {1, 2, 4}, integer biases and integer inputs, every fp32
operation of the tcgen05 'same' kernels (tc_kernels.cu, tc_chain.cu, tc_resident.cu) is exact:

* ``bias1a = bias2a = bias3a = 2^20`` and ``biasNb = -2^20 + k`` (small integer k) keep every
  pre-activation on the linear branch of act_pack8 (tc_common.cuh: ``v + (pre + post)`` when
  ``v > -pre``), and ``pre + post = k`` is exact; the resident kernel's fold ``pre = b1a + cum`` is
  exact too while ``|cum| < 2^23``;
* products are exact and every sum stays below 2^24, so the order of accumulation does not matter;
* the fp16 operand roundings (A1, U, V; VQAE_OPERAND_F16 in tc_common.cuh) are round-to-nearest-even
  of exactly computed fp32 values -- deterministic, and reproduced here with ``.float().half()``;
* ``scale * W3`` (folded at pack time for the resident kernel, pack.cu) is exact in fp16, and the
  tile kernels' ``fmaf(d, scale, b4) + x`` is exact.

A kernel's output therefore equals ``reference`` bit for bit.  The reference checks these
preconditions at every stage and raises ``NotExact`` where one fails, so that a case which drifts out
of the exact regime fails as a bad test, not as a kernel fault.

Growth.  A stack of integer residual blocks compounds: x + B(x) with |B| >= 1 grows geometrically and
54 blocks would overflow fp16.  The channels are therefore split into two random halves, S and T.  In
the first ceil(n / 2) blocks W1 reads only S and W3 writes only T, in the rest the other way round.
Within a half B_j B_i = 0, so the residual grows linearly, and it compounds only once, at the swap.
Every block still has its own random W1, W2 (all nine taps, all channels) and W3, and the swap
makes the channels that one half reads the ones the other half writes.  Inputs and biases are drawn
so that operands of the later blocks pass 2048: the fp16 rounding points are exercised as well.
"""
from __future__ import annotations

from typing import Dict, List

import torch

Tensor = torch.Tensor
BIG = 2.0 ** 20
F16_MAX = 65504.0
EXACT_SUM = 2.0 ** 24


class NotExact(ValueError):
    """A case left the regime in which the kernels compute exactly: the test is wrong, not the kernel."""


def _ternary(shape, density: float, g: torch.Generator) -> Tensor:
    keep = torch.rand(shape, generator=g) < density
    sign = torch.randint(0, 2, shape, generator=g) * 2 - 1
    return (keep * sign).float()


def integer_blocks(c: int, n: int, seed: int) -> List[Dict[str, Tensor]]:
    """n state dicts of 'same' PreActFixupResBlocks (OIHW fp32 weights, 1-element scalars)."""
    g = torch.Generator().manual_seed(seed)
    perm = torch.randperm(c, generator=g)
    halves = (perm[: c // 2], perm[c // 2:])
    damp = min(1.0, 4.0 / n) ** 0.5                       # long runs: sparser W1 and W3
    out = []
    for k in range(n):
        src, dst = halves if k < (n + 1) // 2 else halves[::-1]
        w1 = _ternary((c, c), 2.0 * damp / c, g)          # ~1 input per U channel (short runs)
        w1[:, dst] = 0
        w2 = _ternary((c, c, 3, 3), 2.5 / (9 * c), g)     # ~2.5 taps x channels per V channel
        w3 = _ternary((c, c), 2.0 * damp / c, g)          # ~1 V channel per output of T (short runs)
        w3[src, :] = 0
        ks = torch.randint(-3, 4, (3,), generator=g).tolist()
        b4 = int(torch.randint(1, 4, (1,), generator=g)) * (1 if torch.rand(1, generator=g) < 0.5 else -1)
        scale = float(2 ** int(torch.randint(0, 3, (1,), generator=g)))
        p = {"branch_conv1.weight": w1[:, :, None, None], "branch_conv2.weight": w2,
             "branch_conv3.weight": w3[:, :, None, None]}
        for name, val in (("bias1a", BIG), ("bias1b", -BIG + ks[0]), ("bias2a", BIG),
                          ("bias2b", -BIG + ks[1]), ("bias3a", BIG), ("bias3b", -BIG + ks[2]),
                          ("bias4", float(b4)), ("scale", scale)):
            p[name] = torch.tensor([val])
        out.append(p)
    return out


def integer_input(shape, seed: int, lim: int = 24) -> Tensor:
    """Integer-valued fp32 NHWC input in [-lim, lim]."""
    g = torch.Generator().manual_seed(seed)
    return torch.randint(-lim, lim + 1, shape, generator=g).float()


def load_block(blk, p: Dict[str, Tensor]) -> None:
    """Copy an integer_blocks entry into a PreActFixupResBlock (on any device)."""
    with torch.no_grad():
        sd = blk.state_dict()
        for k, v in p.items():
            sd[k].copy_(v.reshape(sd[k].shape))


class Stats:
    """What the reference saw: the largest operand and how many operand values fp16 rounded."""

    def __init__(self):
        self.max_operand = 0.0
        self.rounded = 0
        self.operands = 0


def _require(cond: bool, what: str) -> None:
    if not cond:
        raise NotExact(what)


def _f16(v: Tensor, where: str, st: Stats) -> Tensor:
    """fp16 rounding of an exactly computed value, as the kernel's operand conversion does."""
    _require(bool((v.abs() < EXACT_SUM).all()), f"{where}: |value| >= 2^24 before the fp16 rounding")
    r = v.float().half().double()
    _require(bool((r.abs() <= F16_MAX).all()), f"{where}: fp16 overflow")
    st.max_operand = max(st.max_operand, float(r.abs().max()))
    st.rounded += int((r != v).sum())
    st.operands += v.numel()
    return r


def _act(v: Tensor, a: float, b: float, where: str) -> Tensor:
    """elu(v + a) + b on its linear branch (requires v > -a): v + (a + b)."""
    _require(bool((v > -a).all()), f"{where}: pre-activation <= -bias (ELU's exponential branch)")
    return v + (a + b)


def _mm(a: Tensor, w: Tensor, where: str) -> Tensor:
    """a [..., C_in] . w[C_out, C_in]^T in float64, exact while sum |w| |a| < 2^24."""
    bound = float(a.abs().amax()) * float(w.abs().sum(1).amax())
    _require(bound < EXACT_SUM, f"{where}: sum |w| |a| may reach 2^24 ({bound:.3g})")
    return a @ w.t()


def block(x: Tensor, p: Dict[str, Tensor], k: int, st: Stats) -> Tensor:
    """One integer 'same' block on NHWC float64 x (any device), with the kernels' fp16 rounding points."""
    _require(bool((x == x.round()).all()), f"block {k}: non-integer input")
    _require(bool((x.abs() < BIG / 2).all()), f"block {k}: |x| >= 2^19")
    f = {n: float(v) for n, v in p.items() if v.numel() == 1}
    dev = x.device
    w1 = p["branch_conv1.weight"][:, :, 0, 0].double().to(dev)
    w2 = p["branch_conv2.weight"].double().to(dev)
    w3 = (p["branch_conv3.weight"][:, :, 0, 0] * f["scale"]).double().to(dev)
    a1 = _f16(_act(x, f["bias1a"], f["bias1b"], f"block {k} A1"), f"block {k} A1", st)
    u = _f16(_act(_mm(a1, w1, f"block {k} G1"), f["bias2a"], f["bias2b"], f"block {k} U"), f"block {k} U", st)
    umax = float(u.abs().amax())
    l1 = float(w2.abs().sum((1, 2, 3)).amax())
    _require(umax * l1 < EXACT_SUM, f"block {k} G2: sum |w| |a| may reach 2^24")
    d2 = torch.zeros(x.shape[:-1] + (w2.shape[0],), dtype=torch.float64, device=dev)
    for ky in range(3):
        for kx in range(3):
            if bool(w2[:, :, ky, kx].any()):
                d2 += torch.roll(u, shifts=(1 - ky, 1 - kx), dims=(1, 2)) @ w2[:, :, ky, kx].t()
    v = _f16(_act(d2, f["bias3a"], f["bias3b"], f"block {k} V"), f"block {k} V", st)
    # the resident kernel accumulates scale * W3 . V straight into the residual: |x| + sum < 2^24
    bound = float(x.abs().amax()) + float(v.abs().amax()) * float(w3.abs().sum(1).amax())
    _require(bound + abs(f["bias4"]) * (k + 1) < EXACT_SUM, f"block {k} G3: residual sum may reach 2^24")
    return x + v @ w3.t() + f["bias4"]


def reference(x: Tensor, blocks: List[Dict[str, Tensor]], st: Stats = None, half_io: bool = False) -> Tensor:
    """The run of ``blocks`` on NHWC x (fp32 or fp16, any device) in float64: what the kernels must
    produce bit for bit.  ``half_io``: the result is rounded to fp16 at the store (fp16 streams)."""
    st = st if st is not None else Stats()
    h = x.double()
    for k, p in enumerate(blocks):
        h = block(h, p, k, st)
    _require(bool((h == h.round()).all()), "output not integer")
    if half_io:
        _require(bool((h.abs() <= F16_MAX).all()), "output overflows fp16")
        return h.float().half()
    return h.float()
