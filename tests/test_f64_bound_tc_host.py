"""CPU: the two checks of tests/test_gpu_tc_exact.py validated without a GPU.

* The float64 bound of tests/f64_bound.py (``FP16_ROUNDED``) against a tcgen05 'same' block emulated in
  fp32 with the fp16 operand roundings of tc_kernels.cu (A1, U, V and the weights), at C = 32, 64, 128;
  and against the resident form (tc_resident.cu: scale * W3 folded at pack time, branch_conv3
  accumulating into the fp32 residual, bias4 carried as a running sum folded into the next bias1a)
  over a telescoped six-block run, each block checked from the previous block's emulated output.  The
  bound holds and is not vacuous.  It grows with K = 9 C (gamma_K of the 3x3 conv), so at C >= 64 it
  is loose: a fault of a few percent in one tap at the wrapped border row, which err/bound flags at
  C = 16 (tests/test_f64_bound_host.py), stays inside it there.  The exact integer runs are the check
  for such faults; the bound is the check for rounding and activation errors.
* tests/exact_blocks.py: its float64 reference equals an fp32 torch evaluation of the same integer
  blocks bit for bit, and it refuses cases outside the exact regime.
"""
import pytest
import torch
import torch.nn.functional as F

import exact_blocks as X
import f64_bound as B
import vqae_oracle as O
from vqae_b200 import synthetic as S


def _f16(t):
    return t.half().float()


def _perturbed(c, seed):
    from vqae_b200.config import pre_activation_fixup
    from vqae_b200.layers.conv_block import PreActFixupResBlock
    conf = pre_activation_fixup(n_layers=12)
    for k in ("_target_", "_recursive_", "in_channels", "out_channels", "mode"):
        conf.pop(k)
    b = PreActFixupResBlock(in_channels=c, out_channels=c, mode="same", **conf).eval()
    b.load_state_dict(S.make_state_dict(b.state_dict(), seed=seed, regime="perturbed", n_layers=12))
    return {k: v.detach() for k, v in b.state_dict().items()}


def _scalars(p):
    return {k: float(v) for k, v in p.items() if v.numel() == 1}


def _branch_v(a1, p, f):
    w1, w2 = (_f16(p[f"branch_conv{i}.weight"].float()) for i in (1, 2))
    u = _f16(O.elu(F.conv2d(a1, w1) + f["bias2a"]) + f["bias2b"])
    return _f16(O.elu(F.conv2d(F.pad(u, (1, 1, 1, 1), mode="circular"), w2) + f["bias3a"]) + f["bias3b"])


def _emulate_tile(x, p):
    """tc_kernels.cu in fp32: fp16 A1, U, V and weights, out = fmaf(D3, scale, b4) + x."""
    f = _scalars(p)
    v = _branch_v(_f16(O.elu(x + f["bias1a"]) + f["bias1b"]), p, f)
    return x + (F.conv2d(v, _f16(p["branch_conv3.weight"].float())) * f["scale"] + f["bias4"])


# The bound is not vacuous: with the rounding points emulated it only covers accumulation order and the
# fp32 elementwise steps, and its gamma_K term (K = 9 C, worst case) outgrows the actual fp32 sum error
# with C: at C = 128 the emulated error is ~0.5 % of the bound.
_NOT_VACUOUS = {32: 1e-2, 64: 1e-2, 128: 2e-3}


@pytest.mark.parametrize("c", [32, 64, 128])
def test_emulated_tc_same_block_within_bound(c):
    p = _perturbed(c, 60)
    x = torch.randn(2, c, 32, 32, generator=torch.Generator().manual_seed(1))
    ok, ratio, err = B.check(_emulate_tile(x, p), B.fixup_block(x, p, B.FP16_ROUNDED))
    print(f"emulated tcgen05 'same' C{c}: max err/bound {ratio:.3g} (max err {err:.3g})")
    assert ok, ratio
    assert ratio >= _NOT_VACUOUS[c], ratio


@pytest.mark.parametrize("c", [32, 64, 128])
def test_emulated_resident_run_telescoped_within_bound(c):
    """tc_resident.cu in fp32 over six blocks: R = x in tensor memory, A1 = f16(elu(R + (b1a + cum)) +
    b1b), R += V . f16(scale W3), cum += bias4, y_k = R + cum.  Block k + 1 is checked from the
    emulated y_k with the carried error of the store and of cum."""
    ps = [_perturbed(c, 100 + k) for k in range(6)]
    x = torch.randn(2, c, 32, 32, generator=torch.Generator().manual_seed(2))
    r, cum = x.clone(), torch.zeros((), dtype=torch.float32)
    ys, b4s = [x], []
    for p in ps:
        f = _scalars(p)
        pre = torch.tensor(f["bias1a"], dtype=torch.float32) + cum
        v = _branch_v(_f16(O.elu(r + pre) + f["bias1b"]), p, f)
        w3s = _f16(p["branch_conv3.weight"].float() * torch.tensor(f["scale"], dtype=torch.float32))
        r = r + F.conv2d(v, w3s)
        cum = cum + torch.tensor(f["bias4"], dtype=torch.float32)
        ys.append(r + cum)
    worst = 0.0
    for k, p in enumerate(ps):
        xin, cum_mag = B.resident_carry(ys[k], b4s)
        ref = B.fixup_block(xin, p, B.FP16_ROUNDED, fold_scale=True, residual_in_acc=True,
                            cum_mag=cum_mag)
        ok, ratio, _ = B.check(ys[k + 1], ref)
        assert ok, (k, ratio)
        worst = max(worst, ratio)
        b4s.append(float(p["bias4"]))
    print(f"emulated resident C{c}, 6 blocks telescoped: max err/bound {worst:.3g}")
    assert worst >= _NOT_VACUOUS[c], worst


def _fp32_torch_run(x_nhwc, blocks):
    """The integer blocks in plain fp32 torch (NCHW convs, circular padding), fp16 operand roundings."""
    h = x_nhwc.permute(0, 3, 1, 2).float()
    for p in blocks:
        f = _scalars(p)
        a1 = _f16(O.elu(h + f["bias1a"]) + f["bias1b"])
        v = _branch_v(a1, p, f)
        h = h + (F.conv2d(v, p["branch_conv3.weight"]) * f["scale"] + f["bias4"])
    return h.permute(0, 2, 3, 1)


@pytest.mark.parametrize("c,hw,n", [(32, 64, 5), (64, 32, 12)])
def test_exact_reference_is_fp32_torch_bit_for_bit(c, hw, n):
    blocks = X.integer_blocks(c, n, seed=1)
    x = X.integer_input((3, hw, hw, c), seed=1)
    st = X.Stats()
    ref = X.reference(x, blocks, st)
    assert ref.dtype == torch.float32
    assert torch.equal(ref, _fp32_torch_run(x, blocks))
    assert st.rounded > 0, "the case never exercises an fp16 rounding point"
    # each half of the run reads one half of the channels and writes the other
    w1 = torch.stack([p["branch_conv1.weight"][:, :, 0, 0] for p in blocks])
    w3 = torch.stack([p["branch_conv3.weight"][:, :, 0, 0] for p in blocks])
    half = (n + 1) // 2
    reads = w1[:half].abs().sum((0, 1)) > 0
    writes = w3[:half].abs().sum((0, 2)) > 0
    assert not bool((reads & writes).any())


def test_exact_reference_refuses_cases_outside_the_exact_regime():
    blocks = X.integer_blocks(32, 2, seed=3)
    x = X.integer_input((1, 32, 32, 32), seed=3)
    X.reference(x, blocks)
    with pytest.raises(X.NotExact, match="non-integer"):
        X.reference(x + 0.5, blocks)
    with pytest.raises(X.NotExact, match="fp16 overflow"):
        X.reference(x + 70000.0, blocks)
    low = [dict(p) for p in blocks]
    low[1]["bias2a"] = torch.tensor([0.0])                 # U on the exponential branch of the ELU
    with pytest.raises(X.NotExact, match="pre-activation"):
        X.reference(x, low)
    big = [dict(p) for p in blocks]
    big[0]["branch_conv2.weight"] = torch.ones_like(big[0]["branch_conv2.weight"]) * 4096
    with pytest.raises(X.NotExact, match="2\\^24"):
        X.reference(x, big)
