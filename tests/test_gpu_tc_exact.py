"""GPU: the tcgen05 'same' kernels block by block -- the image-resident trunk (tc_resident.cu), the
persistent tile chain (tc_chain.cu) and the tile kernel (tc_kernels.cu).

1. Exact integer runs (tests/exact_blocks.py): weights in {-1, 0, 1}, integer biases and inputs, on
   which every fp32 operation of these kernels is exact.  Every image of every launch must equal the
   float64 reference bit for bit, so a fault in one block, one weight slot, one image slot, one halo
   row or one image switch of a 54-block run shows, however small.  Saturated launches (>= 3 units
   per CTA or cluster), ragged ones (the last wave partial, for the resident kernel with one image
   slot of the last cluster idle) and single images.  A negative control changes one weight or one
   bias4 of block 37 in the packed data and checks that the exact comparison fails while the older
   max-normalised 1e-2 bar of tests/test_gpu_tc.py does not see it.
2. A per-element float64 bound with real (perturbed) weights, telescoped: every prefix of the run is
   launched, and block k + 1 of the kernel is checked against tests/f64_bound.py applied to the
   kernel's own output after k blocks.  This checks each block of a 54-block run with a one-block bound
   that does not grow with depth, and covers what the integer runs cannot: the ELU's exponential
   branch, ex2.approx, the rounding points and the bias folds.

The profiler's kernel names confirm which kernel ran, and the launch grids (from the profiler trace)
give the units per CTA or cluster that the test prints.
"""
import json
import tempfile
from pathlib import Path

import pytest
import torch

import exact_blocks as X
import f64_bound as FB
from vqae_b200 import _lib as L
from vqae_b200 import engine as E
from vqae_b200 import synthetic as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _modules(c, params):
    """'same' PreActFixupResBlocks on the GPU: an integer_blocks entry, or a seed for perturbed weights."""
    from vqae_b200.config import pre_activation_fixup
    from vqae_b200.layers.conv_block import PreActFixupResBlock
    conf = pre_activation_fixup(n_layers=12)
    for k in ("_target_", "_recursive_", "in_channels", "out_channels", "mode"):
        conf.pop(k)
    out = []
    for p in params:
        blk = PreActFixupResBlock(in_channels=c, out_channels=c, mode="same", **conf).eval()
        if isinstance(p, dict):
            X.load_block(blk, p)
        else:
            blk.load_state_dict(S.make_state_dict(blk.state_dict(), seed=p, regime="perturbed", n_layers=12))
        out.append(blk.to(DEV))
    return out


# kernel -> (kind, C, H = W, blocks, batches of the exact runs ("ragged": derived from the saturated grid),
#            profiler name)
CASES = {
    "resident64": ("resident", 64, 32, 54, (256, "ragged", 1), "trunk_resident_tc_kernel<64, 32>"),
    "resident128": ("resident", 128, 32, 54, (100, 1), "trunk_resident_tc_kernel<128, 32>"),
    "resident32": ("resident", 32, 64, 5, (256, "ragged", 1), "trunk_resident_tc_kernel<32, 64>"),
    "chain64_64": ("chain", 64, 64, 5, (64,), "same_chain_tc_kernel<64, 64, 16>"),
    "chain64_32": ("chain", 64, 32, 54, (256,), "same_chain_tc_kernel<64, 64, 16>"),
    "chain128_32": ("chain", 128, 32, 3, (40, 3), "same_chain_tc_kernel<128, 128, 8>"),
    "chain128_64": ("chain", 128, 64, 1, (40, 3), "same_chain_tc_kernel<128, 128, 8>"),
    "tile32_128": ("tile", 32, 128, 5, (64, 1), "same_block_tc_kernel<32, 32"),
    "tile64_64": ("tile", 64, 64, 5, (64, 19), "same_block_tc_kernel<64, 64"),
}
CLUSTER = {64: 4, 128: 4, 32: 8}                      # RsCfg<C, W>::CL: one cluster per image
NSLOT = {64: 2, 128: 1, 32: 2}                        # RsCfg<C, W>::NSLOT: images per cluster at once


def _launcher(kind, packed):
    """x -> y through one kernel: the resident kernel and the tile chain through their ABI (a single
    launch for any run length), the tile kernel block by block."""
    lib = L.load()
    if kind == "resident":
        chain = E.PackedChain(packed, resident=True)

        def run(x, out=None):
            out = torch.empty_like(x) if out is None else out
            E.trunk_resident(x, out, chain)
            return out
        return run
    if kind == "chain":
        chain = E.PackedChain(packed)

        def run(x):
            b, h, w, c = x.shape
            bufs = [torch.empty_like(x), torch.empty_like(x)]
            fbytes = lib.vqae_same_chain_flag_bytes(chain.n, b)
            flags = torch.empty(fbytes, dtype=torch.uint8, device=x.device)
            L.check(lib.vqae_same_chain_f16(E._ptr(x), E._ptr(bufs[0]), E._ptr(bufs[1]), E._ptr(chain.weights),
                                            E._ptr(chain.scalars), E._ptr(flags), fbytes, chain.n, b, h, w, c,
                                            E._stream(x.device)), "vqae_same_chain_f16")
            return bufs[(chain.n - 1) & 1]
        return run

    def run(x):
        for pk in packed:
            x = E.fixup_forward_nhwc(pk, x, precision="fp16")
        return x
    return run


def _profiled(fn, *args):
    """fn(*args) under torch.profiler: (result, {kernel name without spaces: [grid.x of each launch]})."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        y = fn(*args)
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = Path(d) / "trace.json"
        prof.export_chrome_trace(str(path))
        events = json.loads(path.read_text())["traceEvents"]
    grids = {}
    for e in events:
        if e.get("cat") == "kernel":
            grids.setdefault(e["name"].replace(" ", ""), []).append(e.get("args", {}).get("grid", [0])[0])
    return y, grids


def _grid_of(grids, kname):
    hits = [g for n, gs in grids.items() if kname.replace(" ", "") in n for g in gs]
    assert hits, (kname, sorted(grids))
    assert all(g > 0 for g in hits), ("no grid in the profiler trace", kname)
    return hits


def _units(kind, c, hw, n, b, grid):
    """(units, units per CTA or cluster) of one launch with this grid (tc_resident.cu:268-282,
    tc_chain.cu:416-439, tc_kernels.cu:410-422)."""
    if kind == "resident":
        clusters = grid // CLUSTER[c]
        groups = -(-b // NSLOT[c])
        return groups, groups / clusters, clusters
    th = 8 if kind == "chain" and c == 128 else 16
    units = b * (hw // th) * (hw // 32) * (n if kind == "chain" else 1)
    return units, units / grid, grid


def _where(y, ref):
    """Where two NHWC batches differ: images, rows, columns, channels (first few of each)."""
    bad = (y != ref).nonzero()
    return {k: sorted(set(bad[:, i].tolist()))[:12] for i, k in enumerate(("image", "row", "col", "channel"))}


def _assert_exact(y, ref, what):
    torch.cuda.synchronize()
    bad = [i for i in range(y.shape[0]) if not torch.equal(y[i], ref[i])]
    assert not bad, f"{what}: {len(bad)} of {y.shape[0]} images differ from the exact reference; " \
                    f"{_where(y, ref)}, max |diff| {float((y.double() - ref.double()).abs().max())}"


def _old_bar(y, ref, x):
    """tests/test_gpu_tc.py's bar: max |y - ref| over the branch maximum."""
    return float((y.double() - ref.double()).abs().max()) / float((ref.double() - x.double()).abs().max())


@pytest.mark.parametrize("case", sorted(CASES))
def test_integer_run_exact(case):
    kind, c, hw, n, batches, kname = CASES[case]
    params = X.integer_blocks(c, n, seed=c + hw + n)
    packed = E.pack_blocks(_modules(c, params))
    run = _launcher(kind, packed)
    if kind == "resident":
        assert L.load().vqae_trunk_resident_supported(256, hw, hw, c)
    elif kind == "chain":
        assert c == 128 or L.load().vqae_same_chain_supported(batches[0], hw, hw, c)
    sat_clusters = None
    for b in batches:
        if b == "ragged":
            # the last wave holds one image group, and that group has one image slot idle
            b = NSLOT[c] * (3 * sat_clusters + 1) - 1
        x = X.integer_input((b, hw, hw, c), seed=b).to(DEV)
        st = X.Stats()
        ref = X.reference(x, params, st)
        y, grids = _profiled(run, x)
        gl = _grid_of(grids, kname)
        assert len(gl) == (n if kind == "tile" else 1)
        units, per, slots = _units(kind, c, hw, n, b, gl[0])
        if b == batches[0]:
            sat_clusters = slots
            assert per >= 3, (units, slots)
        _assert_exact(y, ref, f"{case} B={b}")
        print(f"{case} B={b}: {units} units on {slots} {'clusters' if kind == 'resident' else 'CTAs'} "
              f"= {per:.2f} per {'cluster' if kind == 'resident' else 'CTA'} (last wave {units % slots}); "
              f"max operand {st.max_operand:.0f}, {st.rounded} operand values rounded to fp16")
        if kind == "resident" and b == batches[0]:
            # fp16 stream: loaded and stored as fp16, fp32 on chip
            xh = x.half()
            _assert_exact(run(xh), X.reference(xh, params, half_io=True), f"{case} B={b} fp16 I/O")
            if c == 64:
                xc = x.clone()
                run(xc, xc)                              # out aliases x
                _assert_exact(xc, ref, f"{case} B={b} in place")
        del x, y, ref


@pytest.mark.parametrize("fault", ["weight", "bias4"])
def test_integer_run_negative_control(fault):
    """The exact comparison sees one changed weight or one bias4 off by one in block 37 of 54 (the data
    is changed, not the kernel); the older max-normalised bar of tests/test_gpu_tc.py does not."""
    c, hw, n, b, blk = 64, 32, 54, 256, 37
    params = X.integer_blocks(c, n, seed=c + hw + n)
    packed = E.pack_blocks(_modules(c, params))
    chain = E.PackedChain(packed, resident=True)
    x = X.integer_input((b, hw, hw, c), seed=b).to(DEV)
    ref = X.reference(x, params)
    y = torch.empty_like(x)
    E.trunk_resident(x, y, chain)
    _assert_exact(y, ref, "clean run")
    if fault == "weight":
        # scale * W3 of block 37 (matrix 10, canonical [k-chunk][n][8]): output channel o gains V
        # channel k, where W3 was zero and V_k is not constant (its W2 row is not empty)
        w2 = params[blk]["branch_conv2.weight"]
        w3 = params[blk]["branch_conv3.weight"][:, :, 0, 0]
        k = int((w2.abs().sum((1, 2, 3)) > 0).nonzero()[0])
        o = int((w3[:, k] == 0).nonzero()[0])
        r = (k // 8) * c * 8 + o * 8 + k % 8
        base = (blk * 11 + 10) * c * c
        assert float(chain.weights[base + r]) == 0.0
        chain.weights[base + r] = 1.0
    else:
        chain.scalars[blk, 6] += 1.0                    # bias4 of block 37 (scalars [b1a..b3b, b4, scale])
    E.trunk_resident(x, y, chain)
    torch.cuda.synchronize()
    bad = [i for i in range(b) if not torch.equal(y[i], ref[i])]
    old = _old_bar(y, ref, x)
    print(f"negative control ({fault} of block {blk}): {len(bad)} of {b} images differ from the exact "
          f"reference; old bar: max |diff| / branch max = {old:.2e} (limit 1e-2)")
    assert len(bad) == b
    assert old < 1e-2


# ---- per-element float64 bound, telescoped --------------------------------------------------------------
# kernel -> (kind, C, H = W, blocks, batch)
BOUND_CASES = {
    "resident64": ("resident", 64, 32, 54, 256),
    "resident128": ("resident", 128, 32, 54, 100),
    "resident32": ("resident", 32, 64, 5, 256),
    "chain64": ("chain", 64, 32, 54, 256),
    "chain128": ("chain", 128, 32, 3, 40),
    "tile32": ("tile", 32, 128, 5, 64),
    "tile64": ("tile", 64, 64, 5, 64),
}


@pytest.mark.parametrize("case", sorted(BOUND_CASES))
def test_real_weights_telescoped_f64_bound(case):
    """y_{k+1} of the kernel against the bound of block k + 1 applied to the kernel's own y_k, element by
    element (<= 2 bound) at the first, middle and last image.  The resident kernel never stores y_k
    inside a run, so each prefix of the run is launched on its own; its input carries the error of the
    fp32 store and of the running bias4 sum (f64_bound.resident_carry).  The tile chain and the tile
    kernel store every block's output in fp32, so their y_k is exact input."""
    kind, c, hw, n, b = BOUND_CASES[case]
    blocks = _modules(c, [60 + k for k in range(n)])
    packed = E.pack_blocks(blocks)
    params = [{k: v.detach() for k, v in blk.state_dict().items()} for blk in blocks]
    x = torch.randn(b, hw, hw, c, generator=torch.Generator().manual_seed(c + n)).to(DEV)
    idx = sorted({0, b // 2, b - 1})
    ys = [x[idx]]
    if kind == "tile":
        h = x
        for pk in packed:
            h = E.fixup_forward_nhwc(pk, h, precision="fp16")
            ys.append(h[idx])
    else:
        for k in range(1, n + 1):
            ys.append(_launcher(kind, packed[:k])(x)[idx])
    torch.cuda.synchronize()
    nchw = lambda t: t.permute(0, 3, 1, 2)                                   # noqa: E731
    worst, b4s = 0.0, []
    for k, p in enumerate(params):
        if kind == "resident":
            xin, cum = FB.resident_carry(nchw(ys[k]), b4s)
            ref = FB.fixup_block(xin, p, FB.FP16_ROUNDED, fold_scale=True, residual_in_acc=True, cum_mag=cum)
        else:
            ref = FB.fixup_block(nchw(ys[k]), p, FB.FP16_ROUNDED)
        ok, ratio, err = FB.check(nchw(ys[k + 1]), ref)
        if not ok:
            bad = ((nchw(ys[k + 1]).double() - ref.v).abs() > 2 * ref.e).nonzero()
            raise AssertionError(f"{case}: block {k} outside 2 x bound (err/bound {ratio:.3g}, err {err:.3g}) "
                                 f"at images {sorted(set(bad[:, 0].tolist()))}, rows {sorted(set(bad[:, 2].tolist()))[:12]}, "
                                 f"cols {sorted(set(bad[:, 3].tolist()))[:12]}")
        worst = max(worst, ratio)
        b4s.append(float(p["bias4"]))
    print(f"{case}: {n} blocks telescoped at B={b}, max err/bound {worst:.3g}")
