"""Host-side execution of the hot path over the C-ABI library.

torch is plumbing here: device memory (``torch.empty``), the current CUDA stream, and
``state_dict`` tensors.  Every FLOP is issued through ``libvqae_b200.so``.  There is no CPU
path: tensors that are not on a CUDA device raise.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib as L

Tensor = torch.Tensor

# near-tie threshold on the relative top-2 gap of the un-rooted L4 sums (DESIGN.md section 4)
NEAR_TIE_REL_GAP = 16.0 * 2.0 ** -23

CAMELYON16_MEAN = (0.7279, 0.5955, 0.7762)   # conf/transforms/camelyon16_transforms.yaml:15-23
CAMELYON16_STD = (0.2419, 0.3083, 0.1741)


def _ptr(t: Optional[Tensor]) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def _stream(device: torch.device) -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def require_cuda(t: Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{what}: tensor is on {t.device}; the B200 path has no CPU fallback "
            "(move the module and its inputs to a CUDA device)")


_workspaces: Dict[Tuple[int, int], Tensor] = {}


def workspace(device: torch.device, nbytes: int) -> Tensor:
    """Grow-only scratch buffer per (device, stream).  While the current stream is being captured
    into a CUDA graph the buffer comes from the graph's own memory pool instead (one allocation per
    call, released to that pool after the call): a cached buffer that is replaced by a larger one in the
    middle of a capture would be freed while earlier nodes of the graph still point into it."""
    if torch.cuda.is_current_stream_capturing():
        return torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream)
    buf = _workspaces.get(key)
    if buf is None or buf.numel() < nbytes:
        buf = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = buf
    return buf


def is_channels_last(x: Tensor) -> bool:
    return (x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last)
            and not x.is_contiguous())


def to_nhwc(x: Tensor) -> Tuple[Tensor, bool]:
    """[B,C,H,W] (any strides) -> contiguous [B,H,W,C] fp32, and whether x was channels_last."""
    cl = is_channels_last(x)
    y = x.permute(0, 2, 3, 1)
    if y.dtype != torch.float32:
        y = y.float()
    return y.contiguous(), cl


def from_nhwc(y: Tensor, channels_last: bool) -> Tensor:
    """contiguous [B,H,W,C] -> NCHW-shaped tensor whose strides follow the caller's format."""
    v = y.permute(0, 3, 1, 2)
    return v if channels_last else v.contiguous()


# ----------------------------------------------------------------------------------------------
# weight packing
# ----------------------------------------------------------------------------------------------
def pack_conv_weight(w: Tensor) -> Tensor:
    """OIHW fp32 -> [KH*KW][I][O] fp32 on the device (vqae_pack_conv_weight_f32)."""
    require_cuda(w, "pack_conv_weight")
    w = w.detach().float().contiguous()
    o, i, kh, kw = w.shape
    out = torch.empty(kh * kw, i, o, dtype=torch.float32, device=w.device)
    lib = L.load()
    L.check(lib.vqae_pack_conv_weight_f32(_ptr(w), _ptr(out), o, i, kh, kw, _stream(w.device)),
            "vqae_pack_conv_weight_f32")
    return out


_SCALARS = ("bias1a", "bias1b", "bias2a", "bias2b", "bias3a", "bias3b", "bias4", "scale",
            "bias1c", "bias1d")


def infer_block_mode(block) -> str:
    """'same' / 'down' / 'up' from the structure of a PreActFixupResBlock -- the reference's
    class does not keep its ``mode`` argument (conv_block.py:136-194), so this also serves blocks
    instantiated by the unmodified reference (vqae_b200.accelerate)."""
    c2 = block.branch_conv2
    k2, st = tuple(c2.kernel_size), tuple(c2.stride)
    if hasattr(c2, "upsample") and k2 == (1, 1):
        return "up"
    if k2 == (2, 2) and st == (2, 2):
        return "down"
    if k2 == (3, 3) and st == (1, 1) and c2.padding_mode == "circular":
        return "same"
    raise NotImplementedError(f"PreActFixupResBlock with branch_conv2 {c2} is not built")


def check_block_supported(block) -> None:
    """Everything the kernels assume about a block, checked against the module itself
    (conf/model/layers/conv_block/pre_activation_fixup.yaml)."""
    from torch import nn
    act = block.activation
    if not (isinstance(act, nn.ELU) and act.alpha == 1.0):
        raise NotImplementedError("only nn.ELU(alpha=1) activations are built "
                                  "(conf/model/layers/activation/elu.yaml)")
    convs = (block.branch_conv1, block.branch_conv2, block.branch_conv3, block.skip_conv)
    for conv in convs:
        if conv is None:
            continue
        if conv.bias is not None:
            raise NotImplementedError("branch/skip convs with bias are not built "
                                      "(pre_activation_fixup.yaml sets bias: False)")
        if conv.groups != 1 or tuple(conv.dilation) != (1, 1):
            raise NotImplementedError(f"grouped / dilated conv {conv} is not built")
    for name in ("branch_conv1", "branch_conv3"):
        conv = getattr(block, name)
        if tuple(conv.kernel_size) != (1, 1) or tuple(conv.stride) != (1, 1) \
                or hasattr(conv, "upsample"):
            raise NotImplementedError(f"{name} {conv} is not a plain 1x1 conv")
    mode = infer_block_mode(block)
    declared = getattr(block, "mode", mode)
    if declared != mode:
        raise NotImplementedError(f"mode {declared!r} with branch_conv2 {block.branch_conv2} "
                                  "is not built")
    cb, ci, co = (block.branch_conv1.out_channels, block.branch_conv1.in_channels,
                  block.branch_conv3.out_channels)
    if block.branch_conv2.in_channels != cb or block.branch_conv2.out_channels != cb \
            or block.branch_conv3.in_channels != cb:
        raise NotImplementedError("branch convs with mismatched widths are not built")
    sk = block.skip_conv
    if mode == "same":
        if sk is not None or ci != co:
            raise NotImplementedError("'same' blocks that change the channel count are not built")
    else:
        if sk is None:
            raise NotImplementedError(f"'{mode}' block without skip_conv is not built")
        ks, ss = tuple(sk.kernel_size), tuple(sk.stride)
        ok = (mode == "down" and ks == (2, 2) and ss == (2, 2)) or \
             (mode == "up" and ks == (1, 1) and ss == (1, 1) and hasattr(sk, "upsample"))
        if not ok or sk.in_channels != ci or sk.out_channels != co:
            raise NotImplementedError(f"mode {mode!r} with skip_conv {sk} is not built")


class PackedFixup:
    """Packed weights + the C struct of one PreActFixupResBlock.  Packing is lazy and batched:
    ``ensure_packed`` fills the fp32 and/or tensor-core layouts of any number of blocks with ONE
    launch of vqae_pack_batched."""

    def __init__(self, block, scalars: Sequence[float]):
        w2 = block.branch_conv2.weight
        self.mode = {"same": L.MODE_SAME, "down": L.MODE_DOWN, "up": L.MODE_UP}[
            infer_block_mode(block)]
        self.c_in = block.branch_conv1.weight.shape[1]
        self.c_branch = block.branch_conv1.weight.shape[0]
        self.c_out = block.branch_conv3.weight.shape[0]
        self.device = w2.device
        # fp32 contiguous sources, kept alive until (and after) the asynchronous pack has read them
        self.src = [t.detach().float().contiguous() for t in
                    (block.branch_conv1.weight, w2, block.branch_conv3.weight)]
        self.src.append(block.skip_conv.weight.detach().float().contiguous()
                        if block.skip_conv is not None else None)
        self.scalars = dict(zip(_SCALARS, scalars))
        sc = self.scalars
        p = L.FixupParams()
        p.mode, p.c_in, p.c_out, p.c_branch = self.mode, self.c_in, self.c_out, self.c_branch
        for name, val in sc.items():
            setattr(p, name, float(val))
        self.params = p
        self.w1 = self.w2 = self.w3 = self.w_skip = None           # fp32 [tap][I][O] packs
        # tcgen05 path: bf16 operand packs
        self.tc_weights = self.tc_weights_res = self.mma_weights = None
        self.tc_scalars = None
        self.tc_kind = None
        # fp32-accurate tensor-core mode ("fp32tc"): split fp16 operand packs (hi, lo), the powers
        # of two the matrices were multiplied by, and max|w| of the four convs they derive from
        self.split_hi = self.split_lo = self.split_premul = None
        self.split_mma_hi = self.split_mma_lo = None       # C = 8, 16 'same': warp-MMA layout
        self.wmax: Optional[List[float]] = None
        if self.mode == L.MODE_SAME and self.c_in in (8, 16, 32, 64, 128) and \
                self.c_branch == self.c_in and self.c_out == self.c_in:
            self.tc_kind = "same"
            self.tc_scalars = (C.c_float * 8)(*[float(sc[k]) for k in (
                "bias1a", "bias1b", "bias2a", "bias2b", "bias3a", "bias3b", "bias4", "scale")])
        elif self.mode == L.MODE_UP and self.c_in in (16, 32, 64, 128) and \
                self.c_branch == self.c_in and self.c_out * 2 == self.c_in:
            self.tc_kind = "up"
            self.tc_scalars = (C.c_float * 8)(*(
                [float(sc[k]) for k in ("bias1a", "bias1b", "bias2a", "bias2b", "bias3a",
                                        "bias3b", "bias1c")]
                + [float(sc["bias4"]) + float(sc["bias1d"])]))
        elif self.mode == L.MODE_DOWN and self.c_in in (8, 16, 32, 64) and \
                self.c_branch == 2 * self.c_in and self.c_out == 2 * self.c_in:
            self.tc_kind = "down"
            self.tc_scalars = (C.c_float * 8)(*(
                [float(sc[k]) for k in ("bias1a", "bias1b", "bias2a", "bias2b", "bias3a",
                                        "bias3b", "bias1c")]
                + [float(sc["bias4"]) + float(sc["bias1d"])]))

    @property
    def has_resident(self) -> bool:
        return self.tc_kind == "same" and self.c_in in (32, 64, 128)

    # -- descriptors of the packs that are still missing ----------------------------------------
    def _desc(self, kind, dst, c_in, c_out, taps, srcs, scale=1.0):
        d = L.PackDesc()
        d.kind, d.c_in, d.c_out, d.taps, d.scale = kind, c_in, c_out, taps, float(scale)
        d.n_elems = dst.numel()
        for i, t in enumerate(srcs):
            d.src[i] = t.data_ptr() if t is not None else None
        d.dst = dst.data_ptr()
        return d

    def descs_f32(self) -> List["L.PackDesc"]:
        if self.w1 is not None:
            return []
        out, packs = [], []
        for t in self.src:
            if t is None:
                packs.append(None)
                continue
            o, i, kh, kw = t.shape
            dst = torch.empty(kh * kw, i, o, dtype=torch.float32, device=self.device)
            out.append(self._desc(L.PACK_F32_CONV, dst, i, o, kh * kw, [t]))
            packs.append(dst)
        self.w1, self.w2, self.w3, self.w_skip = packs
        p = self.params
        p.w1, p.w2, p.w3 = self.w1.data_ptr(), self.w2.data_ptr(), self.w3.data_ptr()
        p.w_skip = self.w_skip.data_ptr() if self.w_skip is not None else None
        return out

    def descs_tc(self) -> List["L.PackDesc"]:
        if self.tc_kind is None or self.tc_weights is not None:
            return []
        lib = L.load()
        out = []
        sc = self.scalars
        if self.tc_kind == "same":
            n = lib.vqae_pack_elems(L.PACK_SAME_F16, self.c_in, self.c_in, 9)
            self.tc_weights = torch.empty(n, dtype=torch.float16, device=self.device)
            out.append(self._desc(L.PACK_SAME_F16, self.tc_weights, self.c_in, self.c_in, 9,
                                  self.src[:3]))
            if self.c_in in (8, 16, 32):
                # low-channel form on warp-level MMAs (mma_same.cu): plain [11][n][k]
                self.mma_weights = torch.empty(11 * self.c_in * self.c_in, dtype=torch.float16,
                                               device=self.device)
                out.append(self._desc(L.PACK_SAME_MMA_F16, self.mma_weights, self.c_in, self.c_in, 9,
                                      self.src[:3]))
            if self.has_resident:
                # image-resident trunk kernel: branch_conv3 pre-multiplied by the Fixup scale
                self.tc_weights_res = torch.empty(n, dtype=torch.float16, device=self.device)
                out.append(self._desc(L.PACK_RESIDENT_F16, self.tc_weights_res, self.c_in,
                                      self.c_in, 9, self.src[:3], sc["scale"]))
        elif self.tc_kind == "up":
            n = lib.vqae_pack_elems(L.PACK_UP_MMA_F16, self.c_in, self.c_out, 1)
            self.tc_weights = self.mma_weights = torch.empty(n, dtype=torch.float16,
                                                             device=self.device)
            out.append(self._desc(L.PACK_UP_MMA_F16, self.mma_weights, self.c_in, self.c_out, 1,
                                  [self.src[0], self.src[1], self.src[2], self.src[3]], sc["scale"]))
        else:
            n = lib.vqae_pack_elems(L.PACK_DOWN_F16, self.c_in, self.c_out, 4)
            self.tc_weights = torch.empty(n, dtype=torch.float16, device=self.device)
            out.append(self._desc(L.PACK_DOWN_F16, self.tc_weights, self.c_in, self.c_out, 4,
                                  self.src, sc["scale"]))
            if self.c_in in DOWN_MMA:
                n = lib.vqae_pack_elems(L.PACK_DOWN_MMA_F16, self.c_in, self.c_out, 4)
                self.mma_weights = torch.empty(n, dtype=torch.float16, device=self.device)
                out.append(self._desc(L.PACK_DOWN_MMA_F16, self.mma_weights, self.c_in, self.c_out, 4,
                                      self.src, sc["scale"]))
        return out

    def split_ok(self, h: int, w: int) -> bool:
        """a split-operand (fp32-accurate) tensor-core kernel is built for this block and size"""
        lib = L.load()
        if self.tc_kind == "same" and self.c_in in (8, 16, 32, 64):
            return bool(lib.vqae_same_block_split_supported(h, w, self.c_in))
        if self.tc_kind == "down" and self.c_in in (8, 16, 32):
            return bool(lib.vqae_down_block_mma_supported(h, w, self.c_in))
        return False

    def descs_split(self) -> List["L.PackDesc"]:
        if self.split_hi is not None or self.tc_kind not in ("same", "down"):
            return []
        assert self.wmax is not None, "ensure_wmax first"
        lib = L.load()

        def pm(m: float) -> float:
            # power of two that moves max|w| into (2^13, 2^14]: every low half f16(w - f16(w)) of a
            # weight within 2^-27 of the largest one is then a normal fp16 number
            return 1.0 if not (m > 0.0 and math.isfinite(m)) else 2.0 ** (14 - math.ceil(math.log2(m)))
        w1m, w2m, w3m, wsm = self.wmax
        if self.tc_kind == "same":
            kind, taps, srcs, scale = L.PACK_SAME_F16, 9, self.src[:3], 1.0
            premul = [pm(w1m), pm(w2m), pm(w3m), 1.0]
        else:
            kind, taps, srcs, scale = L.PACK_DOWN_MMA_F16, 4, self.src, self.scalars["scale"]
            p3 = pm(max(w3m * abs(scale), wsm))      # branch_conv3 and skip_conv share an accumulator
            premul = [pm(w1m), pm(w2m), p3, p3]
        n = lib.vqae_pack_elems(kind, self.c_in, self.c_out, taps)
        self.split_hi = torch.empty(n, dtype=torch.float16, device=self.device)
        self.split_lo = torch.empty(n, dtype=torch.float16, device=self.device)
        self.split_premul = (C.c_float * 3)(*premul[:3])
        out = []
        packs = [(kind, self.split_hi, self.split_lo)]
        if self.tc_kind == "same" and self.c_in in SPLIT_MMA:
            n2 = 11 * self.c_in * self.c_in
            self.split_mma_hi = torch.empty(n2, dtype=torch.float16, device=self.device)
            self.split_mma_lo = torch.empty(n2, dtype=torch.float16, device=self.device)
            packs.append((L.PACK_SAME_MMA_F16, self.split_mma_hi, self.split_mma_lo))
        for k, hi, lo in packs:
            for dst, flag in ((hi, 0), (lo, L.PACK_LO)):
                d = self._desc(k | flag, dst, self.c_in, self.c_out, taps, srcs, scale)
                for i, v in enumerate(premul):
                    d.premul[i] = v
                out.append(d)
        return out

    def tc_ok(self, h: int, w: int) -> bool:
        """a tcgen05 kernel is built for this block at this size (16 x 32 pixel tiles; 8 x 32 for
        the C = 128 'same' blocks, which only exist in the persistent chain form)"""
        if self.tc_kind == "up":
            return bool(L.load().vqae_up_block_mma_supported(h, w, self.c_in))
        if self.tc_kind is None or w % 32:
            return False
        return h % 8 == 0 if self.chain_only else h % 16 == 0

    @property
    def chain_only(self) -> bool:
        return self.mode == L.MODE_SAME and self.c_in == 128

    def out_hw(self, h: int, w: int) -> Tuple[int, int]:
        if self.mode == L.MODE_DOWN:
            return h // 2, w // 2
        if self.mode == L.MODE_UP:
            return 2 * h, 2 * w
        return h, w


def block_version(block) -> Tuple:
    return tuple((p.data_ptr(), p._version) for p in block.parameters())


def pack_blocks(blocks: Sequence) -> List[PackedFixup]:
    """Pack a list of PreActFixupResBlocks; scalar parameters are read with ONE host copy."""
    if not blocks:
        return []
    dev = blocks[0].bias1a.device
    zero = torch.zeros(1, device=dev)
    cols = []
    for b in blocks:
        for name in _SCALARS:
            t = getattr(b, name, None)
            cols.append(t.detach().float().reshape(1) if t is not None else zero)
    host = torch.cat(cols).cpu().tolist()
    n = len(_SCALARS)
    return [PackedFixup(b, host[i * n:(i + 1) * n]) for i, b in enumerate(blocks)]


def ensure_wmax(packed: Sequence[PackedFixup]) -> None:
    """max|w| of every conv of the blocks that do not have it yet, with ONE host copy."""
    todo = [pk for pk in packed if pk.wmax is None]
    if not todo:
        return
    zero = torch.zeros((), device=todo[0].device)
    vals = torch.stack([t.abs().max() if t is not None else zero for pk in todo for t in pk.src])
    host = vals.cpu().tolist()
    for i, pk in enumerate(todo):
        pk.wmax = host[4 * i:4 * i + 4]


def ensure_packed(packed: Sequence[PackedFixup], f32: Sequence[bool], tc: Sequence[bool],
                  split: Optional[Sequence[bool]] = None) -> None:
    """Pack whatever is still missing for the requested layouts -- one vqae_pack_batched launch."""
    descs, keep = [], []
    if split is not None and any(split):
        ensure_wmax([pk for pk, want in zip(packed, split) if want and pk.split_hi is None])
    for i, (pk, want_f32, want_tc) in enumerate(zip(packed, f32, tc)):
        if want_f32:
            descs += pk.descs_f32()
        if want_tc:
            descs += pk.descs_tc()
        if split is not None and split[i]:
            descs += pk.descs_split()
    if not descs:
        return
    dev = packed[0].device
    arr = (L.PackDesc * len(descs))(*descs)
    table = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).to(dev)
    L.check(L.load().vqae_pack_batched(_ptr(table), len(descs), max(d.n_elems for d in descs),
                                       _stream(dev)), "vqae_pack_batched")
    # the table is read by the kernel asynchronously: keep it until the stream has passed it
    table.record_stream(torch.cuda.current_stream(dev))


def _plan_layouts(packed: Sequence[PackedFixup], h: int, w: int, precision: str):
    """(needs fp32 pack, needs tensor-core pack, needs split-operand pack) per block for an input
    of h x w."""
    f32, tc, split = [], [], []
    for pk in packed:
        use_tc = precision == "fp16" and pk.tc_ok(h, w)
        use_split = precision == "fp32tc" and pk.split_ok(h, w)
        tc.append(use_tc)
        split.append(use_split)
        f32.append(not (use_tc or use_split))
        h, w = pk.out_hw(h, w)
    return f32, tc, split


# ----------------------------------------------------------------------------------------------
# single calls
# ----------------------------------------------------------------------------------------------
# "fp32": CUDA-core exact path.  "fp16": tensor-core kernels with fp16 operands (what an active
# torch.autocast('cuda') selects).  "fp32tc": tensor-core kernels with split fp16 operands
# (hi + lo, three products each, exact activations) -- fp32-accurate, the reference's fp32 index
# contract holds outside near-ties (csrc/tc_split.cu).
PRECISIONS = ("fp32", "fp16", "fp32tc")
# 'same' blocks of these widths run on warp-level MMAs (mma_same.cu) instead of the tcgen05 tile /
# resident kernels (a set, so that A/B runs can switch single levels).  Measured per block at batch
# 256 on B200: C = 8 @256^2 292 vs 430 us, C = 16 @128^2 162 vs 199 us; C = 32 @64^2 126 us against
# 89 us per block for the image-resident tcgen05 run, which therefore keeps that level.
LOWC_MMA = {8, 16}
# 'down' blocks with these input widths on warp-level MMAs (mma_down.cu) instead of tc_down.cu
DOWN_MMA = {8, 16, 32}
# "fp32tc": 'same' blocks of these widths on warp-level MMAs (mma_same_split.cu) instead of tc_split.cu
# (B200, batch 256: C = 8 @256^2 and C = 16 @128^2 at 1.66 / 0.76 ms per block on the tcgen05 form)
SPLIT_MMA = {8, 16}
# True: in "fp16" mode the NHWC tensors between tensor-core kernels are fp16 instead of fp32.  Built,
# tested (tests/test_gpu_tc.py) and measured on B200 (round 2): halving the block-boundary bytes
# changes the step time by < 1 % (4.56 vs 4.55 ms at batch 256 -- the tile kernels are latency /
# issue bound, not byte bound) while the extra roundings cost code agreement with the reference
# (0.9985 -> 0.9966 on the nd3 golden), so the fp32 stream stays the default.
STREAM_F16 = False


_TORCH_DT = {torch.float32: L.DT_F32, torch.bfloat16: L.DT_BF16, torch.float16: L.DT_F16}


def _io_dt(t: Tensor) -> int:
    return L.DT_F16 if t.dtype == torch.float16 else L.DT_F32


def _as_stream(x: Tensor, half: bool) -> Tensor:
    want = torch.float16 if half else torch.float32
    return x if x.dtype == want else x.to(want)


def trunk_resident(x: Tensor, out: Tensor, chain: "PackedChain") -> None:
    """vqae_trunk_resident_f16 on NHWC x -> out (same dtype: fp32 or fp16; out may alias x)."""
    b, hh, ww, c = x.shape
    L.check(L.load().vqae_trunk_resident_f16(
        _ptr(x), _ptr(out), _io_dt(x), _ptr(chain.weights), _ptr(chain.scalars), chain.n, b, hh, ww,
        c, _stream(x.device)), "vqae_trunk_resident_f16")
# Runs of 'same' blocks at C = 64 / 128 @ 32 x 32 and C = 32 @ 64 x 64 use the
# image-resident kernel (tc_resident.cu); False selects the tile kernels (tc_chain.cu / tc_kernels.cu)
# for A/B measurements (profiles/step_breakdown.py)
TRUNK_RESIDENT = True


def fixup_forward_nhwc(pk: PackedFixup, x: Tensor, out: Optional[Tensor] = None,
                       precision: str = "fp32") -> Tensor:
    """x: contiguous NHWC [B,H,W,c_in] -> NHWC [B,H',W',c_out].

    precision "fp32": CUDA-core exact path, fp32 in and out.  "fp16": tcgen05 kernels (fp16
    operands, fp32 accumulation and fp32 residual add) wherever one is built for the block's shape
    -- they read and write fp32 or fp16 tensors, whatever x is -- and the fp32 kernels elsewhere."""
    lib = L.load()
    b, h, w, c = x.shape
    if c != pk.c_in:
        raise ValueError(f"fixup block expects {pk.c_in} input channels, got {c}")
    ho, wo = pk.out_hw(h, w)
    ensure_packed([pk], *_plan_layouts([pk], h, w, precision))
    tc = precision == "fp16" and pk.tc_ok(h, w)
    if precision == "fp32tc" and pk.split_ok(h, w):
        x = _as_stream(x, False)
        if out is None:
            out = torch.empty(b, ho, wo, pk.c_out, dtype=torch.float32, device=x.device)
        hi, lo = pk.split_hi, pk.split_lo
        if pk.mode == L.MODE_DOWN:
            fn, name = lib.vqae_down_block_split_f16, "vqae_down_block_split_f16"
        elif c in SPLIT_MMA and pk.split_mma_hi is not None and \
                lib.vqae_same_block_mma_split_supported(h, w, c):
            fn, name = lib.vqae_same_block_mma_split_f16, "vqae_same_block_mma_split_f16"
            hi, lo = pk.split_mma_hi, pk.split_mma_lo
        else:
            fn, name = lib.vqae_same_block_split_f16, "vqae_same_block_split_f16"
        L.check(fn(_ptr(x), _ptr(out), _ptr(hi), _ptr(lo), pk.tc_scalars,
                   pk.split_premul, b, h, w, c, _stream(x.device)), name)
        return out
    if tc and pk.chain_only:
        return run_blocks_nhwc([pk], x, "fp16")
    if tc and pk.mode == L.MODE_SAME and c in LOWC_MMA and x.dtype == torch.float32 and \
            lib.vqae_same_block_mma_supported(h, w, c):
        if out is None:
            out = torch.empty_like(x)
        L.check(lib.vqae_same_block_mma_f16(_ptr(x), _ptr(out), _ptr(pk.mma_weights), pk.tc_scalars,
                                            b, h, w, c, _stream(x.device)), "vqae_same_block_mma_f16")
        return out
    if tc and pk.mode == L.MODE_UP:
        x = _as_stream(x, False)
        if out is None:
            out = torch.empty(b, ho, wo, pk.c_out, dtype=torch.float32, device=x.device)
        ws = workspace(x.device, lib.vqae_up_block_mma_scratch_bytes(b, h, w, c))
        L.check(lib.vqae_up_block_mma_f16(_ptr(x), _ptr(out), _ptr(pk.mma_weights), pk.tc_scalars,
                                          _ptr(ws), ws.numel(), b, h, w, c, _stream(x.device)),
                "vqae_up_block_mma_f16")
        return out
    if tc and pk.mode == L.MODE_DOWN and c in DOWN_MMA and x.dtype == torch.float32 and \
            lib.vqae_down_block_mma_supported(h, w, c):
        if out is None:
            out = torch.empty(b, ho, wo, pk.c_out, dtype=torch.float32, device=x.device)
        L.check(lib.vqae_down_block_mma_f16(_ptr(x), _ptr(out), _ptr(pk.mma_weights), pk.tc_scalars,
                                            b, h, w, c, _stream(x.device)), "vqae_down_block_mma_f16")
        return out
    if tc:
        if out is None:
            out = torch.empty(b, ho, wo, pk.c_out, dtype=x.dtype, device=x.device)
        fn, name = ((lib.vqae_down_block_f16, "vqae_down_block_f16") if pk.mode == L.MODE_DOWN
                    else (lib.vqae_same_block_f16, "vqae_same_block_f16"))
        L.check(fn(_ptr(x), _ptr(out), _io_dt(x), _ptr(pk.tc_weights), pk.tc_scalars, b, h, w, c,
                   _stream(x.device)), name)
        return out
    x = _as_stream(x, False)
    if out is None:
        out = torch.empty(b, ho, wo, pk.c_out, dtype=torch.float32, device=x.device)
    need = lib.vqae_fixup_block_scratch_bytes(C.byref(pk.params), b, h, w)
    ws = workspace(x.device, need)
    L.check(lib.vqae_fixup_block_f32(C.byref(pk.params), _ptr(x), _ptr(out), _ptr(ws),
                                     ws.numel(), b, h, w, _stream(x.device)),
            "vqae_fixup_block_f32")
    return out


class PackedChain:
    """Back-to-back bf16 weight packs + device scalar table of a run of tcgen05 'same' blocks."""

    def __init__(self, run: Sequence[PackedFixup], resident: bool = False):
        ensure_packed(run, [False] * len(run), [True] * len(run))
        dev = run[0].device
        self.n = len(run)
        self.c = run[0].c_in
        self.resident = resident
        self.weights = torch.cat([pk.tc_weights_res if resident else pk.tc_weights for pk in run])
        self.scalars = torch.tensor([[float(v) for v in pk.tc_scalars] for pk in run],
                                    dtype=torch.float32).to(dev)


def _chain_runs(packed: Sequence[PackedFixup], h: int, w: int, batch: int = 1 << 30
                ) -> List[Tuple[int, int]]:
    """Maximal runs [start, stop) of >= 2 consecutive tcgen05 'same' blocks of equal width for
    which a multi-block kernel is built (vqae_trunk_resident_supported: C = 64 at 32 x 32, any
    batch; else vqae_same_chain_supported)."""
    lib = L.load()
    runs, i, n = [], 0, len(packed)
    while i < n:
        pk = packed[i]
        hh, ww = h, w
        if pk.mode == L.MODE_SAME and pk.tc_ok(hh, ww):
            j = i + 1
            while j < n and packed[j].mode == L.MODE_SAME and packed[j].c_in == pk.c_in \
                    and packed[j].tc_ok(hh, ww):
                j += 1
            resident = TRUNK_RESIDENT and pk.has_resident and \
                lib.vqae_trunk_resident_supported(batch, hh, ww, pk.c_in)
            lowc = pk.c_in in LOWC_MMA and lib.vqae_same_block_mma_supported(hh, ww, pk.c_in)
            if not lowc and (j - i >= 2 or pk.chain_only) and \
                    (resident or lib.vqae_same_chain_supported(batch, hh, ww, pk.c_in)):
                runs.append((i, j))
            i = j
        else:
            h, w = pk.out_hw(h, w)
            i += 1
    return runs


def run_blocks_nhwc(packed: Sequence[PackedFixup], h: Tensor, precision: str = "fp32",
                    chain_cache: Optional[dict] = None) -> Tensor:
    """A Sequential chain of PreActFixupResBlocks on an NHWC tensor.  In "fp16" mode runs of
    consecutive tcgen05 'same' blocks execute as ONE launch: image-resident (vqae_trunk_resident_f16)
    where a cluster can own an image, the persistent tile chain (vqae_same_chain_f16) otherwise; the
    tensors between tensor-core kernels are fp16 (STREAM_F16), fp32 around the fp32 kernels."""
    ensure_packed(packed, *_plan_layouts(packed, h.shape[1], h.shape[2], precision))
    if precision != "fp16":
        h = _as_stream(h, False)
        for pk in packed:
            h = fixup_forward_nhwc(pk, h, precision=precision)
        return h
    lib = L.load()
    runs = dict(_chain_runs(packed, h.shape[1], h.shape[2], h.shape[0]))
    cache = chain_cache if chain_cache is not None else {}
    i, n = 0, len(packed)
    while i < n:
        if i not in runs:
            pk = packed[i]
            if pk.tc_ok(h.shape[1], h.shape[2]) and not pk.chain_only:
                h = _as_stream(h, STREAM_F16)
            h = fixup_forward_nhwc(pk, h, precision=precision)
            i += 1
            continue
        j = runs[i]
        b, hh, ww, c = h.shape
        resident = TRUNK_RESIDENT and bool(lib.vqae_trunk_resident_supported(b, hh, ww, c))
        key = (i, j, id(packed[i]), resident)
        chain = cache.get(key)
        if chain is None:
            chain = cache[key] = PackedChain(packed[i:j], resident)
        if resident:
            h = _as_stream(h, STREAM_F16)
            out = torch.empty_like(h)
            trunk_resident(h, out, chain)
            h = out
            i = j
            continue
        h = _as_stream(h, False)                       # the tile-chain kernel streams fp32
        bufs = [torch.empty_like(h), torch.empty_like(h)]
        fbytes = lib.vqae_same_chain_flag_bytes(chain.n, b)
        flags = torch.empty(fbytes, dtype=torch.uint8, device=h.device)
        L.check(lib.vqae_same_chain_f16(
            _ptr(h), _ptr(bufs[0]), _ptr(bufs[1]), _ptr(chain.weights), _ptr(chain.scalars),
            _ptr(flags), fbytes, chain.n, b, hh, ww, c, _stream(h.device)), "vqae_same_chain_f16")
        h = bufs[(chain.n - 1) & 1]
        i = j
    return h


def stem_in(x: Tensor, weight: Tensor, bias: Tensor, mean=None, std=None,
            out_dtype: torch.dtype = torch.float32, precision: str = "fp32") -> Tensor:
    """x: fp32 [B,3,H,W] (NCHW or channels_last strides) or u8 [B,H,W,3] -> NHWC [B,H,W,8], fp32 or
    (fp16 stream of the reduced-precision path; needs W % 128 == 0 and H % 8 == 0) fp16."""
    lib = L.load()
    require_cuda(x, "stem_in")
    w = weight.detach().float().contiguous()
    bi = bias.detach().float().contiguous()
    if x.dtype == torch.uint8:
        if x.dim() != 4 or x.shape[-1] != 3:
            raise ValueError("uint8 input must be [B,H,W,3]")
        x = x.contiguous()
        b, h, wd, _ = x.shape
        dt, lay = L.DT_U8, L.LAYOUT_NHWC
        mean_a, std_a = L.f3(mean or CAMELYON16_MEAN), L.f3(std or CAMELYON16_STD)
    else:
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"expected [B,3,H,W] input, got {tuple(x.shape)}")
        b, _, h, wd = x.shape
        if x.dtype != torch.float32:
            x = x.float()
        if is_channels_last(x):
            lay = L.LAYOUT_NHWC
        else:
            x = x.contiguous()
            lay = L.LAYOUT_NCHW
        dt, mean_a, std_a = L.DT_F32, None, None
    if out_dtype == torch.float16 and (wd % 128 or h % 8):
        out_dtype = torch.float32
    out = torch.empty(b, h, wd, w.shape[0], dtype=out_dtype, device=x.device)
    if precision != "fp32" and out_dtype == torch.float32 and \
            lib.vqae_stem_in_mma_supported(h, wd, w.shape[0]):
        # fp32-accurate tensor-core form (csrc/mma_stem.cu); "fp32" keeps the exact CUDA-core kernel
        L.check(lib.vqae_stem_in_mma_f32(_ptr(x), dt, lay, _ptr(w), _ptr(bi), _ptr(out), b, h, wd,
                                         w.shape[0], mean_a, std_a, _stream(x.device)),
                "vqae_stem_in_mma_f32")
        return out
    L.check(lib.vqae_stem_in(_ptr(x), dt, lay, _ptr(w), _ptr(bi), _ptr(out), _TORCH_DT[out_dtype],
                             b, h, wd, w.shape[0], mean_a, std_a, _stream(x.device)),
            "vqae_stem_in")
    return out


# True: in "fp16" mode the encoder's in_stem + 'same' C = 8 + 'down' 8 -> 16 run as ONE kernel
# (csrc/mma_front.cu) where the model starts that way.  Built, tested (tests/test_gpu_front.py) and
# measured on B200 at batch 256 of 256^2 (round 2, profiles/run_front.py): DRAM traffic 261 MB
# instead of 2.4 GB, but 869 us against 756 us for the three separate launches -- each phase of a
# tile is a chain of dependent MMAs / MUFUs per warp with five CTA barriers per tile, and the kernel
# is latency bound at 24 warps per SM (issue slots 60 % busy) -- so the separate launches stay the
# default.
FRONT_FUSED = False


def encoder_front(x: Tensor, weight: Tensor, bias: Tensor, mean, std, packed: Sequence[PackedFixup],
                  precision: str, half_stream: bool = False) -> Tuple[Tensor, int]:
    """in_stem plus as many leading blocks of ``packed`` as one kernel covers: returns the NHWC
    activation and the number of blocks consumed (0 = the stem alone, vqae_stem_in)."""
    lib = L.load()
    fuse = (FRONT_FUSED and precision == "fp16" and not half_stream and len(packed) >= 2
            and weight.shape[0] == 8
            and packed[0].tc_kind == "same" and packed[0].c_in == 8
            and packed[1].tc_kind == "down" and packed[1].c_in == 8)
    if fuse:
        if x.dtype == torch.uint8:
            hh, ww = x.shape[1], x.shape[2]
        else:
            hh, ww = x.shape[2], x.shape[3]
        fuse = bool(lib.vqae_front_fused_supported(hh, ww))
    if not fuse:
        return stem_in(x, weight, bias, mean, std,
                       torch.float16 if half_stream else torch.float32, precision), 0
    require_cuda(x, "encoder_front")
    ensure_packed(packed[:2], [False, False], [True, True])
    w = weight.detach().float().contiguous()
    bi = bias.detach().float().contiguous()
    if x.dtype == torch.uint8:
        if x.dim() != 4 or x.shape[-1] != 3:
            raise ValueError("uint8 input must be [B,H,W,3]")
        x = x.contiguous()
        b = x.shape[0]
        dt, lay = L.DT_U8, L.LAYOUT_NHWC
        mean_a, std_a = L.f3(mean or CAMELYON16_MEAN), L.f3(std or CAMELYON16_STD)
    else:
        if x.dim() != 4 or x.shape[1] != 3:
            raise ValueError(f"expected [B,3,H,W] input, got {tuple(x.shape)}")
        b = x.shape[0]
        if x.dtype != torch.float32:
            x = x.float()
        if is_channels_last(x):
            lay = L.LAYOUT_NHWC
        else:
            x = x.contiguous()
            lay = L.LAYOUT_NCHW
        dt, mean_a, std_a = L.DT_F32, None, None
    out = torch.empty(b, hh // 2, ww // 2, 16, dtype=torch.float32, device=x.device)
    L.check(lib.vqae_front_fused_f16(_ptr(x), dt, lay, _ptr(w), _ptr(bi), mean_a, std_a,
                                     _ptr(packed[0].mma_weights), packed[0].tc_scalars,
                                     _ptr(packed[1].mma_weights), packed[1].tc_scalars, _ptr(out),
                                     b, hh, ww, _stream(x.device)), "vqae_front_fused_f16")
    return out, 2


def stem_out(x_nhwc: Tensor, weight: Tensor, bias: Tensor, channels_last: bool,
             precision: str = "fp32") -> Tensor:
    """NHWC fp32 [B,H,W,8] -> [B,3,H,W] (contiguous NCHW, or channels_last strides).  "fp32": the
    exact CUDA-core kernel; other precisions: split-operand tensor-core kernel (fp32-accurate,
    csrc/mma_stem.cu) where it tiles the image."""
    lib = L.load()
    x_nhwc = _as_stream(x_nhwc, False)
    b, h, wd, c = x_nhwc.shape
    w = weight.detach().float().contiguous()
    bi = bias.detach().float().contiguous()
    if channels_last:
        out = torch.empty(b, h, wd, 3, dtype=torch.float32, device=x_nhwc.device)
        lay = L.LAYOUT_NHWC
    else:
        out = torch.empty(b, 3, h, wd, dtype=torch.float32, device=x_nhwc.device)
        lay = L.LAYOUT_NCHW
    if precision != "fp32" and lib.vqae_stem_out_mma_supported(h, wd, c):
        L.check(lib.vqae_stem_out_mma_f32(_ptr(x_nhwc), _ptr(w), _ptr(bi), _ptr(out), lay, b, h, wd, c,
                                          _stream(x_nhwc.device)), "vqae_stem_out_mma_f32")
    else:
        L.check(lib.vqae_stem_out_f32(_ptr(x_nhwc), _ptr(w), _ptr(bi), _ptr(out), lay, b, h, wd, c,
                                      _stream(x_nhwc.device)), "vqae_stem_out_f32")
    return out.permute(0, 3, 1, 2) if channels_last else out


def stem_out_u8(x_nhwc: Tensor, weight: Tensor, bias: Tensor, canvas: Tensor, first_patch: int = 0,
                grid_cols: int = 1, mean=None, std=None, precision: str = "fp32") -> Tensor:
    """NHWC fp32 [B,H,W,8] -> uint8 RGB pixels, de-normalised with ``mean`` / ``std`` (default: the
    CAMELYON16 constants of ``Encoder.encode``) and rounded half to even (vqae_stem_out_u8).  Image b
    lands at patch ``first_patch + b`` of ``canvas`` (contiguous uint8 [rows, cols, 3], a grid of H x W
    patches with ``grid_cols`` per row); ``grid_cols = 1, first_patch = 0`` on a [B*H, W, 3] view is a
    plain [B,H,W,3] batch.  Kernel choice as in ``stem_out``: "fp32" the exact CUDA-core kernel,
    other precisions the split-operand tensor-core kernel where it tiles the image."""
    lib = L.load()
    require_cuda(x_nhwc, "stem_out_u8")
    x_nhwc = _as_stream(x_nhwc, False).contiguous()
    b, h, wd, c = x_nhwc.shape
    if canvas.dtype != torch.uint8 or canvas.dim() != 3 or canvas.shape[2] != 3 or \
            not canvas.is_contiguous() or canvas.device != x_nhwc.device:
        raise ValueError("canvas must be a contiguous uint8 [rows, cols, 3] tensor on the input's device")
    w = weight.detach().float().contiguous()
    bi = bias.detach().float().contiguous()
    kernel = L.STEM_OUT_EXACT
    if precision != "fp32" and lib.vqae_stem_out_u8_supported(h, wd, c, L.STEM_OUT_TENSOR_CORE):
        kernel = L.STEM_OUT_TENSOR_CORE
    L.check(lib.vqae_stem_out_u8(_ptr(x_nhwc), _ptr(w), _ptr(bi), L.f3(mean or CAMELYON16_MEAN),
                                 L.f3(std or CAMELYON16_STD), _ptr(canvas), canvas.shape[0],
                                 canvas.shape[1], first_patch, grid_cols, b, h, wd, c,
                                 kernel, _stream(x_nhwc.device)), "vqae_stem_out_u8")
    return canvas


def normalize_u8(img: Tensor, mean=CAMELYON16_MEAN, std=CAMELYON16_STD,
                 channels_last: bool = False) -> Tensor:
    """u8 [B,H,W,3] -> fp32 [B,3,H,W]."""
    lib = L.load()
    require_cuda(img, "normalize_u8")
    img = img.contiguous()
    b, h, w, _ = img.shape
    if channels_last:
        out = torch.empty(b, h, w, 3, dtype=torch.float32, device=img.device)
    else:
        out = torch.empty(b, 3, h, w, dtype=torch.float32, device=img.device)
    L.check(lib.vqae_normalize_u8(_ptr(img), _ptr(out), b, h, w, L.f3(mean), L.f3(std),
                                  L.LAYOUT_NHWC if channels_last else L.LAYOUT_NCHW,
                                  _stream(img.device)), "vqae_normalize_u8")
    return out.permute(0, 3, 1, 2) if channels_last else out


class PackedQuantizer:
    """Codebook, proj_in weights and the proj_out(embed) table of one quantiser module."""

    def __init__(self, embed: Tensor, commitment_cost: float, proj_in=None, proj_out=None):
        lib = L.load()
        require_cuda(embed, "quantizer")
        self.embed = embed.detach().float().contiguous()
        self.k, self.d = self.embed.shape
        dev = embed.device
        if proj_in is not None:
            self.c = proj_in.weight.shape[1]
            self.w_in = proj_in.weight.detach().float().reshape(self.d, self.c).contiguous()
            self.b_in = proj_in.bias.detach().float().contiguous()
            self.w_out = proj_out.weight.detach().float().reshape(self.c, self.d).contiguous()
            self.b_out = proj_out.bias.detach().float().contiguous()
        else:
            self.c = self.d
            self.w_in = self.b_in = self.w_out = self.b_out = None
        self.table = torch.empty(self.k, self.c, dtype=torch.float32, device=dev)
        L.check(lib.vqae_quantizer_prepare_f32(_ptr(self.embed), self.k, self.d, _ptr(self.w_out),
                                               _ptr(self.b_out), self.c, _ptr(self.table),
                                               _stream(dev)), "vqae_quantizer_prepare_f32")
        p = L.QuantizerParams()
        p.num_codes, p.dim, p.c = self.k, self.d, self.c
        p.embed = self.embed.data_ptr()
        p.w_in = self.w_in.data_ptr() if self.w_in is not None else None
        p.b_in = self.b_in.data_ptr() if self.b_in is not None else None
        p.table = self.table.data_ptr()
        p.commitment_cost = float(commitment_cost)
        self.params = p


_KERNEL = {"auto": L.QUANT_AUTO, "cuda_core": L.QUANT_CUDA_CORE, "tensor_core": L.QUANT_TENSOR_CORE}


def quantize(pq: PackedQuantizer, x: Tensor, x_nhwc: bool, out_nhwc: bool, batch: int,
             spatial: int, want_out: bool = True, want_z: bool = False, kernel: str = "auto",
             out_dtype: Optional[torch.dtype] = None
             ) -> Tuple[Optional[Tensor], Tensor, Tensor, Tensor, Optional[Tensor]]:
    """x: contiguous fp32 / bf16 / fp16, [B,S,c] if x_nhwc else [B,c,S].  Returns
    (out or None, indices int64 [B*S], loss 0-dim, near_ties uint32 0-dim, z or None).
    kernel: "auto", "cuda_core" (the exact CUDA-core kernel) or "tensor_core" (tcgen05)."""
    lib = L.load()
    dev = x.device
    n = batch * spatial
    out_dtype = out_dtype or x.dtype
    out = torch.empty(n * pq.c, dtype=out_dtype, device=dev) if want_out else None
    idx = torch.empty(n, dtype=torch.int64, device=dev)
    loss = torch.empty((), dtype=torch.float32, device=dev)
    ties = torch.empty((), dtype=torch.int32, device=dev)
    z = torch.empty(n, pq.d, dtype=torch.float32, device=dev) if want_z else None
    need = lib.vqae_quantizer_scratch_bytes(n)
    ws = workspace(dev, need)
    L.check(lib.vqae_quantize(
        C.byref(pq.params), _ptr(x), _TORCH_DT[x.dtype], L.LAYOUT_NHWC if x_nhwc else L.LAYOUT_NCHW,
        _ptr(out), _TORCH_DT[out_dtype], L.LAYOUT_NHWC if out_nhwc else L.LAYOUT_NCHW, _ptr(idx),
        _ptr(loss), _ptr(ties), NEAR_TIE_REL_GAP, _ptr(z), _ptr(ws), ws.numel(), batch, spatial,
        _KERNEL[kernel], _stream(dev)), "vqae_quantize")
    return out, idx, loss, ties, z


# I/O dtypes of the quantiser call for which a kernel is built (config 2 cells)
QUANT_IO_DTYPES = ("fp32", "bf16", "fp16")


def quantize_io_supported(pq: PackedQuantizer, dtype: torch.dtype) -> bool:
    """NHWC in / NHWC out of `dtype` is built (the tcgen05 kernel: fp32 / bf16 / fp16, c in {64, 128})."""
    dt = _TORCH_DT.get(dtype)
    return dt is not None and bool(L.load().vqae_quantize_supported(
        C.byref(pq.params), dt, L.LAYOUT_NHWC, dt, L.LAYOUT_NHWC, 1, L.QUANT_AUTO))


class QuantizeBuffers:
    """Preallocated outputs + scratch of one quantiser call shape (steady-state callers, bench)."""

    def __init__(self, pq: PackedQuantizer, n: int, dtype: torch.dtype, dev: torch.device):
        lib = L.load()
        self.n, self.dtype = n, dtype
        self.out = torch.empty(n * pq.c, dtype=dtype, device=dev)
        self.idx = torch.empty(n, dtype=torch.int64, device=dev)
        self.loss = torch.empty((), dtype=torch.float32, device=dev)
        self.ties = torch.empty((), dtype=torch.int32, device=dev)
        self.ws = workspace(dev, lib.vqae_quantizer_scratch_bytes(n))
        dt = _TORCH_DT[dtype]
        tc = bool(lib.vqae_quantize_supported(C.byref(pq.params), dt, L.LAYOUT_NHWC, dt,
                                              L.LAYOUT_NHWC, 1, L.QUANT_TENSOR_CORE))
        self.kernel_name = ("quantize_tc_kernel (tcgen05 L4 filter + exact fp32 argmin + gather, "
                            "fused loss)" if tc else "quantize_kernel (CUDA-core)")


def quantize_into(pq: PackedQuantizer, x: Tensor, bufs: QuantizeBuffers, batch: int, spatial: int
                  ) -> None:
    """The quantiser call on NHWC input into preallocated buffers (no allocation, no sync)."""
    lib = L.load()
    dt = _TORCH_DT[x.dtype]
    L.check(lib.vqae_quantize(
        C.byref(pq.params), _ptr(x), dt, L.LAYOUT_NHWC, _ptr(bufs.out), _TORCH_DT[bufs.dtype],
        L.LAYOUT_NHWC, _ptr(bufs.idx), _ptr(bufs.loss), _ptr(bufs.ties), NEAR_TIE_REL_GAP, None,
        _ptr(bufs.ws), bufs.ws.numel(), batch, spatial, L.QUANT_AUTO, _stream(x.device)),
        "vqae_quantize")


def embed_codes(pq: PackedQuantizer, idx: Tensor, out_nhwc: bool, batch: int, spatial: int
                ) -> Tensor:
    """out[n,:] = table[idx[n],:] (embed_code -> proj_out); idx int64 or uint8, flat [B*S]."""
    lib = L.load()
    require_cuda(idx, "embed_codes")
    is_u8 = idx.dtype == torch.uint8
    if not is_u8 and idx.dtype != torch.int64:
        idx = idx.long()
    idx = idx.contiguous()
    out = torch.empty(batch * spatial * pq.c, dtype=torch.float32, device=idx.device)
    L.check(lib.vqae_embed_codes_f32(_ptr(idx), int(is_u8), _ptr(pq.table), pq.k, pq.c,
                                     _ptr(out), L.LAYOUT_NHWC if out_nhwc else L.LAYOUT_NCHW,
                                     batch, spatial, _stream(idx.device)),
            "vqae_embed_codes_f32")
    return out


def embed_codemap(pq: PackedQuantizer, code_map: Tensor, code_hw: Tuple[int, int], r0: int, c0: int,
                  region_cols: int, first_patch: int, n: int) -> Tensor:
    """``embed_codes`` of n code tiles gathered straight from a stored map (vqae_embed_codemap_f32):
    code_map uint8 / int64 [rows*th, cols*tw]; patch t is region patch ``first_patch + t`` of the region
    with origin (r0, c0) (in patches) and ``region_cols`` patches per row.  Returns NHWC fp32
    [n, th, tw, C]."""
    lib = L.load()
    require_cuda(code_map, "embed_codemap")
    if code_map.dtype not in (torch.uint8, torch.int64) or code_map.dim() != 2:
        raise ValueError("embed_codemap reads a 2-D uint8 or int64 code map")
    code_map = code_map.contiguous()
    th, tw = code_hw
    out = torch.empty(n, th, tw, pq.c, dtype=torch.float32, device=code_map.device)
    L.check(lib.vqae_embed_codemap_f32(_ptr(code_map), int(code_map.dtype == torch.uint8),
                                       code_map.shape[0], code_map.shape[1], th, tw, r0, c0, region_cols,
                                       first_patch, n, _ptr(pq.table), pq.k, pq.c, _ptr(out),
                                       _stream(code_map.device)), "vqae_embed_codemap_f32")
    return out


def codemap_place(tiles: Tensor, first_patch: int, grid_cols: int, code_map: Tensor) -> None:
    """Place int64 code tiles [P,th,tw] into the u8 map [rows*th, cols*tw] (row-major patches)."""
    lib = L.load()
    require_cuda(tiles, "codemap_place")
    if code_map.dtype != torch.uint8:
        raise ValueError("codemap_place writes uint8 maps (<= 256 codes); see codemap_place_i64")
    tiles = tiles.contiguous()
    p, th, tw = tiles.shape
    L.check(lib.vqae_codemap_place_u8(_ptr(tiles), p, th, tw, first_patch, grid_cols,
                                      _ptr(code_map), code_map.shape[0], code_map.shape[1],
                                      _stream(tiles.device)), "vqae_codemap_place_u8")


def codemap_place_i64(tiles: Tensor, first_patch: int, grid_cols: int, code_map: Tensor) -> None:
    """Like codemap_place, into an int64 map (any codebook size; narrowed on the host later)."""
    lib = L.load()
    require_cuda(tiles, "codemap_place_i64")
    if code_map.dtype != torch.int64 or tiles.dtype != torch.int64:
        raise ValueError("codemap_place_i64 expects int64 tiles and an int64 map")
    tiles = tiles.contiguous()
    p, th, tw = tiles.shape
    L.check(lib.vqae_codemap_place_i64(_ptr(tiles), p, th, tw, first_patch, grid_cols,
                                       _ptr(code_map), code_map.shape[0], code_map.shape[1],
                                       _stream(tiles.device)), "vqae_codemap_place_i64")


def quality_u8(ref_canvas: Tensor, ref_addr: Tuple[int, int, int, int], rec_canvas: Tensor,
               rec_addr: Tuple[int, int, int, int], batch: int, h: int, w: int) -> Tuple[Tensor, Tensor]:
    """Per-patch SSE (int64 [batch, 3]) and SSIM (float64 [batch]) of ``batch`` h x w patches of two
    uint8 RGB canvases (vqae_quality_u8).  Each canvas is a contiguous uint8 [rows, cols, 3] tensor
    holding a grid of h x w patches; ``addr = (r0, c0, region_cols, first)`` puts patch t of the call at
    grid position (r0 + (first + t) // region_cols, c0 + (first + t) % region_cols).  ``(0, 0, 1, 0)``
    on a [batch*h, w, 3] view is a plain batch."""
    lib = L.load()
    require_cuda(ref_canvas, "quality_u8")
    for cv in (ref_canvas, rec_canvas):
        if cv.dtype != torch.uint8 or cv.dim() != 3 or cv.shape[2] != 3 or not cv.is_contiguous() or \
                cv.device != ref_canvas.device:
            raise ValueError("quality_u8 reads contiguous uint8 [rows, cols, 3] canvases on one device")
    dev = ref_canvas.device
    sse = torch.empty(batch, 3, dtype=torch.int64, device=dev)
    ssim = torch.empty(batch, dtype=torch.float64, device=dev)
    ws = workspace(dev, lib.vqae_quality_u8_scratch_bytes(batch, h, w))
    (ar0, ac0, arc, afirst), (br0, bc0, brc, bfirst) = ref_addr, rec_addr
    L.check(lib.vqae_quality_u8(_ptr(ref_canvas), ref_canvas.shape[0], ref_canvas.shape[1], ar0, ac0, arc,
                                afirst, _ptr(rec_canvas), rec_canvas.shape[0], rec_canvas.shape[1], br0, bc0,
                                brc, bfirst, batch, h, w, _ptr(sse), _ptr(ssim), _ptr(ws), ws.numel(),
                                _stream(dev)), "vqae_quality_u8")
    return sse, ssim


def _code_map_arg(code_map: Tensor, what: str) -> Tensor:
    require_cuda(code_map, what)
    if code_map.dtype not in (torch.uint8, torch.int64) or code_map.dim() != 2:
        raise ValueError(f"{what} reads a 2-D uint8 or int64 code map")
    return code_map.contiguous()


def _host_u32(values) -> np.ndarray:
    return np.ascontiguousarray(np.asarray(values, dtype=np.uint32))


def _host_i64(values) -> np.ndarray:
    if isinstance(values, Tensor):
        values = values.cpu().numpy()
    return np.ascontiguousarray(np.asarray(values, dtype=np.int64))


def codemap_histogram(code_map: Tensor, k: int, window: Optional[Tuple[int, int, int, int]] = None
                      ) -> Tuple[Tensor, Tensor]:
    """Code counts of a uint8 / int64 map, or of the window ``(r0, c0, nr, nc)`` of it in codes
    (vqae_codemap_histogram): int64 [k] counts of the codes 0 .. k-1 and an int64 scalar counting the
    codes outside [0, k), both on the map's device."""
    lib = L.load()
    code_map = _code_map_arg(code_map, "codemap_histogram")
    r0, c0, nr, nc = window if window is not None else (0, 0, code_map.shape[0], code_map.shape[1])
    counts = torch.empty(k + 1, dtype=torch.int64, device=code_map.device)
    L.check(lib.vqae_codemap_histogram(_ptr(code_map), int(code_map.dtype == torch.uint8), code_map.shape[0],
                                       code_map.shape[1], r0, c0, nr, nc, k, _ptr(counts),
                                       _stream(code_map.device)), "vqae_codemap_histogram")
    return counts[:k], counts[k]


def codemap_pack(code_map: Tensor, code_hw: Tuple[int, int], freq, scale_bits: int) -> Tuple[Tensor, Tensor]:
    """rANS-pack every th x tw patch of a uint8 / int64 map with the frequency table ``freq`` (k entries
    summing to 2^scale_bits; host values) (vqae_codemap_pack).  Returns the int64 [P + 1] stream offsets
    and the payload buffer (uint8, worst-case sized: the payload is its first ``offsets[P]`` bytes)."""
    lib = L.load()
    code_map = _code_map_arg(code_map, "codemap_pack")
    th, tw = code_hw
    fh = _host_u32(freq)
    dev = code_map.device
    p = (code_map.shape[0] // th) * (code_map.shape[1] // tw)
    offsets = torch.empty(p + 1, dtype=torch.int64, device=dev)
    payload = torch.empty(max(lib.vqae_codemap_pack_worst_bytes(p, th, tw), 1), dtype=torch.uint8, device=dev)
    ws = workspace(dev, lib.vqae_codemap_pack_scratch_bytes(p, th, tw))
    L.check(lib.vqae_codemap_pack(_ptr(code_map), int(code_map.dtype == torch.uint8), code_map.shape[0],
                                  code_map.shape[1], th, tw, fh.ctypes.data_as(C.c_void_p), len(fh), scale_bits,
                                  _ptr(offsets), _ptr(payload), payload.numel(), _ptr(ws), ws.numel(),
                                  _stream(dev)), "vqae_codemap_pack")
    return offsets, payload


def codemap_unpack(payload: Tensor, offsets: Tensor, offsets_host, map_hw: Tuple[int, int],
                   code_hw: Tuple[int, int], freq, scale_bits: int, region: Tuple[int, int, int, int],
                   dtype: torch.dtype = torch.uint8) -> Tuple[Tensor, Tensor]:
    """Decode the patches ``region = (r0, c0, nr, nc)`` of a packed map (vqae_codemap_unpack): payload
    uint8 and offsets int64 [P + 1] on the device, ``offsets_host`` the same offsets on the host, ``freq``
    the host frequency table.  Returns the [nr*th, nc*tw] map (``dtype`` uint8 or int64) and the uint8
    [nr, nc] integrity flags (0: the patch decoded back to the encoder's initial state with its words
    exactly consumed)."""
    lib = L.load()
    require_cuda(payload, "codemap_unpack")
    if payload.dtype != torch.uint8 or offsets.dtype != torch.int64 or offsets.device != payload.device:
        raise ValueError("codemap_unpack reads a uint8 payload and int64 offsets on one device")
    if dtype not in (torch.uint8, torch.int64):
        raise ValueError("codemap_unpack writes uint8 or int64 maps")
    th, tw = code_hw
    r0, c0, nr, nc = region
    fh, oh = _host_u32(freq), _host_i64(offsets_host)
    if oh.shape != (offsets.numel(),) or offsets.numel() != (map_hw[0] // th) * (map_hw[1] // tw) + 1:
        raise ValueError("codemap_unpack: offsets do not match the patch grid")
    dev = payload.device
    out = torch.empty(nr * th, nc * tw, dtype=dtype, device=dev)
    flags = torch.empty(nr, nc, dtype=torch.uint8, device=dev)
    L.check(lib.vqae_codemap_unpack(_ptr(payload), payload.numel(), oh.ctypes.data_as(C.c_void_p),
                                    _ptr(offsets.contiguous()), map_hw[0], map_hw[1], th, tw,
                                    fh.ctypes.data_as(C.c_void_p), len(fh), scale_bits, r0, c0, nr, nc,
                                    _ptr(out), int(dtype == torch.uint8), _ptr(flags), _stream(dev)),
            "vqae_codemap_unpack")
    return out, flags


# ---- f-4: training-mode codebook maintenance, level sums -------------------------------------------
def add_nhwc(a: Tensor, b: Tensor, out: Optional[Tensor] = None) -> Tensor:
    """a + b for two contiguous fp32 tensors of one shape (the level sums of model.py:208, 283-288)."""
    lib = L.load()
    if a.shape != b.shape:
        raise ValueError(f"level sum of tensors of different shapes: {tuple(a.shape)} + {tuple(b.shape)}")
    a = a.float().contiguous()
    b = b.float().contiguous()
    if out is None:
        out = torch.empty_like(a)
    L.check(lib.vqae_add_f32(_ptr(a), _ptr(b), _ptr(out), a.numel(), _stream(a.device)), "vqae_add_f32")
    return out


def column_stats(z: Tensor) -> Tuple[Tensor, Tensor]:
    """(mean, unbiased std) over the rows of z [N, D] fp32 (vq.py:77-78)."""
    lib = L.load()
    n, d = z.shape
    mean = torch.empty(d, dtype=torch.float32, device=z.device)
    std = torch.empty(d, dtype=torch.float32, device=z.device)
    ws = workspace(z.device, lib.vqae_ema_scratch_bytes(n, 1, d))
    L.check(lib.vqae_column_stats_f32(_ptr(z), n, d, _ptr(mean), _ptr(std), _ptr(ws), ws.numel(),
                                      _stream(z.device)), "vqae_column_stats_f32")
    return mean, std


def ema_init(embed: Tensor, embed_avg: Tensor, cluster_size: Tensor, mean: Tensor, std: Tensor,
             cluster_add: float) -> None:
    """vq.py:90-94, in place on the three buffers."""
    k, d = embed.shape
    L.check(L.load().vqae_ema_init_f32(_ptr(embed), _ptr(embed_avg), _ptr(cluster_size), _ptr(mean),
                                       _ptr(std), k, d, float(cluster_add), _stream(embed.device)),
            "vqae_ema_init_f32")


def ema_accumulate(z: Tensor, idx: Tensor, num_codes: int) -> Tensor:
    """One buffer [K * (D + 1)]: dw [K, D] (sum of the z rows of each code) followed by counts [K]
    (vq.py:49-54) -- one buffer so that a data-parallel job needs ONE all-reduce, not two."""
    lib = L.load()
    n, d = z.shape
    buf = torch.empty(num_codes * (d + 1), dtype=torch.float32, device=z.device)
    ws = workspace(z.device, lib.vqae_ema_scratch_bytes(n, num_codes, d))
    dw, counts = buf[:num_codes * d], buf[num_codes * d:]
    L.check(lib.vqae_ema_accumulate_f32(_ptr(z), _ptr(idx), n, num_codes, d, _ptr(counts), _ptr(dw),
                                        _ptr(ws), ws.numel(), _stream(z.device)),
            "vqae_ema_accumulate_f32")
    return buf


def ema_update(embed: Tensor, embed_avg: Tensor, cluster_size: Tensor, acc: Tensor, decay: float,
               laplace_alpha: float) -> None:
    """vq.py:60-74, in place; `acc` is the (all-reduced) buffer of ema_accumulate."""
    k, d = embed.shape
    dw, counts = acc[:k * d], acc[k * d:]
    L.check(L.load().vqae_ema_update_f32(_ptr(embed), _ptr(embed_avg), _ptr(cluster_size), _ptr(counts),
                                         _ptr(dw), k, d, float(decay), float(laplace_alpha),
                                         _stream(embed.device)), "vqae_ema_update_f32")


# launches executed through CUDA-graph replays minus launches merely recorded during a capture
# (graphs.CapturedStep keeps it up to date)
_graph_launch_adjust = 0


def raw_launch_count() -> int:
    """Calls of the library's launching entry points (executed or recorded into a graph)."""
    return int(L.load().vqae_launch_count())


def launch_count() -> int:
    """Kernels of libvqae_b200.so executed so far, graph replays included."""
    return raw_launch_count() + _graph_launch_adjust
