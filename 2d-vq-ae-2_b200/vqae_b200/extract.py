"""The code-extraction caller on the B200 path (scope row f-1).

Counterpart of ``run_eval`` / ``get_encodings`` / ``main`` in
scripts/extract_embeddings/extract_embeddings.py:43-138,176-185: patches in, per-slide code map
out, written as ``<ckpt>/encodings/<parent>/<stem>.npy``.  Differences by design: tiles may arrive
as raw uint8 NHWC (normalisation is fused into the stem kernel instead of running in DataLoader
workers), the quantised tensor is never written (only indices are used,
extract_embeddings.py:125-137), and tiles are placed into the slide map by a kernel instead of
advanced indexing.
"""
from __future__ import annotations

import math
from pathlib import Path
from typing import Dict, Iterable, Iterator, Optional, Sequence, Tuple

import numpy as np
import torch

from . import engine as E
from . import plan as P
from .graphs import CapturedStep
from .plan import resolve_precision
from .quality import ReconstructionQuality, check_u8_patches, reconstruction_quality
from .sharding import gather_code_tiles, shard_range, slide_grid  # noqa: F401


def cast_to_lowest_dtype(array: np.ndarray) -> np.ndarray:
    """extract_embeddings.py:54-59."""
    amin, amax = array.min(), array.max()
    if amin == 0 and amax == 1:
        return array.astype(bool)
    return array.astype(np.result_type(np.min_scalar_type(amin), np.min_scalar_type(amax)))


def extract_path(path: str) -> str:
    """'<...>/<parent>/<name>.tif' -> '<parent>/<name>' (extract_embeddings.py:111-112)."""
    return Path(path).parent.stem + '/' + Path(path).stem


def encoding_path(ckpt_folder, array_name: str) -> Path:
    """Where ``main`` stores a finished slide (extract_embeddings.py:183-185)."""
    return Path(ckpt_folder) / 'encodings' / (array_name + '.npy')


def save_encoding(ckpt_folder, array_name: str, array: np.ndarray) -> Path:
    out_path = encoding_path(ckpt_folder, array_name)
    out_path.parent.mkdir(parents=True, exist_ok=True)
    np.save(str(out_path), array)
    return out_path


@torch.no_grad()
def encode_patches(encoder, patches: torch.Tensor, mean=None, std=None) -> torch.Tensor:
    """patches: uint8 [B,H,W,3] or float [B,3,H,W] on a CUDA device -> int64 codes [B,h,w]."""
    _, idx, _, _, _ = encoder.encode(patches, mean=mean, std=std, want_quantized=False)
    return idx


def _check_u8_codes(encoder) -> None:
    k = int(encoder.vq_layers[0].num_embeddings)
    if k > 256:
        raise ValueError(f"uint8 code maps hold at most 256 codes, the quantiser has {k}; "
                         "use get_encodings (narrowest dtype per slide) instead")


@torch.no_grad()
def compress_slide(encoder, batches: Iterable[Tuple[int, torch.Tensor]], grid: Tuple[int, int],
                   code_hw: Tuple[int, int], device: torch.device, mean=None, std=None
                   ) -> torch.Tensor:
    """Encode (first_patch_index, patch batch) pairs of one slide and place the code tiles into a
    u8 map [rows*h, cols*w] on ``device`` (extract_embeddings.py:47-52,75-89).  Needs a codebook of
    at most 256 entries (the shipped K); wider codebooks go through ``get_encodings``."""
    _check_u8_codes(encoder)
    rows, cols = grid
    th, tw = code_hw
    code_map = torch.zeros(rows * th, cols * tw, dtype=torch.uint8, device=device)
    for first_patch, patches in batches:
        idx = encode_patches(encoder, patches.to(device, non_blocking=True), mean, std)
        E.codemap_place(idx, first_patch, cols, code_map)
    return code_map


@torch.no_grad()
def get_encodings(encoder, batches: Iterable[Tuple[torch.Tensor, Sequence[str], Sequence[int],
                                                   torch.Tensor]],
                  lengths: Sequence[int], sizes: Sequence[Tuple[int, int]],
                  device: Optional[torch.device] = None, mean=None, std=None
                  ) -> Iterator[Tuple[str, np.ndarray]]:
    """The slide-assembly loop of ``get_encodings`` (extract_embeddings.py:43-89) on the B200 path.

    ``batches`` yields what the reference's DataLoader yields per step, minus the labels:
    ``(imgs, img_paths, img_index, patch_index)`` with ``imgs`` uint8 [B,H,W,3] or float
    [B,3,H,W], ``img_paths`` the slide path of every patch, ``img_index`` [B] the slide number and
    ``patch_index`` [B,2] the (row, col) of the patch inside its slide grid.  ``lengths[i]`` /
    ``sizes[i]`` are the dataset's ``_lengths`` / ``_sizes`` (patch count and (rows, cols) grid of
    slide i, datamodules/camelyon16.py:160-168).  Yields ``(name, array)`` when the last patch of a
    slide has been placed, ``name`` = ``extract_path(path)`` and ``array`` narrowed with
    ``cast_to_lowest_dtype`` -- ready for ``save_encoding``."""
    arrays: Dict[str, torch.Tensor] = {}
    counts: Dict[str, int] = {}
    for imgs, paths, img_index, patch_index in batches:
        dev = device or imgs.device
        idx = encode_patches(encoder, imgs.to(dev, non_blocking=True), mean, std)
        th, tw = idx.shape[1:]
        names = [extract_path(p) for p in paths]
        img_index = torch.as_tensor(img_index).tolist()
        patch_index = torch.as_tensor(patch_index).reshape(len(names), 2).tolist()
        # group the batch by slide; runs of row-major consecutive patches go to the device in one
        # placement call (the common case: the tiled dataset walks a slide in row-major order)
        start = 0
        n = len(names)
        while start < n:
            name, image_index = names[start], img_index[start]
            rows, cols = (int(v) for v in sizes[image_index])
            stop = start + 1
            first = patch_index[start][0] * cols + patch_index[start][1]
            while stop < n and names[stop] == name and \
                    patch_index[stop][0] * cols + patch_index[stop][1] == first + (stop - start):
                stop += 1
            if name not in arrays:
                counts[name] = int(lengths[image_index])
                arrays[name] = torch.empty(rows * th, cols * tw, dtype=torch.int64, device=dev)
            E.codemap_place_i64(idx[start:stop], first, cols, arrays[name])
            counts[name] -= stop - start
            if counts[name] == 0:
                counts.pop(name)
                yield name, cast_to_lowest_dtype(arrays.pop(name).cpu().numpy())
            start = stop


def extract_and_save(encoder, batches, lengths, sizes, ckpt_folder, **kw) -> Iterator[Path]:
    """``main``'s inner loop (extract_embeddings.py:176-185): one ``.npy`` per finished slide."""
    for name, array in get_encodings(encoder, batches, lengths, sizes, **kw):
        yield save_encoding(ckpt_folder, name, array)


class StreamingEncoder:
    """Double-buffered host -> device -> host code extraction.

    The copy of batch i+1 from pinned host memory runs on a side stream while batch i is encoded,
    and the code indices of batch i return to pinned host memory asynchronously -- the B200
    counterpart of the reference's DataLoader(pin_memory) + ``imgs.to(device, non_blocking=True)``
    loop (extract_embeddings.py:95-101,118-122).  ``encode_stream`` yields one int64 ``[B,h,w]``
    host tensor per input batch, in order.

    By default every yielded tensor is an independent copy (safe to collect with ``list``).  With
    ``reuse_buffers=True`` the pinned staging buffers themselves are yielded (no host copy): there
    are ``N_OUT`` = 4 of them and results lag one batch behind submission, so a yielded tensor stays
    valid only until the generator has been resumed ``N_OUT - 2`` = 2 more times.

    ``graphs=True`` (default): the encode of a full-size batch is captured into one CUDA graph per
    staging buffer after its first eager run and replayed from then on (``graphs.CapturedStep``): no
    per-launch host work, no idle gaps between the step's kernels.  The graphs read the packed weights
    that existed at capture time: build the ``StreamingEncoder`` after loading the checkpoint, or call
    ``reset_graphs()`` when the weights change."""

    N_OUT = 4

    def __init__(self, encoder, device: torch.device, mean=None, std=None, graphs: bool = True):
        self.encoder, self.device, self.mean, self.std = encoder, device, mean, std
        self._step = CapturedStep(lambda x: encode_patches(self.encoder, x, self.mean, self.std),
                                  key_extra=lambda: resolve_precision(self.encoder)) if graphs else None
        self._idx_read = [None, None]                   # last D2H event of each staging slot's codes
        self.copy_stream = torch.cuda.Stream(device)
        self.out_stream = torch.cuda.Stream(device)     # D2H of the codes: off the compute stream, so
        self._done = torch.cuda.Event()                 # the next batch's kernels start right away
        self._dev_in = [None, None]
        self._host_out = [None] * self.N_OUT
        self._h2d = [torch.cuda.Event() for _ in range(2)]
        self._free = [torch.cuda.Event() for _ in range(2)]     # device input buffer consumed
        self._d2h = [torch.cuda.Event() for _ in range(self.N_OUT)]

    def reset_graphs(self) -> None:
        if self._step is not None:
            self._step.reset()

    def _stage(self, slot: int, host_batch: torch.Tensor, first_use: bool) -> None:
        if self._dev_in[slot] is None or self._dev_in[slot].shape != host_batch.shape \
                or self._dev_in[slot].dtype != host_batch.dtype:
            self._dev_in[slot] = torch.empty(host_batch.shape, dtype=host_batch.dtype,
                                             device=self.device)
            first_use = True
        with torch.cuda.stream(self.copy_stream):
            if not first_use:
                self.copy_stream.wait_event(self._free[slot])
            self._dev_in[slot].copy_(host_batch, non_blocking=True)
            self._h2d[slot].record(self.copy_stream)

    @torch.no_grad()
    def encode_stream(self, host_batches, reuse_buffers: bool = False, to_host: bool = True):
        """``to_host=False`` keeps the codes on the device (freshly allocated int64 tensors, e.g. for
        a code-tile gather): the host -> device staging still overlaps the encode."""
        main = torch.cuda.current_stream(self.device)
        it = iter(host_batches)
        nxt = next(it, None)
        if nxt is None:
            return
        self._stage(0, nxt, True)
        i = 0
        pending = []

        def result(oslot):
            self._d2h[oslot].synchronize()
            out = self._host_out[oslot]
            return out if reuse_buffers else out.clone()

        while nxt is not None:
            slot, oslot = i & 1, i % self.N_OUT
            cur, nxt = nxt, next(it, None)
            if nxt is not None:
                self._stage(slot ^ 1, nxt, i == 0)
            main.wait_event(self._h2d[slot])
            if self._step is not None:
                # a replay overwrites the codes of the batch that used this slot two steps ago
                if self._idx_read[slot] is not None:
                    main.wait_event(self._idx_read[slot])
                idx = self._step(self._dev_in[slot])
            else:
                idx = encode_patches(self.encoder, self._dev_in[slot], self.mean, self.std)
            self._free[slot].record(main)
            if not to_host:
                yield idx.clone() if self._step is not None else idx
                i += 1
                continue
            if self._host_out[oslot] is None or self._host_out[oslot].shape != idx.shape:
                if self._host_out[oslot] is None:
                    # all pinned result buffers at once: a cudaHostAlloc in the middle of the stream
                    # (slot 3 is first used by the fourth batch) stalls the pipeline for milliseconds
                    for o in range(self.N_OUT):
                        if self._host_out[o] is None:
                            self._host_out[o] = torch.empty(idx.shape, dtype=idx.dtype).pin_memory()
                else:                                  # a batch of another size (the short last one)
                    self._host_out[oslot] = torch.empty(idx.shape, dtype=idx.dtype).pin_memory()
            self._done.record(main)
            with torch.cuda.stream(self.out_stream):
                self.out_stream.wait_event(self._done)
                self._host_out[oslot].copy_(idx, non_blocking=True)
                self._d2h[oslot].record(self.out_stream)
            self._idx_read[slot] = self._d2h[oslot]
            # eager results (no graphs, the first batch, a short last batch) are ordinary allocations: the
            # allocator must not hand their memory out again before the copy stream has read it
            idx.record_stream(self.out_stream)
            pending.append(oslot)
            if len(pending) == 2:                  # results lag one batch behind the submission
                yield result(pending.pop(0))
            i += 1
        for oslot in pending:
            yield result(oslot)


def _region_plan(model, code_map: torch.Tensor, code_hw: Tuple[int, int],
                 region: Optional[Tuple[int, int, int, int]], batch: int, who: str):
    """The argument checks of ``decompress_region`` / ``score_region``: returns (packed quantiser,
    decoder, code map (uint8 or int64), (th, tw), (rows, cols), (r0, c0, nr, nc), patch scale)."""
    vq, dec = model.encoder.vq_layers[0], model.decoder
    P.check_u8_decoder(dec, who)
    E.require_cuda(code_map, who)
    if code_map.dim() != 2:
        raise ValueError(f"code_map must be 2-D, got shape {tuple(code_map.shape)}")
    if code_map.dtype not in (torch.uint8, torch.int64):
        if code_map.dtype.is_floating_point or code_map.dtype.is_complex:
            raise ValueError(f"code_map must hold integer codes, got {code_map.dtype}")
        code_map = code_map.long()
    th, tw = (int(v) for v in code_hw)
    if th <= 0 or tw <= 0 or code_map.shape[0] % th or code_map.shape[1] % tw:
        raise ValueError(f"code map {tuple(code_map.shape)} is not a grid of {th} x {tw} code tiles")
    rows, cols = code_map.shape[0] // th, code_map.shape[1] // tw
    r0, c0, nr, nc = (int(v) for v in (region if region is not None else (0, 0, rows, cols)))
    if r0 < 0 or c0 < 0 or nr <= 0 or nc <= 0 or r0 + nr > rows or c0 + nc > cols:
        raise ValueError(f"region {(r0, c0, nr, nc)} leaves the {rows} x {cols} patch grid")
    if batch <= 0:
        raise ValueError("batch must be positive")
    pq = P.packed_quantizer(vq)
    if code_map.dtype != torch.uint8 or pq.k < 256:
        win = code_map[r0 * th:(r0 + nr) * th, c0 * tw:(c0 + nc) * tw]
        if bool(((win < 0) | (win >= pq.k)).any()):
            raise ValueError(f"code map holds codes outside [0, {pq.k})")
    return pq, dec, code_map, (th, tw), (rows, cols), (r0, c0, nr, nc), P.patch_scale(dec)


@torch.no_grad()
def decompress_region(model, code_map: torch.Tensor, code_hw: Tuple[int, int],
                      region: Optional[Tuple[int, int, int, int]] = None, batch: int = 256, mean=None,
                      std=None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """The inverse of ``compress_slide``: decode a stored code map (or a region of it) to uint8 RGB
    pixels on the map's device.

    ``code_map`` [rows*th, cols*tw] of th x tw code tiles (``code_hw``), uint8 or int64 as stored, or any
    other integer / bool dtype that ``cast_to_lowest_dtype`` / ``np.load`` produce (widened to int64
    once).  ``region = (r0, c0, nr, nc)`` in patches, default the whole map.  Patches are gathered from
    the map, decoded and written into the [nr*H, nc*W, 3] result (``out`` if given) by the kernels,
    at most ``batch`` patches per step; H, W = th, tw times 2 per 'up' block of the decoder.  Each patch
    is decoded on its own, exactly like the model decodes a tile.  Reads ``model.encoder.vq_layers[0]``
    and ``model.decoder`` only, so an ``accelerate()``-d reference model works too.  ``mean`` / ``std``:
    the normalisation to undo (default CAMELYON16, as in ``compress_slide``)."""
    pq, dec, code_map, (th, tw), _, (r0, c0, nr, nc), f = _region_plan(model, code_map, code_hw, region,
                                                                       batch, "decompress_region")
    shape = (nr * th * f, nc * tw * f, 3)
    if out is None:
        out = torch.empty(shape, dtype=torch.uint8, device=code_map.device)
    elif tuple(out.shape) != shape or out.dtype != torch.uint8 or out.device != code_map.device \
            or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous uint8 tensor of shape {shape} on {code_map.device}")
    total = nr * nc
    for first in range(0, total, batch):
        n = min(batch, total - first)
        enc = E.embed_codemap(pq, code_map, (th, tw), r0, c0, nc, first, n)
        P.decoder_forward_u8(dec, enc, mean, std, out, first, nc)
    return out


@torch.no_grad()
def compress_slide_scored(model, batches: Iterable[Tuple[int, torch.Tensor]], grid: Tuple[int, int],
                          code_hw: Tuple[int, int], device: torch.device, mean=None, std=None
                          ) -> Tuple[torch.Tensor, ReconstructionQuality]:
    """``compress_slide`` that also scores what the stored codes decode to.  For every
    (first_patch_index, uint8 [B,H,W,3] tiles) batch: encode, place the codes (the returned map is the
    one ``compress_slide`` returns), decode the batch's codes to uint8 pixels (``decode_codes_u8``) and
    score them against the tiles (``reconstruction_quality``).  The decoded pixels live for one batch.
    Returns ``(code_map, quality)``; ``quality`` holds per-patch maps ``sse`` [rows, cols, 3] and
    ``ssim`` [rows, cols] in slide order (patches no batch covers keep sse 0 and ssim NaN).  Reads
    ``model.encoder`` and ``model.decoder``; ``mean`` / ``std`` as in ``compress_slide``."""
    enc_mod, dec = model.encoder, model.decoder
    _check_u8_codes(enc_mod)
    P.check_u8_decoder(dec, "compress_slide_scored")
    rows, cols = grid
    th, tw = code_hw
    f = P.patch_scale(dec)
    hw = (th * f, tw * f)
    code_map = torch.zeros(rows * th, cols * tw, dtype=torch.uint8, device=device)
    sse = torch.zeros(rows * cols, 3, dtype=torch.int64, device=device)
    ssim = torch.full((rows * cols,), math.nan, dtype=torch.float64, device=device)
    vq = enc_mod.vq_layers[0]
    for first_patch, patches in batches:
        check_u8_patches(patches, "compress_slide_scored: a patch batch")
        if tuple(patches.shape[1:3]) != hw:
            raise ValueError(f"patches of {tuple(patches.shape[1:3])} pixels do not decode from "
                             f"{th} x {tw} code tiles ({hw[0]} x {hw[1]} pixels)")
        x = patches.to(device, non_blocking=True)
        idx = encode_patches(enc_mod, x, mean, std)
        E.codemap_place(idx, first_patch, cols, code_map)
        q = reconstruction_quality(x.contiguous(), P.decode_codes_u8(vq, dec, idx, mean, std))
        sse[first_patch:first_patch + len(idx)] = q.sse
        ssim[first_patch:first_patch + len(idx)] = q.ssim
    return code_map, ReconstructionQuality(sse.view(rows, cols, 3), ssim.view(rows, cols), hw)


@torch.no_grad()
def score_region(model, code_map: torch.Tensor, code_hw: Tuple[int, int], slide_u8: torch.Tensor,
                 region: Optional[Tuple[int, int, int, int]] = None, batch: int = 256, mean=None,
                 std=None) -> ReconstructionQuality:
    """Score a stored code map against the original slide: decode the region (as ``decompress_region``
    does, at most ``batch`` patches per step into one reused buffer) and compare each decoded batch with
    the slide's pixels in place.  ``slide_u8``: contiguous uint8 [rows*H, cols*W, 3] on the map's device,
    the whole slide the map was made from.  Returns per-patch maps ``sse`` [nr, nc, 3] and ``ssim``
    [nr, nc] of the region ``(r0, c0, nr, nc)`` (default the whole map).  Argument checks as in
    ``decompress_region``."""
    pq, dec, code_map, (th, tw), (rows, cols), (r0, c0, nr, nc), f = _region_plan(
        model, code_map, code_hw, region, batch, "score_region")
    h, w = th * f, tw * f
    shape = (rows * h, cols * w, 3)
    if not isinstance(slide_u8, torch.Tensor) or tuple(slide_u8.shape) != shape or \
            slide_u8.dtype != torch.uint8 or slide_u8.device != code_map.device or not slide_u8.is_contiguous():
        raise ValueError(f"slide_u8 must be a contiguous uint8 tensor of shape {shape} on {code_map.device}")
    total = nr * nc
    sse = torch.empty(total, 3, dtype=torch.int64, device=code_map.device)
    ssim = torch.empty(total, dtype=torch.float64, device=code_map.device)
    buf = torch.empty(min(batch, total) * h, w, 3, dtype=torch.uint8, device=code_map.device)
    for first in range(0, total, batch):
        n = min(batch, total - first)
        enc = E.embed_codemap(pq, code_map, (th, tw), r0, c0, nc, first, n)
        rec = buf[:n * h]
        P.decoder_forward_u8(dec, enc, mean, std, rec, 0, 1)
        sse[first:first + n], ssim[first:first + n] = E.quality_u8(slide_u8, (r0, c0, nc, first), rec,
                                                                   (0, 0, 1, 0), n, h, w)
    return ReconstructionQuality(sse.view(nr, nc, 3), ssim.view(nr, nc), (h, w))


def tiles_to_map(tiles_u8: torch.Tensor, grid: Tuple[int, int]) -> torch.Tensor:
    """[P,th,tw] tiles in row-major patch order -> [rows*th, cols*tw] map (pure view ops)."""
    rows, cols = grid
    p, th, tw = tiles_u8.shape
    assert p == rows * cols
    return tiles_u8.view(rows, cols, th, tw).permute(0, 2, 1, 3).reshape(rows * th, cols * tw)
