"""Reconstruction scoring on the GPU: the vqae_quality_u8 kernel (per-patch SSE + SSIM) against the same
metric written with torch ops, and the cost of scoring inside a slide round trip.  Prints one JSON line
(also written to --out).

    python profiles/quality_bench.py [--reps 3] [--out FILE]

* Kernel time: batch 256 of 256^2 and batch 64 of 512^2 (100.7 MB of input per call at either size).
  Three input sets are rotated (302 MB, more than the 126 MB L2), so every call reads its inputs from
  HBM.  CUDA events around 10 calls, warmed up, best of --reps runs alternated with the baseline.
* Floors: the algorithmic bytes are the two uint8 images (6 B per pixel).  FLOPs are counted from the
  definition (separable filtering of the five moments plus the SSIM formula, see ``flops_per_patch``).
  The kernel accumulates in fp64, so the arithmetic floor is given for the fp64 rate as well as for the
  fp32 rate; both are estimates from SM count x lanes x clock, not measurements.
* Baseline: five grouped ``conv2d`` in fp32 (x, y, x^2, y^2, xy; the outer product of the same fp32 taps;
  valid padding; TF32 off), the SSIM formula in fp32, SSE in int64.  Reports the speed-up and
  max |ssim - baseline|.
* Scoring overhead: a seeded slide of 64 x 64 patches of 256^2 in "fp16": ``compress_slide`` +
  ``decompress_region`` against ``compress_slide_scored``, patches/s for both.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn.functional as F

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO / "2d-vq-ae-2_b200"))

import vqae_b200  # noqa: E402
from vqae_b200 import engine as E  # noqa: E402
from vqae_b200 import synthetic as S  # noqa: E402
from vqae_b200.extract import compress_slide, compress_slide_scored, decompress_region  # noqa: E402
from vqae_b200.quality import reconstruction_quality  # noqa: E402

DEV = torch.device("cuda:0")
C1, C2 = (0.01 * 255) ** 2, (0.03 * 255) ** 2


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q.stdout.strip()}


def max_sm_clock_hz() -> float:
    q = subprocess.run(["nvidia-smi", "--query-gpu=clocks.max.sm", "--format=csv,noheader,nounits", "-i", "0"],
                       capture_output=True, text=True)
    return float(q.stdout.strip().splitlines()[0]) * 1e6


def timed(fn, reps: int = 1) -> float:
    """Seconds per call, CUDA events around `reps` calls."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def flops_per_patch(h: int, w: int) -> int:
    """Per channel: x^2, y^2, xy at every pixel (3), the horizontal 11-tap pass of five moments over
    h x (w - 10) (110 per output), the vertical pass over (h - 10) x (w - 10) (110), the SSIM formula
    (20: three variances 6, numerator 5, denominator 6, two products and a division 3)."""
    hv, wv = h - 10, w - 10
    return 3 * (3 * h * w + 110 * h * wv + 110 * hv * wv + 20 * hv * wv)


def taps_f32() -> torch.Tensor:
    k = torch.arange(-5, 6, dtype=torch.float64)
    g = torch.exp(-k * k / (2 * 1.5 ** 2))
    return (g / g.sum()).float()


def torch_metric(ref: torch.Tensor, rec: torch.Tensor, w2: torch.Tensor):
    """The same metric with torch ops: int64 SSE, fp32 grouped conv2d moments (valid), fp32 SSIM."""
    d = ref.long() - rec.long()
    sse = (d * d).sum((1, 2))
    x = ref.permute(0, 3, 1, 2).float()
    y = rec.permute(0, 3, 1, 2).float()
    m = F.conv2d(torch.cat([x, y, x * x, y * y, x * y], 1), w2.expand(15, 1, 11, 11), groups=15)
    mx, my, exx, eyy, exy = m.split(3, 1)
    sxx, syy, sxy = exx - mx * mx, eyy - my * my, exy - mx * my
    s = ((2 * mx * my + C1) * (2 * sxy + C2)) / ((mx * mx + my * my + C1) * (sxx + syy + C2))
    return sse, s.mean((1, 2, 3))


def kernel_vs_torch(batch: int, size: int, reps: int, sm: int, clock: float, copy_gbps: float) -> dict:
    g = torch.Generator(device=DEV).manual_seed(size)
    sets = []
    for _ in range(3):
        ref = torch.randint(0, 256, (batch, size, size, 3), device=DEV, generator=g, dtype=torch.uint8)
        rec = (ref.short() + torch.randint(-12, 13, ref.shape, device=DEV, generator=g, dtype=torch.int16))
        sets.append((ref, rec.clamp(0, 255).to(torch.uint8)))
    w2 = torch.outer(taps_f32(), taps_f32()).to(DEV)[None, None]
    state = {"i": 0}

    def run_kernel():
        ref, rec = sets[state["i"] % 3]
        state["i"] += 1
        reconstruction_quality(ref, rec)

    def run_torch():
        ref, rec = sets[state["i"] % 3]
        state["i"] += 1
        torch_metric(ref, rec, w2)

    run_kernel(), run_torch()
    t_k, t_t = [], []
    for _ in range(reps):
        t_k.append(timed(run_kernel, 10))
        t_t.append(timed(run_torch, 3))
    ref, rec = sets[0]
    q = reconstruction_quality(ref, rec)
    sse_t, ssim_t = torch_metric(ref, rec, w2)
    flops = flops_per_patch(size, size) * batch
    nbytes = 6 * batch * size * size
    tk = min(t_k)
    return {
        "batch": batch, "size": size, "kernel_us": round(tk * 1e6, 1), "kernel_us_runs": [round(v * 1e6, 1) for v in t_k],
        "torch_us": round(min(t_t) * 1e6, 1), "speedup_vs_torch": round(min(t_t) / tk, 2),
        "bytes": nbytes, "GBps": round(nbytes / tk / 1e9, 1), "share_of_copy_bandwidth": round(nbytes / tk / 1e9 / copy_gbps, 4),
        "flops": flops, "GFLOPs": round(flops / tk / 1e9, 1),
        "floor_bytes_us": round(nbytes / (copy_gbps * 1e9) * 1e6, 1),
        "floor_fp32_estimate_us": round(flops / (sm * 128 * 2 * clock) * 1e6, 1),
        "floor_fp64_estimate_us": round(flops / (sm * 64 * 2 * clock) * 1e6, 1),
        "sse_equal_torch": bool(torch.equal(q.sse, sse_t)),
        "max_abs_ssim_minus_torch_fp32": float((q.ssim - ssim_t.double()).abs().max()),
    }


def hbm_copy_GBps() -> float:
    a = torch.empty(2 << 30, dtype=torch.uint8, device=DEV)
    b = torch.empty_like(a)
    b.copy_(a)
    sec = min(timed(lambda: b.copy_(a), 5) for _ in range(3))
    return 2 * a.numel() / sec / 1e9


def scoring_overhead(reps: int) -> dict:
    model = vqae_b200.build_vqae(n_down=3).eval()
    model.load_state_dict(S.make_state_dict(model.state_dict(), seed=1, regime="perturbed"))
    model = vqae_b200.set_precision(model.to(DEV), "fp16")
    rows = cols = 64
    batch = 256
    tiles = S.synthetic_patches_u8(batch, 256, 12).to(DEV)
    batches = [(first, tiles) for first in range(0, rows * cols, batch)]
    code_hw = (32, 32)

    def plain():
        cm = compress_slide(model.encoder, batches, (rows, cols), code_hw, DEV)
        decompress_region(model, cm, code_hw, batch=batch)

    def scored():
        compress_slide_scored(model, batches, (rows, cols), code_hw, DEV)

    with torch.no_grad():
        plain(), scored()
        t_p, t_s = [], []
        for _ in range(reps):
            t_p.append(timed(plain))
            t_s.append(timed(scored))
        cm = compress_slide(model.encoder, batches, (rows, cols), code_hw, DEV)
        cm2, q = compress_slide_scored(model, batches, (rows, cols), code_hw, DEV)
    n = rows * cols
    return {"precision": "fp16", "patches": n, "batch": batch,
            "compress_plus_decompress_s": round(min(t_p), 4), "compress_scored_s": round(min(t_s), 4),
            "compress_plus_decompress_patches_per_s": round(n / min(t_p), 1),
            "compress_scored_patches_per_s": round(n / min(t_s), 1),
            "code_maps_equal": bool(torch.equal(cm, cm2)), "summary": q.summary()}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "quality_bench needs a CUDA device"
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    info = card()
    clock = max_sm_clock_hz()
    sm = torch.cuda.get_device_properties(DEV).multi_processor_count
    copy = hbm_copy_GBps()
    with torch.no_grad():
        kern = [kernel_vs_torch(256, 256, args.reps, sm, clock, copy), kernel_vs_torch(64, 512, args.reps, sm, clock, copy)]
    res = {"bench": "quality_u8", **info, "sm_count": sm, "max_sm_clock_MHz": clock / 1e6,
           "hbm_copy_GBps": round(copy, 1), "kernel": kern, "scoring_overhead": scoring_overhead(args.reps)}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
