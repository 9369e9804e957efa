"""Pyramid levels of uint8 RGB slides: the pyramid kernel (csrc/pyramid.cu) against the same levels written
in torch, and, for the config-5 slide, decompress_region followed by slide_pyramid against
decompress_pyramid.  Prints one JSON line (also written to --out).

    python profiles/pyramid_bench.py [--precision fp16] [--reps 20] [--out FILE]

Kernel: batch 256 of 256^2 patches, every factor 2 .. 256 in one launch, timed with CUDA events over
`reps` launches after a warm-up; the launches rotate over 4 inputs (201 MB, more than the 126 MB L2).
Algorithmic bytes = 3 B read per pixel + 3 B / f^2 written per pixel and level; reported over the kernel
time and against a device-to-device copy measured in the same run.  The torch formulation converts the
batch to int32 once, then per level reshape-sums, rounds half up, narrows and places into its canvas.

Config 5: a seeded 6240 x 6240 uint8 map (195 x 195 patches of 32 x 32 codes), the 256-model
(n_down = 3), batches of 256, factors (2, 4, 16, 256).  The two ways alternate, three times each; each
run's time is a host clock around work that ends in a device synchronise, and its peak is
torch.cuda.max_memory_allocated after a reset, both absolute (the model, the map and the other way's last
levels included) and above what was allocated at the start of the run.  The levels of both ways must
be equal."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO / "2d-vq-ae-2_b200"))

import vqae_b200  # noqa: E402
from vqae_b200 import engine as E  # noqa: E402
from vqae_b200 import synthetic as S  # noqa: E402
from vqae_b200.extract import decompress_pyramid, decompress_region  # noqa: E402
from vqae_b200.pyramid import slide_pyramid  # noqa: E402

DEV = torch.device("cuda:0")


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q.stdout.strip(),
            "sm_count": torch.cuda.get_device_properties(DEV).multi_processor_count}


def timed(fn, reps: int) -> float:
    """Seconds per call, CUDA events around `reps` calls."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for i in range(reps):
        fn(i)
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def hbm_copy_GBps() -> float:
    a = torch.empty(2 << 30, dtype=torch.uint8, device=DEV)
    b = torch.empty_like(a)
    b.copy_(a)
    sec = min(timed(lambda i: b.copy_(a), 5) for _ in range(3))
    return 2 * a.numel() / sec / 1e9


def torch_levels(x, h, w, factors, out):
    """x: uint8 [n, h, w, 3] -> out[f] uint8 [n*h/f, w/f, 3], the same definition in torch."""
    n = x.shape[0]
    xi = x.to(torch.int32)
    for f in factors:
        s = xi.view(n, h // f, f, w // f, f, 3).sum((2, 4), dtype=torch.int32)
        out[f].view(n, h // f, w // f, 3).copy_(((s + f * f // 2) >> (2 * (f.bit_length() - 1))).to(torch.uint8))


def kernel_bench(reps: int) -> dict:
    n, h, w = 256, 256, 256
    factors = tuple(1 << k for k in range(1, 9))
    g = torch.Generator(device=DEV).manual_seed(7)
    xs = [torch.randint(0, 256, (n, h, w, 3), device=DEV, generator=g, dtype=torch.uint8) for _ in range(4)]
    mine = {f: torch.empty(n * (h // f), w // f, 3, dtype=torch.uint8, device=DEV) for f in factors}
    ref = {f: torch.empty_like(v) for f, v in mine.items()}
    run_mine = lambda i: E.pyramid_u8(xs[i % 4].view(n * h, w, 3), (0, 0, 1, 0), n, h, w, mine,  # noqa: E731
                                      (0, 0, 1, 0))
    run_torch = lambda i: torch_levels(xs[i % 4], h, w, factors, ref)                           # noqa: E731
    for i in range(4):
        run_mine(i)
        run_torch(i)
    t_mine, t_torch = [], []
    for _ in range(3):                                                                         # alternated
        t_mine.append(timed(run_mine, reps))
        t_torch.append(timed(run_torch, max(reps // 10, 2)))
    run_mine(0)
    run_torch(0)
    equal = all(torch.equal(mine[f], ref[f]) for f in factors)
    px = n * h * w
    nbytes = px * 3 + sum(px * 3 // (f * f) for f in factors)
    sec = min(t_mine)
    return {"batch": n, "size": h, "factors": list(factors), "kernel_us": round(sec * 1e6, 2),
            "kernel_us_runs": [round(v * 1e6, 2) for v in t_mine], "torch_us": round(min(t_torch) * 1e6, 1),
            "speedup_vs_torch": round(min(t_torch) / sec, 2), "algorithmic_bytes": nbytes,
            "GBps": round(nbytes / sec / 1e9, 1), "levels_equal_torch": equal}


def slide_bench(precision: str, batch: int) -> dict:
    model = vqae_b200.build_vqae(n_down=3).eval()
    model.load_state_dict(S.make_state_dict(model.state_dict(), seed=1, regime="perturbed"))
    model = vqae_b200.set_precision(model.to(DEV), precision)
    th = tw = 32
    rows = cols = 195
    g = torch.Generator(device=DEV).manual_seed(5)
    code_map = torch.randint(0, 256, (rows * th, cols * tw), device=DEV, generator=g, dtype=torch.uint8)
    factors = (2, 4, 16, 256)

    def two_step():
        return slide_pyramid(decompress_region(model, code_map, (th, tw), batch=batch), (256, 256), factors)

    def fused():
        return decompress_pyramid(model, code_map, (th, tw), factors, batch=batch)

    def run(fn):
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(DEV)
        base = torch.cuda.memory_allocated(DEV)
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        return out, time.perf_counter() - t0, torch.cuda.max_memory_allocated(DEV), base

    with torch.no_grad():
        for fn in (two_step, fused):                                # warm-up, then drop the outputs
            run(fn)
        res = {"two_step": [], "fused": []}
        outs = {}
        for _ in range(3):
            for name, fn in (("two_step", two_step), ("fused", fused)):
                outs[name] = None
                o, sec, peak, base = run(fn)
                outs[name] = o
                res[name].append((sec, peak, base))
        equal = all(torch.equal(outs["two_step"][f], outs["fused"][f]) for f in factors)
    out = {"precision": precision, "map": [rows * th, cols * tw], "patches": rows * cols, "batch": batch,
           "factors": list(factors), "full_canvas_bytes": rows * 256 * cols * 256 * 3,
           "level_bytes": {str(f): int(outs["fused"][f].numel()) for f in factors}, "levels_equal": equal}
    for name, runs in res.items():
        out[name] = {"s": round(min(r[0] for r in runs), 4), "s_runs": [round(r[0], 4) for r in runs],
                     "peak_allocated_GB": round(max(r[1] for r in runs) / 1e9, 3),
                     "peak_above_start_GB": round(max(r[1] - r[2] for r in runs) / 1e9, 3)}
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "pyramid_bench needs a CUDA device"
    info = card()
    with torch.no_grad():
        kern = kernel_bench(args.reps)
    peak = hbm_copy_GBps()
    kern["share_of_copy_bandwidth"] = round(kern["GBps"] / peak, 3)
    slide = slide_bench(args.precision, args.batch)
    res = {"bench": "pyramid_u8", **info, "hbm_copy_GBps": round(peak, 1), "kernel": kern, "config5_slide": slide}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
