"""Residual layers of the config-5 slide: rate against the empirical entropy, and the time and peak memory of
encode_residual and decompress_region_exact against decompress_region alone.  Prints one JSON line (also
written to --out) with the GPU name and power limit read in the same run.

    python profiles/residual_bench.py [--precision fp16] [--batch 256] [--out FILE]

Config 5: a seeded 6240 x 6240 uint8 map (195 x 195 patches of 32 x 32 codes), the 256-model (n_down = 3) with
synthetic weights, batches of 256.  Two originals are made from the base decode x^: x^ + Laplacian noise of
scale 3 rounded and clamped ("laplace"), and uniform random bytes ("uniform").  For e in {0, 1, 2, 4} the
rate is the container's bits per pixel next to the sum over patches of each patch's empirical order-0
symbol entropy (from the exact GPU histograms).  Times are host clocks around work that ends in a device
synchronise; the three calls alternate, three times each; peaks are torch.cuda.max_memory_allocated after a
reset (the slide canvases, the model and the map included).  Every round trip is checked: equal to the
original at e = 0, within e otherwise."""
from __future__ import annotations

import argparse
import json
import math
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
from vqae_b200.extract import decompress_region, decompress_region_exact, encode_residual  # noqa: E402

DEV = torch.device("cuda:0")


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q.stdout.strip()}


def run(fn):
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats(DEV)
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0, torch.cuda.max_memory_allocated(DEV)


def laplace_like(base: torch.Tensor, scale: float, seed: int) -> torch.Tensor:
    g = torch.Generator(device=DEV).manual_seed(seed)
    out = torch.empty_like(base)
    step = 1024
    for r in range(0, base.shape[0], step):
        b = base[r:r + step]
        u = torch.rand(b.shape, generator=g, device=DEV) - 0.5
        lap = -scale * torch.sign(u) * torch.log1p(-2 * u.abs())
        out[r:r + step] = (b.float() + lap.round()).clamp(0, 255).to(torch.uint8)
    return out


def entropy_bits(slide, base, rows, cols, h, w, e, batch) -> float:
    bits = 0.0
    n = 3 * h * w
    for first in range(0, rows * cols, batch):
        k = min(batch, rows * cols - first)
        hist, _ = E.residual_stats(slide, (0, 0, cols, first), base, (0, 0, cols, first), k, h, w, e)
        c = hist.double()
        p = c / n
        bits += float(-(c * torch.where(c > 0, p.log2(), torch.zeros_like(p))).sum())
    return bits


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "residual_bench needs a CUDA device"
    info = card()
    model = vqae_b200.build_vqae(n_down=3).eval()
    model.load_state_dict(S.make_state_dict(model.state_dict(), seed=1, regime="perturbed"))
    model = vqae_b200.set_precision(model.to(DEV), args.precision)
    th = tw = 32
    rows = cols = 195
    h = w = 256
    px = rows * cols * h * w
    g = torch.Generator(device=DEV).manual_seed(5)
    code_map = torch.randint(0, 256, (rows * th, cols * tw), device=DEV, generator=g, dtype=torch.uint8)
    res = {"bench": "residual", **info, "precision": args.precision, "map": [rows * th, cols * tw],
           "patches": rows * cols, "batch": args.batch, "canvas_bytes": 3 * px}
    with torch.no_grad():
        base = decompress_region(model, code_map, (th, tw), batch=args.batch)
        originals = {"laplace": laplace_like(base, 3.0, 11),
                     "uniform": torch.randint(0, 256, base.shape, device=DEV, generator=g, dtype=torch.uint8)}
        rate = {}
        for name, slide in originals.items():
            rate[name] = {}
            for e in (0, 1, 2, 4):
                layer = encode_residual(model, code_map, (th, tw), slide, max_error=e, batch=args.batch)
                ent = entropy_bits(slide, base, rows, cols, h, w, e, args.batch)
                got = decompress_region_exact(model, code_map, (th, tw), layer, batch=args.batch)
                err = int((got.int() - slide.int()).abs().max()) if e else int(not torch.equal(got, slide))
                assert err <= e, (name, e, err)
                rate[name][str(e)] = {"bits_per_pixel": round(layer.bits_per_pixel(), 4),
                                      "entropy_bits_per_pixel": round(ent / px, 4),
                                      "payload_over_entropy": round(8 * layer.payload_bytes / ent, 4)
                                      if ent else None, "max_abs_error": err}
                del layer, got
        res["rate"] = rate

        slide = originals["laplace"]
        del originals["uniform"]
        out = torch.empty_like(base)
        layer = encode_residual(model, code_map, (th, tw), slide, max_error=0, batch=args.batch)
        calls = {"decompress_region": lambda: decompress_region(model, code_map, (th, tw), batch=args.batch, out=out),
                 "encode_residual": lambda: encode_residual(model, code_map, (th, tw), slide, 0, args.batch),
                 "decompress_region_exact": lambda: decompress_region_exact(model, code_map, (th, tw), layer,
                                                                            batch=args.batch, out=out)}
        for fn in calls.values():                                               # warm-up
            run(fn)
        times = {k: [] for k in calls}
        peaks = {k: 0 for k in calls}
        for _ in range(3):
            for k, fn in calls.items():
                o, sec, peak = run(fn)
                del o
                times[k].append(sec)
                peaks[k] = max(peaks[k], peak)
        assert torch.equal(decompress_region_exact(model, code_map, (th, tw), layer, batch=args.batch), slide)
        base_s = min(times["decompress_region"])
        res["timing_e0_laplace"] = {k: {"s": round(min(v), 4), "s_runs": [round(t, 4) for t in v],
                                        "over_decode": round(min(v) / base_s - 1, 4),
                                        "peak_allocated_GB": round(peaks[k] / 1e9, 3)} for k, v in times.items()}
        res["timing_e0_laplace"]["residual_ms_per_batch"] = {
            k: round((min(times[k]) - base_s) * 1e3 / math.ceil(rows * cols / args.batch), 3)
            for k in ("encode_residual", "decompress_region_exact")}
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
