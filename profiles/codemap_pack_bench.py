"""Rate and cost of packed code maps (vqae_b200.packing): one JSON line per map.

    python profiles/codemap_pack_bench.py [--reps 5] [--out FILE]

Maps (all 6 240 x 6 240 = 195 x 195 tiles of 32 x 32 codes, BASELINE.json config 5):
  slide_perturbed / slide_fixup  the synthetic whole slide of profiles/slide_bench.py (uniform random uint8
                                 pixels per patch, seeded by the patch index) compressed by the 256-model
                                 (n_down = 3) in "fp16", weights from synthetic.make_state_dict in either
                                 regime.  These are synthetic-model maps: the rate on a trained checkpoint
                                 is not measured here.
  uniform256                     uniform random uint8 codes (the incompressible case)
  k1024_int64                    uniform random int64 codes over 1024 symbols
Per map: raw bytes (as stored: uint8 or int64), container bytes and payload bytes, bits per code and per
pixel at 256^2 patches, the empirical entropy bound N H / 8 and the ideal length under the quantised
table, zlib level 9 of the raw map on the host, and device times from CUDA events after a warm-up,
alternated over --reps runs: pack_code_map (histogram, table, pack kernels, offsets read back), the
histogram and pack kernels alone, unpack_code_map of the whole map and of one patch, next to
decompress_region of the same map (uint8 maps).  The card's name and power limit are read in the run."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import zlib
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO / "2d-vq-ae-2_b200"))

import vqae_b200  # noqa: E402
from vqae_b200 import engine as E  # noqa: E402
from vqae_b200 import synthetic as S  # noqa: E402
from vqae_b200.extract import compress_slide, decompress_region  # noqa: E402
from vqae_b200.packing import SCALE_BITS, pack_code_map, quantise_frequencies, unpack_code_map  # noqa: E402

DEV = torch.device("cuda:0")
ROWS = COLS = 195
TH = TW = 32
PATCH = 256


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q.stdout.strip()}


def timed(fn, reps: int = 1) -> float:
    """Seconds per call, CUDA events around ``reps`` calls."""
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3 / reps


def slide_batches(batch: int = 256):
    """(first patch, uint8 [n,256,256,3]) of the slide of profiles/slide_bench.py, generated per batch."""
    g = torch.Generator(device=DEV)
    total = ROWS * COLS
    for first in range(0, total, batch):
        n = min(batch, total - first)
        out = torch.empty(n, PATCH, PATCH, 3, dtype=torch.uint8, device=DEV)
        for i in range(n):
            g.manual_seed(1234 + first + i)
            out[i] = torch.randint(0, 256, (PATCH, PATCH, 3), dtype=torch.uint8, device=DEV, generator=g)
        yield first, out


def slide_map(model) -> torch.Tensor:
    with torch.no_grad():
        return compress_slide(model.encoder, slide_batches(), (ROWS, COLS), (TH, TW), DEV)


def measure(name: str, code_map: torch.Tensor, model, reps: int, k=None) -> dict:
    host = code_map.cpu().numpy()
    counts = np.bincount(host.astype(np.int64).ravel())
    N = int(counts.sum())
    p = counts[counts > 0] / N
    entropy_bytes = float(-(counts[counts > 0] * np.log2(p)).sum() / 8)
    packed = pack_code_map(code_map, (TH, TW), k=k)
    f = packed.freq_host.astype(np.float64)
    cnt = np.bincount(host.astype(np.int64).ravel(), minlength=packed.k)
    used = cnt > 0
    table_bytes = float((cnt[used] * (SCALE_BITS - np.log2(f[used]))).sum() / 8)
    assert torch.equal(unpack_code_map(packed, dtype=code_map.dtype), code_map)

    freq = quantise_frequencies(packed.counts.cpu().numpy())
    fns = {
        "pack_code_map": lambda: pack_code_map(code_map, (TH, TW), k=k),
        "histogram_kernel": lambda: E.codemap_histogram(code_map, packed.k),
        "pack_kernels": lambda: E.codemap_pack(code_map, (TH, TW), freq, SCALE_BITS),
        "unpack_whole": lambda: unpack_code_map(packed, dtype=code_map.dtype),
        "unpack_one_patch": lambda: unpack_code_map(packed, (97, 97, 1, 1), dtype=code_map.dtype),
    }
    decomp = code_map.dtype == torch.uint8 and model is not None
    if decomp:
        canvas = torch.empty(ROWS * PATCH, COLS * PATCH, 3, dtype=torch.uint8, device=DEV)
        fns["decompress_region"] = lambda: decompress_region(model, code_map, (TH, TW), out=canvas)
    with torch.no_grad():
        for fn in fns.values():                                     # warm-up of every shape
            fn()
        t = {k_: [] for k_ in fns}
        for _ in range(reps):                                       # alternated
            for k_, fn in fns.items():
                t[k_].append(timed(fn, 1 if k_ == "decompress_region" else 5))
    raw = host.nbytes
    res = {
        "map": name, "shape": list(code_map.shape), "dtype": str(code_map.dtype).replace("torch.", ""),
        "k": packed.k, "distinct_codes": int(used.sum()), "raw_bytes": raw, "packed_bytes": packed.nbytes(),
        "payload_bytes": packed.payload_bytes, "ratio_vs_raw": round(packed.nbytes() / raw, 5),
        "bits_per_code": round(packed.bits_per_code(), 5),
        "payload_bits_per_code": round(8 * packed.payload_bytes / N, 5),
        "bits_per_pixel_256": round(packed.bits_per_pixel((PATCH, PATCH)), 7),
        "entropy_bound_bytes": round(entropy_bytes, 1), "entropy_bits_per_code": round(8 * entropy_bytes / N, 5),
        "quantised_table_bound_bytes": round(table_bytes, 1),
        "zlib9_bytes": len(zlib.compress(host.tobytes(), 9)),
        "times_ms": {k_: [round(v * 1e3, 4) for v in vals] for k_, vals in t.items()},
        "best_ms": {k_: round(min(vals) * 1e3, 4) for k_, vals in t.items()},
    }
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "codemap_pack_bench needs a CUDA device"
    info = card()
    lines = []
    model = None
    for regime in ("perturbed", "fixup"):
        model = vqae_b200.build_vqae(n_down=3).eval()
        model.load_state_dict(S.make_state_dict(model.state_dict(), seed=1, regime=regime))
        model = vqae_b200.set_precision(model.to(DEV), "fp16")
        cmap = slide_map(model)
        lines.append(measure(f"slide_{regime}", cmap, model, args.reps))
    g = torch.Generator(device=DEV).manual_seed(5)
    uni = torch.randint(0, 256, (ROWS * TH, COLS * TW), device=DEV, generator=g, dtype=torch.uint8)
    lines.append(measure("uniform256", uni, model, args.reps))
    k1024 = torch.randint(0, 1024, (ROWS * TH, COLS * TW), device=DEV, generator=g, dtype=torch.int64)
    lines.append(measure("k1024_int64", k1024, None, args.reps, k=1024))
    out = []
    for res in lines:
        line = json.dumps({"bench": "codemap_pack", **info, **res})
        print(line, flush=True)
        out.append(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(out) + "\n")


if __name__ == "__main__":
    main()
