"""DeepZoom JPEG tiles: the GPU encoder against Pillow on a host thread pool, and export_deepzoom of the config-5
slide phase by phase.  Prints one JSON line (also written to --out) with the GPU name and power limit read in
the same run.
    python profiles/jpeg_bench.py [--precision fp16] [--level-patches 40] [--export-patches 195] [--out FILE]
Level: the decode of a seeded map of level-patches^2 patches of 256^2 (the 256-model, n_down = 3, synthetic
weights), tiled at T = 254 with overlap 1 (tiles of up to 256 px), q = 90, for both subsamplings.  GPU time:
host clock around encode_tiles (payload trimmed, offsets on the host), which ends in a device synchronise;
warm-up, then the best of 5.  Pillow: the same tiles, cropped from the host copy of the level, encoded with
Image.save(quality=90, subsampling=s) on os.cpu_count() threads, best of 2; every GPU tile is checked equal to
Pillow's.  Export: export_deepzoom of an export-patches^2 map to a temporary directory (removed afterwards),
its own per-phase seconds, and torch.cuda.max_memory_allocated after a reset (the model and map included)."""
from __future__ import annotations

import argparse
import io
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO / "2d-vq-ae-2_b200"))

import vqae_b200  # noqa: E402
from vqae_b200 import jpeg as J  # noqa: E402
from vqae_b200 import synthetic as S  # noqa: E402
from vqae_b200.extract import decompress_region, export_deepzoom  # noqa: E402

DEV = torch.device("cuda:0")


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q.stdout.strip()}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--level-patches", type=int, default=40)
    ap.add_argument("--export-patches", type=int, default=195)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "jpeg_bench needs a CUDA device"
    from PIL import Image
    res = {"bench": "jpeg", **card(), "precision": args.precision, "cpu_count": os.cpu_count()}
    model = vqae_b200.build_vqae(n_down=3).eval()
    model.load_state_dict(S.make_state_dict(model.state_dict(), seed=1, regime="perturbed"))
    model = vqae_b200.set_precision(model.to(DEV), args.precision)
    g = torch.Generator(device=DEV).manual_seed(5)
    n = args.level_patches
    with torch.no_grad():
        cm = torch.randint(0, 256, (n * 32, n * 32), device=DEV, generator=g, dtype=torch.uint8)
        level = decompress_region(model, cm, (32, 32))
    img = level.cpu().numpy()
    h, w = img.shape[:2]
    cols, rows = J.tile_grid(w, h, 254)
    rects = [J.tile_rect(c, r, w, h, 254, 1) for r in range(rows) for c in range(cols)]
    res["level"] = {"height": h, "width": w, "tiles": len(rects), "tile": 254, "overlap": 1, "quality": 90}
    for s in (0, 2):
        timed(lambda: J.encode_tiles(level, 254, 1, 90, s))                                # warm-up
        gpu = []
        for _ in range(5):
            tiles, sec = timed(lambda: J.encode_tiles(level, 254, 1, 90, s))
            gpu.append(sec)
        host = tiles.payload.cpu().numpy()

        def pil(rect):
            x0, y0, x1, y1 = rect
            buf = io.BytesIO()
            Image.fromarray(np.ascontiguousarray(img[y0:y1, x0:x1])).save(buf, "JPEG", quality=90, subsampling=s)
            return buf.getvalue()

        cpu = []
        with ThreadPoolExecutor(os.cpu_count()) as ex:
            for _ in range(2):
                t0 = time.perf_counter()
                want = list(ex.map(pil, rects))
                cpu.append(time.perf_counter() - t0)
        assert all(tiles.tile_bytes(i % cols, i // cols, host) == want[i] for i in range(len(rects))), s
        res[f"subsampling_{s}"] = {
            "gpu_s": round(min(gpu), 5), "gpu_s_runs": [round(t, 5) for t in gpu],
            "gpu_tiles_per_s": round(len(rects) / min(gpu)), "pillow_s": round(min(cpu), 4),
            "pillow_s_runs": [round(t, 4) for t in cpu], "pillow_tiles_per_s": round(len(rects) / min(cpu)),
            "gpu_speedup": round(min(cpu) / min(gpu), 2), "payload_bytes": tiles.nbytes(), "bytes_equal": True}
        del tiles
    del level

    n = args.export_patches
    with torch.no_grad():
        cm = torch.randint(0, 256, (n * 32, n * 32), device=DEV, generator=g, dtype=torch.uint8)
    out = Path(tempfile.mkdtemp(prefix="dz_bench_"))
    try:
        torch.cuda.synchronize()
        torch.cuda.reset_peak_memory_stats(DEV)
        t0 = time.perf_counter()
        info = export_deepzoom(model, cm, (32, 32), out, "slide", quality=90, subsampling=2)
        total = time.perf_counter() - t0
        res["export"] = {"patches": n * n, "pixels": (n * 256) ** 2, "levels": info["levels"],
                         "tiles": info["tiles"], "bytes": info["bytes"], "total_s": round(total, 3),
                         "phases_s": {k: round(v, 3) for k, v in info["seconds"].items()},
                         "peak_allocated_GB": round(torch.cuda.max_memory_allocated(DEV) / 1e9, 3)}
    finally:
        shutil.rmtree(out, ignore_errors=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
