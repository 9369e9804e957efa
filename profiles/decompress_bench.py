"""Decompression of a stored slide code map to uint8 RGB: extract.decompress_region against the
same slide decoded the way a caller without it does (decode_codes per batch -> torch de-normalise /
round / clamp -> permute -> stitch by indexing), plus out_stem kernel times of the uint8 and the fp32
NHWC outputs.  Prints one JSON line (also written to --out).

    python profiles/decompress_bench.py [--precision fp16] [--reps 3] [--out FILE]

Geometry of config 5: a seeded 6240 x 6240 uint8 map (195 x 195 patches of 32 x 32 codes), the
256-model (n_down = 3), batches of 256 patches.  Both ways run in this process, alternated, timed with
CUDA events; the two canvases must agree (equal except where the float value lies within 1e-3 of a
half-integer, and there by one level).  The out_stem figures use batch 256 of 256^2 (537 MB of input,
more than L2 holds) and report the algorithmic bytes (32 B in + 3 B or 12 B out per pixel) over the
kernel time against the HBM bandwidth of a device-to-device copy measured in the same run."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO / "2d-vq-ae-2_b200"))

import vqae_b200  # noqa: E402
from vqae_b200 import engine as E  # noqa: E402
from vqae_b200 import synthetic as S  # noqa: E402
from vqae_b200.extract import decompress_region  # noqa: E402

DEV = torch.device("cuda:0")


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                        "-i", "0"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(DEV), "nvidia_smi": q.stdout.strip()}


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


def user_way(model, code_map, th, tw, batch, s, o, canvas):
    rows, cols = code_map.shape[0] // th, code_map.shape[1] // tw
    tiles_all = code_map.view(rows, th, cols, tw).permute(0, 2, 1, 3)
    ph, pw = canvas.shape[0] // rows, canvas.shape[1] // cols
    view = canvas.view(rows, ph, cols, pw, 3)
    total = rows * cols
    for first in range(0, total, batch):
        ids = torch.arange(first, min(first + batch, total), device=code_map.device)
        pr, pc = ids // cols, ids % cols
        f = model.decode_codes(tiles_all[pr, pc])                               # fp32 [n,3,H,W]
        u = (f * s[:, None, None] + o[:, None, None]).round_().clamp_(0, 255).to(torch.uint8)
        view[pr, :, pc] = u.permute(0, 2, 3, 1)
    return canvas


def check_agreement(model, code_map, th, tw, batch, fused):
    """The rule of tests/test_gpu_decompress.py: equal except within 1e-3 of a half-integer (there by 1)."""
    rows, cols = code_map.shape[0] // th, code_map.shape[1] // tw
    tiles_all = code_map.view(rows, th, cols, tw).permute(0, 2, 1, 3)
    s = (torch.tensor(E.CAMELYON16_STD, dtype=torch.float32) * 255).double().to(DEV)
    o = (torch.tensor(E.CAMELYON16_MEAN, dtype=torch.float32) * 255).double().to(DEV)
    ph, pw = fused.shape[0] // rows, fused.shape[1] // cols
    view = fused.view(rows, ph, cols, pw, 3)
    n_diff = 0
    for first in range(0, rows * cols, batch):
        ids = torch.arange(first, min(first + batch, rows * cols), device=DEV)
        pr, pc = ids // cols, ids % cols
        pre = model.decode_codes(tiles_all[pr, pc]).permute(0, 2, 3, 1).double() * s + o
        ref = pre.round().clamp(0, 255)
        d = (view[pr, :, pc].double() - ref).abs()
        near = (pre - pre.floor() - 0.5).abs() < 1e-3
        assert not bool((d[~near] > 0).any()), "fused canvas differs from the float path"
        assert float(d.max()) <= 1
        n_diff += int((d > 0).sum())
    return n_diff


def stem_times(precision: str, reps: int) -> dict:
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(256, 256, 256, 8, device=DEV, generator=g)
    w = torch.randn(3, 8, 3, 3, device=DEV, generator=g) * 0.1
    b = torch.randn(3, device=DEV, generator=g) * 0.1
    canvas = torch.empty(256 * 256, 256, 3, dtype=torch.uint8, device=DEV)
    f32 = lambda: E.stem_out(x, w, b, True, precision)                          # noqa: E731
    u8 = lambda: E.stem_out_u8(x, w, b, canvas, 0, 1, precision=precision)      # noqa: E731
    for fn in (f32, u8):
        fn()
    t = {"fp32_nhwc": [], "u8": []}
    for _ in range(3):                                                          # alternated
        t["fp32_nhwc"].append(timed(f32, reps))
        t["u8"].append(timed(u8, reps))
    npix = 256 * 256 * 256
    out = {}
    for k, per_px in (("fp32_nhwc", 32 + 12), ("u8", 32 + 3)):
        sec = min(t[k])
        out[k] = {"us": round(sec * 1e6, 1), "us_all": [round(v * 1e6, 1) for v in t[k]],
                  "algorithmic_bytes": npix * per_px, "GBps": round(npix * per_px / sec / 1e9, 1)}
    return out


def hbm_copy_GBps() -> float:
    a = torch.empty(2 << 30, dtype=torch.uint8, device=DEV)
    b = torch.empty_like(a)
    b.copy_(a)
    sec = min(timed(lambda: b.copy_(a), 5) for _ in range(3))
    return 2 * a.numel() / sec / 1e9


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=256)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "decompress_bench needs a CUDA device"
    info = card()

    model = vqae_b200.build_vqae(n_down=3).eval()
    model.load_state_dict(S.make_state_dict(model.state_dict(), seed=1, regime="perturbed"))
    model = vqae_b200.set_precision(model.to(DEV), args.precision)
    th = tw = 32
    rows = cols = 195
    g = torch.Generator(device=DEV).manual_seed(5)
    code_map = torch.randint(0, 256, (rows * th, cols * tw), device=DEV, generator=g, dtype=torch.uint8)
    s = (torch.tensor(E.CAMELYON16_STD, dtype=torch.float32) * 255).to(DEV)
    o = (torch.tensor(E.CAMELYON16_MEAN, dtype=torch.float32) * 255).to(DEV)
    fused = torch.empty(rows * 256, cols * 256, 3, dtype=torch.uint8, device=DEV)
    ref = torch.empty_like(fused)

    with torch.no_grad():
        # warm-up of every shape the timed window uses (full batches and the short last one)
        decompress_region(model, code_map, (th, tw), batch=args.batch, out=fused)
        user_way(model, code_map, th, tw, args.batch, s, o, ref)
        t_fused, t_user = [], []
        for _ in range(args.reps):
            t_fused.append(timed(lambda: decompress_region(model, code_map, (th, tw), batch=args.batch,
                                                           out=fused)))
            t_user.append(timed(lambda: user_way(model, code_map, th, tw, args.batch, s, o, ref)))
        n_diff = check_agreement(model, code_map, th, tw, args.batch, fused)
        n_diff_user = int((fused != ref).sum())
        stems = {p: stem_times(p, 20) for p in ("fp32", args.precision)}
    peak = hbm_copy_GBps()
    for p in stems.values():
        for v in p.values():
            v["share_of_copy_bandwidth"] = round(v["GBps"] / peak, 3)
    n = rows * cols
    res = {
        "bench": "decompress_region", **info, "precision": args.precision, "map": [rows * th, cols * tw],
        "patches": n, "batch": args.batch, "canvas_bytes": fused.numel(),
        "fused_s": [round(v, 4) for v in t_fused], "user_way_s": [round(v, 4) for v in t_user],
        "fused_patches_per_s": round(n / min(t_fused), 1), "user_way_patches_per_s": round(n / min(t_user), 1),
        "speedup": round(min(t_user) / min(t_fused), 3),
        "bytes_differing_from_float_path": n_diff, "bytes_differing_from_user_way": n_diff_user,
        "stem_out_batch256_256sq": {("cuda_core" if p == "fp32" else f"tensor_core[{p}]"): v
                                    for p, v in stems.items()},
        "hbm_copy_GBps": round(peak, 1),
    }
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
