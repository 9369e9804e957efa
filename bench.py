#!/usr/bin/env python
"""bench.py -- the hot path of 2D-VQ-AE-2 on N B200s, with roofline and CPU baseline.

Contract (one JSON line on stdout from rank 0):
  python bench.py --gpus N --steps K --warmup W [--workload encode256|roundtrip512|slide] [--dump-outputs DIR]
  python bench.py --impl reference --gpus N ...    # the reference's own CPU implementation
--dump-outputs DIR writes what the last timed step returned on rank 0 as DIR/<name>.npy (float32), so that
two builds can be compared output for output on the same seeded inputs.
For N > 1 launch with torch.distributed.run (one rank per GPU); patches shard by rank with no
data-path collective (weak scaling); only the slide workload gathers code tiles with NCCL.

Workloads (BASELINE.json `configs`):
  encode256     config 3 (the headline metric): encode + quantise of 256 synthetic 256x256x3 patches per
                GPU per step, 256-model (n_down=3, C_lat=64, 32x32 codes)
  roundtrip512  config 4: 512x512x3 -> 32x32 codes -> 512x512x3, as-shipped 512-model (n_down=4), 64
                patches per GPU per step
  slide         config 5: one synthetic 50 000^2 px slide (38 025 patches of 256^2) per step, sharded by
                patch over the ranks, u8 code tiles all-gathered and placed into the 6 240^2 code map
  value : patches/s with the inputs already resident in HBM (CUDA events, max over ranks)
  e2e   : the same through the public API from pinned HOST uint8 tiles, H2D + D2H inside the timed region
The encode256 line also carries config 2 (`quantizer_microbench`: every built (C, dtype) cell) and
config 1 (`cpu_baseline.config1`: as-shipped model, 8 patches, encode+quantise+decode on the host).
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
# the benchmark writes nothing into the tree: its CPU legs import oracle/ modules that build() never
# imported, and their bytecode would otherwise land in oracle/__pycache__
sys.dont_write_bytecode = True
for _p in (REPO / "2d-vq-ae-2_b200", REPO / "oracle"):
    if str(_p) not in sys.path:
        sys.path.insert(0, str(_p))

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    "encode256": dict(
        metric="patches_per_sec_encode_quantize_256", n_down=3, patch=256, batch=256,
        flop_per_patch=6.255e9,          # SURVEY.md 8(d): 3.127 GMAC encode + quantise, 256-model
        text="encode+quantise 256x256x3 patches, 256-model (n_down=3, C_lat=64, 32x32 codes), "
             "batch 256/GPU"),
    "roundtrip512": dict(
        metric="patches_per_sec_roundtrip_512", n_down=4, patch=512, batch=64,
        flop_per_patch=54.3e9,           # SURVEY.md 8(d): 27.16 encode + 27.16 decode GFLOP, 512-model
        text="encode+quantise+decode round trip of 512x512x3 patches, as-shipped 512-model "
             "(n_down=4, C_lat=128, 32x32 codes), batch 64/GPU"),
    "slide": dict(
        metric="patches_per_sec_slide_256", n_down=3, patch=256, batch=256, flop_per_patch=6.255e9,
        text="synthetic whole slide 50000x50000 px -> 195x195 patches of 256^2 -> 6240x6240 u8 code "
             "map per step, 256-model, patches sharded over the ranks, NCCL all-gather of code tiles"),
}
SLIDE_LEVEL = (50_000, 50_000)


def load_peaks():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        return json.loads(p.read_text()), "measured (MEASURED_PEAKS.json)"
    # B200_PROFILING.md fallback figures
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, \
        "fallback (B200_PROFILING.md)"


def ncu_traffic(kernel_key: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel_key`, from the committed
    `ncu --set full` capture index profiles/ncu_traffic.json (written by profiles/summarize_ncu.py);
    None when no capture of that kernel at the bench shape is committed."""
    p = REPO / "profiles" / "ncu_traffic.json"
    if not p.exists():
        return None, None
    rec = json.loads(p.read_text()).get(kernel_key)
    if not rec:
        return None, None
    return float(rec["dram_bytes_read"]) + float(rec["dram_bytes_write"]), rec.get("source")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])), smax.append(float(r[1]))
            except (ValueError, IndexError):
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown",
                                "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def dist_env():
    return (int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1")),
            int(os.environ.get("LOCAL_RANK", "0")))


def build_model_and_state(n_down: int, seed: int = 1):
    import vqae_b200
    from vqae_b200 import synthetic as S
    model = vqae_b200.build_vqae(n_down=n_down).eval()
    sd = S.make_state_dict(model.state_dict(), seed=seed, regime="perturbed")
    model.load_state_dict(sd)
    return model, sd


# --------------------------------------------------------------------------------------------
# CPU legs: the reference itself (oracle/_ref through oracle/ref_shim.py) when its copy travelled
# with the repository, else the oracle port -- the only places bench.py executes oracle/
# --------------------------------------------------------------------------------------------
class CpuPath:
    """The reference's CPU implementation of the path: `kind` "reference" = the unmodified
    vq_ae.model.VQAE of oracle/_ref run by stock PyTorch CPU kernels; "port" = oracle/vqae_oracle.py."""

    def __init__(self, n_down: int, sd):
        import vqae_oracle as O
        self.O, self.sd, self.model = O, sd, None
        try:
            import ref_shim
            if ref_shim.reference_available():
                from vqae_b200.config import compose_vqae_conf
                model_mod, *_ = ref_shim.load_reference()
                conf = compose_vqae_conf(n_down=n_down)
                conf.pop("_target_"), conf.pop("_recursive_")
                self.model = model_mod.VQAE(**conf).eval()
                self.model.load_state_dict(sd)
        except Exception as e:  # noqa: BLE001 -- fall back to the port, say why
            self.why_port = f"{type(e).__name__}: {e}"
        self.kind = "reference" if self.model is not None else "port"

    @torch.no_grad()
    def encode(self, img_u8: np.ndarray):
        # input normalisation: albumentations is not installed anywhere here; its published formula
        # (oracle/vqae_oracle.py:normalize_u8) stands in for it in both kinds
        x = torch.from_numpy(self.O.normalize_u8(img_u8))
        if self.model is not None:
            return tuple(zip(*self.model.encoder(x)))[0]          # extract_embeddings.py:125
        (e,), (i,), (l,) = self.O.encoder_forward(x, self.sd)
        return e, i, l

    @torch.no_grad()
    def roundtrip(self, img_u8: np.ndarray):
        x = torch.from_numpy(self.O.normalize_u8(img_u8))
        if self.model is not None:
            return self.model(x)[0]
        (e,), _, _ = self.O.encoder_forward(x, self.sd)
        return self.O.decoder_forward((e,), self.sd)


def host_threads() -> int:
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU legs run on rank 0 alone and are
    # meant to use all the host threads they can
    try:
        avail = len(os.sched_getaffinity(0))
    except AttributeError:
        avail = os.cpu_count() or 1
    if torch.get_num_threads() < avail:
        torch.set_num_threads(avail)
    return torch.get_num_threads()


def cpu_sample(cpu: CpuPath, workload: str, n_patches: int, seed: int) -> float:
    """One bounded CPU sample of `workload`; returns seconds."""
    from vqae_b200 import synthetic as S
    w = WORKLOADS[workload]
    img = S.synthetic_patches_u8(n_patches, w["patch"], seed).numpy()
    t0 = time.perf_counter()
    if workload == "roundtrip512":
        cpu.roundtrip(img)
    else:
        _, idx, _ = cpu.encode(img)
        if workload == "slide":                                  # placement of the sample's tiles
            cpu.O.stitch_code_map(idx.numpy(), 1, n_patches)
    return time.perf_counter() - t0


CPU_SAMPLE = {"encode256": 32, "roundtrip512": 4, "slide": 32}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the workload on the box's host cores,
    all host threads, each step a bounded sample (CPU_SAMPLE patches) of the workload."""
    rank, world, _ = dist_env()
    if rank != 0:
        return
    cores = host_threads()
    w = WORKLOADS[args.workload]
    _, sd = build_model_and_state(w["n_down"])
    cpu = CpuPath(w["n_down"], sd)
    sample = CPU_SAMPLE[args.workload]
    for i in range(args.warmup):
        cpu_sample(cpu, args.workload, sample, i)
    dt = sum(cpu_sample(cpu, args.workload, sample, 100 + s) for s in range(args.steps))
    value = sample * args.steps / dt
    what = ("the unmodified reference modules (oracle/_ref via oracle/ref_shim.py)"
            if cpu.kind == "reference" else "oracle/vqae_oracle.py (port)")
    line = {
        "impl": "reference", "metric": w["metric"], "value": value, "unit": "patches/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": w["text"]},
        "cpu_baseline": {"value": value, "unit": "patches/s", "cores": cores, "kind": cpu.kind,
                         "sample": f"{sample} patches per step x {args.steps} steps of the workload, "
                                   f"{what}, torch {torch.__version__} CPU kernels, {cores} threads"},
        "e2e": {"value": value, "unit": "patches/s", "h2d_bytes_per_step": 0,
                "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# GPU leg: isolated-kernel timings (roofline) and the config-2 microbench
# --------------------------------------------------------------------------------------------
def _event_time(launch, reps, dev, warm=3):
    for i in range(warm):
        launch(i)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(dev)
    e0.record()
    for i in range(reps):
        launch(i)
    e1.record()
    torch.cuda.synchronize(dev)
    return e0.elapsed_time(e1) / reps


def time_trunk_kernel(dev, peaks, model, C: int, B: int):
    """CUDA-event timing of the dominant kernel alone at the bench shape: the image-resident trunk
    launch (54 'same' blocks, C channels at 32x32, batch B) with THE MODEL'S OWN packed weights,
    launched through the C-ABI on the current stream, rotating over 4 buffer pairs (> 126 MB L2)."""
    from vqae_b200 import _lib as L
    from vqae_b200 import engine as E
    from vqae_b200 import plan as P
    lib = L.load()
    H = W = 32
    blocks = [b for b in P.flat_blocks(model.encoder.down_layers) +
              P.flat_blocks(model.encoder.pre_enc_layers)
              if b.branch_conv1.in_channels == C and tuple(b.branch_conv2.kernel_size) == (3, 3)]
    packed = E.pack_blocks(blocks)
    chain = E.PackedChain(packed, resident=True)
    nblk = chain.n
    nbuf = 4
    xs = [torch.randn(B, H, W, C, device=dev) for _ in range(nbuf)]
    ys = [torch.empty(B, H, W, C, device=dev) for _ in range(nbuf)]
    st = E._stream(dev)
    assert lib.vqae_trunk_resident_supported(B, H, W, C)

    def launch(i):
        E.trunk_resident(xs[i % nbuf], ys[i % nbuf], chain)
    ms = _event_time(launch, 5, dev)
    flops = 2.0 * B * H * W * C * C * 11 * nblk
    achieved = flops / (ms * 1e-3) / 1e12
    key = f"trunk_resident_tc_kernel<{C},32>@B{B}"
    traffic, traffic_src = ncu_traffic(key)
    return {
        "bound": "tensor", "achieved": achieved, "peak": peaks["bf16_tflops"], "unit": "TFLOP/s",
        "frac": achieved / peaks["bf16_tflops"],
        "peak_kind": "burst (bf16_tflops): the kernel is timed alone, 5 launches",
        "frac_of_sustained": achieved / peaks["bf16_tflops_sustained"],
        "traffic": traffic, "traffic_source": traffic_src,
        "kernel": f"trunk_resident_tc_kernel<{C},32> ({nblk} fused PreActFixupResBlocks 'same' per "
                  f"launch, C={C}, 32x32, batch {B}; tcgen05 bf16 operands, fp32 residual resident in "
                  "tensor memory, 4-CTA clusters, halo rows through distributed shared memory)",
        "us_per_launch": ms * 1e3, "algorithmic_flops_per_launch": flops,
        "weights": "the benchmarked model's own blocks (random-init 'perturbed' regime)",
        "timing": f"CUDA events on the launch stream, {nbuf} rotating buffer pairs, 3 warm-up launches"}


def time_quantizer_cells(dev, peaks):
    """Config 2: ProjectedEMAVectorQuantizer2d on [512,C,32,32] NHWC, N = 524 288 vectors, every
    (C, I/O dtype) cell the library builds: the C-ABI call on preallocated buffers, three rotating
    inputs (> L2), CUDA events on the launch stream.  Algorithmic bytes = read N*C*s + write N*C*s +
    write N*8 (int64 indices), SURVEY.md 8(d)."""
    from vqae_b200 import engine as E
    from vqae_b200.layers.vq import ProjectedEMAVectorQuantizer2d
    n = 512 * 1024
    cells = {}
    for c in (64, 128):
        q = ProjectedEMAVectorQuantizer2d(256, c, 1.0, 0.99, 1e-5, 8).eval().to(dev)
        pq = q.packed()
        for dt in E.QUANT_IO_DTYPES:
            tdt = {"fp32": torch.float32, "bf16": torch.bfloat16, "fp16": torch.float16}[dt]
            xs = [torch.randn(n, c, device=dev).to(tdt) for _ in range(3)]
            bufs = E.QuantizeBuffers(pq, n, tdt, dev)

            def call(i, xs=xs, bufs=bufs, pq=pq):
                E.quantize_into(pq, xs[i % 3], bufs, 512, 1024)

            us = _event_time(call, 20, dev) * 1e3
            s = xs[0].element_size()
            byts = n * c * s * 2 + n * 8
            gbs = byts / (us * 1e-6) / 1e9
            cells[f"C{c}_{dt}"] = {
                "kernel": bufs.kernel_name, "us_per_call": us, "algorithmic_bytes": byts,
                "achieved_gbs": gbs, "peak_gbs": peaks["hbm_gbs"], "frac": gbs / peaks["hbm_gbs"],
                "vectors_per_s": n / (us * 1e-6), "near_ties": int(bufs.ties.item())}
            del xs, bufs
    head = cells["C64_fp32"]
    return {"workload": "ProjectedEMAVectorQuantizer2d [512,C,32,32] NHWC, K=256, D=8, N=524288",
            "headline_cell": "C64_fp32", "us_per_call": head["us_per_call"],
            "achieved_gbs": head["achieved_gbs"], "peak_gbs": head["peak_gbs"], "frac": head["frac"],
            "cells": cells}


# --------------------------------------------------------------------------------------------
# GPU leg: workloads
# --------------------------------------------------------------------------------------------
def device_patches(first: int, count: int, patch: int, dev) -> torch.Tensor:
    """uint8 [count,patch,patch,3] tiles that depend only on the patch index (slide workload)."""
    out = torch.empty(count, patch, patch, 3, dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev)
    for i in range(count):                       # one generator state per patch: shard-independent
        g.manual_seed(1234 + first + i)
        out[i] = torch.randint(0, 256, (patch, patch, 3), dtype=torch.uint8, device=dev, generator=g)
    return out


DUMP_MAX_ELEMS = 1 << 22        # per array: 16 MB of float32; at most two arrays per workload, 32 MB


def host_outputs(outs, names) -> dict:
    """float32 host copies of a step's outputs, taken before later steps reuse the graph's output
    buffers.  An array larger than DUMP_MAX_ELEMS is stored as `<name>_sample`: the flattened array at
    DUMP_MAX_ELEMS positions drawn from a fixed seed, the same positions in every run."""
    outs = outs if isinstance(outs, tuple) else (outs,)
    res = {}
    for name, t in zip(names, outs, strict=True):
        if t.numel() > DUMP_MAX_ELEMS:
            pos = torch.randint(t.numel(), (DUMP_MAX_ELEMS,), generator=torch.Generator().manual_seed(0))
            t, name = t.reshape(-1)[pos.to(t.device)], name + "_sample"
        res[name] = t.float().cpu().numpy()
    return res


def run_gpu(args):
    rank, world, local = dist_env()
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)
    else:
        dist = None

    import vqae_b200
    from vqae_b200 import engine as E
    from vqae_b200 import synthetic as S
    from vqae_b200.extract import StreamingEncoder, encode_patches
    from vqae_b200.graphs import CapturedStep
    from vqae_b200.plan import resolve_precision
    from vqae_b200.sharding import bind_host_to_gpu_numa_node, gather_code_tiles, shard_range, slide_grid

    numa_node = bind_host_to_gpu_numa_node(local) if world > 1 else None   # before any pinned allocation
    w = WORKLOADS[args.workload]
    peaks, peaks_kind = load_peaks()
    model, sd = build_model_and_state(w["n_down"])
    model = vqae_b200.set_precision(model.to(dev), args.precision)
    enc = model.encoder
    B, PATCH = w["batch"], w["patch"]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def allmax(ms):
        if dist is None:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- per-workload step functions --------------------------------------------------------
    # every step is captured into a CUDA graph per input buffer after its first eager run and replayed
    # from then on (vqae_b200.graphs.CapturedStep; --no-graphs: eager launches every step)
    def captured(fn):
        if args.no_graphs:
            return fn
        return CapturedStep(fn, key_extra=lambda: (resolve_precision(enc), resolve_precision(model.decoder)))

    encode_step = captured(lambda x: encode_patches(enc, x))
    extra = {}
    if args.workload == "slide":
        rows, cols = slide_grid(SLIDE_LEVEL, PATCH)
        n_total = rows * cols
        lo, hi = shard_range(n_total, rank, world)
        batches = [(s, device_patches(s, min(B, hi - s), PATCH, dev)) for s in range(lo, hi, B)]
        units_per_step = n_total                       # whole job, all ranks
        code_map = torch.zeros(rows * 32, cols * 32, dtype=torch.uint8, device=dev)
        gather_ms = []

        def step_resident(i):
            tiles = torch.cat([encode_step(p).to(torch.uint8) for _, p in batches])
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            full = gather_code_tiles(tiles, n_total)   # NCCL all-gather (N > 1)
            E.codemap_place(full.long(), 0, cols, code_map)
            g1.record()
            gather_ms.append((g0, g1))
            return code_map
        out_names = ("code_map",)
        pool = [S.synthetic_patches_u8(B, PATCH, 42 + rank + 1000 * j).pin_memory() for j in range(4)]
        n_b = len(batches)
        h2d = sum(int(p.numel()) for _, p in batches)
        d2h = int(code_map.numel()) if rank == 0 else 0
        host_map = torch.empty(code_map.shape, dtype=torch.uint8).pin_memory()
        streamer = StreamingEncoder(enc, dev, graphs=not args.no_graphs)

        def run_e2e(n_steps):
            """Per slide: this rank's patch batches from pinned host memory (a pool of 4 distinct
            pinned batches stands in for the 7.5 GB of tiles) -> H2D -> encode -> gather -> map -> D2H
            of the code map on rank 0."""
            acc = 0
            for _ in range(n_steps):
                sizes = [p.shape[0] for _, p in batches]
                outs = [o[:k].to(torch.uint8) for o, k in zip(
                    streamer.encode_stream((pool[j % 4] for j in range(n_b)), to_host=False), sizes)]
                full = gather_code_tiles(torch.cat(outs), n_total)
                E.codemap_place(full.long(), 0, cols, code_map)
                if rank == 0:
                    host_map.copy_(code_map, non_blocking=True)
                torch.cuda.synchronize(dev)
                acc += int(host_map[0, 0])
            return acc
        api = ("StreamingEncoder.encode_stream over the rank's pinned uint8 batches, "
               "sharding.gather_code_tiles (NCCL all-gather), engine.codemap_place, D2H of the u8 map")
    else:
        host = [S.synthetic_patches_u8(B, PATCH, 42 + rank + 1000 * j).pin_memory() for j in range(2)]
        resident = [h.to(dev) for h in host]
        units_per_step = world * B
        if args.workload == "encode256":
            def step_resident(i):
                return encode_step(resident[i % 2])
            out_names = ("codes",)
            streamer = StreamingEncoder(enc, dev, graphs=not args.no_graphs)
            h2d, d2h = int(B * PATCH * PATCH * 3), int(B * 32 * 32 * 8)

            def run_e2e(n_steps):
                """Pinned uint8 tiles -> H2D (side stream, overlapped with the previous batch's
                encode) -> encode -> D2H of the int64 code indices into pinned memory."""
                acc = 0
                for out in streamer.encode_stream((host[i % 2] for i in range(n_steps)),
                                                  reuse_buffers=True):
                    acc += int(out[0, 0, 0])             # touch the host result
                return acc
            api = ("vqae_b200.extract.StreamingEncoder(model.encoder).encode_stream(pinned uint8 "
                   "tiles): double-buffered H2D on a side stream, D2H of int64 codes")
        else:                                           # roundtrip512
            def roundtrip(x):
                _, idx, _, _, _ = enc.encode(x, want_quantized=True)
                return idx, model.decode_codes(idx)
            roundtrip_step = captured(roundtrip)

            def step_resident(i):
                return roundtrip_step(resident[i % 2])
            out_names = ("codes", "reconstruction")
            dev_in = [torch.empty_like(resident[0]) for _ in range(2)]
            host_idx = [torch.empty(B, 32, 32, dtype=torch.int64).pin_memory() for _ in range(2)]
            host_stat = torch.empty(2, dtype=torch.float32).pin_memory()
            h2d, d2h = int(B * PATCH * PATCH * 3), int(B * 32 * 32 * 8 + 8)

            copy_stream = torch.cuda.Stream(dev)
            ev_in = [torch.cuda.Event() for _ in range(2)]
            ev_free = [torch.cuda.Event() for _ in range(2)]

            def run_e2e(n_steps):
                """Pinned uint8 tiles -> H2D (side stream: the copy of batch i + 1 runs under the compute of
                batch i) -> encode -> decode_codes -> D2H of the int64 codes (the stored representation)
                and of two reconstruction statistics (mean, mean |.|), read on the host every step; the
                200 MB fp32 reconstruction itself stays on the device."""
                acc = 0.0
                cur = torch.cuda.current_stream(dev)

                def prefetch(j):
                    t = j & 1
                    with torch.cuda.stream(copy_stream):
                        copy_stream.wait_event(ev_free[t])       # the compute that last read this buffer
                        dev_in[t].copy_(host[t], non_blocking=True)
                        ev_in[t].record(copy_stream)
                for t in range(2):
                    ev_free[t].record(cur)
                prefetch(0)
                for i in range(n_steps):
                    s = i & 1
                    if i + 1 < n_steps:
                        prefetch(i + 1)
                    cur.wait_event(ev_in[s])
                    idx, rec = roundtrip_step(dev_in[s])
                    ev_free[s].record(cur)
                    host_idx[s].copy_(idx, non_blocking=True)
                    host_stat.copy_(torch.stack([rec.mean(), rec.abs().mean()]), non_blocking=True)
                    cur.synchronize()
                    acc += float(host_stat[1]) + int(host_idx[s][0, 0, 0])
                return acc
            api = ("Encoder.encode(uint8 tiles) + VQAE.decode_codes: double-buffered H2D of pinned uint8 tiles "
                   "on a side stream, D2H of int64 codes + reconstruction statistics every step")

    def timed(fn, steps, warmup):
        """(max over ranks of the device time of `steps` calls of fn in ms, launches, last call's result)"""
        with torch.no_grad():
            for i in range(warmup):
                fn(i)
            barrier()
            l0 = E.launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                out = fn(i)
            e1.record()
            barrier()
            ms = e0.elapsed_time(e1)
            launches = E.launch_count() - l0
        return allmax(ms), launches, out

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # at least three untimed steps: eager run, then one graph capture per input buffer
    warm = max(args.warmup, 3)
    ms, launches, last_out = timed(step_resident, args.steps, warm)
    clocks = sampler.stop() if rank == 0 else None
    dumped = host_outputs(last_out, out_names) if args.dump_outputs and rank == 0 else None
    del last_out

    with torch.no_grad():
        run_e2e(3 if args.workload == "slide" else warm)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        run_e2e(args.steps)
        e1.record()
        barrier()
        wall_ms = (time.perf_counter() - t0) * 1e3
        ms_e2e = allmax(max(e0.elapsed_time(e1), 0.0))

    value = units_per_step * args.steps / (ms * 1e-3)
    e2e = units_per_step * args.steps / (ms_e2e * 1e-3)

    # the other arithmetic modes on the same resident batch, next to the headline mode
    modes = {}
    if args.workload == "encode256" and not args.no_extras:
        for prec in E.PRECISIONS:
            if prec == args.precision:
                modes[prec] = value / world
                continue
            vqae_b200.set_precision(model, prec)
            k = 3 if prec == "fp32" else max(3, args.steps // 2)
            ms_p, _, _ = timed(step_resident, k, 2)
            modes[prec] = B * k / (ms_p * 1e-3)
        vqae_b200.set_precision(model, args.precision)

    if rank == 0:
        C = 64 if w["n_down"] == 3 else 128
        roofline = time_trunk_kernel(dev, peaks, model, C, B)
        roofline["peak_source"] = peaks_kind
        line = {
            "metric": w["metric"], "value": value, "unit": "patches/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "f16",
            "data": "synthetic",
            "config": {"workload": w["text"]},
            "detail": {"precision": args.precision,
                       "parallelism": f"patch-sharded x{world}, no data-path collective"
                       + (" (one NCCL all-gather of u8 code tiles per slide)"
                          if args.workload == "slide" else ""),
                       "host_numa_node_rank0": numa_node,
                       "cuda_graphs": not args.no_graphs,
                       "l2": "two rotating resident batches; per-step activation traffic >> 126 MB L2",
                       "whole_step_tflops_per_gpu": value * w["flop_per_patch"] / 1e12 / world,
                       "whole_step_frac_of_sustained_bf16_peak":
                           value * w["flop_per_patch"] / 1e12 / world / peaks["bf16_tflops_sustained"],
                       "patches_per_s_per_gpu_by_precision": modes or None},
            "e2e": {"value": e2e, "unit": "patches/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": api,
                    "host_wall_ms_per_step": wall_ms / args.steps},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roofline,
        }
        if args.workload == "slide":
            torch.cuda.synchronize(dev)
            gm = [a.elapsed_time(b) for a, b in gather_ms[-args.steps:]]
            line["detail"].update({
                "patches_per_slide": units_per_step, "gather_and_place_ms": float(np.median(gm)),
                "gathered_bytes_per_rank": int(sum(p.shape[0] for _, p in batches) * 1024),
                "code_map_sha256_16": hashlib.sha256(code_map.cpu().numpy().tobytes()).hexdigest()[:16]})
        if args.workload == "encode256" and not args.no_extras:
            line["quantizer_microbench"] = time_quantizer_cells(dev, peaks)
        if world == 1 and not args.no_extras:
            cores = host_threads()
            cpu = CpuPath(w["n_down"], sd)
            n_s = CPU_SAMPLE[args.workload] // (4 if args.workload != "roundtrip512" else 2)
            best = min(cpu_sample(cpu, args.workload, n_s, 7 + r) for r in range(3))
            line["cpu_baseline"] = {
                "value": n_s / best, "unit": "patches/s", "cores": cores, "kind": cpu.kind,
                "sample": f"{n_s} patches of the workload, best of 3, "
                          + ("unmodified reference modules from oracle/_ref" if cpu.kind == "reference"
                             else "oracle port") + f", torch {torch.__version__} CPU, {cores} threads"}
            if args.workload == "encode256":
                # BASELINE.json config 1 as written: as-shipped conf (n_down=4), 8 normalised 256^2
                # patches, encode + quantise + decode (16x16 code grid for this conf)
                _, sd4 = build_model_and_state(4)
                cpu4 = CpuPath(4, sd4)
                img = S.synthetic_patches_u8(8, 256, 5).numpy()
                cpu4.roundtrip(img)
                ts = []
                for _ in range(3):
                    t0 = time.perf_counter()
                    cpu4.roundtrip(img)
                    ts.append(time.perf_counter() - t0)
                line["cpu_baseline"]["config1"] = {
                    "workload": "as-shipped VQ-AE (n_down=4), encode+quantise+decode of 8 synthetic "
                                "256x256x3 patches (16x16 codes)",
                    "seconds": min(ts), "patches_per_s": 8 / min(ts), "kind": cpu4.kind, "cores": cores}
        if dumped is not None:
            out_dir = Path(args.dump_outputs)
            out_dir.mkdir(parents=True, exist_ok=True)
            for name, arr in dumped.items():
                np.save(out_dir / f"{name}.npy", arr)
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="encode256", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp16")
    ap.add_argument("--no-graphs", action="store_true",
                    help="launch every kernel of every step from the host instead of replaying CUDA graphs")
    ap.add_argument("--no-extras", action="store_true",
                    help="skip the side measurements (other precisions, config 2, CPU baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32; arrays above "
                         f"{DUMP_MAX_ELEMS} elements as a seeded sample, <name>_sample.npy).  --impl b200 only: "
                         "the reference leg times small CPU samples, not the inputs of the B200 path")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the B200 path (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_gpu(args)


if __name__ == "__main__":
    main()
