#!/usr/bin/env python
"""Benchmark of the animal-vision per-frame pixel pipeline on B200 (BASELINE.json metric:
Mpix/s and 4K frames/s at 1/2/4/8 GPUs, % of HBM roofline).

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
        --master-port P bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU path (oracle port) on host cores
    python bench.py ... --dump-outputs DIR    # also write the last timed step's outputs to DIR/<name>.npy

Workload (BASELINE.json configs[4], the one the metric is quoted on): a synthetic 4K (3840x2160)
60-frame uint8 video batch PER GPU (weak scaling: frames are independent, no collective), species
round-robin Dog -> Cat -> HoneyBee, frame s filled by numpy default_rng(seed s).  One step = one
pass of the hot path over that batch: 20 Dog + 20 Cat + 20 HoneyBee frames.

  value     whole-job Mpix/s with the frames already resident in HBM (CUDA events, max over ranks)
  e2e       same metric through the public host API: pinned host frames in, pinned host frames out,
            H2D + kernels + D2H all inside the timed region (HostBatchPipeline)
  roofline  dominant kernel: algorithmic bytes per launch / its mean launch time, measured live
            with CUDA events on the launching stream (avb_profile_begin/end)
  cpu_baseline  oracle (CPU restatement of the reference; tests pin it bit-exact to the reference)
            timed on this host's cores on a bounded sample of the same workload
Prints ONE JSON line on rank 0.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time


def _affinity_cores() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


if "reference" in sys.argv:
    # torchrun exports OMP_NUM_THREADS=1 to every rank; the CPU arm is ONE process that may use every core
    # this process is allowed on.  BLAS / OpenMP read these at import time, so set them before numpy / torch.
    for _v in ("OMP_NUM_THREADS", "OPENBLAS_NUM_THREADS", "MKL_NUM_THREADS"):
        os.environ[_v] = str(_affinity_cores())

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

H4K, W4K = 2160, 3840
FRAMES_PER_GPU = 60
SPECIES = ("Dog", "Cat", "HoneyBee")
# algorithmic bytes per pixel (uint8 in + uint8 out(s)); SURVEY.md 8(d)
ALGO_BYTES_PER_PX = {"Dog": 6, "Cat": 9, "HoneyBee": 6}
# per KERNEL: bytes it must read + write per output pixel (cat warp: u8 frame in, cat view out; the
# centre zoom's output belongs to cat_center_zoom)
KERNEL_ALGO_BYTES_PER_PX = {"k2_gauss_dichromat": 6.0, "k2_gauss_cat_warp": 6.0, "cat_center_zoom": 3.0 + 3.0 / 2.25,
                            "k3_uv_map": 6.0, "k3_uv_hist": 3.0, "k3_uv_stats": 3.0, "k3_uv_compact": 8.0, "k2_streak": 6.0}
# measured DRAM traffic per launch comes from a committed ncu capture of THIS launch shape, never from a constant:
# tools/ncu_dram_table.py turns an .ncu-rep (ncu --set full on `tools/prof_one.py ... 20` = the bench's 20-frame 4K
# launches) into this JSON; a kernel / shape that is not in it reports traffic = null.
NCU_DRAM_TABLE = os.path.join(ROOT, "profiles", "ncu_dram_table.json")
KERNEL_SPECIES = {"k2_gauss_dichromat": "Dog", "k2_gauss_cat_warp": "Cat", "cat_center_zoom": "Cat",
                  "k3_uv_stats": "HoneyBee", "k3_uv_map": "HoneyBee", "k3_uv_hist": "HoneyBee", "k3_uv_compact": "HoneyBee",
                  "k3_uv_prep": "HoneyBee", "k3_uv_scan": "HoneyBee", "k3_uv_select": "HoneyBee", "k2_streak": "Dog",
                  "frame_flags": "Cat", "k2_gauss_dichromat_fixup": "Dog", "k2_gauss_cat_warp_fixup": "Cat"}


def bench_config():
    """`config` of the JSON line: byte-identical in the GPU arm and the --impl reference arm (extras go to `detail`)."""
    return {"workload": "4K 60-frame mixed-species video batch per GPU (Dog/Cat/HoneyBee round-robin), BASELINE configs[4]",
            "resolution": f"{W4K}x{H4K}", "frames_per_gpu": FRAMES_PER_GPU, "species": list(SPECIES)}


def ncu_traffic(kernel: str, frames: int, H: int, W: int):
    """(bytes per launch, source) measured by ncu for this kernel at exactly this launch shape, else (None, why)."""
    try:
        with open(NCU_DRAM_TABLE) as fh:
            tab = json.load(fh)
    except Exception:
        return None, "no profiles/ncu_dram_table.json"
    for rec in tab.get("kernels", []):
        if rec.get("bench_name") == kernel and (rec.get("frames"), rec.get("H"), rec.get("W")) == (frames, H, W):
            return float(rec["dram_bytes_per_launch"]), f"{tab.get('source', 'profiles/ncu_dram_table.json')}: ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of one {frames}-frame {W}x{H} launch"
    return None, f"profiles/ncu_dram_table.json has no capture of {kernel} at {frames} x {W}x{H}"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.idx)],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 8:
                continue
            try:
                clk, cmax = float(parts[1]), float(parts[2])
            except ValueError:
                continue
            if t0 - 0.05 <= ts <= t1 + 0.25:
                sm.append(clk)
                mx.append(cmax)
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        if not sm:  # region shorter than one sample: use whatever we saw
            for ts, line in self.lines:
                parts = [p.strip() for p in line.split(",")]
                try:
                    sm.append(float(parts[1])); mx.append(float(parts[2]))
                except Exception:
                    pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- workload
def make_host_frames(rank: int, world: int, n_frames: int, H: int, W: int, pinned: bool):
    """This rank's shard of the world x n_frames synthetic video, grouped per species: a uint8
    [k, H, W, 3] host tensor each; global frame s is default_rng(s), its species round-robin in s."""
    import torch
    from animal_vision_b200 import sharding
    plan = sharding.shard_plan(world * n_frames, rank, world, SPECIES)
    out = {}
    for sp in SPECIES:
        idx = [i for i, s in plan if s == sp]
        t = torch.empty((len(idx), H, W, 3), dtype=torch.uint8)
        if pinned:
            t = t.pin_memory()
        view = t.numpy()
        for j, s in enumerate(idx):
            view[j] = np.random.default_rng(s).integers(0, 256, (H, W, 3), dtype=np.uint8)
        out[sp] = t
    return out


DUMP_BYTES = 64 * 10 ** 6
DUMP_SEED = 0


def dump_outputs(directory: str, dev_out):
    """Write the outputs of the last timed step as float32 .npy files, DUMP_BYTES in all, so that two builds can
    be compared output for output.  An output larger than its share of the budget is sampled: the same
    default_rng(DUMP_SEED) draw of pixels (all three channels, in raster order) for every output of that shape."""
    import torch
    arrays = {"dog": dev_out["Dog"], "cat_human": dev_out["Cat"][0], "cat_view": dev_out["Cat"][1],
              "honeybee": dev_out["HoneyBee"]}
    budget_px = (DUMP_BYTES // len(arrays) - 1024) // (3 * 4)        # 1 KB per file for the .npy header
    os.makedirs(directory, exist_ok=True)
    picks = {}
    for name, t in arrays.items():
        n_px = t.numel() // 3
        if n_px <= budget_px:
            a = t.float().cpu().numpy()
        else:
            if t.shape not in picks:
                idx = np.sort(np.random.default_rng(DUMP_SEED).choice(n_px, budget_px, replace=False))
                picks[t.shape] = torch.from_numpy(idx).to(t.device)
            a = t.reshape(n_px, 3).index_select(0, picks[t.shape]).float().cpu().numpy()
        np.save(os.path.join(directory, name + ".npy"), a)
    log(f"[rank 0] outputs of the last timed step written to {directory} ({', '.join(arrays)})")


def peak_numbers():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as fh:
            d = json.load(fh)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


# ----------------------------------------------------------------------------- CPU arms
def oracle_step_time(frames_by_species, reps: int = 1):
    """Seconds for one pass of the oracle (reference restatement) over the given frames."""
    from oracle import mammals as M
    from oracle import uv
    t0 = time.perf_counter()
    for _ in range(reps):
        for sp, frames in frames_by_species.items():
            for f in frames:
                if sp == "Dog":
                    M.mammal_visualize(f, "dog")
                elif sp == "Cat":
                    M.cat_visualize(f)
                else:
                    uv.honeybee_visualize(f)
    return (time.perf_counter() - t0) / reps


def host_threads():
    info = {"os_cpu_count": os.cpu_count()}
    try:
        info["sched_affinity"] = len(os.sched_getaffinity(0))
    except Exception:
        pass
    try:
        import cv2
        info["cv2_threads"] = cv2.getNumThreads()
    except Exception:
        pass
    try:
        import torch
        info["torch_threads"] = torch.get_num_threads()
    except Exception:
        pass
    return info


def cpu_sample(rows: int):
    """One frame per species, `rows` x 3840 (a full-width band of a 4K frame)."""
    return {sp: [np.random.default_rng(1000 + k).integers(0, 256, (rows, W4K, 3), dtype=np.uint8)]
            for k, sp in enumerate(SPECIES)}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle port; the reference
    is Python and cannot travel to the GPU box, tests pin the port bit-exact to it) on the host."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = _affinity_cores()
    try:                                            # one process, every core it may run on (see the top of this file)
        import cv2
        cv2.setNumThreads(cores)
    except Exception:
        pass
    try:
        import torch
        torch.set_num_threads(cores)
    except Exception:
        pass
    threads = host_threads()
    # size the per-step sample so that (warmup + steps) steps finish in ~150 s
    probe = cpu_sample(270)
    t_probe = oracle_step_time(probe)                         # 3 x 270x3840 frames
    px_probe = 3 * 270 * W4K
    budget = 150.0 / max(1, args.steps + args.warmup)
    rows = int(min(H4K, max(64, 270 * budget / max(t_probe, 1e-6) * 0.8)))
    sample = cpu_sample(rows)
    px = 3 * rows * W4K
    for _ in range(args.warmup):
        oracle_step_time(sample)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_step_time(sample)
    dt = (time.perf_counter() - t0) / max(1, args.steps)
    mpix = px / dt / 1e6
    desc = (f"per step: 1 Dog + 1 Cat + 1 HoneyBee frame of {rows}x{W4K} (full-width band of a 4K frame of the config's video: a bounded "
            f"sample, the metric is a rate), oracle port, ONE process on {cores} host cores (rank 0 only when launched under torchrun)")
    line = {
        "impl": "reference", "metric": "Mpix/s", "value": mpix, "unit": "Mpix/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(),
        "fps_4k": mpix * 1e6 / (H4K * W4K),
        "cpu_baseline": {"value": mpix, "unit": "Mpix/s", "cores": cores, "kind": "port", "sample": desc, "threads": threads},
        "e2e": {"value": mpix, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "probe": {"px": px_probe, "seconds": t_probe},
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- per-config legs
CONFIG_TEXT = {"Dog": "BASELINE configs[0]: Dog dichromat transform on one synthetic 1920x1080 image",
               "Cat": "BASELINE configs[1]: Cat LMS + acuity blur + wide-vision remap on 1080p frames",
               "HoneyBee": "BASELINE configs[2]: HoneyBee UV via 31-band reconstruction + receptor projection at 1080p"}


def run_config_legs(dev, species, peak, with_cpu: bool):
    """BASELINE configs[0..2]: ONE synthetic 1080p uint8 frame.
      visualize_*   the reference-facing call `Animal.visualize(np.ndarray)` (NumPy in, NumPy out: pinned H2D, kernels,
                    D2H and one synchronise inside) -- median latency of 10 calls after 3 warm-up calls
      device_*      `visualize_batch` on one device-resident frame, CUDA events; the frames rotate through a ring of 24
                    distinct frames (149 MB in + >= 149 MB out, larger than the 126 MB L2) so no call finds its input in L2
      roofline      whole species path (all its kernels) on one frame: algorithmic bytes (uint8 in + uint8 out(s)) / device time
      cpu_reference the oracle port on the same frame on this host's cores (best of 2), N = 1 only"""
    import torch
    H, W = 1080, 1920
    px = H * W
    ring_n = 24
    ring = torch.empty((ring_n, H, W, 3), dtype=torch.uint8)
    for i in range(ring_n):
        ring[i] = torch.from_numpy(np.random.default_rng(i).integers(0, 256, (H, W, 3), dtype=np.uint8))
    f0 = ring[0].numpy().copy()
    d_ring = ring.to(dev)
    out = {}
    for name in SPECIES:
        sp = species[name]
        n_out = int(getattr(sp, "N_OUTPUTS", 1))
        for _ in range(3):
            sp.visualize(f0)
        lat = []
        for _ in range(10):
            t0 = time.perf_counter()
            sp.visualize(f0)
            lat.append(time.perf_counter() - t0)
        lat_s = float(np.median(lat))
        outs = [torch.empty_like(d_ring) for _ in range(n_out)]

        def one(i):
            o = tuple(t[i:i + 1] for t in outs) if n_out == 2 else outs[0][i:i + 1]
            sp.visualize_batch(d_ring[i:i + 1], out=o)
        for i in range(ring_n):
            one(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for rep in range(2):
            for i in range(ring_n):
                one(i)
        e1.record()
        torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1) / (2 * ring_n)
        bpp = ALGO_BYTES_PER_PX[name]
        ach = bpp * px / (dev_ms * 1e-3) / 1e9
        rec = {"config": CONFIG_TEXT[name], "frame": f"{W}x{H} uint8, default_rng(0)",
               "visualize_ms": lat_s * 1e3, "visualize_mpix_per_s": px / lat_s / 1e6, "visualize_fps": 1.0 / lat_s,
               "device_ms": dev_ms, "device_mpix_per_s": px / (dev_ms * 1e-3) / 1e6,
               "roofline": {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                            "algorithmic_bytes_per_frame": bpp * px,
                            "note": f"{bpp} B/px x {W}x{H}; one frame per call, ring of {ring_n} frames (> L2), all kernels of the species path"}}
        if with_cpu:
            from oracle import mammals as M
            from oracle import uv
            fn = {"Dog": lambda: M.mammal_visualize(f0, "dog"), "Cat": lambda: M.cat_visualize(f0), "HoneyBee": lambda: uv.honeybee_visualize(f0)}[name]
            ts = []
            for _ in range(2):
                t0 = time.perf_counter()
                fn()
                ts.append(time.perf_counter() - t0)
            rec["cpu_reference"] = {"ms": min(ts) * 1e3, "mpix_per_s": px / min(ts) / 1e6, "kind": "port", "cores": _affinity_cores()}
        out[name] = rec
        del outs
    return out


# ----------------------------------------------------------------------------- UV species leg (SURVEY.md 8f-1 / 8f-2)
UV_SPECIES = [("Reindeer", "reindeer"), ("RatUV", "rat_uv"), ("Goldfish", "goldfish"), ("Damselfish", "damselfish"),
              ("Anableps", "anableps"), ("Anchovy", "anchovy"), ("Guppy", "guppy"), ("Morpho", "morpho"), ("Heliconius", "heliconius"),
              ("Pieris", "pieris"), ("MantisShrimp", "mantis_shrimp"), ("Kestrel", "kestrel"), ("JumpingSpider", "jumping_spider"),
              ("Dragonfly", "dragonfly"), ("Hummingbird", "hummingbird")]


def run_uv_species_leg(dev, peak, with_cpu: bool):
    """The 15 panorama / UV species on 1080p uint8 frames (two outputs each: warped baseline + view, 9 B/px algorithmic).
      device_ms     `visualize_batch` on a device-resident batch of 4 frames, CUDA events, per frame; the batch rotates over
                    8 distinct batches (199 MB of input, > L2)
      launches      kernels per call (K6 operators + K7 fused element-wise programs)
      cpu_reference the oracle port (bit-equal to the reference on the golden frames) on ONE 540x960 frame, this host's cores"""
    import torch
    import animal_vision_b200.animals as A
    from animal_vision_b200.engine import get_engine
    eng = get_engine(dev)
    H, W, nb, ring_n = 1080, 1920, 4, 8
    ring = torch.randint(0, 256, (ring_n, nb, H, W, 3), dtype=torch.uint8, device=dev)
    small = np.random.default_rng(0).integers(0, 256, (540, 960, 3), dtype=np.uint8)
    out = {}
    for cls, fn in UV_SPECIES:
        sp = getattr(A, cls)()
        for i in range(2):
            sp.visualize_batch(ring[i])
        torch.cuda.synchronize()
        l0 = eng.launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(ring_n):
            sp.visualize_batch(ring[i])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / (ring_n * nb)
        ach = 9 * H * W / (ms * 1e-3) / 1e9
        rec = {"device_ms_per_frame": ms, "device_mpix_per_s": H * W / (ms * 1e-3) / 1e6, "launches_per_call": (eng.launches - l0) // ring_n,
               "roofline_frac_hbm": ach / peak}
        if with_cpu:
            from oracle import uv_species as O
            t0 = time.perf_counter()
            getattr(O, fn)(small)
            dt = time.perf_counter() - t0
            rec["cpu_reference"] = {"ms": dt * 1e3, "mpix_per_s": small.shape[0] * small.shape[1] / dt / 1e6, "frame": "540x960", "kind": "port",
                                    "cores": _affinity_cores()}
        out[cls] = rec
    return {"frame": f"{W}x{H} uint8, batches of {nb}", "algorithmic_bytes_per_px": 9, "species": out}


# ----------------------------------------------------------------------------- K4 leg
MSTPP_FLOP_PER_PATCH = 169.2e9      # SURVEY.md 8a-19: 482x512 patch, 2 x MAC, unpadded channel counts


def run_mstpp_leg(args, dev, rank, world, max_over_ranks, barrier):
    """MST++ (K4) throughput on `--mstpp-batch` 482x512 patches per GPU, seeded weights; reported as an
    extra object beside the headline metric (the 4K video workload has no MST++ species)."""
    import torch
    if args.mstpp_batch <= 0:
        return None
    from animal_vision_b200.mstpp import MSTPlusPlus, synthetic_state_dict
    net = MSTPlusPlus(synthetic_state_dict(0), dev)
    nb = args.mstpp_batch
    x = torch.rand(nb, 482, 512, 3, generator=torch.Generator().manual_seed(1 + rank)).to(dev)
    parts = min(4, nb)             # patches are independent: the batch runs as `parts` concurrent forwards
    for _ in range(3):
        net.forward_nhwc_streams(x, parts)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    iters = 5
    e0.record()
    for _ in range(iters):
        net.forward_nhwc_streams(x, parts)
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1) / iters)
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            peak = float(json.load(fh)["bf16_tflops_sustained"]); src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)"
    except Exception:
        peak, src = 1400.0, "fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)"
    tf = MSTPP_FLOP_PER_PATCH * nb * world / (ms * 1e-3) / 1e12
    # single patch, one stream (latency), then the ten mantis-shrimp bands + safe_norm on its cube (configs[3])
    from animal_vision_b200.mstpp import mantis_bands, safe_norm_maps
    x1 = x[:1].contiguous()
    for _ in range(3):
        cube = net.forward_nhwc(x1)
    s0, s1, s2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    s0.record()
    for _ in range(iters):
        cube = net.forward_nhwc(x1)
    s1.record()
    for _ in range(iters):
        bands = safe_norm_maps(mantis_bands(cube, net))
    s2.record()
    # configs[3] as BASELINE words it: forward with the ten-band projection fused on the output (no cube written)
    from animal_vision_b200 import tables as _tables
    Wm = _tables.mantis_band_matrix(np.linspace(400.0, 700.0, 31, dtype=np.float32))
    for _ in range(3):
        net.forward_bands(x1, Wm)
    s3, s4 = (torch.cuda.Event(enable_timing=True) for _ in range(2))
    s3.record()
    for _ in range(iters):
        fused_bands = net.forward_bands(x1, Wm)
    s4.record()
    barrier()
    fused_ms = s3.elapsed_time(s4) / iters
    single_ms, bands_ms = s0.elapsed_time(s1) / iters, s1.elapsed_time(s2) / iters
    cpu_ref = None
    if world == 1 and not args.no_cpu:
        from oracle import mstpp as O                    # the checker, timed as the CPU baseline of configs[3]
        torch.set_num_threads(_affinity_cores())
        xc = x1.permute(0, 3, 1, 2).cpu().contiguous()
        sd = synthetic_state_dict(0)
        t0 = time.perf_counter()
        yc = O.forward(xc, sd)
        cpu_s = time.perf_counter() - t0
        rel = float((cube.permute(0, 3, 1, 2).cpu() - yc).abs().max() / yc.abs().max())
        cpu_ref = {"ms_per_patch": cpu_s * 1e3, "patches_per_s": 1.0 / cpu_s, "kind": "port", "cores": _affinity_cores(),
                   "what": "fp32 torch-CPU forward of the reference architecture (oracle restatement, pinned to the reference module), one 482x512 patch, all host threads",
                   "gpu_vs_cpu_max_abs_rel": rel}
    return {"single_patch_ms": single_ms, "mantis_bands_ms": bands_ms, "single_patch_fused_bands_ms": fused_ms, "cpu_reference": cpu_ref,
            "workload": f"MST++ forward, {nb} x 3x482x512 patches per GPU (BASELINE configs[3]), seeded weights, bf16 operands / fp32 accumulate",
            "patches_per_s": nb * world / (ms * 1e-3), "ms_per_forward": ms, "batch_per_gpu": nb, "concurrent_forwards": parts,
            "roofline": {"bound": "tensor", "achieved": tf / world, "peak": peak, "unit": "TFLOP/s", "frac": tf / world / peak,
                         "peak_source": src, "algorithmic_flop_per_patch": MSTPP_FLOP_PER_PATCH,
                         "note": "whole forward (104 dependent launches chained with programmatic dependent launch), not one kernel; at C=31 the network is bound by per-kernel latency and HBM, not by the tensor pipe (SURVEY.md section 7)"}}


# ----------------------------------------------------------------------------- GPU arm
def run_b200(args):
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout must carry the ONE JSON line and nothing else, but native libraries (NCCL's "NCCL version ..."
    # banner) print to file descriptor 1: park the real stdout, point fd 1 at stderr for the whole run and
    # write the JSON line to the parked descriptor at the end
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    from animal_vision_b200 import _abi
    import animal_vision_b200.animals as A
    from animal_vision_b200.engine import get_engine
    from animal_vision_b200.pipeline import HostBatchPipeline

    lib = _abi.load()
    eng = get_engine(dev)
    H, W, nf = args.height, args.width, args.frames
    species = {sp: getattr(A, sp)() for sp in SPECIES}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    t_gen = time.time()
    host = make_host_frames(rank, world, nf, H, W, pinned=True)
    log(f"[rank {rank}] generated {nf} host frames {W}x{H} in {time.time() - t_gen:.1f}s")
    dev_in = {sp: host[sp].to(dev, non_blocking=True) for sp in SPECIES}
    dev_out = {sp: ((torch.empty_like(dev_in[sp]), torch.empty_like(dev_in[sp])) if sp == "Cat" else torch.empty_like(dev_in[sp]))
               for sp in SPECIES}
    torch.cuda.synchronize()
    px_step = nf * H * W                                   # per GPU

    # The three species batches are independent: each runs on its own stream (fork / join with events on
    # the timing stream), so the partially filled last wave of one kernel overlaps the next species' work.
    nsplit = max(0, args.streams)
    side = {(sp, k): torch.cuda.Stream(device=dev) for sp in SPECIES for k in range(nsplit)} if nsplit else None

    def run_part(sp, k, parts):
        n = dev_in[sp].shape[0]
        a, b = n * k // parts, n * (k + 1) // parts
        if a == b:
            return
        o = dev_out[sp]
        species[sp].visualize_batch(dev_in[sp][a:b], out=(o[0][a:b], o[1][a:b]) if isinstance(o, tuple) else o[a:b])

    def step(single: bool = False):
        if side is None or single:
            for sp in SPECIES:
                run_part(sp, 0, 1)
            return
        main = torch.cuda.current_stream(dev)
        fork = torch.cuda.Event()
        fork.record(main)
        for k in range(nsplit):
            for sp in SPECIES:
                st = side[(sp, k)]
                st.wait_event(fork)
                with torch.cuda.stream(st):
                    run_part(sp, k, nsplit)
                    done = torch.cuda.Event()
                    done.record(st)
                main.wait_event(done)

    def checksum():
        outs = []
        for sp in SPECIES:
            o = dev_out[sp]
            outs += list(o) if isinstance(o, tuple) else [o]
        return [int(t.reshape(-1).view(torch.int32).sum(dtype=torch.int64).item()) for t in outs]

    # ---- device-resident throughput ("value")
    for _ in range(args.warmup):
        step()
    barrier()
    sampler = ClockSampler(local).start() if rank == 0 else None
    launches0 = eng.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    for _ in range(args.steps):
        step()
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms_step = max_over_ranks(e0.elapsed_time(e1) / args.steps)
    launches = eng.launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dev_out)

    # ---- per-kernel timing over the same steps (roofline leg): CUDA events around every launch
    prof_steps = max(1, min(args.steps, 3))
    sum_streams = checksum()                        # outputs of the concurrent steps ...
    step(single=True)                               # per-kernel times are taken on ONE stream: no overlap between kernels
    torch.cuda.synchronize()
    streams_ok = checksum() == sum_streams          # ... equal those of a single-stream step
    lib.avb_profile_begin()
    for _ in range(prof_steps):
        step(single=True)
    cap = 4096
    names = C.create_string_buffer(cap * 48)
    msbuf = (C.c_float * cap)()
    nrec = lib.avb_profile_end(names, 48, msbuf, cap)
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    kern = {}
    for i in range(nrec):
        nm = names.raw[i * 48:(i + 1) * 48].split(b"\0", 1)[0].decode()
        k = kern.setdefault(nm, [0.0, 0])
        k[0] += float(msbuf[i])
        k[1] += 1
    total_ms = sum(v[0] for v in kern.values()) or 1.0
    shares = {nm: {"ms_per_launch": v[0] / v[1], "launches_per_step": v[1] / prof_steps, "share": v[0] / total_ms}
              for nm, v in sorted(kern.items(), key=lambda kv: -kv[1][0])}
    dom = next(iter(shares))
    dom_sp = KERNEL_SPECIES.get(dom, "Dog")
    frames_per_launch = dev_in[dom_sp].shape[0]
    bpp = KERNEL_ALGO_BYTES_PER_PX.get(dom, ALGO_BYTES_PER_PX[dom_sp])
    algo_bytes = bpp * frames_per_launch * H * W
    traffic, traffic_src = ncu_traffic(dom, frames_per_launch, H, W)
    peak, peak_src = peak_numbers()
    achieved = algo_bytes / (shares[dom]["ms_per_launch"] * 1e-3) / 1e9
    # the same figure for every kernel that has an algorithmic byte count, and per species path (all its kernels, uint8 in + out(s))
    for nm, rec in shares.items():
        if nm in KERNEL_ALGO_BYTES_PER_PX:
            n_fr = dev_in[KERNEL_SPECIES.get(nm, "Dog")].shape[0]
            gbs = KERNEL_ALGO_BYTES_PER_PX[nm] * n_fr * H * W / (rec["ms_per_launch"] * 1e-3) / 1e9
            rec["algorithmic_gbs"] = gbs
            rec["frac_of_hbm_peak"] = gbs / peak
    paths = {}
    for sp in SPECIES:
        ms_sp = sum(rec["ms_per_launch"] * rec["launches_per_step"] for nm, rec in shares.items() if KERNEL_SPECIES.get(nm) == sp)
        if ms_sp > 0:
            gbs = ALGO_BYTES_PER_PX[sp] * dev_in[sp].shape[0] * H * W / (ms_sp * 1e-3) / 1e9
            paths[sp] = {"kernel_ms_per_step": ms_sp, "algorithmic_bytes_per_px": ALGO_BYTES_PER_PX[sp], "algorithmic_gbs": gbs,
                         "frac_of_hbm_peak": gbs / peak}
    roofline = {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "peak_source": peak_src, "traffic_source": traffic_src,
                "algorithmic_bytes_per_launch": algo_bytes,
                "note": f"{bpp:g} B/px x {frames_per_launch} frames x {W}x{H}; duration = mean CUDA-event time of this kernel over {prof_steps} step(s)",
                "kernel_shares": shares, "species_paths": paths}

    # ---- end to end through the host API: pinned host in -> pinned host out
    pipe = HostBatchPipeline(dev, chunk_frames=args.chunk)
    host_out = {sp: pipe.pinned_like(host[sp], pipe.n_outputs(species[sp])) for sp in SPECIES}
    jobs = [(species[sp], host[sp], host_out[sp]) for sp in SPECIES]
    for _ in range(max(1, min(args.warmup, 2))):
        pipe.run(jobs)
    barrier()
    e2e_steps = max(1, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        h2d, d2h = pipe.run(jobs)
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps)
    barrier()

    # ---- K1 leg (north_star kernel 1, BASELINE configs[0]'s species family): the pure colorimetric kernel
    # (Rat: LUT decode, 3x3, row gain, encode) on the Dog shard, device resident, CUDA events
    rat = A.Rat()
    rat_out = torch.empty_like(dev_in["Dog"])
    for _ in range(3):
        rat.visualize_batch(dev_in["Dog"], out=rat_out)
    barrier()
    k0, k1e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k0.record()
    for _ in range(10):
        rat.visualize_batch(dev_in["Dog"], out=rat_out)
    k1e.record()
    barrier()
    k1_ms = max_over_ranks(k0.elapsed_time(k1e) / 10)
    k1_bytes = 6.0 * dev_in["Dog"].shape[0] * H * W
    colorimetric = {"kernel": "k1_colorimetric (+ its AVB_NORM_AUTO fixup launch)", "species": "Rat", "frames": int(dev_in["Dog"].shape[0]),
                    "ms": k1_ms, "mpix_per_s": dev_in["Dog"].shape[0] * H * W / (k1_ms * 1e-3) / 1e6,
                    "roofline": {"bound": "hbm", "achieved": k1_bytes / (k1_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                 "frac": k1_bytes / (k1_ms * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": k1_bytes}}

    # ---- K4 leg (BASELINE configs[3]): MST++ forward on 482x512 patches, tensor-pipe roofline
    mstpp = run_mstpp_leg(args, dev, rank, world, max_over_ranks, barrier)

    # ---- BASELINE configs[0..2]: one 1080p frame per species through visualize(np.ndarray) (rank 0 only)
    configs = run_config_legs(dev, species, peak, with_cpu=(world == 1 and not args.no_cpu)) if rank == 0 and not args.no_configs else None
    uv_species = run_uv_species_leg(dev, peak, with_cpu=(world == 1 and not args.no_cpu)) if rank == 0 and not args.no_configs else None
    barrier()

    # sanity: the e2e outputs equal the device-resident outputs (same kernels, same inputs)
    ok = bool(torch.equal(host_out["Dog"][0][:2], dev_out["Dog"][:2].cpu()))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    value = world * px_step / (ms_step * 1e-3) / 1e6
    e2e_val = world * px_step / (e2e_ms * 1e-3) / 1e6
    line = {
        "metric": "Mpix/s", "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": dict(bench_config(), resolution=f"{W}x{H}", frames_per_gpu=nf),
        "detail": {"parallelism": f"frame-sharded x{world}, no collective",
                   "streams": f"{3 * nsplit} CUDA streams: every species batch in {nsplit} part(s), fork/join on the timed stream; outputs equal the single-stream step: {streams_ok}" if nsplit else "single stream",
                   "l2": f"inputs {nf * H * W * 3 / 1e6:.0f} MB per step per GPU, larger than the 126 MB L2 (no flush needed)",
                   "normalisation": "AVB_NORM_AUTO (reference semantics, decided per frame on device)"},
        "fps_4k": value * 1e6 / (H4K * W4K),
        "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": "Mpix/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "ms_per_step": e2e_ms, "steps": e2e_steps, "fps_4k": e2e_val * 1e6 / (H4K * W4K),
                "api": "HostBatchPipeline.run: pinned host frames -> H2D -> Animal.visualize_batch -> D2H -> pinned host frames",
                "outputs_match_device_path": ok},
        "gpu_launches": int(launches),
        "roofline": roofline,
    }
    line["mstpp"] = mstpp
    line["configs"] = configs
    line["uv_species"] = uv_species
    line["colorimetric"] = colorimetric
    if world == 1 and not args.no_cpu:
        threads = host_threads()
        rows = args.cpu_rows
        sample = cpu_sample(rows)
        oracle_step_time(cpu_sample(64))                                  # warm up imports / thread pools
        dt = oracle_step_time(sample)
        line["cpu_baseline"] = {
            "value": 3 * rows * W4K / dt / 1e6, "unit": "Mpix/s",
            "cores": threads.get("sched_affinity") or threads.get("os_cpu_count") or 1, "kind": "port",
            "sample": f"1 Dog + 1 Cat + 1 HoneyBee frame of {rows}x{W4K} (full-width band of a 4K frame), {dt:.1f} s of CPU work, oracle port with OpenCV/BLAS threads = all cores",
            "threads": threads}
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--height", type=int, default=H4K)
    ap.add_argument("--width", type=int, default=W4K)
    ap.add_argument("--frames", type=int, default=FRAMES_PER_GPU, help="frames per GPU per step (multiple of 3)")
    ap.add_argument("--chunk", type=int, default=2, help="frames per pipeline chunk in the e2e leg")
    ap.add_argument("--cpu-rows", type=int, default=1080, help="rows of the 3840-wide CPU-baseline sample frames")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-configs", action="store_true", help="skip the per-config 1080p single-frame legs")
    ap.add_argument("--streams", type=int, default=1, help="streams per species batch in the device-resident step (the batch is cut into that many parts); 0: a single stream")
    ap.add_argument("--mstpp-batch", type=int, default=4, help="482x512 patches per GPU in the MST++ leg (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step (rank 0's frames) as DIR/<name>.npy, float32, "
                         "at most 64 MB in all: a fixed seeded pixel sample of a larger output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
