"""JPEG with optimized Huffman tables (K8's optimized mode, cv2.IMWRITE_JPEG_OPTIMIZE) against the standard tables.

    python tools/jpeg_opt_bench.py [--out profiles/jpeg_opt_bench.jsonl] [--iters 10] [--rounds 3]

One run measures, with the card name and power limit read in the same process:
  - encode_jpeg of 20 frames at 1080p and at 4K (tests/frames.py natural and noise), quality 75 and 95: CUDA events
    around `iters` calls after warm-up (each call includes its D2H of the lengths and of the used bytes), the standard
    and the optimized mode alternated `rounds` times; per-stage kernel times from the library's profiler on one extra
    call of each mode; the mean file size of each mode; whether every file equals cv2.imencode's;
  - cv2.imencode of the same 20 frames on the host, with and without IMWRITE_JPEG_OPTIMIZE, one call per frame;
  - bench.py's e2e workload (bench.make_host_frames: 60 4K frames, Dog / Cat / HoneyBee, pinned) through
    HostBatchPipeline.run_split_jpeg in chunks of 2 at depth 3, quality 95, standard against optimized, alternated,
    with a host clock around each call (which ends in a device synchronise) and the D2H bytes each copies.
Appends one JSON line to --out."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import animal_vision_b200.animals as A  # noqa: E402
import frames  # noqa: E402
from animal_vision_b200 import _abi  # noqa: E402
from animal_vision_b200.jpeg import encode_jpeg  # noqa: E402
from animal_vision_b200.pipeline import HostBatchPipeline  # noqa: E402
from bench import H4K, SPECIES, W4K, make_host_frames  # noqa: E402
from split_bench import card  # noqa: E402

N = 20
MODES = {"standard": False, "optimized": True}


def stage_times(batch, q, optimize):
    lib = _abi.load()
    lib.avb_profile_begin()
    encode_jpeg(batch, q, optimize=optimize)
    names = C.create_string_buffer(64 * 32)
    ms = (C.c_float * 32)()
    n = lib.avb_profile_end(names, 64, ms, 32)
    return {names.raw[64 * i:64 * (i + 1)].split(b"\0")[0].decode(): round(float(ms[i]), 4) for i in range(n)}


def time_device(batch, q, optimize, iters):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        out = encode_jpeg(batch, q, optimize=optimize)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, out


def host_encode(imgs, q, optimize):
    params = [cv2.IMWRITE_JPEG_QUALITY, q] + ([cv2.IMWRITE_JPEG_OPTIMIZE, 1] if optimize else [])
    t0 = time.perf_counter()
    out = [cv2.imencode(".jpg", im, params)[1].tobytes() for im in imgs]
    return (time.perf_counter() - t0) * 1e3, out


class CountingSink:
    def __init__(self):
        self.records = self.jpeg_bytes = self.frames = 0

    def write_records(self, records, jpeg_lengths):
        self.records += len(records)
        self.jpeg_bytes += sum(jpeg_lengths)
        self.frames += len(jpeg_lengths)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "jpeg_opt_bench.jsonl"))
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=3)
    a = ap.parse_args()
    rec = {"tool": "jpeg_opt_bench", "card": card(), "host_cores": os.cpu_count(), "frames": N, "cases": []}
    cv2.setNumThreads(1)
    for h, w in ((1080, 1920), (H4K, W4K)):
        for kind in ("natural", "noise"):
            imgs = [frames.natural(h, w, s) if kind == "natural" else frames.noise(h, w, s) for s in range(N)]
            batch = torch.from_numpy(np.stack(imgs)).cuda()
            for q in (75, 95):
                for opt in MODES.values():
                    encode_jpeg(batch, q, optimize=opt)
                torch.cuda.synchronize()
                ms = {m: [] for m in MODES}
                out = {}
                for _ in range(a.rounds):
                    for m, opt in MODES.items():
                        t, out[m] = time_device(batch, q, opt, a.iters)
                        ms[m].append(round(t, 3))
                c = {"shape": [h, w], "content": kind, "quality": q}
                for m, opt in MODES.items():
                    host_ms, ref = host_encode(imgs, q, opt)
                    med = statistics.median(ms[m])
                    c[m] = {"device_ms_per_call": ms[m], "device_ms_per_frame": round(med / N, 4),
                            "mean_bytes": round(sum(len(b) for b in out[m]) / N), "identical_to_cv2": out[m] == ref,
                            "host_cv2_ms_per_frame": round(host_ms / N, 2), "stages_ms": stage_times(batch, q, opt)}
                c["optimized_smaller_by"] = round(1 - c["optimized"]["mean_bytes"] / c["standard"]["mean_bytes"], 4)
                c["device_time_ratio"] = round(c["optimized"]["device_ms_per_frame"] / c["standard"]["device_ms_per_frame"], 3)
                print(json.dumps(c), flush=True)
                rec["cases"].append(c)
            del batch
            torch.cuda.empty_cache()

    host = make_host_frames(0, 1, 60, H4K, W4K, pinned=True)
    species = {sp: getattr(A, sp)() for sp in SPECIES}
    jobs = [(species[sp], host[sp]) for sp in SPECIES]
    pipe = HostBatchPipeline(chunk_frames=2, depth=3)
    e2e = {m: {"ms": []} for m in MODES}
    for opt in MODES.values():                             # warm-up: every shape and slot set of both modes
        pipe.run_split_jpeg(jobs, quality=95, optimize=opt, out=CountingSink())
    for _ in range(a.rounds):
        for m, opt in MODES.items():
            sink = CountingSink()
            t0 = time.perf_counter()
            h2d, d2h = pipe.run_split_jpeg(jobs, quality=95, optimize=opt, out=sink)
            e2e[m]["ms"].append(round((time.perf_counter() - t0) * 1e3, 1))
            e2e[m].update(h2d_bytes=int(h2d), d2h_bytes=int(d2h), mean_jpeg_bytes=round(sink.jpeg_bytes / sink.frames))
    for m in MODES:
        e2e[m]["median_ms"] = statistics.median(e2e[m]["ms"])
        e2e[m]["frames_per_s"] = round(60 / (e2e[m]["median_ms"] * 1e-3), 1)
    rec["run_split_jpeg_e2e"] = {"workload": {"frames": 60, "resolution": f"{W4K}x{H4K}", "species": list(SPECIES),
                                              "chunk": 2, "depth": 3, "quality": 95}, **e2e}
    print(json.dumps(rec["run_split_jpeg_e2e"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fh:
        fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
