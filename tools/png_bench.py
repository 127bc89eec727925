"""Device PNG encode (K10) against cv2.imencode(".png") on the host, and the server path with each encoder.

    python tools/png_bench.py [--out profiles/png_bench.jsonl] [--iters 10]

One run measures, on the same frames (tests/frames.py natural and noise; noise codes as stored blocks, the largest
output):
  - encode_png on batches of 20 frames at 1080p and 4K: CUDA events around `iters` calls after warm-up (each call
    includes its D2H of the lengths and of the used bytes), per-stage kernel times from the library's profiler on one
    extra call;
  - cv2.imencode(".png") of the same frames on the host, one call per frame, with the host's core count;
  - process_image_png throughput for 16 concurrent 1080p requests (Dog): the default device batcher (device encode)
    against a batcher whose runner returns host arrays (host encode), alternated.
Appends one JSON line to --out, with the card name and power limit."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

import frames  # noqa: E402
from animal_vision_b200 import _abi, serving  # noqa: E402
from animal_vision_b200.png import encode_png  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def stage_times(batch):
    lib = _abi.load()
    lib.avb_profile_begin()
    encode_png(batch)
    names = C.create_string_buffer(64 * 32)
    ms = (C.c_float * 32)()
    n = lib.avb_profile_end(names, 64, ms, 32)
    return {names.raw[64 * i:64 * (i + 1)].split(b"\0")[0].decode(): round(float(ms[i]), 4) for i in range(n)}


def time_device(batch, iters):
    for _ in range(3):
        encode_png(batch)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        out = encode_png(batch)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, out


def time_host(imgs, reps):
    cv2.imencode(".png", imgs[0])
    t0 = time.perf_counter()
    for _ in range(reps):
        for im in imgs:
            cv2.imencode(".png", im)
    return (time.perf_counter() - t0) * 1e3 / reps


def host_runner():
    dev = serving._device_runner()

    def run(key, batch):
        return dev(key, batch).cpu().numpy()           # species on the device, view back as pixels: cv2 encodes
    return run


def serve_rate(fb, reqs, rounds):
    def one():
        ths = [threading.Thread(target=serving.process_image_png, args=(r, "dog", fb)) for r in reqs]
        [t.start() for t in ths]
        [t.join() for t in ths]
    one()
    t0 = time.perf_counter()
    for _ in range(rounds):
        one()
    return len(reqs) * rounds / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "png_bench.jsonl"))
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    rec = {"tool": "png_bench", "card": card(), "host_cores": os.cpu_count(), "cases": []}
    for (h, w, n) in ((1080, 1920, 20), (2160, 3840, 20)):
        for kind in ("natural", "noise"):
            imgs = [frames.natural(h, w, s) if kind == "natural" else frames.noise(h, w, s) for s in range(n)]
            batch = torch.from_numpy(np.stack(imgs)).cuda()
            ms, out = time_device(batch, a.iters)
            ref = [cv2.imencode(".png", im)[1].tobytes() for im in imgs]
            host_ms = time_host(imgs, 1)
            nbytes = sum(len(b) for b in out)
            c = {"shape": [h, w], "frames": n, "content": kind, "identical_to_cv2": out == ref,
                 "device_ms_per_frame": round(ms / n, 4), "device_gpix_s": round(n * h * w / ms / 1e6, 3),
                 "bytes_per_frame": nbytes // n,
                 "host_cv2_ms_per_frame": round(host_ms / n, 3), "host_cv2_gpix_s": round(n * h * w / host_ms / 1e6, 4),
                 "stages_ms": stage_times(batch)}
            print(json.dumps(c), flush=True)
            rec["cases"].append(c)
            del batch
    reqs = [cv2.imencode(".jpg", frames.natural(1080, 1920, s))[1].tobytes() for s in range(16)]
    dev_rates, host_rates = [], []
    with serving.FrameBatcher(max_batch=16, max_delay_ms=5.0) as fd, \
            serving.FrameBatcher(host_runner(), max_batch=16, max_delay_ms=5.0) as fh:
        for _ in range(3):
            dev_rates.append(round(serve_rate(fd, reqs, 3), 2))
            host_rates.append(round(serve_rate(fh, reqs, 1), 2))
    rec["process_image_png_16x1080p_req_s"] = {"device_encode": dev_rates, "host_encode": host_rates}
    print(json.dumps(rec["process_image_png_16x1080p_req_s"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fh_:
        fh_.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
