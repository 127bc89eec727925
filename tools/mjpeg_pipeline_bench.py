"""Split-compare video as a Motion-JPEG AVI: frames encoded on the host against frames encoded on the device.

    python tools/mjpeg_pipeline_bench.py [--rounds 3] [--out profiles/mjpeg_pipeline.jsonl] [--dir /dev/shm]

Workload: bench.py's e2e leg (bench.make_host_frames: 60 4K frames, Dog / Cat / HoneyBee, pinned; chunks of 2 frames,
depth 3), quality 95.  After warm-up every round times, one after the other, with a host clock around work that ends in a
device synchronise and a closed file:
  (a) run_split, then cv2.imencode of every split frame (channels swapped, as VideoRenderer.render does) and
      MjpegAviWriter.write_jpeg, on one thread: the host route a caller of run_split has today;
  (b) run_split_jpeg into an MjpegAviWriter: frames encoded on the device (K8 RGB + K11), only records cross;
  (b1) the same on a pipeline of depth 1, which shows what the overlap of chunks is worth;
  (c) run_split alone, the reference point (no encode, no file).
(a) and (c) overwrite their frames, so they run on a copy restored before every step, outside the timed region; (b)
leaves them unchanged.  The videos go to --dir (tmpfs by default, so the disk is not what is timed); (a)'s and (b)'s
files are compared byte for byte.  K8 and K11 are timed alone, per kernel with CUDA events, on one chunk of 4K split
frames.  The card name and power limit are read in the same process.  Appends one JSON line to --out."""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)

import ctypes as C  # noqa: E402

import cv2  # noqa: E402
import torch  # noqa: E402

import animal_vision_b200.animals as A  # noqa: E402
from animal_vision_b200._abi import check  # noqa: E402
from animal_vision_b200.engine import get_engine  # noqa: E402
from animal_vision_b200.jpeg import JpegLauncher  # noqa: E402
from animal_vision_b200.pipeline import HostBatchPipeline  # noqa: E402
from animal_vision_b200.renderers.mjpeg import MjpegAviWriter  # noqa: E402
from bench import H4K, SPECIES, W4K, make_host_frames  # noqa: E402
from split_bench import card  # noqa: E402

FRAMES, CHUNK, DEPTH, QUALITY, FPS = 60, 2, 3, 95, 30
LABELS = ("Original", "Transformed")


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return (time.perf_counter() - t0) * 1e3, r


def kernel_ms(frames_dev, iters=10):
    """Per-kernel CUDA-event times (avb_profile_begin / _end), per frame, of K8 (RGB) on a chunk of 4K frames and of
    K11 packing its files."""
    eng = get_engine()
    lib = eng.lib
    k8 = JpegLauncher(lib, H4K, W4K, QUALITY, rgb=True)
    n = frames_dev.shape[0]
    ws = torch.empty(k8.workspace_bytes(n), dtype=torch.uint8, device="cuda")
    slots = torch.empty(n * k8.slot, dtype=torch.uint8, device="cuda")
    packed = torch.empty(n * (8 + ((k8.slot + 3) & ~3)), dtype=torch.uint8, device="cuda")
    meta = torch.empty(2 * n + 1, dtype=torch.int64, device="cuda")

    def step():
        st = eng.stream_ptr()
        check(k8.launch(frames_dev.data_ptr(), n, H4K * W4K * 3, W4K * 3, ws.data_ptr(), slots.data_ptr(), k8.slot,
                        meta[n + 1:].data_ptr(), st), k8.name)
        check(lib.avb_mjpeg_pack_u8(slots.data_ptr(), k8.slot, meta[n + 1:].data_ptr(), n, packed.data_ptr(),
                                    meta.data_ptr(), st), "avb_mjpeg_pack_u8")
    for _ in range(3):
        step()
    torch.cuda.synchronize()
    lib.avb_profile_begin()
    for _ in range(iters):
        step()
    names, ms = C.create_string_buffer(256 * 48), (C.c_float * 256)()
    got = lib.avb_profile_end(names, 48, ms, 256)
    agg = {}
    for i in range(got):
        nm = names.raw[i * 48:(i + 1) * 48].split(b"\0", 1)[0].decode()
        agg[nm] = agg.get(nm, 0.0) + ms[i] / iters / n
    k8_total = sum(v for k, v in agg.items() if k.startswith("jpeg_"))
    return {"k8_ms_per_frame": round(k8_total, 3), "k11_ms_per_frame": round(agg.get("mjpeg_pack", 0.0), 4),
            "k8_kernels_ms_per_frame": {k: round(v, 4) for k, v in agg.items() if k.startswith("jpeg_")}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "mjpeg_pipeline.jsonl"))
    ap.add_argument("--dir", default="/dev/shm" if os.path.isdir("/dev/shm") else None)
    a = ap.parse_args()
    tmp = tempfile.mkdtemp(prefix="mjpeg_bench_", dir=a.dir)
    rec = {"tool": "mjpeg_pipeline_bench", "card": card(), "host_cores": os.cpu_count(),
           "workload": {"frames": FRAMES, "resolution": f"{W4K}x{H4K}", "species": list(SPECIES), "chunk": CHUNK,
                        "depth": DEPTH, "quality": QUALITY, "labels": list(LABELS), "video_dir": a.dir},
           "rounds": a.rounds}
    host = make_host_frames(0, 1, FRAMES, H4K, W4K, pinned=True)
    work = {sp: torch.empty_like(host[sp]).pin_memory() for sp in SPECIES}
    species = {sp: getattr(A, sp)() for sp in SPECIES}
    pipe = HostBatchPipeline(chunk_frames=CHUNK, depth=DEPTH)
    pipe1 = HostBatchPipeline(chunk_frames=CHUNK, depth=1)
    split_jobs = [(species[sp], work[sp]) for sp in SPECIES]
    jpeg_jobs = [(species[sp], host[sp]) for sp in SPECIES]
    paths = {r: os.path.join(tmp, f"{r}.avi") for r in ("host_encode", "device_encode", "device_encode_depth1")}

    def restore():
        for sp in SPECIES:
            work[sp].copy_(host[sp])

    def route_a():
        h2d, d2h = pipe.run_split(split_jobs, labels=LABELS)
        nbytes = 0
        with MjpegAviWriter(paths["host_encode"], FPS, (W4K, H4K)) as wr:
            for sp in SPECIES:
                for f in work[sp].numpy():
                    j = cv2.imencode(".jpg", f[..., ::-1], [cv2.IMWRITE_JPEG_QUALITY, QUALITY])[1]
                    nbytes += j.size
                    wr.write_jpeg(j.tobytes())
        return h2d, d2h, nbytes

    def route_b():
        with MjpegAviWriter(paths["device_encode"], FPS, (W4K, H4K)) as wr:
            h2d, d2h = pipe.run_split_jpeg(jpeg_jobs, labels=LABELS, quality=QUALITY, out=wr)
        return h2d, d2h, os.path.getsize(paths["device_encode"])

    def route_b1():
        with MjpegAviWriter(paths["device_encode_depth1"], FPS, (W4K, H4K)) as wr:
            h2d, d2h = pipe1.run_split_jpeg(jpeg_jobs, labels=LABELS, quality=QUALITY, out=wr)
        return h2d, d2h, os.path.getsize(paths["device_encode_depth1"])

    def route_c():
        h2d, d2h = pipe.run_split(split_jobs, labels=LABELS)
        return h2d, d2h, 0

    routes = {"run_split_host_imencode": route_a, "run_split_jpeg": route_b, "run_split_jpeg_depth1": route_b1,
              "run_split": route_c}
    for fn in routes.values():                        # warm-up: every shape, slot set and file path
        restore()
        fn()
    threads, cv_threads = torch.get_num_threads(), cv2.getNumThreads()
    ms = {r: [] for r in routes}
    res = {}
    for _ in range(a.rounds):
        for name, fn in routes.items():
            restore()
            one = name == "run_split_host_imencode"
            if one:                                   # the host route on one thread, as the reference's loop runs
                torch.set_num_threads(1)
                cv2.setNumThreads(1)
            dt, res[name] = timed(fn)
            if one:
                torch.set_num_threads(threads)
                cv2.setNumThreads(cv_threads)
            ms[name].append(dt)
        print(json.dumps({k: round(v[-1], 1) for k, v in ms.items()}), flush=True)
    files = {r: open(p, "rb").read() for r, p in paths.items()}
    same = files["host_encode"] == files["device_encode"] == files["device_encode_depth1"]
    px = FRAMES * H4K * W4K
    for name, v in ms.items():
        med = statistics.median(v)
        h2d, d2h, _ = res[name]
        rec[name] = {"ms_per_step": [round(x, 1) for x in v], "median_ms_per_step": round(med, 1),
                     "frames_per_s": round(FRAMES / (med * 1e-3), 1), "h2d_bytes_per_step": int(h2d),
                     "d2h_bytes_per_step": int(d2h), "d2h_bytes_per_px": round(d2h / px, 4)}
    rec["mean_jpeg_bytes"] = round(res["run_split_host_imencode"][2] / FRAMES)
    rec["run_split_jpeg"]["file_bytes"] = res["run_split_jpeg"][2]
    rec["files_identical"] = bool(same)
    restore()
    pipe.run_split([(species["Dog"], work["Dog"][:CHUNK])], labels=LABELS)
    rec["kernels_4k"] = kernel_ms(work["Dog"][:CHUNK].cuda())
    for p in paths.values():
        os.remove(p)
    os.rmdir(tmp)
    print(json.dumps(rec), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fh:
        fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
