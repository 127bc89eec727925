"""HostBatchPipeline.run_split against run(), and against run() plus the host compose a caller needs for split frames.

    python tools/split_pipeline_bench.py [--rounds 5] [--steps 3] [--out profiles/split_pipeline.jsonl]

Workload: bench.py's e2e leg (bench.make_host_frames: 60 4K frames, Dog / Cat / HoneyBee, pinned; chunks of 2 frames,
depth 3).  After warm-up every round times, one after the other:
  (a) run(): every species output comes back (Dog and HoneyBee one frame, Cat two);
  (b) run() plus the host compose of the labelled split frames that the caller of (a) does today: split_compare_batch on
      CPU tensors, then draw_split_labels, one frame at a time on one thread (also reported per frame);
  (c) run_split(): the labelled split frames in place, only the label band and columns [W/2, W) copied back.
(a) and (c) are timed over --steps steps, (b) over one (its host compose dominates), each with a host clock around work
that ends in a device synchronise.  run_split overwrites its frames, so (c) runs on a copy restored before every step,
outside the timed region.  Some (c) frames are compared with (b)'s.  A copy probe times the split fetch of 20 4K frames
against one contiguous device-to-host copy of the same byte count (CUDA events), to show whether the pitched rows
(5.8 KB right halves at 4K) copy slower.  The card name and power limit are read in the same process.  Appends one
JSON line to --out."""
from __future__ import annotations

import argparse
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
from animal_vision_b200.engine import get_engine  # noqa: E402
from animal_vision_b200.pipeline import HostBatchPipeline  # noqa: E402
from animal_vision_b200.renderers.video import draw_split_labels, split_compare_batch  # noqa: E402
from bench import H4K, SPECIES, W4K, make_host_frames  # noqa: E402
from split_bench import card  # noqa: E402

FRAMES, CHUNK = 60, 2
LABELS = ("Original", "Transformed")


def host_compose(frames_host, view_host):
    """The split frames of one species batch as the caller of run() builds them: one frame at a time."""
    return [draw_split_labels(split_compare_batch(frames_host[k:k + 1], view_host[k:k + 1])[0].numpy(), *LABELS)
            for k in range(frames_host.shape[0])]


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return (time.perf_counter() - t0) * 1e3, r


def fetch_probe(iters=20):
    eng = get_engine()
    n = 20
    band = eng.split_stencil(H4K, W4K, *LABELS)[0]
    src = torch.randint(0, 256, (n, H4K, W4K, 3), dtype=torch.uint8, device="cuda")
    dst = torch.empty((n, H4K, W4K, 3), dtype=torch.uint8).pin_memory()
    nbytes = eng.split_fetch(src, dst, band)
    flat_src, flat_dst = src.view(-1)[:nbytes], dst.view(-1)[:nbytes]
    res = {"frames": n, "bytes": nbytes}
    for name, fn in (("split_fetch", lambda: eng.split_fetch(src, dst, band)),
                     ("contiguous_copy", lambda: flat_dst.copy_(flat_src, non_blocking=True))):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / iters
        res[name] = {"ms": round(ms, 3), "gb_s": round(nbytes / ms / 1e6, 1)}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "split_pipeline.jsonl"))
    a = ap.parse_args()
    rec = {"tool": "split_pipeline_bench", "card": card(), "host_cores": os.cpu_count(),
           "workload": {"frames": FRAMES, "resolution": f"{W4K}x{H4K}", "species": list(SPECIES), "chunk": CHUNK,
                        "depth": 3, "labels": list(LABELS)},
           "rounds": a.rounds, "steps": a.steps}
    px = FRAMES * H4K * W4K
    host = make_host_frames(0, 1, FRAMES, H4K, W4K, pinned=True)
    work = {sp: torch.empty_like(host[sp]).pin_memory() for sp in SPECIES}
    species = {sp: getattr(A, sp)() for sp in SPECIES}
    pipe = HostBatchPipeline(chunk_frames=CHUNK)
    outs = {sp: pipe.pinned_like(host[sp], pipe.n_outputs(species[sp])) for sp in SPECIES}
    jobs = [(species[sp], host[sp], outs[sp]) for sp in SPECIES]
    split_jobs = [(species[sp], work[sp]) for sp in SPECIES]

    def restore():
        for sp in SPECIES:
            work[sp].copy_(host[sp])

    for _ in range(2):
        pipe.run(jobs)
        restore()
        pipe.run_split(split_jobs, labels=LABELS)
    threads, cv_threads = torch.get_num_threads(), cv2.getNumThreads()
    ms = {"run": [], "run_plus_host_compose": [], "run_split": []}
    compose_ms = []
    for _ in range(a.rounds):
        t = 0.0
        for _ in range(a.steps):
            dt, (h2d_a, d2h_a) = timed(lambda: pipe.run(jobs))
            t += dt
        ms["run"].append(t / a.steps)
        torch.set_num_threads(1)
        cv2.setNumThreads(1)
        dt_run, _ = timed(lambda: pipe.run(jobs))
        dt, split_host = timed(lambda: {sp: host_compose(host[sp], outs[sp][-1]) for sp in SPECIES})
        torch.set_num_threads(threads)
        cv2.setNumThreads(cv_threads)
        ms["run_plus_host_compose"].append(dt_run + dt)
        compose_ms.append(dt / FRAMES)
        t = 0.0
        for _ in range(a.steps):
            restore()
            dt, (h2d_c, d2h_c) = timed(lambda: pipe.run_split(split_jobs, labels=LABELS))
            t += dt
        ms["run_split"].append(t / a.steps)
        print(json.dumps({k: round(v[-1], 2) for k, v in ms.items()}), flush=True)
    same = all(np.array_equal(work[sp][k].numpy(), split_host[sp][k])
               for sp in SPECIES for k in (0, host[sp].shape[0] - 1))
    bytes_per_step = {"run": (h2d_a, d2h_a), "run_plus_host_compose": (h2d_a, d2h_a), "run_split": (h2d_c, d2h_c)}
    for name, v in ms.items():
        med = statistics.median(v)
        h2d, d2h = bytes_per_step[name]
        rec[name] = {"ms_per_step": [round(x, 2) for x in v], "median_ms_per_step": round(med, 2),
                     "gpix_s": round(px / (med * 1e-3) / 1e9, 2), "h2d_bytes_per_step": int(h2d),
                     "d2h_bytes_per_step": int(d2h), "d2h_bytes_per_px": round(d2h / px, 3)}
    rec["run_plus_host_compose"]["host_compose_ms_per_frame_one_thread"] = round(statistics.median(compose_ms), 2)
    rec["run_split_equals_host_route"] = bool(same)
    rec["fetch_probe"] = fetch_probe()
    print(json.dumps(rec), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fh:
        fh.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
