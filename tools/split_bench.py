"""K9 split-compare compose against the torch slice copies it replaces, the host label route, and the server's split path.

    python tools/split_bench.py [--out profiles/split_bench.jsonl] [--iters 50]

One run measures, with the card name and power limit:
  - K9 (`split_compare_batch` on CUDA tensors) on 20 frames at 1080p and 4K, unlabelled and labelled, against the two
    strided torch copies + seam fill of the previous device path: CUDA events around `iters` calls after warm-up, as
    achieved GB/s at 6 B/px (3 read, 3 written; inputs and output exceed L2 at both sizes, so no flush is needed),
    beside a plain device-to-device copy of the same bytes in the same run and the measured copy peak of the B200
    (SURVEY.md: 6 545 GB/s);
    the K9 output is compared with the torch copies (unlabelled) and with the host route (labelled, one frame);
  - the host route per frame: CPU slice copies + draw_split_labels (cv2), single thread of this host;
  - the label table build (tables.split_label_stencil) at 1080p and 4K, uncached;
  - process_split_image for 16 concurrent 1080p requests (Dog): the default device batcher (K9 + K8) against a batcher
    whose runner returns host arrays (host compose, cv2 labels, cv2.imencode), alternated.
Appends one JSON line to --out."""
from __future__ import annotations

import argparse
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
from animal_vision_b200 import serving, tables  # noqa: E402
from animal_vision_b200.renderers.video import draw_split_labels, split_compare_batch  # noqa: E402

COPY_PEAK_GBS = 6545.0          # HBM copy peak measured on the B200 (SURVEY.md, MEASURED_PEAKS)
LABELS = ("Original", "Transformed")


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def torch_copies(a, b, out):
    """The device path before K9: two strided slice copies and the seam fill."""
    mid = a.shape[2] // 2
    out[:, :, :mid].copy_(a[:, :, :mid])
    out[:, :, mid:].copy_(b[:, :, mid:])
    out[:, :, mid:mid + 1] = 255
    return out


def time_ms(fn, iters):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def host_runner():
    dev = serving._device_runner()

    def run(key, batch):
        return dev(key, batch).cpu().numpy()           # species on the device, view back as pixels: the host composes
    return run


def serve_rate(fb, reqs, rounds):
    def one():
        ths = [threading.Thread(target=serving.process_split_image, args=(r, "dog", LABELS, fb)) for r in reqs]
        [t.start() for t in ths]
        [t.join() for t in ths]
    one()
    t0 = time.perf_counter()
    for _ in range(rounds):
        one()
    return len(reqs) * rounds / (time.perf_counter() - t0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "split_bench.jsonl"))
    ap.add_argument("--iters", type=int, default=50)
    a = ap.parse_args()
    rec = {"tool": "split_bench", "card": card(), "host_cores": os.cpu_count(), "copy_peak_gbs": COPY_PEAK_GBS,
           "frames": 20, "cases": []}
    for (h, w) in ((1080, 1920), (2160, 3840)):
        n = 20
        left = torch.from_numpy(np.stack([frames.natural(h, w, s % 4) for s in range(n)])).cuda()
        right = torch.flip(left, dims=(1, 2)).contiguous()
        out = torch.empty_like(left)
        nbytes = 6 * n * h * w
        c = {"shape": [h, w]}
        ref = torch_copies(left, right, torch.empty_like(left))
        split_compare_batch(left, right, out)
        c["k9_unlabelled_equals_torch_copies"] = bool(torch.equal(out, ref))
        split_compare_batch(left, right, out, labels=LABELS)
        host = draw_split_labels(ref[0].cpu().numpy().copy(), *LABELS)
        c["k9_labelled_equals_host_route"] = bool(np.array_equal(out[0].cpu().numpy(), host))
        for name, fn in (("dtod_copy", lambda: out.copy_(left)),
                         ("torch_copies", lambda: torch_copies(left, right, out)),
                         ("k9_unlabelled", lambda: split_compare_batch(left, right, out)),
                         ("k9_labelled", lambda: split_compare_batch(left, right, out, labels=LABELS))):
            ms = time_ms(fn, a.iters)
            gbs = nbytes / ms / 1e6
            c[name] = {"ms_per_20_frames": round(ms, 4), "gb_s_at_6_b_per_px": round(gbs, 1),
                       "frac_of_copy_peak": round(gbs / COPY_PEAK_GBS, 3)}
        hl, hr = left[:2].cpu(), right[:2].cpu()
        split_compare_batch(hl[:1], hr[:1])
        t0 = time.perf_counter()
        reps = 10
        for _ in range(reps):
            for k in range(2):
                draw_split_labels(split_compare_batch(hl[k:k + 1], hr[k:k + 1])[0].numpy(), *LABELS)
        c["host_compose_labels_ms_per_frame"] = round((time.perf_counter() - t0) * 1e3 / (2 * reps), 3)
        tables.split_label_stencil.cache_clear()
        t0 = time.perf_counter()
        st = tables.split_label_stencil(h, w, *LABELS)
        c["stencil_build_s"] = round(time.perf_counter() - t0, 3)
        c["stencil"] = {"band_rows": st.band_rows, "tables": int(st.luts.shape[0])}
        print(json.dumps(c), flush=True)
        rec["cases"].append(c)
        del left, right, out, ref
        torch.cuda.empty_cache()
    reqs = [cv2.imencode(".jpg", frames.natural(1080, 1920, s))[1].tobytes() for s in range(16)]
    dev_rates, host_rates = [], []
    with serving.FrameBatcher(max_batch=16, max_delay_ms=5.0) as fd, \
            serving.FrameBatcher(host_runner(), max_batch=16, max_delay_ms=5.0) as fh:
        same = serving.process_split_image(reqs[0], "dog", LABELS, fd) == serving.process_split_image(reqs[0], "dog", LABELS, fh)
        for _ in range(3):
            dev_rates.append(round(serve_rate(fd, reqs, 5), 2))
            host_rates.append(round(serve_rate(fh, reqs, 5), 2))
    rec["process_split_image_16x1080p_req_s"] = {"device_route": dev_rates, "host_route": host_rates,
                                                 "same_data_uri": same}
    print(json.dumps(rec["process_split_image_16x1080p_req_s"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "a") as fh_:
        fh_.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
