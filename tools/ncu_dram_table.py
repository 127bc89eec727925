#!/usr/bin/env python
"""Turn an .ncu-rep of `tools/prof_one.py <species> H W N` (ncu --set full) into profiles/ncu_dram_table.json:
the measured DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of every kernel, keyed by
the name bench.py's per-kernel timer uses, together with the launch shape it was measured at.  bench.py reports
`roofline.traffic` from this file only when the shape equals the benchmarked launch -- never from a constant.

    python tools/ncu_dram_table.py gpurun_out/x.ncu-rep FRAMES H W profiles/<summary file the numbers are kept in>
"""
import csv
import io
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# substring of the CUDA kernel name -> name used by AVB_TIMED / bench.py
NAMES = [("DogProducer", "k2_gauss_dichromat"), ("cat_warp_kernel", "k2_gauss_cat_warp"), ("center_zoom", "cat_center_zoom"),
         ("tcblur", "k2_tcblur"), ("frame_flags", "frame_flags"),
         ("uv_stats", "k3_uv_stats"), ("uv_hist", "k3_uv_hist"), ("uv_compact", "k3_uv_compact"), ("uv_map", "k3_uv_map"),
         ("uv_prep", "k3_uv_prep"), ("uv_scan", "k3_uv_scan"), ("uv_select", "k3_uv_select"), ("uv_fused", "k3_uv_fused"),
         ("streak_kernel", "k2_streak"), ("k1_contig", "k1_colorimetric")]
UNIT = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}
TIME = {"ns": 1e-3, "us": 1.0, "ms": 1e3, "s": 1e6, "nsecond": 1e-3, "usecond": 1.0, "msecond": 1e3, "second": 1e6}


def main():
    rep, frames, H, W, source = sys.argv[1], int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), sys.argv[5]
    out = subprocess.run(["ncu", "-i", rep, "--page", "raw", "--csv"], capture_output=True, text=True).stdout
    rows = list(csv.reader(io.StringIO(out)))
    hdr, units = rows[0], rows[1]
    ix = {h: i for i, h in enumerate(hdr)}
    best = {}
    for r in rows[2:]:
        kname = r[ix["Kernel Name"]]
        bench = next((b for sub, b in NAMES if sub in kname), None)
        if bench is None:
            continue

        def val(metric, table):
            i = ix[metric]
            return float(r[i].replace(",", "")) * table.get(units[i], 1.0)
        rd, wr = val("dram__bytes_read.sum", UNIT), val("dram__bytes_write.sum", UNIT)
        us = val("gpu__time_duration.sum", TIME)
        rec = {"bench_name": bench, "kernel": kname[:120], "frames": frames, "H": H, "W": W,
               "dram_bytes_read": rd, "dram_bytes_write": wr, "dram_bytes_per_launch": rd + wr,
               "dram_bytes_per_px": (rd + wr) / (frames * H * W), "ncu_us": us}
        # several launches of one kernel (fixup passes exit early): keep the longest = the real pass
        if bench not in best or us > best[bench]["ncu_us"]:
            best[bench] = rec
    tab = {"source": source, "how": "ncu --set full --clock-control none; dram__bytes_read.sum + dram__bytes_write.sum per launch",
           "kernels": sorted(best.values(), key=lambda d: d["bench_name"])}
    path = os.path.join(ROOT, "profiles", "ncu_dram_table.json")
    with open(path, "w") as fh:
        json.dump(tab, fh, indent=1)
    for k in tab["kernels"]:
        print(f"{k['bench_name']:22s} {k['dram_bytes_per_px']:6.2f} B/px  rd {k['dram_bytes_read'] / 1e6:8.1f} MB  wr {k['dram_bytes_write'] / 1e6:8.1f} MB  {k['ncu_us']:8.1f} us")
    print("wrote", path)


if __name__ == "__main__":
    main()
