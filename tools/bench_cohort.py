#!/usr/bin/env python
"""bench_cohort.py -- per-sample `depth region` over cohorts of more than 64 samples, which the library counts a group of samples
at a time (bdepth_set_samples_per_pass).  Two inputs, generated with tools/bamgen.c from fixed seeds:

  cohort : --files per-sample BAMs (one @RG each, --sample S<k>) over chr20, read together as several inputs;
  merged : one BAM with --rgs read groups (bamgen --samples), every read's RG:Z drawn from the generator.

Each is timed over --steps region runs (after --warmup) through the C ABI: host wall clock around bdepth_run_regions, and the
library's CUDA-event times: device time per sample pass (ms_total_device / n_sample_passes) and K2 (ms_scan).  After the timed
runs every row is checked against the oracle: the cohort per file (oracle_segment_stats of that file = its sample's rows), the
merged file through the oracle CLI against this project's CLI, byte for byte.  Prints one JSON line; the GPU's name and power
limit are part of it.

  python tools/bench_cohort.py [--files 96] [--rgs 256] [--reads 200000] [--steps 3] [--warmup 1] [--json out.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import helpers  # noqa: E402
import sambamba_b200 as sb  # noqa: E402

CHR20 = 64444167


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = [x.strip() for x in out.split(",")]
        return {"gpu": name, "power_limit": power}
    except Exception as e:      # the numbers below are then without the card they were measured on: say so
        return {"gpu": None, "power_limit": None, "gpu_info_error": repr(e)}


def panel(n=2000, length=200, seed=5):
    rnd = np.random.default_rng(seed)
    starts = np.sort(rnd.choice(np.arange(0, CHR20 - length, length * 4), n, replace=False))
    return [(0, int(s), int(s) + length) for s in starts]


def timed(open_handle, regions, thr, steps, warmup):
    walls, dev, k2, passes = [], [], [], None
    rows = None
    for i in range(warmup + steps):
        with open_handle() as h:
            t0 = time.perf_counter()
            rows = h.run_regions(regions, thr)
            wall = (time.perf_counter() - t0) * 1e3
            st = h.stats()
        if i >= warmup:
            walls.append(wall); dev.append(st["ms_total_device"]); k2.append(st["ms_scan"]); passes = st["n_sample_passes"]
    return rows, {"n_sample_passes": passes, "host_wall_ms": float(np.median(walls)), "device_ms": float(np.median(dev)),
                  "device_ms_per_pass": float(np.median(dev)) / max(1, passes or 1), "k2_ms": float(np.median(k2)), "steps": steps}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--files", type=int, default=96)
    ap.add_argument("--rgs", type=int, default=256)
    ap.add_argument("--reads", type=int, default=200000, help="reads per cohort file; the merged file has files x reads")
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    regions, thr = panel(), [1, 10, 20]
    res = {"workload": {"cohort_files": a.files, "merged_read_groups": a.rgs, "reads_per_file": a.reads, "regions": len(regions), "thresholds": thr}}
    res.update(gpu_info())
    ok = True
    with tempfile.TemporaryDirectory() as d:
        paths = []
        for k in range(a.files):
            paths.append(helpers.gen_bam(os.path.join(d, f"s{k:03d}.bam"), "-r", f"chr20:{CHR20}", "-n", a.reads, "-s", 100 + k, "-t", 8, "--sample", f"S{k:03d}"))
        merged = helpers.gen_bam(os.path.join(d, "merged.bam"), "-r", f"chr20:{CHR20}", "-n", a.reads * a.files, "-s", 7, "-t", 8, "--samples", a.rgs)

        def open_cohort():
            h = sb.BDepth(paths[0])
            for p in paths[1:]:
                h.add_input(p)
            return h
        rows, res["cohort"] = timed(open_cohort, regions, thr, a.steps, a.warmup)
        # verification (outside the timed runs): sample k's rows are what the oracle computes for file k alone
        got = {}
        for r in rows:      # (ref_id, start, end, n_reads, n_bases, cov_ge, sample_id), regions outer, samples inner
            got.setdefault(r[6], []).append(r)
        seg_a = np.array([s for _, s, _ in regions], np.uint64); seg_b = np.array([e for _, _, e in regions], np.uint64)
        bad = 0
        for k, p in enumerate(paths):
            want_r, want_b, want_c = helpers.oracle_segment_stats(p, seg_a, seg_b, thr)
            mine = got.get(k, [])
            if len(mine) != len(regions) or any((m[3], m[4], list(m[5])) != (int(want_r[i]), int(want_b[i]), [int(x) for x in want_c[:, i]]) for i, m in enumerate(mine)):
                bad += 1
        res["cohort"]["files_differing"] = bad
        ok &= bad == 0

        rows_m, res["merged"] = timed(lambda: sb.BDepth(merged), regions, thr, a.steps, a.warmup)
        bed = os.path.join(d, "panel.bed")
        with open(bed, "w") as f:
            f.writelines(f"chr20\t{s}\t{e}\n" for _, s, e in regions)
        args = ["region", "-L", bed] + sum((["-T", str(t)] for t in thr), [])
        rc1, out1, err1 = helpers.run_cli(args + [merged])
        rc2, out2, err2 = helpers.oracle_cli(args + [merged])
        res["merged"]["cli_equals_oracle"] = rc1 == 0 and rc2 == 0 and out1 == out2
        res["merged"]["rows"] = len(rows_m)
        ok &= res["merged"]["cli_equals_oracle"] and len(rows_m) == len(regions) * a.rgs
    res["verified"] = bool(ok)
    line = json.dumps(res)
    print(line)
    if a.json:
        with open(a.json, "w") as f:
            f.write(line + "\n")
    return 0 if ok else 1


if __name__ == "__main__":
    sys.exit(main())
