#!/usr/bin/env python
"""bench.py -- headline benchmark of the depth hot path (BASELINE.json metric: BAM GB/s for `depth base`).

  python bench.py --gpus N --steps K --warmup W            # our arm (libbdepth.so through the C ABI)
  python bench.py --impl reference --gpus N --steps K ...  # reference arm: the CPU implementation on host cores
  python bench.py ... --dump-outputs DIR                   # also write a seeded sample of the counters the last e2e step delivered
                                                           # (DIR/positions.npy, DIR/counts.npy; the sampling runs inside that step)

Workload (config.workload): BASELINE configs[1], the synthetic 30x chr20 BAM (64,444,167 bp, 12,888,833 x 150 bp
reads, seed 20, zlib level 6, 0xFF00-byte BGZF blocks) generated on the box by tools/bamgen.c.  At N > 1 GPUs
the input grows with N (N chromosomes of that size, weak scaling, the shape of BASELINE configs[3]) and is sharded
by BGZF virtual offset at BAI linear-index record starts; boundary counters are exchanged over NCCL.

A "step" is one complete `depth base` pass over the whole input:
  value  : input already resident in HBM  -> K1 inflate -> K2 scan -> K3 coverage (+ NCCL boundary exchange),
           timed with CUDA events on the library's stream (bdepth_stats.ms_span_device), max over ranks.
  e2e    : bdepth_open_memory() on the BAM image in PINNED HOST memory + bdepth_run_base(): H2D of the compressed
           bytes, all kernels, and D2H of the 7 x u32 per-position counters into pinned host memory, all inside
           the timed region (host wall clock around the call, which ends in a stream synchronize).
The file is 2.26 GB compressed / 3.76 GB inflated per chromosome unit, far larger than the 126 MB L2, so no L2
flush is needed between steps (config.l2: "inputs >> L2").
"""
import argparse
import datetime
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
if os.environ.get("BDEPTH_EMULATE") == "1":        # TEST INFRASTRUCTURE (run by hand: minutes even for a tiny workload): the bench logic on the CPU over the CUDA-on-CPU emulation of the library; never a benchmark
    import sambamba_b200._lib as _L
    _L.lib_path = lambda: os.path.join(ROOT, "tests", "emul", "libbdepth_emul.so")

READS_PER_UNIT = 12888833
UNIT_LEN = int(os.environ.get("BDEPTH_BENCH_UNIT_LEN", "64444167"))      # (the override is for tests/run_bench_emul.py: the CPU emulation cannot sweep 64 Mbp in a test's time)


def ncu_traffic(kernel_key):
    """roofline.traffic = dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel, parsed from the ncu
    summary profiles/CURRENT.json names for it (the capture of the shipped build; tools/ncu_summary.py wrote it)."""
    try:
        with open(os.path.join(ROOT, "profiles", "CURRENT.json")) as f:
            ent = json.load(f)[kernel_key]
        tot, inside = 0.0, False
        with open(os.path.join(ROOT, ent["summary"])) as f:
            for line in f:
                if line.startswith("== kernel:"):
                    inside = any(m in line for m in ent["kernel_match"])        # the K1 stage is two launches (k1_huff, k1_lz): their traffic adds
                elif inside and ("dram__bytes_read.sum" in line or "dram__bytes_write.sum" in line):
                    unit = line.split("[")[1].split("]")[0].lower()
                    v = float(line.rsplit("=", 1)[1].replace(",", ""))
                    tot += v * {"gbyte": 1e9, "mbyte": 1e6, "kbyte": 1e3, "byte": 1.0, "tbyte": 1e12}[unit]
                elif inside and line.startswith("== hottest"):
                    inside = False
        return (int(tot) if tot else None), ent["summary"]
    except Exception as e:                                    # no capture of this build yet: say so instead of quoting a stale one
        return None, f"none ({type(e).__name__})"


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs, copy bandwidth)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def workload_path(n_units, reads_per_unit):
    d = os.environ.get("BDEPTH_BENCH_DIR", "/tmp/bdepth_bench")
    os.makedirs(d, exist_ok=True)
    return os.path.join(d, f"synth_chr20x{n_units}_{reads_per_unit}" + ("" if UNIT_LEN == 64444167 else f"_len{UNIT_LEN}") + ".bam")


def ensure_workload(n_units, reads_per_unit, load=True):
    import __graft_entry__ as g
    g.build(quiet=True, load=load)          # load=False (reference arm): the product library is never mapped into that process
    path = workload_path(n_units, reads_per_unit)
    if os.path.exists(path) and os.path.exists(path + ".bai"):
        return path
    tmp = path + f".tmp{os.getpid()}"
    refs = []
    for i in range(n_units):
        refs += ["-r", (f"chr20:{UNIT_LEN}" if n_units == 1 else f"chr20_{i + 1}:{UNIT_LEN}")]
    cmd = [os.path.join(ROOT, "tools", "_build", "bamgen"), "-o", tmp, "-n", str(reads_per_unit * n_units), "-s", "20",
           "-t", str(min(64, os.cpu_count() or 8))] + refs
    subprocess.check_call(cmd, stderr=subprocess.DEVNULL)
    os.replace(tmp + ".bai", path + ".bai")
    os.replace(tmp, path)
    return path


GRCH38 = [248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422, 135086622, 133275309, 114364328,
          107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167, 46709983, 50818468, 156040895, 57227415]
WGS_SCALE = int(os.environ.get("BDEPTH_BENCH_WGS_SCALE", "10"))       # every chromosome at 1 / WGS_SCALE of its GRCh38 length, still 30x
WGS_READS = 620000000


def wgs_refs(scale=None):
    scale = scale or WGS_SCALE
    return [((f"chr{i + 1}" if i < 22 else ("chrX" if i == 22 else "chrY")), GRCH38[i] // scale) for i in range(24)]


def ensure_wgs(load=True):
    """BASELINE configs[2..4] input: the 24 GRCh38 primary chromosomes, 30x of 150 bp reads, seed 30 (SURVEY 8d) -- at 1 / WGS_SCALE
    linear scale: a full-size one is 108 GB of BAM, more than the box's 79 GB disk and ~10 minutes of generation per bench run.
    Every per-position ratio (reads per tile, bytes per position, blocks per Mbp) is that of the full genome; 62 M reads,
    10.8 GB of BAM, 18 GB inflated = three 6 GiB HBM batches, so the carry / tile-window / prefetch paths are all in the timing."""
    import __graft_entry__ as g
    g.build(quiet=True, load=load)
    d = os.environ.get("BDEPTH_BENCH_DIR", "/tmp/bdepth_bench")
    os.makedirs(d, exist_ok=True)
    n = WGS_READS // WGS_SCALE
    path = os.path.join(d, f"synth_wgs_div{WGS_SCALE}_{n}.bam")
    if os.path.exists(path) and os.path.exists(path + ".bai"):
        return path
    tmp = path + f".tmp{os.getpid()}"
    cmd = [os.path.join(ROOT, "tools", "_build", "bamgen"), "-o", tmp, "-n", str(n), "-s", "30", "-t", str(min(64, os.cpu_count() or 8))]
    for name, ln in wgs_refs():
        cmd += ["-r", f"{name}:{ln}"]
    subprocess.check_call(cmd, stderr=subprocess.DEVNULL)
    os.replace(tmp + ".bai", path + ".bai")
    os.replace(tmp, path)
    return path


def exome_bed(refs, n_total, seed=50):
    """SURVEY 8d C5: sorted, non-overlapping intervals, lengths ~ lognormal (median 150, clipped 50..2000), spread over the
    references in proportion to their length.  Returns an [n, 3] uint32 array (ref_id, start, end)."""
    import numpy as np
    rs = np.random.RandomState(seed)
    total = sum(l for _, l in refs)
    out = []
    for ri, (_, L) in enumerate(refs):
        k = max(1, int(round(n_total * L / total)))
        lens = np.clip(np.exp(rs.normal(np.log(150.0), 0.6, k)), 50, 2000).astype(np.int64)
        slack = L - int(lens.sum()) - k
        if slack <= 0:
            k = max(1, int(L // 4000)); lens = lens[:k]; slack = L - int(lens.sum()) - k
        gaps = np.diff(np.concatenate([[0], np.sort(rs.randint(0, slack + 1, k))])) + 1          # >= 1 between consecutive intervals
        starts = np.cumsum(gaps + np.concatenate([[0], lens[:-1]]))
        out.append(np.stack([np.full(k, ri, np.int64), starts, starts + lens], axis=1))
    return np.concatenate(out).astype(np.uint32)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx), "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def pinned_file(path):
    """Read a file into page-locked host memory (cudaHostAlloc through the runtime the library links)."""
    rt = C.CDLL("libcudart.so.12")
    n = os.path.getsize(path)
    p = C.c_void_p()
    rc = rt.cudaHostAlloc(C.byref(p), C.c_size_t(n), 0)
    if rc:
        raise RuntimeError(f"cudaHostAlloc failed: {rc}")
    buf = (C.c_ubyte * n).from_address(p.value)
    with open(path, "rb") as f:
        got = f.readinto(buf)
    assert got == n
    import numpy as np
    return np.ctypeslib.as_array(buf), (rt, p)


def cpu_baseline(path, threads, sample_bytes):
    """The reference's algorithm on the host cores (oracle port: zlib inflate on `threads` threads + the serial
    column sweep and per-base printer), on a bounded prefix of the same BAM.  kind = "port": the reference is D
    and cannot be compiled in this image."""
    exe = os.path.join(ROOT, "oracle", "_build", "depth_oracle")
    cmd = [exe, "--inflate-threads", str(threads)] + (["--max-file-bytes", str(sample_bytes)] if sample_bytes else []) + ["--stats", "depth", "base", path, "-o", "/dev/null"]
    t0 = time.time()
    r = subprocess.run(cmd, capture_output=True, text=True)
    dt = time.time() - t0
    if r.returncode != 0:
        raise RuntimeError(f"the CPU baseline failed (exit {r.returncode}): {r.stderr[-300:]}")
    st = {}
    for line in r.stderr.splitlines():
        if line.startswith("{"):
            st = json.loads(line)
    nbytes = st.get("file_bytes", sample_bytes or os.path.getsize(path))
    return {"value": nbytes / 1e9 / dt, "unit": "GB/s", "cores": threads, "kind": "port",
            "sample": f"{'first ' if sample_bytes else 'all '}{nbytes / 1e6:.0f} MB of the BAM ({st.get('columns', 0)} covered positions): inflate {st.get('t_inflate', 0):.2f} s on {threads} threads + serial pileup sweep/print {st.get('t_sweep', 0):.2f} s; wall {dt:.2f} s",
            "covered_mbases_per_s": st.get("columns", 0) / 1e6 / dt}, dt, nbytes, st


CK_A, CK_B = 0x9E3779B97F4A7C15, 0xC2B2AE3D27D4EB4F


def plane_checksums(planes, lin_start):
    """Order-sensitive checksum of a [7, n] block of counters whose first column is linear position lin_start: the sum over
    planes p and positions g of count * ((g * CK_A + (p + 1) * CK_B) | 1) modulo 2^64, the plain sum, and the number of
    covered positions.  All three add over disjoint tiles, so ranks (and tiles) can be summed in any order."""
    import numpy as np
    n = planes.shape[1]
    g = np.arange(lin_start, lin_start + n, dtype=np.uint64) * np.uint64(CK_A)
    ck, tot = 0, 0
    with np.errstate(over="ignore"):
        for p in range(7):
            c = planes[p].astype(np.uint64)
            w = (g + np.uint64(((p + 1) * CK_B) & 0xFFFFFFFFFFFFFFFF)) | np.uint64(1)
            ck = (ck + int((c * w).sum(dtype=np.uint64))) & 0xFFFFFFFFFFFFFFFF
            tot += int(c.sum(dtype=np.uint64))
    covered = int(np.count_nonzero(planes.sum(axis=0, dtype=np.uint64)))
    return ck, tot, covered


def checksum_run(h, lin0):
    """One more (untimed) bdepth_run_base whose tile callback folds every delivered tile into the checksums."""
    import numpy as np
    import sambamba_b200._lib as L
    acc = [0, 0, 0, 0]

    def cb(_user, tp):
        t = tp.contents
        src = np.ctypeslib.as_array(t.counts, shape=(6 * t.stride + t.len,))
        planes = np.stack([src[p * t.stride:p * t.stride + t.len] for p in range(7)])
        ck, tot, cov = plane_checksums(planes, int(lin0[t.ref_id]) + t.start)
        acc[0] = (acc[0] + ck) & 0xFFFFFFFFFFFFFFFF
        acc[1] += tot
        acc[2] += cov
        acc[3] += t.len
        return 0
    h._ck(h.L.bdepth_run_base(h.h, L.TILE_CB(cb), None))
    return acc


DUMP_POSITIONS = 1 << 20      # 8 + 7 x 4 bytes per position: 36 MiB of .npy files


def counter_sampler(lin0, seed=20):
    """A tile callback for bdepth_run_base that keeps the 7 counters of a fixed, seeded, sorted sample of linear positions
    (the same sample for every run on the same input).  Returns (positions, counts[7, n] float32, callback); positions
    another rank delivers stay zero."""
    import numpy as np
    import sambamba_b200._lib as L
    total = int(lin0[-1])
    pos = np.sort(np.random.default_rng(seed).choice(total, size=min(DUMP_POSITIONS, total), replace=False))
    counts = np.zeros((7, len(pos)), np.float32)         # counters stay far below 2^24: exact in float32

    def cb(_user, tp):
        t = tp.contents
        a = int(lin0[t.ref_id]) + t.start
        lo, hi = np.searchsorted(pos, (a, a + t.len))
        if hi > lo:
            src = np.ctypeslib.as_array(t.counts, shape=(6 * t.stride + t.len,))
            off = pos[lo:hi] - a
            for p in range(7):
                counts[p, lo:hi] = src[p * t.stride + off]
        return 0
    return pos, counts, L.TILE_CB(cb)


def oracle_checksums(path, threads):
    """The same three numbers from the CPU oracle's closed-form counters over the whole genome (test infrastructure; the
    only use of oracle/ in our arm is this check AFTER the timed region)."""
    import helpers
    want, st = helpers.oracle_counts(path, threads=threads)
    ck = tot = cov = 0
    step = 1 << 24
    for a0 in range(0, want.shape[1], step):
        c, t, v = plane_checksums(want[:, a0:a0 + step], a0)
        ck = (ck + c) & 0xFFFFFFFFFFFFFFFF
        tot += t
        cov += v
    return [ck, tot, cov, want.shape[1]], st


T_PROCESS_START = time.time()
# The driver gives one bench launch 870 s (SCALE_r01.json per_n_timeout_s).  The oracle's whole-file closed form is the one leg whose duration grows
# with N (about 30 s per chr20 unit on 64 host threads): it runs under a deadline, and a run that cannot finish the check in time still prints
# its line -- with "verified": null and the reason -- instead of being killed without one.
BENCH_BUDGET_S = float(os.environ.get("BDEPTH_BENCH_BUDGET_S", "780"))


def with_deadline(fn, reserve_s=45.0):
    """fn() on a worker thread (the oracle is a ctypes call: the GIL is released); None when the launch's time budget would be overrun."""
    import threading
    box = {}

    def work():
        try:
            box["r"] = fn()
        except BaseException as e:          # noqa: BLE001 -- re-raised on the caller's thread
            box["e"] = e
    t = threading.Thread(target=work, daemon=True)
    t.start()
    t.join(max(5.0, BENCH_BUDGET_S - (time.time() - T_PROCESS_START) - reserve_s))
    if t.is_alive():
        return None
    if "e" in box:
        raise box["e"]
    return box["r"]


def setup_dist(world, local_rank):
    if world <= 1:
        return None
    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(minutes=30))      # rank 0 checks the counters against the CPU oracle (minutes at N = 8) while the others wait in a collective
    return dist


def run_wgs_config(a, rank, world, local_rank):
    """BASELINE configs[2] (`depth window -w 1000`, 1 GPU), [3] (`depth base` sharded over 2/4/8 GPUs, one file: strong scaling) and
    [4] (`depth region -L exome.bed`, 8 GPUs) on the GRCh38-shaped 30x BAM.  Same JSON contract as the headline config."""
    import numpy as np
    refs = wgs_refs()
    lin0 = np.concatenate([[0], np.cumsum([l for _, l in refs])]).astype(np.int64)
    n_bed = max(1000, 200000 // WGS_SCALE)
    mode = {"window": "depth window -w 1000", "wgs-shard": "depth base", "exome": f"depth region -L exome.bed ({n_bed} intervals)"}[a.config]
    workload = (f"synthetic 30x whole-genome BAM, GRCh38 primary chromosomes at 1/{WGS_SCALE} length (BASELINE configs[{ {'window': 2, 'wgs-shard': 3, 'exome': 4}[a.config] }] shape): "
                f"24 references, {sum(l for _, l in refs):,} bp, {WGS_READS // WGS_SCALE:,} x 150 bp reads, seed 30, zlib-6 BGZF; `{mode}`, default filter"
                + (f"; BED: {n_bed} sorted intervals (200,000 x 1/{WGS_SCALE}: the interval density of the full-size case), lognormal lengths, seed 50" if a.config == "exome" else ""))
    config = {"workload": workload, "mode": mode, "filter": "mapping_quality > 0 and not duplicate and not failed_quality_control",
              "parallelism": f"bgzf-shard x{a.gpus} (one file, strong scaling)" if a.gpus > 1 else "single GPU", "l2": "inputs >> L2 (10.8 GB compressed, 18 GB inflated, three 6 GiB HBM batches)"}
    metric = {"window": "bam_gb_per_s_depth_window", "wgs-shard": "bam_gb_per_s_depth_base", "exome": "bam_gb_per_s_depth_region"}[a.config]
    bed = exome_bed(refs, n_bed) if a.config == "exome" else None

    # ------------------------------------------------------------------ reference arm (CPU port, bounded sample of the same command)
    if a.impl == "reference":
        if rank != 0:
            return 0
        path = ensure_wgs(load=False)
        threads = os.cpu_count() or 1
        exe = os.path.join(ROOT, "oracle", "_build", "depth_oracle")
        sample = a.cpu_sample_mb << 20
        extra = []
        if a.config == "exome":
            bp = path + f".exome{n_bed}.bed"
            with open(bp, "w") as f:
                f.write("".join(f"{refs[r][0]}\t{s}\t{e}\n" for r, s, e in bed.tolist()))
            extra = ["-L", bp]
        sub = {"window": ["depth", "window", "-w", "1000"], "wgs-shard": ["depth", "base"], "exome": ["depth", "region"] + extra}[a.config]
        times = []
        for i in range(a.warmup + a.steps):
            t0 = time.time()
            r = subprocess.run([exe, "--inflate-threads", str(threads), "--max-file-bytes", str(sample), "--stats"] + sub + [path, "-o", "/dev/null"], capture_output=True, text=True)
            if r.returncode != 0:
                raise RuntimeError(f"the CPU baseline failed (exit {r.returncode}): {r.stderr[-300:]}")
            if i >= a.warmup:
                times.append(time.time() - t0)
        dt = sum(times) / len(times)
        nb = min(sample, os.path.getsize(path))
        v = nb / 1e9 / dt
        cb = {"value": v, "unit": "GB/s", "cores": threads, "kind": "port", "sample": f"first {nb / 1e6:.0f} MB of the BAM, `{mode}` by the oracle port: zlib inflate on {threads} threads + serial sweep; wall {dt:.2f} s",
              "probe": {"sambamba": shutil.which("sambamba"), "ldc2": shutil.which("ldc2")}}
        print(json.dumps({"impl": "reference", "metric": metric, "value": v, "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt * 1e3,
                          "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": config, "cpu_baseline": cb,
                          "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return 0

    # ------------------------------------------------------------------ our arm
    import sambamba_b200 as sb
    dist = setup_dist(world, local_rank)
    if rank == 0:
        path = ensure_wgs()
    if dist is not None:
        dist.barrier()
    path = ensure_wgs()
    file_bytes = os.path.getsize(path)

    def barrier():
        if dist is not None:
            dist.barrier()

    def reduce(x, op):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    def fresh_uid():
        if dist is None:
            return None
        obj = [sb.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        return obj[0]

    def one_pass(h, collect=False):
        if a.config == "window":
            return h.run_windows(1000, 0, (1, 10, 30) if collect else (), collect="arrays" if collect else False)
        if a.config == "exome":
            return h.run_regions(bed, (1, 10, 30) if collect else (), collect="arrays" if collect else False)
        return h.run_base(collect=False)

    # ---- value: the (shard of the) compressed file resident in HBM
    b = sb.BDepth(path, device=local_rank)
    if world > 1:
        b.set_shard(rank, world, fresh_uid())
    b.stage()                # (with the shard resident a region query takes the plain path: sparse staging of the regions' BAI chunks is an H2D matter and is what `e2e` measures)
    for _ in range(a.warmup):
        barrier()
        one_pass(b) if a.config != "wgs-shard" else b.run_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    span, k1, k2, k3, ex, red, launches = [], [], [], [], [], [], 0
    barrier()
    for _ in range(a.steps):
        barrier()
        t0 = time.perf_counter()
        one_pass(b) if a.config != "wgs-shard" else b.run_resident()
        wall = (time.perf_counter() - t0) * 1e3
        st = b.stats()
        dev = st["ms_span_device"] + st["ms_reduce"]
        span.append(reduce(dev, "MAX"))
        k1.append(st["ms_inflate"]); k2.append(st["ms_scan"]); k3.append(st["ms_coverage"]); ex.append(st["ms_exchange"]); red.append(st["ms_reduce"])
        launches += st["gpu_launches"]
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    st = b.stats()
    ms_step = sum(span) / len(span)
    k1_ms = sum(k1) / len(k1)
    k1_bytes = st["cdata_bytes"] + st["inflated_bytes"]
    n_batches = st["n_batches"]
    staged_bytes = reduce(st["file_bytes"], "SUM")
    covered = reduce(st["covered_positions"], "SUM") if a.config == "wgs-shard" else None
    total_launches = reduce(launches, "SUM")
    b.close()

    # ---- e2e: pinned host BAM image in, results in host memory out, everything inside the timed region
    try:
        img, keep = pinned_file(path)
        host_kind = "pinned"
    except Exception:
        img, keep, host_kind = np.fromfile(path, dtype=np.uint8), None, "pageable (cudaHostAlloc of the whole image failed)"
    bai = np.fromfile(path + ".bai", dtype=np.uint8)
    h = sb.BDepth(memory=img, bai=bai, device=local_rank)
    if world > 1:
        h.set_shard(rank, world, fresh_uid())
    e2e_t, d2h_bytes, h2d_bytes = [], 0, 0
    n_w = max(1, min(a.warmup, 3))
    for i in range(n_w + a.steps):
        barrier()
        t0 = time.perf_counter()
        one_pass(h)
        dt = reduce(time.perf_counter() - t0, "MAX")
        s2 = h.stats()
        h2d_bytes = reduce(s2["file_bytes"], "SUM")
        d2h_bytes = reduce((s2["own_hi"] - s2["own_lo"]) * 28, "SUM") if a.config == "wgs-shard" else None
        if i >= n_w:
            e2e_t.append(dt)
    e2e_stats = h.stats()
    e2e_s = sum(e2e_t) / len(e2e_t)

    # ---- verification after the timed regions, against the CPU oracle's closed forms over the whole file
    verify = None
    if not a.no_verify:
        if a.config == "wgs-shard":
            mine = checksum_run(h, lin0)
            allv = [None] * world
            if dist is not None:
                dist.all_gather_object(allv, mine)
            else:
                allv = [mine]
            if rank == 0:
                got = [sum(v[0] for v in allv) & 0xFFFFFFFFFFFFFFFF, sum(v[1] for v in allv), sum(v[2] for v in allv), sum(v[3] for v in allv)]
                t0 = time.perf_counter()
                want, ost = oracle_checksums(path, min(64, os.cpu_count() or 8))
                verify = {"ok": got == want and got[2] == int(covered), "checksum": f"{got[0]:016x}", "oracle_checksum": f"{want[0]:016x}", "counts_total": got[1], "oracle_counts_total": want[1],
                          "covered_positions": got[2], "oracle_covered_positions": want[2], "positions_delivered": got[3], "oracle_seconds": time.perf_counter() - t0,
                          "what": "order-sensitive checksum of every rank's delivered counter tiles vs the CPU oracle's closed-form counters of the whole file"}
        else:
            rows = one_pass(h, collect=True)           # every rank holds the all-reduced table; rank 0 checks it
            if rank == 0:
                import helpers
                t0 = time.perf_counter()
                if a.config == "window":
                    sa = np.concatenate([lin0[r] + np.arange(0, (L // 1000) * 1000, 1000, dtype=np.int64) for r, (_, L) in enumerate(refs)]).astype(np.uint64)
                    sb_ = sa + np.uint64(1000)
                else:
                    sa = (lin0[bed[:, 0].astype(np.int64)] + bed[:, 1].astype(np.int64)).astype(np.uint64)
                    sb_ = (lin0[bed[:, 0].astype(np.int64)] + bed[:, 2].astype(np.int64)).astype(np.uint64)
                wr, wb, wc = helpers.oracle_segment_stats(path, sa, sb_, (1, 10, 30), threads=min(64, os.cpu_count() or 8))
                same_rows = len(rows["n_reads"]) == len(sa) and np.array_equal(lin0[rows["ref_id"]] + rows["start"], sa.astype(np.int64))
                ok_r = same_rows and np.array_equal(rows["n_reads"], wr)
                ok_b = same_rows and np.array_equal(rows["n_bases"], wb)
                ok_c = same_rows and np.array_equal(rows["cov_ge"].T, wc)
                verify = {"ok": bool(ok_r and ok_b and ok_c), "rows": int(len(sa)), "n_reads_equal": bool(ok_r), "n_bases_equal": bool(ok_b), "cov_ge_1_10_30_equal": bool(ok_c),
                          "sum_n_reads": int(rows["n_reads"].sum()), "sum_n_bases": int(rows["n_bases"].astype(np.uint64).sum()), "oracle_seconds": time.perf_counter() - t0,
                          "what": "readCount, n_bases and the positions with COV >= 1 / 10 / 30 of every row vs the CPU oracle's closed form (oracle_segment_stats, itself checked against the faithful sweep in tests/test_oracle_golden.py)"}
    h.close()
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    peak, peak_src = peaks()
    traffic, traffic_src = ncu_traffic("roofline")
    value = file_bytes / 1e9 / (ms_step / 1e3)
    out = {
        "metric": metric, "value": value, "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_step, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "u32", "data": "synthetic", "config": config,
        "covered_mbases_per_s": (covered / 1e6 / (ms_step / 1e3)) if covered is not None else None,
        "stage_ms": {"k1_inflate": k1_ms, "k2_scan": sum(k2) / len(k2), "k3_coverage": sum(k3) / len(k3), "nccl_exchange": sum(ex) / len(ex), "reduce": sum(red) / len(red), "hbm_batches": n_batches},
        "staged_bytes_per_step": int(staged_bytes),
        "e2e": {"value": file_bytes / 1e9 / e2e_s, "unit": "GB/s", "h2d_bytes_per_step": int(h2d_bytes), "d2h_bytes_per_step": int(d2h_bytes) if d2h_bytes is not None else "result table only",
                "ms_per_step": e2e_s * 1e3, "device_ms": {k: e2e_stats[k] for k in ("ms_h2d", "ms_inflate", "ms_scan", "ms_coverage", "ms_reduce", "ms_d2h", "ms_span_device")},
                "path": "bdepth_open_memory(pinned host BAM image) + " + {"window": "bdepth_run_windows", "wgs-shard": "bdepth_run_base", "exome": "bdepth_run_regions"}[a.config], "host_input": host_kind},
        "gpu_launches": int(total_launches),
        "roofline": {"kernel": "K1 two-phase inflate (k1_huff + k1_lz)", "bound": "hbm", "achieved": k1_bytes / 1e9 / (k1_ms / 1e3) if k1_ms else None, "peak": peak, "unit": "GB/s",
                     "frac": (k1_bytes / 1e9 / (k1_ms / 1e3) / peak) if k1_ms else None, "traffic": None, "traffic_source": "per-launch capture exists for the chr20 workload only (" + str(traffic_src) + ")",
                     "algorithmic_bytes_per_launch": int(k1_bytes / max(1, n_batches)), "launches_per_step": n_batches, "peak_source": peak_src,
                     "note": "C + U of this rank's shard / CUDA-event time of its K1 launches"},
        "clocks": clocks, "verified": (verify["ok"] if verify else None), "verification": verify,
    }
    if not a.no_cpu_baseline:
        exe = os.path.join(ROOT, "oracle", "_build", "depth_oracle")
        sample = a.cpu_sample_mb << 20
        sub = {"window": ["depth", "window", "-w", "1000"], "wgs-shard": ["depth", "base"], "exome": None}[a.config]
        if sub is not None:
            threads = os.cpu_count() or 1
            t0 = time.time()
            r = subprocess.run([exe, "--inflate-threads", str(threads), "--max-file-bytes", str(sample), "--stats"] + sub + [path, "-o", "/dev/null"], capture_output=True, text=True)
            dt = time.time() - t0
            if r.returncode != 0:
                raise RuntimeError(f"the CPU baseline failed (exit {r.returncode}): {r.stderr[-300:]}")
            out["cpu_baseline"] = {"value": min(sample, file_bytes) / 1e9 / dt, "unit": "GB/s", "cores": threads, "kind": "port",
                                   "sample": f"first {min(sample, file_bytes) / 1e6:.0f} MB of the BAM, `{mode}` by the oracle port; wall {dt:.2f} s"}
        else:
            out["cpu_baseline"] = {"value": None, "unit": "GB/s", "cores": os.cpu_count(), "kind": "port", "sample": "see `bench.py --impl reference --config exome` (needs the BED file on disk)"}
    print(json.dumps(out))
    if dist is not None:
        dist.destroy_process_group()
    if verify is not None and not verify["ok"]:
        sys.stderr.write("bench.py: VERIFICATION FAILED\n")
        return 3
    return 0


def main():
    if os.environ.get("BDEPTH_BENCH_WATCHDOG"):        # development aid: dump every thread's Python stack and exit if the run takes longer than this many seconds
        import faulthandler
        faulthandler.dump_traceback_later(int(os.environ["BDEPTH_BENCH_WATCHDOG"]), exit=True)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="chr20", choices=["chr20", "window", "wgs-shard", "exome"],
                    help="chr20: BASELINE configs[1] (headline; N > 1: N chromosomes, weak scaling).  window / wgs-shard / exome: configs[2] / [3] / [4] on the GRCh38-shaped 30x BAM")
    ap.add_argument("--reads-per-unit", type=int, default=READS_PER_UNIT, help="smaller values are for smoke tests only")
    ap.add_argument("--cpu-sample-mb", type=int, default=256)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-full-file", action="store_true", help="reference arm: skip the one whole-file run of the port")
    ap.add_argument("--no-verify", action="store_true", help="development only: skip the bit-exact check of the counters after the timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the counters the last timed end-to-end step delivered (a fixed, seeded sample of "
                    "positions) to DIR/positions.npy and DIR/counts.npy, so that two builds can be compared output for output")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "ours" or a.config != "chr20"):
        ap.error("--dump-outputs applies to the chr20 `depth base` workload of --impl ours")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.config != "chr20":
        return run_wgs_config(a, rank, world, local_rank)
    n_units = max(1, a.gpus)
    workload = (f"synthetic 30x chr20 BAM (BASELINE configs[1]): {n_units} x 64,444,167 bp, {a.reads_per_unit * n_units} x 150 bp reads, seed 20, "
                "zlib-6 BGZF 0xFF00 blocks; `depth base`, default filter")
    config = {"workload": workload, "mode": "depth base", "filter": "mapping_quality > 0 and not duplicate and not failed_quality_control",
              "parallelism": f"bgzf-shard x{a.gpus}" if a.gpus > 1 else "single GPU", "l2": "inputs >> L2 (2.3 GB compressed, 3.8 GB inflated per unit)"}

    # ------------------------------------------------------------------ reference arm (CPU)
    if a.impl == "reference":
        if rank != 0:
            return 0
        path = ensure_workload(n_units, a.reads_per_unit, load=False)
        threads = os.cpu_count() or 1
        probe = {"sambamba": shutil.which(os.environ.get("BDEPTH_SAMBAMBA", "sambamba")), "ldc2": shutil.which("ldc2")}
        times, nb = [], 0
        if probe["sambamba"]:
            # the real thing (BASELINE.md 3.1): `sambamba depth base -t $(nproc)` over the whole file; without -t it is serial (depth.d:1081,1154)
            nb = os.path.getsize(path)
            n_warm = min(a.warmup, 1)           # a whole-file run of the real thing takes most of a minute: at most one warm-up
            for i in range(n_warm + a.steps):
                t0 = time.time()
                r = subprocess.run([probe["sambamba"], "depth", "base", "-t", str(threads), path, "-o", "/dev/null"], capture_output=True, text=True)
                if r.returncode != 0:
                    raise RuntimeError(f"sambamba failed (exit {r.returncode}): {r.stderr[-300:]}")
                if i >= n_warm:
                    times.append(time.time() - t0)
            dt = sum(times) / len(times)
            cb = {"value": nb / 1e9 / dt, "unit": "GB/s", "cores": threads, "kind": "sambamba", "timed_runs": len(times),
                  "sample": f"whole file ({nb / 1e6:.0f} MB), {probe['sambamba']} depth base -t {threads}; {len(times)} timed runs"}
        else:
            for i in range(a.warmup + a.steps):
                cb, dt, nb, st = cpu_baseline(path, threads, a.cpu_sample_mb << 20)
                if i >= a.warmup:
                    times.append(dt)
            dt = sum(times) / len(times)
            if n_units == 1 and not a.no_full_file:
                # the bounded sample is a prefix; time the port over the WHOLE file once as well, so that the per-step number is not an extrapolation
                full, fdt, fnb, fst = cpu_baseline(path, threads, 0)
                cb["full_file"] = {"value": fnb / 1e9 / fdt, "unit": "GB/s", "seconds": fdt, "bytes": fnb, "covered_positions": fst.get("columns", 0)}
        v = nb / 1e9 / dt
        cb["value"] = v
        cb["probe"] = probe
        print(json.dumps({"impl": "reference", "metric": "bam_gb_per_s_depth_base", "value": v, "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                          "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
                          "config": config, "cpu_baseline": cb, "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "gpu_launches": 0}))
        return 0

    # ------------------------------------------------------------------ our arm
    import numpy as np
    import sambamba_b200 as sb
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(minutes=30))      # rank 0 checks the counters against the CPU oracle (minutes at N = 8) while the others wait in a collective
        if rank == 0:
            path = ensure_workload(n_units, a.reads_per_unit)
        dist.barrier()
        path = workload_path(n_units, a.reads_per_unit)
    else:
        path = ensure_workload(n_units, a.reads_per_unit)

    def fresh_uid():
        """A NCCL unique id can seed exactly one communicator: every handle gets its own (rank 0 creates, all receive)."""
        if dist is None:
            return None
        obj = [sb.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(obj, src=0)
        return obj[0]

    file_bytes = os.path.getsize(path)

    def barrier():
        if dist is not None:
            dist.barrier()

    def max_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x):
        if dist is None:
            return x
        import torch
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- value: inputs resident in HBM
    b = sb.BDepth(path, device=local_rank)
    if world > 1:
        b.set_shard(rank, world, fresh_uid())
    b.stage()
    for _ in range(a.warmup):
        barrier()
        b.run_resident()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    span, k1, k2, k3, ex, launches = [], [], [], [], [], 0
    barrier()
    for _ in range(a.steps):
        barrier()
        b.run_resident()
        st = b.stats()
        span.append(max_over_ranks(st["ms_span_device"]))
        k1.append(st["ms_inflate"]); k2.append(st["ms_scan"]); k3.append(st["ms_coverage"]); ex.append(st["ms_exchange"])
        launches += st["gpu_launches"]
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    st = b.stats()
    ms_step = sum(span) / len(span)
    covered = sum_over_ranks(st["covered_positions"])
    total_launches = sum_over_ranks(launches)
    k1_ms = sum(k1) / len(k1)
    k1_bytes = st["cdata_bytes"] + st["inflated_bytes"]              # C + U of this rank's shard (SURVEY 8d)
    k1_launches_per_step = st["n_batches"]
    # ---- A/B on the same resident handle (one GPU only; the library reads its switches at every run): kernels this build replaced,
    # measured beside the shipped ones so that a change made without access to a GPU shows its effect in the line the driver records
    ab = None
    if world == 1:
        ab = {"what": "stage times (ms) of 3 resident passes with one library switch each, same handle and input as `value`",
              "shipped": {"k1_inflate": k1_ms, "k3_coverage": sum(k3) / len(k3), "ms_per_step": ms_step}}
        for name, env in (("k1_lz_v12_literal_table", {"BDEPTH_K1LZ": "v12"}), ("k3_gather_round1", {"BDEPTH_K3": "gather"})):
            try:
                os.environ.update(env)
                b.run_resident()
                t = []
                for _ in range(3):
                    b.run_resident()
                    s3 = b.stats()
                    t.append((s3["ms_inflate"], s3["ms_coverage"], s3["ms_span_device"]))
                ab[name] = {"env": env, "k1_inflate": sum(x[0] for x in t) / 3, "k3_coverage": sum(x[1] for x in t) / 3, "ms_per_step": sum(x[2] for x in t) / 3}
            except Exception as e:                                  # an A/B leg must never take the bench line down
                ab[name] = {"env": env, "error": repr(e)[:200]}
            finally:
                for k in env:
                    os.environ.pop(k, None)
    b.close()

    # ---- e2e: host (pinned) buffers in, host (pinned) counters out, everything inside the timed region
    try:
        img, keep = pinned_file(path)
        host_kind = "pinned"
    except Exception:                                                 # N ranks pin N copies of the whole image: fall back rather than die
        img, keep, host_kind = np.fromfile(path, dtype=np.uint8), None, "pageable (cudaHostAlloc of the whole image failed)"
    bai = np.fromfile(path + ".bai", dtype=np.uint8)
    e2e_t, d2h_bytes = [], 0
    t0 = time.perf_counter()
    h = sb.BDepth(memory=img, bai=bai, device=local_rank)          # session setup (BGZF index, header, buffers) is outside the steps
    if world > 1:
        h.set_shard(rank, world, fresh_uid())
    chunk_blocks = int(os.environ.get("BDEPTH_BENCH_CHUNK_BLOCKS", "0"))       # tuning sweep: BGZF blocks per H2D chunk = per K1 sub-launch = per sub-batch
    if chunk_blocks:
        h.set_tuning(0, chunk_blocks)
    open_s = time.perf_counter() - t0
    cold_s = None
    n_w = max(1, min(a.warmup, 3))
    if a.dump_outputs:
        lin0 = np.concatenate([[0], np.cumsum([l for _, l in h.refs])]).astype(np.int64)
        dump_pos, dump_counts, dump_cb = counter_sampler(lin0)
    for i in range(n_w + a.steps):
        barrier()
        t0 = time.perf_counter()
        if a.dump_outputs and i == n_w + a.steps - 1:
            h._ck(h.L.bdepth_run_base(h.h, dump_cb, None))          # the last step hands its counters to the sampler
        else:
            h.run_base(collect=False)                               # H2D of the compressed bytes + kernels + D2H of the counters
        dt = time.perf_counter() - t0
        s2 = h.stats()
        d2h_bytes = (s2["own_hi"] - s2["own_lo"]) * 28
        dt = max_over_ranks(dt)
        if i == 0:
            cold_s = dt + max_over_ranks(open_s)
        if i >= n_w:
            e2e_t.append(dt)
    e2e_stats = h.stats()
    if a.dump_outputs:
        if dist is not None:                                        # ranks deliver disjoint positions: their samples add up
            parts = [None] * world
            dist.all_gather_object(parts, dump_counts)
            dump_counts = sum(parts)
        if rank == 0:
            os.makedirs(a.dump_outputs, exist_ok=True)
            np.save(os.path.join(a.dump_outputs, "positions.npy"), dump_pos.astype(np.float64))
            np.save(os.path.join(a.dump_outputs, "counts.npy"), dump_counts)
    # ---- rows of `depth base` formatted on the GPU (SURVEY 8d: "text formatting timed as its own line"): the same pass,
    # delivered as the text PerBasePrinter would print instead of counter planes (single GPU only; host wall clock)
    text = None
    if world == 1:
        tt, tbytes = [], 0
        for i in range(2):
            box = {"n": 0}

            def text_sink(_u, _p, n, box=box):
                box["n"] += n
                return 0
            t0 = time.perf_counter()
            h._ck(h.L.bdepth_run_base_text(h.h, C.byref(sb._lib.TextOpts(1.0, 1e50, 0)), sb._lib.TEXT_CB(text_sink), None))
            dt = time.perf_counter() - t0
            if i:
                tt.append(dt)
                tbytes = box["n"]
        text = {"ms_per_step": 1e3 * sum(tt) / len(tt), "text_bytes": tbytes, "text_gb_per_s": tbytes / 1e9 / (sum(tt) / len(tt)), "bam_gb_per_s": file_bytes / 1e9 / (sum(tt) / len(tt)),
                "path": "bdepth_run_base_text: H2D + kernels + k_text_len/scan/write + D2H of the row text (default `depth base`, min coverage 1)"}
    # ---- verification AFTER the timed regions: the counters this very session delivers (every rank's owned tiles) against the
    # CPU oracle over the whole input -- order-sensitive checksum, total count, covered positions, positions delivered
    verify, abandoned = None, False
    if not a.no_verify:
        lin0 = np.concatenate([[0], np.cumsum([l for _, l in h.refs])]).astype(np.int64)
        mine = checksum_run(h, lin0)
        if dist is not None:
            allv = [None] * world
            dist.all_gather_object(allv, mine)
        else:
            allv = [mine]
        if rank == 0:
            got = [sum(v[0] for v in allv) & 0xFFFFFFFFFFFFFFFF, sum(v[1] for v in allv), sum(v[2] for v in allv), sum(v[3] for v in allv)]
            t0 = time.perf_counter()
            try:
                res = with_deadline(lambda: oracle_checksums(path, min(64, os.cpu_count() or 8)))
            except Exception as e:            # the checker itself failed (host memory, ...): the measured line is still printed, unverified, with the reason
                res = e
            if isinstance(res, Exception):
                verify = {"ok": None, "skipped": "the CPU oracle failed: " + repr(res)[:300], "checksum": f"{got[0]:016x}", "counts_total": got[1], "covered_positions": got[2], "positions_delivered": got[3]}
            elif res is None:
                abandoned = True
                verify = {"ok": None, "skipped": f"the CPU oracle did not finish the whole-file closed form inside this launch's {BENCH_BUDGET_S:.0f} s budget (BDEPTH_BENCH_BUDGET_S)",
                          "checksum": f"{got[0]:016x}", "counts_total": got[1], "covered_positions": got[2], "positions_delivered": got[3]}
            else:
                want, ost = res
                verify = {"ok": got == want and got[2] == int(covered), "checksum": f"{got[0]:016x}", "oracle_checksum": f"{want[0]:016x}", "counts_total": got[1], "oracle_counts_total": want[1],
                      "covered_positions": got[2], "oracle_covered_positions": want[2], "positions_delivered": got[3], "oracle_seconds": time.perf_counter() - t0,
                      "what": "sum over planes p, positions g of count*((g*A+(p+1)*B)|1) mod 2^64 over every rank's delivered tiles vs the CPU oracle's closed-form counters of the whole file"}
    h.close()
    e2e_s = sum(e2e_t) / len(e2e_t)
    h2d_total = file_bytes
    d2h_total = sum_over_ranks(d2h_bytes)

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0
    peak, peak_src = peaks()
    traffic, traffic_src = ncu_traffic("roofline")
    value = file_bytes / 1e9 / (ms_step / 1e3)
    out = {
        "metric": "bam_gb_per_s_depth_base", "value": value, "unit": "GB/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": config,
        "covered_mbases_per_s": covered / 1e6 / (ms_step / 1e3),
        "stage_ms": {"k1_inflate": k1_ms, "k2_scan": sum(k2) / len(k2), "k3_coverage": sum(k3) / len(k3), "nccl_exchange": sum(ex) / len(ex)},
        "e2e": {"value": file_bytes / 1e9 / e2e_s, "unit": "GB/s", "h2d_bytes_per_step": int(h2d_total), "d2h_bytes_per_step": int(d2h_total),
                "ms_per_step": e2e_s * 1e3, "covered_mbases_per_s": covered / 1e6 / e2e_s, "first_call_incl_open_ms": cold_s * 1e3,
                "device_ms": {k: e2e_stats[k] for k in ("ms_h2d", "ms_inflate", "ms_scan", "ms_coverage", "ms_d2h", "ms_span_device")},
                "path": "bdepth_open_memory(pinned host BAM image) + bdepth_run_base -> 7 x u32 counters in pinned host memory", "host_input": host_kind, "chunk_blocks": chunk_blocks or "default (6656)",
                "variants": {k: os.environ[k] for k in ("BDEPTH_K1_STREAM_WARPS", "BDEPTH_K1_LIT3", "BDEPTH_K3_PREFETCH") if k in os.environ}},
        "text_rows": text, "ab": ab,
        "gpu_launches": int(total_launches),
        "roofline": {"kernel": "K1 two-phase inflate: k1_huff (lane-per-BGZF-block Huffman phase) + k1_lz (warp-per-block LZ77 phase), timed together", "bound": "hbm", "achieved": k1_bytes / 1e9 / (k1_ms / 1e3), "peak": peak, "unit": "GB/s",
                     "frac": k1_bytes / 1e9 / (k1_ms / 1e3) / peak, "traffic": traffic if (a.gpus == 1 and a.reads_per_unit == READS_PER_UNIT) else None, "traffic_source": traffic_src,
                     "algorithmic_bytes_per_launch": int(k1_bytes / max(1, k1_launches_per_step)), "launches_per_step": k1_launches_per_step,
                     "peak_source": peak_src, "note": "C + U per pass (SURVEY 8d) / CUDA-event duration of the K1 launches (k1_huff + k1_lz + k1_fallback) on the library stream; phase 1 is instruction-latency bound, phase 2 issue bound, neither HBM bound"},
        "clocks": clocks,
        "verified": (verify["ok"] if verify else None), "verification": verify,
    }
    if not a.no_cpu_baseline:
        cb, _, _, _ = cpu_baseline(path, os.cpu_count() or 1, a.cpu_sample_mb << 20)
        out["cpu_baseline"] = cb
    print(json.dumps(out))
    sys.stdout.flush()
    if dist is not None:
        dist.destroy_process_group()
    if verify is not None and verify["ok"] is False:
        sys.stderr.write("bench.py: VERIFICATION FAILED: the counters differ from the CPU oracle's\n")
        return 3
    if abandoned:
        os._exit(0)          # the oracle's worker thread is still inside its C call
    return 0


if __name__ == "__main__":
    sys.dont_write_bytecode = True          # the bench leaves the tree it runs from untouched (no __pycache__ of the modules it imports)
    sys.exit(main())
