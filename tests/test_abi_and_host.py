"""CPU-side checks: the C-ABI library loads and exports every symbol include/bdepth.h declares (no compute
calls), the product path fails loudly without a GPU, and host-only logic (shard planning, BED handling in the
CLI) behaves.  No GPU needed."""
import ctypes as C
import os
import re
import subprocess

import pytest

import helpers
from helpers import GOLDEN, ROOT


def test_library_exports_every_declared_symbol():
    import sambamba_b200 as sb
    from sambamba_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "bdepth.h")).read()
    declared = set(re.findall(r"\b(bdepth_[a-z_0-9]+)\s*\(", hdr)) - {"bdepth_tile_cb", "bdepth_stat_cb"}
    L = C.CDLL(sb.lib_path())
    for name in sorted(declared):
        assert hasattr(L, name), f"libbdepth.so does not export {name}"
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)


def _no_gpu():
    import sambamba_b200 as sb
    return sb.load_library().bdepth_device_count() == 0


def test_no_cpu_fallback_without_gpu():
    if not _no_gpu():
        pytest.skip("a GPU is present")
    import sambamba_b200 as sb
    with pytest.raises(sb.BDepthError) as e:
        sb.BDepth(os.path.join(GOLDEN, "issue_193.bam"))
    assert e.value.code == -5 and "no CPU fallback" in e.value.msg
    rc, out, err = helpers.run_cli(["depth", "base", os.path.join(GOLDEN, "issue_193.bam")])
    assert rc == 1 and err.startswith(b"sambamba-depth: ") and b"no CPU fallback" in err


def test_product_sources_never_touch_the_oracle():
    for root, _, files in os.walk(os.path.join(ROOT, "sambamba_b200")):
        for f in files:
            if f.endswith((".cu", ".cuh", ".cpp", ".hpp", ".py", ".h", ".d")):
                txt = open(os.path.join(root, f), errors="ignore").read()
                assert "oracle/" not in txt and "liboracle" not in txt and "depth_oracle" not in txt, f
    assert "oracle" not in open(os.path.join(ROOT, "include", "bdepth.h")).read()


def test_cli_usage_and_argument_errors_need_no_gpu():
    rc, out, err = helpers.run_cli([])
    assert rc == 0 and b"Usage: sambamba-depth region|window|base" in err
    rc, out, err = helpers.run_cli(["depth", "frobnicate", "x.bam"])
    assert rc == 0 and b"Usage:" in err
    rc, out, err = helpers.run_cli(["depth", "region", "x.bam"])
    assert rc == 1 and b"BED file or a region must be provided in region mode" in err
    rc, out, err = helpers.run_cli(["depth", "window", "x.bam"])
    assert rc == 1 and b"positive window size must be specified" in err
    rc, out, err = helpers.run_cli(["depth", "window", "-w", "10", "--overlap", "10", "x.bam"])
    assert rc == 1 and b"specified overlap is larger than window size" in err
    rc, out, err = helpers.run_cli(["depth", "base", "/nonexistent/x.bam"])
    assert rc == 1 and b"Cannot open file" in err


def test_shard_plan_is_a_partition_at_record_starts(tmp_path):
    """bdepth_plan_shards is host-only: boundaries must be BAI linear-index record starts, increasing, and each
    must be the start of a record in the inflated stream."""
    import sambamba_b200 as sb
    p = helpers.gen_bam(str(tmp_path / "s.bam"), "-r", "chrA:900000", "-r", "chrB:600000", "-n", 60000, "-s", 3, "-t", 2)
    u = helpers.oracle_inflate(p)
    first, _ = helpers.header_first_record_offset(u)
    starts = {r[0] for r in helpers.parse_records(u, first)}
    # block table: compressed offset -> inflated offset
    raw = open(p, "rb").read()
    off, uoff, table = 0, 0, {}
    while off + 18 <= len(raw):
        bs = int.from_bytes(raw[off + 16:off + 18], "little") + 1
        isz = int.from_bytes(raw[off + bs - 4:off + bs], "little")
        if isz == 0:
            break
        table[off] = uoff
        uoff += isz
        off += bs
    for world in (2, 3, 4, 8):
        cuts = sb.plan_shards(p, world)
        assert len(cuts) == world - 1
        real = [c for c in cuts if c != 2 ** 64 - 1]
        assert real == sorted(real)
        for k, vo in enumerate(cuts, start=1):
            if vo == 2 ** 64 - 1:
                continue
            assert (vo >> 16) in table, "boundary must point at a BGZF block start"
            assert table[vo >> 16] + (vo & 0xFFFF) in starts, "boundary must be a record start"
            assert (vo >> 16) >= k * len(raw) // world - 70000


def test_region_chunk_plan_covers_every_overlapping_record(tmp_path):
    """bdepth_plan_region_chunks is host-only: every record that overlaps a region must start inside one of the planned
    virtual-offset ranges (a superset is fine -- the reference also only narrows by bins, randomaccessmanager.d:247-294),
    ranges are sorted, disjoint and begin at record starts; narrow queries must plan far less than the file."""
    import random
    import sambamba_b200 as sb
    p = helpers.gen_bam(str(tmp_path / "s.bam"), "-r", "chrA:2000000", "-r", "chrB:300", "-r", "chrC:700000", "-n", 150000, "-s", 5, "-t", 3)
    u = helpers.oracle_inflate(p)
    first, refs = helpers.header_first_record_offset(u)
    recs = helpers.parse_records(u, first)
    raw = open(p, "rb").read()
    off, uoff, blocks = 0, 0, []          # (inflated offset, file offset)
    while off + 18 <= len(raw):
        bs = int.from_bytes(raw[off + 16:off + 18], "little") + 1
        isz = int.from_bytes(raw[off + bs - 4:off + bs], "little")
        if isz == 0:
            break
        blocks.append((uoff, off))
        uoff += isz
        off += bs
    import bisect
    ustarts = [b[0] for b in blocks]

    def voffset(o):
        k = bisect.bisect_right(ustarts, o) - 1
        return (blocks[k][1] << 16) | (o - blocks[k][0])
    rec_vo = [voffset(r[0]) for r in recs]
    vo_set = set(rec_vo)
    rnd = random.Random(1)
    queries = [[(0, 1000, 1200)], [(2, 0, 700000)], [(0, 1999000, 2000000), (2, 10, 20)], [(1, 0, 300)],
               [(0, rnd.randrange(0, 1990000), 0) for _ in range(40)]]
    queries[-1] = sorted((r, s, s + rnd.randrange(1, 3000)) for r, s, _ in queries[-1])
    total_span = max(rec_vo) - min(rec_vo)
    for q in queries:
        chunks = sb.plan_region_chunks(p, q)
        assert chunks == sorted(chunks) and all(b < e for b, e in chunks)
        assert all(chunks[i][1] < chunks[i + 1][0] for i in range(len(chunks) - 1)), "ranges must be disjoint"
        assert all(b in vo_set for b, _ in chunks), "a range must begin at a record start"
        begs = [b for b, _ in chunks]
        for r, vo in zip(recs, rec_vo):
            _, ref, pos, _flag, _mq, _nc, span = r
            if ref < 0 or not any(ref == g[0] and pos < g[2] and pos + max(span, 1) > g[1] for g in q):
                continue
            k = bisect.bisect_right(begs, vo) - 1
            assert k >= 0 and chunks[k][0] <= vo < chunks[k][1], (q, r)
    small = sb.plan_region_chunks(p, [(0, 1000, 1200)])
    assert sum((e >> 16) - (b >> 16) for b, e in small) < 0.05 * (total_span >> 16)


def test_bench_reference_arm_prints_its_line(tmp_path):
    """`bench.py --impl reference` (the CPU arm the driver times beside the GPU one) on a small workload: one JSON line with
    the contract's keys, measured on a bounded sample that ends mid-stream (the oracle tolerates the cut only there)."""
    import json
    import subprocess
    import sys
    env = dict(os.environ, BDEPTH_BENCH_DIR=str(tmp_path))
    r = subprocess.run([sys.executable, os.path.join(helpers.ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--reads-per-unit", "60000", "--cpu-sample-mb", "2"], capture_output=True, text=True, env=env, timeout=600)
    assert r.returncode == 0, r.stderr[-400:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["unit"] == "GB/s" and line["gpu_launches"] == 0
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and "covered positions" in line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    sample_mb = float(line["cpu_baseline"]["sample"].split()[1])
    assert 0 < sample_mb <= 2.2, line["cpu_baseline"]["sample"]


def test_bench_own_arm_control_flow_under_the_emulation(tmp_path):
    """bench.py's own arm with the product library replaced by its CUDA-on-CPU emulation build (tests/run_bench_emul.py): warm-up, timed
    passes, the A/B legs, e2e, text rows and the verification against the oracle all run and the line carries the contract's keys.
    (What the numbers are is meaningless here; that the round-end launch cannot die of a Python error is the point.)"""
    import json
    import subprocess
    import sys
    env = dict(os.environ, BDEPTH_BENCH_DIR=str(tmp_path), BDEPTH_BENCH_UNIT_LEN="300000")
    r = subprocess.run([sys.executable, os.path.join(helpers.ROOT, "tests", "run_bench_emul.py"), "--reads-per-unit", "15000", "--steps", "1", "--warmup", "1", "--cpu-sample-mb", "1",
                        "--dump-outputs", str(tmp_path / "dump")], capture_output=True, text=True, env=env, timeout=900)
    assert r.returncode == 0, r.stderr[-600:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["verified"] is True and line["verification"]["checksum"] == line["verification"]["oracle_checksum"]
    # --dump-outputs: the counters of the last timed e2e step at the sampled positions (here all 300,000 of them) are the oracle's
    import numpy as np
    pos, counts = np.load(tmp_path / "dump" / "positions.npy"), np.load(tmp_path / "dump" / "counts.npy")
    assert pos.dtype == np.float64 and counts.dtype == np.float32 and counts.shape == (7, 300000) and np.array_equal(pos, np.arange(300000))
    want, _ = helpers.oracle_counts(str(next(tmp_path.glob("*.bam"))))
    assert counts.sum() > 0 and np.array_equal(counts, want)
    assert line["metric"] == "bam_gb_per_s_depth_base" and line["unit"] == "GB/s" and line["n_gpus"] == 1 and line["gpu_launches"] > 0
    assert set(line["roofline"]) >= {"bound", "achieved", "peak", "unit", "frac", "traffic"} and line["cpu_baseline"]["kind"] == "port"
    assert line["e2e"]["h2d_bytes_per_step"] > 0 and line["e2e"]["d2h_bytes_per_step"] == 300000 * 28
    assert all("error" not in v for k, v in line["ab"].items() if isinstance(v, dict)), line["ab"]
    assert line["text_rows"]["text_bytes"] > 0


def test_bench_verification_deadline():
    """The oracle leg runs under the launch's time budget: overrun -> None (the line is printed with "verified": null), errors propagate."""
    import time
    import bench
    saved = bench.BENCH_BUDGET_S
    try:
        bench.BENCH_BUDGET_S = 0.0
        t0 = time.time()
        assert bench.with_deadline(lambda: time.sleep(30)) is None and time.time() - t0 < 10
        bench.BENCH_BUDGET_S = 1e9
        assert bench.with_deadline(lambda: 42) == 42
        with pytest.raises(ZeroDivisionError):
            bench.with_deadline(lambda: 1 // 0)
    finally:
        bench.BENCH_BUDGET_S = saved
