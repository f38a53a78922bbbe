"""Per-sample region and window statistics for cohorts of more than 64 samples: the library counts the samples a group at a
time (bdepth_set_samples_per_pass) and delivers every row at the end.  The CLI over many per-sample files must print what the
oracle prints for ONE file holding their coordinate-sorted union under a header with every file's @RG lines (depth.d:1170-1181;
MultiBamReader)."""
import hashlib
import os
import random
import struct

import pytest

import helpers

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(1800)]

REFS = [("c1", 6000), ("c2", 3000), ("c3", 2000)]      # c3 never has reads: the window carry quirk (depth.d:1070-1076)
CIGARS = [[(50, 0)], [(20, 0), (3, 2), (30, 0)], [(25, 0), (100, 3), (25, 0)], [(10, 4), (40, 0)], [(20, 0), (2, 1), (28, 0)]]
BED = "c1\t100\t900\nc1\t800\t1200\nc1\t2000\t2600\nc2\t0\t3000\nc3\t10\t500\n"


def _reads(rnd, n, name, rgs):
    """n reads on c1 / c2; rgs: the RG ids to draw from (None in the list: a read without an RG tag)."""
    out, quals, tags = [], [], []
    for i in range(n):
        ref = 0 if rnd.random() < 0.75 else 1
        cig = rnd.choice(CIGARS)
        qlen = sum(l for l, op in cig if op in (0, 1, 4))
        pos = rnd.randrange(0, REFS[ref][1] - 300)
        flag = 0x400 if rnd.random() < 0.05 else 0
        out.append((ref, pos, rnd.choice((0, 20, 60, 60)), flag, cig, "".join(rnd.choice("ACGT") for _ in range(qlen)), f"{name}r{i}"))
        quals.append([rnd.randrange(5, 41) for _ in range(qlen)])
        rg = rnd.choice(rgs)
        tags.append(b"" if rg is None else b"RGZ" + rg.encode() + b"\0")
    order = sorted(range(n), key=lambda k: (out[k][0], out[k][1]))
    return [out[k] for k in order], [quals[k] for k in order], [tags[k] for k in order]


def _records(path):
    """(header bytes, [(ref (unplaced last), pos, raw record)]) of a BAM, records in file order."""
    u = helpers.oracle_inflate(path)
    first, _ = helpers.header_first_record_offset(u)
    b = u.tobytes()
    out, o = [], first
    while o + 4 <= len(b):
        bs = struct.unpack_from("<i", b, o)[0]
        if o + 4 + bs > len(b):
            break
        ref, pos = struct.unpack_from("<ii", b, o + 4)
        out.append(((ref if ref >= 0 else 1 << 30), pos, b[o:o + 4 + bs]))
        o += 4 + bs
    return b[:first], out


def _merge(paths, dst):
    """One file with the coordinate-sorted union of the files' records (stable: ties keep file order) behind the first file's header,
    whose @RG lines are replaced by every file's @RG lines in file order -- the order in which several inputs number their samples."""
    head, recs, rgs = None, [], []
    for fi, p in enumerate(paths):
        h, rr = _records(p)
        lt = struct.unpack_from("<i", h, 4)[0]
        rgs += [ln for ln in h[8:8 + lt].decode().split("\n") if ln.startswith("@RG")]
        head = head or h
        recs += [(a, b2, fi, i, raw) for i, (a, b2, raw) in enumerate(rr)]
    recs.sort(key=lambda t: t[:4])
    lt = struct.unpack_from("<i", head, 4)[0]
    text = "".join(ln + "\n" for ln in head[8:8 + lt].decode().split("\n") if ln and not ln.startswith("@RG")) + "".join(ln + "\n" for ln in rgs)
    n_ref = struct.unpack_from("<i", head, 8 + lt)[0]
    head = b"BAM\1" + struct.pack("<i", len(text)) + text.encode() + head[8 + lt:]
    return helpers.write_bgzf(dst, head + b"".join(t[4] for t in recs), n_ref)


def _cohort(d, n_files, shared_every):
    """n_files per-sample BAMs (ID f<k>, SM S<k>); every shared_every-th file reuses the sample name of the file before it; the last
    file also holds a few reads without an RG tag (sample 0, which another pass counts)."""
    rnd = random.Random(n_files)
    paths = []
    for f in range(n_files):
        sm = f"S{f - 1}" if shared_every and f % shared_every == shared_every - 1 else f"S{f}"
        rgs = [f"f{f}"] + ([None] if f == n_files - 1 else [])
        reads, quals, tags = _reads(rnd, 14, f"f{f}", rgs)
        paths.append(helpers.write_bam(str(d / f"s{f:03d}.bam"), REFS, reads, rg=[(f"f{f}", sm)], quals=quals, tags=tags))
    merged = _merge(paths, str(d / "merged.bam"))
    bed = d / "r.bed"
    bed.write_text(BED)
    return paths, merged, str(bed)


def _commands(bed):
    return [["region", "-L", bed, "-T", "3", "-T", "10"], ["region", "-L", bed, "-a", "-c", "2", "-C", "40"], ["region", "-L", bed, "-q", "20"],
            ["window", "-w", "500"], ["window", "-w", "300", "--overlap", "100", "-T", "5"], ["region", "-L", bed, "--combined"], ["window", "-w", "500", "--combined"]]


@pytest.mark.parametrize("n_files,shared_every,n_samples", [(65, 0, 65), (100, 10, 90), (130, 100, 129)])
def test_many_files_equal_the_merged_file(tmp_path, n_files, shared_every, n_samples):
    paths, merged, bed = _cohort(tmp_path, n_files, shared_every)
    for args in _commands(bed):
        rc1, out1, err1 = helpers.run_cli(args + paths)
        rc2, out2, err2 = helpers.oracle_cli(args + [merged])
        assert rc1 == 0 and rc2 == 0, (args, err1, err2)
        assert out1 == out2, args
        assert err1 == err2, args       # the "Processing reference #k" lines: references with reads in any pass
    import sambamba_b200 as sb
    with sb.BDepth(paths[0]) as h:
        for p in paths[1:]:
            h.add_input(p)
        assert len(h.samples) == n_samples
        h.run_regions([(0, 0, 6000), (1, 0, 3000)], [1])
        st = h.stats()
    ost = helpers.oracle_scan(merged)
    assert st["n_sample_passes"] == (n_samples + 63) // 64
    assert st["n_records"] == ost.n_records and st["n_records_pass"] == ost.n_pass


def _merged_rg_file(path, rgs, n=1500, seed=9, extra_tag=None):
    rnd = random.Random(seed)
    reads, quals, tags = _reads(rnd, n, "m", [i for i, _ in rgs] + [None])
    if extra_tag is not None:
        tags[n // 2] = extra_tag
    return helpers.write_bam(path, REFS, reads, rg=rgs, quals=quals, tags=tags)


def test_one_file_with_200_read_groups_over_150_samples(tmp_path):
    rgs = [(f"g{i}", f"P{i % 150}") for i in range(200)]       # P0..P49 have two read groups each
    path = _merged_rg_file(str(tmp_path / "m.bam"), rgs)
    bed = tmp_path / "r.bed"
    bed.write_text(BED)
    for args in _commands(str(bed)):
        rc1, out1, err1 = helpers.run_cli(args + [path])
        rc2, out2, err2 = helpers.oracle_cli(args + [path])
        assert rc1 == 0 and rc2 == 0, (args, err1, err2)
        assert out1 == out2 and err1 == err2, args
    bad = _merged_rg_file(str(tmp_path / "bad.bam"), rgs, extra_tag=b"RGZnot-in-header\0")
    for args in (["region", "-L", str(bed)], ["window", "-w", "500"]):
        rc, out, err = helpers.run_cli(args + [bad])
        assert rc == 1 and b"read group is not present in the header" in err, (args, err)


@pytest.fixture(scope="module")
def forty(tmp_path_factory):
    d = tmp_path_factory.mktemp("s40")
    return helpers.gen_bam(str(d / "s40.bam"), "-r", "c1:60000", "-r", "c2:3000", "-r", "c3:5000", "-r", "c4:4000", "-n", 4000, "-s", 3, "-t", 2, "--samples", 40)


def test_forced_passes_agree(forty):
    import sambamba_b200 as sb
    ost = helpers.oracle_scan(forty)
    regions = [(0, 100, 9000), (0, 30000, 31000), (1, 0, 3000), (3, 5, 4000)]
    results = []
    for k, passes in ((1, 40), (7, 6), (0, 1)):
        with sb.BDepth(forty) as h:
            assert len(h.samples) == 40
            h.set_samples_per_pass(k)
            reg = h.run_regions(regions, [1, 5])
            st = h.stats()
            has_r = [h.L.bdepth_ref_has_reads(h.h, i) for i in range(4)]
            win = h.run_windows(1000, 200, [2])
            stw = h.stats()
            has_w = [h.L.bdepth_ref_has_reads(h.h, i) for i in range(4)]
        assert st["n_sample_passes"] == passes and stw["n_sample_passes"] == passes
        assert stw["n_records"] == ost.n_records and stw["n_records_pass"] == ost.n_pass
        results.append((reg, has_r, win, has_w))
    assert results[0] == results[1] == results[2]
    assert len(results[0][0]) == len(regions) * 40


def test_refusals_name_the_limit(tmp_path):
    paths, merged, bed = _cohort(tmp_path, 65, 0)
    rc, out, err = helpers.run_cli(["base"] + paths)
    assert rc == 1 and b"at most 64" in err and b"--combined" in err, err
    rc, out, err = helpers.run_cli(["base", merged])
    assert rc == 1 and b"at most 64" in err, err
    rc, out, err = helpers.run_cli(["region", "-L", bed, "-m", merged])
    assert rc == 1 and b"fix-mate-overlaps" in err and b"at most 64 samples" in err, err
    import sambamba_b200 as sb
    rgs = [(f"g{i}", f"P{i}") for i in range(5)]
    small = _merged_rg_file(str(tmp_path / "five.bam"), rgs, n=200)
    with sb.BDepth(small) as h:
        h.set_samples_per_pass(2)
        h.set_fix_mates(True)
        with pytest.raises(sb.BDepthError, match="at most 2 samples"):
            h.run_regions([(0, 0, 6000)], [1])
        h.set_samples_per_pass(0)
        assert len(h.run_regions([(0, 0, 6000)], [1])) == 5      # every sample fits one pass: -m runs as before


def _rank_main(rank, world, path, uid, regions, q):
    try:
        import sambamba_b200 as sb
        with sb.BDepth(path, device=rank) as b:
            b.set_shard(rank, world, uid)
            rows = b.run_regions(regions, [2, 8])
            q.put((rank, "ok", rows, b.stats()))
    except Exception as e:  # pragma: no cover
        q.put((rank, "err", repr(e), None))


def test_100_samples_on_two_ranks(tmp_path):
    import sambamba_b200 as sb
    emulate = os.environ.get("BDEPTH_EMULATE") == "1"
    if not emulate and sb.load_library().bdepth_device_count() < 2:
        pytest.skip("needs 2 GPUs")
    path = helpers.gen_bam(str(tmp_path / "s100.bam"), "-r", "chrA:200000", "-r", "chrB:700", "-r", "chrC:150000", "-n", 20000, "-s", 11, "-t", 4, "--samples", 100)
    regions = [(0, 100, 9000), (0, 60000, 140000), (2, 5, 100000)]
    with sb.BDepth(path) as b:
        want = b.run_regions(regions, [2, 8])
        assert b.stats()["n_sample_passes"] == 2
    uid = sb.nccl_unique_id()
    if emulate:          # ranks are threads over the NCCL stand-in (tests/emul)
        import queue
        import threading
        q = queue.Queue()
        ts = [threading.Thread(target=_rank_main, args=(r, 2, path, uid, regions, q)) for r in range(2)]
    else:
        import multiprocessing as mp
        ctx = mp.get_context("spawn")
        q = ctx.Queue()
        ts = [ctx.Process(target=_rank_main, args=(r, 2, path, uid, regions, q)) for r in range(2)]
    for t in ts:
        t.start()
    res = sorted([q.get(timeout=1500) for _ in range(2)], key=lambda r: r[0])
    for t in ts:
        t.join(timeout=60)
    for r in res:
        assert r[1] == "ok", r
        assert r[2] == want          # the statistics are all-reduced: every rank holds the full table
        assert r[3]["n_sample_passes"] == 2


def test_bamgen_defaults_unchanged(tmp_path):
    """--samples / --sample leave the default output alone: the benchmark inputs stay what they were (inflated stream; the
    compressed bytes also depend on the zlib build)."""
    want = {"tiny": "1d83b870f6bffe5ed4c7d623cbf76dcb", "chr20": "96633ffe80d5c55c08bfe56970a22656"}
    a = helpers.gen_bam(str(tmp_path / "t.bam"), "--preset", "tiny")
    b = helpers.gen_bam(str(tmp_path / "c.bam"), "-r", "chr20:64444167", "-n", 20000, "-s", 7)
    got = {k: hashlib.md5(helpers.oracle_inflate(p).tobytes()).hexdigest() for k, p in (("tiny", a), ("chr20", b))}
    assert got == want
    k = helpers.gen_bam(str(tmp_path / "k.bam"), "--preset", "tiny", "--samples", 5)
    s = helpers.gen_bam(str(tmp_path / "s.bam"), "--preset", "tiny", "--sample", "NA12878")
    import sambamba_b200 as sb
    with sb.BDepth(k) as h:
        assert h.samples == ["S1", "S2", "S3", "S4", "S5"]
    with sb.BDepth(s) as h:
        assert h.samples == ["NA12878"]
