#!/usr/bin/env python
"""Differential fuzzer (TEST INFRASTRUCTURE): random coordinate-sorted BAM files through the product's host pipeline and kernels compiled
over the CUDA-on-CPU emulation (tests/emul/libbdepth_emul.so, tests/emul/sambamba-depth-emul) against the CPU oracle
(oracle/_build/depth_oracle, liboracle.so).  Needs no GPU; never touches libbdepth.so.

Every case: a random header (1-4 references, 0-3 samples), random reads (every CIGAR operation, clipping, insertions at the ends, skips,
unmapped and unplaced reads, duplicates / QC failures / secondary / supplementary reads, name-sharing pairs and triples that overlap,
random qualities), random BGZF member sizes and compression levels (stored, fixed and dynamic deflate blocks), then
  * the BAI the GPU builder writes, byte for byte against the oracle's IndexBuilder restatement,
  * the per-position counters of the C API with small batches / sub-batches (several HBM batches, carries, ghosts) against the
    oracle's closed form, without and with -m,
  * a handful of random `depth base|region|window` command lines, stdout and exit code against the oracle CLI.
A mismatch is kept under --keep (files + command line) and reported; exit code 1 if there was any.

    python tools/fuzz_emul.py --seed 1 --cases 200 [--keep /tmp/fuzz_fail]

Deliberately not generated (refused or documented, DESIGN.md 8): a CIGAR that begins with N AND ends in M/=/X (one that begins with N and ends
otherwise is generated in one case in six; region / window statistics of such files only on one rank, without -m and --overlap), reads that reach past the end of their reference, more than eight reads of one
name over one position under -m.
"""
import argparse
import os
import random
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
EMUL = os.environ.get("BDEPTH_FUZZ_EMUL", os.path.join(ROOT, "tests", "emul"))      # a snapshot of the built harness, so that a fuzz run survives rebuilds

import numpy as np      # noqa: E402

import helpers          # noqa: E402

LEGS = {}      # how many comparisons of each kind ran
TEXTS = {}     # ranks leg: the row text every rank delivered (rank -> bytes)
OPS = "MIDNSHP=X"
REF_CONSUMING = (0, 2, 3, 7, 8)
QUERY_CONSUMING = (0, 1, 4, 7, 8)


def rand_cigar(rng, max_span):
    """A valid CIGAR whose reference span is in [1, max_span]: [H][S] body [S][H], body starts and ends with M/=/X (or D in the middle)."""
    body = []
    n_body = rng.choice([1, 1, 1, 2, 3, 4, 6])
    span = 0
    for k in range(n_body):
        first, last = k == 0, k == n_body - 1
        if first or last:
            op = rng.choice([0, 0, 0, 7, 8])
        else:
            op = rng.choice([0, 0, 1, 2, 2, 3, 6, 7, 8, 1])
        if op == 3:
            ln = rng.choice([1, 5, 50, 400, 1500, 3000])
        elif op in (1, 6):
            ln = rng.randint(1, 6)
        elif op == 2:
            ln = rng.randint(1, 12)
        else:
            ln = rng.choice([1, 2, 3, rng.randint(1, 40), rng.randint(20, 151)])
        if op in REF_CONSUMING:
            if span + ln > max_span:
                ln = max_span - span
                if ln <= 0:
                    continue
            span += ln
        body.append((ln, op))
    # an insertion right after the first / before the last operation, and at the very ends (the reference's cursor skips them)
    if rng.random() < 0.1:
        body.insert(0, (rng.randint(1, 4), 1))
    if rng.random() < 0.1:
        body.append((rng.randint(1, 4), 1))
    if not any(op in (0, 7, 8) for _, op in body):
        body = [(max(1, min(max_span, 10)), 0)]
    # no leading N (deviation), and the first reference-consuming operation decides it
    while body and body[0][1] == 3:
        body.pop(0)
    pre, post = [], []
    if rng.random() < 0.25:
        pre.append((rng.randint(1, 20), 4))
    if rng.random() < 0.1:
        pre.insert(0, (rng.randint(1, 30), 5))
    if rng.random() < 0.25:
        post.append((rng.randint(1, 20), 4))
    if rng.random() < 0.1:
        post.append((rng.randint(1, 30), 5))
    cig = pre + body + post
    span = sum(l for l, op in cig if op in REF_CONSUMING)
    if span < 1 or span > max_span:
        cig = [(max(1, min(max_span, 30)), 0)]
    return cig


def rand_case(rng, d, idx, n_cohort=0):
    n_ref = rng.choice([1, 1, 2, 3, 4])
    refs = [("r%d" % i, rng.choice([60, 300, 1000, 5000, 20000, 40000, 70000])) for i in range(n_ref)]
    n_samp = rng.choice([0, 0, 1, 2, 3])
    if n_cohort:        # a cohort of more than 64 samples (region / window runs count them a group at a time)
        n_samp = n_cohort
    rg = [("g%d" % i, "S%d" % (i if rng.random() < 0.8 else 0)) for i in range(n_samp)] or None
    n_reads = rng.choice([0, 1, 5, 40, 200, 600, 1500])
    dense = rng.random() < 0.5
    reads, quals, tags = [], [], []
    names = 0
    placed = []
    for _ in range(n_reads):
        ref = rng.randrange(n_ref)
        L = refs[ref][1]
        if dense:
            pos = min(L - 1, int(abs(rng.gauss(L * 0.3, L * 0.05))))
        else:
            pos = rng.randrange(L)
        placed.append((ref, pos))
    placed.sort()
    pending_mates = []       # (ref, pos_min, name) to emit later as an overlapping same-name read
    out = []
    for ref, pos in placed:
        L = refs[ref][1]
        cig = rand_cigar(rng, L - pos)
        flag = 0
        r = rng.random()
        if r < 0.05:
            flag |= 0x400
        elif r < 0.10:
            flag |= 0x200
        elif r < 0.15:
            flag |= 0x100
        elif r < 0.20:
            flag |= 0x800
        if rng.random() < 0.5:
            flag |= 0x1 | (0x40 if rng.random() < 0.5 else 0x80)
        if rng.random() < 0.5:
            flag |= 0x10
        mapq = 0 if rng.random() < 0.08 else rng.randint(1, 60)
        if rng.random() < 0.03:
            flag |= 0x4                 # placed but unmapped
            if rng.random() < 0.5:
                cig = []
        name = "q%d" % names
        names += 1
        out.append([ref, pos, mapq, flag, cig, name])
        if rng.random() < 0.3:
            pending_mates.append((ref, pos, name, rng.choice([1, 1, 1, 2, 3, 1, 1, 12])))
    # same-name partners: placed a little to the right of their mate so that most overlap
    for ref, pos, name, k in pending_mates:
        L = refs[ref][1]
        x = pos
        for _ in range(k):
            if k > 3:                      # a chain of supplementary alignments: each a little further right
                x = min(L - 1, x + rng.randint(20, 70))
                p2 = x
            else:
                p2 = min(L - 1, pos + rng.choice([0, 0, 1, 5, 30, 80, 140, 300]))
            cig = rand_cigar(rng, L - p2)
            flag = 0x1 | 0x80 | (0x10 if rng.random() < 0.5 else 0)
            out.append([ref, p2, 0 if rng.random() < 0.05 else rng.randint(1, 60), flag, cig, name])
    out.sort(key=lambda r: (r[0], r[1]))
    # quirk 1 (one case in six): some reads begin with N -- never ending in M/=/X (the reference reads past the sequence there, the product
    # refuses the file); region / window statistics of such a case only on one rank, without -m and without --overlap (refused otherwise)
    lead_n = rng.random() < 0.17
    if lead_n:
        for r in out:
            cig = r[4]
            if not cig or rng.random() > 0.25:
                continue
            L = refs[r[0]][1]
            span = sum(l for l, op in cig if op in REF_CONSUMING)
            room = L - r[1] - span
            if room < 1:
                continue
            k = next(i for i, (l, op) in enumerate(cig) if op in REF_CONSUMING)
            if cig[k][1] == 3:
                continue
            lead = [(rng.randint(1, min(room, 40)), 3)]
            if room - lead[0][0] >= 1 and rng.random() < 0.2:                      # two leading N operations, something that consumes only the query in between
                lead += [(rng.randint(1, 3), 1), (rng.randint(1, min(room - lead[0][0], 10)), 3)]
            cig = cig[:k] + lead + cig[k:]
            if cig[-1][1] in (0, 7, 8):
                cig = cig + [rng.choice([(rng.randint(1, 5), 4), (rng.randint(1, 5), 5), (rng.randint(1, 3), 1), (rng.randint(1, 4), 6)])]
            r[4] = cig
    for _ in range(rng.choice([0, 0, 0, 3, 30])):                      # unplaced reads at the end of the file
        out.append([-1, -1, 0, 0x4, [], "u%d" % names])
        names += 1
    reads = []
    for ref, pos, mapq, flag, cig, name in out:
        lseq = sum(l for l, op in cig if op in QUERY_CONSUMING)
        if not cig:
            lseq = rng.choice([0, 10, 50])
        seq = "".join(rng.choice("ACGTACGTACGTACGTN") for _ in range(lseq))
        reads.append((ref, pos, mapq, flag, cig, seq, name))
        qmode = rng.random()
        if qmode < 0.6:
            quals.append([rng.randint(0, 45) for _ in range(lseq)])
        elif qmode < 0.8:
            quals.append([rng.choice([2, 37])] * lseq)
        else:
            quals.append([255] * lseq)
        t = b""
        if rng.random() < 0.3:
            t += b"NMC" + bytes([rng.randrange(10)])
        if rg:
            t += b"RGZ" + rng.choice(rg)[0].encode() + b"\0"
        if rng.random() < 0.2:
            t += b"XSZ" + b"x" * rng.randint(0, 40) + b"\0"
        tags.append(t)
    block = rng.choice([150, 400, 1000, 4000, 20000, 0xFF00])
    level = rng.choice([0, 1, 6, 6, 9])
    path = os.path.join(d, "c%d.bam" % idx)
    helpers.write_bam(path, refs, reads, rg=rg, block=block, level=level, quals=quals, tags=tags, bins="auto", index=False)
    return path, refs, reads, rg, lead_n


def emul_cli(args, env=None):
    r = subprocess.run([os.path.join(EMUL, "sambamba-depth-emul")] + list(args), capture_output=True, env=env, timeout=600)
    return r.returncode, r.stdout, r.stderr


def rand_region(rng, refs):
    name, L = rng.choice(refs)
    k = rng.random()
    if k < 0.3:
        return name
    a = rng.randrange(L)
    if k < 0.36:                           # region strings that hold no position, or reach past the reference's end
        return rng.choice(["%s:%d-%d" % (name, a + 2, a + 1), "%s:%d" % (name, L + 5), "%s:%d-%d" % (name, L + 1, L + 100), "%s:%d-%d" % (name, max(1, L - 5), L + 50), "%s:%d" % (name, a + 1)])
    b = min(L, a + rng.choice([1, 10, 100, 1000, 5000]))
    return "%s:%d-%d" % (name, a + 1, max(a + 1, b))


def rand_bed(rng, refs, path):
    lines = []
    for _ in range(rng.choice([1, 2, 5, 20, 60])):
        name, L = rng.choice(refs)
        a = rng.randrange(L)
        b = min(L, a + rng.choice([1, 10, 100, 1000, 5000]))
        if b <= a:
            b = a + 1
        extra = rng.choice(["", "\tg%d" % len(lines), "\tx\ty"])
        lines.append("%s\t%d\t%d%s" % (name, a, b, extra))
    if rng.random() < 0.2:
        lines.append("nope\t1\t5")
    if rng.random() < 0.5:
        lines.sort(key=lambda s: (s.split("\t")[0], int(s.split("\t")[1])))
    with open(path, "w") as f:
        f.write("\n".join(lines) + "\n")
    return path


def rand_commands(rng, path, refs, d, has_rg, mates_ok, base_only=False, many=False):
    cmds = []
    for _ in range(rng.choice([3, 5, 8])):
        mode = rng.choice(["base", "base", "region", "window"])
        a = [mode]
        if rng.random() < 0.3:
            a += ["-q", str(rng.choice([1, 10, 20, 30, 40, 46]))]
        if rng.random() < 0.25:
            a += ["-F", ""]
        if rng.random() < 0.3:
            a += ["-c", rng.choice(["0", "1", "2", "3.5", "10"])]
        if rng.random() < 0.15:
            a += ["-C", rng.choice(["1", "4", "9.5", "30"])]
        if rng.random() < 0.25:
            a += ["-a"]
        if has_rg and rng.random() < 0.3 or many and mode == "base":      # (depth base holds at most 64 samples' counters at once)
            a += ["--combined"]
        if mates_ok and not many and rng.random() < 0.35 and not (base_only and mode != "base"):      # (CIGARs that begin with N: region / window statistics only without -m ...
            a += ["-m"]
        if mode == "base":
            if rng.random() < 0.2:
                a += ["-z"]
            k = rng.random()
            if k < 0.25:
                a += ["-L", rand_region(rng, refs)]
            elif k < 0.45:
                a += ["-L", rand_bed(rng, refs, os.path.join(d, "b%d.bed" % len(cmds)))]
        elif mode == "region":
            a += ["-L", rand_region(rng, refs) if rng.random() < 0.4 else rand_bed(rng, refs, os.path.join(d, "b%d.bed" % len(cmds)))]
            for _ in range(rng.choice([0, 1, 3, 3, 20])):
                a += ["-T", str(rng.choice([0, 1, 2, 5, 10, 30]))]
        else:
            # (a reducer block per window costs ~2 ms under the emulation: keep the number of windows in the low thousands)
            tot = sum(l for _, l in refs)
            w = rng.choice([x for x in (1, 7, 100, 640, 1000, 5000, 100000) if tot // x <= 3000])
            a += ["-w", str(w)]
            if w > 1 and rng.random() < 0.4 and not base_only:                              # ... and only for windows that do not overlap)
                a += ["--overlap", str(rng.randrange(max(1, w - max(1, tot // 3000)) ))]
            for _ in range(rng.choice([0, 1, 2])):
                a += ["-T", str(rng.choice([0, 1, 2, 5, 10]))]
        cmds.append(a + [path])
    return cmds


def max_same_name_overlap(reads):
    """Largest number of placed reads of one name over one position (the -m walk holds at most eight; any read counts here, whatever
    the filter would say: an upper bound)."""
    by = {}
    for ref, pos, mapq, flag, cig, seq, name in reads:
        if ref < 0:
            continue
        span = sum(l for l, op in cig if op in REF_CONSUMING)
        by.setdefault((name, ref), []).append((pos, pos + span))
    worst = 1
    for v in by.values():
        ev = sorted([(a, 1) for a, b in v] + [(b, -1) for a, b in v], key=lambda e: (e[0], e[1]))
        n = 0
        for _, d in ev:
            n += d
            worst = max(worst, n)
    return worst


def run_ranks(world, path, fix, tuning, minq, combined, regions, window, text_cov=None):
    """`world` ranks as threads over the emulation's NCCL stand-in (as tests/test_gpu_multi.py does): every rank's owned counters, region rows
    and window rows."""
    import queue
    import threading
    import sambamba_b200 as sb
    uid = sb.nccl_unique_id()
    q = queue.Queue()

    def main(rank):
        try:
            with sb.BDepth(path, device=rank) as b:
                b.set_shard(rank, world, uid)
                if tuning:
                    b.set_tuning(*tuning)
                b.set_min_baseq(minq)
                if fix:
                    b.set_fix_mates(True)
                if combined:
                    b.set_combined(True)
                got = b.run_base()
                st = b.stats()
                lo, hi = st["own_lo"], st["own_hi"]
                rr = b.run_regions(regions, [1, 3]) if regions else None
                ww = b.run_windows(window[0], window[1], [2]) if window else None
                if text_cov is not None:
                    TEXTS[rank] = b.run_base_text(min_cov=text_cov)
                q.put((rank, "ok", lo, hi, np.asarray(got)[..., lo:hi].copy(), rr, ww))
        except Exception as e:
            q.put((rank, "err", 0, 0, repr(e)[:300], None, None))

    ts = [threading.Thread(target=main, args=(r,)) for r in range(world)]
    for t in ts:
        t.start()
    res = [q.get(timeout=900) for _ in range(world)]
    for t in ts:
        t.join(timeout=60)
    res.sort(key=lambda r: r[0])
    return res


def one_case(seed, idx, keep):
    rng = random.Random(seed * 1000003 + idx)
    d = tempfile.mkdtemp(prefix="bdfuzz_")
    fails = []

    def fail(what, detail=""):
        fails.append((what, detail))

    try:
        # a share of the cases is a cohort of 65..150 samples, drawn apart from rng: the other cases stay the ones earlier campaigns ran
        rc_ = random.Random("cohort%d:%d" % (seed, idx))
        n_cohort = rc_.randint(65, 150) if rc_.random() < 0.1 else 0
        path, refs, reads, rg, lead_n = rand_case(rng, d, idx, n_cohort)
        many = bool(rg) and len({s for _, s in rg}) > 64
        # ---- index: GPU builder (emulated) vs the oracle's IndexBuilder
        rc, out, err = emul_cli(["index", path])
        if rc != 0:
            fail("index rc", err.decode()[-300:])
            return fails, d
        want = helpers.oracle_build_bai(path)
        got = open(path + ".bai", "rb").read()
        if got != want:
            fail("index bytes", "len %d vs %d" % (len(got), len(want)))
        if rng.random() < 0.15:      # an index that exists but does not describe the file (the reference only checks that one exists)
            import struct
            with open(path + ".bai", "wb") as f:
                f.write(b"BAI\1" + struct.pack("<i", len(refs)) + b"".join(struct.pack("<ii", 0, 0) for _ in refs) + struct.pack("<Q", 0))
        # ---- counters through the C API with small batches
        import sambamba_b200 as sb
        tot = sum(l for _, l in refs)
        n_over = max_same_name_overlap(reads)
        mates_ok = n_over <= 8
        for fix in ([False, True] if mates_ok else [False]):
            tuning = rng.choice([None, (1 << 20, 1), (1 << 20, 3), (0, 2), (1 << 16, 1)])
            minq = rng.choice([0, 0, 13, 30])
            LEGS["counters"] = LEGS.get("counters", 0) + 1
            try:
                with sb.BDepth(path) as b:
                    if tuning:
                        b.set_tuning(*tuning)
                    b.set_min_baseq(minq)
                    if fix:
                        b.set_fix_mates(True)
                    if rg and rng.random() < 0.5 or (rg and len(b.samples) > 1):
                        b.set_combined(True)
                    got_c = b.run_base()
            except Exception as e:
                fail("run_base fix=%s tuning=%s" % (fix, tuning), repr(e)[:300])
                continue
            if fix:
                want_c, _ = helpers.oracle_counts_fix_mates(path, min_bq=minq)
            else:
                want_c, _ = helpers.oracle_counts(path, min_bq=minq)
            g = np.asarray(got_c).reshape(-1, tot)[:7] if tot else np.zeros((7, 0), np.uint32)
            if g.shape != want_c.shape or not np.array_equal(g, want_c):
                bad = np.argwhere(g != want_c)[:3].tolist() if g.shape == want_c.shape else "shape %s vs %s" % (g.shape, want_c.shape)
                fail("counters fix=%s tuning=%s minq=%d" % (fix, tuning, minq), str(bad))
        # ---- samples counted a group at a time: bdepth_set_samples_per_pass 1, 3 and 0 (as many as fit) give the same rows (the command
        # lines below hold the default against the oracle)
        if rg and 1 < len({s for _, s in rg}) <= 16 and rc_.random() < 0.5:      # (one pass per sample is for small sample counts: the cohorts run as many passes as they need in the command lines)
            LEGS["passes"] = LEGS.get("passes", 0) + 1
            tot = sum(l for _, l in refs)
            minq = rc_.choice([0, 20])
            outs = []
            for k in (1, 3, 0):
                try:
                    with sb.BDepth(path) as b:
                        b.set_samples_per_pass(k)
                        b.set_min_baseq(minq)
                        outs.append((b.run_regions([(i, 0, L) for i, (_, L) in enumerate(refs)], [1, 5]), b.run_windows(max(100, tot // 500), 0, [2])))
                except Exception as e:
                    outs.append(repr(e)[:200])
            if not outs[0] == outs[1] == outs[2]:
                fail("samples per pass 1 / 3 / 0 minq=%d" % minq, str([o if isinstance(o, str) else len(o[0]) for o in outs]))
        # ---- several ranks (threads): the owned counters tile the genome and equal the oracle's; region / window rows equal one rank's
        if len(reads) >= 40 and rng.random() < 0.5:
            world = rng.choice([2, 2, 3, 4])
            fix = mates_ok and rng.random() < 0.4
            tuning = rng.choice([None, None, (1 << 20, 1), (0, 2), (1 << 16, 1)])
            minq = rng.choice([0, 0, 20])
            regions = None
            if rng.random() < 0.6 and not lead_n:
                regions = []
                for _ in range(rng.choice([1, 3, 10])):
                    r = rng.randrange(len(refs))
                    a0 = rng.randrange(refs[r][1])
                    regions.append((r, a0, min(refs[r][1], a0 + rng.choice([1, 50, 500, 5000]))))
                regions.sort()
            window = None
            if rng.random() < 0.5 and not lead_n:
                w = rng.choice([x for x in (100, 640, 1000, 5000) if tot // x <= 2000] or [100000])
                window = (w, rng.choice([0, 0, w // 2 if tot // max(1, w // 2) <= 3000 else 0]))
            LEGS["ranks"] = LEGS.get("ranks", 0) + 1
            what = "ranks world=%d fix=%s tuning=%s minq=%d regions=%s window=%s" % (world, fix, tuning, minq, regions, window)
            try:
                with sb.BDepth(path) as b:
                    b.set_min_baseq(minq)
                    if fix:
                        b.set_fix_mates(True)
                    if rg:
                        b.set_combined(True)
                    one_r = b.run_regions(regions, [1, 3]) if regions else None
                    one_w = b.run_windows(window[0], window[1], [2]) if window else None
                # ... and the rows of `depth base` every rank formats for its own positions, concatenated in rank order, are the one-process output
                text_cov = rng.choice([None, 0.0, 1.0, 2.0])
                TEXTS.clear()
                res = run_ranks(world, path, fix, tuning, minq, bool(rg), regions, window, text_cov)
                want_c = (helpers.oracle_counts_fix_mates(path, min_bq=minq) if fix else helpers.oracle_counts(path, min_bq=minq))[0]
                got = np.zeros_like(want_c)
                prev_hi, bad = 0, None
                if fix and any(st_ != "ok" and "64 BGZF blocks past a shard boundary" in str(arr_) for _, st_, _, _, arr_, _, _ in res):
                    # a documented refusal (DESIGN.md 8) of the rank that owns the chain's leader; the others must have stopped with it (run_ranks
                    # waits for every rank: a rank left waiting in a collective would have been a timeout above)
                    LEGS["ranks_refused"] = LEGS.get("ranks_refused", 0) + 1
                    if not all(st_ != "ok" for _, st_, _, _, _, _, _ in res):
                        fail(what, "one rank refused, another delivered: " + str([(r_, st_) for r_, st_, _, _, _, _, _ in res]))
                    res = []
                    prev_hi = tot
                    got = want_c
                for rank, status, lo, hi, arr, rr, ww in res:
                    if status != "ok":
                        bad = "rank %d: %s" % (rank, arr)
                        break
                    if hi > lo:
                        if lo != prev_hi:
                            bad = "owned ranges do not tile: rank %d owns [%d, %d) after %d" % (rank, lo, hi, prev_hi)
                            break
                        got[:, lo:hi] = np.asarray(arr).reshape(-1, hi - lo)[:7]
                        prev_hi = hi
                    if rank == 0 and regions and rr != one_r:
                        bad = "region rows differ from one rank's"
                    if rank == 0 and window and ww != one_w:
                        bad = "window rows differ from one rank's"
                if bad is None and text_cov is not None and res:
                    a_ = ["base", "-c", "%g" % text_cov, "-q", str(minq)] + (["-m"] if fix else []) + (["--combined"] if rg else []) + [path]
                    rc2, o2, e2 = helpers.oracle_cli(a_)
                    got_t = b"".join(TEXTS.get(r_, b"") for r_ in range(world))
                    want_t = o2.split(b"\n", 1)[1] if b"\n" in o2 else b""
                    LEGS["ranks_text"] = LEGS.get("ranks_text", 0) + 1
                    if rc2 != 0 or got_t != want_t:
                        k = next((i for i in range(min(len(got_t), len(want_t))) if got_t[i] != want_t[i]), min(len(got_t), len(want_t)))
                        bad = "row text of the ranks (-c %g): first difference at byte %d: %r vs %r" % (text_cov, k, got_t[max(0, k - 60):k + 60], want_t[max(0, k - 60):k + 60])
                if bad is None and prev_hi != tot:
                    bad = "owned ranges end at %d of %d" % (prev_hi, tot)
                if bad is None and not np.array_equal(got, want_c):
                    bad = "counters: " + str(np.argwhere(got != want_c)[:3].tolist())
                if bad:
                    fail(what, bad)
            except Exception as e:
                import traceback
                fail(what, traceback.format_exc()[-600:])
        # ---- several BAM files in one run: the records dealt out to two or three files (same header), every command line must print what
        # the oracle prints for the one file (the N-way merge of coordinate-sorted files; no -m there: refused)
        if len(reads) >= 5 and rng.random() < 0.3:
            import struct
            u = helpers.oracle_inflate(path)
            first, _refs = helpers.header_first_record_offset(u)
            raw = u.tobytes()
            nf = rng.choice([2, 2, 3])
            parts = [[raw[:first]] for _ in range(nf)]
            o = first
            while o + 4 <= len(raw):
                bs = struct.unpack_from("<i", raw, o)[0]
                parts[rng.randrange(nf)].append(raw[o:o + 4 + bs])
                o += 4 + bs
            files = []
            for k in range(nf):
                f = os.path.join(d, "part%d.bam" % k)
                helpers.write_bgzf(f, b"".join(parts[k]), len(refs), block=rng.choice([300, 4000, 0xFF00]), level=rng.choice([1, 6]))
                if os.path.exists(f + ".bai"):
                    os.remove(f + ".bai")
                rc, out, err = emul_cli(["index", f])
                if rc != 0:
                    fail("multi index rc", err.decode()[-300:])
                files.append(f)
            for a in rand_commands(rng, path, refs, d, bool(rg), False, base_only=lead_n, many=many)[:3]:
                LEGS["multi"] = LEGS.get("multi", 0) + 1
                rc1, o1, e1 = emul_cli(["depth"] + a[:-1] + files)
                rc2, o2, e2 = helpers.oracle_cli(a)
                if rc1 != rc2 or o1 != o2:
                    k = next((i for i in range(min(len(o1), len(o2))) if o1[i] != o2[i]), min(len(o1), len(o2)))
                    fail("multi %d files: " % nf + " ".join(a), "rc %d vs %d; first difference at byte %d: %r vs %r; stderr %r / %r" % (rc1, rc2, k, o1[max(0, k - 60):k + 60], o2[max(0, k - 60):k + 60], e1[-200:], e2[-200:]))
        # ---- -F queries: the command line with a query on the whole file against the oracle with -F "" on the file reduced to the reads a
        # Python statement of the query keeps (the oracle knows no queries; method checked in tests/test_emul_filter.py)
        if len(reads) >= 5 and rng.random() < 0.3:
            import test_emul_filter as tef
            _, recs = tef.parse_all(helpers.oracle_inflate(path))
            qk = rng.randint(0, 60)
            sl = rng.choice([5, 40, 100])
            cands = [("mapping_quality >= %d" % qk, lambda r: r.mapq >= qk),
                     ("not (duplicate or failed_quality_control) and mapping_quality > %d" % (qk // 2), lambda r: not r.flag & 0x600 and r.mapq > qk // 2),
                     ("paired and first_of_pair or mapping_quality < %d" % qk, lambda r: bool(r.flag & 1 and r.flag & 0x40) or r.mapq < qk),
                     ("sequence_length >= %d and not secondary_alignment" % sl, lambda r: r.lseq >= sl and not r.flag & 0x100),
                     ("reverse_strand and not supplementary", lambda r: bool(r.flag & 0x10) and not r.flag & 0x800),
                     ("read_name =~ /^q[0-9]*[02468]$/", lambda r: len(r.name) >= 2 and r.name[:1] == b"q" and r.name[1:].isdigit() and r.name[-1:] in b"02468"),
                     ("ref_id == 0 and position >= %d" % (refs[0][1] // 3), lambda r: r.ref == 0 and r.pos >= refs[0][1] // 3)]
            qtxt, fn = rng.choice(cands)
            sub = helpers.subset_bam(path, os.path.join(d, "sub.bam"), [bool(fn(r)) for r in recs])
            for a in rand_commands(rng, path, refs, d, bool(rg), mates_ok, base_only=lead_n, many=many)[:3]:
                a = [x for i, x in enumerate(a) if not (x == "-F" or (i and a[i - 1] == "-F"))]
                LEGS["filter"] = LEGS.get("filter", 0) + 1
                rc1, o1, e1 = emul_cli(["depth"] + a[:-1] + ["-F", qtxt, path])
                rc2, o2, e2 = helpers.oracle_cli(a[:-1] + ["-F", "", sub])
                if rc1 != rc2 or o1 != o2:
                    k = next((i for i in range(min(len(o1), len(o2))) if o1[i] != o2[i]), min(len(o1), len(o2)))
                    fail("filter -F '%s': " % qtxt + " ".join(a), "rc %d vs %d; first difference at byte %d: %r vs %r; stderr %r / %r" % (rc1, rc2, k, o1[max(0, k - 60):k + 60], o2[max(0, k - 60):k + 60], e1[-200:], e2[-200:]))
        # ---- command lines
        for a in rand_commands(rng, path, refs, d, bool(rg), mates_ok, base_only=lead_n, many=many):
            LEGS["cli"] = LEGS.get("cli", 0) + 1
            rc1, o1, e1 = emul_cli(["depth"] + a)
            rc2, o2, e2 = helpers.oracle_cli(a)
            if rc1 != rc2 or o1 != o2:
                k = next((i for i in range(min(len(o1), len(o2))) if o1[i] != o2[i]), min(len(o1), len(o2)))
                fail("cli " + " ".join(a), "rc %d vs %d; first difference at byte %d: %r vs %r; stderr %r / %r" % (rc1, rc2, k, o1[max(0, k - 60):k + 60], o2[max(0, k - 60):k + 60], e1[-200:], e2[-200:]))
        return fails, d
    except Exception as e:
        import traceback
        fail("exception", traceback.format_exc()[-800:])
        return fails, d
    finally:
        if fails and keep:
            dst = os.path.join(keep, "seed%d_case%d" % (seed, idx))
            shutil.rmtree(dst, ignore_errors=True)
            shutil.copytree(d, dst)
            with open(os.path.join(dst, "FAILS.txt"), "w") as f:
                for w, det in fails:
                    f.write(w + "\n    " + det + "\n")
        shutil.rmtree(d, ignore_errors=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--cases", type=int, default=50)
    ap.add_argument("--first", type=int, default=0)
    ap.add_argument("--seconds", type=float, default=0, help="stop after this many seconds (0: run all cases)")
    ap.add_argument("--keep", default=None)
    a = ap.parse_args()
    import __graft_entry__ as g
    if "BDEPTH_FUZZ_EMUL" not in os.environ:
        g.build(quiet=True, load=False)          # oracle, emulation harness (and the product library, which this script never loads)
    import sambamba_b200._lib as L
    L.lib_path = lambda: os.path.join(EMUL, "libbdepth_emul.so")
    L._lib = None
    if a.keep:
        os.makedirs(a.keep, exist_ok=True)
    t0 = time.time()
    n_fail = n = 0
    for i in range(a.first, a.first + a.cases):
        fails, _ = one_case(a.seed, i, a.keep)
        n += 1
        if fails:
            n_fail += 1
            print("case %d (seed %d): %d mismatches" % (i, a.seed, len(fails)))
            for w, det in fails[:4]:
                print("   ", w, "\n       ", det[:600])
            sys.stdout.flush()
        if a.seconds and time.time() - t0 > a.seconds:
            break
    print("fuzz: %d cases, %d with mismatches, %.0f s; comparisons: %s" % (n, n_fail, time.time() - t0, LEGS))
    return 1 if n_fail else 0


if __name__ == "__main__":
    sys.exit(main())
