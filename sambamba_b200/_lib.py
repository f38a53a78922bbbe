"""ctypes binding of libbdepth.so.  Fails loudly if the CUDA library is missing: there is no
CPU fallback anywhere in the product path."""
import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))


def lib_path():
    return os.path.join(_HERE, "_build", "libbdepth.so")


class BDepthError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"bdepth error {code}: {msg}")
        self.code = code
        self.msg = msg


class Region(C.Structure):
    _fields_ = [("ref_id", C.c_uint32), ("start", C.c_uint32), ("end", C.c_uint32)]


class Tile(C.Structure):
    _fields_ = [("ref_id", C.c_int32), ("start", C.c_uint32), ("len", C.c_uint32), ("stride", C.c_uint32),
                ("counts", C.POINTER(C.c_uint32)), ("n_samples", C.c_uint32), ("sample_stride", C.c_uint32)]


class RegionStat(C.Structure):
    _fields_ = [("ref_id", C.c_int32), ("start", C.c_uint32), ("end", C.c_uint32), ("n_reads", C.c_uint32),
                ("n_bases", C.c_uint32), ("cov_ge", C.POINTER(C.c_uint32)), ("sample_id", C.c_int32)]


class Stats(C.Structure):
    _fields_ = [(n, C.c_uint64) for n in ("file_bytes", "n_blocks", "cdata_bytes", "inflated_bytes", "n_records",
                                          "n_records_pass", "n_cigar_ops", "seq_bytes", "positions",
                                          "covered_positions", "long_reads", "chain_fixups")] + \
               [("gpu_launches", C.c_uint32), ("n_batches", C.c_uint32)] + \
               [(n, C.c_float) for n in ("ms_h2d", "ms_inflate", "ms_scan", "ms_coverage", "ms_reduce", "ms_d2h",
                                         "ms_total_device")] + [("host_wall_ms", C.c_double), ("ms_span_device", C.c_float), ("ms_exchange", C.c_float),
                                                                 ("own_lo", C.c_uint64), ("own_hi", C.c_uint64), ("halo_bytes_sent", C.c_uint64),
                                                                 ("mate_pairs", C.c_uint64), ("mate_pair_columns", C.c_uint64), ("mate_groups", C.c_uint64), ("ms_mates", C.c_float),
                                                                 ("n_sample_passes", C.c_uint32)]

    def as_dict(self):
        return {n: getattr(self, n) for n, _ in self._fields_}


class TextOpts(C.Structure):
    _fields_ = [("min_cov", C.c_double), ("max_cov", C.c_double), ("annotate", C.c_int)]


TEXT_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_size_t)
TILE_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(Tile))
STAT_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.POINTER(RegionStat), C.c_uint64)

_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    p = lib_path()
    if not os.path.exists(p):
        raise ImportError(f"{p} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    L = C.CDLL(p)
    vp = C.c_void_p
    L.bdepth_device_count.restype = C.c_int
    L.bdepth_open.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
    L.bdepth_open_lazy.argtypes = [C.c_char_p, C.c_int, C.POINTER(vp)]
    L.bdepth_open_memory.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.c_int, C.POINTER(vp)]
    L.bdepth_add_input.argtypes = [vp, C.c_char_p]
    L.bdepth_close.argtypes = [vp]
    L.bdepth_close.restype = None
    L.bdepth_last_error.argtypes = [vp]
    L.bdepth_last_error.restype = C.c_char_p
    L.bdepth_n_ref.argtypes = [vp]
    L.bdepth_ref_name.argtypes = [vp, C.c_int]
    L.bdepth_ref_name.restype = C.c_char_p
    L.bdepth_ref_length.argtypes = [vp, C.c_int]
    L.bdepth_ref_length.restype = C.c_uint32
    L.bdepth_header_text.argtypes = [vp, C.POINTER(C.c_size_t)]
    L.bdepth_header_text.restype = C.c_char_p
    L.bdepth_is_coordinate_sorted.argtypes = [vp]
    L.bdepth_has_index.argtypes = [vp]
    L.bdepth_n_samples.argtypes = [vp]
    L.bdepth_sample_name.argtypes = [vp, C.c_int]
    L.bdepth_sample_name.restype = C.c_char_p
    L.bdepth_set_filter.argtypes = [vp, C.c_int, C.c_uint32]
    L.bdepth_set_filter_query.argtypes = [vp, C.c_char_p]
    L.bdepth_set_min_baseq.argtypes = [vp, C.c_uint32]
    L.bdepth_set_fix_mates.argtypes = [vp, C.c_int]
    L.bdepth_set_combined.argtypes = [vp, C.c_int]
    L.bdepth_set_samples_per_pass.argtypes = [vp, C.c_uint32]
    L.bdepth_set_regions.argtypes = [vp, C.POINTER(Region), C.c_size_t]
    L.bdepth_set_shard.argtypes = [vp, C.c_int, C.c_int, vp]
    L.bdepth_nccl_unique_id.argtypes = [vp]
    L.bdepth_set_tuning.argtypes = [vp, C.c_uint64, C.c_uint64]
    L.bdepth_stage.argtypes = [vp]
    L.bdepth_run_resident.argtypes = [vp]
    L.bdepth_plan_shards.argtypes = [C.c_char_p, C.c_int, C.POINTER(C.c_uint64)]
    L.bdepth_plan_region_chunks.argtypes = [C.c_char_p, C.POINTER(Region), C.c_size_t, C.POINTER(C.c_uint64), C.c_size_t]
    L.bdepth_plan_region_chunks.restype = C.c_long
    L.bdepth_run_base.argtypes = [vp, TILE_CB, vp]
    L.bdepth_run_base_text.argtypes = [vp, C.POINTER(TextOpts), TEXT_CB, vp]
    L.bdepth_run_windows.argtypes = [vp, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), C.c_size_t, STAT_CB, vp]
    L.bdepth_run_regions.argtypes = [vp, C.POINTER(Region), C.c_size_t, C.POINTER(C.c_uint32), C.c_size_t, STAT_CB, vp]
    L.bdepth_get_stats.argtypes = [vp, C.POINTER(Stats)]
    L.bdepth_ref_has_reads.argtypes = [vp, C.c_int]
    L.bdepth_inflate_to_host.argtypes = [vp, vp, C.c_uint64]
    L.bdepth_inflate_to_host.restype = C.c_int64
    L.bdepth_scan_to_host.argtypes = [vp, C.c_uint64] + [vp] * 7
    L.bdepth_scan_to_host.restype = C.c_int64
    L.bdepth_build_index.argtypes = [vp, vp, C.c_uint64]
    L.bdepth_build_index.restype = C.c_int64
    _lib = L
    return L


EXPORTED_SYMBOLS = [
    "bdepth_device_count", "bdepth_open", "bdepth_open_lazy", "bdepth_open_memory", "bdepth_add_input", "bdepth_close", "bdepth_last_error", "bdepth_n_ref",
    "bdepth_ref_name", "bdepth_ref_length", "bdepth_header_text", "bdepth_is_coordinate_sorted", "bdepth_has_index",
    "bdepth_n_samples", "bdepth_sample_name", "bdepth_set_filter", "bdepth_set_filter_query", "bdepth_set_min_baseq", "bdepth_set_fix_mates", "bdepth_set_combined", "bdepth_set_samples_per_pass", "bdepth_set_regions",
    "bdepth_set_shard", "bdepth_nccl_unique_id", "bdepth_plan_shards", "bdepth_plan_region_chunks", "bdepth_set_tuning", "bdepth_stage", "bdepth_run_resident", "bdepth_run_base", "bdepth_run_base_text",
    "bdepth_run_windows", "bdepth_run_regions", "bdepth_get_stats", "bdepth_ref_has_reads", "bdepth_inflate_to_host", "bdepth_scan_to_host", "bdepth_build_index",
]


def nccl_unique_id():
    L = load_library()
    buf = (C.c_char * 128)()
    rc = L.bdepth_nccl_unique_id(buf)
    if rc:
        raise BDepthError(rc, L.bdepth_last_error(None).decode())
    return bytes(buf)


def plan_shards(path, world):
    L = load_library()
    out = (C.c_uint64 * max(1, world - 1))()
    rc = L.bdepth_plan_shards(os.fsencode(path), world, out)
    if rc:
        raise BDepthError(rc, L.bdepth_last_error(None).decode())
    return list(out)[:world - 1]


def plan_region_chunks(path, regions):
    """Host-only: merged BGZF virtual-offset ranges [(beg, end), ...] a query for regions [(ref_id, start, end)] reads."""
    L = load_library()
    arr = (Region * max(1, len(regions)))(*[Region(*r) for r in regions])
    n = L.bdepth_plan_region_chunks(os.fsencode(path), arr, len(regions), None, 0)
    if n < 0:
        raise BDepthError(n, L.bdepth_last_error(None).decode())
    out = (C.c_uint64 * max(1, 2 * n))()
    L.bdepth_plan_region_chunks(os.fsencode(path), arr, len(regions), out, n)
    return [(out[2 * i], out[2 * i + 1]) for i in range(n)]


class BDepth:
    """Thin object wrapper over the C ABI (mirrors what the CLI host does)."""

    def __init__(self, path=None, device=0, memory=None, bai=None, lazy=False):
        self.L = load_library()
        self.h = C.c_void_p()
        if memory is not None:
            self._keep = (memory, bai)
            mp = memory.ctypes.data_as(C.c_void_p)
            bp = bai.ctypes.data_as(C.c_void_p) if bai is not None else None
            rc = self.L.bdepth_open_memory(mp, memory.size, bp, 0 if bai is None else bai.size, device, C.byref(self.h))
        else:
            rc = (self.L.bdepth_open_lazy if lazy else self.L.bdepth_open)(os.fsencode(path), device, C.byref(self.h))
        if rc:
            raise BDepthError(rc, self.L.bdepth_last_error(None).decode())

    def _ck(self, rc):
        if rc < 0:
            raise BDepthError(rc, self.L.bdepth_last_error(self.h).decode())
        return rc

    def add_input(self, path):
        self._ck(self.L.bdepth_add_input(self.h, os.fsencode(path)))

    def close(self):
        if self.h:
            self.L.bdepth_close(self.h)
            self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    # header
    @property
    def refs(self):
        return [(self.L.bdepth_ref_name(self.h, i).decode(), self.L.bdepth_ref_length(self.h, i))
                for i in range(self.L.bdepth_n_ref(self.h))]

    @property
    def samples(self):
        return [self.L.bdepth_sample_name(self.h, i).decode() for i in range(self.L.bdepth_n_samples(self.h))]

    @property
    def coordinate_sorted(self):
        return bool(self.L.bdepth_is_coordinate_sorted(self.h))

    @property
    def has_index(self):
        return bool(self.L.bdepth_has_index(self.h))

    # config
    def set_filter(self, mapq_gt=0, flag_reject=0x600):
        self._ck(self.L.bdepth_set_filter(self.h, mapq_gt, flag_reject))

    def set_filter_query(self, query):
        self._ck(self.L.bdepth_set_filter_query(self.h, query.encode()))

    def set_min_baseq(self, q):
        self._ck(self.L.bdepth_set_min_baseq(self.h, q))

    def set_fix_mates(self, on=True):
        self._ck(self.L.bdepth_set_fix_mates(self.h, 1 if on else 0))

    def set_combined(self, on=True):
        self._ck(self.L.bdepth_set_combined(self.h, 1 if on else 0))

    def set_samples_per_pass(self, n=0):
        """Region / window runs: count at most n samples per pipeline pass (0: as many as fit, up to 64)."""
        self._ck(self.L.bdepth_set_samples_per_pass(self.h, n))

    def set_regions(self, regions):
        arr = (Region * max(1, len(regions)))(*[Region(*r) for r in regions])
        self._ck(self.L.bdepth_set_regions(self.h, arr, len(regions)))

    def set_shard(self, rank, world, uid=None):
        self._uid = C.create_string_buffer(uid, 128) if uid is not None else None
        self._ck(self.L.bdepth_set_shard(self.h, rank, world, self._uid))

    def set_tuning(self, batch_bytes=0, chunk_blocks=0):
        self._ck(self.L.bdepth_set_tuning(self.h, batch_bytes, chunk_blocks))

    def stage(self):
        self._ck(self.L.bdepth_stage(self.h))

    def run_resident(self):
        self._ck(self.L.bdepth_run_resident(self.h))

    def stats(self):
        s = Stats()
        self.L.bdepth_get_stats(self.h, C.byref(s))
        return s.as_dict()

    # runs
    def lin_to_regions(self, a, b):
        """Split the linear window [a, b) at reference boundaries -> [(ref_id, start, end)]."""
        refs = self.refs
        out, lin = [], 0
        for i, (_, L) in enumerate(refs):
            lo, hi = max(a, lin), min(b, lin + L)
            if lo < hi:
                out.append((i, lo - lin, hi - lin))
            lin += L
        return out

    def run_base(self, collect=True, window=None):
        """Returns counts[7, n] over the linear window (default: the concatenated references)."""
        refs = self.refs
        lin0 = np.concatenate([[0], np.cumsum([l for _, l in refs])]).astype(np.int64)
        wa, wb = (0, int(lin0[-1])) if window is None else window
        if window is not None:
            self.set_regions(self.lin_to_regions(wa, wb))
        box = {}

        def cb(_user, tp):
            t = tp.contents
            if "out" not in box:
                box["out"] = np.zeros((t.n_samples, 7, max(0, wb - wa)), np.uint32)
            a = int(lin0[t.ref_id]) + t.start - wa
            src = np.ctypeslib.as_array(t.counts, shape=((t.n_samples - 1) * t.sample_stride + 6 * t.stride + t.len,))
            for si in range(t.n_samples):
                for p in range(7):
                    o = si * t.sample_stride + p * t.stride
                    box["out"][si, p, a:a + t.len] = src[o:o + t.len]
            return 0

        cbf = TILE_CB(cb) if collect else C.cast(None, TILE_CB)
        try:
            self._ck(self.L.bdepth_run_base(self.h, cbf, None))
        finally:
            if window is not None:
                self.set_regions([])
        if not collect:
            return None
        out = box.get("out")
        if out is None:
            return np.zeros((7, max(0, wb - wa)), np.uint32)
        return out[0] if out.shape[0] == 1 else out          # [7, n] for a single counter set, [S, 7, n] per sample

    def run_base_text(self, min_cov=1.0, max_cov=1e50, annotate=False, collect=True):
        """`depth base` rows formatted on the GPU; returns the text (bytes) when collect=True."""
        parts = []

        def cb(_user, ptr, n):
            if collect:
                parts.append(C.string_at(ptr, n))
            return 0
        opts = TextOpts(min_cov, max_cov, 1 if annotate else 0)
        self._ck(self.L.bdepth_run_base_text(self.h, C.byref(opts), TEXT_CB(cb), None))
        return b"".join(parts)

    def _run_stats(self, fn, collect=True):
        """collect=True: list of rows; "arrays": numpy columns (large runs); False: no callback at all (timing)."""
        if collect is False:
            self._ck(fn(C.cast(None, STAT_CB)))
            return None
        nthr = self._nthr
        if collect == "arrays":
            cap = [1 << 16]
            cols = {"ref_id": np.zeros(cap[0], np.int32), "start": np.zeros(cap[0], np.uint32), "end": np.zeros(cap[0], np.uint32), "n_reads": np.zeros(cap[0], np.uint32),
                    "n_bases": np.zeros(cap[0], np.uint32), "cov_ge": np.zeros((cap[0], max(1, nthr)), np.uint32), "sample_id": np.zeros(cap[0], np.int32)}
            n = [0]

            def cba(_user, sp, idx):
                s = sp.contents
                i = n[0]
                if i == cap[0]:
                    cap[0] *= 2
                    for k in cols:
                        cols[k] = np.concatenate([cols[k], np.zeros_like(cols[k])])
                cols["ref_id"][i] = s.ref_id; cols["start"][i] = s.start; cols["end"][i] = s.end; cols["n_reads"][i] = s.n_reads; cols["n_bases"][i] = s.n_bases; cols["sample_id"][i] = s.sample_id
                for t in range(nthr):
                    cols["cov_ge"][i, t] = s.cov_ge[t]
                n[0] = i + 1
                return 0
            self._ck(fn(STAT_CB(cba)))
            return {k: v[:n[0]] for k, v in cols.items()}
        rows = []

        def cb(_user, sp, idx):
            s = sp.contents
            rows.append((s.ref_id, s.start, s.end, s.n_reads, s.n_bases, [s.cov_ge[i] for i in range(nthr)], s.sample_id))
            return 0
        self._ck(fn(STAT_CB(cb)))
        return rows

    def run_windows(self, window, overlap=0, thresholds=(), collect=True):
        thr = (C.c_uint32 * max(1, len(thresholds)))(*thresholds)
        self._nthr = len(thresholds)
        return self._run_stats(lambda cb: self.L.bdepth_run_windows(self.h, window, overlap, thr, len(thresholds), cb, None), collect)

    def run_regions(self, regions, thresholds=(), collect=True):
        thr = (C.c_uint32 * max(1, len(thresholds)))(*thresholds)
        if isinstance(regions, np.ndarray):          # [n, 3] uint32 (ref_id, start, end): no per-region Python objects
            flat = np.ascontiguousarray(regions, np.uint32)
            arr = C.cast(flat.ctypes.data_as(C.c_void_p), C.POINTER(Region)); n = len(flat); self._keep_regions = flat
        else:
            arr = (Region * max(1, len(regions)))(*[Region(*r) for r in regions]); n = len(regions)
        self._nthr = len(thresholds)
        return self._run_stats(lambda cb: self.L.bdepth_run_regions(self.h, arr, n, thr, len(thresholds), cb, None), collect)

    def inflate(self):
        n = self._ck(self.L.bdepth_inflate_to_host(self.h, None, 0))
        buf = np.zeros(max(1, n), np.uint8)
        n2 = self._ck(self.L.bdepth_inflate_to_host(self.h, buf.ctypes.data_as(C.c_void_p), n))
        assert n2 == n
        return buf[:n]

    def build_index(self):
        """The BAI index of the file, built on the GPU (bytes); the handle adopts it."""
        n = self._ck(self.L.bdepth_build_index(self.h, None, 0))
        buf = np.zeros(max(1, n), np.uint8)
        n2 = self._ck(self.L.bdepth_build_index(self.h, buf.ctypes.data_as(C.c_void_p), n))
        assert n2 == n
        return buf[:n].tobytes()

    def scan(self, cap):
        cols = dict(ref_id=np.zeros(cap, np.int32), pos=np.zeros(cap, np.int32), span=np.zeros(cap, np.uint32),
                    flag=np.zeros(cap, np.uint16), mapq=np.zeros(cap, np.uint8), n_cigar=np.zeros(cap, np.uint16),
                    rec_off=np.zeros(cap, np.uint64))
        n = self._ck(self.L.bdepth_scan_to_host(self.h, cap, *[c.ctypes.data_as(C.c_void_p) for c in cols.values()]))
        return n, {k: v[:min(n, cap)] for k, v in cols.items()}
