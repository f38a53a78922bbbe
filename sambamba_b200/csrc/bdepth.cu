// bdepth.cu -- host pipeline and C ABI of libbdepth.so (see include/bdepth.h for the contract and
// the reference seams each entry point replaces).
//
// Pipeline per batch of BGZF blocks (all on one CUDA stream; a second stream feeds H2D):
//   H2D (pinned or pageable)  ->  K1 inflate  ->  K2 guess/walk (+ host chain verification)
//   ->  K2 decode (SoA)  ->  K3 tile index / long-read scatter / per-position gather
// then reducers + D2H for the chosen front end (base tiles, window stats, region stats).
// There is no CPU fallback anywhere: if CUDA is unavailable every run returns BDEPTH_ERR_CUDA.
#include "launch.cuh"
#include <dlfcn.h>
#include <fcntl.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <chrono>
#include <map>
#include <string>
#include <vector>

#include "../../include/bdepth.h"
#include "host_bam.hpp"
#include "kernels.cuh"
#include "mates.cuh"
#include "host_filter.hpp"

using namespace bdk;

namespace {

thread_local std::string g_open_error;

struct DevBuf {
    void* p = nullptr; size_t cap = 0;
    cudaError_t ensure(size_t n) {
        if (n <= cap) return cudaSuccess;
        if (p) { cudaFree(p); p = nullptr; cap = 0; }
        size_t want = n + n / 8 + 256;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T* as() const { return (T*)p; }
};

// Small control-plane transfers (block tables up, chain/scan results down) do not go through the copy engines:
// those queue in order behind the bulk H2D of the compressed file and the bulk D2H of finished counters, which
// cost every sub-batch milliseconds.  They live in mapped pinned memory and a tiny kernel moves the words.
struct HostScratch {
    uint8_t* hp = nullptr; uint8_t* dp = nullptr; size_t cap = 0, used = 0;
    cudaError_t ensure(size_t n) {          // only while nothing in flight refers to it
        if (n <= cap) return cudaSuccess;
        if (hp) { cudaDeviceSynchronize(); cudaFreeHost(hp); hp = nullptr; dp = nullptr; cap = 0; }
        cudaError_t e = cudaHostAlloc((void**)&hp, n + n / 4, cudaHostAllocMapped);
        if (e != cudaSuccess) return e;
        e = cudaHostGetDevicePointer((void**)&dp, hp, 0);
        if (e == cudaSuccess) cap = n + n / 4;
        used = 0;
        return e;
    }
    uint8_t* take(size_t n) { size_t a = (used + 15) & ~size_t(15); if (a + n > cap) return nullptr; used = a + n; return hp + a; }
    uint8_t* dev(const void* host) const { return dp + ((const uint8_t*)host - hp); }
    void release() { if (hp) cudaFreeHost(hp); hp = nullptr; dp = nullptr; cap = used = 0; }
};
__global__ void k_copy_words(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, size_t n) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

#ifdef BDEPTH_EMULATE_SHIM
constexpr unsigned COUNT_GRID = 4;           // grid-stride reducer: any grid gives the same sum; the CPU emulation runs blocks one by one
#else
constexpr unsigned COUNT_GRID = 2048;
#endif
constexpr size_t CARRY_MAX = 64ull << 20;
constexpr size_t EMIT_CHUNK = 4ull << 20;     // positions per D2H chunk
constexpr uint32_t SHARD_EXTRA_BLOCKS = 8;
constexpr uint32_t MATE_ZONE_BLOCKS = 64;       // -m on several ranks: blocks read behind the shard so that pairs cut by the boundary are seen whole

enum RunMode { RUN_FULL = 0, RUN_INFLATE_ONLY = 1, RUN_SCAN_ONLY = 2, RUN_INDEX = 3 };
constexpr int RC_RETRY_WINDOW = 1;      // internal: a read lies outside the counter window a multi-input run was given

// ---- NCCL, bound at run time (dlopen) so that single-GPU users need no NCCL at all and so that a host
// process that already loaded NCCL (e.g. through torch) shares that one instance (same SONAME).
struct NcclUid { char b[128]; };
typedef void* NcclComm;
struct NcclApi {
    bool ok = false; std::string err;
    int (*GetUniqueId)(NcclUid*) = nullptr;
    int (*CommInitRank)(NcclComm*, int, NcclUid, int) = nullptr;
    int (*CommDestroy)(NcclComm) = nullptr;
    int (*AllGather)(const void*, void*, size_t, int, NcclComm, cudaStream_t) = nullptr;
    int (*AllReduce)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*Send)(const void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*Recv)(void*, size_t, int, int, NcclComm, cudaStream_t) = nullptr;
    int (*GroupStart)() = nullptr;
    int (*GroupEnd)() = nullptr;
    const char* (*GetErrorString)(int) = nullptr;
};
constexpr int NCCL_UINT32 = 3, NCCL_UINT64 = 5, NCCL_SUM = 0;    // ncclDataType_t / ncclRedOp_t values (nccl.h)
NcclApi& nccl() {
    static NcclApi api; static bool tried = false;
    if (tried) return api;
    tried = true;
#ifdef BDEPTH_EMULATE_SHIM      // test build only (launch.cuh): ranks are threads, the collectives are rendezvous between them
    api.GetUniqueId = [](NcclUid* u) { return emu_ncclGetUniqueId(u->b); };
    api.CommInitRank = [](NcclComm* c, int w, NcclUid u, int r) { return emu_ncclCommInitRank(c, w, u.b, r); };
    api.CommDestroy = emu_ncclCommDestroy; api.AllGather = emu_ncclAllGather; api.AllReduce = emu_ncclAllReduce; api.Send = emu_ncclSend; api.Recv = emu_ncclRecv;
    api.GroupStart = emu_ncclGroupStart; api.GroupEnd = emu_ncclGroupEnd; api.GetErrorString = emu_ncclGetErrorString; api.ok = true;
    return api;
#endif
    void* lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!lib) { api.err = std::string("cannot load libnccl.so.2: ") + dlerror(); return api; }
    bool all = true;
    auto sym = [&](const char* n) { void* p = dlsym(lib, n); if (!p) { all = false; api.err = std::string("missing NCCL symbol ") + n; } return p; };
    api.GetUniqueId = (int (*)(NcclUid*))sym("ncclGetUniqueId");
    api.CommInitRank = (int (*)(NcclComm*, int, NcclUid, int))sym("ncclCommInitRank");
    api.CommDestroy = (int (*)(NcclComm))sym("ncclCommDestroy");
    api.AllGather = (int (*)(const void*, void*, size_t, int, NcclComm, cudaStream_t))sym("ncclAllGather");
    api.AllReduce = (int (*)(const void*, void*, size_t, int, int, NcclComm, cudaStream_t))sym("ncclAllReduce");
    api.Send = (int (*)(const void*, size_t, int, int, NcclComm, cudaStream_t))sym("ncclSend");
    api.Recv = (int (*)(void*, size_t, int, int, NcclComm, cudaStream_t))sym("ncclRecv");
    api.GroupStart = (int (*)())sym("ncclGroupStart");
    api.GroupEnd = (int (*)())sym("ncclGroupEnd");
    api.GetErrorString = (const char* (*)(int))sym("ncclGetErrorString");
    api.ok = all;
    return api;
}

}  // namespace

struct bdepth {
    // ---- input
    const uint8_t* file = nullptr; size_t file_len = 0; bool mapped = false; int fd = -1;
    std::vector<HostBlock> blocks; uint64_t total_u = 0;
    // lazy open (bdepth_open_lazy): `blocks` is a prefix of the file's BGZF members (enough for the header) until somebody
    // needs them all; a region query never does (plan_sparse frames the members of its BAI chunks on its own)
    bool lazy = false, framed_all = true; size_t framed_off = 0;
    BamHeader hdr; BaiIndex bai; bool has_index = false;
    int device = 0;
    // ---- config
    int mapq_gt = 0; uint32_t flag_reject = 0x600; uint32_t minq = 0;
    std::vector<bdepth_region> regions;   // merged, sorted
    int rank = 0, world = 1;
    NcclComm comm = nullptr; bool have_uid = false; NcclUid uid{};
    uint64_t own_lo = 0, own_hi = 0;      // linear range owned by this rank (whole genome when world == 1)
    bool bai_window_ok = true;            // cleared when the linear index turns out not to describe the file
    bool combined = false;                // --combined: one counter set for all samples
    bool fix_mates = false;               // -m: overlapping mates count once per column (mates.cuh)
    bool k1lz_v12 = false;                // BDEPTH_K1LZ=v12: k1_lz with the uncompacted literal table (A/B)
    bool k1lz_flat = false;               // BDEPTH_K1LZ=flat: phase 2 with one output byte per lane (k1_lz_flat) instead of one token per lane (k1_lz)
    int k1h_variant = -1;                 // BDEPTH_K1H_VARIANT: which instantiation of k1_huff runs (-1: by launch size; 0: limits in registers, 4 CTAs/SM; 2: limits in shared memory, 5 CTAs/SM)
    bool k1_onephase = false;             // BDEPTH_K1_ONEPHASE=1: the round-1 one-phase K1 for every block (A/B against the two-phase inflater)
    bool k3_pre = false;                  // BDEPTH_K3_PREFETCH=0: k3_gather without the lane-parallel record prefetch
    bool k3_tile = true;                  // BDEPTH_K3=gather: the round-1 per-position gather kernel instead of k3_tile
    bool has_fprog = false; FilterProg fprog; DevBuf fprog_d;      // -F: compiled query (filter.cuh); otherwise mapq_gt / flag_reject
    DevBuf m_hash, m_flag, m_flt, m_ctl;
    uint32_t S = 1;                       // counter sets in the current run (samples, or 1)
    uint32_t samples_per_pass = 0;        // bdepth_set_samples_per_pass: region / window runs hold at most this many samples' counters at once (0: as many as fit, up to 64)
    uint32_t pass_g0 = 0, pass_n = 0;     // a sample pass (run_segments): the run counts samples [pass_g0, pass_g0 + pass_n) only; pass_n == 0: every sample at once
    bool pass_untagged = false;           // set by a sample pass that met passing reads without an RG tag while it did not hold sample 0
    DevBuf rg_ids, rg_offs, rg_samp, rg_hash, rg_tab;
    DevBuf text[2], text_tiles, text_offs, text_zero, text_samp, present;
    int coll_pending = 0;                 // several ranks: collectives of the current run this rank has not joined yet (2: the sparse decision and the boundary table; 1: the boundary table) -- a rank that stops with an error joins them with a "failed" mark, so that the others stop too instead of waiting for it
    bool want_presence = false;           // -a with -q and a positive minimum coverage: mark the positions reads cover (k_presence)
    uint64_t batch_u = 6ull << 30;
    uint64_t chunk_blocks = 13 * 32 * 16;              // BGZF blocks per H2D chunk = per K1 sub-launch = per sub-batch: 6656 blocks = 16 K1 CTAs, ~260 MB compressed
    // ---- shard (resolved lazily)
    bool shard_ready = false;
    size_t blk_lo = 0, blk_hi = 0; int64_t entry0 = 0; uint64_t limit_abs_u = 0;
    uint64_t zone_lin_lo = UINT64_MAX;    // several ranks: linear coordinate of the 16 kbp window in which this rank's first record begins (its counter window starts there)
    uint64_t own_lo_abs_u = 0;            // several ranks: the stream begins before the shard does (zone of the previous rank); own records start here
    // Sparse staging for region queries (SURVEY 8a row a17): only the BGZF blocks inside the BAI chunk list of the
    // regions are copied, inflated and scanned.  vblocks = those blocks with uoff re-based to a compact stream;
    // a segment is one merged chunk: it starts at a record (seg_entry = offset inside its first block) and ends at
    // one (seg_limit = offset inside its last block at which the walk stops).
    bool sparse_ok = true;                            // cleared when the index turns out not to describe the file
    bool sparse_on = false;                           // this run uses vblocks
    std::vector<HostBlock> vblocks; std::vector<int32_t> seg_entry /* -1: not a segment start */; std::vector<uint32_t> seg_limit /* UINT32_MAX: none */;
    DevBuf anchors_idx, anchors_val, chunk_limit;
    // ---- device state
    cudaStream_t s_main = nullptr, s_copy = nullptr, s_d2h = nullptr;
    cudaEvent_t ev[32] = {};
    DevBuf comp2[2];
    cudaStream_t s_k1[16] = {};                       // K1 sub-launches of one batch run side by side (one stream each)
    std::vector<cudaEvent_t> chunk_ev[2], k1_ev;      // per H2D chunk (per slot) / per K1 sub-launch
    std::vector<size_t> chunk_end[2];                  // block index (exclusive) covered by each H2D chunk of a slot
    bool staged = false; uint64_t staged_file_off = 0;
    DevBuf tok, lits, aux, segi, littab;              // two-phase K1: match tokens, packed literals, per-block counts, segment starts, literal tables
    DevBuf comp, descs, status, ubuf, chunk_start, entry, exitb, count, slot_base, slots, rec_base, walk_list;
    DevBuf soa_start, soa_span, soa_meta, soa_off, soa_ncl, soa_lseq, long_list, tile_first, tile_lo, counts, ref_len_d, ref_lin0_d, scan_stats, ref_has, ref_has_all, flt_d, lead_list, misc;
    uint64_t cnt_base = 0, win_len = 0;
    void* pinned = nullptr; size_t pinned_cap = 0;
    HostScratch hs;
    std::vector<uint32_t> ref_has_host;
    // ---- optional per-read segment counting (window / region front ends), device arrays
    struct SegSet { bool on = false; uint32_t n = 0; bool has_min = false, has_u = false; uint64_t ext_max = 0; DevBuf s, e, pmax, id, reads, minstart, bases_reads, mbases, ustart, da, dac, db, dthr, dbases, dcov, dscr; } seg;
    // ---- BAI builder (bdepth_build_index): device tables of k_index_scan, the runs / exceptions it handed out, the finished index
    struct IndexSet { DevBuf lin, lin_len, lin_base, lin_cap, n_mapped, n_unmapped, carry, ctl, runs, excs; std::vector<uint32_t> base, cap; std::vector<IndexRun> h_runs; std::vector<IndexExc> h_excs; uint64_t n_lin = 0; } ix;
    std::vector<uint8_t> built_bai;
    // ---- several BAM files (bdepth_add_input; MultiBamReader, multireader.d:218-268): the additional files are whole handles that
    // only hold their input (file, BGZF members, header, index, shard / sparse plan); a run swaps them into this handle one after
    // the other and accumulates into the same counters -- per-position counters and per-segment sums are additive over reads,
    // and without -m nothing depends on the order in which the merged stream would have delivered them
    std::vector<bdepth*> extra;
    bool accum = false;                   // the run continues on the counters of the previous input
    bool force_window = false;            // counter window fixed by the caller (union over the inputs)
    // ---- results
    bdepth_stats st{}; std::string err;
};

namespace {

int fail(bdepth* h, int code, const char* fmt, ...) {
    char buf[1024]; va_list ap; va_start(ap, fmt); vsnprintf(buf, sizeof buf, fmt, ap); va_end(ap);
    if (h) h->err = buf; else g_open_error = buf;
    return code;
}
#define NK(call) do { int r__ = (call); if (r__ != 0) return fail(h, BDEPTH_ERR_NCCL, "NCCL error at %s:%d: %s", __FILE__, __LINE__, nccl().GetErrorString ? nccl().GetErrorString(r__) : "?"); } while (0)
#define CK(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(h, BDEPTH_ERR_CUDA, "CUDA error %s at %s:%d: %s", cudaGetErrorName(e__), __FILE__, __LINE__, cudaGetErrorString(e__)); } while (0)

int ensure_pinned(bdepth* h, size_t n) {
    if (n <= h->pinned_cap) return 0;
    if (h->pinned) cudaFreeHost(h->pinned);
    h->hs.release();
    h->pinned = nullptr; h->pinned_cap = 0;
    CK(cudaMallocHost(&h->pinned, n));
    h->pinned_cap = n;
    return 0;
}

int init_device(bdepth* h) {
    int n = 0; cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) return fail(h, BDEPTH_ERR_CUDA, "no CUDA device available (%s); libbdepth has no CPU fallback", cudaGetErrorString(e));
    if (h->device < 0 || h->device >= n) return fail(h, BDEPTH_ERR_ARG, "device %d out of range (%d devices)", h->device, n);
    CK(cudaSetDevice(h->device));
    if (!h->s_main) { CK(cudaStreamCreateWithFlags(&h->s_main, cudaStreamNonBlocking)); CK(cudaStreamCreateWithFlags(&h->s_copy, cudaStreamNonBlocking)); CK(cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking)); for (auto& ks : h->s_k1) CK(cudaStreamCreateWithFlags(&ks, cudaStreamNonBlocking)); for (auto& e2 : h->ev) CK(cudaEventCreate(&e2)); }
    CK(cudaFuncSetAttribute(k1_inflate, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_SMEM));
    CK(cudaFuncSetAttribute(k1_fallback, cudaFuncAttributeMaxDynamicSharedMemorySize, K1_SMEM));
    CK(cudaFuncSetAttribute(k1_huff<false, 4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); CK(cudaFuncSetAttribute(k1_huff<false, 6>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    CK(cudaFuncSetAttribute(k1_huff<true, 5>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)); CK(cudaFuncSetAttribute(k1_huff<true, 4>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    { const char* e = getenv("BDEPTH_K1H_VARIANT"); h->k1h_variant = e ? atoi(e) : -1; }      // A/B of the phase-1 instantiations (kernels.cuh)
    { const char* e = getenv("BDEPTH_K3"); h->k3_tile = !(e && !strcmp(e, "gather")); }
    CK(cudaFuncSetAttribute(k3_tile<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K3T_SMEM)); CK(cudaFuncSetAttribute(k3_tile<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)K3T_SMEM));
    { const char* e = getenv("BDEPTH_K1LZ"); h->k1lz_flat = e && !strcmp(e, "flat"); h->k1lz_v12 = e && !strcmp(e, "v12"); }      // A/B of the two phase-2 kernels
    { const char* e = getenv("BDEPTH_K1_ONEPHASE"); h->k1_onephase = e && atoi(e) == 1; }
    { const char* e = getenv("BDEPTH_K3_PREFETCH"); h->k3_pre = !e || atoi(e) != 0; }      // default since round 2: measured 10.4 -> 8.4 ms on chr20 (profiles/k3_history.md)
    return 0;
}

// Inflate blocks [b0, b1) into a host vector (used for the header only: a few blocks).
int inflate_blocks_to_host(bdepth* h, size_t b0, size_t b1, std::vector<uint8_t>& out) {
    size_t nb = b1 - b0; if (!nb) { out.clear(); return 0; }
    uint64_t f0 = h->blocks[b0].coff & ~3ull, f1 = h->blocks[b1 - 1].coff + h->blocks[b1 - 1].bsize;
    uint64_t ulen = h->blocks[b1 - 1].uoff + h->blocks[b1 - 1].isize - h->blocks[b0].uoff;
    CK(h->comp.ensure(f1 - f0 + 256)); CK(h->descs.ensure(nb * sizeof(BlockDesc))); CK(h->status.ensure(nb * sizeof(int))); CK(h->ubuf.ensure(CARRY_MAX + ulen + 256));
    std::vector<BlockDesc> d(nb);
    for (size_t i = 0; i < nb; i++) { const HostBlock& b = h->blocks[b0 + i]; d[i] = BlockDesc{b.coff + b.cdata_off - f0, b.uoff - h->blocks[b0].uoff, b.csize, b.isize}; }
    CK(cudaMemcpyAsync(h->comp.p, h->file + f0, f1 - f0, cudaMemcpyHostToDevice, h->s_main));
    CK(cudaMemsetAsync((uint8_t*)h->comp.p + (f1 - f0), 0, 128, h->s_main));
    CK(cudaMemcpyAsync(h->descs.p, d.data(), nb * sizeof(BlockDesc), cudaMemcpyHostToDevice, h->s_main));
    BD_LAUNCH((unsigned)((nb + 32 * K1_WARPS - 1) / (32 * K1_WARPS)), 32 * K1_WARPS, K1_SMEM, h->s_main, k1_inflate)(h->comp.as<uint32_t>(), h->descs.as<BlockDesc>(), (uint32_t)nb, h->ubuf.as<uint8_t>() + CARRY_MAX, h->status.as<int>());
    CK(cudaGetLastError());
    std::vector<int> stt(nb); out.resize(ulen);
    CK(cudaMemcpyAsync(stt.data(), h->status.p, nb * sizeof(int), cudaMemcpyDeviceToHost, h->s_main));
    CK(cudaMemcpyAsync(out.data(), h->ubuf.as<uint8_t>() + CARRY_MAX, ulen, cudaMemcpyDeviceToHost, h->s_main));
    CK(cudaStreamSynchronize(h->s_main));
    h->st.gpu_launches += 1;
    for (size_t i = 0; i < nb; i++) if (stt[i]) return fail(h, BDEPTH_ERR_FORMAT, "DEFLATE error %d in BGZF block at offset %llu", stt[i], (unsigned long long)h->blocks[b0 + i].coff);
    return 0;
}

// frame up to `more` further BGZF members (all of them: SIZE_MAX)
int frame_more(bdepth* h, size_t more) {
    if (h->framed_all) return 0;
    bool eof = false;
    std::string e = frame_bgzf(h->file, h->file_len, &h->framed_off, &h->total_u, more, UINT64_MAX, h->blocks, &eof);
    if (!e.empty()) return fail(h, BDEPTH_ERR_FORMAT, "%s", e.c_str());
    if (eof) h->framed_all = true;
    return 0;
}
int ensure_all_blocks(bdepth* h) { return frame_more(h, SIZE_MAX); }

int finish_open(bdepth* h) {
    h->blocks.clear(); h->total_u = 0; h->framed_off = 0; h->framed_all = false;
    { int rcf = frame_more(h, h->lazy ? 4 : SIZE_MAX); if (rcf) return rcf; }
    if (h->blocks.empty()) return fail(h, BDEPTH_ERR_FORMAT, "Invalid file format: expected BAM\\1");
    int rc = init_device(h); if (rc) return rc;
    // header: inflate a growing prefix of blocks on the GPU until it parses
    size_t nb = std::min<size_t>(4, h->blocks.size());
    for (;;) {
        std::vector<uint8_t> u; rc = inflate_blocks_to_host(h, 0, nb, u); if (rc) return rc;
        std::string perr; int pr = parse_bam_header(u.data(), u.size(), h->hdr, perr);
        if (pr == 0) break;
        if (pr < 0) return fail(h, BDEPTH_ERR_FORMAT, "%s", perr.c_str());
        if (nb == h->blocks.size() && !h->framed_all) { rc = frame_more(h, nb * 3); if (rc) return rc; }
        if (nb == h->blocks.size()) return fail(h, BDEPTH_ERR_FORMAT, "truncated BAM header");
        nb = std::min(h->blocks.size(), nb * 4);
    }
    size_t nref = h->hdr.ref_len.size();
    CK(h->ref_len_d.ensure((nref + 1) * 4)); CK(h->ref_lin0_d.ensure((nref + 1) * 8));
    if (nref) { CK(cudaMemcpy(h->ref_len_d.p, h->hdr.ref_len.data(), nref * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(h->ref_lin0_d.p, h->hdr.ref_lin0.data(), nref * 8, cudaMemcpyHostToDevice)); }
    return 0;
}

// Candidate shard boundaries: every distinct record start recorded in the BAI linear index.
std::vector<uint64_t> shard_candidates(const BaiIndex& bai) {
    std::vector<uint64_t> vos;
    for (auto& v : bai.ioffsets) for (uint64_t x : v) if (x) vos.push_back(x);
    std::sort(vos.begin(), vos.end()); vos.erase(std::unique(vos.begin(), vos.end()), vos.end());
    return vos;
}
// k-th of `world` boundaries: first candidate whose compressed offset is >= k * file_len / world.
uint64_t shard_cut_voffset(const std::vector<uint64_t>& vos, uint64_t file_len, int k, int world) {
    uint64_t target = (uint64_t)((__uint128_t)file_len * (unsigned)k / (unsigned)world);
    auto it = std::lower_bound(vos.begin(), vos.end(), target << 16);
    return it == vos.end() ? UINT64_MAX : *it;
}

// Resolve the block range / entry / limit of this rank's shard.
int prepare_shard(bdepth* h) {
    if (h->shard_ready) return 0;
    { int rcf = ensure_all_blocks(h); if (rcf) return rcf; }
    const auto& B = h->blocks;
    auto block_of_u = [&](uint64_t u) { size_t lo = 0, hi = B.size(); while (lo + 1 < hi) { size_t m = (lo + hi) / 2; if (B[m].uoff <= u) lo = m; else hi = m; } return lo; };
    auto block_of_c = [&](uint64_t c) { size_t lo = 0, hi = B.size(); while (lo + 1 < hi) { size_t m = (lo + hi) / 2; if (B[m].coff <= c) lo = m; else hi = m; } return lo; };
    uint64_t start_u = h->hdr.first_rec_off, end_u = h->total_u;
    if (h->world > 1) {
        if (!h->bai.valid) return fail(h, BDEPTH_ERR_NOINDEX, "sharding needs the BAI linear index");
        std::vector<uint64_t> vos = shard_candidates(h->bai);
        auto cut = [&](int k) -> uint64_t {   // absolute inflated offset of the k-th shard boundary
            if (k <= 0) return h->hdr.first_rec_off;
            if (k >= h->world) return h->total_u;
            uint64_t vo = shard_cut_voffset(vos, h->file_len, k, h->world);
            if (vo == UINT64_MAX) return h->total_u;
            size_t b = block_of_c(vo >> 16);
            if (B[b].coff != (vo >> 16)) return h->total_u;      // index does not match the file
            uint64_t u = B[b].uoff + (vo & 0xFFFF);
            return u < h->hdr.first_rec_off ? h->hdr.first_rec_off : u;
        };
        start_u = cut(h->rank); end_u = cut(h->rank + 1);
        if (end_u < start_u) end_u = start_u;
    }
    if (start_u >= h->total_u) { h->blk_lo = h->blk_hi = B.size(); h->entry0 = 0; h->limit_abs_u = h->total_u; h->shard_ready = true; return 0; }
    h->blk_lo = block_of_u(start_u); h->entry0 = (int64_t)(start_u - B[h->blk_lo].uoff);
    h->limit_abs_u = end_u; h->own_lo_abs_u = start_u;
    if (end_u >= h->total_u) h->blk_hi = B.size();
    else h->blk_hi = std::min(B.size(), block_of_u(end_u) + 1 + (h->fix_mates ? MATE_ZONE_BLOCKS : SHARD_EXTRA_BLOCKS));
    h->zone_lin_lo = UINT64_MAX;
    if (h->world > 1 && h->rank > 0) {      // (with -m: the same zone, read for the mate kernels; without: its reads are counted where they reach into this rank's positions)
        // The zone before the shard.  The BAI linear index holds, per 16 kbp window, the first record that overlaps the window:
        // starting at the entry of the window of the shard's first read includes every read that overlaps any column at or
        // after that window's start, i.e. every read the rank's own components and their columns can involve.
        std::vector<uint8_t> u; int rc = inflate_blocks_to_host(h, h->blk_lo, std::min(B.size(), h->blk_lo + 2), u); if (rc) return rc;
        const uint64_t o = (uint64_t)h->entry0;
        if (o + 12 <= u.size()) {
            int32_t ref = (int32_t)h_rd32(u.data() + o + 4), pos = (int32_t)h_rd32(u.data() + o + 8);
            if (ref >= 0 && (size_t)ref < h->bai.ioffsets.size() && pos >= 0) {
                const auto& lin = h->bai.ioffsets[ref]; size_t w = (size_t)pos >> 14;
                uint64_t vo = w < lin.size() ? lin[w] : 0;
                if (vo) {
                    size_t b = block_of_c(vo >> 16);
                    if (B[b].coff != (vo >> 16)) return fail(h, BDEPTH_ERR_FORMAT, "fix-mate-overlaps on several ranks: the linear index does not match the file");
                    uint64_t zu = B[b].uoff + (vo & 0xFFFF);
                    if (zu < h->hdr.first_rec_off) zu = h->hdr.first_rec_off;
                    if (zu < start_u) { h->blk_lo = block_of_u(zu); h->entry0 = (int64_t)(zu - B[h->blk_lo].uoff); }
                    h->zone_lin_lo = h->hdr.ref_lin0[ref] + ((uint64_t)w << 14);      // this rank's own positions begin at or after the first record's position, i.e. inside this window
                }
            }
        }
    }
    h->shard_ready = true;
    return 0;
}

// ---- base-mode delivery: D2H of finished counter ranges in EMIT_CHUNK pieces on a separate stream, double
// buffered in pinned memory, split at reference boundaries for the callback.  advance(limit) may be called after
// every batch: positions below the first read start of the following batch can no longer change (the file is
// coordinate sorted), so their D2H overlaps the next batch's inflate.
struct Emitter {
    bdepth* h; bdepth_tile_cb cb; void* user;
    struct Range { uint64_t a, b; };
    std::vector<Range> ranges; size_t ri = 0; uint64_t pos = 0; bool started = false;
    uint64_t lo_clip = 0, hi_clip = UINT64_MAX;      // several ranks: only the positions this rank owns are delivered
    struct Slot { uint64_t a = 0, b = 0; } slot[2];
    int head = 0, inflight = 0;
    uint64_t d2h_bytes = 0;
    // the pinned double buffer holds 2 x [S][7][chunk] ; chunk shrinks with the number of samples
    size_t chunk() const { return EMIT_CHUNK / h->S; }
    int issue(int si, uint64_t a, uint64_t b) {
        const int NP = N_PLANES * (int)h->S; const size_t CH = chunk();
        uint32_t* dst = (uint32_t*)h->pinned + (size_t)si * EMIT_CHUNK * N_PLANES;
        uint64_t wa = std::max(a, h->cnt_base), wb = std::min(b, h->cnt_base + h->win_len);   // outside the window: zeros
        if (wa >= wb || wa > a || wb < b) for (int pl = 0; pl < NP; pl++) memset(dst + (size_t)pl * CH, 0, (b - a) * 4);
        if (wa < wb) for (int pl = 0; pl < NP; pl++) CK(cudaMemcpyAsync(dst + (size_t)pl * CH + (wa - a), h->counts.as<uint32_t>() + (uint64_t)pl * h->win_len + (wa - h->cnt_base), (wb - wa) * 4, cudaMemcpyDeviceToHost, h->s_d2h));
        CK(cudaEventRecord(h->ev[8 + si], h->s_d2h));
        slot[si].a = a; slot[si].b = b; d2h_bytes += (b - a) * NP * 4;
        return 0;
    }
    int deliver_oldest() {
        int si = (head + 2 - inflight) & 1;     // oldest in-flight slot
        CK(cudaEventSynchronize(h->ev[8 + si]));
        inflight--;
        if (!cb) return 0;
        const uint32_t* src = (const uint32_t*)h->pinned + (size_t)si * EMIT_CHUNK * N_PLANES;
        uint64_t a = slot[si].a, bnd = slot[si].b; const size_t nref = h->hdr.ref_len.size();
        size_t ref = std::upper_bound(h->hdr.ref_lin0.begin(), h->hdr.ref_lin0.end(), a) - h->hdr.ref_lin0.begin() - 1;
        while (a < bnd && ref < nref) {
            uint64_t rend = h->hdr.ref_lin0[ref] + h->hdr.ref_len[ref];
            if (a >= rend) { ref++; continue; }
            uint64_t e = std::min(bnd, rend);
            bdepth_tile t{(int32_t)ref, (uint32_t)(a - h->hdr.ref_lin0[ref]), (uint32_t)(e - a), (uint32_t)chunk(), src + (a - slot[si].a), h->S, (uint32_t)(chunk() * N_PLANES)};
            if (cb(user, &t)) return fail(h, BDEPTH_ERR_CALLBACK, "tile callback aborted");
            a = e;
        }
        return 0;
    }
    // everything below `limit` (linear coordinate) is final once `ready` (recorded on the main stream) has fired
    int advance(uint64_t limit, cudaEvent_t ready) {
        if (ready) CK(cudaStreamWaitEvent(h->s_d2h, ready, 0));
        if (!started) { started = true; if (!ranges.empty()) pos = ranges[0].a; }
        while (ri < ranges.size()) {
            const Range& r = ranges[ri];
            const uint64_t rb = std::min(r.b, hi_clip);
            uint64_t a = std::max(std::max(pos, r.a), lo_clip);
            if (a >= rb) { if (r.b > hi_clip) break; ri++; if (ri < ranges.size()) pos = ranges[ri].a; continue; }      // (nothing beyond hi_clip is this rank's)
            if (a >= limit) break;
            uint64_t b = std::min(std::min(rb, limit), a + (uint64_t)chunk());
            if (inflight == 2) { int rc = deliver_oldest(); if (rc) return rc; }
            int rc = issue(head, a, b); if (rc) return rc;
            head ^= 1; inflight++; pos = b;
        }
        return 0;
    }
    int finish() { while (inflight) { int rc = deliver_oldest(); if (rc) return rc; } return 0; }
};

__global__ void k_add_u32(uint32_t* __restrict__ dst, const uint32_t* __restrict__ src, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) dst[i] += src[i];
}

// Multi-GPU boundary exchange (SURVEY 8e).  Rank k holds the counters of ITS reads, which start in
// [min_k, min_{k+1}) but may run past min_{k+1}.  Ownership of position p goes to the last rank whose first
// read starts at or before p; every rank sends the part of its counters that lies in a later rank's range
// (7 planes, packed) with ncclSend/ncclRecv inside one group, and the owner adds it.  One all-gather of
// (min_start, max_end) per rank tells everybody the ranges.  Also reduces the per-reference "has reads" bits.
constexpr uint64_t PEER_FAILED = 0xFFFFFFFFFFFFFFFDull;      // in the boundary table instead of a rank's smallest start: that rank stopped with an error
constexpr uint32_t SPARSE_PEER_FAILED = 1u << 16;            // the same in the sum of the sparse decision

// A rank that stops with an error before the boundary table has been gathered still joins that all-gather (or, on a -L run, the decision
// before it) and says so there: the other ranks then stop with an error of their own instead of waiting in the collective for ever (a
// refusal such as "reads of one name reach too far past a shard boundary" concerns one rank only).  Best effort: errors in here are ignored.
void abort_collectives(bdepth* h) {
    const int p = h->coll_pending; h->coll_pending = 0;
    if (!p || h->world <= 1 || !h->comm) return;
    NcclApi& N = nccl(); cudaStream_t sm = h->s_main;
    if (p == 2) {
        uint32_t flag = SPARSE_PEER_FAILED;
        if (h->misc.ensure(16) != cudaSuccess) return;
        cudaMemcpyAsync(h->misc.p, &flag, 4, cudaMemcpyHostToDevice, sm);
        N.AllReduce(h->misc.p, h->misc.p, 1, NCCL_UINT32, NCCL_SUM, h->comm, sm);
        cudaStreamSynchronize(sm);
        return;
    }
    DevBuf dpair, dall; if (dpair.ensure(16) != cudaSuccess || dall.ensure(16 * (size_t)h->world) != cudaSuccess) return;
    uint64_t mine[2] = {PEER_FAILED, 0};
    cudaMemcpyAsync(dpair.p, mine, 16, cudaMemcpyHostToDevice, sm);
    N.AllGather(dpair.p, dall.p, 2, NCCL_UINT64, h->comm, sm);
    cudaStreamSynchronize(sm);
    dpair.release(); dall.release();
}

int exchange_boundaries(bdepth* h, uint64_t shard_min, uint64_t shard_max, bool with_counters) {
    NcclApi& N = nccl(); cudaStream_t sm = h->s_main; const int W = h->world, me = h->rank;
    cudaEvent_t e0 = h->ev[12], e1 = h->ev[13];
    CK(cudaEventRecord(e0, sm));
    DevBuf dpair, dall; CK(dpair.ensure(16)); CK(dall.ensure(16 * (size_t)W));
    uint64_t mine[2] = {shard_min, shard_max};
    CK(cudaMemcpyAsync(dpair.p, mine, 16, cudaMemcpyHostToDevice, sm));
    NK(N.AllGather(dpair.p, dall.p, 2, NCCL_UINT64, h->comm, sm));
    h->coll_pending = 0;
    std::vector<uint64_t> all(2 * (size_t)W);
    CK(cudaMemcpyAsync(all.data(), dall.p, 16 * (size_t)W, cudaMemcpyDeviceToHost, sm));
    CK(cudaStreamSynchronize(sm));
    for (int r = 0; r < W; r++) if (all[2 * (size_t)r] == PEER_FAILED) return fail(h, BDEPTH_ERR_NCCL, "rank %d of the run stopped with an error (its own message says why): nothing was exchanged, no result", r);
    auto nonempty = [&](int r) { return all[2 * r] != UINT64_MAX; };
    auto own_lo = [&](int r) -> uint64_t { return r == 0 ? 0 : all[2 * r]; };      // rank 0 owns from 0 (whether it has reads or not): every rank knows where its own positions begin before it has heard of the others
    auto own_hi = [&](int r) -> uint64_t { for (int q = r + 1; q < W; q++) if (nonempty(q)) return all[2 * q]; return h->hdr.total_len; };
    struct Xfer { int peer; uint64_t lo, hi; };
    std::vector<Xfer> sends, recvs;
    // with_counters == false (plain shards without -m): every rank has counted the reads of the previous ranks' zone itself, so its own
    // positions are complete and only the table of boundaries is exchanged
    if (with_counters) {
    if (nonempty(me)) for (int j = me + 1; j < W; j++) if (nonempty(j) && all[2 * j] < shard_max) { uint64_t lo = std::max(all[2 * j], shard_min), hi = std::min(shard_max, own_hi(j)); if (lo < hi) sends.push_back({j, lo, hi}); }
    if (nonempty(me)) for (int i = 0; i < me; i++) if (nonempty(i) && all[2 * i + 1] > all[2 * me]) { uint64_t lo = std::max(all[2 * me], all[2 * i]), hi = std::min(all[2 * i + 1], own_hi(me)); if (lo < hi) recvs.push_back({i, lo, hi}); }
    }
    uint64_t tot = 0; for (auto& x : sends) tot += x.hi - x.lo; uint64_t sent = tot; for (auto& x : recvs) tot += x.hi - x.lo;
    const int NP = N_PLANES * (int)h->S;      // all counter planes of all samples
    DevBuf stage; CK(stage.ensure((size_t)std::max<uint64_t>(tot, 1) * NP * 4));
    uint32_t* sp = stage.as<uint32_t>(); uint64_t off = 0;
    std::vector<uint64_t> soff, roff;
    for (auto& x : sends) {   // pack the 7 planes of the slice contiguously
        uint64_t n = x.hi - x.lo; soff.push_back(off);
        // one copy per plane: a pitched 2D copy would need a source pitch of win_len * 4 bytes, which exceeds cudaDeviceProp::memPitch
        // (2^31 - 1) as soon as the references total more than ~536 Mbp -- and with several ranks the window is the whole genome
        for (int pl = 0; pl < NP; pl++) CK(cudaMemcpyAsync(sp + off + (uint64_t)pl * n, h->counts.as<uint32_t>() + (uint64_t)pl * h->win_len + (x.lo - h->cnt_base), n * 4, cudaMemcpyDeviceToDevice, sm));
        off += n * NP;
    }
    for (auto& x : recvs) { roff.push_back(off); off += (x.hi - x.lo) * NP; }
    NK(N.GroupStart());
    for (size_t i = 0; i < sends.size(); i++) NK(N.Send(sp + soff[i], (sends[i].hi - sends[i].lo) * NP, NCCL_UINT32, sends[i].peer, h->comm, sm));
    for (size_t i = 0; i < recvs.size(); i++) NK(N.Recv(sp + roff[i], (recvs[i].hi - recvs[i].lo) * NP, NCCL_UINT32, recvs[i].peer, h->comm, sm));
    NK(N.GroupEnd());
    for (size_t i = 0; i < recvs.size(); i++) {
        uint64_t n = recvs[i].hi - recvs[i].lo;
        for (int pl = 0; pl < NP; pl++) BD_LAUNCH((unsigned)((n + 255) / 256), 256, 0, sm, k_add_u32)(h->counts.as<uint32_t>() + (uint64_t)pl * h->win_len + (recvs[i].lo - h->cnt_base), sp + roff[i] + (uint64_t)pl * n, n);
        h->st.gpu_launches += NP;
    }
    // which references have reads: OR over ranks == (sum > 0)
    size_t nw = h->hdr.ref_len.size() / 32 + 2;
    DevBuf bits; CK(bits.ensure(nw * 32 * 4));
    {   // expand bits -> counts, all-reduce, compress back (tiny)
        std::vector<uint32_t> hb(nw); CK(cudaMemcpyAsync(hb.data(), h->ref_has.p, nw * 4, cudaMemcpyDeviceToHost, sm)); CK(cudaStreamSynchronize(sm));
        std::vector<uint32_t> ex(nw * 32); for (size_t i = 0; i < nw * 32; i++) ex[i] = (hb[i >> 5] >> (i & 31)) & 1;
        CK(cudaMemcpyAsync(bits.p, ex.data(), nw * 32 * 4, cudaMemcpyHostToDevice, sm));
        NK(N.AllReduce(bits.p, bits.p, nw * 32, NCCL_UINT32, NCCL_SUM, h->comm, sm));
        CK(cudaMemcpyAsync(ex.data(), bits.p, nw * 32 * 4, cudaMemcpyDeviceToHost, sm)); CK(cudaStreamSynchronize(sm));
        for (size_t i = 0; i < nw; i++) { uint32_t v = 0; for (int b = 0; b < 32; b++) if (ex[i * 32 + b]) v |= 1u << b; hb[i] = v; }
        CK(cudaMemcpyAsync(h->ref_has.p, hb.data(), nw * 4, cudaMemcpyHostToDevice, sm));
    }
    CK(cudaEventRecord(e1, sm)); CK(cudaStreamSynchronize(sm));
    float t = 0; CK(cudaEventElapsedTime(&t, e0, e1)); h->st.ms_exchange = t; h->st.halo_bytes_sent = sent * NP * 4;
    // ownership: an empty rank owns nothing
    if (nonempty(me) || me == 0) { h->own_lo = own_lo(me); h->own_hi = own_hi(me); } else { h->own_lo = h->own_hi = 0; }
    dpair.release(); dall.release(); stage.release(); bits.release();
    return 0;
}

// Build the sparse block list for the current regions.  Returns false when sparse staging does not apply (no
// regions, no usable index, several ranks, input staged as a whole) or would not save anything.
static bool plan_sparse(bdepth* h) {
    h->sparse_on = false;
    if (h->regions.empty() || !h->sparse_ok || (h->world != 1 && h->fix_mates) || h->staged || !h->bai.valid || h->bai.bins.size() != h->hdr.ref_len.size()) return false;
    const auto& P = h->blocks; if (P.empty()) return false;          // the framed prefix of the file: at least the header's members
    uint64_t vo_first;
    {   // a credible index starts where the records start (a dummy or foreign .bai is accepted by the reference, which only
        // checks that one exists, depth.d:1166 -- it must not make reads disappear here)
        uint64_t mn = UINT64_MAX; for (uint64_t v : h->bai.min_chunk_beg) mn = std::min(mn, v);
        size_t lo = 0, hi = P.size(); while (lo + 1 < hi) { size_t m = (lo + hi) / 2; if (P[m].uoff <= h->hdr.first_rec_off) lo = m; else hi = m; }
        vo_first = (P[lo].coff << 16) | (h->hdr.first_rec_off - P[lo].uoff);
        if (h->hdr.first_rec_off - P[lo].uoff >= P[lo].isize) vo_first = (P[lo].coff + P[lo].bsize) << 16;      // the first record begins the next member
        if (mn != vo_first) { h->sparse_ok = false; return false; }
    }
    std::vector<HostRegion> rg; rg.reserve(h->regions.size());
    for (auto& g : h->regions) rg.push_back(HostRegion{g.ref_id, g.start, g.end});
    std::vector<BaiChunk> cs = region_chunks(h->bai, rg);
    // The members the chunks touch: the handle's table when it already covers the whole file (every open but the lazy one), else framed
    // straight from the file as far as the chunks reach (sorted by offset; no need for the whole file's table).
    const bool have_all = h->framed_all;
    std::vector<HostBlock> Lown; const std::vector<HostBlock>& L = have_all ? P : Lown;
    bool file_end = have_all; uint64_t end_coff = have_all ? P.back().coff + P.back().bsize : 0;      // end_coff: offset after the last member once the end has been seen
    auto frame_to = [&](uint64_t from, uint64_t to) -> bool {       // make sure every member starting in [from, to] is in L; from must be a member start
        if (have_all) return true;
        std::vector<HostBlock>& L = Lown;
        if (from >= h->file_len) return true;
        size_t off = (size_t)from; uint64_t dummy = 0; bool eof = false;
        if (!L.empty() && L.back().coff >= from) { if (L.back().coff >= to) return true; off = (size_t)(L.back().coff + L.back().bsize); }
        else if (!L.empty() && L.back().coff + L.back().bsize > from) return false;       // begins inside a member framed before: not a member start
        std::vector<HostBlock> add; std::string e = frame_bgzf(h->file, h->file_len, &off, &dummy, SIZE_MAX, to, add, &eof);
        if (!e.empty()) return false;
        if (eof) { file_end = true; end_coff = off; }
        L.insert(L.end(), add.begin(), add.end());
        return true;
    };
    auto block_at = [&](uint64_t coff) -> long { if (L.empty()) return -1; size_t lo = 0, hi = L.size(); while (lo + 1 < hi) { size_t m = (lo + hi) / 2; if (L[m].coff <= coff) lo = m; else hi = m; } return L[lo].coff == coff ? (long)lo : -1; };
    struct Seg { size_t b0, b1; uint32_t entry, limit; };      // members L[b0..b1], entry inside b0, limit inside b1
    std::vector<Seg> segs;
    for (const BaiChunk& c : cs) {
        if (c.beg < vo_first) { h->sparse_ok = false; return false; }                        // the header's members are never part of a chunk
        if (!frame_to(c.beg >> 16, c.end >> 16)) { h->sparse_ok = false; return false; }      // the index does not describe this file
        long kb = block_at(c.beg >> 16), ke = block_at(c.end >> 16);
        uint32_t wb = (uint32_t)(c.beg & 0xFFFF), we = (uint32_t)(c.end & 0xFFFF);
        if (kb < 0) { if (file_end && (c.beg >> 16) >= end_coff) continue; h->sparse_ok = false; return false; }
        if (ke < 0) { if (file_end && (c.end >> 16) >= end_coff) { ke = (long)L.size() - 1; we = L.back().isize; } else { h->sparse_ok = false; return false; } }
        if (wb >= L[kb].isize) { kb++; wb = 0; if ((size_t)kb >= L.size()) continue; }      // "end of block" == start of the next one
        if (we == 0) { if (ke == 0) continue; ke--; we = L[ke].isize; }
        if (we > L[ke].isize) { h->sparse_ok = false; return false; }
        if (ke < kb || (ke == kb && we <= wb)) continue;
        if (!segs.empty() && (size_t)kb <= segs.back().b1) {         // touches the previous segment's last block: one segment
            if ((size_t)ke > segs.back().b1 || ((size_t)ke == segs.back().b1 && we > segs.back().limit)) { segs.back().b1 = (size_t)ke; segs.back().limit = we; }
            continue;
        }
        segs.push_back(Seg{(size_t)kb, (size_t)ke, wb, we});
    }
    uint64_t sel_bytes = 0; size_t nsel = 0; for (auto& sg : segs) for (size_t k = sg.b0; k <= sg.b1; k++) { sel_bytes += L[k].bsize; nsel++; }
    if (sel_bytes * 10 > (uint64_t)h->file_len * 9) return false;      // nearly the whole file: the plain path is simpler
    if (h->world > 1) {      // several ranks: consecutive segments (each begins and ends at a record) by compressed bytes; file order = coordinate order, so
        std::vector<Seg> mine; uint64_t cum = 0;                        // the ranks' reads still lie in consecutive coordinate ranges and the boundary exchange applies as it is
        for (auto& sg : segs) { uint64_t bytes = 0; for (size_t k = sg.b0; k <= sg.b1; k++) bytes += L[k].bsize; int owner = sel_bytes ? (int)std::min<uint64_t>((uint64_t)h->world - 1, (cum + bytes / 2) * (uint64_t)h->world / sel_bytes) : 0; if (owner == h->rank) mine.push_back(sg); cum += bytes; }
        segs.swap(mine); nsel = 0; for (auto& sg : segs) nsel += sg.b1 - sg.b0 + 1;
    }
    h->vblocks.clear(); h->seg_entry.clear(); h->seg_limit.clear();
    h->vblocks.reserve(nsel); h->seg_entry.reserve(nsel); h->seg_limit.reserve(nsel);
    uint64_t vu = 0;
    for (auto& sg : segs) for (size_t k = sg.b0; k <= sg.b1; k++) {
        HostBlock hb = L[k]; hb.uoff = vu; vu += hb.isize;
        h->vblocks.push_back(hb); h->seg_entry.push_back(k == sg.b0 ? (int32_t)sg.entry : -1); h->seg_limit.push_back(k == sg.b1 ? sg.limit : UINT32_MAX);
    }
    h->sparse_on = true;
    return true;
}

__global__ void k_scatter_i64(int64_t* __restrict__ dst, const uint32_t* __restrict__ idx, const int64_t* __restrict__ val, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) dst[idx[i]] = val[i];
}

struct RunOut {                    // optional sinks for the kernel-level entry points
    uint8_t* inflate_dst = nullptr; uint64_t inflate_cap = 0; uint64_t inflate_len = 0;
    uint64_t scan_cap = 0; uint64_t scan_n = 0;
    int32_t* ref_id = nullptr; int32_t* pos = nullptr; uint32_t* span = nullptr; uint16_t* flag = nullptr; uint8_t* mapq = nullptr; uint16_t* n_cigar = nullptr; uint64_t* rec_off = nullptr;
};

__global__ void k_fill_u32(uint32_t* p, uint32_t v, uint64_t n) { uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; if (i < n) p[i] = v; }

// The pipeline: leaves the per-position counters of the whole shard in h->counts (RUN_FULL).
int run_pipeline_body(bdepth* h, RunMode mode, RunOut* ro, Emitter* em);
int run_pipeline(bdepth* h, RunMode mode, RunOut* ro, Emitter* em = nullptr) {
    const int rc = run_pipeline_body(h, mode, ro, em);
    if (rc && rc != RC_RETRY_WINDOW) abort_collectives(h);      // (a nested run -- the restarts below -- has done that itself: nothing is pending then)
    return rc;
}
int run_pipeline_body(bdepth* h, RunMode mode, RunOut* ro, Emitter* em) {
    h->coll_pending = 0;
    int rc = init_device(h); if (rc) return rc;
    auto t_host0 = std::chrono::steady_clock::now();
    bdepth_stats& st = h->st; uint32_t launches0 = 0;
    st = bdepth_stats{}; st.gpu_launches = launches0;
    const bool sparse = mode == RUN_FULL && plan_sparse(h);
    h->coll_pending = (mode == RUN_FULL && h->world > 1 && h->comm) ? (sparse ? 2 : 1) : 0;
    if (!sparse) { rc = prepare_shard(h); if (rc) return rc; }      // the plain path needs the whole file's member table (a lazily opened handle frames it now)
    // -m pairs reads of one name wherever they sit in the shard.  A batch is scanned as a whole (no sub-batches), and every
    // batch after the first re-reads the end of the previous one as "ghost" records -- from the earliest record that can
    // still meet a mate (mates.cuh) -- so that a pair cut by a batch boundary is seen complete by the batch that closes it.
    const bool fix = mode == RUN_FULL && h->fix_mates;
    bool flt_uploaded = false;            // -L regions on the device for k_ref_seen (once per run)
    if (fix && h->world > 1 && !h->comm) return fail(h, BDEPTH_ERR_ARG, "fix-mate-overlaps on several ranks needs the boundary exchange (bdepth_set_shard with a NCCL id)");
    const uint64_t eff_batch_u = h->batch_u;
    size_t ghost_b = 0; int64_t ghost_entry = 0; uint64_t ghost_below_abs = 0, prev_s_last = 0, covered_from = 0;      // -m: where the next batch's stream begins
    const std::vector<HostBlock>& B = sparse ? h->vblocks : h->blocks;
    const size_t blk_lo = sparse ? 0 : h->blk_lo, blk_hi = sparse ? B.size() : h->blk_hi;
    const size_t nref = h->hdr.ref_len.size();
    cudaStream_t sm = h->s_main;

    // ---- counter window (28 B/position).  With a BAI the linear index bounds where reads can lie, so only that
    // span of the linear genome is allocated; without one the whole genome is (87 GB for GRCh38, fits 180 GB HBM).
    if (mode == RUN_FULL && h->accum) {
        // a further input of the same run: counters, window, sample planes stay as the first input left them
    } else if (mode == RUN_FULL) {
        uint64_t lo = 0, hi = h->hdr.total_len;
        if (h->force_window) { lo = h->cnt_base; hi = h->cnt_base + h->win_len; }
        else
        if (h->bai.valid && h->bai_window_ok && h->bai.ioffsets.size() == nref && h->world > 1 && !sparse && !fix && blk_hi > blk_lo) {
            // a shard: from the window in which its first record begins (its own positions begin there or later) to the end of the last
            // 16 kbp window that any read before the shard's end overlaps (the linear index holds, per window, the first such read)
            const uint64_t vo_end = blk_hi < B.size() ? (B[blk_hi].coff << 16) : (h->file_len << 16);
            lo = h->rank == 0 ? UINT64_MAX : h->zone_lin_lo; hi = 0;
            for (size_t r = 0; r < nref; r++) {
                const auto& v = h->bai.ioffsets[r];
                for (size_t k = 0; k < v.size(); k++) if (v[k] && v[k] < vo_end) {
                    const uint64_t a = h->hdr.ref_lin0[r] + std::min<uint64_t>((uint64_t)k << 14, h->hdr.ref_len[r]), e = h->hdr.ref_lin0[r] + std::min<uint64_t>((uint64_t)(k + 1) << 14, h->hdr.ref_len[r]);
                    if (h->rank == 0) lo = std::min(lo, a);
                    if (e > hi) hi = e;
                }
            }
            if (lo == UINT64_MAX || lo >= hi) { lo = 0; hi = h->hdr.total_len; }
        } else if (h->bai.valid && h->bai_window_ok && h->bai.ioffsets.size() == nref && h->world == 1) {
            lo = UINT64_MAX; hi = 0;
            for (size_t r = 0; r < nref; r++) {
                const auto& v = h->bai.ioffsets[r]; if (v.empty()) continue;
                size_t k = 0; while (k < v.size() && v[k] == 0) k++;
                if (k == v.size()) continue;
                lo = std::min<uint64_t>(lo, h->hdr.ref_lin0[r] + std::min<uint64_t>((uint64_t)k << 14, h->hdr.ref_len[r]));
                hi = std::max<uint64_t>(hi, h->hdr.ref_lin0[r] + std::min<uint64_t>((uint64_t)v.size() << 14, h->hdr.ref_len[r]));
            }
            if (lo >= hi) { lo = 0; hi = h->hdr.total_len; }      // an index without linear entries says nothing
        }
        if (!h->force_window) {
            h->cnt_base = lo / TILE_POS * TILE_POS;
            h->win_len = ((hi - h->cnt_base + TILE_POS - 1) / TILE_POS + 1) * TILE_POS;
        }
        if (h->pass_n) h->S = h->pass_n;
        else {
            h->S = (h->combined || h->hdr.sample_names.size() <= 1) ? 1u : (uint32_t)h->hdr.sample_names.size();
            // (region and window runs with more samples count them a group at a time, run_segments)
            if (h->S > 64) return fail(h, BDEPTH_ERR_ARG, "%u samples: per-base output holds every sample's counters at once and supports at most 64 (use --combined, or depth region / depth window, which take any number of samples)", h->S);
        }
        size_t need = (size_t)h->win_len * N_PLANES * 4 * h->S;
        size_t free_b = 0, tot_b = 0; CK(cudaMemGetInfo(&free_b, &tot_b));
        if (need > h->counts.cap && need > free_b + h->counts.cap) return fail(h, BDEPTH_ERR_CUDA, "counter window needs %zu bytes of HBM, %zu free", need, free_b);
        CK(h->counts.ensure(need));
        CK(cudaMemsetAsync(h->counts.p, 0, need, sm));
        if (h->want_presence) { CK(h->present.ensure((h->win_len / 32 + 2) * 4)); CK(cudaMemsetAsync(h->present.p, 0, (h->win_len / 32 + 2) * 4, sm)); }
        CK(h->ref_has.ensure((nref / 32 + 2) * 4)); CK(cudaMemsetAsync(h->ref_has.p, 0, (nref / 32 + 2) * 4, sm));
    }
    CK(h->scan_stats.ensure(sizeof(ScanStats)));
    const FilterProg* d_fprog = nullptr;
    if (h->has_fprog) { CK(h->fprog_d.ensure(sizeof(FilterProg))); CK(cudaMemcpyAsync(h->fprog_d.p, &h->fprog, sizeof(FilterProg), cudaMemcpyHostToDevice, sm)); CK(cudaStreamSynchronize(sm)); d_fprog = h->fprog_d.as<FilterProg>(); }
    RgTable rgt{nullptr, nullptr, nullptr, nullptr, 0, 0, 0};
    h->pass_untagged = false;
    if (mode == RUN_FULL && (h->S > 1 || h->pass_n || (fix && h->hdr.sample_names.size() > 1))) {      // @RG ID -> sample table for the per-read RG lookup (depth.d:240-250); mates pair within a sample
        // a sample pass maps the read groups of its samples to pass-local ids and every other one to RG_OTHER
        auto local = [&](uint32_t s) -> uint16_t { return !h->pass_n ? (uint16_t)s : s - h->pass_g0 < h->pass_n ? (uint16_t)(s - h->pass_g0) : RG_OTHER; };
        const size_t n_rg = h->hdr.rg_ids.size();
        if (n_rg >= RG_OTHER) return fail(h, BDEPTH_ERR_ARG, "%zu read groups: at most %u are supported", n_rg, (unsigned)RG_OTHER - 1);
        std::vector<uint8_t> ids; std::vector<uint32_t> offs; std::vector<uint16_t> samp;
        for (size_t g = 0; g < n_rg; g++) { offs.push_back((uint32_t)ids.size()); ids.insert(ids.end(), h->hdr.rg_ids[g].begin(), h->hdr.rg_ids[g].end()); ids.push_back(0); samp.push_back(local((uint32_t)h->hdr.rg_sample[g])); }
        uint32_t slots = 2; while (slots < 2 * n_rg) slots *= 2;
        std::vector<uint32_t> tab(slots, 0);
        for (size_t g = 0; g < n_rg; g++) {      // (an ID that occurs twice keeps its first line, as the linear scan it replaces did)
            const std::string& id = h->hdr.rg_ids[g]; uint32_t hs = FNV1A_INIT; for (char c : id) hs = fnv1a_step(hs, (uint8_t)c);
            uint32_t k = hs & (slots - 1);
            while (tab[k] && h->hdr.rg_ids[tab[k] - 1] != id) k = (k + 1) & (slots - 1);
            if (!tab[k]) tab[k] = (uint32_t)g + 1;
        }
        CK(h->rg_ids.ensure(ids.size() + 8)); CK(h->rg_offs.ensure(offs.size() * 4 + 8)); CK(h->rg_samp.ensure(samp.size() * 2 + 8)); CK(h->rg_hash.ensure(slots * 4));
        if (n_rg) { CK(cudaMemcpyAsync(h->rg_ids.p, ids.data(), ids.size(), cudaMemcpyHostToDevice, sm)); CK(cudaMemcpyAsync(h->rg_offs.p, offs.data(), offs.size() * 4, cudaMemcpyHostToDevice, sm)); CK(cudaMemcpyAsync(h->rg_samp.p, samp.data(), samp.size() * 2, cudaMemcpyHostToDevice, sm)); }
        CK(cudaMemcpyAsync(h->rg_hash.p, tab.data(), slots * 4, cudaMemcpyHostToDevice, sm));
        rgt = RgTable{h->rg_ids.as<uint8_t>(), h->rg_offs.as<uint32_t>(), h->rg_samp.as<uint16_t>(), h->rg_hash.as<uint32_t>(), slots - 1, (uint32_t)n_rg, local(0)};
        CK(h->rg_tab.ensure(sizeof(RgTable))); CK(cudaMemcpyAsync(h->rg_tab.p, &rgt, sizeof(RgTable), cudaMemcpyHostToDevice, sm));
        CK(cudaStreamSynchronize(sm));
    }
    const RgTable* d_rgt = rgt.n_rg ? h->rg_tab.as<RgTable>() : nullptr;
    { uint64_t shard_u = blk_hi > blk_lo ? B[blk_hi - 1].uoff + B[blk_hi - 1].isize - B[blk_lo].uoff : 0; CK(h->ubuf.ensure(CARRY_MAX + std::min<uint64_t>(eff_batch_u + 65536, shard_u) + 256)); }
    CK(h->misc.ensure(64));
    HostScratch& hs = h->hs;
    // up(): host words -> device buffer; down(): device words -> mapped host memory, readable after the next
    // synchronisation of the main stream.  Both are stream-ordered kernels on the main stream.
    auto up = [&](void* dst_dev, const void* src, size_t bytes) -> int {
        if (!bytes) return 0;
        uint8_t* m = hs.take(bytes); if (!m) return fail(h, BDEPTH_ERR_CUDA, "internal: host scratch exhausted");
        memcpy(m, src, bytes);
        BD_LAUNCH((unsigned)std::min<size_t>((bytes / 4 + 255) / 256, 512), 256, 0, sm, k_copy_words)((uint32_t*)dst_dev, (const uint32_t*)hs.dev(m), bytes / 4);
        st.gpu_launches++;
        return 0;
    };
    auto down = [&](const void* src_dev, size_t bytes) -> uint8_t* {
        uint8_t* m = hs.take(bytes ? bytes : 4); if (!m) return nullptr;
        if (bytes) { BD_LAUNCH((unsigned)std::min<size_t>((bytes / 4 + 255) / 256, 512), 256, 0, sm, k_copy_words)((uint32_t*)hs.dev(m), (const uint32_t*)src_dev, bytes / 4); st.gpu_launches++; }
        return m;
    };
#define UP(dst, src, bytes) do { int rcu_ = up((dst), (src), (bytes)); if (rcu_) return rcu_; } while (0)
#define DOWN(var, type, src, bytes) type* var = (type*)down((src), (bytes)); if (!var) return fail(h, BDEPTH_ERR_CUDA, "internal: host scratch exhausted")

    float ms_h2d = 0, ms_k1 = 0, ms_k2 = 0, ms_k3 = 0;
    uint64_t carry_len = 0; bool first_batch = true;
    bool sparse_bad = false;         // a region chunk's record chain did not end at the chunk end (several ranks: decided together after the batches)
    uint64_t shard_min = UINT64_MAX, shard_max = 0;
    if (mode == RUN_INDEX) {      // tables of k_index_scan: one linear-index row per reference (16 kbp windows up to one past the reference end), counters, carry
        auto& X = h->ix; X.base.assign(nref + 1, 0); X.cap.assign(nref + 1, 0); uint64_t acc = 0;
        for (size_t r = 0; r < nref; r++) { X.base[r] = (uint32_t)acc; X.cap[r] = (uint32_t)std::min<uint64_t>(32769, ((uint64_t)h->hdr.ref_len[r] >> 14) + 2); acc += X.cap[r]; if (acc > 0xFFFFFFF0ull) return fail(h, BDEPTH_ERR_ARG, "too many references for the linear index tables"); }
        X.n_lin = acc; X.h_runs.clear(); X.h_excs.clear();
        CK(X.lin.ensure((acc + 1) * 8)); CK(X.lin_len.ensure((nref + 1) * 4)); CK(X.lin_base.ensure((nref + 1) * 4)); CK(X.lin_cap.ensure((nref + 1) * 4));
        CK(X.n_mapped.ensure((nref + 1) * 8)); CK(X.n_unmapped.ensure((nref + 1) * 8)); CK(X.carry.ensure(sizeof(IndexCarry))); CK(X.ctl.ensure(sizeof(IndexCtl)));
        CK(cudaMemsetAsync(X.lin.p, 0xFF, (acc + 1) * 8, sm)); CK(cudaMemsetAsync(X.lin_len.p, 0, (nref + 1) * 4, sm)); CK(cudaMemsetAsync(X.n_mapped.p, 0, (nref + 1) * 8, sm)); CK(cudaMemsetAsync(X.n_unmapped.p, 0, (nref + 1) * 8, sm));
        CK(cudaMemsetAsync(X.carry.p, 0, sizeof(IndexCarry), sm));
        CK(cudaMemcpyAsync(X.lin_base.p, X.base.data(), (nref + 1) * 4, cudaMemcpyHostToDevice, sm)); CK(cudaMemcpyAsync(X.lin_cap.p, X.cap.data(), (nref + 1) * 4, cudaMemcpyHostToDevice, sm));
        IndexCtl c0{0, 0, 0, ~0ull, ~0ull, 0, ~0ull, 0};
        CK(cudaMemcpyAsync(X.ctl.p, &c0, sizeof c0, cudaMemcpyHostToDevice, sm)); CK(cudaStreamSynchronize(sm));
    }
    CK(cudaEventRecord(h->ev[10], sm));
    size_t b = blk_lo;
    if (ro) { ro->inflate_len = 0; ro->scan_n = 0; }
    if (!h->staged) {   // size both compressed-data buffers for the largest batch up front (ensure() must not reallocate mid-flight)
        uint64_t mx = 0;
        for (size_t bb = blk_lo; bb < blk_hi;) {
            size_t e = bb; uint64_t u = 0, cb = 0; while (e < blk_hi && (e == bb || u + B[e].isize <= eff_batch_u)) { u += B[e].isize; cb += B[e].bsize; e++; }
            mx = std::max<uint64_t>(mx, sparse ? cb + 8 : B[e - 1].coff + B[e - 1].bsize - (B[bb].coff & ~3ull)); bb = e;
        }
        CK(h->comp2[0].ensure(mx + 256)); CK(h->comp2[1].ensure(mx + 256));
    }
    size_t batch_no = 0;
    auto batch_end = [&](size_t bb) { size_t e = bb; uint64_t u = 0; while (e < blk_hi && (e == bb || u + B[e].isize <= eff_batch_u)) { u += B[e].isize; e++; } return e; };
    // H2D of blocks [bb, be) into comp2[slot]; waits until K1 of the batch that used the slot two batches ago is done
    const size_t H2D_CHUNK_BLOCKS = h->chunk_blocks;
    // dco[slot][i] = where block bb+i of the batch sits in comp2[slot].  Plain runs keep the file layout (one copy
    // per chunk); sparse runs pack the selected blocks back to back (one copy per run of file-adjacent blocks).
    std::vector<uint64_t> dco[2];
    auto issue_h2d = [&](size_t no, size_t bb, size_t be) -> int {
        int slot = (int)(no & 1);
        uint64_t g0 = B[bb].coff & ~3ull;
        if (no >= 2) CK(cudaStreamWaitEvent(h->s_copy, h->ev[16 + slot], 0));
        CK(cudaEventRecord(h->ev[18 + slot], h->s_copy));
        h->chunk_end[slot].clear();
        dco[slot].resize(be - bb);
        { uint64_t acc = 0; for (size_t i = bb; i < be; i++) { dco[slot][i - bb] = sparse ? acc : B[i].coff - g0; acc += B[i].bsize; } }
        size_t nch = 0;
        for (size_t c0 = bb; c0 < be; c0 += H2D_CHUNK_BLOCKS, nch++) {
            size_t c1 = std::min(be, c0 + H2D_CHUNK_BLOCKS);
            uint64_t dev_end;
            if (!sparse) {
                uint64_t a = c0 == bb ? g0 : B[c0].coff, e = B[c1 - 1].coff + B[c1 - 1].bsize;
                CK(cudaMemcpyAsync((uint8_t*)h->comp2[slot].p + (a - g0), h->file + a, e - a, cudaMemcpyHostToDevice, h->s_copy));
                dev_end = e - g0;
            } else {
                for (size_t r0 = c0; r0 < c1;) {
                    size_t r1 = r0 + 1; while (r1 < c1 && B[r1].coff == B[r1 - 1].coff + B[r1 - 1].bsize) r1++;
                    CK(cudaMemcpyAsync((uint8_t*)h->comp2[slot].p + dco[slot][r0 - bb], h->file + B[r0].coff, B[r1 - 1].coff + B[r1 - 1].bsize - B[r0].coff, cudaMemcpyHostToDevice, h->s_copy));
                    r0 = r1;
                }
                dev_end = dco[slot][c1 - 1 - bb] + B[c1 - 1].bsize;
            }
            if (c1 == be) CK(cudaMemsetAsync((uint8_t*)h->comp2[slot].p + dev_end, 0, 128, h->s_copy));
            if (h->chunk_ev[slot].size() <= nch) { cudaEvent_t ne; CK(cudaEventCreateWithFlags(&ne, cudaEventDisableTiming)); h->chunk_ev[slot].push_back(ne); }
            CK(cudaEventRecord(h->chunk_ev[slot][nch], h->s_copy));
            h->chunk_end[slot].push_back(c1);
        }
        CK(cudaEventRecord(h->ev[14 + slot], h->s_copy));
        return 0;
    };
    while (b < blk_hi) {
        // ---- batch extent
        size_t b1 = b; uint64_t ub_new = 0;
        while (b1 < blk_hi && (b1 == b || ub_new + B[b1].isize <= eff_batch_u)) { ub_new += B[b1].isize; b1++; }
        const bool last_batch = b1 == blk_hi;
        st.n_batches++; st.n_blocks += b1 - b; st.inflated_bytes += ub_new;
        const size_t new_b = b;                                                          // first block that has not been scanned yet
        const size_t stream_b = (fix && batch_no > 0) ? std::min(ghost_b, b) : b;          // -m: the batch's stream begins with re-read blocks
        {   // from here to the end of the sub-batch loop `b` is the first block of the batch's stream
        const size_t b = stream_b;
        const size_t nb = b1 - b;
        const uint64_t batch_u0 = B[b].uoff;               // absolute inflated offset of the batch start
        const uint64_t ub = B[b1 - 1].uoff + B[b1 - 1].isize - batch_u0;
        // ---- compressed bytes on the device: H2D runs on the copy stream into one of two buffers, so the copy of
        // batch i+1 overlaps the kernels of batch i
        const uint32_t* d_comp;
        cudaEvent_t e0 = h->ev[0], e1 = h->ev[1], e2 = h->ev[2], e3 = h->ev[3], e4 = h->ev[4];
        CK(cudaEventRecord(e0, sm));
        if (h->staged) d_comp = h->comp.as<uint32_t>();
        else {
            if (fix) {       // no prefetch: where a batch begins is only known when the previous one has been scanned
                uint64_t need = 8; if (sparse) for (size_t i = b; i < b1; i++) need += B[i].bsize; else need = B[b1 - 1].coff + B[b1 - 1].bsize - (B[b].coff & ~3ull);
                CK(h->comp2[batch_no & 1].ensure(need + 256));
                int rcp = issue_h2d(batch_no, b, b1); if (rcp) return rcp;
            } else if (batch_no == 0) { int rcp = issue_h2d(0, b, b1); if (rcp) return rcp; }
            d_comp = h->comp2[batch_no & 1].as<uint32_t>();
        }
        // ---- descriptors
        std::vector<BlockDesc> d(nb); uint64_t csum = 0, tok_words = 0;
        for (size_t i = 0; i < nb; i++) {
            const HostBlock& hb = B[b + i];
            uint64_t dev_off = h->staged ? hb.coff - h->staged_file_off : dco[batch_no & 1][i];
            d[i] = BlockDesc{dev_off + hb.cdata_off, hb.uoff - batch_u0, hb.csize, hb.isize, tok_words};
            tok_words += tok_cap_of(hb.isize);
            if (b + i >= new_b) { csum += hb.csize; st.file_bytes += hb.bsize; }
        }
        st.cdata_bytes += csum;
        CK(h->descs.ensure(nb * sizeof(BlockDesc))); CK(h->status.ensure(nb * sizeof(int))); CK(h->ubuf.ensure(CARRY_MAX + ub + 256));
        if (!h->k1_onephase) { CK(h->tok.ensure(tok_words * 4 + 64)); CK(h->lits.ensure(ub + 16 * nb + 64)); CK(h->aux.ensure(nb * sizeof(BlockAux))); CK(h->segi.ensure(nb * MAX_SEG * 4)); CK(h->littab.ensure(nb * (size_t)MAX_SEG * 256)); }
        CK(hs.ensure(nb * (sizeof(BlockDesc) + 192) + 16384)); hs.used = 0;      // nothing is in flight here: every sub-batch ends synchronised
        UP(h->descs.p, d.data(), nb * sizeof(BlockDesc));
        uint8_t* u0 = h->ubuf.as<uint8_t>() + CARRY_MAX;     // offset 0 of this batch's inflated bytes
        CK(cudaEventRecord(e1, sm));
        struct Sub { size_t s0, s1; int ev_lo, ev_hi; };     // blocks [s0, s1) are inflated once k1_ev[ev_lo..ev_hi] have fired
        std::vector<Sub> subs;
        // ---- K1: when the input is streaming in, one sub-launch per H2D chunk, spread over a few streams so that
        // they run side by side (a lone sub-launch cannot fill the GPU: every lane owns a whole BGZF block)
        // K1 of blocks [c0, c0 + n) of the batch on stream ks: the two-phase inflater (k1_huff, k1_lz) and the exact one-phase kernel
        // for whatever phase 1 handed back (normally nothing: it returns at once); BDEPTH_K1_ONEPHASE=1 runs the round-1 kernel alone (A/B)
        auto launch_k1 = [&](cudaStream_t ks, size_t c0, uint32_t n) -> int {
            const BlockDesc* dd = h->descs.as<BlockDesc>() + (c0 - b); int* stp = h->status.as<int>() + (c0 - b);
            if (h->k1_onephase) {
                BD_LAUNCH((n + 32 * K1_WARPS - 1) / (32 * K1_WARPS), 32 * K1_WARPS, K1_SMEM, ks, k1_inflate)(d_comp, dd, n, u0, stp);
                CK(cudaGetLastError()); st.gpu_launches++;
                return 0;
            }
            BlockAux* ax = h->aux.as<BlockAux>() + (c0 - b); uint32_t* sgi = h->segi.as<uint32_t>() + (c0 - b) * MAX_SEG; uint8_t* ltb = h->littab.as<uint8_t>() + (c0 - b) * (size_t)MAX_SEG * 256;
            const unsigned hg = (n + 32 * K1H_WARPS - 1) / (32 * K1H_WARPS); const uint32_t blk0 = (uint32_t)(c0 - b);
#define K1H(LIMS, MINB) BD_LAUNCH(hg, 32 * K1H_WARPS, k1h_smem<LIMS>(), ks, k1_huff<LIMS, MINB>)(d_comp, dd, n, blk0, stp, h->tok.as<uint32_t>(), h->lits.as<uint8_t>(), ax, sgi, ltb)
            // which instantiation: limits in registers at 4 CTAs per SM (16 warps) is the faster loop; when a launch has more warps than that
            // holds at once, limits in shared memory at 5 CTAs (20 warps) wins by its occupancy (profiles/k1_history.md)
            const int variant = h->k1h_variant >= 0 ? h->k1h_variant : (n > 148u * 16u * 32u ? 2 : 0);
            switch (variant) { case 1: K1H(false, 6); break; case 2: K1H(true, 5); break; case 3: K1H(true, 4); break; default: K1H(false, 4); }
#undef K1H
            if (h->k1lz_flat) BD_LAUNCH((n + K1L_WARPS - 1) / K1L_WARPS, 32 * K1L_WARPS, 0, ks, k1_lz_flat)(dd, n, blk0, u0, stp, h->tok.as<uint32_t>(), h->lits.as<uint8_t>(), ax, sgi, ltb);
            else if (h->k1lz_v12) BD_LAUNCH((n + K1L_WARPS - 1) / K1L_WARPS, 32 * K1L_WARPS, 0, ks, k1_lz<false>)(dd, n, blk0, u0, stp, h->tok.as<uint32_t>(), h->lits.as<uint8_t>(), ax, sgi, ltb);
            else BD_LAUNCH((n + K1L_WARPS - 1) / K1L_WARPS, 32 * K1L_WARPS, 0, ks, k1_lz<true>)(dd, n, blk0, u0, stp, h->tok.as<uint32_t>(), h->lits.as<uint8_t>(), ax, sgi, ltb);
            BD_LAUNCH((n + 32 * K1_WARPS - 1) / (32 * K1_WARPS), 32 * K1_WARPS, K1_SMEM, ks, k1_fallback)(d_comp, dd, n, u0, stp);
            CK(cudaGetLastError()); st.gpu_launches += 3;
            return 0;
        };
        if (h->staged) {
            { int rck = launch_k1(sm, b, (uint32_t)nb); if (rck) return rck; }
            subs.push_back(Sub{b, b1, 0, -1});
        } else {
            int slot = (int)(batch_no & 1); size_t c0 = b;
            for (size_t j = 0; j < h->chunk_end[slot].size(); j++) {
                size_t c1 = h->chunk_end[slot][j]; cudaStream_t ks = h->s_k1[j & 15];
                CK(cudaStreamWaitEvent(ks, e1, 0)); CK(cudaStreamWaitEvent(ks, h->chunk_ev[slot][j], 0));
                uint32_t n = (uint32_t)(c1 - c0);
                { int rck = launch_k1(ks, c0, n); if (rck) return rck; }
                if (h->k1_ev.size() <= j) { cudaEvent_t ne; CK(cudaEventCreateWithFlags(&ne, cudaEventDisableTiming)); h->k1_ev.push_back(ne); }
                CK(cudaEventRecord(h->k1_ev[j], ks));
                // Sub-batches: a lane needs ~60 ms for its block however empty the GPU is, so the scan / coverage /
                // delivery of the blocks that arrived first runs while the later chunks are still being inflated.
                if ((mode == RUN_FULL || mode == RUN_INDEX) && !fix) subs.push_back(Sub{c0, c1, (int)j, (int)j}); else { if (subs.empty()) subs.push_back(Sub{b, b1, 0, (int)j}); subs[0].ev_hi = (int)j; }
                c0 = c1;
            }
        }
        if (!h->staged && !fix && b1 < blk_hi) { int rcp = issue_h2d(batch_no + 1, b1, batch_end(b1)); if (rcp) return rcp; }
        const size_t mb = b, mb1 = b1; const uint64_t m_u0abs = batch_u0; uint8_t* const m_u0 = u0; const bool m_last = last_batch;
        for (size_t sbi = 0; sbi < subs.size(); sbi++) {
        const size_t b = subs[sbi].s0, b1 = subs[sbi].s1, nb = b1 - b;                  // from here on: the sub-batch
        const uint64_t batch_u0 = B[b].uoff, ub = B[b1 - 1].uoff + B[b1 - 1].isize - batch_u0;
        uint8_t* const u0 = m_u0 + (batch_u0 - m_u0abs);
        const bool last_sub = sbi + 1 == subs.size(), last_batch = m_last && last_sub;
        for (int j = subs[sbi].ev_lo; j <= subs[sbi].ev_hi; j++) CK(cudaStreamWaitEvent(sm, h->k1_ev[j], 0));
        CK(cudaEventRecord(e2, sm));
        if (!h->staged && last_sub) CK(cudaEventRecord(h->ev[16 + (batch_no & 1)], sm));     // this batch's compressed buffer is free again
        DOWN(stt, int, h->status.as<int>() + (b - mb), nb * sizeof(int));
        if (mode == RUN_INFLATE_ONLY) {
            CK(cudaStreamSynchronize(sm));
            for (size_t i = 0; i < nb; i++) if (stt[i]) return fail(h, BDEPTH_ERR_FORMAT, "DEFLATE error %d in BGZF block at offset %llu", stt[i], (unsigned long long)B[b + i].coff);
            if (ro && ro->inflate_dst) {
                if (ro->inflate_len + ub > ro->inflate_cap) return fail(h, BDEPTH_ERR_ARG, "inflate buffer too small");
                CK(cudaMemcpy(ro->inflate_dst + ro->inflate_len, u0, ub, cudaMemcpyDeviceToHost));
            }
            if (ro) ro->inflate_len += ub;
            float t; CK(cudaEventElapsedTime(&t, e1, e2)); ms_k1 += t;
            continue;
        }
        // ---- K2: chunk table
        const bool seg0 = sparse && h->seg_entry[b] >= 0;      // the sub-batch begins a new region-query chunk: nothing is carried into it
        if (seg0) carry_len = 0;
        std::vector<int64_t> cstart(nb + 1); std::vector<uint32_t> sbase(nb + 1);
        { uint64_t acc = 0; for (size_t i = 0; i < nb; i++) { cstart[i] = (int64_t)(B[b + i].uoff - batch_u0); sbase[i] = (uint32_t)acc; uint64_t sz = B[b + i].isize + (i == 0 ? carry_len : 0); acc += sz / 36 + 2; } cstart[nb] = (int64_t)ub; sbase[nb] = (uint32_t)acc; cstart[0] = -(int64_t)carry_len;
          if (acc > 0xFFFFFFFFull) return fail(h, BDEPTH_ERR_ARG, "batch too large"); }
        const uint64_t n_slots = sbase[nb];
        CK(h->chunk_start.ensure((nb + 1) * 8)); CK(h->slot_base.ensure((nb + 1) * 4)); CK(h->entry.ensure(nb * 8)); CK(h->exitb.ensure(nb * 8)); CK(h->count.ensure(nb * 4)); CK(h->rec_base.ensure((nb + 1) * 4)); CK(h->slots.ensure(n_slots * 2 + 64)); CK(h->walk_list.ensure(64));
        UP(h->chunk_start.p, cstart.data(), (nb + 1) * 8);
        UP(h->slot_base.p, sbase.data(), (nb + 1) * 4);
        CK(cudaMemsetAsync(h->entry.p, ENTRY_NONE_BYTE, nb * 8, sm));
        // (-m: a stream that begins exactly where a region-query chunk begins starts at that chunk's first record)
        int64_t anchor = (fix && batch_no > 0) ? ((seg0 && ghost_entry < (int64_t)h->seg_entry[b]) ? (int64_t)h->seg_entry[b] : ghost_entry) : seg0 ? (int64_t)h->seg_entry[b] : first_batch ? h->entry0 : -(int64_t)carry_len;
        UP(h->entry.p, &anchor, 8);
        CK(cudaMemsetAsync(h->misc.p, 0, 64, sm));
        // records that START at or after the shard limit belong to the next rank
        int64_t u_limit = (int64_t)ub; if (!sparse && h->limit_abs_u < batch_u0 + ub) u_limit = (int64_t)h->limit_abs_u - (int64_t)batch_u0;      // may be negative: the limit lies before this sub-batch, and a carried record that starts at or after it is not ours either
        ScanParams sp{u0, -(int64_t)carry_len, (int64_t)ub, (int)nref, h->ref_len_d.as<uint32_t>(), h->ref_lin0_d.as<uint64_t>()};
        BD_LAUNCH((unsigned)((nb * 32 + 255) / 256), 256, 0, sm, k2_guess_entries)(sp, h->chunk_start.as<int64_t>(), (uint32_t)nb, h->entry.as<int64_t>());
        CK(cudaGetLastError()); st.gpu_launches++;
        const int64_t* d_limit = nullptr;
        if (sparse) {       // chunks of the region query: exact entries at their first blocks, walk limits at their last ones
            std::vector<uint32_t> ai; std::vector<int64_t> av; std::vector<int64_t> lim(nb, INT64_MAX);
            for (size_t i = 0; i < nb; i++) {
                if (i && h->seg_entry[b + i] >= 0) { ai.push_back((uint32_t)i); av.push_back(cstart[i] + h->seg_entry[b + i]); }
                if (h->seg_limit[b + i] != UINT32_MAX) lim[i] = (i ? cstart[i] : 0) + (int64_t)h->seg_limit[b + i];
            }
            CK(h->chunk_limit.ensure(nb * 8)); UP(h->chunk_limit.p, lim.data(), nb * 8); d_limit = h->chunk_limit.as<int64_t>();
            if (!ai.empty()) {
                CK(h->anchors_idx.ensure(ai.size() * 4)); CK(h->anchors_val.ensure(av.size() * 8));
                UP(h->anchors_idx.p, ai.data(), ai.size() * 4); UP(h->anchors_val.p, av.data(), av.size() * 8);
                BD_LAUNCH((unsigned)((ai.size() + 255) / 256), 256, 0, sm, k_scatter_i64)(h->entry.as<int64_t>(), h->anchors_idx.as<uint32_t>(), h->anchors_val.as<int64_t>(), (uint32_t)ai.size());
                CK(cudaGetLastError()); st.gpu_launches++;
            }
        }
        ScanParams spw = sp;
        BD_LAUNCH((unsigned)((nb + 127) / 128), 128, 0, sm, k2_walk)(spw, h->chunk_start.as<int64_t>(), (uint32_t)nb, h->entry.as<int64_t>(), h->slot_base.as<uint32_t>(), h->slots.as<uint16_t>(), h->count.as<uint32_t>(), h->exitb.as<int64_t>(), (int*)h->misc.p, nullptr, 0, d_limit);
        CK(cudaGetLastError()); st.gpu_launches++;
        DOWN(ent, int64_t, h->entry.p, nb * 8); DOWN(ext, int64_t, h->exitb.p, nb * 8); DOWN(cnt, uint32_t, h->count.p, nb * 4);      // host-owned once synchronised
        DOWN(werr, int, h->misc.p, 4);
        CK(cudaStreamSynchronize(sm));
        int walk_err = *werr;
        for (size_t i = 0; i < nb; i++) if (stt[i]) return fail(h, BDEPTH_ERR_FORMAT, "DEFLATE error %d in BGZF block at offset %llu", stt[i], (unsigned long long)B[b + i].coff);
        // ---- exact chain verification (host, control plane): entry[i] must equal the running exit
        int64_t cur = anchor; int64_t tail = (int64_t)ub;
        for (size_t i = 0; i < nb; i++) {
            if (sparse && i && h->seg_entry[b + i] >= 0) cur = cstart[i] + h->seg_entry[b + i];     // a new chunk: the chain restarts at its first record
            int64_t true_e = (cur < cstart[i + 1]) ? cur : ENTRY_NONE;
            if (true_e != ENTRY_NONE && true_e < cstart[i]) return fail(h, BDEPTH_ERR_FORMAT, "internal: record chain went backwards");
            if (ent[i] != true_e) {
                st.chain_fixups++;
                uint32_t ci = (uint32_t)i;
                UP((int64_t*)h->entry.p + i, &true_e, 8);
                UP(h->walk_list.p, &ci, 4);
                BD_LAUNCH(1, 32, 0, sm, k2_walk)(spw, h->chunk_start.as<int64_t>(), (uint32_t)nb, h->entry.as<int64_t>(), h->slot_base.as<uint32_t>(), h->slots.as<uint16_t>(), h->count.as<uint32_t>(), h->exitb.as<int64_t>(), (int*)h->misc.p, h->walk_list.as<uint32_t>(), 1, d_limit);
                CK(cudaGetLastError()); st.gpu_launches++;
                DOWN(fx_ext, int64_t, (int64_t*)h->exitb.p + i, 8); DOWN(fx_cnt, uint32_t, (uint32_t*)h->count.p + i, 4); DOWN(fx_err, int, h->misc.p, 4);
                CK(cudaStreamSynchronize(sm));
                ext[i] = *fx_ext; cnt[i] = *fx_cnt; walk_err = *fx_err;
                ent[i] = true_e;
            }
            if (true_e != ENTRY_NONE) {
                cur = ext[i];
                if (sparse && h->seg_limit[b + i] != UINT32_MAX) {      // last block of a chunk: the chain must end exactly at the chunk end
                    if (ext[i] != (i ? cstart[i] : 0) + (int64_t)h->seg_limit[b + i]) {
                        // the index does not describe this file (the reference only checks that one exists): plain pass instead.
                        // On several ranks that decision has to be taken by all of them together (below, after the batches):
                        // a rank falling back on its own would leave the union of the ranks' records no partition of the file.
                        if (h->world == 1) { h->sparse_ok = false; CK(cudaDeviceSynchronize()); return run_pipeline(h, mode, ro, em); }
                        sparse_bad = true; break;
                    }
                    cur = INT64_MAX / 2;                                  // nothing follows until the next chunk begins
                    continue;
                }
                if (ext[i] < cstart[i + 1]) {      // the walk stopped inside its own block: incomplete tail record
                    for (size_t j = i + 1; j < nb; j++) cnt[j] = 0;
                    break;
                }
            }
        }
        if (sparse_bad) break;
        if (walk_err) return fail(h, BDEPTH_ERR_FORMAT, "corrupt BAM record chain (block_size < 32)");
        tail = cur < (int64_t)ub ? cur : (int64_t)ub;     // first byte not consumed by a complete record
        // ---- shard limit: drop records starting at/after u_limit (host trims counts; offsets are sorted)
        std::vector<uint32_t> rbase(nb + 1); uint64_t R = 0;
        bool limited = u_limit < (int64_t)ub && !fix;        // (-m keeps the records behind the limit: they are marked as the next rank's by k2_decode)
        std::vector<uint16_t> tmp_slots;
        for (size_t i = 0; i < nb; i++) {
            if (limited && cnt[i]) {
                if (cstart[i] >= u_limit) cnt[i] = 0;
                else if (cstart[i + 1] > u_limit) {   // partial: count slots below the limit
                    tmp_slots.resize(cnt[i]);
                    CK(cudaMemcpy(tmp_slots.data(), (uint16_t*)h->slots.p + sbase[i], cnt[i] * 2, cudaMemcpyDeviceToHost));
                    uint32_t k = 0; while (k < cnt[i] && ((k == 0 || cstart[i] > 0) ? cstart[i] : 0) + tmp_slots[k] < u_limit) k++;     // slot encoding: see k2_walk
                    cnt[i] = k;
                }
            }
            rbase[i] = (uint32_t)R; R += cnt[i];
        }
        rbase[nb] = (uint32_t)R;
        if (R > 0xFFFFFFF0ull) return fail(h, BDEPTH_ERR_ARG, "batch too large");
        UP(h->count.p, cnt, nb * 4);
        if (limited && last_batch && tail < u_limit && tail < (int64_t)ub && b1 < B.size()) return fail(h, BDEPTH_ERR_FORMAT, "record at the shard boundary spans more than %u BGZF blocks", SHARD_EXTRA_BLOCKS);
        UP(h->rec_base.p, rbase.data(), (nb + 1) * 4);
        st.n_records += R;
        // ---- K2 decode
        size_t Rc = R ? R : 1;
        CK(h->soa_start.ensure(Rc * 8)); CK(h->soa_span.ensure(Rc * 4)); CK(h->soa_meta.ensure(Rc * 4)); CK(h->soa_off.ensure(Rc * 8)); CK(h->soa_ncl.ensure(Rc * 4)); CK(h->soa_lseq.ensure(Rc * 4)); CK(h->long_list.ensure(Rc * 4));
        RecordSoA soa{h->soa_start.as<uint64_t>(), h->soa_span.as<uint32_t>(), h->soa_meta.as<uint32_t>(), h->soa_off.as<int64_t>(), h->soa_ncl.as<uint32_t>(), h->soa_lseq.as<int32_t>()};
        ScanStats zs{0, 0, 0, 0, ~0ull, 0, 0, ~0ull, 0, 0, ~0ull, 0, ~0ull, ~0ull, 0};
        const int64_t ghost_below = (fix && batch_no > 0) ? (int64_t)ghost_below_abs - (int64_t)batch_u0 : INT64_MIN;
        const int64_t own_lo = (fix && h->world > 1) ? (int64_t)h->own_lo_abs_u - (int64_t)batch_u0 : INT64_MIN;           // -m on several ranks: records outside belong to the neighbours
        const int64_t own_hi = (fix && h->world > 1 && h->limit_abs_u < h->total_u) ? (int64_t)h->limit_abs_u - (int64_t)batch_u0 : INT64_MAX;
        const int64_t zone_below = (!fix && !sparse && h->world > 1) ? (int64_t)h->own_lo_abs_u - (int64_t)batch_u0 : INT64_MIN;       // records of the previous ranks' zone
        UP(h->scan_stats.p, &zs, sizeof zs);
        if ((mode == RUN_SCAN_ONLY || mode == RUN_INDEX) && !h->ref_has.p) { CK(h->ref_has.ensure((nref / 32 + 2) * 4)); CK(cudaMemsetAsync(h->ref_has.p, 0, (nref / 32 + 2) * 4, sm)); }
        // runs with -L regions: K2's every-passing-read bits go to a scratch word array, k_ref_seen marks the references of the reads that overlap a region
        uint32_t* has_dst = h->ref_has.as<uint32_t>();
        const uint32_t n_flt_k2 = mode == RUN_FULL ? (uint32_t)h->regions.size() : 0u;
        if (n_flt_k2) {
            if (!flt_uploaded) {
                std::vector<uint64_t> fl; fl.reserve(2 * (size_t)n_flt_k2);
                for (auto& g : h->regions) fl.push_back(h->hdr.ref_lin0[g.ref_id] + g.start);
                for (auto& g : h->regions) fl.push_back(h->hdr.ref_lin0[g.ref_id] + g.end);
                CK(h->flt_d.ensure(fl.size() * 8)); CK(cudaMemcpyAsync(h->flt_d.p, fl.data(), fl.size() * 8, cudaMemcpyHostToDevice, sm)); CK(cudaStreamSynchronize(sm));      // (fl is a local)
                CK(h->ref_has_all.ensure((nref / 32 + 2) * 4)); CK(cudaMemsetAsync(h->ref_has_all.p, 0, (nref / 32 + 2) * 4, sm));
                flt_uploaded = true;
            }
            has_dst = h->ref_has_all.as<uint32_t>();
        }
#define K2_DECODE(F, G) do { if (d_rgt) K2_DECODE_RG(F, G, true); else K2_DECODE_RG(F, G, false); } while (0)
#define K2_DECODE_RG(F, G, R) BD_LAUNCH((unsigned)((nb * 32 + 255) / 256), 256, 0, sm, k2_decode<F, G, R>)(sp, h->chunk_start.as<int64_t>(), (uint32_t)nb, h->slot_base.as<uint32_t>(), h->slots.as<uint16_t>(), h->count.as<uint32_t>(), h->rec_base.as<uint32_t>(), soa, h->mapq_gt, h->flag_reject, h->scan_stats.as<ScanStats>(), h->long_list.as<uint32_t>(), has_dst, d_rgt, d_fprog, ghost_below, own_lo, own_hi, zone_below)
        if (fix) { if (d_fprog) K2_DECODE(true, true); else K2_DECODE(false, true); }
        else if (d_fprog) K2_DECODE(true, false);
        else K2_DECODE(false, false);
#undef K2_DECODE
#undef K2_DECODE_RG
        CK(cudaGetLastError()); st.gpu_launches++;
        if (R && mode != RUN_INDEX && mode != RUN_SCAN_ONLY) {      // quirk 1: CIGARs that begin with N, rewritten to what the reference's cursor makes of them (the index and the raw scan see the file as it is)
            // region mode proper (no window slots, no -m, one rank): the statistics of such a read are reproduced (kernels.cuh); otherwise refused
            const bool lead_n_regions = h->seg.on && h->seg.n && !h->seg.has_u && !h->seg.has_min && !fix && h->world == 1;
            LeadNSegs lsg{nullptr, nullptr, nullptr, nullptr, 0u, nullptr, nullptr, 1u, h->minq};
            if (lead_n_regions) lsg = LeadNSegs{h->seg.s.as<uint64_t>(), h->seg.e.as<uint64_t>(), h->seg.pmax.as<uint64_t>(), h->seg.id.as<uint32_t>(), h->seg.n, h->seg.reads.as<uint32_t>(), h->seg.mbases.as<uint32_t>(),
                                                h->S, h->minq};
            CK(h->lead_list.ensure(Rc * 4));
            BD_LAUNCH((unsigned)((R + 255) / 256), 256, 0, sm, k2_lead_n_find)(soa, u0, (uint32_t)R, h->lead_list.as<uint32_t>(), h->scan_stats.as<ScanStats>());
            BD_LAUNCH(32, 128, 0, sm, k2_lead_n_fix)(soa, u0, h->lead_list.as<uint32_t>(), h->scan_stats.as<ScanStats>(), (h->seg.on && !lead_n_regions) ? 1 : 0,
                                                    n_flt_k2 ? h->flt_d.as<uint64_t>() : nullptr, n_flt_k2 ? h->flt_d.as<uint64_t>() + n_flt_k2 : nullptr, n_flt_k2, lsg);
            CK(cudaGetLastError()); st.gpu_launches += 2;
        }
        if (n_flt_k2 && R) {
            BD_LAUNCH((unsigned)((R + 255) / 256), 256, 0, sm, k_ref_seen)(soa, (uint32_t)R, h->flt_d.as<uint64_t>(), h->flt_d.as<uint64_t>() + n_flt_k2, n_flt_k2, h->ref_lin0_d.as<uint64_t>(), (uint32_t)nref, h->ref_has.as<uint32_t>());
            CK(cudaGetLastError()); st.gpu_launches++;
        }
        DOWN(ssp, ScanStats, h->scan_stats.p, sizeof(ScanStats));
        CK(cudaEventRecord(e3, sm));
        CK(cudaStreamSynchronize(sm));
        const ScanStats ss = *ssp;
        st.n_records -= ss.n_ghost + ss.n_ghost_right;          // re-read records of the previous batch / of the neighbours' zones are counted there
        if (ss.bad_rec != ~0ull) return fail(h, BDEPTH_ERR_FORMAT, "corrupt BAM record (#%llu of the batch): its name, CIGAR, sequence and qualities do not fit its block_size", ss.bad_rec);
        if (ss.lead_n != ~0ull) return fail(h, BDEPTH_ERR_FORMAT, "read #%llu of the batch: its CIGAR begins with N%s (pileup.d:180-189): there is no result to reproduce", ss.lead_n,
                                             h->seg.on ? " -- the reference computes region / window statistics of such a read partly from its CIGAR as written and partly from a cursor that skips the leading N" : " and ends in a match -- the reference's pileup cursor runs past the read's sequence on such a read");
        if (ss.rg_err != ~0ull) return fail(h, BDEPTH_ERR_FORMAT, "error in read #%llu of the batch: its read group is not present in the header", ss.rg_err);
        if (ss.untagged_elsewhere) h->pass_untagged = true;
        st.n_records_pass += ss.n_pass; st.n_cigar_ops += ss.n_cigar; st.seq_bytes += ss.seq_bytes; st.long_reads += ss.n_long;
        if (ss.n_pass) { shard_min = std::min<uint64_t>(shard_min, ss.min_start); shard_max = std::max<uint64_t>(shard_max, ss.max_end); }
        if (mode == RUN_SCAN_ONLY) {
            if (ro && R) {
                uint64_t n = std::min<uint64_t>(R, ro->scan_cap > ro->scan_n ? ro->scan_cap - ro->scan_n : 0);
                std::vector<uint64_t> hs(n), ho(n); std::vector<uint32_t> hsp(n), hm(n), hn(n);
                CK(cudaMemcpy(hs.data(), soa.start, n * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(ho.data(), soa.off, n * 8, cudaMemcpyDeviceToHost));
                CK(cudaMemcpy(hsp.data(), soa.span, n * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(hm.data(), soa.meta, n * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(hn.data(), soa.ncl, n * 4, cudaMemcpyDeviceToHost));
                for (uint64_t i = 0; i < n; i++) {
                    uint64_t k = ro->scan_n + i; int32_t rid = -1, p = -1;
                    if (hs[i] != START_UNPLACED) { size_t lo = 0, hi = nref; while (lo + 1 < hi) { size_t m = (lo + hi) / 2; if (h->hdr.ref_lin0[m] <= hs[i]) lo = m; else hi = m; } while (lo + 1 < nref && h->hdr.ref_lin0[lo + 1] <= hs[i] && h->hdr.ref_len[lo] == 0) lo++; rid = (int32_t)lo; p = (int32_t)(hs[i] - h->hdr.ref_lin0[lo]); }
                    if (ro->ref_id) ro->ref_id[k] = rid; if (ro->pos) ro->pos[k] = p; if (ro->span) ro->span[k] = hsp[i];
                    if (ro->flag) ro->flag[k] = (uint16_t)(hm[i] >> 16); if (ro->mapq) ro->mapq[k] = (uint8_t)(hm[i] >> 8); if (ro->n_cigar) ro->n_cigar[k] = (uint16_t)(hn[i] >> 8);
                    if (ro->rec_off) ro->rec_off[k] = batch_u0 + ho[i] - 4;       // absolute offset of the block_size field
                }
            }
            if (ro) ro->scan_n += R;
        }
        // ---- BAI builder: the per-record part of IndexBuilder.put (bai/indexing.d:290-333) for this sub-batch's records
        if (mode == RUN_INDEX && R) {
            auto& X = h->ix;
            CK(X.runs.ensure(R * sizeof(IndexRun))); CK(X.excs.ensure(R * sizeof(IndexExc)));
            BD_LAUNCH((unsigned)((R + 255) / 256), 256, 0, sm, k_index_scan)(soa, u0, (uint32_t)R, (unsigned long long)batch_u0, (int)nref, X.lin_base.as<uint32_t>(), X.lin_cap.as<uint32_t>(), X.lin.as<unsigned long long>(), X.lin_len.as<uint32_t>(),
                                                                               X.n_mapped.as<unsigned long long>(), X.n_unmapped.as<unsigned long long>(), X.carry.as<IndexCarry>(), X.runs.as<IndexRun>(), X.excs.as<IndexExc>(), X.ctl.as<IndexCtl>());
            BD_LAUNCH(1, 32, 0, sm, k_index_carry)(soa, u0, (unsigned long long)batch_u0, X.carry.as<IndexCarry>(), X.ctl.as<IndexCtl>());
            CK(cudaGetLastError()); st.gpu_launches += 2;
            DOWN(icp, IndexCtl, X.ctl.p, sizeof(IndexCtl));
            CK(cudaStreamSynchronize(sm));
            const IndexCtl ic = *icp;
            if (ic.bad_ref != ~0ull) return fail(h, BDEPTH_ERR_FORMAT, "record #%llu of the batch names a reference the header does not have", ic.bad_ref);
            if (ic.unsorted != ~0ull) return fail(h, BDEPTH_ERR_FORMAT, "BAM file is not coordinate-sorted (record #%llu of the batch lies before the read in front of it)", ic.unsorted);
            if (ic.past_end) return fail(h, BDEPTH_ERR_FORMAT, "%llu reads reach more than 16 kbp past the end of their reference: no index is built for such a file", ic.past_end);
            if (ic.n_runs) { size_t o = X.h_runs.size(); X.h_runs.resize(o + ic.n_runs); CK(cudaMemcpy(X.h_runs.data() + o, X.runs.p, ic.n_runs * sizeof(IndexRun), cudaMemcpyDeviceToHost)); std::sort(X.h_runs.begin() + o, X.h_runs.end(), [](const IndexRun& a, const IndexRun& b) { return a.start_abs < b.start_abs; }); }
            if (ic.n_exc) { size_t o = X.h_excs.size(); X.h_excs.resize(o + ic.n_exc); CK(cudaMemcpy(X.h_excs.data() + o, X.excs.p, ic.n_exc * sizeof(IndexExc), cudaMemcpyDeviceToHost)); std::sort(X.h_excs.begin() + o, X.h_excs.end(), [](const IndexExc& a, const IndexExc& b) { return a.start_abs < b.start_abs; }); }
            CK(cudaMemsetAsync(X.ctl.p, 0, 16, sm));      // n_runs, n_exc
        }
        // ---- per-read segment counting (countRead, depth.d:661-669) for the window / region front ends
        if (mode == RUN_FULL && h->seg.on && h->seg.n && ss.n_pass) {
            if (h->minq) BD_LAUNCH((unsigned)((R + 127) / 128), 128, 0, sm, k_read_segments<true>)(soa, u0, (uint32_t)R, h->seg.s.as<uint64_t>(), h->seg.e.as<uint64_t>(), h->seg.pmax.as<uint64_t>(), h->seg.id.as<uint32_t>(), h->seg.has_min ? h->seg.minstart.as<uint64_t>() : nullptr, h->seg.n, h->seg.reads.as<uint32_t>(), h->minq, h->S, h->seg.has_min ? h->seg.bases_reads.as<uint32_t>() : nullptr);
            else BD_LAUNCH((unsigned)((R + 127) / 128), 128, 0, sm, k_read_segments<false>)(soa, u0, (uint32_t)R, h->seg.s.as<uint64_t>(), h->seg.e.as<uint64_t>(), h->seg.pmax.as<uint64_t>(), h->seg.id.as<uint32_t>(), h->seg.has_min ? h->seg.minstart.as<uint64_t>() : nullptr, h->seg.n, h->seg.reads.as<uint32_t>(), 0, h->S, h->seg.has_min ? h->seg.bases_reads.as<uint32_t>() : nullptr);
            CK(cudaGetLastError()); st.gpu_launches++;
        }
        uint64_t idx_tiles_base = 0; uint32_t idx_n_tiles = 0;      // K3's per-tile read index of this sub-batch (the mate kernels look reads up through it)
        // ---- K3
        uint64_t gmin = std::min<uint64_t>(ss.min_start, ss.min_start_all), gmax = ss.max_end;
        if (ss.n_zone_pass && gmin < h->cnt_base) gmin = h->cnt_base;      // a zone read may begin before the window; only what reaches this rank's positions matters
        // (a sub-batch of the zone's first blocks can hold nothing but reads that end before this rank's first position -- the linear index
        // points at the first read that overlaps the 16 kbp window, the short reads behind it need not: nothing to count then)
        if (mode == RUN_FULL && (ss.n_pass || ss.n_zone_pass) && gmax > gmin) {
            if (gmin < h->cnt_base || gmax > h->cnt_base + h->win_len) {
                // the index does not describe this file (the reference only checks that one exists, depth.d:1166):
                // start over with the whole genome as the counter window
                if (!h->bai_window_ok) return fail(h, BDEPTH_ERR_FORMAT, "read extends past the end of the reference space");
                h->bai_window_ok = false; CK(cudaDeviceSynchronize());
                if (h->force_window || h->accum) return RC_RETRY_WINDOW;      // several inputs: the caller starts over with the whole genome as the window
                return run_pipeline(h, mode, ro, em);
            }
            uint64_t t_lo = (gmin - h->cnt_base) / TILE_POS, t_hi = (gmax - h->cnt_base + TILE_POS - 1) / TILE_POS;
            uint64_t n_tiles = t_hi - t_lo; uint64_t tiles_base = h->cnt_base + t_lo * TILE_POS;
            idx_tiles_base = tiles_base; idx_n_tiles = (uint32_t)n_tiles;
            if (t_hi * TILE_POS > h->win_len) return fail(h, BDEPTH_ERR_FORMAT, "read extends past the end of the reference space");
            CK(h->tile_first.ensure((n_tiles + 2) * 4)); CK(h->tile_lo.ensure((n_tiles + 2) * 4));
            BD_LAUNCH((unsigned)((n_tiles + 2 + 255) / 256), 256, 0, sm, k_fill_u32)(h->tile_first.as<uint32_t>(), (uint32_t)R, n_tiles + 2);
            CK(cudaMemsetAsync(h->tile_lo.p, 0xFF, (n_tiles + 2) * 4, sm));
            if (h->want_presence) { BD_LAUNCH((unsigned)((R + 255) / 256), 256, 0, sm, k_presence)(soa, (uint32_t)R, h->cnt_base, h->win_len, h->present.as<uint32_t>()); st.gpu_launches++; }
            BD_LAUNCH((unsigned)((R + 255) / 256), 256, 0, sm, k3_tile_index)(soa, (uint32_t)R, tiles_base, (uint32_t)n_tiles, h->tile_first.as<uint32_t>(), h->tile_lo.as<uint32_t>());
            CK(cudaGetLastError()); st.gpu_launches += 2;
            for (uint32_t si = 0; si < h->S; si++) {      // one counter set per sample (one pass when combined / single sample)
                if (h->pass_n && rgt.n_rg && !((ss.seen_samples >> si) & 1ull)) continue;      // a sample pass: only the samples this sub-batch holds reads of
                uint32_t* cnt = h->counts.as<uint32_t>() + (uint64_t)si * N_PLANES * h->win_len; int sel = h->S > 1 ? (int)si : -1;
                if (ss.n_long) {
                    if (h->minq) BD_LAUNCH((unsigned)((ss.n_long * 32 + 255) / 256), 256, 0, sm, k3_scatter_long<true>)(soa, u0, h->long_list.as<uint32_t>(), (uint32_t)ss.n_long, h->cnt_base, h->win_len, cnt, h->minq, sel);
                    else BD_LAUNCH((unsigned)((ss.n_long * 32 + 255) / 256), 256, 0, sm, k3_scatter_long<false>)(soa, u0, h->long_list.as<uint32_t>(), (uint32_t)ss.n_long, h->cnt_base, h->win_len, cnt, 0, sel);
                    CK(cudaGetLastError()); st.gpu_launches++;
                }
                if (h->k3_tile) {      // CTA per tile, shared-memory counters, records staged by cp.async.bulk
                    if (h->minq) BD_LAUNCH((unsigned)n_tiles, 256, K3T_SMEM, sm, k3_tile<true>)(soa, u0, (int64_t)ub, (uint32_t)R, tiles_base, h->cnt_base, h->win_len, h->tile_first.as<uint32_t>(), h->tile_lo.as<uint32_t>(), cnt, h->minq, sel);
                    else BD_LAUNCH((unsigned)n_tiles, 256, K3T_SMEM, sm, k3_tile<false>)(soa, u0, (int64_t)ub, (uint32_t)R, tiles_base, h->cnt_base, h->win_len, h->tile_first.as<uint32_t>(), h->tile_lo.as<uint32_t>(), cnt, 0, sel);
                } else if (h->k3_pre) {       // round-1 gather kernel with lane-parallel record prefetch (BDEPTH_K3=gather)
                    if (h->minq) BD_LAUNCH((unsigned)n_tiles, 256, 0, sm, k3_gather<true, true>)(soa, u0, tiles_base, h->cnt_base, h->win_len, h->tile_first.as<uint32_t>(), h->tile_lo.as<uint32_t>(), cnt, h->minq, sel);
                    else BD_LAUNCH((unsigned)n_tiles, 256, 0, sm, k3_gather<false, true>)(soa, u0, tiles_base, h->cnt_base, h->win_len, h->tile_first.as<uint32_t>(), h->tile_lo.as<uint32_t>(), cnt, 0, sel);
                } else if (h->minq) BD_LAUNCH((unsigned)n_tiles, 256, 0, sm, k3_gather<true, false>)(soa, u0, tiles_base, h->cnt_base, h->win_len, h->tile_first.as<uint32_t>(), h->tile_lo.as<uint32_t>(), cnt, h->minq, sel);
                else BD_LAUNCH((unsigned)n_tiles, 256, 0, sm, k3_gather<false, false>)(soa, u0, tiles_base, h->cnt_base, h->win_len, h->tile_first.as<uint32_t>(), h->tile_lo.as<uint32_t>(), cnt, 0, sel);
                CK(cudaGetLastError()); st.gpu_launches++;
            }
        }
        // ---- -m: take the worse mate of every overlapping pair out again (mates.cuh)
        if (fix) {      // where the next batch's stream begins if nothing is open: the first record this batch did not consume
            const uint64_t tail_abs = batch_u0 + (uint64_t)tail; size_t lo = 0, hi = B.size(); while (lo + 1 < hi) { size_t m2 = (lo + hi) / 2; if (B[m2].uoff <= tail_abs) lo = m2; else hi = m2; }
            ghost_b = lo; ghost_entry = (int64_t)(tail_abs - B[lo].uoff); ghost_below_abs = tail_abs;
        }
        if (fix && R && (ss.n_pass || ss.n_ghost || ss.n_ghost_right)) {
            if (subs.size() != 1) return fail(h, BDEPTH_ERR_ARG, "internal: fix-mate-overlaps scans a batch as a whole");
            uint64_t s_last = 0;       // start of the batch's last record: nothing that follows starts before it
            CK(cudaMemcpyAsync(&s_last, soa.start + (R - 1), 8, cudaMemcpyDeviceToHost, sm)); CK(cudaStreamSynchronize(sm));
            cudaEvent_t em0 = h->ev[20], em1 = h->ev[21];
            CK(cudaEventRecord(em0, sm));
            CK(h->m_hash.ensure(Rc * 8)); CK(h->m_flag.ensure(Rc * 4)); CK(h->m_ctl.ensure(64));
            std::vector<uint64_t> fl;                 // -L: merged regions (sorted, disjoint) in linear coordinates, starts then ends
            for (auto& g : h->regions) fl.push_back(h->hdr.ref_lin0[g.ref_id] + g.start);
            for (auto& g : h->regions) fl.push_back(h->hdr.ref_lin0[g.ref_id] + g.end);
            const uint32_t n_flt = (uint32_t)h->regions.size();
            CK(h->m_flt.ensure(fl.size() * 8 + 16));
            if (n_flt) CK(cudaMemcpyAsync(h->m_flt.p, fl.data(), fl.size() * 8, cudaMemcpyHostToDevice, sm));
            CK(cudaMemsetAsync(h->m_ctl.p, 0, 64, sm)); CK(cudaMemsetAsync((uint8_t*)h->m_ctl.p + 48, 0xFF, 16, sm));       // err, stat; open_off = open_start = none
            const bool segm = h->seg.on && h->seg.n;
            MateParams mp{soa.start, soa.span, soa.meta, soa.off, soa.ncl, soa.lseq, u0, (uint32_t)R, h->m_hash.as<uint64_t>(), h->m_flag.as<uint32_t>(),
                          h->m_flt.as<uint64_t>(), h->m_flt.as<uint64_t>() + n_flt, n_flt, h->counts.as<uint32_t>(), h->cnt_base, h->win_len, h->S, h->minq,
                          segm ? h->seg.s.as<uint64_t>() : nullptr, segm ? h->seg.e.as<uint64_t>() : nullptr, segm ? h->seg.pmax.as<uint64_t>() : nullptr, segm ? h->seg.id.as<uint32_t>() : nullptr,
                          segm ? h->seg.n : 0u, segm ? h->seg.reads.as<uint32_t>() : nullptr, segm ? h->seg.mbases.as<uint32_t>() : nullptr, h->S,
                          segm && h->seg.has_u ? h->seg.ustart.as<uint64_t>() : nullptr, segm && h->seg.has_u && h->seg.has_min ? h->seg.minstart.as<uint64_t>() : nullptr, segm && h->seg.has_u ? h->seg.ext_max : 0ull,
                          h->tile_lo.as<uint32_t>(), idx_tiles_base, idx_n_tiles, h->long_list.as<uint32_t>(), (uint32_t)ss.n_long,
                          (uint32_t)ss.n_ghost, s_last, prev_s_last, covered_from, last_batch ? 1 : 0, (unsigned long long*)((uint8_t*)h->m_ctl.p + 48), (unsigned long long*)((uint8_t*)h->m_ctl.p + 56),
                          (last_batch && blk_hi < B.size()) ? 1 : 0, (unsigned long long*)((uint8_t*)h->m_ctl.p + 40), (uint32_t)ss.n_ghost_right, ghost_below == INT64_MIN ? INT64_MIN : ghost_below + 4, 0,
                          (int*)h->m_ctl.p, (unsigned long long*)((uint8_t*)h->m_ctl.p + 16)};
            const unsigned mg = (unsigned)((R + 127) / 128);
            BD_LAUNCH(mg, 128, 0, sm, km_hash)(mp); BD_LAUNCH(mg, 128, 0, sm, km_link)(mp); BD_LAUNCH(mg, 128, 0, sm, km_fix)(mp);
            if (!last_batch) { BD_LAUNCH(mg, 128, 0, sm, km_cover)(mp); st.gpu_launches++; }
            CK(cudaGetLastError()); st.gpu_launches += 3;
            CK(cudaEventRecord(em1, sm));
            struct { int err[4]; unsigned long long stat[3]; unsigned long long fix_max_end; unsigned long long open_off, open_start; } ctl;
            CK(cudaMemcpyAsync(&ctl, h->m_ctl.p, sizeof ctl, cudaMemcpyDeviceToHost, sm));
            CK(cudaStreamSynchronize(sm));
            if (ctl.err[0] == MATE_ERR_TOO_MANY) return fail(h, BDEPTH_ERR_ARG, "fix-mate-overlaps: more than %d reads of one name cover one position (record #%d of the batch)", MATE_MAX_MEMBERS, ctl.err[1]);
            if (ctl.err[0] == MATE_ERR_CROSS) return fail(h, BDEPTH_ERR_ARG, "fix-mate-overlaps: four or more overlapping reads of one name next to a batch boundary (record #%d of the batch): not reproduced there, use larger batches", ctl.err[1]);
            st.mate_pairs += ctl.stat[0]; st.mate_pair_columns += ctl.stat[1]; st.mate_groups += ctl.stat[2];
            if (!last_batch && ctl.open_off != ~0ull && batch_u0 + (ctl.open_off - 4) < ghost_below_abs) {      // something is still open: re-read from its first record
                const uint64_t g_abs = batch_u0 + (ctl.open_off - 4); size_t lo = 0, hi = B.size(); while (lo + 1 < hi) { size_t m2 = (lo + hi) / 2; if (B[m2].uoff <= g_abs) lo = m2; else hi = m2; }
                ghost_b = lo; ghost_entry = (int64_t)(g_abs - B[lo].uoff);
            }
            if (ctl.err[0] == MATE_ERR_ZONE) return fail(h, BDEPTH_ERR_ARG, "fix-mate-overlaps on several ranks: overlapping reads of one name reach more than %u BGZF blocks past a shard boundary (record #%d of the batch)", MATE_ZONE_BLOCKS, ctl.err[1]);
            if (ctl.fix_max_end > shard_max && shard_min != UINT64_MAX) shard_max = ctl.fix_max_end;      // the halo exchange carries the corrections to their owners
            prev_s_last = s_last; covered_from = ctl.open_start;
            { float t = 0; CK(cudaEventElapsedTime(&t, em0, em1)); st.ms_mates += t; }
        }
        CK(cudaEventRecord(e4, sm));
        // Progressive delivery: positions below the start of the sub-batch's last own read are final (the file is coordinate sorted).  Several ranks
        // (plain shards): a rank's own positions begin at its first passing read -- known once such a read has been seen -- and the reads of the
        // previous ranks that reach into them come first in its stream (the zone), so the same holds; where its positions end it learns at the end.
        const bool zone_mode = h->world > 1 && h->comm && !fix && !sparse;
        if (em && zone_mode && h->rank > 0 && shard_min != UINT64_MAX) em->lo_clip = shard_min;
        if (em && mode == RUN_FULL && (h->world == 1 || (zone_mode && (h->rank == 0 || shard_min != UINT64_MAX))) && !fix && !last_batch && ss.n_pass) { int rce = em->advance(ss.max_start / TILE_POS * TILE_POS, e4); if (rce) return rce; }
        // ---- carry the incomplete tail record to the front of the next batch
        uint64_t new_carry = (uint64_t)((int64_t)ub - tail);
        // the file ends inside a record: readExact throws "not enough data in stream" (readrange.d:169); fewer than 4 left-over bytes end the stream quietly (:139-149)
        if (last_batch && last_sub && !sparse && !limited && b1 == B.size() && new_carry >= 4) return fail(h, BDEPTH_ERR_FORMAT, "truncated BAM record at the end of the file (not enough data in stream)");
        if (!last_batch && last_sub && new_carry && !fix) {      // inside a batch the tail already sits right below the next sub-batch; -m re-reads it with the next batch
            if (new_carry > CARRY_MAX) return fail(h, BDEPTH_ERR_FORMAT, "BAM record larger than %zu bytes", CARRY_MAX);
            CK(cudaMemcpyAsync(m_u0 - new_carry, u0 + tail, new_carry, cudaMemcpyDeviceToDevice, sm));
        }
        CK(cudaStreamSynchronize(sm));
        { float t; if (!h->staged && last_sub) { CK(cudaEventElapsedTime(&t, h->ev[18 + (batch_no & 1)], h->ev[14 + (batch_no & 1)])); ms_h2d += t; } if (last_sub) { CK(cudaEventElapsedTime(&t, e1, e2)); ms_k1 += t; } CK(cudaEventElapsedTime(&t, e2, e3)); ms_k2 += t; CK(cudaEventElapsedTime(&t, e3, e4)); ms_k3 += t; }
        carry_len = (last_batch || fix) ? 0 : new_carry; first_batch = false;
        hs.used = 0;      // synchronised above: the scratch is free again
        }   // sub-batches
        if (sparse_bad) break;
        }   // stream scope
        b = b1; batch_no++;
    }
    if (sparse && h->world > 1) {      // did the region chunks end where the index says, on EVERY rank?
        if (h->comm) {
            uint32_t flag = sparse_bad ? 1u : 0u;
            CK(cudaMemcpyAsync(h->misc.p, &flag, 4, cudaMemcpyHostToDevice, sm));
            NK(nccl().AllReduce(h->misc.p, h->misc.p, 1, NCCL_UINT32, NCCL_SUM, h->comm, sm));
            h->coll_pending = 1;
            CK(cudaMemcpyAsync(&flag, h->misc.p, 4, cudaMemcpyDeviceToHost, sm)); CK(cudaStreamSynchronize(sm));
            if (flag >= SPARSE_PEER_FAILED) { h->coll_pending = 0; return fail(h, BDEPTH_ERR_NCCL, "another rank of the run stopped with an error (its own message says why): no result"); }
            sparse_bad = flag != 0;
        } else if (sparse_bad) return fail(h, BDEPTH_ERR_FORMAT, "the index does not describe this file (a region chunk does not end at a record); several ranks without a NCCL id cannot fall back together");
        if (sparse_bad) { h->sparse_ok = false; CK(cudaDeviceSynchronize()); return run_pipeline(h, mode, ro, em); }
    }
    st.ms_h2d = ms_h2d; st.ms_inflate = ms_k1; st.ms_scan = ms_k2; st.ms_coverage = ms_k3;
    st.positions = mode == RUN_FULL ? h->hdr.total_len : 0;
    h->own_lo = 0; h->own_hi = h->hdr.total_len;
    if (mode == RUN_FULL) {
        if (h->world > 1 && h->comm) { rc = exchange_boundaries(h, shard_min, shard_max, sparse || fix); if (rc) return rc; }      // plain shards: the boundary table only (every rank counted its zone)
        h->ref_has_host.assign(nref / 32 + 2, 0);
        CK(cudaMemcpyAsync(h->ref_has_host.data(), h->ref_has.p, (nref / 32 + 2) * 4, cudaMemcpyDeviceToHost, sm));
    }
    CK(cudaEventRecord(h->ev[11], sm));
    CK(cudaStreamSynchronize(sm));
    { float t = 0; CK(cudaEventElapsedTime(&t, h->ev[10], h->ev[11])); st.ms_span_device = t; }
    st.own_lo = h->own_lo; st.own_hi = h->own_hi;
    st.host_wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_host0).count();
    return 0;
}

// ---- several inputs --------------------------------------------------------------------------------------------------------
// Exchange the input of two handles: everything that describes the file and the plan made for it, nothing of the device state.
void swap_inputs(bdepth* a, bdepth* b) {
    std::swap(a->file, b->file); std::swap(a->file_len, b->file_len); std::swap(a->mapped, b->mapped); std::swap(a->fd, b->fd);
    std::swap(a->blocks, b->blocks); std::swap(a->total_u, b->total_u); std::swap(a->lazy, b->lazy); std::swap(a->framed_all, b->framed_all); std::swap(a->framed_off, b->framed_off);
    std::swap(a->hdr, b->hdr); std::swap(a->bai, b->bai); std::swap(a->has_index, b->has_index); std::swap(a->bai_window_ok, b->bai_window_ok);
    std::swap(a->shard_ready, b->shard_ready); std::swap(a->blk_lo, b->blk_lo); std::swap(a->blk_hi, b->blk_hi); std::swap(a->entry0, b->entry0);
    std::swap(a->limit_abs_u, b->limit_abs_u); std::swap(a->own_lo_abs_u, b->own_lo_abs_u); std::swap(a->zone_lin_lo, b->zone_lin_lo);
    std::swap(a->sparse_ok, b->sparse_ok); std::swap(a->sparse_on, b->sparse_on); std::swap(a->vblocks, b->vblocks); std::swap(a->seg_entry, b->seg_entry); std::swap(a->seg_limit, b->seg_limit);
}
// where the linear index of the handle's current input says reads can lie (whole genome when it says nothing)
void index_extent(const bdepth* h, uint64_t& lo, uint64_t& hi) {
    const size_t nref = h->hdr.ref_len.size();
    lo = 0; hi = h->hdr.total_len;
    if (!(h->bai.valid && h->bai_window_ok && h->bai.ioffsets.size() == nref)) return;
    uint64_t a = UINT64_MAX, b = 0;
    for (size_t r = 0; r < nref; r++) {
        const auto& v = h->bai.ioffsets[r]; if (v.empty()) continue;
        size_t k = 0; while (k < v.size() && v[k] == 0) k++;
        if (k == v.size()) continue;
        a = std::min<uint64_t>(a, h->hdr.ref_lin0[r] + std::min<uint64_t>((uint64_t)k << 14, h->hdr.ref_len[r]));
        b = std::max<uint64_t>(b, h->hdr.ref_lin0[r] + std::min<uint64_t>((uint64_t)v.size() << 14, h->hdr.ref_len[r]));
    }
    if (a < b) { lo = a; hi = b; }
}
void add_stats(bdepth_stats& t, const bdepth_stats& s) {
    t.file_bytes += s.file_bytes; t.n_blocks += s.n_blocks; t.cdata_bytes += s.cdata_bytes; t.inflated_bytes += s.inflated_bytes; t.n_records += s.n_records; t.n_records_pass += s.n_records_pass;
    t.n_cigar_ops += s.n_cigar_ops; t.seq_bytes += s.seq_bytes; t.long_reads += s.long_reads; t.chain_fixups += s.chain_fixups; t.gpu_launches += s.gpu_launches; t.n_batches += s.n_batches;
    t.ms_h2d += s.ms_h2d; t.ms_inflate += s.ms_inflate; t.ms_scan += s.ms_scan; t.ms_coverage += s.ms_coverage; t.ms_span_device += s.ms_span_device; t.host_wall_ms += s.host_wall_ms;
}
// One pass of a region / window run whose samples are counted a group at a time (run_segments; the group is h->pass_g0 / pass_n).
// It reads the inputs whose @RG samples meet the group, and -- when the group holds sample 0 -- those in which an earlier pass met
// reads without an RG tag (they belong to sample 0, depth.d:240-250; the pass that holds sample 0 runs last).  Every input's records
// enter n_records once, in the first pass that reads it.
struct SamplePass {
    std::vector<char> counted, untagged;      // per input (0: the handle's own, i: extra[i - 1])
    bool reads(const bdepth* h, size_t i) const {
        const BamHeader& hd = h->hdr;
        if (hd.rg_ids.empty()) return h->pass_g0 == 0;          // no @RG lines: every read is sample 0
        if (h->pass_g0 == 0 && untagged[i]) return true;
        for (int s : hd.rg_sample) if ((uint32_t)s - h->pass_g0 < h->pass_n) return true;
        return false;
    }
    void note(bdepth* h, size_t i) {
        if (counted[i]) h->st.n_records = 0;
        counted[i] = 1;
        if (h->pass_untagged) untagged[i] = 1;
    }
};
// The pipeline over every input of the handle, into one set of counters (RUN_FULL).  One input: run_pipeline as it is.
int run_all_inputs(bdepth* h, Emitter* em = nullptr, SamplePass* sp = nullptr) {
    if (h->extra.empty()) {
        const int rc = run_pipeline(h, RUN_FULL, nullptr, em);
        if (!rc && sp) sp->note(h, 0);
        return rc;
    }
    if (h->fix_mates) return fail(h, BDEPTH_ERR_ARG, "fix-mate-overlaps with several BAM files: not available (mates are paired within one file's stream)");
    if (h->world > 1) return fail(h, BDEPTH_ERR_ARG, "several BAM files on several ranks: not available");
    h->staged = false;
    for (int attempt = 0; attempt < 2; attempt++) {
        // the counter window: the union of what the inputs' indices say (second attempt: an index lied -- the whole genome)
        uint64_t lo = UINT64_MAX, hi = 0;
        for (size_t i = 0; i <= h->extra.size(); i++) {
            if (i) swap_inputs(h, h->extra[i - 1]);
            uint64_t a, b; index_extent(h, a, b); if (attempt) { a = 0; b = h->hdr.total_len; }
            lo = std::min(lo, a); hi = std::max(hi, b);
            if (i) swap_inputs(h, h->extra[i - 1]);
        }
        h->cnt_base = lo / TILE_POS * TILE_POS; h->win_len = ((hi - h->cnt_base + TILE_POS - 1) / TILE_POS + 1) * TILE_POS;
        h->force_window = true;
        bdepth_stats total{}; int rc = 0; size_t n_run = 0;
        const SamplePass sp0 = sp ? *sp : SamplePass{};      // (what a second attempt starts from)
        for (size_t i = 0; i <= h->extra.size() && !rc; i++) {
            if (i) swap_inputs(h, h->extra[i - 1]);
            if (!sp || sp->reads(h, i)) {
                h->accum = n_run++ > 0;
                rc = run_pipeline(h, RUN_FULL, nullptr, nullptr);       // (delivery starts when every input has been counted)
                if (!rc && sp) sp->note(h, i);
                add_stats(total, h->st);
            }
            if (i) swap_inputs(h, h->extra[i - 1]);
        }
        h->accum = false; h->force_window = false;
        if (rc == RC_RETRY_WINDOW) { if (attempt) return fail(h, BDEPTH_ERR_FORMAT, "read extends past the end of the reference space"); if (sp) *sp = sp0; continue; }
        if (rc) return rc;
        if (!n_run) return fail(h, BDEPTH_ERR_ARG, "internal: a sample pass that reads no input");
        total.positions = h->hdr.total_len; total.own_lo = h->own_lo; total.own_hi = h->own_hi;
        h->st = total;
        return 0;
    }
    return fail(h, BDEPTH_ERR_FORMAT, "internal: counter window");
}

// merged, sorted regions clipped to reference lengths
void normalize_regions(const bdepth* h, const bdepth_region* r, size_t n, std::vector<bdepth_region>& out) {
    out.clear();
    for (size_t i = 0; i < n; i++) {
        if (r[i].ref_id >= h->hdr.ref_len.size() || r[i].start >= r[i].end) continue;
        bdepth_region g = r[i]; if (g.end > h->hdr.ref_len[g.ref_id]) g.end = h->hdr.ref_len[g.ref_id]; if (g.start >= g.end) continue;
        out.push_back(g);
    }
    std::sort(out.begin(), out.end(), [](const bdepth_region& a, const bdepth_region& b) { return a.ref_id != b.ref_id ? a.ref_id < b.ref_id : a.start != b.start ? a.start < b.start : a.end < b.end; });
    size_t m = 0;
    for (size_t i = 0; i < out.size(); i++) { if (m && out[m - 1].ref_id == out[i].ref_id && out[m - 1].end >= out[i].start) out[m - 1].end = std::max(out[m - 1].end, out[i].end); else out[m++] = out[i]; }
    out.resize(m);
}

}  // namespace

// =============================================================================== C ABI
extern "C" {

int bdepth_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) return 0; return n; }

static int open_common(bdepth* h, bdepth_t** out) {
    int rc = finish_open(h);
    if (rc) { g_open_error = h->err; bdepth_close(h); return rc; }
    *out = h; return 0;
}

static int open_path(const char* bam_path, int device, bool lazy, bdepth_t** out);
int bdepth_open(const char* bam_path, int device, bdepth_t** out) { return open_path(bam_path, device, false, out); }
int bdepth_open_lazy(const char* bam_path, int device, bdepth_t** out) { return open_path(bam_path, device, true, out); }
static int open_path(const char* bam_path, int device, bool lazy, bdepth_t** out) {
    if (!bam_path || !out) return fail(nullptr, BDEPTH_ERR_ARG, "null argument");
    bdepth* h = new bdepth(); h->device = device; h->lazy = lazy;
    h->fd = open(bam_path, O_RDONLY);
    if (h->fd < 0) { delete h; return fail(nullptr, BDEPTH_ERR_IO, "Cannot open file `%s' in mode `rb' (No such file or directory)", bam_path); }
    struct stat sb; if (fstat(h->fd, &sb) != 0 || sb.st_size == 0) { close(h->fd); delete h; return fail(nullptr, BDEPTH_ERR_IO, "cannot stat `%s' or file is empty", bam_path); }
    h->file_len = (size_t)sb.st_size;
    void* m = mmap(nullptr, h->file_len, PROT_READ, MAP_PRIVATE, h->fd, 0);
    if (m == MAP_FAILED) { close(h->fd); delete h; return fail(nullptr, BDEPTH_ERR_IO, "cannot mmap `%s'", bam_path); }
    madvise(m, h->file_len, MADV_SEQUENTIAL);
    h->file = (const uint8_t*)m; h->mapped = true;
    // index lookup as BaiFile does (baifile.d:98-113): <file>.bai, else <file minus extension>.bai
    std::string p1 = std::string(bam_path) + ".bai", p2; { std::string s(bam_path); size_t dot = s.rfind('.'); p2 = (dot == std::string::npos ? s + "." : s.substr(0, dot + 1)) + "bai"; }
    for (const std::string& bp : {p1, p2}) {
        FILE* f = fopen(bp.c_str(), "rb"); if (!f) continue;
        fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET);
        std::vector<uint8_t> buf(n > 0 ? n : 0); if (n > 0 && fread(buf.data(), 1, n, f) != (size_t)n) { fclose(f); continue; }
        fclose(f); h->has_index = true; parse_bai(buf.data(), buf.size(), h->bai); break;
    }
    return open_common(h, out);
}

int bdepth_open_memory(const void* bam, size_t bam_len, const void* bai, size_t bai_len, int device, bdepth_t** out) {
    if (!bam || !bam_len || !out) return fail(nullptr, BDEPTH_ERR_ARG, "null argument");
    bdepth* h = new bdepth(); h->device = device; h->file = (const uint8_t*)bam; h->file_len = bam_len;
    if (bai && bai_len) { h->has_index = true; parse_bai((const uint8_t*)bai, bai_len, h->bai); }
    return open_common(h, out);
}

// MultiBamReader(string[] filenames) (multireader.d:244-246, depth.d:1162-1163): one more coordinate-sorted, indexed BAM whose reads
// are counted together with the handle's.  Its reference dictionary must be the handle's (the reference's SamHeaderMerger only
// supports its "simple" strategy, multireader.d:225); its read groups join the sample table: a sample name keeps its number, new
// names are appended in the order of the file's @RG lines (the reference numbers samples in the iteration order of a D
// associative array, samheadermerger.d:202: not reproducible -- with --combined or one sample there is no order).
int bdepth_add_input(bdepth_t* h, const char* bam_path) {
    if (!h || !bam_path) return fail(h, BDEPTH_ERR_ARG, "null argument");
    bdepth* x = nullptr;
    int rc = open_path(bam_path, h->device, h->lazy, &x);
    if (rc) { h->err = g_open_error; return rc; }
    if (x->hdr.ref_names != h->hdr.ref_names || x->hdr.ref_len != h->hdr.ref_len) { bdepth_close(x); return fail(h, BDEPTH_ERR_ARG, "%s: its reference sequences differ from the first file's (only identical sequence dictionaries can be merged)", bam_path); }
    // merged sample table, the same in every input's header
    const bool first_has_rg = !h->hdr.rg_ids.empty(), this_has_rg = !x->hdr.rg_ids.empty();
    std::vector<std::string> merged = first_has_rg ? h->hdr.sample_names : std::vector<std::string>();
    std::vector<int> remap(x->hdr.sample_names.size(), 0);
    if (this_has_rg) for (size_t i = 0; i < x->hdr.sample_names.size(); i++) {
        int id = -1; for (size_t k = 0; k < merged.size(); k++) if (merged[k] == x->hdr.sample_names[i]) id = (int)k;
        if (id < 0) { id = (int)merged.size(); merged.push_back(x->hdr.sample_names[i]); }
        remap[i] = id;
    }
    if (merged.empty()) merged.push_back("*");
    for (auto& sid : x->hdr.rg_sample) sid = remap[sid];
    x->hdr.sample_names = merged; h->hdr.sample_names = merged;
    for (bdepth* e : h->extra) e->hdr.sample_names = merged;
    // the additional handle only holds its input from here on
    x->comp.release(); x->descs.release(); x->status.release(); x->ubuf.release();
    h->extra.push_back(x);
    h->staged = false;
    return 0;
}

void bdepth_close(bdepth_t* h) {
    if (!h) return;
    for (bdepth* e : h->extra) bdepth_close(e);
    h->extra.clear();
    cudaSetDevice(h->device);
    h->anchors_idx.release(); h->anchors_val.release(); h->chunk_limit.release(); h->tok.release(); h->lits.release(); h->aux.release(); h->segi.release(); h->littab.release();
    DevBuf* bufs[] = {&h->comp, &h->descs, &h->status, &h->ubuf, &h->chunk_start, &h->entry, &h->exitb, &h->count, &h->slot_base, &h->slots, &h->rec_base, &h->walk_list, &h->soa_start, &h->soa_span, &h->soa_meta, &h->soa_off, &h->soa_ncl, &h->soa_lseq, &h->long_list, &h->tile_first, &h->tile_lo, &h->counts, &h->ref_len_d, &h->ref_lin0_d, &h->scan_stats, &h->ref_has, &h->ref_has_all, &h->flt_d, &h->lead_list, &h->misc};
    for (DevBuf* b : bufs) b->release();
    h->rg_ids.release(); h->rg_offs.release(); h->rg_samp.release(); h->rg_hash.release(); h->rg_tab.release();
    h->text[0].release(); h->text[1].release(); h->text_tiles.release(); h->text_offs.release(); h->text_zero.release(); h->text_samp.release(); h->present.release();
    h->seg.s.release(); h->seg.e.release(); h->seg.pmax.release(); h->seg.id.release(); h->seg.reads.release(); h->seg.minstart.release(); h->seg.bases_reads.release(); h->seg.mbases.release(); h->seg.ustart.release(); h->seg.dscr.release(); h->seg.da.release(); h->seg.dac.release(); h->seg.db.release(); h->seg.dthr.release(); h->seg.dbases.release(); h->seg.dcov.release();
    { auto& X = h->ix; X.lin.release(); X.lin_len.release(); X.lin_base.release(); X.lin_cap.release(); X.n_mapped.release(); X.n_unmapped.release(); X.carry.release(); X.ctl.release(); X.runs.release(); X.excs.release(); }
    h->m_hash.release(); h->m_flag.release(); h->m_flt.release(); h->m_ctl.release(); h->fprog_d.release();
    if (h->comm) { nccl().CommDestroy(h->comm); h->comm = nullptr; }
    if (h->pinned) cudaFreeHost(h->pinned);
    h->hs.release();
    if (h->s_main) { cudaStreamDestroy(h->s_main); cudaStreamDestroy(h->s_copy); cudaStreamDestroy(h->s_d2h); for (auto& ks : h->s_k1) cudaStreamDestroy(ks); for (auto& e : h->ev) cudaEventDestroy(e); for (int q = 0; q < 2; q++) for (auto& e : h->chunk_ev[q]) cudaEventDestroy(e); for (auto& e : h->k1_ev) cudaEventDestroy(e); }
    h->comp2[0].release(); h->comp2[1].release();
    if (h->mapped) munmap((void*)h->file, h->file_len);
    if (h->fd >= 0) close(h->fd);
    delete h;
}

const char* bdepth_last_error(const bdepth_t* h) { return h ? h->err.c_str() : g_open_error.c_str(); }

int bdepth_n_ref(const bdepth_t* h) { return (int)h->hdr.ref_len.size(); }
const char* bdepth_ref_name(const bdepth_t* h, int i) { return (i >= 0 && (size_t)i < h->hdr.ref_names.size()) ? h->hdr.ref_names[i].c_str() : nullptr; }
uint32_t bdepth_ref_length(const bdepth_t* h, int i) { return (i >= 0 && (size_t)i < h->hdr.ref_len.size()) ? h->hdr.ref_len[i] : 0; }
const char* bdepth_header_text(const bdepth_t* h, size_t* len) { if (len) *len = h->hdr.text.size(); return h->hdr.text.c_str(); }
int bdepth_is_coordinate_sorted(const bdepth_t* h) { for (const bdepth* e : h->extra) if (!e->hdr.so_coordinate) return 0; return h->hdr.so_coordinate ? 1 : 0; }      // "All files must be coordinate-sorted" (depth.d:1164)
int bdepth_has_index(const bdepth_t* h) { for (const bdepth* e : h->extra) if (!e->has_index) return 0; return h->has_index ? 1 : 0; }
int bdepth_n_samples(const bdepth_t* h) { return (int)h->hdr.sample_names.size(); }
const char* bdepth_sample_name(const bdepth_t* h, int i) { return (i >= 0 && (size_t)i < h->hdr.sample_names.size()) ? h->hdr.sample_names[i].c_str() : nullptr; }

int bdepth_set_filter(bdepth_t* h, int mapq_gt, uint32_t flag_reject_mask) { h->mapq_gt = mapq_gt; h->flag_reject = flag_reject_mask; h->has_fprog = false; return 0; }
int bdepth_set_filter_query(bdepth_t* h, const char* query) {
    if (!query) return fail(h, BDEPTH_ERR_ARG, "null filter");
    const std::string q(query);
    if (q.empty()) return bdepth_set_filter(h, -1, 0);                                                     // NullFilter, filtering.d:41-42
    if (q == "mapping_quality > 0 and not duplicate and not failed_quality_control") return bdepth_set_filter(h, 0, 0x600);   // depth.d:1159
    FilterCompiler fc(h->hdr.ref_names);
    std::string e = fc.compile(q, h->fprog);
    if (!e.empty()) { h->has_fprog = false; return fail(h, BDEPTH_ERR_ARG, "%s", e.c_str()); }
    h->has_fprog = true;
    return 0;
}
int bdepth_set_combined(bdepth_t* h, int combined) { h->combined = combined != 0; return 0; }
int bdepth_set_samples_per_pass(bdepth_t* h, uint32_t n) { h->samples_per_pass = n; return 0; }
int bdepth_set_fix_mates(bdepth_t* h, int on) { if (h->fix_mates != (on != 0)) h->shard_ready = false; h->fix_mates = on != 0; return 0; }      // (with -m a shard is read with zones around it)
int bdepth_set_min_baseq(bdepth_t* h, uint32_t q) { h->minq = q > 255 ? 255 : q; return 0; }
int bdepth_set_regions(bdepth_t* h, const bdepth_region* r, size_t n) { normalize_regions(h, r, n, h->regions); return 0; }
int bdepth_set_shard(bdepth_t* h, int rank, int world, const void* nccl_unique_id) {
    if (world < 1 || rank < 0 || rank >= world) return fail(h, BDEPTH_ERR_ARG, "bad shard %d/%d", rank, world);
    if (world > 1 && !h->bai.valid) return fail(h, BDEPTH_ERR_NOINDEX, "sharding needs the BAI linear index");
    if (h->comm) { nccl().CommDestroy(h->comm); h->comm = nullptr; }
    h->rank = rank; h->world = world; h->shard_ready = false; h->staged = false;
    if (world > 1 && nccl_unique_id) {
        NcclApi& N = nccl();
        if (!N.ok) return fail(h, BDEPTH_ERR_NCCL, "%s", N.err.c_str());
        int rc = init_device(h); if (rc) return rc;
        memcpy(h->uid.b, nccl_unique_id, 128);
        NK(N.CommInitRank(&h->comm, world, h->uid, rank));
    }
    return 0;
}
int bdepth_nccl_unique_id(void* out128) {
    NcclApi& N = nccl();
    if (!N.ok) return fail(nullptr, BDEPTH_ERR_NCCL, "%s", N.err.c_str());
    NcclUid u; int r = N.GetUniqueId(&u);
    if (r) return fail(nullptr, BDEPTH_ERR_NCCL, "ncclGetUniqueId: %s", N.GetErrorString(r));
    memcpy(out128, u.b, 128);
    return 0;
}
// Host-only shard planning: needs the BGZF block index and the BAI, no device.
int bdepth_plan_shards(const char* bam_path, int world, uint64_t* out) {
    if (!bam_path || world < 1 || (world > 1 && !out)) return fail(nullptr, BDEPTH_ERR_ARG, "bad argument");
    int fd = open(bam_path, O_RDONLY); if (fd < 0) return fail(nullptr, BDEPTH_ERR_IO, "cannot open %s", bam_path);
    struct stat sb; fstat(fd, &sb);
    void* m = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
    if (m == MAP_FAILED) { close(fd); return fail(nullptr, BDEPTH_ERR_IO, "cannot mmap %s", bam_path); }
    std::vector<HostBlock> blocks; uint64_t tu = 0;
    std::string e = index_bgzf((const uint8_t*)m, (size_t)sb.st_size, blocks, &tu);
    munmap(m, (size_t)sb.st_size); close(fd);
    if (!e.empty()) return fail(nullptr, BDEPTH_ERR_FORMAT, "%s", e.c_str());
    BaiIndex bai;
    { std::string p1 = std::string(bam_path) + ".bai"; FILE* f = fopen(p1.c_str(), "rb"); if (!f) return fail(nullptr, BDEPTH_ERR_NOINDEX, "no index %s", p1.c_str());
      fseek(f, 0, SEEK_END); long n = ftell(f); fseek(f, 0, SEEK_SET); std::vector<uint8_t> buf(n); if (fread(buf.data(), 1, n, f) != (size_t)n) { fclose(f); return fail(nullptr, BDEPTH_ERR_IO, "read error"); } fclose(f);
      if (!parse_bai(buf.data(), buf.size(), bai)) return fail(nullptr, BDEPTH_ERR_FORMAT, "bad BAI"); }
    std::vector<uint64_t> vos = shard_candidates(bai);
    for (int k = 1; k < world; k++) out[k - 1] = shard_cut_voffset(vos, (uint64_t)sb.st_size, k, world);
    return 0;
}
// Host-only: the merged BAI chunk list a region query reads (what bdepth_run_* stage when regions are set).
long bdepth_plan_region_chunks(const char* bam_path, const bdepth_region* regions, size_t n, uint64_t* out_pairs, size_t cap) {
    if (!bam_path || (n && !regions)) return fail(nullptr, BDEPTH_ERR_ARG, "bad argument");
    BaiIndex bai;
    { std::string p1 = std::string(bam_path) + ".bai"; FILE* f = fopen(p1.c_str(), "rb"); if (!f) return fail(nullptr, BDEPTH_ERR_NOINDEX, "no index %s", p1.c_str());
      fseek(f, 0, SEEK_END); long nb = ftell(f); fseek(f, 0, SEEK_SET); std::vector<uint8_t> buf(nb); if (fread(buf.data(), 1, nb, f) != (size_t)nb) { fclose(f); return fail(nullptr, BDEPTH_ERR_IO, "read error"); } fclose(f);
      if (!parse_bai(buf.data(), buf.size(), bai)) return fail(nullptr, BDEPTH_ERR_FORMAT, "bad BAI"); }
    std::vector<HostRegion> rg;
    for (size_t i = 0; i < n; i++) if (regions[i].start < regions[i].end) rg.push_back(HostRegion{regions[i].ref_id, regions[i].start, regions[i].end});
    std::sort(rg.begin(), rg.end(), [](const HostRegion& a, const HostRegion& b) { return a.ref != b.ref ? a.ref < b.ref : a.start < b.start; });
    std::vector<BaiChunk> cs = region_chunks(bai, rg);
    for (size_t i = 0; i < cs.size() && i < cap; i++) { out_pairs[2 * i] = cs[i].beg; out_pairs[2 * i + 1] = cs[i].end; }
    return (long)cs.size();
}
int bdepth_set_tuning(bdepth_t* h, uint64_t batch_inflated_bytes, uint64_t chunk_blocks) {
    if (batch_inflated_bytes) h->batch_u = std::max<uint64_t>(batch_inflated_bytes, 1 << 16);
    if (chunk_blocks) h->chunk_blocks = chunk_blocks;
    h->staged = false;
    return 0;
}

int bdepth_stage(bdepth_t* h) {
    int rc = init_device(h); if (rc) return rc;
    rc = prepare_shard(h); if (rc) return rc;
    if (h->blk_lo >= h->blk_hi) { h->staged = false; return 0; }
    const auto& B = h->blocks;
    uint64_t f0 = B[h->blk_lo].coff & ~3ull, f1 = B[h->blk_hi - 1].coff + B[h->blk_hi - 1].bsize;
    CK(h->comp.ensure(f1 - f0 + 256));
    CK(cudaMemcpyAsync(h->comp.p, h->file + f0, f1 - f0, cudaMemcpyHostToDevice, h->s_main));
    CK(cudaMemsetAsync((uint8_t*)h->comp.p + (f1 - f0), 0, 128, h->s_main));
    CK(cudaStreamSynchronize(h->s_main));
    h->staged = true; h->staged_file_off = f0;
    return 0;
}

// The part of the counter window this rank owns, window-relative: [a, b), empty when b <= a.  (A rank without a passing read of its own
// owns nothing -- own_lo = own_hi = 0 -- while its window begins at its shard: the differences must not wrap.)
static inline void owned_window(const bdepth* h, uint64_t& a, uint64_t& b) {
    const uint64_t lo = std::max(h->own_lo, h->cnt_base), hi = std::min(h->own_hi, h->cnt_base + h->win_len);
    if (hi > lo) { a = lo - h->cnt_base; b = hi - h->cnt_base; } else { a = b = 0; }
}

int bdepth_run_resident(bdepth_t* h) {
    int rc = run_all_inputs(h); if (rc) return rc;
    cudaStream_t sm = h->s_main;
    CK(cudaMemsetAsync(h->misc.p, 0, 8, sm));
    uint64_t a, b; owned_window(h, a, b);
    if (b > a) { BD_LAUNCH(COUNT_GRID, 256, 0, sm, k_count_covered)(h->counts.as<uint32_t>(), h->win_len, a, b, (unsigned long long*)h->misc.p, N_PLANES * (int)h->S); CK(cudaGetLastError()); h->st.gpu_launches++; }
    unsigned long long cov = 0; CK(cudaMemcpyAsync(&cov, h->misc.p, 8, cudaMemcpyDeviceToHost, sm)); CK(cudaStreamSynchronize(sm));
    h->st.covered_positions = cov;
    h->st.ms_total_device = h->st.ms_h2d + h->st.ms_inflate + h->st.ms_scan + h->st.ms_coverage + h->st.ms_exchange;
    return 0;
}

// ---- base mode: D2H of the counters in EMIT_CHUNK pieces, split at reference boundaries
int bdepth_run_base(bdepth_t* h, bdepth_tile_cb cb, void* user) {
    int rc = init_device(h); if (rc) return rc;
    rc = ensure_pinned(h, 2 * EMIT_CHUNK * N_PLANES * 4); if (rc) return rc;
    Emitter em{h, cb, user};
    // ranges to deliver: whole genome, or the merged regions (sorted)
    if (h->regions.empty()) { if (h->hdr.total_len) em.ranges.push_back({0, h->hdr.total_len}); }
    else for (auto& g : h->regions) em.ranges.push_back({h->hdr.ref_lin0[g.ref_id] + g.start, h->hdr.ref_lin0[g.ref_id] + g.end});
    rc = run_all_inputs(h, &em); if (rc) { em.finish(); return rc; }
    cudaStream_t sm = h->s_main;
    cudaEvent_t e0 = h->ev[5], e1 = h->ev[6];
    // covered positions (rows of default `depth base`), over the range this rank owns
    CK(cudaMemsetAsync(h->misc.p, 0, 8, sm));
    { uint64_t ca, cb2; owned_window(h, ca, cb2);
      if (cb2 > ca) { BD_LAUNCH(COUNT_GRID, 256, 0, sm, k_count_covered)(h->counts.as<uint32_t>(), h->win_len, ca, cb2, (unsigned long long*)h->misc.p, N_PLANES * (int)h->S); CK(cudaGetLastError()); h->st.gpu_launches++; } }
    unsigned long long cov = 0; CK(cudaMemcpyAsync(&cov, h->misc.p, 8, cudaMemcpyDeviceToHost, sm));
    CK(cudaEventRecord(e0, sm));
    if (h->world > 1) { em.lo_clip = h->own_lo; em.hi_clip = h->own_hi; }      // multi-GPU: ranks deliver disjoint, ordered pieces (what was delivered on the way lies inside)
    rc = em.advance(UINT64_MAX, e0); if (rc) { em.finish(); return rc; }
    rc = em.finish(); if (rc) return rc;
    CK(cudaEventRecord(e1, h->s_d2h)); CK(cudaStreamSynchronize(h->s_d2h)); CK(cudaStreamSynchronize(sm));
    h->st.covered_positions = cov;
    float t = 0; CK(cudaEventElapsedTime(&t, e0, e1)); h->st.ms_d2h = t;      // the part of the D2H that was not hidden behind the kernels
    h->st.ms_total_device = h->st.ms_h2d + h->st.ms_inflate + h->st.ms_scan + h->st.ms_coverage + h->st.ms_exchange + h->st.ms_d2h;
    return 0;
}

// ---- base mode with GPU-side text (SURVEY 8f rank 1)
int bdepth_run_base_text(bdepth_t* h, const bdepth_text_opts* o, bdepth_text_cb cb, void* user) {
    if (!o) return fail(h, BDEPTH_ERR_ARG, "null options");
    // a position that reads cover but whose every base fails -q still has a column: with -a and a positive minimum coverage
    // the reference prints it (flag n); the counters cannot tell it from an empty position, a bitmap can (one rank only)
    // (with -m a column can be empty as well: a read left in state `detected` without a partner is skipped, depth.d:521-525)
    const bool presence = o->annotate && (h->minq > 0 || h->fix_mates) && o->min_cov > 0 && h->world == 1;
    h->want_presence = presence;
    int rc = run_all_inputs(h); h->want_presence = false; if (rc) return rc;
    const bool ms = h->S > 1;             // one row per sample and position (k_text_len_ms / k_text_write_ms)
    cudaStream_t sm = h->s_main;
    cudaEvent_t e0 = h->ev[5], e1 = h->ev[6];
    CK(cudaEventRecord(e0, sm));
    CK(cudaMemsetAsync(h->misc.p, 0, 8, sm));
    { uint64_t ca, cb2; owned_window(h, ca, cb2);
      if (cb2 > ca) { BD_LAUNCH(COUNT_GRID, 256, 0, sm, k_count_covered)(h->counts.as<uint32_t>(), h->win_len, ca, cb2, (unsigned long long*)h->misc.p, N_PLANES * (int)h->S); CK(cudaGetLastError()); h->st.gpu_launches++; } }
    unsigned long long cov = 0; CK(cudaMemcpyAsync(&cov, h->misc.p, 8, cudaMemcpyDeviceToHost, sm));
    TextParams tp; memset(&tp, 0, sizeof tp);
    tp.min_cov = o->min_cov; tp.max_cov = o->max_cov; tp.annotate = o->annotate ? 1 : 0; tp.with_sample = h->combined ? 0 : 1;
    const std::string& sn = h->hdr.sample_names[0];
    if (sn.size() > 255) return fail(h, BDEPTH_ERR_ARG, "sample name too long");
    tp.sample_len = (uint32_t)sn.size(); memcpy(tp.sample, sn.data(), sn.size());
    TextParamsMS tpm; memset(&tpm, 0, sizeof tpm); size_t max_sample = sn.size();
    if (ms) {
        std::vector<char> names; std::vector<uint32_t> offs;
        for (uint32_t si = 0; si < h->S; si++) { const std::string& x = h->hdr.sample_names[si]; offs.push_back((uint32_t)names.size()); names.insert(names.end(), x.begin(), x.end()); max_sample = std::max(max_sample, x.size()); }
        offs.push_back((uint32_t)names.size());
        const size_t off_bytes = (names.size() + 15) & ~size_t(15);
        CK(h->text_samp.ensure(off_bytes + offs.size() * 4 + 16));
        if (!names.empty()) CK(cudaMemcpyAsync(h->text_samp.p, names.data(), names.size(), cudaMemcpyHostToDevice, sm));
        CK(cudaMemcpyAsync((uint8_t*)h->text_samp.p + off_bytes, offs.data(), offs.size() * 4, cudaMemcpyHostToDevice, sm));
        CK(cudaStreamSynchronize(sm));
        tpm.min_cov = o->min_cov; tpm.max_cov = o->max_cov; tpm.annotate = o->annotate ? 1 : 0; tpm.S = h->S;
        tpm.samp = h->text_samp.as<char>(); tpm.samp_off = (const uint32_t*)((uint8_t*)h->text_samp.p + off_bytes);
    }
    constexpr size_t TEXT_BUF = 128ull << 20;
    rc = ensure_pinned(h, std::max<size_t>(2 * TEXT_BUF, 2 * EMIT_CHUNK * N_PLANES * 4)); if (rc) return rc;
    CK(h->text[0].ensure(TEXT_BUF)); CK(h->text[1].ensure(TEXT_BUF));
    // linear ranges to print (whole genome or merged regions), clipped to what this rank owns, cut at reference ends,
    // at the counter-window edges (outside it every counter is zero) and into chunks whose text fits the buffer
    struct Piece { uint32_t ref; uint64_t a, b; bool in_window; };
    std::vector<Piece> pieces;
    // --min-coverage=0: the reference writes the empty rows of the references in front of the first one it sees reads on, of those behind the
    // last one, and of the gaps of the ones it sees -- but when the sweep moves from one reference to a later one, only the tail of the
    // former and the head of the latter are written (PerBasePrinter.push, depth.d:578-581): a reference in between, which has no column,
    // gets no rows at all.  (No reference with reads: close() writes every one, :597-599.)
    long first_seen = -1, last_seen = -1;
    { const size_t nref = h->hdr.ref_len.size(); for (size_t r = 0; r < nref && !h->ref_has_host.empty(); r++) if ((h->ref_has_host[r >> 5] >> (r & 31)) & 1) { if (first_seen < 0) first_seen = (long)r; last_seen = (long)r; } }
    auto ref_rows = [&](size_t ref) { return first_seen < 0 || (long)ref <= first_seen || (long)ref >= last_seen || ((h->ref_has_host[ref >> 5] >> (ref & 31)) & 1); };
    auto add_range = [&](uint64_t a, uint64_t b) {
        a = std::max(a, h->own_lo); b = std::min(b, h->own_hi);
        while (a < b) {
            size_t ref = std::upper_bound(h->hdr.ref_lin0.begin(), h->hdr.ref_lin0.end(), a) - h->hdr.ref_lin0.begin() - 1;
            while (ref < h->hdr.ref_len.size() && a >= h->hdr.ref_lin0[ref] + h->hdr.ref_len[ref]) ref++;
            if (ref >= h->hdr.ref_len.size()) break;
            uint64_t e = std::min(b, h->hdr.ref_lin0[ref] + h->hdr.ref_len[ref]);
            bool inw = a >= h->cnt_base && a < h->cnt_base + h->win_len;
            if (inw) e = std::min(e, h->cnt_base + h->win_len); else if (a < h->cnt_base) e = std::min(e, h->cnt_base);
            size_t max_row = (h->hdr.ref_names[ref].size() + max_sample + 96) * (ms ? h->S : 1);
            uint64_t cp = std::max<uint64_t>(TEXT_TILE, (TEXT_BUF / max_row) / TEXT_TILE * TEXT_TILE);
            e = std::min(e, a + cp);
            if (o->min_cov > 0 ? inw : ref_rows(ref)) pieces.push_back({(uint32_t)ref, a, e, inw});      // zero rows only exist when min_cov == 0 (a skipped reference has no read, so no row of any kind)
            a = e;
        }
    };
    if (h->regions.empty()) add_range(0, h->hdr.total_len);
    else for (auto& g : h->regions) add_range(h->hdr.ref_lin0[g.ref_id] + g.start, h->hdr.ref_lin0[g.ref_id] + g.end);
    uint64_t max_piece = 0; for (auto& p : pieces) max_piece = std::max(max_piece, p.b - p.a);
    CK(h->text_tiles.ensure((max_piece / TEXT_TILE + 2) * 4)); CK(h->text_offs.ensure((max_piece / TEXT_TILE + 2) * 8 + 16));
    bool need_zero = false; for (auto& p : pieces) need_zero |= !p.in_window;
    if (need_zero) { CK(h->text_zero.ensure(max_piece * 4 + 64)); CK(cudaMemsetAsync(h->text_zero.p, 0, max_piece * 4 + 64, sm)); }
    size_t pend_len[2] = {0, 0}; bool pend[2] = {false, false};
    auto deliver = [&](int slot) -> int {
        if (!pend[slot]) return 0;
        CK(cudaEventSynchronize(h->ev[8 + slot])); pend[slot] = false;
        if (cb && pend_len[slot] && cb(user, (const char*)h->pinned + (size_t)slot * TEXT_BUF, pend_len[slot])) return fail(h, BDEPTH_ERR_CALLBACK, "text callback aborted");
        return 0;
    };
    for (size_t i = 0; i < pieces.size(); i++) {
        const Piece& p = pieces[i]; int slot = (int)(i & 1);
        rc = deliver(slot); if (rc) return rc;                       // the slot's previous chunk must be consumed before reuse
        const std::string& nm = h->hdr.ref_names[p.ref];
        if (nm.size() > 255) return fail(h, BDEPTH_ERR_ARG, "reference name too long");
        tp.name_len = (uint32_t)nm.size(); memcpy(tp.name, nm.data(), nm.size());
        tpm.name_len = tp.name_len; memcpy(tpm.name, nm.data(), nm.size()); tpm.sample_stride = p.in_window ? (uint64_t)N_PLANES * h->win_len : 0;
        tp.present = tpm.present = (presence && p.in_window) ? h->present.as<uint32_t>() : nullptr;      // indexed like the counters (idx0 is window-relative)
        uint32_t n = (uint32_t)(p.b - p.a), n_tiles = (n + TEXT_TILE - 1) / TEXT_TILE, pos0 = (uint32_t)(p.a - h->hdr.ref_lin0[p.ref]);
        const uint32_t* cnt = p.in_window ? h->counts.as<uint32_t>() : h->text_zero.as<uint32_t>();
        uint64_t wl = p.in_window ? h->win_len : 0, idx0 = p.in_window ? p.a - h->cnt_base : 0;
        unsigned long long* tot_d = (unsigned long long*)((uint8_t*)h->text_offs.p + (size_t)(max_piece / TEXT_TILE + 2) * 8);
        if (ms) BD_LAUNCH(n_tiles, 256, 0, sm, k_text_len_ms)(tpm, cnt, wl, idx0, pos0, n, h->text_tiles.as<uint32_t>());
        else BD_LAUNCH(n_tiles, 256, 0, sm, k_text_len)(tp, cnt, wl, idx0, pos0, n, h->text_tiles.as<uint32_t>());
        BD_LAUNCH(1, 1024, 0, sm, k_text_scan)(h->text_tiles.as<uint32_t>(), n_tiles, (unsigned long long*)h->text_offs.p, tot_d);
        unsigned long long tot = 0; CK(cudaMemcpyAsync(&tot, tot_d, 8, cudaMemcpyDeviceToHost, sm));
        CK(cudaStreamSynchronize(sm));
        if (tot > TEXT_BUF) return fail(h, BDEPTH_ERR_ARG, "internal: text chunk larger than its buffer");
        if (tot) {
            if (ms) BD_LAUNCH(n_tiles, 256, 0, sm, k_text_write_ms)(tpm, cnt, wl, idx0, pos0, n, (const unsigned long long*)h->text_offs.p, h->text[slot].as<char>());
            else BD_LAUNCH(n_tiles, 256, 0, sm, k_text_write)(tp, cnt, wl, idx0, pos0, n, (const unsigned long long*)h->text_offs.p, h->text[slot].as<char>());
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync((char*)h->pinned + (size_t)slot * TEXT_BUF, h->text[slot].p, tot, cudaMemcpyDeviceToHost, sm));
        }
        h->st.gpu_launches += tot ? 3 : 2;
        CK(cudaEventRecord(h->ev[8 + slot], sm)); pend[slot] = true; pend_len[slot] = tot;
        rc = deliver(slot ^ 1); if (rc) return rc;                   // hand out the previous chunk while this one is in flight
    }
    rc = deliver(0); if (rc) return rc; rc = deliver(1); if (rc) return rc;
    CK(cudaEventRecord(e1, sm)); CK(cudaStreamSynchronize(sm));
    h->st.covered_positions = cov;
    float t = 0; CK(cudaEventElapsedTime(&t, e0, e1)); h->st.ms_d2h = t;
    h->st.ms_total_device = h->st.ms_h2d + h->st.ms_inflate + h->st.ms_scan + h->st.ms_coverage + h->st.ms_exchange + h->st.ms_d2h;
    return 0;
}

// How many samples one pass of a region / window run counts: at most 64 (the sample field of RecordSoA.meta), at most what the
// counter window leaves room for in HBM (the arithmetic of the check in run_pipeline_body), at most bdepth_set_samples_per_pass.
// Several ranks take the smallest answer of any of them, so that their passes -- and the collectives inside -- line up.
static int pass_group_size(bdepth* h, size_t NS, uint32_t& G) {
    const uint32_t cap = h->samples_per_pass ? std::min<uint32_t>(h->samples_per_pass, 64) : 64;
    G = cap;
    const bool shared = h->world > 1 && h->comm;
    if (NS <= 1 || (shared && NS <= cap)) return 0;      // (several ranks: decided from what they all know)
    // the counter window as run_all_inputs takes it, the union of what the inputs' indices say: no smaller than any rank's own
    uint64_t lo = UINT64_MAX, hi = 0;
    for (size_t i = 0; i <= h->extra.size(); i++) {
        if (i) swap_inputs(h, h->extra[i - 1]);
        uint64_t a, b; index_extent(h, a, b); lo = std::min(lo, a); hi = std::max(hi, b);
        if (i) swap_inputs(h, h->extra[i - 1]);
    }
    const uint64_t base = lo / TILE_POS * TILE_POS, win = ((hi - base + TILE_POS - 1) / TILE_POS + 1) * TILE_POS;
    size_t free_b = 0, tot_b = 0; CK(cudaMemGetInfo(&free_b, &tot_b));
    const uint64_t fit = (free_b + h->counts.cap) / (win * N_PLANES * 4);
    G = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(G, fit));      // (nothing fits: one sample, refused by the check itself)
    if (shared) {
        cudaStream_t sm = h->s_main; DevBuf mine, all; CK(mine.ensure(16)); CK(all.ensure(16 * (size_t)h->world));
        CK(cudaMemcpyAsync(mine.p, &G, 4, cudaMemcpyHostToDevice, sm));
        NK(nccl().AllGather(mine.p, all.p, 1, NCCL_UINT32, h->comm, sm));
        std::vector<uint32_t> v((size_t)h->world); CK(cudaMemcpyAsync(v.data(), all.p, 4 * (size_t)h->world, cudaMemcpyDeviceToHost, sm)); CK(cudaStreamSynchronize(sm));
        G = *std::min_element(v.begin(), v.end());
        mine.release(); all.release();
    }
    return 0;
}

// Shared by window and region modes.  segs: output-order list of (ref, start, end) with end possibly
// past the reference end (windows); stats are computed over the part inside the reference.
// Results are laid out [sample][segment].  When the samples' counters do not fit at once (more than 64 samples, HBM, or
// bdepth_set_samples_per_pass), the pipeline runs once per group of samples and each pass fills its samples' part.
struct SegDef { uint32_t ref, start, end; uint32_t cov_ext = 0;  /* thresholds are counted from start - cov_ext */ uint32_t min_read_start = 0;  /* != 0: only reads starting at/after it count (quirk 6) */ };
static int run_segments(bdepth* h, const std::vector<SegDef>& segs, const uint32_t* thr, size_t n_thr,
                        std::vector<uint32_t>& reads, std::vector<uint32_t>& bases, std::vector<uint32_t>& cov) {
    int rc = init_device(h); if (rc) return rc;
    const size_t n = segs.size();
    const size_t NS = (h->combined || h->hdr.sample_names.size() <= 1) ? 1 : h->hdr.sample_names.size();   // layout: [sample][..]
    const size_t nt1 = std::max<size_t>(n_thr, 1);
    uint32_t G = 0; rc = pass_group_size(h, NS, G); if (rc) return rc;
    const size_t n_pass = (NS + G - 1) / G, PS = n_pass > 1 ? G : NS;      // PS: counter sets on the device at once
    if (n_pass > 1 && h->fix_mates) return fail(h, BDEPTH_ERR_ARG, "fix-mate-overlaps counts every sample in one pass: %zu samples need %zu passes of at most %u samples (use --combined)", NS, n_pass, G);
    reads.assign(NS * n, 0); bases.assign(NS * n, 0); cov.assign(NS * n * nt1, 0);
    // linear-coordinate segments, clipped to the reference
    std::vector<uint64_t> a(n), b(n);
    for (size_t i = 0; i < n; i++) {
        uint64_t L = h->hdr.ref_len[segs[i].ref], l0 = h->hdr.ref_lin0[segs[i].ref];
        a[i] = l0 + std::min<uint64_t>(segs[i].start, L); b[i] = l0 + std::min<uint64_t>(segs[i].end, L);
        if (b[i] < a[i]) b[i] = a[i];
    }
    // sorted view for the per-read kernel
    std::vector<uint32_t> order(n); for (size_t i = 0; i < n; i++) order[i] = (uint32_t)i;
    if (!std::is_sorted(a.begin(), a.end()))      // windows and a sorted BED already are: 310 k windows would cost ~20 ms to sort again
        std::sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return a[x] != a[y] ? a[x] < a[y] : x < y; });
    std::vector<uint64_t> ss(n), se(n), pm(n), ms(n), us(n); uint64_t mx = 0, ext_max = 0; bool has_min = false, has_u = false;
    for (size_t i = 0; i < n; i++) {
        ss[i] = a[order[i]]; se[i] = b[order[i]]; mx = std::max(mx, se[i]); pm[i] = mx;
        const SegDef& sd = segs[order[i]]; ms[i] = sd.min_read_start ? h->hdr.ref_lin0[sd.ref] + sd.min_read_start : 0; has_min |= ms[i] != 0;
        // first column in which the reference updates this slot (thresholds and, with -m, the per-column terms start there)
        uint64_t sc = sd.start - std::min(sd.cov_ext, sd.start);
        us[i] = std::min(ss[i], h->hdr.ref_lin0[sd.ref] + std::min<uint64_t>(sc, h->hdr.ref_len[sd.ref])); has_u |= sd.cov_ext != 0 || sd.min_read_start != 0; ext_max = std::max<uint64_t>(ext_max, ss[i] - us[i]);
    }
    auto& S = h->seg;
    size_t nn = n ? n : 1;
    CK(S.s.ensure(nn * 8)); CK(S.e.ensure(nn * 8)); CK(S.pmax.ensure(nn * 8)); CK(S.id.ensure(nn * 4)); CK(S.reads.ensure(PS * nn * 4)); CK(S.minstart.ensure(nn * 8)); CK(S.bases_reads.ensure(PS * nn * 4)); CK(S.mbases.ensure(PS * nn * 4));
    if (n) {
        CK(cudaMemcpy(S.s.p, ss.data(), n * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(S.e.p, se.data(), n * 8, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(S.pmax.p, pm.data(), n * 8, cudaMemcpyHostToDevice)); CK(cudaMemcpy(S.id.p, order.data(), n * 4, cudaMemcpyHostToDevice));
    }
    if (n) CK(cudaMemcpy(S.minstart.p, ms.data(), n * 8, cudaMemcpyHostToDevice));
    CK(S.ustart.ensure(nn * 8)); if (n) CK(cudaMemcpy(S.ustart.p, us.data(), n * 8, cudaMemcpyHostToDevice));
    CK(S.da.ensure(nn * 8)); CK(S.dac.ensure(nn * 8)); CK(S.db.ensure(nn * 8)); CK(S.dthr.ensure(std::max<size_t>(64, n_thr * 4))); if (n_thr > 16) CK(S.dscr.ensure(PS * nn * 4)); CK(S.dbases.ensure(PS * nn * 4)); CK(S.dcov.ensure(PS * nn * 4 * nt1));
    S.has_min = has_min; S.has_u = has_u; S.ext_max = ext_max;
    SamplePass spass; spass.counted.assign(h->extra.size() + 1, 0); spass.untagged.assign(h->extra.size() + 1, 0);
    bdepth_stats total{}; float ms_reduce = 0, ms_exchange = 0; std::vector<uint32_t> has_union;
    std::vector<uint64_t> wa(n), wb(n), acv(n);      // window-relative segment bounds of a pass (allocated here: not between the device events of the reduction)
    for (size_t pi = 0; pi < n_pass; pi++) {
    const size_t g0 = n_pass > 1 ? (pi + 1) % n_pass * G : 0, gn = std::min(PS, NS - g0);      // (the group that holds sample 0 runs last: SamplePass)
    h->pass_g0 = (uint32_t)g0; h->pass_n = n_pass > 1 ? (uint32_t)gn : 0;
    CK(cudaMemset(S.reads.p, 0, PS * nn * 4)); CK(cudaMemset(S.bases_reads.p, 0, PS * nn * 4)); CK(cudaMemset(S.mbases.p, 0, PS * nn * 4));
    S.on = true; S.n = (uint32_t)n;
    rc = run_all_inputs(h, nullptr, n_pass > 1 ? &spass : nullptr);
    S.on = false; h->pass_g0 = h->pass_n = 0;
    if (rc) return rc;
    cudaStream_t sm = h->s_main;
    cudaEvent_t e0 = h->ev[5], e1 = h->ev[6];
    CK(cudaEventRecord(e0, sm));
    // per-segment sums over the counters (original order)
    DevBuf &da = S.da, &dac = S.dac, &db = S.db, &dthr = S.dthr, &dbases = S.dbases, &dcov = S.dcov;      // the handle's (sized before the pipeline ran, released with it): no allocation per call
    std::vector<uint32_t> qbases, mbases;
    for (size_t i = 0; i < n; i++) {
        uint64_t lo = std::max(h->cnt_base, h->own_lo), hi = std::min(h->cnt_base + h->win_len, h->own_hi); if (hi < lo) hi = lo;
        uint64_t sc = segs[i].start - std::min(segs[i].cov_ext, segs[i].start);
        uint64_t acov = h->hdr.ref_lin0[segs[i].ref] + std::min<uint64_t>(sc, h->hdr.ref_len[segs[i].ref]);
        uint64_t xa = std::min(std::max(a[i], lo), hi), xb = std::min(std::max(b[i], lo), hi), xc = std::min(std::max(acov, lo), hi);
        wa[i] = xa - h->cnt_base; wb[i] = xb - h->cnt_base; acv[i] = xc - h->cnt_base;
    }
    if (n) { CK(cudaMemcpyAsync(da.p, wa.data(), n * 8, cudaMemcpyHostToDevice, sm)); CK(cudaMemcpyAsync(dac.p, acv.data(), n * 8, cudaMemcpyHostToDevice, sm)); CK(cudaMemcpyAsync(db.p, wb.data(), n * 8, cudaMemcpyHostToDevice, sm)); }
    if (n_thr) CK(cudaMemcpyAsync(dthr.p, thr, n_thr * 4, cudaMemcpyHostToDevice, sm));
    CK(cudaMemsetAsync(dbases.p, 0, PS * nn * 4, sm)); CK(cudaMemsetAsync(dcov.p, 0, PS * nn * 4 * nt1, sm));
    if (n) {
        for (size_t si = 0; si < gn; si++) {
            // the kernel keeps 16 threshold counters in registers: more thresholds (the reference has no limit) take further passes over the segments,
            // whose base sums go to a scratch array (they were added by the first pass)
            for (size_t t0 = 0; t0 < std::max<size_t>(n_thr, 1); t0 += 16) {
                const uint32_t nt = n_thr ? (uint32_t)std::min<size_t>(16, n_thr - t0) : 0u;
                BD_LAUNCH((unsigned)((n * 32 + 255) / 256), 256, 0, sm, k_segment_stats)(h->counts.as<uint32_t>() + (uint64_t)si * N_PLANES * h->win_len, h->win_len, da.as<uint64_t>(), dac.as<uint64_t>(), db.as<uint64_t>(), (uint32_t)n, dthr.as<uint32_t>() + t0, nt,
                                                                                          (t0 ? S.dscr.as<uint32_t>() : dbases.as<uint32_t>()) + si * n, dcov.as<uint32_t>() + si * n * nt1 + t0 * n);
                CK(cudaGetLastError()); h->st.gpu_launches++;
            }
        }
        if (h->world > 1 && h->comm) {   // per-segment partial sums are additive over ranks; a failed collective is an error, never a partial sum handed out as the result
            NcclApi& N = nccl();
            NK(N.AllReduce(dbases.p, dbases.p, gn * n, NCCL_UINT32, NCCL_SUM, h->comm, sm));
            if (n_thr) NK(N.AllReduce(dcov.p, dcov.p, gn * n * n_thr, NCCL_UINT32, NCCL_SUM, h->comm, sm));
            NK(N.AllReduce(S.reads.p, S.reads.p, gn * n, NCCL_UINT32, NCCL_SUM, h->comm, sm));
            if (has_min) NK(N.AllReduce(S.bases_reads.p, S.bases_reads.p, gn * n, NCCL_UINT32, NCCL_SUM, h->comm, sm));
            if (h->fix_mates) NK(N.AllReduce(S.mbases.p, S.mbases.p, gn * n, NCCL_UINT32, NCCL_SUM, h->comm, sm));
        }
        CK(cudaMemcpyAsync(bases.data() + g0 * n, dbases.p, gn * n * 4, cudaMemcpyDeviceToHost, sm));
        if (n_thr) CK(cudaMemcpyAsync(cov.data() + g0 * n * nt1, dcov.p, gn * n * n_thr * 4, cudaMemcpyDeviceToHost, sm));
        CK(cudaMemcpyAsync(reads.data() + g0 * n, S.reads.p, gn * n * 4, cudaMemcpyDeviceToHost, sm));
        if (has_min) { qbases.resize(gn * n); CK(cudaMemcpyAsync(qbases.data(), S.bases_reads.p, gn * n * 4, cudaMemcpyDeviceToHost, sm)); }
        if (h->fix_mates || h->world == 1) { mbases.resize(gn * n); CK(cudaMemcpyAsync(mbases.data(), S.mbases.p, gn * n * 4, cudaMemcpyDeviceToHost, sm)); }      // what n_bases has on top of the base planes: -m (mates.cuh), CIGARs that begin with N (k2_lead_n; zero otherwise)
    }
    CK(cudaEventRecord(e1, sm));
    CK(cudaStreamSynchronize(sm));
    CK(cudaGetLastError());
    if (!qbases.empty()) for (size_t si = 0; si < gn; si++) for (size_t i = 0; i < n; i++) if (segs[i].min_read_start) bases[(g0 + si) * n + i] = qbases[si * n + i];
    if (!mbases.empty()) for (size_t k = 0; k < gn * n; k++) bases[g0 * n + k] += mbases[k];
    float t = 0; CK(cudaEventElapsedTime(&t, e0, e1)); ms_reduce += t; ms_exchange += h->st.ms_exchange;
    if (n_pass > 1) {      // a reference has reads if it has them in any pass
        add_stats(total, h->st);
        if (has_union.empty()) has_union = h->ref_has_host; else for (size_t k = 0; k < has_union.size(); k++) has_union[k] |= h->ref_has_host[k];
    }
    }   // sample passes
    if (n_pass > 1) {
        const bdepth_stats last = h->st;
        h->st = total; h->st.positions = last.positions; h->st.own_lo = last.own_lo; h->st.own_hi = last.own_hi; h->st.halo_bytes_sent = last.halo_bytes_sent; h->st.ms_exchange = ms_exchange;
        h->ref_has_host = has_union;
    }
    h->st.n_sample_passes = (uint32_t)n_pass;
    h->st.ms_reduce = ms_reduce;
    h->st.ms_total_device = h->st.ms_h2d + h->st.ms_inflate + h->st.ms_scan + h->st.ms_coverage + h->st.ms_reduce;
    return 0;
}

// results are laid out [sample][segment] (cov: [sample][threshold][segment]); delivery order is the reference's:
// regions outer, samples inner (depth.d:925-930, :946-949)
static int deliver_one(bdepth* h, const SegDef& sd, size_t i, size_t n, size_t n_thr, const std::vector<uint32_t>& reads, const std::vector<uint32_t>& bases,
                       const std::vector<uint32_t>& cov, bool zero, bdepth_stat_cb cb, void* user, uint64_t idx) {
    const size_t NS = (h->combined || h->hdr.sample_names.size() <= 1) ? 1 : h->hdr.sample_names.size(), nt1 = std::max<size_t>(n_thr, 1);
    std::vector<uint32_t> c(nt1, 0);
    for (size_t si = 0; si < NS; si++) {
        if (!zero) for (size_t t = 0; t < n_thr; t++) c[t] = cov[si * n * nt1 + t * n + i];
        bdepth_region_stat st{(int32_t)sd.ref, sd.start, sd.end, zero ? 0u : reads[si * n + i], zero ? 0u : bases[si * n + i], c.data(), (int32_t)si};
        if (cb(user, &st, idx)) return fail(h, BDEPTH_ERR_CALLBACK, "stat callback aborted");
    }
    return 0;
}

int bdepth_run_windows(bdepth_t* h, uint32_t window, uint32_t overlap, const uint32_t* thr, size_t n_thr, bdepth_stat_cb cb, void* user) {
    if (!h) return BDEPTH_ERR_ARG;
    if (window == 0) return fail(h, BDEPTH_ERR_ARG, "positive window size must be specified");
    if (!(overlap < window)) return fail(h, BDEPTH_ERR_ARG, "specified overlap is larger than window size");      // (depth.d:959; a step of zero has no next window)
    // -m: a window is a segment with an update range (ring slots are updated before their window begins when the step does
    // not divide the window) and, for reference 0's first slots, without a first occurrence; mates.cuh replays both.
    const uint32_t step = window - overlap;
    const uint32_t nslot = (window + step - 1) / step;          // ring slots of PerWindowPrinter (depth.d:1026-1029)
    const uint32_t ext = nslot * step - window;                  // a slot reused for window m >= nslot starts collecting
                                                                 // thresholds `ext` positions before the window (WindowStatsCollector
                                                                 // updates all nslot slots once position >= window, depth.d:215-226)
    // every window slot the reference could print: full windows when the reference has reads
    // (depth.d:1057,1071), ref_length / step windows when it has none (printEmptyWindows, depth.d:1039-1044)
    std::vector<SegDef> segs; std::vector<uint32_t> n_full(h->hdr.ref_len.size()), n_empty(h->hdr.ref_len.size()); std::vector<size_t> first(h->hdr.ref_len.size());
    for (size_t r = 0; r < h->hdr.ref_len.size(); r++) {
        uint64_t L = h->hdr.ref_len[r];
        n_full[r] = L >= window ? (uint32_t)((L - window) / step + 1) : 0; n_empty[r] = (uint32_t)(L / step);
        // + nslot: the ring's content after the last full window (partial windows at the reference end), see below
        uint32_t m = std::max(n_full[r] + nslot, n_empty[r]); first[r] = segs.size();
        for (uint32_t k = 0; k < m; k++) {
            SegDef sd{(uint32_t)r, k * step, k * step + window};
            if (k >= nslot) sd.cov_ext = ext;
            // slots start with is_first_occurrence == false (depth.d:1031-1032); until a slot has been finished once it only
            // counts reads that start inside it.  That affects windows 1..nslot-1 of reference 0 (later references are
            // preceded by resetAllWindows, depth.d:951-960).
            if (r == 0 && k >= 1 && k < nslot) sd.min_read_start = k * step;
            segs.push_back(sd);
        }
    }
    std::vector<uint32_t> reads, bases, cov;
    int rc = run_segments(h, segs, thr, n_thr, reads, bases, cov); if (rc) return rc;
    // Which slots the reference prints: full windows of references with reads (depth.d:1057,1071), length/step
    // windows of references without (printEmptyWindows, depth.d:1039-1044).  Quirk kept for drop-in output: in
    // close() (depth.d:1070-1076) the FIRST trailing reference without reads is printed before the window state is
    // reset, so its windows continue from where the last reference with reads stopped -- and its first nslot rows
    // carry what the ring still holds: the statistics of the partial windows at the end of that last reference.
    const size_t nref = h->hdr.ref_len.size();
    long last_has = -1;
    for (size_t r = 0; r < nref; r++) if ((h->ref_has_host[r >> 5] >> (r & 31)) & 1) last_has = (long)r;
    if (!cb) return 0;
    uint64_t idx = 0;
    for (size_t r = 0; r < nref; r++) {
        bool has = (h->ref_has_host[r >> 5] >> (r & 31)) & 1;
        uint32_t m = has ? n_full[r] : n_empty[r];
        const bool carry = !has && last_has >= 0 && (long)r == last_has + 1;      // (also when that reference was shorter than a window: shift 0, the ring holds its only, partial, window)
        const uint32_t shift = carry ? n_full[last_has] * step : 0;
        for (uint32_t k = 0; k < m; k++) {
            size_t i = first[r] + k;
            SegDef sd = segs[i];
            if (carry) { sd = SegDef{(uint32_t)r, shift + k * step, shift + k * step + window}; i = first[last_has] + n_full[last_has] + k; }
            rc = deliver_one(h, sd, i, segs.size(), n_thr, reads, bases, cov, carry && k >= nslot, cb, user, idx++); if (rc) return rc;
        }
    }
    return 0;
}

int bdepth_run_regions(bdepth_t* h, const bdepth_region* regions, size_t n, const uint32_t* thr, size_t n_thr, bdepth_stat_cb cb, void* user) {
    std::vector<SegDef> segs(n);
    for (size_t i = 0; i < n; i++) {
        if (regions[i].ref_id >= h->hdr.ref_len.size()) return fail(h, BDEPTH_ERR_ARG, "region %zu: reference id out of range", i);
        segs[i] = SegDef{regions[i].ref_id, regions[i].start, regions[i].end};
    }
    std::vector<uint32_t> reads, bases, cov;
    // only reads overlapping a region matter: let the pipeline stage just the BAI chunks of these regions
    const bool tmp_regions = h->regions.empty() && n;
    if (tmp_regions) normalize_regions(h, regions, n, h->regions);
    int rc = run_segments(h, segs, thr, n_thr, reads, bases, cov);
    if (tmp_regions) h->regions.clear();
    if (rc) return rc;
    if (!cb) return 0;
    for (size_t i = 0; i < n; i++) { rc = deliver_one(h, segs[i], i, n, n_thr, reads, bases, cov, false, cb, user, i); if (rc) return rc; }
    return 0;
}

// ---- BAI builder ------------------------------------------------------------------------------------------------------------------
// The per-run part of IndexBuilder (bai/indexing.d): chunks from the runs (updateChunks :219-246), metadata (:117-131, :198-203), the
// linear index with its gaps filled from the left (:163-182), empty references (:98-101), n_no_coor (:348).  Bins are written in
// ascending order (the reference: iteration order of a D associative array, :188 -- not defined by anything but that runtime).
static int assemble_bai(bdepth* h) {
    auto& X = h->ix; const auto& B = h->blocks; const size_t nref = h->hdr.ref_len.size();
    std::vector<unsigned long long> lin(X.n_lin + 1), nm(nref + 1), nu(nref + 1); std::vector<uint32_t> ll(nref + 1);
    IndexCtl ctl; IndexCarry carry;
    CK(cudaMemcpy(lin.data(), X.lin.p, (X.n_lin + 1) * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(ll.data(), X.lin_len.p, (nref + 1) * 4, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(nm.data(), X.n_mapped.p, (nref + 1) * 8, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(nu.data(), X.n_unmapped.p, (nref + 1) * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&ctl, X.ctl.p, sizeof ctl, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(&carry, X.carry.p, sizeof carry, cudaMemcpyDeviceToHost));
    const uint64_t end_coff = B.empty() ? 0 : B.back().coff + B.back().bsize;
    auto vo = [&](uint64_t u) -> uint64_t {      // BgzfInputStream.virtualTell() at inflated offset u: the end of a member is the start of the next one
        if (B.empty() || u >= h->total_u) return end_coff << 16;
        size_t lo = 0, hi = B.size(); while (lo + 1 < hi) { size_t m = (lo + hi) / 2; if (B[m].uoff <= u) lo = m; else hi = m; }
        return (B[lo].coff << 16) | (u - B[lo].uoff);
    };
    std::vector<uint8_t>& out = h->built_bai; out.clear();
    auto p32 = [&](uint32_t v) { for (int i = 0; i < 4; i++) out.push_back((uint8_t)(v >> (8 * i))); };
    auto p64 = [&](uint64_t v) { p32((uint32_t)v); p32((uint32_t)(v >> 32)); };
    out.insert(out.end(), {'B', 'A', 'I', 1}); p32((uint32_t)nref);
    const auto& R = X.h_runs; const auto& E = X.h_excs;
    size_t next_ref = 0, e_i = 0;
    for (size_t i0 = 0; i0 < R.size();) {
        size_t i1 = i0; while (i1 < R.size() && R[i1].ref == R[i0].ref) i1++;
        const size_t r = (size_t)R[i0].ref;
        for (; next_ref < r; next_ref++) { p32(0); p32(0); }
        std::map<uint32_t, std::vector<std::pair<uint64_t, uint64_t>>> bins;
        for (size_t k = i0; k < i1; k++) {
            const uint64_t beg = vo(R[k].prev_end_abs == ~0ull ? R[k].start_abs : R[k].prev_end_abs), end = vo(k + 1 < R.size() ? R[k + 1].prev_end_abs : carry.end_abs);
            auto& cs = bins[R[k].bin];
            if (cs.empty() || (cs.back().second >> 16) != (beg >> 16)) cs.push_back({beg, end}); else cs.back().second = end;
        }
        // metadata: reads with a reference but no position count where the stream stood (before the next reference's first valid read)
        const uint64_t next_start = i1 < R.size() ? R[i1].start_abs : UINT64_MAX;
        uint64_t mapped = nm[r], unmapped = nu[r], end_abs = i1 < R.size() ? R[i1].prev_end_abs : carry.end_abs;
        for (; e_i < E.size() && E[e_i].start_abs < next_start; e_i++) { if (E[e_i].unmapped) unmapped++; else mapped++; if (E[e_i].end_abs > end_abs) end_abs = E[e_i].end_abs; }
        const uint64_t beg_vo = i0 == 0 ? vo(ctl.first_placed_abs) : vo(R[i0].prev_end_abs);
        p32((uint32_t)bins.size() + 1);
        for (auto& kv : bins) { p32(kv.first); p32((uint32_t)kv.second.size()); for (auto& c : kv.second) { p64(c.first); p64(c.second); } }
        p32(37450); p32(2); p64(beg_vo); p64(vo(end_abs)); p64(mapped); p64(unmapped);
        p32(ll[r]);
        uint64_t last = 0;
        for (uint32_t w = 0; w < ll[r]; w++) { unsigned long long a = lin[X.base[r] + w]; uint64_t v = a == ~0ull ? 0 : vo(a); if (v == 0) v = last; else last = v; p64(v); }
        next_ref = r + 1; i0 = i1;
    }
    for (; next_ref < nref; next_ref++) { p32(0); p32(0); }
    p64(ctl.no_coord);
    return 0;
}

int64_t bdepth_build_index(bdepth_t* h, void* dst, uint64_t cap) {
    if (!h) return BDEPTH_ERR_ARG;
    if (h->world > 1) return fail(h, BDEPTH_ERR_ARG, "the index is built by one rank (the shards of a run are cut from it)");
    if (h->built_bai.empty()) {
        const bool save_staged = h->staged; h->staged = false;
        int rc = run_pipeline(h, RUN_INDEX, nullptr);
        h->staged = save_staged;
        if (rc) return rc;
        rc = assemble_bai(h); if (rc) return rc;
        h->ix.h_runs.clear(); h->ix.h_runs.shrink_to_fit(); h->ix.h_excs.clear();
        // the handle adopts what it built: sharding, counter windows and region queries work on un-indexed input from here on
        h->bai = BaiIndex{}; if (!parse_bai(h->built_bai.data(), h->built_bai.size(), h->bai)) return fail(h, BDEPTH_ERR_FORMAT, "internal: the built index does not parse");
        h->has_index = true; h->sparse_ok = true; h->bai_window_ok = true; h->shard_ready = false;
    }
    if (dst && cap >= h->built_bai.size()) memcpy(dst, h->built_bai.data(), h->built_bai.size());
    return (int64_t)h->built_bai.size();
}

int bdepth_ref_has_reads(const bdepth_t* h, int ref) {
    if (ref < 0 || (size_t)ref >= h->hdr.ref_len.size() || h->ref_has_host.empty()) return 0;
    return (h->ref_has_host[ref >> 5] >> (ref & 31)) & 1;
}

int bdepth_get_stats(const bdepth_t* h, bdepth_stats* out) { if (!h || !out) return BDEPTH_ERR_ARG; *out = h->st; return 0; }

int64_t bdepth_inflate_to_host(bdepth_t* h, void* dst, uint64_t cap) {
    RunOut ro; ro.inflate_dst = (uint8_t*)dst; ro.inflate_cap = cap;
    // whole shard block range, including header blocks, so the result is comparable to a plain inflate of the file
    int rc = init_device(h); if (rc) return rc;
    rc = prepare_shard(h); if (rc) return rc;
    size_t save_lo = h->blk_lo; if (h->world == 1) h->blk_lo = 0;
    bool save_staged = h->staged; h->staged = false;
    rc = run_pipeline(h, RUN_INFLATE_ONLY, &ro);
    h->blk_lo = save_lo; h->staged = save_staged;
    if (rc) return rc;
    return (int64_t)ro.inflate_len;
}

int64_t bdepth_scan_to_host(bdepth_t* h, uint64_t cap, int32_t* ref_id, int32_t* pos, uint32_t* span, uint16_t* flag, uint8_t* mapq, uint16_t* n_cigar, uint64_t* rec_off) {
    RunOut ro; ro.scan_cap = cap; ro.ref_id = ref_id; ro.pos = pos; ro.span = span; ro.flag = flag; ro.mapq = mapq; ro.n_cigar = n_cigar; ro.rec_off = rec_off;
    int rc = run_pipeline(h, RUN_SCAN_ONLY, &ro);
    if (rc) return rc;
    return (int64_t)ro.scan_n;
}

}  // extern "C"
