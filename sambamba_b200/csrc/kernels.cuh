// kernels.cuh -- the sm_100a kernels of the depth hot path.
//
//   K1  k1_inflate          lane-per-BGZF-block DEFLATE (inflate_core.cuh)
//   K2  k2_guess_entries    first record start of every BGZF block (speculative, verified)
//       k2_walk             per-block record chain walk -> record offsets, exit offset
//       k2_decode           record header + CIGAR -> columnar SoA (warp per block)
//   K3  k3_tile_index       per-tile read ranges (tile_first / tile_lo)
//       k3_gather           per-position gather: every thread owns 4 consecutive positions and
//                           accumulates all reads covering them in registers (no atomics)
//       k3_scatter_long     reads spanning > SPAN_SHORT (spliced / long reads): warp per read,
//                           RED atomics
//   R   k_tile_covered, k_bucket_stats, k_read_windows, k_read_regions : reducers for the
//       base / window / region front ends
//
// Semantics restated (file:line under /root/reference):
//   record layout      BioD/bio/std/hts/bam/read.d:907-1003, readrange.d:118-173
//   CIGAR predicates   BioD/bio/std/hts/bam/cigar.d:58-148 (CIGAR_TYPE :116)
//   filter             sambamba/depth.d:1159, filtering.d:163-167,194-214
//   basesCovered()>0   BioD/bio/std/hts/bam/pileup.d:509-519, read.d:255-262
//   per-base counters  sambamba/depth.d:495-556 (writeColumn), base.d:186 (nt16 -> nt5)
//   region/window      sambamba/depth.d:661-698 (countRead), :760-845 (push), :847-876
#pragma once
#include "launch.cuh"
#include <stdint.h>
#include "inflate_core.cuh"
#include "inflate2_core.cuh"
#include "filter.cuh"

namespace bdk {

constexpr int TILE_POS = 1024;          // positions per K3 CTA (256 threads x 4)
constexpr uint32_t SPAN_SHORT = 1024;   // reads spanning more go to the scatter path
constexpr int N_PLANES = 7;
// "no record starts in this block".  Not -1: an entry of -1 is legal (a sub-batch that begins with one carried byte of
// the next record's size field).  The byte pattern 0x80.. lets cudaMemset initialise an entry table.
constexpr int64_t ENTRY_NONE = (int64_t)0x8080808080808080ull;
constexpr int ENTRY_NONE_BYTE = 0x80;

// ------------------------------------------------------------------------------------- K1
struct BlockDesc {
    uint64_t coff;      // byte offset of the raw deflate data inside the compressed buffer
    uint64_t uoff;      // byte offset of the output inside the inflated buffer
    uint32_t csize;
    uint32_t isize;
    uint64_t tok_off;   // first word of the block's token area (two-phase K1; capacity tok_cap_of(isize) words)
};
// Token area per block: a match is at least 3 bytes, so isize / 3 tokens is the worst case; BAM data needs about isize / 9.
// A block that needs more than isize / 4 takes the one-phase fallback instead of everybody paying for the worst case.
BD_HD uint32_t tok_cap_of(uint32_t isize) { return isize / 4u + 16u; }
struct BlockAux { uint32_t n_tok, n_seg, n_lit, pad; };      // what phase 1 found in the block
// Literal area of block i of a batch (16-byte aligned, >= isize bytes, disjoint from its neighbours'): derived from the output offset.
BD_HD uint64_t lit_off_of(uint64_t uoff, uint64_t block_index) { return (uoff & ~15ull) + 16ull * block_index; }

// One CTA of 13 warps per SM: 13 x 17,664 B = 229,632 B of dynamic shared memory (the per-CTA 1 KB system
// reservation is paid once, which is what lets a 13th warp fit).  148 x 13 x 32 = 61,568 BGZF blocks in flight:
// a 30x chromosome (57.6 k blocks) is a single wave with no tail (12 one-warp CTAs per SM left 5 warps for a
// second wave that cost 35 % of the kernel time, profiles/k1_history.md).
constexpr int K1_WARPS = 13;
constexpr int K1_SMEM = K1_WARPS * SMEM_BYTES_PER_WARP;         // 229,632 B
__global__ void __launch_bounds__(K1_WARPS * 32, 1) k1_inflate(const uint32_t* __restrict__ comp, const BlockDesc* __restrict__ blocks,
                                                               uint32_t n_blocks, uint8_t* __restrict__ u, int* __restrict__ status) {
    BD_DYN_SMEM(uint32_t, smem);
    uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t b = (blockIdx.x * K1_WARPS + warp) * 32u + lane;
    uint32_t scratch[96];
    const bool active = b < n_blocks;
    BlockDesc d = active ? blocks[b] : BlockDesc{0, 0, 0, 0, 0};
    uint32_t* wbase = smem + warp * (SMEM_BYTES_PER_WARP / 4);
    SmemTab tab{wbase + lane, (uint32_t)__cvta_generic_to_shared(wbase + T_WORDS * 32) + lane * 16, (uint32_t)__cvta_generic_to_shared(wbase + T_FAR * 32 + lane)};
    ByteOut out{u};
    int rc = inflate_block(tab, comp, d.coff, d.csize, out, d.uoff, d.isize, scratch, active);
    if (active) status[b] = rc;
}


// ------------------------------------------------------------------------------------- K1, two phases (inflate2_core.cuh)
// Phase 1: one lane per BGZF block, Huffman decoding only.  256 (+64) B of shared memory per lane and no output window:
// 4-warp CTAs, several per SM; the block scheduler spreads a chromosome's 450 CTAs evenly.
constexpr int K1H_WARPS = 4;
template <bool LIMS> constexpr int k1h_smem() { return K1H_WARPS * (H_SMEM_BYTES_PER_WARP + (LIMS ? H_LIM_BYTES_PER_WARP : 0)); }      // 32 KB / 40 KB
// LIMS / MINB: where the Huffman limits live and how many CTAs per SM the register allocation aims at -- the variants
// measured against each other in profiles/k1_history.md.  blk0: index of blocks[0] in the batch (literal areas are per batch).
template <bool LIMS, int MINB>
__global__ void __launch_bounds__(K1H_WARPS * 32, MINB) k1_huff(const uint32_t* __restrict__ comp, const BlockDesc* __restrict__ blocks, uint32_t n_blocks, uint32_t blk0,
                                                                int* __restrict__ status, uint32_t* __restrict__ tok, uint8_t* __restrict__ lits, BlockAux* __restrict__ aux,
                                                                uint32_t* __restrict__ seg_info, uint8_t* __restrict__ lit_tab) {
    BD_DYN_SMEM(uint32_t, smem);
    uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t b = (blockIdx.x * K1H_WARPS + warp) * 32u + lane;
    uint32_t scratch[96];
    const bool active = b < n_blocks;
    BlockDesc d = active ? blocks[b] : BlockDesc{0, 0, 0, 0, 0};
    constexpr int PER_WARP = (H_SMEM_BYTES_PER_WARP + (LIMS ? H_LIM_BYTES_PER_WARP : 0)) / 4;
    uint32_t* wbase = smem + warp * PER_WARP;
    uint32_t* limb = wbase + H_WORDS * 32 + (32 * RING_BYTES_PER_LANE) / 4;
    SmemTab2 tab{wbase + lane, limb + lane * 4, (uint32_t)__cvta_generic_to_shared(wbase + H_WORDS * 32) + lane * 16};
    HuffOut ho{tok + d.tok_off, tok_cap_of(d.isize), lits + lit_off_of(d.uoff, (uint64_t)blk0 + b), lit_tab + (size_t)b * (MAX_SEG * 256), seg_info + (size_t)b * MAX_SEG};
    uint32_t n_tok = 0, n_seg = 0, n_lit = 0;
    int rc = huff_phase<SmemTab2, LIMS>(tab, comp, d.coff, d.csize, d.isize, scratch, ho, n_tok, n_seg, n_lit, active);
    if (active) { status[b] = rc; aux[b] = BlockAux{n_tok, n_seg, n_lit, 0u}; }
}

// Phase 2: one warp per BGZF block, 32 tokens at a time.  A warp scan of (literals + length) and of (literals) gives every
// token its place in the output and in the packed literal stream.  (1) the group's literals: lanes stride over the packed
// ranks (coalesced), find their token by a binary search over the 32 prefix sums in shared memory, translate through the
// deflate block's rank -> byte table (shared memory) and store.  (2) the matches: lane = token; a source byte that lies
// inside the group's own output range is resolved through the group's tokens (pointer jumping: a byte of match j is the
// byte `distance_j` before it, repeated until the position is a literal or lies before the group), so all copies of a
// group read only finished bytes and need no order among themselves; groups are separated by __syncwarp.  Distances
// and sizes are validated here; a violation ends the block with the error zlib would report.
// little-endian 32-bit load at any byte address (shared or global)
__device__ __forceinline__ uint32_t ld_u32_any(const uint8_t* p) {
    uintptr_t a = reinterpret_cast<uintptr_t>(p); const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    return __funnelshift_r(w[0], w[1], (uint32_t)(a & 3) * 8);
}
constexpr int K1L_WARPS = 8;
#ifndef BDEPTH_EMULATE_SHIM
__device__ __forceinline__ uint32_t warp_max_u32(uint32_t v) { return __reduce_max_sync(0xFFFFFFFFu, v); }
#else
static inline uint32_t warp_max_u32(uint32_t v) { return ~__reduce_min_sync(0xFFFFFFFFu, ~v); }
static inline bool emu_k1lz_warp() { static const bool on = getenv("BDEPTH_EMU_K1LZ_WARP") && atoi(getenv("BDEPTH_EMU_K1LZ_WARP")) == 1; return on; }
#endif
template <bool COMPACT>      // COMPACT = false: round 2's first literal stage (table of all 32 tokens, BDEPTH_K1LZ=v12), kept for the A/B bench.py prints
__global__ void __launch_bounds__(K1L_WARPS * 32, 6) k1_lz(const BlockDesc* __restrict__ blocks, uint32_t n_blocks, uint32_t blk0, uint8_t* __restrict__ u, int* __restrict__ status,
                                                        const uint32_t* __restrict__ tok, const uint8_t* __restrict__ lits, const BlockAux* __restrict__ aux,
                                                        const uint32_t* __restrict__ seg_info, const uint8_t* __restrict__ lit_tab) {
    __shared__ uint32_t s_tab[K1L_WARPS][64];
    __shared__ uint32_t s_il[K1L_WARPS][33], s_dl[K1L_WARPS][33];      // (one slot of slack: the stepping loop looks one token ahead)
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t b = blockIdx.x * K1L_WARPS + warp;
    if (b >= n_blocks || status[b] != INF_OK) return;            // warp-uniform
    const BlockDesc d = blocks[b]; const BlockAux ax = aux[b];
    uint8_t* const ub = u + d.uoff;
    const uint8_t* const lt = lits + lit_off_of(d.uoff, (uint64_t)blk0 + b);
    const uint32_t* const sgi = seg_info + (size_t)b * MAX_SEG;
    const uint8_t* const ltab = lit_tab + (size_t)b * (MAX_SEG * 256);
#ifdef BDEPTH_EMULATE_SHIM
    // TEST BUILD ONLY: a warp collective costs 32 fiber switches under the CPU emulation, which makes this kernel ~30x slower than
    // the rest of the emulated pipeline.  The big emulated suites therefore run the serial restatement of phase 2 (one fiber per
    // block); tests/test_emul_inflate.py runs the warp code below on every fixture with BDEPTH_EMU_K1LZ_WARP=1.
    if (!emu_k1lz_warp()) {
        if (lane == 0) { int rcs = lz_phase_serial(ub, d.isize, tok + d.tok_off, ax.n_tok, lt, ax.n_lit, ltab, sgi, ax.n_seg); if (rcs) status[b] = rcs; }
        return;
    }
#endif
    const uint8_t* const tb = reinterpret_cast<const uint8_t*>(s_tab[warp]);
    // current deflate block (segment) of the literal stream: literals [seg_lo, seg_hi)
    uint32_t sg = 0, seg_hi = ax.n_seg > 1 ? (sgi[1] & 0x7FFFFFFFu) : 0xFFFFFFFFu; bool seg_raw = ax.n_seg == 0 || (sgi[0] & SEG_RAW);
    if (!seg_raw) { const uint32_t* tg = reinterpret_cast<const uint32_t*>(ltab); s_tab[warp][lane] = tg[lane]; s_tab[warp][lane + 32] = tg[lane + 32]; }
    __syncwarp();
    const uint32_t* tk = tok + d.tok_off;
    uint32_t base = 0, lbase = 0;           // output position / literal index at which the group begins
    int err = INF_OK;
    for (uint32_t g = 0; g < ax.n_tok; g += 32) {
        const uint32_t t = g + lane < ax.n_tok ? tk[g + lane] : TOK_NOMATCH;
        const uint32_t lit = t & 0xFFu, len = (t >> 31) ? 0u : ((t >> 8) & 0xFFu) + 3u, dist = ((t >> 16) & 0x7FFFu) + 1u;
        uint32_t incl = lit + len, il = lit;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o), w = __shfl_up_sync(0xFFFFFFFFu, il, o); if ((int)lane >= o) { incl += v; il += w; } }
        const uint32_t tot = __shfl_sync(0xFFFFFFFFu, incl, 31), totl = __shfl_sync(0xFFFFFFFFu, il, 31);
        const uint32_t dlit = base + incl - len - lit, dst = dlit + lit;
        {   // what zlib checks while it copies: "invalid distance too far back", output larger than ISIZE
            const bool far = len && dist > dst;
            if (__ballot_sync(0xFFFFFFFFu, far)) { err = INF_ERR_DIST; break; }
            if (base + tot > d.isize || lbase + totl > ax.n_lit) { err = INF_ERR_OVERRUN; break; }
        }
        // ---- (1) literals of the group.  Lanes stride over the packed ranks four at a time (one unaligned word per lane and round:
        // a group's ~130 literals are one round); the token a literal belongs to is found by a binary search over the 32
        // inclusive counts in shared memory for the first of the four and by stepping for the others; rank -> byte through the
        // deflate block's table in shared memory; byte stores (runs are a few bytes at arbitrary alignment).
        if (totl) {
            while (sg + 1 < ax.n_seg && lbase >= seg_hi) {        // the group begins in a later deflate block: its table
                sg++; seg_hi = sg + 1 < ax.n_seg ? (sgi[sg + 1] & 0x7FFFFFFFu) : 0xFFFFFFFFu; seg_raw = (sgi[sg] & SEG_RAW) != 0;
                __syncwarp();
                if (!seg_raw) { const uint32_t* tg = reinterpret_cast<const uint32_t*>(ltab + sg * 256u); s_tab[warp][lane] = tg[lane]; s_tab[warp][lane + 32] = tg[lane + 32]; }
                __syncwarp();
            }
            const bool one_seg = lbase + totl <= seg_hi;
            // lanes stride over the packed ranks four at a time (one unaligned word per lane and round: a group's ~130 literals are one
            // round); the token a literal belongs to is found by a binary search over the 32 inclusive counts in shared memory for the
            // first of the four and by stepping for the others; rank -> byte through the deflate block's table in shared memory
            // (measured against a lane-per-token copy of the runs: 11.6 vs 12.9 ms, profiles/k1_history.md)
            // Only the tokens that have literals enter the table (compacted by a ballot): every entry then covers at least one literal, so
            // from one literal to the next the token changes by at most one entry -- one predicated step per byte instead of a loop over
            // the match-only tokens in between (that loop was 13 % of the kernel's instructions at 7 of 32 lanes).
            int n_ent = 32;
            if (COMPACT) {
                const unsigned has_l = __ballot_sync(0xFFFFFFFFu, lit != 0);
                if (lit) { const uint32_t e = __popc(has_l & ((1u << lane) - 1u)); s_il[warp][e] = il; s_dl[warp][e] = dlit; }
                n_ent = __popc(has_l);
            } else { s_il[warp][lane] = il; s_dl[warp][lane] = dlit; }
            __syncwarp();
            for (uint32_t j0 = 4 * lane; j0 < totl; j0 += 128) {
                const uint32_t w = ld_u32_any(lt + lbase + j0);
                int lo = 0, hi = n_ent - 1;                       // the first entry whose inclusive literal count exceeds j0 (the last one's is totl > j0)
                while (lo < hi) { int mid = (lo + hi) >> 1; if (s_il[warp][mid] > j0) hi = mid; else lo = mid + 1; }
                uint32_t tend = s_il[warp][lo], tbeg = lo ? s_il[warp][lo - 1] : 0u, tdst = s_dl[warp][lo];
#pragma unroll
                for (uint32_t bq = 0; bq < 4; bq++) {
                    const uint32_t j = j0 + bq;
                    if (j >= totl) break;
                    if (COMPACT) { if (j >= tend) { lo++; tbeg = tend; tend = s_il[warp][lo]; tdst = s_dl[warp][lo]; } }      // j == tend here, and the next entry has at least one literal
                    else while (j >= tend) { lo++; tbeg = tend; tend = s_il[warp][lo]; tdst = s_dl[warp][lo]; }            // (tokens without literals are stepped over)
                    const uint32_t r = (w >> (8 * bq)) & 0xFFu;
                    uint32_t v;
                    if (one_seg) v = seg_raw ? r : (uint32_t)tb[r];
                    else {                                        // the group straddles deflate blocks (at most MAX_SEG - 1 groups per block): table from global memory
                        uint32_t s2 = sg; while (s2 + 1 < ax.n_seg && lbase + j >= (sgi[s2 + 1] & 0x7FFFFFFFu)) s2++;
                        v = (sgi[s2] & SEG_RAW) ? r : (uint32_t)ltab[s2 * 256u + r];
                    }
                    ub[tdst + (j - tbeg)] = (uint8_t)v;
                }
            }
            __syncwarp();
        }
        // ---- (2) matches of the group, in rounds.  Everything before the first match that has not been copied yet is final
        // (all earlier matches, all literals of the group), so a match whose source bytes -- those it does not produce itself --
        // end at or before that position can go now; the first pending match always can.  A lane copies its match front to back,
        // four bytes at a time when the distance is at least four (then the four source bytes lie before the four it writes), byte
        // by byte otherwise, so a match that overlaps its own source (distance < length) needs no special case.  Dependent
        // matches (a record header copied from the previous record, which was itself copied) take another round.
        {
            const uint32_t need = len ? ((dst - dist + len < dst) ? dst - dist + len : dst) : 0u;       // end of the source bytes other lanes (or earlier groups) produce
            uint8_t* dp = ub + dst; const uint8_t* sp = dp - dist;
            unsigned pending = __ballot_sync(0xFFFFFFFFu, len != 0);
            while (pending) {
                const uint32_t ready = __shfl_sync(0xFFFFFFFFu, dst, __ffs(pending) - 1);
                const bool go = ((pending >> lane) & 1u) && need <= ready;
                const uint32_t ml = warp_max_u32(go ? len : 0u);
                for (uint32_t k = 0; k < ml; k += 4) {
                    if (!go || k >= len) continue;
                    const uint32_t n = len - k < 4u ? len - k : 4u;
                    if (dist >= 4) {
                        const uint32_t w = ld_u32_any(sp + k);
                        dp[k] = (uint8_t)w;
                        if (n > 1) dp[k + 1] = (uint8_t)(w >> 8);
                        if (n > 2) dp[k + 2] = (uint8_t)(w >> 16);
                        if (n > 3) dp[k + 3] = (uint8_t)(w >> 24);
                    } else for (uint32_t q = 0; q < n; q++) dp[k + q] = sp[k + q];
                }
                pending &= ~__ballot_sync(0xFFFFFFFFu, go);
                __syncwarp();
            }
        }
        base += tot; lbase += totl;
    }
    if (!err && (base != d.isize || lbase != ax.n_lit)) err = INF_ERR_SHORT;
    if (err && lane == 0) status[b] = err;
}

// Phase 2, flattened: the same job as k1_lz with one output BYTE per lane and round instead of one token per lane.  After the two warp
// scans every lane knows its token's range; a round covers 32 consecutive output positions: the tokens that begin inside the round
// set a bit each (one warp OR), so a lane finds its token with a POPC instead of a search; a literal byte comes from the packed
// stream through the rank -> byte table, a match byte from `distance` before it -- and if that position lies inside the group's own
// range, it is resolved through the group's tokens (binary search over the 32 ends in shared memory, repeated until the position is
// a literal or lies before the group: pointer jumping), so all bytes of a group are independent: no rounds of dependent copies,
// 32 consecutive byte stores per round (one or two sectors).
__global__ void __launch_bounds__(K1L_WARPS * 32) k1_lz_flat(const BlockDesc* __restrict__ blocks, uint32_t n_blocks, uint32_t blk0, uint8_t* __restrict__ u, int* __restrict__ status,
                                                             const uint32_t* __restrict__ tok, const uint8_t* __restrict__ lits, const BlockAux* __restrict__ aux,
                                                             const uint32_t* __restrict__ seg_info, const uint8_t* __restrict__ lit_tab) {
    __shared__ uint32_t s_tab[K1L_WARPS][64];
    __shared__ uint32_t s_end[K1L_WARPS][32], s_il[K1L_WARPS][32], s_dist[K1L_WARPS][32];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint32_t b = blockIdx.x * K1L_WARPS + warp;
    if (b >= n_blocks || status[b] != INF_OK) return;            // warp-uniform
    const BlockDesc d = blocks[b]; const BlockAux ax = aux[b];
    uint8_t* const ub = u + d.uoff;
    const uint8_t* const lt = lits + lit_off_of(d.uoff, (uint64_t)blk0 + b);
    const uint32_t* const sgi = seg_info + (size_t)b * MAX_SEG;
    const uint8_t* const ltab = lit_tab + (size_t)b * (MAX_SEG * 256);
    const uint8_t* const tb = reinterpret_cast<const uint8_t*>(s_tab[warp]);
    uint32_t sg = 0, seg_hi = ax.n_seg > 1 ? (sgi[1] & 0x7FFFFFFFu) : 0xFFFFFFFFu; bool seg_raw = ax.n_seg == 0 || (sgi[0] & SEG_RAW);
    if (!seg_raw) { const uint32_t* tg = reinterpret_cast<const uint32_t*>(ltab); s_tab[warp][lane] = tg[lane]; s_tab[warp][lane + 32] = tg[lane + 32]; }
    __syncwarp();
    const uint32_t* tk = tok + d.tok_off;
    uint32_t base = 0, lbase = 0;
    int err = INF_OK;
    for (uint32_t g = 0; g < ax.n_tok; g += 32) {
        const uint32_t t = g + lane < ax.n_tok ? tk[g + lane] : TOK_NOMATCH;
        const uint32_t lit = t & 0xFFu, len = (t >> 31) ? 0u : ((t >> 8) & 0xFFu) + 3u, dist = ((t >> 16) & 0x7FFFu) + 1u;
        uint32_t incl = lit + len, il = lit;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { uint32_t v = __shfl_up_sync(0xFFFFFFFFu, incl, o), w = __shfl_up_sync(0xFFFFFFFFu, il, o); if ((int)lane >= o) { incl += v; il += w; } }
        const uint32_t tot = __shfl_sync(0xFFFFFFFFu, incl, 31), totl = __shfl_sync(0xFFFFFFFFu, il, 31);
        const uint32_t tstart = incl - len - lit;                 // where the token's literals begin, relative to the group
        {
            const bool far = len && dist > base + tstart + lit;
            if (__ballot_sync(0xFFFFFFFFu, far)) { err = INF_ERR_DIST; break; }
            if (base + tot > d.isize || lbase + totl > ax.n_lit) { err = INF_ERR_OVERRUN; break; }
        }
        if (totl) {
            while (sg + 1 < ax.n_seg && lbase >= seg_hi) {        // the group begins in a later deflate block: its table
                sg++; seg_hi = sg + 1 < ax.n_seg ? (sgi[sg + 1] & 0x7FFFFFFFu) : 0xFFFFFFFFu; seg_raw = (sgi[sg] & SEG_RAW) != 0;
                __syncwarp();
                if (!seg_raw) { const uint32_t* tg = reinterpret_cast<const uint32_t*>(ltab + sg * 256u); s_tab[warp][lane] = tg[lane]; s_tab[warp][lane + 32] = tg[lane + 32]; }
                __syncwarp();
            }
        }
        const bool one_seg = lbase + totl <= seg_hi;
        auto literal = [&](uint32_t li) -> uint32_t {           // the byte of literal li of the block
            const uint32_t r = lt[li];
            if (one_seg) return seg_raw ? r : (uint32_t)tb[r];
            uint32_t s2 = sg; while (s2 + 1 < ax.n_seg && li >= (sgi[s2 + 1] & 0x7FFFFFFFu)) s2++;      // the group straddles deflate blocks: table from global memory
            return (sgi[s2] & SEG_RAW) ? r : (uint32_t)ltab[s2 * 256u + r];
        };
        s_end[warp][lane] = incl; s_il[warp][lane] = il; s_dist[warp][lane] = dist;
        __syncwarp();
        const bool real = lit + len != 0;
        for (uint32_t o0 = 0; o0 < tot; o0 += 32) {
            // the tokens that begin inside this round, one bit each; the token the round begins in
            const uint32_t mbits = __reduce_or_sync(0xFFFFFFFFu, (real && tstart >= o0 && tstart < o0 + 32) ? (1u << (tstart - o0)) : 0u);
            const uint32_t first = (uint32_t)__popc(__ballot_sync(0xFFFFFFFFu, real && tstart <= o0)) - 1u;
            const uint32_t o = o0 + lane;
            if (o < tot) {
                uint32_t i = first + (uint32_t)__popc(mbits & ((2u << lane) - 1u) & ~1u);
                uint32_t ts = i ? s_end[warp][i - 1] : 0u, lb = i ? s_il[warp][i - 1] : 0u, li = s_il[warp][i] - lb, off = o - ts;
                uint32_t v;
                if (off < li) v = literal(lbase + lb + off);
                else {
                    uint32_t k = off - li, dd = s_dist[warp][i], ms = base + ts + li;
                    uint32_t s = ms - dd + (dd <= k ? k % dd : k);             // inside its own match: period `dd`
                    bool done = false; v = 0;
                    while (s >= base) {                                        // the source lies in the group: through its tokens
                        const uint32_t so = s - base;
                        int lo = 0, hi = (int)i;                                // the first token whose end exceeds so (it is <= i)
                        while (lo < hi) { int mid = (lo + hi) >> 1; if (s_end[warp][mid] > so) hi = mid; else lo = mid + 1; }
                        ts = lo ? s_end[warp][lo - 1] : 0u; lb = lo ? s_il[warp][lo - 1] : 0u; li = s_il[warp][lo] - lb; off = so - ts;
                        if (off < li) { v = literal(lbase + lb + off); done = true; break; }
                        k = off - li; dd = s_dist[warp][lo]; ms = base + ts + li;
                        s = ms - dd + (dd <= k ? k % dd : k);
                    }
                    if (!done) v = ub[s];
                }
                ub[base + o] = (uint8_t)v;
            }
        }
        base += tot; lbase += totl;
        __syncwarp();
    }
    if (!err && (base != d.isize || lbase != ax.n_lit)) err = INF_ERR_SHORT;
    if (err && lane == 0) status[b] = err;
}

// The exact one-phase decoder for the blocks phase 1 marked INF_FALLBACK (more than MAX_SEG deflate blocks, more tokens
// than the token area holds).  Launched after every two-phase inflate; a warp without such a block returns at once.
__global__ void __launch_bounds__(K1_WARPS * 32, 1) k1_fallback(const uint32_t* __restrict__ comp, const BlockDesc* __restrict__ blocks,
                                                                uint32_t n_blocks, uint8_t* __restrict__ u, int* __restrict__ status) {
    BD_DYN_SMEM(uint32_t, smem);
    uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t b = (blockIdx.x * K1_WARPS + warp) * 32u + lane;
    uint32_t scratch[96];
    const bool active = b < n_blocks && status[b] == INF_FALLBACK;
#ifndef BDEPTH_EMULATE_SHIM
    if (!__any_sync(0xFFFFFFFFu, active)) return;
#endif
    BlockDesc d = active ? blocks[b] : BlockDesc{0, 0, 0, 0, 0};
    uint32_t* wbase = smem + warp * (SMEM_BYTES_PER_WARP / 4);
    SmemTab tab{wbase + lane, (uint32_t)__cvta_generic_to_shared(wbase + T_WORDS * 32) + lane * 16, (uint32_t)__cvta_generic_to_shared(wbase + T_FAR * 32 + lane)};
    ByteOut out{u};
    int rc = inflate_block(tab, comp, d.coff, d.csize, out, d.uoff, d.isize, scratch, active);
    if (active) status[b] = rc;
}

// ------------------------------------------------------------------------------------- K2
// Unaligned little-endian loads from the inflated stream: two aligned 32-bit loads + funnel shift (records are
// byte-aligned; four byte loads per field made k2_decode LSU-queue bound: profiles/r1_k2_k3_ncu_full_summary.txt).
// The buffer has >= 256 readable bytes after its end, so touching the following word is always legal.
__device__ __forceinline__ uint32_t ldu32(const uint8_t* p) {
    uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(a & ~uintptr_t(3));
    uint32_t lo = __ldg(w), hi = __ldg(w + 1);
    return __funnelshift_r(lo, hi, (uint32_t)(a & 3) * 8);
}
__device__ __forceinline__ uint32_t ldu16(const uint8_t* p) { return ldu32(p) & 0xFFFFu; }

struct ScanParams {
    const uint8_t* u;          // inflated stream; offsets below are relative to it (may be negative for the carry)
    int64_t u_begin;           // first valid byte (<= 0 when a carry precedes the batch)
    int64_t u_end;             // one past the last valid byte
    int n_ref;
    const uint32_t* ref_len;
    const uint64_t* ref_lin0;  // linear coordinate of position 0 of each reference
};

// A record header at offset o is plausible if its fixed fields are mutually consistent.
__device__ __forceinline__ bool plausible_record(const ScanParams& sp, int64_t o, int64_t* next) {
    if (o + 36 > sp.u_end) return false;
    const uint8_t* p = sp.u + o;
    uint32_t bs = ldu32(p);
    if (bs < 32u || bs > (1u << 28)) return false;
    int32_t ref = (int32_t)ldu32(p + 4), pos = (int32_t)ldu32(p + 8);
    if (ref < -1 || ref >= sp.n_ref || pos < -1) return false;
    if (ref >= 0 && (uint32_t)pos > sp.ref_len[ref]) return false;
    uint32_t l_name = p[12];
    uint32_t n_cigar = ldu16(p + 16);
    int32_t l_seq = (int32_t)ldu32(p + 20);
    int32_t nref = (int32_t)ldu32(p + 24), npos = (int32_t)ldu32(p + 28);
    if (l_name < 1 || l_seq < 0 || nref < -1 || nref >= sp.n_ref || npos < -1) return false;
    uint64_t need = 32ull + l_name + 4ull * n_cigar + ((uint64_t)l_seq + 1) / 2 + (uint64_t)l_seq;
    if (need > bs) return false;
    int64_t nul = o + 36 + l_name - 1;
    if (nul < sp.u_end && sp.u[nul] != 0) return false;
    *next = o + 4 + (int64_t)bs;
    return true;
}

// One warp per BGZF block: the smallest offset in the block at which a chain of 3 plausible
// records starts.  Result is only a GUESS; k2_walk + host verification make it exact.
__global__ void k2_guess_entries(ScanParams sp, const int64_t* __restrict__ chunk_start, uint32_t n_chunks, int64_t* __restrict__ entry) {
    uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n_chunks) return;
    if (warp == 0) return;                 // chunk 0 is anchored by the caller
    int64_t c0 = chunk_start[warp], c1 = chunk_start[warp + 1];
    int64_t found = ENTRY_NONE;
    for (int64_t base = c0; base < c1; base += 32) {
        int64_t o = base + lane, nx = 0;
        bool ok = o < c1 && plausible_record(sp, o, &nx);
        if (ok) {
            // follow two more records (each must be plausible unless it runs off the stream end)
            int64_t o2 = nx, n2 = 0;
            if (o2 + 36 <= sp.u_end) { ok = plausible_record(sp, o2, &n2); if (ok && n2 + 36 <= sp.u_end) { int64_t n3; ok = plausible_record(sp, n2, &n3); } }
        }
        unsigned m = __ballot_sync(0xFFFFFFFFu, ok);
        if (m) { found = base + (__ffs(m) - 1); break; }
    }
    if (lane == 0) entry[warp] = found;
}

// One thread per block: walk the record chain from entry[c] while the record STARTS inside the
// block.  Writes the start offsets (relative to chunk_start) and the exit offset.
// walk_list (optional) restricts the launch to the listed chunks (fix-up passes).
__global__ void k2_walk(ScanParams sp, const int64_t* __restrict__ chunk_start, uint32_t n_chunks, const int64_t* __restrict__ entry,
                        const uint32_t* __restrict__ slot_base, uint16_t* __restrict__ slots, uint32_t* __restrict__ count,
                        int64_t* __restrict__ exit_off, int* __restrict__ err, const uint32_t* __restrict__ walk_list, uint32_t n_list,
                        const int64_t* __restrict__ chunk_limit /* optional: the walk of chunk c stops at this offset (end of a region-query chunk) */) {
    uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t c;
    if (walk_list) { if (t >= n_list) return; c = walk_list[t]; } else { if (t >= n_chunks) return; c = t; }
    int64_t o = entry[c], c0 = chunk_start[c], c1 = chunk_start[c + 1];
    if (chunk_limit && chunk_limit[c] < c1) c1 = chunk_limit[c];
    uint32_t n = 0;
    if (o != ENTRY_NONE) {
        uint16_t* sl = slots + slot_base[c];
        while (o < c1) {
            if (o + 4 > sp.u_end) break;                       // size field itself is cut: tail
            uint32_t bs = ldu32(sp.u + o);
            if (bs < 32u) { atomicExch(err, 1); break; }       // corrupt chain
            if (o + 4 + (int64_t)bs > sp.u_end) break;          // incomplete record: tail, carried to the next batch
            // 16-bit offsets: relative to the chunk start, except that after the first record of a chunk that begins
            // inside the carried tail (c0 < 0) the base is 0 -- a full 64 KB block plus a carry does not fit 16 bits
            sl[n] = (uint16_t)(o - ((n == 0 || c0 > 0) ? c0 : 0)); n++;
            o += 4 + (int64_t)bs;
        }
    }
    count[c] = n;
    exit_off[c] = o;
}

// Columnar SoA written by k2_decode (one row per record, file order).
struct RecordSoA {
    uint64_t* start;     // linear coordinate of the first reference base (UINT64_MAX-1 when unplaced)
    uint32_t* span;      // reference bases covered, clipped to the reference end; 0 => contributes nothing
    uint32_t* meta;      // flag << 16 | mapq << 8 | sample << 2 | bit1 long | bit0 pass
    int64_t* off;        // offset of the record's refID field relative to the batch's inflated bytes (negative inside the carry)
    uint32_t* ncl;       // n_cigar << 8 | l_read_name
    int32_t*  lseq;
};
struct ScanStats {      // device-side accumulators
    unsigned long long n_pass, n_cigar, seq_bytes, max_end, min_start, n_long, max_start, rg_err;   // rg_err: 1 + index of the first read with an unknown RG
    unsigned long long n_ghost;     // -m: records before the batch's own ones (re-read from the previous batch / the previous rank's zone), k2_decode<.., true>
    unsigned long long n_ghost_right;   // -m on several ranks: records at or after the shard limit (the next rank's zone)
    unsigned long long bad_rec;     // 1 + index of the first record whose name + CIGAR + sequence + qualities do not fit its block_size (~0: none)
    unsigned long long n_zone_pass, min_start_all;      // several ranks without -m: passing reads of the previous ranks' zone; smallest start over own and zone reads
    unsigned long long lead_n;      // 1 + index of the first read whose CIGAR begins with N and cannot be reproduced (k2_lead_n_fix; ~0: none)
    unsigned long long n_lead;      // reads whose first reference-consuming operation is N (k2_lead_n_find's list)
    unsigned long long seen_samples;        // RG lookup on: bit s set iff a passing read of pass-local sample s was seen (K3 runs for those only in a sample pass)
    unsigned long long untagged_elsewhere;  // RG lookup on: nonzero iff a passing read without an RG tag (sample 0) was left to the pass that holds sample 0
};
constexpr uint64_t START_UNPLACED = 0xFFFFFFFFFFFFFFFEull;      // RecordSoA.start of a record without a position on a known reference
constexpr uint32_t NCL_GHOST = 1u << 31;      // RecordSoA.ncl: a record that is only re-read for the mate kernels and passes the filter (its pass bit is clear)
constexpr uint32_t NCL_FOREIGN = 1u << 30;    // ... and belongs to another rank's shard (-m on several ranks: the zones left and right of the shard)
// @RG ID -> sample table of one sample pass (depth.d:1170-1181).  ids: the @RG IDs, NUL-terminated, concatenated (offs: where each
// begins); hash: open-addressing table of 1 + read-group index (0: empty slot), FNV-1a of the ID, linear probing, mask + 1 slots (a power
// of two >= 2 n_rg, so a probe always ends); sample_of: the read group's pass-local sample id, or RG_OTHER when its sample is counted
// in another pass; no_tag: the same for sample 0, which reads without an RG tag belong to.  It lives in device memory: k2_decode takes
// a pointer to it (nullptr: no lookup, every read is sample 0).
constexpr uint16_t RG_OTHER = 0xFFFFu;
struct RgTable { const uint8_t* ids; const uint32_t* offs; const uint16_t* sample_of; const uint32_t* hash; uint32_t mask; uint32_t n_rg; uint32_t no_tag; };
__host__ __device__ __forceinline__ uint32_t fnv1a_step(uint32_t h, uint8_t c) { return (h ^ c) * 16777619u; }
constexpr uint32_t FNV1A_INIT = 2166136261u;

// CustomBamRead (depth.d:240-250): scan of the aux area for RG:Z (read.d:1070-1087), the ID hashed while it is walked, then one
// string compare per probe.  Returns the read's pass-local sample id or RG_OTHER.  A read group that is not in the header is booked
// in st->rg_err (the run fails; the read counts as sample 0 meanwhile).  Out of line, and only in the k2_decode<.., .., true>
// instantiations: the kernel of single-sample runs keeps its registers.
__device__ BD_NOINLINE uint32_t sample_of_record(const RgTable* rgp, const uint8_t* aux, const uint8_t* end, ScanStats* st, uint32_t r) {
    const RgTable rg = *rgp;
    while (aux + 3 <= end) {
        uint8_t t0 = aux[0], t1 = aux[1], ty = aux[2];
        const uint8_t* v = aux + 3;
        if (t0 == 'R' && t1 == 'G' && ty == 'Z') {
            uint32_t hs = FNV1A_INIT; const uint8_t* q = v;
            while (q < end && *q) { hs = fnv1a_step(hs, *q); q++; }
            const size_t len = (size_t)(q - v);
            for (uint32_t k = hs & rg.mask;; k = (k + 1) & rg.mask) {
                const uint32_t g1 = rg.hash[k];
                if (!g1) break;
                const uint8_t* id = rg.ids + rg.offs[g1 - 1]; size_t i = 0;
                while (i < len && id[i] == v[i]) i++;
                if (i == len && id[len] == 0) {
                    const uint32_t s = rg.sample_of[g1 - 1];
                    if (s != RG_OTHER && !((st->seen_samples >> s) & 1ull)) atomicOr(&st->seen_samples, 1ull << s);
                    return s;
                }
            }
            atomicMin(&st->rg_err, (unsigned long long)r + 1);
            return rg.no_tag == RG_OTHER ? 0u : rg.no_tag;
        }
        size_t n = 0;
        switch (ty) {
        case 'A': case 'c': case 'C': n = 1; break;
        case 's': case 'S': n = 2; break;
        case 'i': case 'I': case 'f': n = 4; break;
        case 'Z': case 'H': { const uint8_t* q = v; while (q < end && *q) q++; n = (size_t)(q - v) + 1; break; }
        case 'B': { if (v + 5 > end) { aux = end; continue; } uint8_t bt = v[0]; uint32_t cnt = ldu32(v + 1); size_t es = (bt == 'c' || bt == 'C') ? 1 : (bt == 's' || bt == 'S') ? 2 : 4; n = 5 + es * cnt; break; }
        default: aux = end; continue;      // (an unknown type ends the scan: no RG tag)
        }
        aux = v + n;
    }
    // no RG tag: sample 0
    if (rg.no_tag == RG_OTHER) { if (!st->untagged_elsewhere) atomicExch(&st->untagged_elsewhere, 1ull); }
    else if (!((st->seen_samples >> rg.no_tag) & 1ull)) atomicOr(&st->seen_samples, 1ull << rg.no_tag);
    return rg.no_tag;
}

__device__ __forceinline__ bool cig_rcons(uint32_t op) { return op == 0 || op == 2 || op == 3 || op == 7 || op == 8; }
__device__ __forceinline__ bool cig_qcons(uint32_t op) { return op == 0 || op == 1 || op == 4 || op == 7 || op == 8; }
__device__ __forceinline__ bool cig_match(uint32_t op) { return op == 0 || op == 7 || op == 8; }

// out of line: the default predicate's path through k2_decode keeps its registers
__device__ BD_NOINLINE bool filter_eval_cold(const FilterProg* fp, const uint8_t* rec, uint32_t rec_size) { return filter_eval(*fp, rec, rec_size); }

// FILTER: a compiled -F query decides (its own instantiation, so that the default predicate's kernel keeps its register count).
// RG: per-sample counters -- the read's @RG sample is looked up (sample_of_record; rg: the table of the run or sample pass).
// GHOST (-m across batches and ranks, mates.cuh): records that start below ghost_below were counted by the previous batch,
// records outside [own_lo, own_hi) belong to a neighbouring rank's shard; both are read only so that the mate kernels see
// them: their pass bit stays clear (K3, the per-read reducers and the statistics ignore them), NCL_GHOST marks the ones
// that pass the filter, NCL_FOREIGN the ones of another rank.
template <bool FILTER, bool GHOST, bool RG>
__global__ void k2_decode(ScanParams sp, const int64_t* __restrict__ chunk_start, uint32_t n_chunks, const uint32_t* __restrict__ slot_base,
                          const uint16_t* __restrict__ slots, const uint32_t* __restrict__ count, const uint32_t* __restrict__ rec_base,
                          RecordSoA soa, int mapq_gt, uint32_t flag_reject, ScanStats* __restrict__ st, uint32_t* __restrict__ long_list,
                          uint32_t* __restrict__ ref_has_reads, const RgTable* __restrict__ rg, const FilterProg* __restrict__ fprog /* compiled -F query, or nullptr: mapq_gt / flag_reject */,
                          int64_t ghost_below, int64_t own_lo, int64_t own_hi, int64_t zone_below /* several ranks without -m: records below this offset
                          belong to the previous ranks' shards and are read only because they reach into this rank's positions: counted by K3, kept out of the statistics */) {
    uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n_chunks) return;
    uint32_t n = count[warp];
    int64_t c0 = chunk_start[warp];
    const uint16_t* sl = slots + slot_base[warp];
    uint32_t rb = rec_base[warp];
    unsigned long long loc_pass = 0, loc_cig = 0, loc_seq = 0, loc_maxend = 0, loc_minstart = ~0ull, loc_maxstart = 0;
    uint32_t has_word = 0xFFFFFFFFu, has_bits = 0;      // per-lane pending "reference has reads" bits (one atomic per warp, not per read)
    unsigned long long loc_ghost = 0, loc_ghost_r = 0, loc_zone = 0, loc_minall = ~0ull;
    for (uint32_t k = lane; k < n; k += 32) {
        int64_t o = ((k == 0 || c0 > 0) ? c0 : 0) + sl[k];
        const uint8_t* p = sp.u + o + 4;
        // refID, pos, bin_mq_nl, flag_nc, l_seq: 20 consecutive bytes = 6 aligned words + 5 funnel shifts
        uintptr_t pa = reinterpret_cast<uintptr_t>(p);
        const uint32_t* pw = reinterpret_cast<const uint32_t*>(pa & ~uintptr_t(3)); uint32_t psh = (uint32_t)(pa & 3) * 8;
        uint32_t h0 = __ldg(pw), h1 = __ldg(pw + 1), h2 = __ldg(pw + 2), h3 = __ldg(pw + 3), h4 = __ldg(pw + 4), h5 = __ldg(pw + 5);
        int32_t ref = (int32_t)__funnelshift_r(h0, h1, psh), pos = (int32_t)__funnelshift_r(h1, h2, psh);
        uint32_t bmn = __funnelshift_r(h2, h3, psh), fnc = __funnelshift_r(h3, h4, psh);
        int32_t l_seq = (int32_t)__funnelshift_r(h4, h5, psh);
        uint32_t l_name = bmn & 0xFF, mapq = (bmn >> 8) & 0xFF, flag = fnc >> 16, n_cigar = fnc & 0xFFFF;
        const uint8_t* cg = p + 32 + l_name;
        uint64_t span = 0;
        {   // a record whose fields overrun its block_size (corrupt file) must not send anybody reading past it: the reference
            // slices without bounds checks there (release build), this engine refuses the file (bdepth.cu reports bad_rec)
            const uint32_t bs = __funnelshift_r(__ldg(pw - 1), h0, psh);
            const uint64_t need = 32ull + l_name + 4ull * n_cigar + (l_seq > 0 ? ((uint64_t)(uint32_t)l_seq + 1) / 2 + (uint32_t)l_seq : 0ull);
            if (l_seq < 0 || need > bs) { atomicMin(&st->bad_rec, (unsigned long long)(rb + k) + 1); n_cigar = 0; l_seq = 0; ref = -1; }
        }
        for (uint32_t i = 0; i < n_cigar; i++) { uint32_t c = ldu32(cg + 4 * i); if (cig_rcons(c & 15)) span += c >> 4; }
        bool placed = ref >= 0 && ref < sp.n_ref && pos >= 0;
        bool pass = placed && !(flag & 4u) && span > 0;
        if (pass) { if (FILTER) pass = filter_eval_cold(fprog, p, ldu32(sp.u + o)); else pass = ((int)mapq > mapq_gt) && !(flag & flag_reject); }
        uint64_t start = placed ? sp.ref_lin0[ref] + (uint64_t)pos : START_UNPLACED;
        uint32_t span_eff = 0;
        if (pass) {
            uint64_t room = (uint32_t)pos < sp.ref_len[ref] ? (uint64_t)sp.ref_len[ref] - (uint32_t)pos : 0;
            span_eff = (uint32_t)(span < room ? span : room);
            if (span_eff == 0) pass = false;
        }
        bool is_long = pass && span_eff > SPAN_SHORT;
        uint32_t r = rb + k;
        uint32_t sample = 0;
        if (RG && pass) {
            uint32_t bs = ldu32(sp.u + o);
            const uint32_t sid = sample_of_record(rg, cg + 4u * n_cigar + ((uint32_t)l_seq + 1) / 2 + (uint32_t)l_seq, p + bs, st, r);
            if (sid == RG_OTHER) { pass = false; is_long = false; }      // counted in the pass that holds its sample
            else sample = sid & 63u;
        }
        uint32_t ghost_bit = 0;
        if (GHOST) {
            const bool foreign = o < own_lo || o >= own_hi;
            if (foreign || o < ghost_below) { if (o >= own_hi) loc_ghost_r++; else loc_ghost++; if (pass) ghost_bit = NCL_GHOST | (foreign ? NCL_FOREIGN : 0u); pass = false; is_long = false; }
        }
        const bool zone = !GHOST && o < zone_below;
        if (zone) { loc_ghost++; if (pass) ghost_bit = NCL_FOREIGN; }
        soa.start[r] = start; soa.span[r] = span_eff;
        soa.meta[r] = (flag << 16) | (mapq << 8) | (sample << 2) | (pass ? 1u : 0u) | (is_long ? 2u : 0u);
        soa.off[r] = o + 4; soa.ncl[r] = (n_cigar << 8) | l_name | ghost_bit; soa.lseq[r] = l_seq;
        if (!zone) loc_cig += n_cigar;
        if (pass && zone) {      // a zone read: its extent bounds the tiles K3 has to visit; it is not one of this rank's reads otherwise
            loc_zone++;
            if (start < loc_minall) loc_minall = start;
            if (start + span_eff > loc_maxend) loc_maxend = start + span_eff;
            if (is_long) { uint32_t idx = (uint32_t)atomicAdd(&st->n_long, 1ull); long_list[idx] = r; }
        } else if (pass) {
            loc_pass++; loc_seq += ((uint64_t)l_seq + 1) / 2;
            if (start + span_eff > loc_maxend) loc_maxend = start + span_eff;
            if (start < loc_minstart) loc_minstart = start;
            if (start > loc_maxstart) loc_maxstart = start;
            if ((uint32_t)(ref >> 5) != has_word) { if (has_bits) atomicOr(&ref_has_reads[has_word], has_bits); has_word = (uint32_t)(ref >> 5); has_bits = 0; }
            has_bits |= 1u << (ref & 31);
            if (is_long) { uint32_t idx = (uint32_t)atomicAdd(&st->n_long, 1ull); long_list[idx] = r; }
        }
    }
    if (loc_zone) { atomicAdd(&st->n_zone_pass, loc_zone); atomicMin(&st->min_start_all, loc_minall); }
    if (loc_ghost) atomicAdd(&st->n_ghost, loc_ghost);       // per lane: only a batch's first blocks hold ghosts / zone records
    if (GHOST && loc_ghost_r) atomicAdd(&st->n_ghost_right, loc_ghost_r);
    {   // flush the has-reads bits: in the common case the whole warp saw one bitmap word -> one atomic
        uint32_t w0 = __shfl_sync(0xFFFFFFFFu, has_word, 0);
        bool same = __all_sync(0xFFFFFFFFu, has_word == w0 || has_bits == 0);
        if (same) { uint32_t allb = __reduce_or_sync(0xFFFFFFFFu, has_bits); uint32_t ww = __reduce_min_sync(0xFFFFFFFFu, has_bits ? has_word : 0xFFFFFFFFu); if (lane == 0 && allb) atomicOr(&ref_has_reads[ww], allb); }
        else if (has_bits) atomicOr(&ref_has_reads[has_word], has_bits);
    }
    for (int s = 16; s; s >>= 1) {
        loc_pass += __shfl_xor_sync(0xFFFFFFFFu, loc_pass, s); loc_cig += __shfl_xor_sync(0xFFFFFFFFu, loc_cig, s); loc_seq += __shfl_xor_sync(0xFFFFFFFFu, loc_seq, s);
        unsigned long long m = __shfl_xor_sync(0xFFFFFFFFu, loc_maxend, s); if (m > loc_maxend) loc_maxend = m;
        m = __shfl_xor_sync(0xFFFFFFFFu, loc_minstart, s); if (m < loc_minstart) loc_minstart = m;
        m = __shfl_xor_sync(0xFFFFFFFFu, loc_maxstart, s); if (m > loc_maxstart) loc_maxstart = m;
    }
    if (lane == 0) {
        if (loc_pass) atomicAdd(&st->n_pass, loc_pass);
        if (loc_cig) atomicAdd(&st->n_cigar, loc_cig);
        if (loc_seq) atomicAdd(&st->seq_bytes, loc_seq);
        if (loc_maxend) atomicMax(&st->max_end, loc_maxend);
        if (loc_minstart != ~0ull) atomicMin(&st->min_start, loc_minstart);
        if (loc_maxstart) atomicMax(&st->max_start, loc_maxstart);
    }
}

// ------------------------------------------------------------------------------------- K3
// tile t covers linear positions [win_base + t*TILE_POS, +TILE_POS).
// tile_first[t] = first record index whose start >= tile start   (n_tiles + 1 entries, pre-set to R)
// tile_lo[t]    = smallest index of a passing short read overlapping tile t (pre-set to 0xFFFFFFFF)
__global__ void k3_tile_index(RecordSoA soa, uint32_t R, uint64_t win_base, uint32_t n_tiles, uint32_t* __restrict__ tile_first, uint32_t* __restrict__ tile_lo) {
    uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    uint64_t s = soa.start[r];
    // A record that is not placed (pos = -1 on a reference, or a reference id the header does not have) can sit anywhere
    // in a sorted file; its start is the sentinel, which is not monotone: it takes no part in the index, and the placed
    // record behind it looks back past it.
    if (s == START_UNPLACED) return;
    // boundaries: tiles whose start lies in (prev_start, s] get first = r
    // tile_first[t] = min{ r : start[r] >= tile_start(t) }.  Record r is that minimum for all t with
    // start[r-1] < tile_start(t) <= start[r].
    int64_t t_hi = s >= win_base ? (int64_t)((s - win_base) / TILE_POS) : -1;                        // last tile with tile_start <= s
    int64_t t_lo;
    uint32_t q = r; while (q > 0 && soa.start[q - 1] == START_UNPLACED) q--;
    if (q == 0) t_lo = 0;
    else { uint64_t ps = soa.start[q - 1]; t_lo = ps >= win_base ? (int64_t)((ps - win_base) / TILE_POS) + 1 : 0; }
    if (t_hi > (int64_t)n_tiles) t_hi = n_tiles;
    for (int64_t t = t_lo; t <= t_hi; t++) tile_first[t] = r;
    uint32_t m = soa.meta[r];
    if ((m & 3u) == 1u) {      // (a read of the previous rank's zone may begin before the first tile and still reach into it)
        uint64_t e = s + soa.span[r] - 1;
        if (e >= win_base) {
            uint64_t ta = s >= win_base ? (s - win_base) / TILE_POS : 0, tb = (e - win_base) / TILE_POS;
            for (uint64_t t = ta; t <= tb && t < n_tiles; t++) atomicMin(&tile_lo[t], r);
        }
    }
}

__device__ __forceinline__ uint32_t ldg8(const uint8_t* p) { return (uint32_t)__ldg(p); }

struct GatherAcc {
    uint32_t packed[4];          // A,C,G,T as 4 x 8-bit fields per position
    uint32_t wide[4][4];         // flushed A,C,G,T
    uint32_t nN[4], del[4], skip[4];
};

// add base with reference offset x (relative to the read start) at query index q for slot j
template <bool MINQ>
__device__ __forceinline__ void add_base(GatherAcc& a, int j, const uint8_t* seq, const uint8_t* qual, uint32_t q, uint32_t lseq, uint32_t minq) {
    if (q >= lseq) return;
    if (MINQ) { if (ldg8(qual + q) < minq) return; }
    uint32_t b = ldg8(seq + (q >> 1));
    uint32_t nib = (q & 1) ? (b & 15u) : (b >> 4);
    // nt16 -> nt5 (base.d:186): 1,2,4,8 -> A,C,G,T ; everything else N
    if (__popc(nib) == 1) a.packed[j] += 1u << ((31 - __clz(nib)) * 8);
    else a.nN[j]++;
}

// PRE (EXPERIMENT, off by default, BDEPTH_K3_PREFETCH=1): the lane that holds candidate read base+i also loads that
// read's off / ncl / lseq / first CIGAR word, 32 reads per load instruction, and the per-read step takes them by
// shuffle.  Without it every selected read costs a chain of four dependent global loads (off -> ncl/lseq -> CIGAR
// word -> sequence bytes) that all 32 lanes wait for: ~56 reads per warp x ~2 us; the kernel's 7.4 ms is about what
// that latency chain predicts at 32 resident warps per SM.  Never measured: DESIGN.md section 10.
template <bool MINQ, bool PRE>
__global__ void __launch_bounds__(256) k3_gather(RecordSoA soa, const uint8_t* __restrict__ u, uint64_t tiles_base, uint64_t cnt_base, uint64_t win_len,
                                                  const uint32_t* __restrict__ tile_first, const uint32_t* __restrict__ tile_lo,
                                                  uint32_t* __restrict__ counts, uint32_t minq, int sample_sel) {
    uint32_t tile = blockIdx.x;
    uint32_t lo = tile_lo[tile];
    if (lo == 0xFFFFFFFFu) return;                       // no passing short read touches this tile
    uint32_t hi = tile_first[tile + 1];
    uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint64_t w0 = tiles_base + (uint64_t)tile * TILE_POS + warp * 128u, w1 = w0 + 128;
    uint64_t p0 = w0 + 4u * lane;
    GatherAcc a;
#pragma unroll
    for (int j = 0; j < 4; j++) { a.packed[j] = 0; a.nN[j] = a.del[j] = a.skip[j] = 0; for (int c = 0; c < 4; c++) a.wide[j][c] = 0; }
    uint32_t since_flush = 0;
    for (uint32_t base = lo; base < hi; base += 32) {
        uint32_t r = base + lane;
        uint64_t s = 0; uint32_t sp = 0; bool ov = false;
        int64_t off_l = 0; uint32_t ncl_l = 0, lseq_l = 0, c0_l = 0;
        if (r < hi) {
            s = soa.start[r]; sp = soa.span[r];
            uint32_t mt = soa.meta[r];
            ov = (mt & 3u) == 1u && (sample_sel < 0 || (int)((mt >> 2) & 63u) == sample_sel) && s < w1 && s + sp > w0;
            if (PRE && ov) { off_l = soa.off[r]; ncl_l = soa.ncl[r]; lseq_l = (uint32_t)max(soa.lseq[r], 0); c0_l = ldu32(u + off_l + 32 + (ncl_l & 0xFF)); }
        }
        // reads are sorted by start: once the first PLACED read of a group starts at or past w1, we are done (an
        // unplaced record in the middle of the file carries the sentinel start and says nothing about the ones behind it)
        unsigned placed_m = __ballot_sync(0xFFFFFFFFu, r < hi && s != START_UNPLACED);
        if (placed_m) { uint64_t s_first = __shfl_sync(0xFFFFFFFFu, s, __ffs(placed_m) - 1); if (s_first >= w1) break; }
        unsigned m = __ballot_sync(0xFFFFFFFFu, ov);
        while (m) {
            int bsel = __ffs(m) - 1; m &= m - 1;
            uint32_t rr = base + bsel;
            uint64_t rs = __shfl_sync(0xFFFFFFFFu, s, bsel);
            uint32_t rspan = __shfl_sync(0xFFFFFFFFu, sp, bsel);
            int64_t off; uint32_t ncl, lseq;
            if (PRE) { off = __shfl_sync(0xFFFFFFFFu, off_l, bsel); ncl = __shfl_sync(0xFFFFFFFFu, ncl_l, bsel); lseq = __shfl_sync(0xFFFFFFFFu, lseq_l, bsel); }
            else { off = soa.off[rr]; ncl = soa.ncl[rr]; lseq = (uint32_t)max(soa.lseq[rr], 0); }
            uint32_t n_cigar = (ncl >> 8) & 0xFFFFu, l_name = ncl & 0xFF;      // (bits 30-31 of ncl are the ghost / foreign marks)
            const uint8_t* rec = u + off;
            const uint8_t* cg = rec + 32 + l_name;
            const uint8_t* seq = cg + 4u * n_cigar;
            const uint8_t* qual = seq + (lseq + 1) / 2;
            const int32_t rp = (int32_t)((int64_t)p0 - (int64_t)rs);      // reference offset of this lane's first position (|rp| < span + 128)
            const uint32_t c0 = PRE ? __shfl_sync(0xFFFFFFFFu, c0_l, bsel) : ldu32(cg);
            if (n_cigar == 1 && cig_match(c0 & 15)) {
                // ---- fast path (90 % of short reads): one M/=/X op.  The 4 bases of this lane sit in at most 3
                // sequence bytes: one unaligned 32-bit load, nibbles picked by shifts.
                uint32_t L = min(min(c0 >> 4, rspan), lseq);
                if (rp + 3 >= 0 && rp < (int32_t)L) {
                    uint32_t xb = rp > 0 ? (uint32_t)rp : 0u, bq = xb >> 1;
                    uint32_t w = ldu32(seq + bq), wq = 0;
                    if (MINQ) wq = ldu32(qual + xb);
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        int32_t x = rp + j;
                        if (x >= 0 && x < (int32_t)L) {
                            bool okq = true;
                            if (MINQ) okq = ((wq >> (8 * ((uint32_t)x - xb))) & 0xFFu) >= minq;
                            uint32_t n = (uint32_t)x - 2 * bq;                       // nibble index inside w (0..7), high nibble first
                            uint32_t nib = (w >> (8 * (n >> 1) + ((n & 1) ? 0 : 4))) & 15u;
                            if (okq) { if (__popc(nib) == 1) a.packed[j] += 1u << ((31 - __clz(nib)) * 8); else a.nN[j]++; }
                        }
                    }
                }
            } else {
                uint32_t rpos = 0, qpos = 0;
                for (uint32_t i = 0; i < n_cigar; i++) {
                    uint32_t c = i == 0 ? c0 : ldu32(cg + 4 * i), len = c >> 4, op = c & 15;
                    if (cig_match(op)) {
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            int32_t x = rp + j - (int32_t)rpos;
                            if (x >= 0 && x < (int32_t)len && (uint32_t)(rp + j) < rspan) add_base<MINQ>(a, j, seq, qual, qpos + (uint32_t)x, lseq, minq);
                        }
                        rpos += len; qpos += len;
                    } else if (op == 2 || op == 3) {
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            int32_t x = rp + j - (int32_t)rpos;
                            if (x >= 0 && x < (int32_t)len && (uint32_t)(rp + j) < rspan) { if (op == 2) a.del[j]++; else a.skip[j]++; }
                        }
                        rpos += len;
                    } else if (cig_qcons(op)) qpos += len;
                    if ((int32_t)rpos > rp + 3) break;          // (warp-divergent exit is fine: remaining ops cannot touch this lane)
                }
            }
            if (++since_flush == 255) {
                since_flush = 0;
#pragma unroll
                for (int j = 0; j < 4; j++) { for (int c = 0; c < 4; c++) a.wide[j][c] += (a.packed[j] >> (8 * c)) & 255u; a.packed[j] = 0; }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 4; j++) for (int c = 0; c < 4; c++) a.wide[j][c] += (a.packed[j] >> (8 * c)) & 255u;
    // read-modify-write of this thread's 4 positions in each plane (16-byte vector accesses)
    uint64_t idx = p0 - cnt_base;
    if (idx + 4 > win_len) return;
    uint32_t any = 0;
#pragma unroll
    for (int j = 0; j < 4; j++) any |= a.wide[j][0] | a.wide[j][1] | a.wide[j][2] | a.wide[j][3] | a.nN[j] | a.del[j] | a.skip[j];
    if (!any) return;
#pragma unroll
    for (int pl = 0; pl < N_PLANES; pl++) {
        uint32_t v[4];
#pragma unroll
        for (int j = 0; j < 4; j++) v[j] = pl < 4 ? a.wide[j][pl] : pl == 4 ? a.nN[j] : pl == 5 ? a.del[j] : a.skip[j];
        if (!(v[0] | v[1] | v[2] | v[3])) continue;
        uint4* dst = reinterpret_cast<uint4*>(counts + (uint64_t)pl * win_len + idx);
        uint4 cur = *dst;
        cur.x += v[0]; cur.y += v[1]; cur.z += v[2]; cur.w += v[3];
        *dst = cur;
    }
}

// ---- k3_tile: CTA per 1024-position tile, counters in shared memory, records staged by bulk async copy (TMA) ----------
// The reads that can touch a tile are the records [tile_lo, tile_first[tile + 1]) of the sorted file, and they are
// CONTIGUOUS in the inflated stream: one cp.async.bulk (UBLKCP, completion on an mbarrier) per chunk brings their bytes --
// CIGARs, packed sequences, qualities -- into shared memory, instead of every warp chasing off -> CIGAR -> sequence
// through dependent global loads per read (k3_gather: 190 instructions per read and 128-position window, long-scoreboard
// bound).  A warp takes a record, walks its CIGAR (warp-uniform), lanes stride over the bases of an op clipped to the tile
// and add into the 7 x 1024 shared-memory counters (ATOMS; the 32 lanes of a round hit 32 consecutive positions: no bank
// conflicts).  One coalesced read-modify-write of the tile's counters at the end.  Reads longer than SPAN_SHORT stay with
// k3_scatter_long.  A record that does not fit the stage on its own is read from global memory by the same code.
constexpr uint32_t K3T_STAGE = 40 * 1024;                          // bytes of records staged per chunk
constexpr uint32_t K3T_SMEM = N_PLANES * TILE_POS * 4 + K3T_STAGE + 64;      // 28,672 + 40,960 + 64 = 69,696 B -> 3 CTAs per SM
#ifndef BDEPTH_EMULATE_SHIM
__device__ __forceinline__ void mbar_init(uint32_t mbar_sa, uint32_t count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(mbar_sa), "r"(count) : "memory"); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void bulk_g2s(uint32_t dst_sa, const void* src, uint32_t bytes, uint32_t mbar_sa) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(mbar_sa), "r"(bytes) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" :: "r"(dst_sa), "l"(src), "r"(bytes), "r"(mbar_sa) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t mbar_sa, uint32_t parity) {
    asm volatile("{\n.reg .pred p;\nWAIT_%=:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra DONE_%=;\nbra WAIT_%=;\nDONE_%=:\n}" :: "r"(mbar_sa), "r"(parity) : "memory");
}
#endif
template <bool MINQ>
__global__ void __launch_bounds__(256) k3_tile(RecordSoA soa, const uint8_t* __restrict__ u, int64_t u_end, uint32_t R, uint64_t tiles_base, uint64_t cnt_base, uint64_t win_len,
                                               const uint32_t* __restrict__ tile_first, const uint32_t* __restrict__ tile_lo, uint32_t* __restrict__ counts, uint32_t minq, int sample_sel) {
    BD_DYN_SMEM(uint8_t, smem_raw);
    uint32_t* cnt = reinterpret_cast<uint32_t*>(smem_raw);                                  // [7][1024]
    uint8_t* stage = smem_raw + N_PLANES * TILE_POS * 4;                                    // K3T_STAGE bytes, 16-byte aligned
    __shared__ unsigned long long s_mbar; __shared__ uint32_t s_r1;
    const uint32_t tile = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t lo = tile_lo[tile];
    if (lo == 0xFFFFFFFFu) return;                        // no passing short read touches this tile
    const uint32_t hi = tile_first[tile + 1];
    const uint64_t t0 = tiles_base + (uint64_t)tile * TILE_POS;
    for (uint32_t i = tid; i < N_PLANES * TILE_POS; i += 256) cnt[i] = 0;
#ifndef BDEPTH_EMULATE_SHIM
    const uint32_t mbar_sa = (uint32_t)__cvta_generic_to_shared(&s_mbar);
    if (tid == 0) mbar_init(mbar_sa, 1);
#endif
    __syncthreads();
    uint32_t parity = 0;
    for (uint32_t r0 = lo; r0 < hi;) {
        // ---- the chunk: records [r0, r1) whose bytes fit the stage (at least one record; a record larger than the stage is read in place)
        const int64_t c0 = (int64_t)((reinterpret_cast<uintptr_t>(u) + (uintptr_t)(soa.off[r0] - 4)) & ~uintptr_t(15)) - (int64_t)reinterpret_cast<uintptr_t>(u);      // start of the chunk relative to u, at a 16-byte aligned ADDRESS
        if (warp == 0) {
            // largest r1 <= hi with end(r1 - 1) - c0 <= K3T_STAGE, end(r) = start of record r + 1 (or the end of the stream): binary search on the monotone offsets
            uint32_t a = r0 + 1, b = hi;                               // r1 in [a, b]
            while (a < b) { uint32_t m = (a + b + 1) >> 1; int64_t e = m < R ? soa.off[m] - 4 : u_end; if (e - c0 <= (int64_t)K3T_STAGE) a = m; else b = m - 1; }
            if (lane == 0) s_r1 = a;
        }
        __syncthreads();
        const uint32_t r1 = s_r1;
        const int64_t c1 = r1 < R ? soa.off[r1] - 4 : u_end;
        const bool staged = c1 - c0 <= (int64_t)K3T_STAGE;             // false only for a single oversized record
        if (staged) {
            const uint32_t bytes = (uint32_t)((c1 - c0 + 15) & ~int64_t(15));       // (the stream has >= 256 readable bytes behind its end)
#ifndef BDEPTH_EMULATE_SHIM
            if (tid == 0) bulk_g2s((uint32_t)__cvta_generic_to_shared(stage), u + c0, bytes, mbar_sa);
            mbar_wait(mbar_sa, parity); parity ^= 1;
#else
            for (uint32_t i = tid; i < bytes; i += 256) stage[i] = u[c0 + i];
            __syncthreads();
#endif
        }
        const uint8_t* const rb = staged ? stage - c0 : u;             // record bytes: rb + off
        // the chunk's records are divided among the warps in contiguous runs; a warp takes 32 of its records at a time: lane i
        // loads the SoA row of record i (coalesced; one round trip for 32 records instead of a chain of dependent loads per
        // record), a ballot finds the ones that pass and touch the tile, their rows go round by shuffle
        const uint32_t per_warp = (r1 - r0 + 7) / 8, wa = r0 + warp * per_warp, wb = min(r1, wa + per_warp);
        for (uint32_t rb0 = wa; rb0 < wb; rb0 += 32) {
            const uint32_t rl = rb0 + lane;
            uint32_t mt_l = 0, span_l = 0, ncl_l = 0, lseq_l = 0; uint64_t rs_l = 0; int64_t off_l = 0; bool want = false;
            if (rl < wb) {
                mt_l = soa.meta[rl]; rs_l = soa.start[rl]; span_l = soa.span[rl];
                want = (mt_l & 3u) == 1u && (sample_sel < 0 || (int)((mt_l >> 2) & 63u) == sample_sel) && rs_l < t0 + TILE_POS && rs_l + span_l > t0;
                if (want) { off_l = soa.off[rl]; ncl_l = soa.ncl[rl]; lseq_l = (uint32_t)max(soa.lseq[rl], 0); }
            }
            unsigned todo = __ballot_sync(0xFFFFFFFFu, want);
            while (todo) {
            const int src = __ffs(todo) - 1; todo &= todo - 1;
            const uint64_t rs = __shfl_sync(0xFFFFFFFFu, rs_l, src); const uint32_t rspan = __shfl_sync(0xFFFFFFFFu, span_l, src);
            const int64_t off = __shfl_sync(0xFFFFFFFFu, off_l, src); const uint32_t ncl = __shfl_sync(0xFFFFFFFFu, ncl_l, src), lseq = __shfl_sync(0xFFFFFFFFu, lseq_l, src);
            const uint32_t n_cigar = (ncl >> 8) & 0xFFFFu, l_name = ncl & 0xFF;
            const uint8_t* cg = rb + off + 32 + l_name; const uint8_t* seq = cg + 4u * n_cigar; const uint8_t* qual = seq + (lseq + 1) / 2;
            // window of the read's reference offsets that fall into the tile: [w_lo, w_hi)
            const uint32_t w_lo = rs < t0 ? (uint32_t)(t0 - rs) : 0u;
            const uint32_t w_hi = (uint32_t)min((uint64_t)rspan, t0 + TILE_POS - rs);
            const uint32_t pbase = (uint32_t)(rs - t0);                        // position in the tile of reference offset 0 (mod 2^32)
            uint32_t rpos = 0, qpos = 0;
            for (uint32_t i = 0; i < n_cigar && rpos < w_hi; i++) {
                const uint32_t c = ld_u32_any(cg + 4 * i), len = c >> 4, op = c & 15;
                if (cig_match(op)) {
                    const uint32_t xa = rpos < w_lo ? w_lo - rpos : 0u, xb = min(len, w_hi - rpos);
                    for (uint32_t x = xa + lane; x < xb; x += 32) {
                        const uint32_t q = qpos + x;
                        if (q >= lseq) break;
                        if (MINQ) { if ((uint32_t)qual[q] < minq) continue; }
                        const uint32_t b = seq[q >> 1], nib = (q & 1) ? (b & 15u) : (b >> 4);
                        const uint32_t pl = (__popc(nib) == 1) ? (31 - __clz(nib)) : 4;        // nt16 -> nt5 (base.d:186)
                        atomicAdd(&cnt[pl * TILE_POS + (pbase + rpos + x)], 1u);
                    }
                    rpos += len; qpos += len;
                } else if (op == 2 || op == 3) {
                    const uint32_t xa = rpos < w_lo ? w_lo - rpos : 0u, xb = min(len, w_hi - rpos);
                    const uint32_t pl = op == 2 ? 5u : 6u;
                    for (uint32_t x = xa + lane; x < xb; x += 32) atomicAdd(&cnt[pl * TILE_POS + (pbase + rpos + x)], 1u);
                    rpos += len;
                } else if (cig_qcons(op)) qpos += len;
            }
            }   // records of the batch that pass
        }
        __syncthreads();                                               // the stage is reused by the next chunk
        r0 = r1;
    }
    // ---- add the tile's counters to the window (16-byte read-modify-writes; tiles are exclusive to their CTA)
    const uint64_t idx0 = t0 - cnt_base;
    if (idx0 + TILE_POS > win_len) return;
    for (uint32_t i = tid; i < N_PLANES * TILE_POS / 4; i += 256) {
        const uint4 v = reinterpret_cast<const uint4*>(cnt)[i];
        if (!(v.x | v.y | v.z | v.w)) continue;
        const uint32_t pl = i / (TILE_POS / 4), p4 = i % (TILE_POS / 4);
        uint4* dst = reinterpret_cast<uint4*>(counts + (uint64_t)pl * win_len + idx0) + p4;
        uint4 cur = *dst; cur.x += v.x; cur.y += v.y; cur.z += v.z; cur.w += v.w; *dst = cur;
    }
}

// Long reads: one warp per read, lanes stride over the bases of each op, RED atomics.
template <bool MINQ>
__global__ void k3_scatter_long(RecordSoA soa, const uint8_t* __restrict__ u, const uint32_t* __restrict__ long_list, uint32_t n_long,
                                uint64_t win_base, uint64_t win_len, uint32_t* __restrict__ counts, uint32_t minq, int sample_sel) {
    uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n_long) return;
    uint32_t rr = long_list[warp];
    if (sample_sel >= 0 && (int)((soa.meta[rr] >> 2) & 63u) != sample_sel) return;
    uint64_t rs = soa.start[rr]; uint32_t rspan = soa.span[rr];
    int64_t off = soa.off[rr]; uint32_t ncl = soa.ncl[rr]; uint32_t lseq = (uint32_t)max(soa.lseq[rr], 0);
    uint32_t n_cigar = (ncl >> 8) & 0xFFFFu, l_name = ncl & 0xFF;      // (bits 30-31 of ncl are the ghost / foreign marks)
    const uint8_t* rec = u + off; const uint8_t* cg = rec + 32 + l_name; const uint8_t* seq = cg + 4u * n_cigar; const uint8_t* qual = seq + (lseq + 1) / 2;
    uint32_t rpos = 0, qpos = 0;
    for (uint32_t i = 0; i < n_cigar; i++) {
        uint32_t c = ldu32(cg + 4 * i), len = c >> 4, op = c & 15;
        if (cig_match(op)) {
            for (uint32_t x = lane; x < len; x += 32) {
                uint32_t rp = rpos + x, q = qpos + x;
                if (rp >= rspan || q >= lseq) continue;
                uint64_t g = rs + rp; if (g < win_base || g - win_base >= win_len) continue;
                if (MINQ) { if (ldg8(qual + q) < minq) continue; }
                uint32_t b = ldg8(seq + (q >> 1)); uint32_t nib = (q & 1) ? (b & 15u) : (b >> 4);
                uint32_t pl = (__popc(nib) == 1) ? (31 - __clz(nib)) : 4;
                atomicAdd(counts + (uint64_t)pl * win_len + (g - win_base), 1u);
            }
            rpos += len; qpos += len;
        } else if (op == 2 || op == 3) {
            uint32_t pl = op == 2 ? 5 : 6;
            for (uint32_t x = lane; x < len; x += 32) {
                uint32_t rp = rpos + x; if (rp >= rspan) continue;
                uint64_t g = rs + rp; if (g < win_base || g - win_base >= win_len) continue;
                atomicAdd(counts + (uint64_t)pl * win_len + (g - win_base), 1u);
            }
            rpos += len;
        } else if (cig_qcons(op)) qpos += len;
    }
}

// ------------------------------------------------------------------------------------- BAI builder (SURVEY 8f rank 2)
// What `sambamba index` computes over the record stream (IndexBuilder, BioD/bio/std/hts/bam/bai/indexing.d:56-351), split so that the
// per-record part runs here, one thread per record of a sub-batch, and only the per-run part (one entry per change of bin) is left to the
// host (bdepth.cu: assemble_bai):
//   * linear index (:133-161): every read with a reference and a position >= 0 ("valid") offers its start to the 16 kbp windows it covers
//     -- [pos, pos + basesCovered - 1], an unmapped read only its own window; the smallest start offset wins (= the first in file order);
//     offsets here are positions in the inflated stream, the host turns them into virtual offsets;
//   * chunks (:219-246, :325-330): a chunk ends where the bin of the valid reads changes (or a new reference begins): such a read emits a
//     run entry with the end of the valid read before it (the reference's _current_chunk_beg);
//   * metadata (:117-131): mapped / unmapped reads per reference, reads without reference; the rare reads that have a reference but no
//     position take no part in the index yet count in the metadata of whatever reference is current: they go to the host as exceptions;
//   * the sortedness check (:259-271) against the previous valid read.
// The previous valid read of the sub-batch's first records is the carry (written by k_index_carry at the end of the previous sub-batch).
struct IndexCarry { unsigned long long has, key, end_abs; int ref, pos; };
struct IndexRun { unsigned long long start_abs, prev_end_abs; int ref; uint32_t bin; };       // prev_end_abs = ~0: no valid read before it
struct IndexExc { unsigned long long start_abs, end_abs; int ref; uint32_t unmapped; };
struct IndexCtl {
    unsigned long long n_runs, n_exc, last_valid /* 1 + record index */, first_placed_abs, unsorted /* 1 + record index */, past_end, bad_ref, no_coord;
};
struct IndexRec { int ref, pos; uint32_t bin, unmapped; int64_t end_pos /* pos + basesCovered */; unsigned long long abs_s, abs_e; };

__device__ __forceinline__ IndexRec index_rec(const RecordSoA& soa, const uint8_t* u, uint32_t r, unsigned long long batch_u0) {
    const int64_t o = soa.off[r];                       // of refID; block_size sits 4 bytes below
    const uint8_t* p = u + o;
    IndexRec x;
    x.ref = (int)ldu32(p); x.pos = (int)ldu32(p + 4);
    const uint32_t bmn = ldu32(p + 8), fnc = ldu32(p + 12), bs = ldu32(p - 4);
    x.bin = bmn >> 16; x.unmapped = (fnc >> 16) & 4u ? 1u : 0u;
    const uint32_t l_name = bmn & 0xFF, n_cigar = fnc & 0xFFFF;
    int64_t bc = 0;
    if (!x.unmapped) { const uint8_t* cg = p + 32 + l_name; for (uint32_t i = 0; i < n_cigar; i++) { uint32_t c = ldu32(cg + 4 * i); if (cig_rcons(c & 15)) bc += c >> 4; } }      // basesCovered (read.d:255-262)
    x.end_pos = (int64_t)x.pos + bc;
    x.abs_s = batch_u0 + (unsigned long long)(o - 4); x.abs_e = x.abs_s + 4ull + bs;
    return x;
}

__global__ void k_index_scan(RecordSoA soa, const uint8_t* __restrict__ u, uint32_t R, unsigned long long batch_u0, int n_ref,
                             const uint32_t* __restrict__ lin_base, const uint32_t* __restrict__ lin_cap, unsigned long long* __restrict__ lin, uint32_t* __restrict__ lin_len,
                             unsigned long long* __restrict__ n_mapped, unsigned long long* __restrict__ n_unmapped,
                             const IndexCarry* __restrict__ carry, IndexRun* __restrict__ runs, IndexExc* __restrict__ excs, IndexCtl* __restrict__ ctl) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x, lane = threadIdx.x & 31;
    const bool in = r < R;
    IndexRec x{-1, -1, 0, 0, 0, 0, 0};
    if (in) x = index_rec(soa, u, r, batch_u0);
    const bool valid = in && x.ref >= 0 && x.pos >= 0, placed = in && x.ref != -1;
    if (in && x.ref >= n_ref) { atomicMin(&ctl->bad_ref, (unsigned long long)r + 1); }
    const bool ok_ref = x.ref < n_ref;
    if (placed) {
        // the valid read before this one: normally r - 1; reads without position are rare, a tail of unplaced reads never looks back
        bool have = false; int pref = -1, ppos = -1; unsigned long long pkey = 0, pend = ~0ull;
        for (int64_t q = (int64_t)r - 1; q >= 0; q--) {
            IndexRec y = index_rec(soa, u, (uint32_t)q, batch_u0);
            if (y.ref >= 0 && y.pos >= 0) { have = true; pref = y.ref; ppos = y.pos; pkey = ((unsigned long long)(uint32_t)y.ref << 32) | y.bin; pend = y.abs_e; break; }
        }
        if (!have && carry->has) { have = true; pref = carry->ref; ppos = carry->pos; pkey = carry->key; pend = carry->end_abs; }
        if (have && !(pref < x.ref) && !(x.ref == pref && x.pos >= ppos)) atomicMin(&ctl->unsorted, (unsigned long long)r + 1);      // checkThatInputIsSorted
        if (ctl->first_placed_abs > x.abs_s) atomicMin(&ctl->first_placed_abs, x.abs_s);
        if (valid && ok_ref) {
            const unsigned long long key = ((unsigned long long)(uint32_t)x.ref << 32) | x.bin;
            if (!have || key != pkey) { unsigned long long i = atomicAdd(&ctl->n_runs, 1ull); runs[i] = IndexRun{x.abs_s, have ? pend : ~0ull, x.ref, x.bin}; }
            const int64_t last = x.unmapped ? (int64_t)x.pos : x.end_pos - 1;
            const uint32_t w0 = (uint32_t)x.pos >> 14, w1 = last < 0 ? 0u : (uint32_t)(last >> 14);
            const uint32_t cap = lin_cap[x.ref]; unsigned long long* L = lin + lin_base[x.ref];
            for (uint32_t w = w0; w <= w1; w++) {
                if (w >= cap) { atomicAdd(&ctl->past_end, 1ull); break; }
                if (L[w] > x.abs_s) atomicMin(&L[w], x.abs_s);
            }
            if (w1 + 1 <= cap && lin_len[x.ref] < w1 + 1) atomicMax(&lin_len[x.ref], w1 + 1);
        } else if (!valid) {
            unsigned long long i = atomicAdd(&ctl->n_exc, 1ull); excs[i] = IndexExc{x.abs_s, x.abs_e, x.ref, x.unmapped};
        }
    }
    // metadata counters: one atomic per warp when the warp's reads share a reference (sorted input: nearly always)
    const int cref = !in ? -2 : (valid && ok_ref) ? x.ref : (x.ref == -1 ? -1 : -2);      // -1: no reference; -2: counted elsewhere (exception) or nothing
    const int cref0 = __shfl_sync(0xFFFFFFFFu, cref, 0);
    const bool same = __all_sync(0xFFFFFFFFu, cref == cref0 || cref == -2);
    if (same) {
        const uint32_t bm = __ballot_sync(0xFFFFFFFFu, cref >= 0 && !x.unmapped), bu = __ballot_sync(0xFFFFFFFFu, cref >= 0 && x.unmapped), bn = __ballot_sync(0xFFFFFFFFu, cref == -1);
        const uint32_t any = __ballot_sync(0xFFFFFFFFu, cref >= 0); const int rr = __shfl_sync(0xFFFFFFFFu, cref, any ? (31 - __clz(any)) : 0);
        if (lane == 0) { if (bm) atomicAdd(&n_mapped[rr], (unsigned long long)__popc(bm)); if (bu) atomicAdd(&n_unmapped[rr], (unsigned long long)__popc(bu)); if (bn) atomicAdd(&ctl->no_coord, (unsigned long long)__popc(bn)); }
    } else {
        if (cref >= 0) { if (x.unmapped) atomicAdd(&n_unmapped[cref], 1ull); else atomicAdd(&n_mapped[cref], 1ull); }
        else if (cref == -1) atomicAdd(&ctl->no_coord, 1ull);
    }
    const uint32_t bv = __ballot_sync(0xFFFFFFFFu, valid && ok_ref);
    if (bv && lane == 31 - __clz(bv)) { if (ctl->last_valid < (unsigned long long)r + 1) atomicMax(&ctl->last_valid, (unsigned long long)r + 1); }
}

// the last valid read of the sub-batch becomes the carry of the next one
__global__ void k_index_carry(RecordSoA soa, const uint8_t* __restrict__ u, unsigned long long batch_u0, IndexCarry* __restrict__ carry, IndexCtl* __restrict__ ctl) {
    if (threadIdx.x || blockIdx.x) return;
    if (ctl->last_valid) {
        IndexRec y = index_rec(soa, u, (uint32_t)(ctl->last_valid - 1), batch_u0);
        carry->has = 1; carry->key = ((unsigned long long)(uint32_t)y.ref << 32) | y.bin; carry->end_abs = y.abs_e; carry->ref = y.ref; carry->pos = y.pos;
    }
    ctl->last_valid = 0;
}

// ------------------------------------------------------------------------------------- reducers
// number of positions in [a, b) (window-relative) whose 7 counters sum to > 0
__global__ void k_count_covered(const uint32_t* __restrict__ counts, uint64_t win_len, uint64_t a, uint64_t b, unsigned long long* __restrict__ out, int n_planes) {
    uint64_t i = a + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    unsigned long long n = 0;
    for (; i < b; i += stride) {
        uint32_t s = 0;
        for (int pl = 0; pl < n_planes; pl++) s |= counts[(uint64_t)pl * win_len + i];
        n += s != 0;
    }
    for (int sft = 16; sft; sft >>= 1) n += __shfl_xor_sync(0xFFFFFFFFu, n, sft);
    if ((threadIdx.x & 31) == 0 && n) atomicAdd(out, n);
}

// Segment statistics over the counters: one warp per segment [seg_a[i], seg_b[i]) (window-relative).
// out_bases[i] += sum(A+C+G+T+N); out_cov[t][i] += #positions with all-7 sum >= thr[t].
__global__ void k_segment_stats(const uint32_t* __restrict__ counts, uint64_t win_len, const uint64_t* __restrict__ seg_a, const uint64_t* __restrict__ seg_a_cov, const uint64_t* __restrict__ seg_b,
                                uint32_t n_seg, const uint32_t* __restrict__ thr, uint32_t n_thr, uint32_t* __restrict__ out_bases, uint32_t* __restrict__ out_cov /* [n_thr][n_seg] */) {
    uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= n_seg) return;
    // bases are summed over [a, b); thresholds are counted over [a_cov, b) with a_cov <= a (the reference's window
    // slots start collecting coverage before their window begins when the step does not divide the window)
    uint64_t a = seg_a[warp], ac = seg_a_cov[warp], b = seg_b[warp];
    uint32_t bases = 0; uint32_t cge[16];
#pragma unroll
    for (int t = 0; t < 16; t++) cge[t] = 0;
    for (uint64_t i = ac + lane; i < b; i += 32) {
        uint32_t s5 = 0, s = 0;
#pragma unroll
        for (int pl = 0; pl < N_PLANES; pl++) { uint32_t v = counts[(uint64_t)pl * win_len + i]; s += v; if (pl < 5) s5 += v; }
        if (i >= a) bases += s5;
        if (s) {
#pragma unroll
            for (int t = 0; t < 16; t++) if ((uint32_t)t < n_thr) cge[t] += s >= thr[t];
        }
    }
    for (int sft = 16; sft; sft >>= 1) {
        bases += __shfl_xor_sync(0xFFFFFFFFu, bases, sft);
#pragma unroll
        for (int t = 0; t < 16; t++) cge[t] += __shfl_xor_sync(0xFFFFFFFFu, cge[t], sft);
    }
    if (lane == 0) {
        if (bases) atomicAdd(&out_bases[warp], bases);
#pragma unroll
        for (int t = 0; t < 16; t++) if ((uint32_t)t < n_thr && cge[t]) atomicAdd(&out_cov[(uint64_t)t * n_seg + warp], cge[t]);
    }
}

// Per-read "countRead" (depth.d:661-669) against sorted segments: a read adds 1 to n_reads of every
// segment in which it has >= 1 M/=/X base with quality >= minq.  Segments are given sorted by start
// in LINEAR coordinates with pmax_end[i] = max(end[0..i]) for pruning; seg_id maps to the output slot.
template <bool MINQ>
__global__ void k_read_segments(RecordSoA soa, const uint8_t* __restrict__ u, uint32_t R, const uint64_t* __restrict__ seg_s, const uint64_t* __restrict__ seg_e,
                                const uint64_t* __restrict__ pmax_end, const uint32_t* __restrict__ seg_id, const uint64_t* __restrict__ seg_min_start, uint32_t n_seg,
                                uint32_t* __restrict__ out_reads /* [n_samples][n_seg] */, uint32_t minq, uint32_t n_samples, uint32_t* __restrict__ out_bases_reads) {
    uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    if (!(soa.meta[r] & 1u) || (soa.ncl[r] & NCL_FOREIGN)) return;      // (a zone read is counted by the rank whose shard holds it)
    const uint32_t samp = n_samples > 1 ? ((soa.meta[r] >> 2) & 63u) : 0u;
    uint64_t rs = soa.start[r]; uint32_t rspan = soa.span[r]; uint64_t re = rs + rspan;
    // candidates: segments with seg_s < re ; walk down from the last such while pmax_end > rs
    uint32_t lo = 0, hi = n_seg;
    while (lo < hi) { uint32_t mid = (lo + hi) >> 1; if (seg_s[mid] < re) lo = mid + 1; else hi = mid; }
    if (lo == 0) return;
    int64_t off = soa.off[r]; uint32_t ncl = soa.ncl[r]; uint32_t lseq = (uint32_t)max(soa.lseq[r], 0);
    uint32_t n_cigar = (ncl >> 8) & 0xFFFFu, l_name = ncl & 0xFF;      // (bits 30-31 of ncl are the ghost / foreign marks)
    const uint8_t* rec = u + off; const uint8_t* cg = rec + 32 + l_name; const uint8_t* qual = cg + 4u * n_cigar + (lseq + 1) / 2;
    for (int64_t k = (int64_t)lo - 1; k >= 0; k--) {
        if (pmax_end[k] <= rs) break;
        uint64_t a = seg_s[k], b = seg_e[k];
        if (b <= rs || a >= re) continue;
        const bool q6 = seg_min_start && seg_min_start[k] != 0;     // window-mode first-occurrence quirk (depth.d:1031-1032):
        if (q6 && rs < seg_min_start[k]) continue;                  // such a slot only ever sees reads that START inside it
        // any M base with q >= minq inside [a,b)?  (for quirk slots: how many, their n_bases comes from countRead alone)
        bool hit = false; uint32_t rpos = 0, qpos = 0, nb = 0;
        for (uint32_t i = 0; i < n_cigar && (q6 || !hit); i++) {
            uint32_t c = ldu32(cg + 4 * i), len = c >> 4, op = c & 15;
            if (cig_match(op)) {
                uint64_t ma = rs + rpos, mb = ma + len; if (mb > re) mb = re;
                uint64_t xa = ma > a ? ma : a, xb = mb < b ? mb : b;
                if (xa < xb) {
                    if (!MINQ && !q6) hit = (qpos + (uint32_t)(xa - ma)) < lseq;
                    else for (uint64_t g = xa; g < xb && (q6 || !hit); g++) { uint32_t q = qpos + (uint32_t)(g - ma); if (q < lseq && (!MINQ || ldg8(qual + q) >= minq)) { hit = true; nb++; } }
                }
                rpos += len; qpos += len;
            } else if (op == 2 || op == 3) rpos += len;
            else if (cig_qcons(op)) qpos += len;
        }
        if (q6 && nb && out_bases_reads) atomicAdd(&out_bases_reads[(uint64_t)samp * n_seg + seg_id[k]], nb);
        if (hit) atomicAdd(&out_reads[(uint64_t)samp * n_seg + seg_id[k]], 1u);
    }
}


// ------------------------------------------------------------------------------------- text (SURVEY 8f rank 1)
// GPU formatting of `depth base` rows (PerBasePrinter.writeColumn, depth.d:534-555, and the zero rows of
// writeEmptyColumns, depth.d:452-487) for one sample / --combined:
//   <ref>\t<pos>\t<COV>\t<A>\t<C>\t<G>\t<T>\t<DEL>\t<REFSKIP>[\t<sample>][\t<y|n>]\n
// Pass 1 sums the row lengths per 1024-position tile, a single block scans the tile sums, pass 2 re-derives the
// lengths, scans inside the tile and writes the bytes.  The host only fwrite()s.
struct TextParams {
    double min_cov, max_cov;
    int annotate, with_sample;
    uint32_t name_len, sample_len;
    char name[256], sample[256];
    const uint32_t* present;      // optional bitmap (window-relative): a read covers the position even if -q left no counted base (k_presence)
};
// With -a, -q and a positive minimum coverage the reference still prints a row (flag n) for a position that reads cover but
// whose every base fails -q: the column exists, its counters are zero (depth.d:534-555).  The counters alone cannot tell
// that from "no read here", so such runs also mark the covered positions: one bit per position, thread per passing read.
__global__ void k_presence(RecordSoA soa, uint32_t R, uint64_t cnt_base, uint64_t win_len, uint32_t* __restrict__ present) {
    uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R || !(soa.meta[r] & 1u)) return;
    uint64_t a = soa.start[r], b = a + soa.span[r];
    if (a < cnt_base) a = cnt_base;
    if (b > cnt_base + win_len) b = cnt_base + win_len;
    if (a >= b) return;
    a -= cnt_base; b -= cnt_base;
    for (uint64_t w = a >> 5; w <= (b - 1) >> 5; w++) {
        uint32_t lo = w == (a >> 5) ? (uint32_t)(a & 31) : 0u, hi = w == ((b - 1) >> 5) ? (uint32_t)((b - 1) & 31) : 31u;
        uint32_t m = (hi == 31 ? 0xFFFFFFFFu : ((1u << (hi + 1)) - 1u)) & ~((1u << lo) - 1u);
        atomicOr(&present[w], m);
    }
}
// Quirk 1 (SURVEY 8a): PileupRead's constructor looks for the first M/=/X/D operation and steps over N operations on the way WITHOUT
// consuming them (pileup.d:180-189), while the read still occupies basesCovered() columns from its position.  The cursor therefore
// runs through the rest of the CIGAR that many columns early and, once past the last operation, stays on the last one it examined --
// cigar[$ - 1] -- for the columns that are left (incrementPosition leaves _cur_op alone when it finds nothing, :207-218): a D counts
// deletions there, every operation that does not consume both query and reference (N, S, I, H, P) counts reference skips
// (depth.d:507-513).  That is exactly the CIGAR with its leading N operations taken out and as many skipped (or deleted) columns
// appended: k2_lead_n_find / k2_lead_n_fix rewrite such a CIGAR in the inflated stream, in place and in the same number of operations (
// after k2_decode -- the -F query has seen the original -- and before anything walks CIGARs), and every later kernel then computes what the
// reference computes.  If the last operation is M/=/X the reference indexes the sequence and the qualities past their end for those
// columns (release build: unchecked reads): there is nothing to reproduce, the run is refused.  Real aligners never write a leading N;
// the cost for ordinary reads is one look at the first reference-consuming operation.
// Region and window statistics mix the two views: readCount and meanCoverage go through countOverlappingBases, which walks the CIGAR
// from the read's position as written (depth.d:671-698), the percentages through the shifted cursor.  Window mode, -m and several
// ranks keep per-slot / per-pair / per-rank books of their own on top of that: with refuse_all such a read ends the run whatever
// its last operation is.
// (With -L only reads that overlap a region are in the reference's stream at all: flt_s / flt_e as in k_ref_seen; the others cannot end the run.)
// Region mode on one rank without -m (seg.n_seg != 0) is reproduced as well: the reducers take n_bases from the counter planes and the
// read count from k_read_segments, both of which will see the rewritten CIGAR, so this kernel books the difference to the CIGAR as
// written for every region the read overlaps -- (+ bases, + read) before the rewrite, (- bases, - read) after it -- into the arrays the
// reducers add on top (seg_mbases, seg_reads: the ones the mate kernels use for the same purpose).
struct LeadNSegs { const uint64_t* s; const uint64_t* e; const uint64_t* pmax; const uint32_t* id; uint32_t n_seg; uint32_t* reads; uint32_t* mbases; uint32_t n_samples; uint32_t minq; };
__device__ BD_NOINLINE void lead_n_book(const LeadNSegs& sg, const RecordSoA& soa, const uint8_t* u, uint32_t r, uint32_t sign) {
    const uint64_t rs = soa.start[r], re = rs + soa.span[r];
    uint32_t lo = 0, hi = sg.n_seg;
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (sg.s[mid] < re) lo = mid + 1; else hi = mid; }
    const uint32_t ncl = soa.ncl[r], n_cigar = (ncl >> 8) & 0xFFFFu, l_name = ncl & 0xFFu, lseq = (uint32_t)max(soa.lseq[r], 0);
    const uint8_t* cg = u + soa.off[r] + 32 + l_name; const uint8_t* qual = cg + 4u * n_cigar + (lseq + 1) / 2;
    const uint32_t samp = sg.n_samples > 1 ? ((soa.meta[r] >> 2) & 63u) : 0u;
    for (int64_t k = (int64_t)lo - 1; k >= 0; k--) {
        if (sg.pmax[k] <= rs) break;
        const uint64_t a = sg.s[k], b = sg.e[k];
        if (b <= rs || a >= re) continue;
        uint32_t rpos = 0, qpos = 0, nb = 0;                       // countOverlappingBases (depth.d:671-698) of the CIGAR as it stands in the stream
        for (uint32_t i = 0; i < n_cigar; i++) {
            const uint8_t* q4 = cg + 4 * i; const uint32_t c = (uint32_t)q4[0] | ((uint32_t)q4[1] << 8) | ((uint32_t)q4[2] << 16) | ((uint32_t)q4[3] << 24), len = c >> 4, op = c & 15u;
            if (cig_match(op)) {
                uint64_t ma = rs + rpos, mb = ma + len; if (mb > re) mb = re;
                const uint64_t xa = ma > a ? ma : a, xb = mb < b ? mb : b;
                for (uint64_t g = xa; g < xb; g++) { const uint32_t q = qpos + (uint32_t)(g - ma); if (q < lseq && qual[q] >= sg.minq) nb++; }
                rpos += len; qpos += len;
            } else if (op == 2u || op == 3u) rpos += len;
            else if (cig_qcons(op)) qpos += len;
        }
        if (nb) { atomicAdd(&sg.mbases[(uint64_t)samp * sg.n_seg + sg.id[k]], sign * nb); atomicAdd(&sg.reads[(uint64_t)samp * sg.n_seg + sg.id[k]], sign); }
    }
}
// Step 1, every record: does the first reference-consuming operation say N?  (the usual answer after one or two loads is no)
__global__ void __launch_bounds__(256) k2_lead_n_find(RecordSoA soa, const uint8_t* u, uint32_t R, uint32_t* __restrict__ list, ScanStats* __restrict__ st) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    const uint32_t ncl = soa.ncl[r];
    if (!((soa.meta[r] & 1u) || (ncl & (NCL_GHOST | NCL_FOREIGN)))) return;      // only reads that are counted (or re-read for the mate kernels)
    const uint32_t n_cigar = (ncl >> 8) & 0xFFFFu;
    if (n_cigar < 2) return;                                      // (an N in front of an M/=/X/D takes two operations: most reads are one M and never touch their CIGAR here)
    const uint8_t* cg = u + soa.off[r] + 32 + (ncl & 0xFFu);
    for (uint32_t i = 0; i < n_cigar; i++) {
        const uint32_t op = ld_u32_any(cg + 4 * i) & 15u;       // (plain loads: step 2 writes CIGAR bytes)
        if (!cig_rcons(op)) continue;
        if (op == 3u) list[(uint32_t)atomicAdd(&st->n_lead, 1ull)] = r;
        return;
    }
}
// Step 2, the records step 1 listed (none, in any file an aligner wrote): a few blocks stride over the list.
__global__ void __launch_bounds__(128) k2_lead_n_fix(RecordSoA soa, uint8_t* u, const uint32_t* __restrict__ list, ScanStats* __restrict__ st, int refuse_all,
                                                     const uint64_t* __restrict__ flt_s, const uint64_t* __restrict__ flt_e, uint32_t n_flt, LeadNSegs sg) {
    const unsigned long long n = st->n_lead;
    for (unsigned long long li = blockIdx.x * blockDim.x + threadIdx.x; li < n; li += (unsigned long long)gridDim.x * blockDim.x) {
        const uint32_t r = list[li];
        const uint32_t ncl = soa.ncl[r], n_cigar = (ncl >> 8) & 0xFFFFu, l_name = ncl & 0xFFu;
        uint8_t* cg = u + soa.off[r] + 32 + l_name;
        auto ld = [&](uint32_t j) { const uint8_t* q = cg + 4 * j; return (uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24); };
        auto st4 = [&](uint32_t j, uint32_t v) { uint8_t* q = cg + 4 * j; q[0] = (uint8_t)v; q[1] = (uint8_t)(v >> 8); q[2] = (uint8_t)(v >> 16); q[3] = (uint8_t)(v >> 24); };
        uint32_t first = 0, k = 0; uint64_t nlead = 0; bool found = false, zero = false;
        for (; first < n_cigar; first++) {
            const uint32_t c = ld(first), op = c & 15u;
            if (!cig_rcons(op)) continue;
            if (op != 3u) { found = true; break; }
            nlead += c >> 4; k++; zero |= (c >> 4) == 0;
        }
        if (!k || !found) continue;          // nothing but N consumes the reference: the cursor never leaves the last operation and every column is a skip, as the CIGAR says
        const uint32_t last_op = ld(n_cigar - 1) & 15u;
        if (refuse_all || last_op == 0u || last_op == 7u || last_op == 8u || zero || nlead >= (1ull << 28)) {
            bool in_stream = true;
            if (n_flt) {
                const uint64_t s0 = soa.start[r], e0 = s0 + soa.span[r];
                uint32_t lo = 0, hi = n_flt;
                while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (flt_e[mid] <= s0) lo = mid + 1; else hi = mid; }
                in_stream = lo < n_flt && flt_s[lo] < e0;
            }
            if (in_stream) atomicMin(&st->lead_n, (unsigned long long)r + 1);
            continue;
        }
        const bool book = sg.n_seg != 0 && (soa.meta[r] & 1u) && !(ncl & NCL_FOREIGN);
        if (book) lead_n_book(sg, soa, u, r, 1u);
        uint32_t w = 0;
        for (uint32_t j = 0; j < n_cigar; j++) { const uint32_t c = ld(j); if (j < first && (c & 15u) == 3u) continue; st4(w++, c); }      // w <= j: a slot is read before it is overwritten
        const uint32_t tail_op = last_op == 2u ? 2u : 3u;
        for (uint32_t t = 0; t + 1 < k; t++) st4(w++, (1u << 4) | tail_op);                     // k operations went out, k come in: k - 1 of one column ...
        st4(w, ((uint32_t)(nlead - (k - 1)) << 4) | tail_op);                                       // ... and the rest (every leading N had at least one column: nlead >= k)
        if (book) lead_n_book(sg, soa, u, r, 0xFFFFFFFFu);
    }
}

// With -L the reference's pileup only ever sees the reads that overlap a region (getReadsOverlapping, randomaccessmanager.d:316-338): a
// reference "has reads" -- is announced, gets its empty rows with --min-coverage=0 (depth.d:574-586), carries window state -- iff such a
// read passes the filter.  K2 marks every passing read's reference; runs with regions mark through this kernel instead (thread per read;
// flt_s / flt_e: the merged regions in linear coordinates, sorted and disjoint, as mates.cuh uses them).
__global__ void k_ref_seen(RecordSoA soa, uint32_t R, const uint64_t* __restrict__ flt_s, const uint64_t* __restrict__ flt_e, uint32_t n_flt,
                           const uint64_t* __restrict__ ref_lin0, uint32_t n_ref, uint32_t* __restrict__ ref_has_reads) {
    const uint32_t r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R || !(soa.meta[r] & 1u) || !n_ref) return;
    const uint64_t s = soa.start[r], e = s + soa.span[r];
    uint32_t lo = 0, hi = n_flt;                                   // first region that ends after the read starts; the read is in the stream iff it reaches it
    while (lo < hi) { const uint32_t mid = (lo + hi) >> 1; if (flt_e[mid] <= s) lo = mid + 1; else hi = mid; }
    if (lo >= n_flt || flt_s[lo] >= e) return;
    uint32_t a = 0, b = n_ref;                                     // the last reference that begins at or before s (an empty reference shares its successor's origin)
    while (a + 1 < b) { const uint32_t mid = (a + b) >> 1; if (ref_lin0[mid] <= s) a = mid; else b = mid; }
    atomicOr(&ref_has_reads[a >> 5], 1u << (a & 31));
}
__device__ __forceinline__ uint32_t dec_digits(uint32_t v) {
    return v < 10u ? 1u : v < 100u ? 2u : v < 1000u ? 3u : v < 10000u ? 4u : v < 100000u ? 5u : v < 1000000u ? 6u : v < 10000000u ? 7u : v < 100000000u ? 8u : v < 1000000000u ? 9u : 10u;
}
__device__ __forceinline__ char* put_dec(char* p, uint32_t v) {     // writes v, returns the end
    uint32_t n = dec_digits(v); char* e = p + n;
    do { *--e = (char)('0' + v % 10u); v /= 10u; } while (v);
    return p + n;
}
// row length of one position, 0 when the row is not printed
__device__ __forceinline__ uint32_t text_row(const TextParams& tp, const uint32_t* __restrict__ counts, uint64_t win_len, uint64_t idx, uint32_t pos, uint32_t* v, bool* okp) {
    uint32_t total = 0;
#pragma unroll
    for (int pl = 0; pl < N_PLANES; pl++) { v[pl] = counts[(uint64_t)pl * win_len + idx]; total += v[pl]; }
    bool ok = (double)total >= tp.min_cov && (double)total <= tp.max_cov;
    *okp = ok;
    if (!ok && !tp.annotate) return 0;
    if (total == 0 && tp.min_cov > 0 && !(tp.present && tp.annotate && ((tp.present[idx >> 5] >> (idx & 31)) & 1u))) return 0;          // no column at all: nothing is written when min_cov > 0 (depth.d:568-572)
    uint32_t len = tp.name_len + 1 + dec_digits(pos) + 1 + dec_digits(total);
    len += 1 + dec_digits(v[0]) + 1 + dec_digits(v[1]) + 1 + dec_digits(v[2]) + 1 + dec_digits(v[3]) + 1 + dec_digits(v[5]) + 1 + dec_digits(v[6]);
    if (tp.with_sample) len += 1 + tp.sample_len;
    if (tp.annotate) len += 2;
    return len + 1;
}
// pass 1: tile_sum[t] = bytes of tile t (TEXT_TILE positions starting at idx0 + t*TEXT_TILE)
constexpr int TEXT_TILE = 1024;
__global__ void __launch_bounds__(256) k_text_len(TextParams tp, const uint32_t* __restrict__ counts, uint64_t win_len, uint64_t idx0, uint32_t pos0, uint32_t n, uint32_t* __restrict__ tile_sum) {
    __shared__ uint32_t wsum[8];
    uint32_t base = blockIdx.x * TEXT_TILE, s = 0;
    for (int k = 0; k < 4; k++) {
        uint32_t i = base + threadIdx.x * 4 + k; uint32_t v[N_PLANES]; bool ok;
        if (i < n) s += text_row(tp, counts, win_len, idx0 + i, pos0 + i, v, &ok);
    }
    for (int sh = 16; sh; sh >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, sh);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < 8; w++) t += wsum[w]; tile_sum[blockIdx.x] = t; }
}
// exclusive scan of up to 1024*16 tile sums by one block (64-bit offsets)
__global__ void __launch_bounds__(1024) k_text_scan(const uint32_t* __restrict__ tile_sum, uint32_t n_tiles, unsigned long long* __restrict__ tile_off, unsigned long long* __restrict__ total) {
    __shared__ unsigned long long wtot[32];
    const uint32_t per = (n_tiles + 1023) / 1024, lo = threadIdx.x * per, hi = min(n_tiles, lo + per), lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned long long s = 0;
    for (uint32_t i = lo; i < hi; i++) s += tile_sum[i];
    // exclusive scan of the 1024 partial sums: a shuffle scan inside every warp, then one over the 32 warp totals
    unsigned long long incl = s;
    for (uint32_t sh = 1; sh < 32; sh <<= 1) { unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, incl, sh); if (lane >= sh) incl += t; }
    if (lane == 31) wtot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const unsigned long long w = wtot[lane]; unsigned long long wi = w;
        for (uint32_t sh = 1; sh < 32; sh <<= 1) { unsigned long long t = __shfl_up_sync(0xFFFFFFFFu, wi, sh); if (lane >= sh) wi += t; }
        wtot[lane] = wi - w;
        if (lane == 31) *total = wi;
    }
    __syncthreads();
    unsigned long long a = wtot[warp] + incl - s;
    for (uint32_t i = lo; i < hi; i++) { tile_off[i] = a; a += tile_sum[i]; }
}
// pass 2: write the rows
__global__ void __launch_bounds__(256) k_text_write(TextParams tp, const uint32_t* __restrict__ counts, uint64_t win_len, uint64_t idx0, uint32_t pos0, uint32_t n,
                                                    const unsigned long long* __restrict__ tile_off, char* __restrict__ out) {
    __shared__ uint32_t wsum[8];
    uint32_t base = blockIdx.x * TEXT_TILE, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t len[4], v[4][N_PLANES]; bool ok[4]; uint32_t mine = 0;
    for (int k = 0; k < 4; k++) { uint32_t i = base + threadIdx.x * 4 + k; len[k] = i < n ? text_row(tp, counts, win_len, idx0 + i, pos0 + i, v[k], &ok[k]) : 0; mine += len[k]; }
    uint32_t incl = mine;
    for (int sh = 1; sh < 32; sh <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, sh); if (lane >= (uint32_t)sh) incl += t; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    uint32_t woff = 0; for (uint32_t w = 0; w < warp; w++) woff += wsum[w];
    char* p = out + tile_off[blockIdx.x] + woff + (incl - mine);
    for (int k = 0; k < 4; k++) {
        if (!len[k]) continue;
        uint32_t i = base + threadIdx.x * 4 + k; const uint32_t* c = v[k];
        uint32_t total = c[0] + c[1] + c[2] + c[3] + c[4] + c[5] + c[6];
        for (uint32_t q = 0; q < tp.name_len; q++) *p++ = tp.name[q];
        *p++ = '\t'; p = put_dec(p, pos0 + i); *p++ = '\t'; p = put_dec(p, total);
        *p++ = '\t'; p = put_dec(p, c[0]); *p++ = '\t'; p = put_dec(p, c[1]); *p++ = '\t'; p = put_dec(p, c[2]); *p++ = '\t'; p = put_dec(p, c[3]);
        *p++ = '\t'; p = put_dec(p, c[5]); *p++ = '\t'; p = put_dec(p, c[6]);
        if (tp.with_sample) { *p++ = '\t'; for (uint32_t q = 0; q < tp.sample_len; q++) *p++ = tp.sample[q]; }
        if (tp.annotate) { *p++ = '\t'; *p++ = total == 0 ? (tp.min_cov > 0 ? 'n' : 'y') : (ok[k] ? 'y' : 'n'); }
        *p++ = '\n';
    }
}

// ---- the same for several samples: every position prints one row per sample, in sample order, and the first sample whose
// COV is out of bounds ends the position (writeColumn returns instead of continuing, depth.d:540-541 -- SURVEY quirk 2);
// a position without any read prints nothing when min_cov > 0 and one zero row per sample otherwise (depth.d:452-487).
struct TextParamsMS {
    double min_cov, max_cov; int annotate; uint32_t name_len; char name[256];
    uint32_t S; const char* samp; const uint32_t* samp_off;      // sample names concatenated, S + 1 offsets
    uint64_t sample_stride;                                       // elements between the counter sets of two samples (0: all read the same planes)
    const uint32_t* present;                                      // as in TextParams
};
// length of the rows of one position; writes them when p != nullptr
__device__ __forceinline__ uint32_t text_rows_ms(const TextParamsMS& tp, const uint32_t* __restrict__ counts, uint64_t win_len, uint64_t idx, uint32_t pos, char* p) {
    uint32_t any = 0;
    for (uint32_t s = 0; s < tp.S; s++) for (int pl = 0; pl < N_PLANES; pl++) any |= counts[(uint64_t)s * tp.sample_stride + (uint64_t)pl * win_len + idx];
    if (!any && tp.present && ((tp.present[idx >> 5] >> (idx & 31)) & 1u)) any = 1;      // the column exists although -q left nothing to count
    if (!any && tp.min_cov > 0) return 0;
    uint32_t len = 0;
    for (uint32_t s = 0; s < tp.S; s++) {
        uint32_t v[N_PLANES], total = 0;
#pragma unroll
        for (int pl = 0; pl < N_PLANES; pl++) { v[pl] = counts[(uint64_t)s * tp.sample_stride + (uint64_t)pl * win_len + idx]; total += v[pl]; }
        const bool ok = (double)total >= tp.min_cov && (double)total <= tp.max_cov;
        if (!ok && !tp.annotate) break;
        const uint32_t sl = tp.samp_off[s + 1] - tp.samp_off[s];
        uint32_t rl = tp.name_len + 1 + dec_digits(pos) + 1 + dec_digits(total) + 1 + dec_digits(v[0]) + 1 + dec_digits(v[1]) + 1 + dec_digits(v[2]) + 1 + dec_digits(v[3]) + 1 + dec_digits(v[5]) + 1 + dec_digits(v[6]) + 1 + sl + (tp.annotate ? 2 : 0) + 1;
        if (p) {
            char* q = p + len;
            for (uint32_t k = 0; k < tp.name_len; k++) *q++ = tp.name[k];
            *q++ = '\t'; q = put_dec(q, pos); *q++ = '\t'; q = put_dec(q, total);
            *q++ = '\t'; q = put_dec(q, v[0]); *q++ = '\t'; q = put_dec(q, v[1]); *q++ = '\t'; q = put_dec(q, v[2]); *q++ = '\t'; q = put_dec(q, v[3]);
            *q++ = '\t'; q = put_dec(q, v[5]); *q++ = '\t'; q = put_dec(q, v[6]);
            *q++ = '\t'; for (uint32_t k = 0; k < sl; k++) *q++ = tp.samp[tp.samp_off[s] + k];
            if (tp.annotate) { *q++ = '\t'; *q++ = !any ? (tp.min_cov > 0 ? 'n' : 'y') : (ok ? 'y' : 'n'); }
            *q++ = '\n';
        }
        len += rl;
    }
    return len;
}
__global__ void __launch_bounds__(256) k_text_len_ms(TextParamsMS tp, const uint32_t* __restrict__ counts, uint64_t win_len, uint64_t idx0, uint32_t pos0, uint32_t n, uint32_t* __restrict__ tile_sum) {
    __shared__ uint32_t wsum[8];
    uint32_t base = blockIdx.x * TEXT_TILE, s = 0;
    for (int k = 0; k < 4; k++) { uint32_t i = base + threadIdx.x * 4 + k; if (i < n) s += text_rows_ms(tp, counts, win_len, idx0 + i, pos0 + i, nullptr); }
    for (int sh = 16; sh; sh >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, sh);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < 8; w++) t += wsum[w]; tile_sum[blockIdx.x] = t; }
}
__global__ void __launch_bounds__(256) k_text_write_ms(TextParamsMS tp, const uint32_t* __restrict__ counts, uint64_t win_len, uint64_t idx0, uint32_t pos0, uint32_t n,
                                                       const unsigned long long* __restrict__ tile_off, char* __restrict__ out) {
    __shared__ uint32_t wsum[8];
    uint32_t base = blockIdx.x * TEXT_TILE, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t len[4], mine = 0;
    for (int k = 0; k < 4; k++) { uint32_t i = base + threadIdx.x * 4 + k; len[k] = i < n ? text_rows_ms(tp, counts, win_len, idx0 + i, pos0 + i, nullptr) : 0; mine += len[k]; }
    uint32_t incl = mine;
    for (int sh = 1; sh < 32; sh <<= 1) { uint32_t t = __shfl_up_sync(0xFFFFFFFFu, incl, sh); if (lane >= (uint32_t)sh) incl += t; }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    uint32_t woff = 0; for (uint32_t w = 0; w < warp; w++) woff += wsum[w];
    char* p = out + tile_off[blockIdx.x] + woff + (incl - mine);
    for (int k = 0; k < 4; k++) { if (!len[k]) continue; uint32_t i = base + threadIdx.x * 4 + k; text_rows_ms(tp, counts, win_len, idx0 + i, pos0 + i, p); p += len[k]; }
}

}  // namespace bdk
