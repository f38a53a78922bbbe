/*
 * bdepth.h -- C ABI of libbdepth.so, the B200-native engine behind `sambamba depth`.
 *
 * The reference has NO foreign-function boundary on this path (SURVEY.md F4): `depth` is D
 * ranges composed in one function, sambamba/depth.d:1211-1232.  This header therefore DEFINES
 * the drop-in boundary at the seam where the reference hands data between layers:
 *
 *   reference seam (what each entry point replaces)                      entry point
 *   -------------------------------------------------------------------  ----------------------
 *   new MultiBamReader(files)            sambamba/depth.d:1163,          bdepth_open /
 *     BamReader.this                     BioD/bio/std/hts/bam/reader.d:101-125   bdepth_open_memory
 *   bam.header.sorting_order, has_index  depth.d:1164-1166               bdepth_is_coordinate_sorted,
 *                                                                        bdepth_has_index
 *   bam.reference_sequences[i].name/.length  reader.d:588-598            bdepth_n_ref/_ref_name/_ref_length
 *   bam.header.read_groups -> sample table   depth.d:1170-1181           bdepth_n_samples/_sample_name
 *   createFilterFromQuery(default)       depth.d:1159, filtering.d:40-51 bdepth_set_filter
 *   printer.min_base_quality             depth.d:280,1129                bdepth_set_min_baseq
 *   bam.getReadsOverlapping(bed)         depth.d:1211, multireader.d:357 bdepth_set_regions
 *   foreach (column; pileupColumns(..)) printer.push(column)             bdepth_run_base   (PerBasePrinter,  depth.d:402-607)
 *     BGZF inflate   BioD/bio/core/bgzf/block.d:127-216                  bdepth_run_windows(PerWindowPrinter, depth.d:933-1077)
 *     record walk    BioD/bio/std/hts/bam/readrange.d:118-173            bdepth_run_regions(PerBedRegionPrinter, depth.d:879-931)
 *     column sweep   BioD/bio/std/hts/bam/pileup.d:345-424
 *
 * Conventions: every entry returns 0 on success or a negative bdepth_status; the message is
 * available through bdepth_last_error().  No exception crosses the boundary.  There is no CPU
 * fallback: a missing GPU or a CUDA failure is BDEPTH_ERR_CUDA.  The library owns all device and
 * pinned memory; pointers handed to callbacks are valid only during the callback (like the
 * reference's transient Column, pileup.d:660-664).  Callbacks run on the calling thread, in
 * (ref_id, position) order, never concurrently.  The caller owns path strings and region arrays
 * for the duration of the call that receives them.
 */
#ifndef BDEPTH_H
#define BDEPTH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bdepth bdepth_t;

typedef enum {
    BDEPTH_OK = 0,
    BDEPTH_ERR_IO = -1,        /* cannot open / read / mmap                                  */
    BDEPTH_ERR_FORMAT = -2,    /* BGZF / BAM / BAI / DEFLATE format error                    */
    BDEPTH_ERR_UNSORTED = -3,  /* header does not say SO:coordinate  (depth.d:1164)          */
    BDEPTH_ERR_NOINDEX = -4,   /* no .bai next to the file           (depth.d:1166)          */
    BDEPTH_ERR_CUDA = -5,      /* no device, CUDA error, out of device memory                */
    BDEPTH_ERR_NCCL = -6,      /* a NCCL call failed -- or another rank of the run stopped with an error: every rank then returns this instead of waiting for it */
    BDEPTH_ERR_ARG = -7,       /* bad argument / unsupported combination                     */
    BDEPTH_ERR_CALLBACK = -8   /* a callback returned non-zero                               */
} bdepth_status;

/* 0-based half-open interval on a reference, same meaning as BamRegion
 * (BioD/bio/std/hts/bam/region.d:28-31). */
typedef struct { uint32_t ref_id, start, end; } bdepth_region;

/* One position-ordered tile of per-base counters.  counts is SoA: plane p (A,C,G,T,N,DEL,REFSKIP
 * = the seven counters of PerBasePrinter.writeColumn, depth.d:495-556) occupies
 * counts[p * stride .. p * stride + len).  COV of the reference = sum of the 7 planes. */
typedef struct {
    int32_t  ref_id;
    uint32_t start;      /* first position of the tile on ref_id          */
    uint32_t len;        /* number of positions                           */
    uint32_t stride;     /* elements between planes                       */
    const uint32_t* counts;
    uint32_t n_samples;  /* counter sets in the tile: samples of the @RG table (depth.d:1170-1181), or 1 */
    uint32_t sample_stride; /* elements between the plane-0 starts of consecutive samples            */
} bdepth_tile;
enum { BDEPTH_PLANE_A = 0, BDEPTH_PLANE_C, BDEPTH_PLANE_G, BDEPTH_PLANE_T, BDEPTH_PLANE_N, BDEPTH_PLANE_DEL, BDEPTH_PLANE_REFSKIP, BDEPTH_N_PLANES };

typedef int (*bdepth_tile_cb)(void* user, const bdepth_tile* tile);

/* Per-window / per-region statistics = PerSampleRegionData (depth.d:609-635):
 * n_reads, n_bases and, for every -T threshold, the number of positions with coverage >= it. */
typedef struct {
    int32_t  ref_id;
    uint32_t start, end;
    uint32_t n_reads;
    uint32_t n_bases;
    const uint32_t* cov_ge;   /* n_thresholds entries */
    int32_t  sample_id;       /* regions outer, samples inner, as the reference prints them */
} bdepth_region_stat;
typedef int (*bdepth_stat_cb)(void* user, const bdepth_region_stat* stat, uint64_t index);

/* Counters and device timings of the last run (all times in milliseconds, CUDA events). */
typedef struct {
    uint64_t file_bytes;          /* compressed .bam bytes consumed (this shard)                    */
    uint64_t n_blocks;            /* BGZF data blocks inflated                                      */
    uint64_t cdata_bytes;         /* C: sum of raw deflate payload bytes                            */
    uint64_t inflated_bytes;      /* U: sum of ISIZE                                                */
    uint64_t n_records;           /* R: alignment records scanned                                   */
    uint64_t n_records_pass;      /* records passing filter with basesCovered() > 0                 */
    uint64_t n_cigar_ops;         /* K: sum of n_cigar over scanned records                         */
    uint64_t seq_bytes;           /* Q: sum of ceil(l_seq/2) over passing records                   */
    uint64_t positions;           /* T: positions of the counter tiles processed                    */
    uint64_t covered_positions;   /* positions with >=1 passing read (rows of default `depth base`) */
    uint64_t long_reads;          /* passing reads routed to the atomic scatter path                */
    uint64_t chain_fixups;        /* record-chain entry guesses corrected by verification           */
    uint32_t gpu_launches;        /* kernels launched by the library in the run                     */
    uint32_t n_batches;
    float ms_h2d, ms_inflate, ms_scan, ms_coverage, ms_reduce, ms_d2h, ms_total_device;
    double host_wall_ms;          /* wall clock of the whole call, host side                        */
    float ms_span_device;         /* CUDA-event time from the first to the last device operation    */
    float ms_exchange;            /* multi-GPU boundary exchange (NCCL)                             */
    uint64_t own_lo, own_hi;      /* linear-coordinate range this rank owns after the exchange      */
    uint64_t halo_bytes_sent;     /* boundary counters sent to the next ranks                       */
    uint64_t mate_pairs;          /* -m: overlapping pairs of one name fixed                        */
    uint64_t mate_pair_columns;   /* -m: (pair, column) decisions of selectBetterMate               */
    uint64_t mate_groups;         /* -m: names with three or more overlapping reads                 */
    float ms_mates;               /* -m: km_hash + km_link + km_fix (contained in ms_coverage)      */
    uint32_t n_sample_passes;     /* region / window runs: pipeline passes over groups of samples (1: every sample at once); 0 otherwise */
} bdepth_stats;

/* ------------------------------------------------------------------ lifecycle */
int  bdepth_device_count(void);
/* Open a BAM by path (mmap) -- also looks for <path>.bai / <path minus ext>.bai. */
int  bdepth_open(const char* bam_path, int device, bdepth_t** out);
/* The same, but the BGZF members of the file are framed only as far as the header needs.  A region query (regions set,
 * usable .bai) then touches nothing but the header and the members inside its BAI chunks, as the reference's
 * RandomAccessManager does (randomaccessmanager.d:316-338) -- bdepth_open reads the 18-byte header and the footer of every
 * member of the file up front, which for a cold multi-100-GB file is most of the cost of a small query.  Any run that
 * needs the whole file frames the rest when it starts (framing errors are then reported by that run). */
int  bdepth_open_lazy(const char* bam_path, int device, bdepth_t** out);
/* Open a BAM image held in host memory (pinned memory gives full-rate H2D).  bai may be NULL. */
int  bdepth_open_memory(const void* bam, size_t bam_len, const void* bai, size_t bai_len, int device, bdepth_t** out);
/* One more BAM whose reads are counted together with the handle's: new MultiBamReader(bam_filenames), depth.d:1162-1163,
 * BioD/bio/std/hts/bam/multireader.d:244-268 (nWayUnion of the files' sorted streams).  The file needs the handle's reference
 * dictionary; its @RG samples join the sample table (bdepth_n_samples / _sample_name afterwards).  bdepth_is_coordinate_sorted and
 * bdepth_has_index then answer for all files.  Not with -m, not on several ranks.  Call before the first run. */
int  bdepth_add_input(bdepth_t* h, const char* bam_path);
void bdepth_close(bdepth_t* h);
/* h == NULL returns the message of the last failed open on this thread. */
const char* bdepth_last_error(const bdepth_t* h);

/* ------------------------------------------------------------------ header */
int         bdepth_n_ref(const bdepth_t* h);
const char* bdepth_ref_name(const bdepth_t* h, int i);
uint32_t    bdepth_ref_length(const bdepth_t* h, int i);
const char* bdepth_header_text(const bdepth_t* h, size_t* len);
int         bdepth_is_coordinate_sorted(const bdepth_t* h);
int         bdepth_has_index(const bdepth_t* h);
int         bdepth_n_samples(const bdepth_t* h);                 /* >= 1; "*" when there is no @RG */
const char* bdepth_sample_name(const bdepth_t* h, int i);

/* ------------------------------------------------------------------ configuration */
/* keep a read iff mapq > mapq_gt && (flag & flag_reject_mask) == 0.
 * default (depth.d:1159): mapq_gt = 0, mask = 0x400 | 0x200.  -F "" : mapq_gt = -1, mask = 0. */
int bdepth_set_filter(bdepth_t* h, int mapq_gt, uint32_t flag_reject_mask);
/* -F / --filter (depth.d:1121, createFilterFromQuery filtering.d:40-51): a query in sambamba's filter language
 * (queryparser.d), compiled to a small postfix program that the record scan evaluates per read.  "" keeps every
 * read.  Supported: flag conditions, integer fields incl. avg_base_quality, [XX] tags against integers, strings and
 * null, read_name / strand / sequence / cigar string comparisons, ref_name / mate_ref_name == / !=, `=~ /regex/flags` on
 * read_name, sequence, cigar and string tags (patterns without back-references / look-around, at most 64 NFA states), and /
 * or / not / brackets.  BDEPTH_ERR_ARG (with the message) for syntax errors and for what is not supported: regular
 * expressions outside that subset or on reference names, ordering comparisons of reference names. */
int bdepth_set_filter_query(bdepth_t* h, const char* query);
int bdepth_set_min_baseq(bdepth_t* h, uint32_t min_base_quality);
/* -m / --fix-mate-overlaps (depth.d:1133; detectOverlappingMates :319-388, selectBetterMate :391-399, the -m branches
 * of writeColumn :521-530 and PerRegionPrinter.push :760-845): where two reads of one name (same sample) overlap,
 * every column counts only the better mate.  Available for bdepth_run_base / _run_base_text / _run_regions /
 * _run_windows / _run_resident; batches re-read the end of the previous batch and ranks a zone of their neighbours'
 * records, so that pairs cut by a batch or shard boundary are seen whole.  Names with three or more overlapping
 * reads (a chain of any length) follow the reference's none/detected/fixed/past state machine; more than eight reads
 * of one name over a single position are refused (BDEPTH_ERR_ARG). */
int bdepth_set_fix_mates(bdepth_t* h, int on);
/* --combined (depth.d:1131): one counter set for all samples.  Default: one per @RG sample.  bdepth_run_base / _run_base_text /
 * _run_resident hold every sample's counters at once: at most 64 samples (BDEPTH_ERR_ARG beyond).  bdepth_run_regions / _run_windows
 * take any number: see bdepth_set_samples_per_pass. */
int bdepth_set_combined(bdepth_t* h, int combined);
/* Region and window runs count the samples a group at a time when their counters do not fit at once: the pipeline runs once per group
 * of consecutive samples and each run adds the statistics of its group (a read counts in the pass of its sample only; every input is
 * read by the passes whose groups hold one of its @RG samples).  A group holds at most 64 samples, at most what the counter window
 * leaves room for in HBM and at most n; n = 0 (the default): as many as fit, up to 64.  Several ranks take the smallest group size of
 * any of them.  With -m every sample has to fit one pass (BDEPTH_ERR_ARG otherwise).  bdepth_stats.n_sample_passes tells how many
 * passes a run took. */
int bdepth_set_samples_per_pass(bdepth_t* h, uint32_t n);
/* Restrict runs to reads overlapping these regions (any order; merged internally).  n = 0 clears.  Regions that hold no position
 * (start >= end, or start behind the reference's end) are dropped; if none is left the restriction is cleared as with n = 0 -- a host that
 * wants "nothing" for such a query (the reference prints its header only) does not run at all, as the CLI does. */
int bdepth_set_regions(bdepth_t* h, const bdepth_region* regions, size_t n);
/* Multi-GPU: this process handles shard `rank` of `world` (BGZF virtual-offset ranges cut at BAI
 * linear-index record starts).  nccl_unique_id (128 bytes, identical on all ranks, from
 * bdepth_nccl_unique_id on rank 0) enables the boundary-counter exchange over NCCL; NULL with
 * world > 1 processes the shard without exchange (tiles then carry only this shard's reads). */
int bdepth_set_shard(bdepth_t* h, int rank, int world, const void* nccl_unique_id);
int bdepth_nccl_unique_id(void* out128);
/* Host-only (no GPU needed): the world-1 interior shard boundaries as BGZF virtual offsets, i.e.
 * the first linear-index record start at or after k * file_size / world (k = 1..world-1);
 * UINT64_MAX when there is none.  Used by the sharding tests. */
int bdepth_plan_shards(const char* bam_path, int world, uint64_t* out_voffsets);
/* Host-only (no GPU needed): the merged list of BGZF virtual-offset ranges [beg, end) a query for `regions`
 * has to read, computed from the BAI bins and linear index as getGroupChunks does
 * (BioD/bio/std/hts/bam/randomaccessmanager.d:247-294).  Writes up to `cap` (beg, end) pairs, returns the number
 * of ranges (or a negative error).  With regions set, the run entry points stage and inflate only these. */
long bdepth_plan_region_chunks(const char* bam_path, const bdepth_region* regions, size_t n, uint64_t* out_pairs, size_t cap);
/* Tuning knobs (0 = default): uncompressed bytes per batch (one inflate buffer in HBM); BGZF blocks per
 * host-to-device chunk, which is also the sub-batch whose scan / coverage / delivery overlaps the inflate of
 * the chunks that arrive after it. */
int bdepth_set_tuning(bdepth_t* h, uint64_t batch_inflated_bytes, uint64_t chunk_blocks);

/* ------------------------------------------------------------------ runs */
/* Stage the (shard of the) compressed file into HBM ahead of time; later runs then start with
 * inputs resident on the device (kernel-only timing).  Without it every run streams H2D itself. */
int bdepth_stage(bdepth_t* h);
/* Run the pipeline and leave the counters on the device (no tile delivery): kernel-only timing. */
int bdepth_run_resident(bdepth_t* h);
/* depth base: deliver every tile of the processed range in order.  cb may be NULL (benchmark). */
int bdepth_run_base(bdepth_t* h, bdepth_tile_cb cb, void* user);
/* depth window -w W --overlap O -T t...: stats for every window slot the reference would print
 * (all full windows of every reference, in order; depth.d:1051-1076), any O < W.  The reference's ring-slot
 * behaviour is reproduced in closed form (early threshold collection when W-O does not divide W, the
 * first-occurrence quirk of reference 0, the leftovers printed under the first trailing empty reference). */
int bdepth_run_windows(bdepth_t* h, uint32_t window, uint32_t overlap, const uint32_t* thresholds, size_t n_thresholds, bdepth_stat_cb cb, void* user);
/* depth region: stats for the given regions, delivered in the given order.
 * Both: one record per (segment, sample), segments outer, samples inner; with several sample passes
 * (bdepth_set_samples_per_pass) delivery starts when the last pass is done, in the same order. */
int bdepth_run_regions(bdepth_t* h, const bdepth_region* regions, size_t n, const uint32_t* thresholds, size_t n_thresholds, bdepth_stat_cb cb, void* user);

/* `depth base` with the row text produced on the GPU (SURVEY 8f rank 1): the rows PerBasePrinter would print
 * (depth.d:534-555, zero rows :452-487), delivered in order as text chunks: one row per position for one sample or
 * --combined, one row per sample and position otherwise (a sample whose COV is out of bounds ends the position, as
 * writeColumn's early return does). */
typedef struct { double min_cov, max_cov; int annotate; } bdepth_text_opts;
typedef int (*bdepth_text_cb)(void* user, const char* text, size_t len);
int bdepth_run_base_text(bdepth_t* h, const bdepth_text_opts* opts, bdepth_text_cb cb, void* user);

int bdepth_get_stats(const bdepth_t* h, bdepth_stats* out);
/* After a run: 1 if the reference has at least one read that produced a pileup column (the
 * condition under which depth.d:1225-1229 prints "Processing reference #k").  With regions set
 * only reads that overlap a region count: the reference's stream holds no others
 * (getReadsOverlapping, BioD/bio/std/hts/bam/randomaccessmanager.d:316-338). */
int bdepth_ref_has_reads(const bdepth_t* h, int ref);

/* ------------------------------------------------------------------ kernel-level entry points
 * (used by the parity tests and the roofline bench; same kernels as the runs above) */
/* Inflate the whole (shard of the) file on the GPU and copy the concatenated payload to dst. */
int64_t bdepth_inflate_to_host(bdepth_t* h, void* dst, uint64_t cap);
/* Build the BAI index of the opened BAM on the GPU -- what `sambamba index` writes: createIndex / IndexBuilder,
 * BioD/bio/std/hts/bam/bai/indexing.d:56-366 (bins with their chunks as the reference cuts them -- a chunk ends where the bin of
 * consecutive reads changes, chunks of one bin merge when they meet in one BGZF member --, the metadata pseudo-bin 37450, the linear
 * index with its gaps filled, n_no_coor).  K1 inflate and the K2 record scan as in every run, then one thread per record
 * (k_index_scan); the host assembles the per-bin lists from one entry per change of bin.  Bins are written in ascending order (the
 * reference: iteration order of a D associative array); a file that is not coordinate sorted is refused as there (:259-271).
 * Returns the size of the index in bytes (copied to dst when cap suffices; the first call builds, later calls only copy) or a negative
 * error.  The handle adopts the index: bdepth_has_index turns 1, and sharding, counter windows and region queries work on input
 * that came without a .bai (the reference refuses such input, depth.d:1166 -- the CLI still does unless --build-index is given). */
int64_t bdepth_build_index(bdepth_t* h, void* dst, uint64_t cap);
/* Scan records on the GPU; copy out up to cap rows of the columnar SoA (any pointer may be NULL). */
int64_t bdepth_scan_to_host(bdepth_t* h, uint64_t cap, int32_t* ref_id, int32_t* pos, uint32_t* span, uint16_t* flag, uint8_t* mapq, uint16_t* n_cigar, uint64_t* rec_off);

#ifdef __cplusplus
}
#endif
#endif /* BDEPTH_H */
