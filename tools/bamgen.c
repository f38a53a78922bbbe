/*
 * bamgen.c -- seeded synthetic coordinate-sorted BAM + BAI generator.
 *
 * Produces the benchmark inputs described in SURVEY.md 8(d) / BASELINE.md
 * (config 2: chr20-30x; configs 3-5: WGS-30x shaped) without any network or
 * third-party tool.  Output is a standard BGZF/BAM file: 0xFF00-byte payload
 * blocks (the reference writer's block size, BioD/bio/core/bgzf/constants.d:61),
 * zlib level 6 raw deflate, 28-byte EOF block, plus a standard .bai
 * (bins + 16 kb linear index), because `depth` insists on an index
 * (sambamba/depth.d:1166) and the multi-GPU sharder splits on linear-index
 * record starts.
 *
 * Deterministic for a given (seed, refs, n_reads) regardless of thread count:
 * every 4096-read chunk owns an RNG seeded from (seed, chunk index).
 *
 * usage: bamgen -o out.bam [-n reads] [-s seed] [-t threads] [-l level]
 *               [-r name:len]... | --preset chr20|wgs|tiny  [--stored-every K] [--pairs K]
 *               [--samples K | --sample NAME]
 *
 * --samples K: K read groups rgN / SM:SN (N = 1..K); every read's RG:Z is drawn from the seeded generator.
 * --sample NAME: the one read group is ID:NAME / SM:NAME (files of one cohort, one sample each).
 * Without either the file has the read group rg1 / S1, byte for byte as before these options existed.
 */
#define _GNU_SOURCE
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <math.h>
#include <pthread.h>
#include <zlib.h>

#define BLK 0xFF00u
#define CHUNK_READS 4096u
#define READ_LEN 150

static void die(const char *m) { fprintf(stderr, "bamgen: %s\n", m); exit(1); }

/* ---- rng: splitmix64 seeding xoshiro256** */
typedef struct { uint64_t s[4]; } Rng;
static uint64_t splitmix(uint64_t *x) { uint64_t z = (*x += 0x9E3779B97F4A7C15ULL); z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL; z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL; return z ^ (z >> 31); }
static void rng_seed(Rng *r, uint64_t a, uint64_t b) { uint64_t x = a * 0xD1342543DE82EF95ULL + b; for (int i = 0; i < 4; i++) r->s[i] = splitmix(&x); }
static inline uint64_t rotl(uint64_t x, int k) { return (x << k) | (x >> (64 - k)); }
static inline uint64_t rng_next(Rng *r) { uint64_t *s = r->s; uint64_t res = rotl(s[1] * 5, 7) * 9, t = s[1] << 17; s[2] ^= s[0]; s[3] ^= s[1]; s[1] ^= s[2]; s[0] ^= s[3]; s[2] ^= t; s[3] = rotl(s[3], 45); return res; }
static inline double rng_u(Rng *r) { return (double)(rng_next(r) >> 11) * (1.0 / 9007199254740992.0); }
static inline uint32_t rng_below(Rng *r, uint32_t n) { return (uint32_t)(((rng_next(r) >> 32) * (uint64_t)n) >> 32); }

/* ---- refs */
typedef struct { char name[64]; uint32_t len; uint64_t lin0; /* start in usable linear space */ uint64_t usable; } Ref;
static Ref *g_refs; static int g_nref;
static uint64_t g_G; /* total usable */

static const uint32_t GRCH38[24] = {248956422, 242193529, 198295559, 190214555, 181538259, 170805979, 159345973, 145138636, 138394717, 133797422, 135086622, 133275309, 114364328, 107043718, 101991189, 90338345, 83257441, 80373285, 58617616, 64444167, 46709983, 50818468, 156040895, 57227415};

static uint8_t g_qual_tab[1024];
static void init_qual_tab(void) {
    /* inverse CDF of N(30,8) clipped to [2,41], 1024 quantiles */
    for (int i = 0; i < 1024; i++) {
        double p = (i + 0.5) / 1024.0, lo = -8, hi = 8;
        for (int it = 0; it < 60; it++) { double m = 0.5 * (lo + hi); if (0.5 * erfc(-m / sqrt(2.0)) < p) lo = m; else hi = m; }
        double q = 30.0 + 8.0 * lo; if (q < 2) q = 2; if (q > 41) q = 41; g_qual_tab[i] = (uint8_t)lrint(q);
    }
}

static int reg2bin(int64_t beg, int64_t end) {
    --end;
    if (beg >> 14 == end >> 14) return (int)(((1 << 15) - 1) / 7 + (beg >> 14));
    if (beg >> 17 == end >> 17) return (int)(((1 << 12) - 1) / 7 + (beg >> 17));
    if (beg >> 20 == end >> 20) return (int)(((1 << 9) - 1) / 7 + (beg >> 20));
    if (beg >> 23 == end >> 23) return (int)(((1 << 6) - 1) / 7 + (beg >> 23));
    if (beg >> 26 == end >> 26) return (int)(((1 << 3) - 1) / 7 + (beg >> 26));
    return 0;
}

typedef struct { int32_t ref; int32_t beg, end; uint32_t bin; uint64_t u0, u1; } Meta;  /* u0/u1: global uncompressed offsets */

typedef struct {
    uint64_t first_read, n_reads, total_reads; uint64_t seed;
    uint8_t *buf; size_t len, cap; Meta *meta; size_t nmeta, capmeta;
} GenJob;

static inline void put32(uint8_t *p, uint32_t v) { p[0] = (uint8_t)v; p[1] = (uint8_t)(v >> 8); p[2] = (uint8_t)(v >> 16); p[3] = (uint8_t)(v >> 24); }

static uint64_t g_pairs = 0;
static uint32_t g_nsamp = 1; static const char *g_sample = NULL;
static void gen_read(GenJob *j, Rng *r, uint64_t idx) {
    /* stratified-uniform sorted position in usable linear space */
    double x = ((double)idx + rng_u(r)) / (double)j->total_reads * (double)g_G;
    uint64_t lx = (uint64_t)x; if (lx >= g_G) lx = g_G - 1;
    int ref = 0; { int lo = 0, hi = g_nref - 1; while (lo < hi) { int m = (lo + hi + 1) / 2; if (g_refs[m].lin0 <= lx) lo = m; else hi = m - 1; } ref = lo; }
    int32_t pos = (int32_t)(lx - g_refs[ref].lin0);
    uint32_t rlen = g_refs[ref].len;
    /* CIGAR */
    uint32_t cig[3]; int nc = 1; uint32_t span = READ_LEN; uint32_t u = rng_below(r, 100);
    if (u < 90) { cig[0] = (READ_LEN << 4) | 0; }
    else if (u < 94) { uint32_t b = 1 + rng_below(r, 10), a = 10 + rng_below(r, READ_LEN - 20 - b); cig[0] = (a << 4) | 0; cig[1] = (b << 4) | 1; cig[2] = ((READ_LEN - a - b) << 4) | 0; nc = 3; span = READ_LEN - b; }
    else if (u < 98) { uint32_t b = 1 + rng_below(r, 10), a = 10 + rng_below(r, READ_LEN - 20); cig[0] = (a << 4) | 0; cig[1] = (b << 4) | 2; cig[2] = ((READ_LEN - a) << 4) | 0; nc = 3; span = READ_LEN + b; }
    else if (u < 99) { uint32_t s = 1 + rng_below(r, 50); cig[0] = (s << 4) | 4; cig[1] = ((READ_LEN - s) << 4) | 0; nc = 2; span = READ_LEN - s; }
    else { uint32_t b = 100 + rng_below(r, 4901), a = 10 + rng_below(r, READ_LEN - 20); cig[0] = (a << 4) | 0; cig[1] = (b << 4) | 3; cig[2] = ((READ_LEN - a) << 4) | 0; nc = 3; span = READ_LEN + b; }
    if ((uint64_t)pos + span > rlen) { cig[0] = (READ_LEN << 4) | 0; nc = 1; span = READ_LEN; }
    /* flags / mapq */
    uint32_t flag = 0x1 | 0x2 | ((rng_next(r) & 1) ? 0x40 : 0x80) | ((rng_next(r) & 1) ? 0x10 : 0x20);
    uint32_t f = rng_below(r, 1000);
    if (f < 20) flag |= 0x400; else if (f < 25) flag |= 0x200; else if (f < 35) flag |= 0x100; else if (f < 40) flag |= 0x800;
    uint32_t mq, m = rng_below(r, 100); if (m < 93) mq = 60; else if (m < 98) mq = 0; else mq = 1 + rng_below(r, 59);
    int32_t mpos = pos + (int32_t)rng_below(r, 1001) - 500; if (mpos < 0) mpos = 0; if ((uint32_t)mpos >= rlen) mpos = (int32_t)rlen - 1;
    int32_t tlen = mpos >= pos ? mpos - pos + READ_LEN : -(pos - mpos + READ_LEN);
    /* record */
    /* --pairs K: read idx and read idx + K (about K read spacings further along) share a name, like overlapping mates */
    uint64_t name_id = g_pairs ? (idx / (2 * g_pairs)) * g_pairs + (idx % g_pairs) : idx;
    char name[16]; int l_name = snprintf(name, sizeof name, "r%09llu", (unsigned long long)name_id) + 1;
    char rg[80]; int l_rg = g_sample ? snprintf(rg, sizeof rg, "%s", g_sample) : snprintf(rg, sizeof rg, "rg%u", g_nsamp > 1 ? 1 + rng_below(r, g_nsamp) : 1u);
    size_t rec = 32 + (size_t)l_name + 4 * (size_t)nc + (READ_LEN + 1) / 2 + READ_LEN + (size_t)(4 + l_rg) + 4 + 4;
    if (j->len + 4 + rec > j->cap) { j->cap = (j->cap + 4 + rec) * 2; j->buf = realloc(j->buf, j->cap); if (!j->buf) die("oom"); }
    uint8_t *p = j->buf + j->len; size_t start = j->len;
    uint32_t bin = (uint32_t)reg2bin(pos, pos + (int64_t)span);
    put32(p, (uint32_t)rec); p += 4;
    put32(p, (uint32_t)ref); put32(p + 4, (uint32_t)pos); put32(p + 8, (bin << 16) | (mq << 8) | (uint32_t)l_name); put32(p + 12, (flag << 16) | (uint32_t)nc);
    put32(p + 16, READ_LEN); put32(p + 20, (uint32_t)ref); put32(p + 24, (uint32_t)mpos); put32(p + 28, (uint32_t)tlen); p += 32;
    memcpy(p, name, (size_t)l_name); p += l_name;
    for (int k = 0; k < nc; k++) { put32(p, cig[k]); p += 4; }
    /* bases: nibble codes 1,2,4,8 ; ~0.1% N (15) */
    static const uint8_t NT[4] = {1, 2, 4, 8};
    uint8_t bases[READ_LEN]; uint64_t bits = 0; int nb = 0;
    for (int k = 0; k < READ_LEN; k++) { if (!nb) { bits = rng_next(r); nb = 32; } bases[k] = NT[bits & 3]; bits >>= 2; nb--; }
    { double un = rng_u(r); int nn = un < 0.8607 ? 0 : un < 0.9899 ? 1 : un < 0.99947 ? 2 : 3; for (int k = 0; k < nn; k++) bases[rng_below(r, READ_LEN)] = 15; }
    for (int k = 0; k < READ_LEN; k += 2) *p++ = (uint8_t)((bases[k] << 4) | (k + 1 < READ_LEN ? bases[k + 1] : 0));
    for (int k = 0; k < READ_LEN; ) { uint64_t q = rng_next(r); for (int t = 0; t < 6 && k < READ_LEN; t++, k++) { *p++ = g_qual_tab[q & 1023]; q >>= 10; } }
    p[0] = 'R'; p[1] = 'G'; p[2] = 'Z'; memcpy(p + 3, rg, (size_t)l_rg + 1); p += 4 + l_rg;
    p[0] = 'N'; p[1] = 'M'; p[2] = 'C'; p[3] = (uint8_t)rng_below(r, 6); p += 4;
    p[0] = 'A'; p[1] = 'S'; p[2] = 'C'; p[3] = (uint8_t)(100 + rng_below(r, 51)); p += 4;
    j->len = (size_t)(p - j->buf);
    if (j->len - start != 4 + rec) die("internal: record size mismatch");
    if (j->nmeta == j->capmeta) { j->capmeta = j->capmeta ? j->capmeta * 2 : 4096; j->meta = realloc(j->meta, j->capmeta * sizeof(Meta)); }
    Meta mt = { ref, pos, pos + (int32_t)span, bin, start, j->len }; j->meta[j->nmeta++] = mt;
}

static void *gen_worker(void *arg) {
    GenJob *j = arg; j->len = 0; j->nmeta = 0;
    for (uint64_t i = 0; i < j->n_reads; ) {
        uint64_t idx = j->first_read + i, chunk = idx / CHUNK_READS;
        Rng r; rng_seed(&r, j->seed, chunk);
        uint64_t chunk_end = (chunk + 1) * CHUNK_READS, stop = j->first_read + j->n_reads; if (chunk_end < stop) stop = chunk_end;
        /* first_read is always chunk aligned, so the RNG stream of a chunk is consumed identically for any thread count */
        for (; idx < stop; idx++, i++) gen_read(j, &r, idx);
    }
    return NULL;
}

/* ---- compression */
typedef struct { const uint8_t *src; size_t n_blocks; size_t first; int nthreads, tid, level; uint32_t last_len; uint8_t *dst /* n_blocks * 65536 */; uint32_t *dlen; int stored_every; uint64_t blk_index0; } CompJob;

static uint32_t compress_block(const uint8_t *src, uint32_t n, uint8_t *dst, int level) {
    z_stream zs; memset(&zs, 0, sizeof zs);
    if (deflateInit2(&zs, level, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) die("deflateInit2");
    zs.next_in = (Bytef *)src; zs.avail_in = n; zs.next_out = dst + 18; zs.avail_out = 65536 - 18 - 8;
    int rc = deflate(&zs, Z_FINISH);
    if (rc != Z_STREAM_END) {   /* incompressible: fall back to stored */
        deflateEnd(&zs); memset(&zs, 0, sizeof zs);
        deflateInit2(&zs, 0, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY);
        zs.next_in = (Bytef *)src; zs.avail_in = n; zs.next_out = dst + 18; zs.avail_out = 65536 - 18 - 8;
        if (deflate(&zs, Z_FINISH) != Z_STREAM_END) die("deflate stored failed");
    }
    uint32_t clen = (uint32_t)zs.total_out; deflateEnd(&zs);
    static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    memcpy(dst, hdr, 16);
    uint32_t total = 18 + clen + 8; dst[16] = (uint8_t)((total - 1) & 0xFF); dst[17] = (uint8_t)((total - 1) >> 8);
    uint32_t crc = (uint32_t)crc32(crc32(0, NULL, 0), src, n);
    put32(dst + 18 + clen, crc); put32(dst + 22 + clen, n);
    return total;
}
static void *comp_worker(void *arg) {
    CompJob *c = arg;
    for (size_t b = c->tid; b < c->n_blocks; b += c->nthreads) {
        uint32_t n = (b + 1 == c->n_blocks) ? c->last_len : BLK;
        int lvl = c->level;
        if (c->stored_every > 0 && ((c->blk_index0 + b) % (uint64_t)c->stored_every) == (uint64_t)c->stored_every - 1) lvl = 0;
        if (c->stored_every > 0 && ((c->blk_index0 + b) % (uint64_t)c->stored_every) == 0 && c->stored_every > 2) lvl = -2; /* marker: fixed huffman */
        if (lvl == -2) {
            /* Z_FIXED strategy forces fixed-Huffman (btype 1) blocks */
            uint8_t *dst = c->dst + b * 65536; z_stream zs; memset(&zs, 0, sizeof zs);
            deflateInit2(&zs, 6, Z_DEFLATED, -15, 8, Z_FIXED);
            zs.next_in = (Bytef *)(c->src + b * (size_t)BLK); zs.avail_in = n; zs.next_out = dst + 18; zs.avail_out = 65536 - 26;
            if (deflate(&zs, Z_FINISH) == Z_STREAM_END) {
                uint32_t clen = (uint32_t)zs.total_out; deflateEnd(&zs);
                static const uint8_t hdr[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
                memcpy(dst, hdr, 16); uint32_t total = 18 + clen + 8; dst[16] = (uint8_t)((total - 1) & 0xFF); dst[17] = (uint8_t)((total - 1) >> 8);
                put32(dst + 18 + clen, (uint32_t)crc32(crc32(0, NULL, 0), c->src + b * (size_t)BLK, n)); put32(dst + 22 + clen, n);
                c->dlen[b] = total; continue;
            }
            deflateEnd(&zs); lvl = c->level;
        }
        c->dlen[b] = compress_block(c->src + b * (size_t)BLK, n, c->dst + b * 65536, lvl);
    }
    return NULL;
}

/* ---- BAI accumulation */
typedef struct { uint64_t beg, end; } Chunk;
typedef struct { Chunk *c; uint32_t n, cap; } BinV;
typedef struct { BinV *bins; /* 37450 */ uint64_t *lin; uint32_t nlin, caplin; int used; uint64_t off_beg, off_end, n_mapped; } RefIdx;
static RefIdx *g_idx; static int32_t g_last_ref = -1; static uint32_t g_last_bin = 0xFFFFFFFFu; static uint64_t g_chunk_beg;

static void idx_close_chunk(uint64_t end_vo) {
    if (g_last_ref < 0 || g_last_bin == 0xFFFFFFFFu) return;
    RefIdx *ri = &g_idx[g_last_ref]; BinV *bv = &ri->bins[g_last_bin];
    if (bv->n == bv->cap) { bv->cap = bv->cap ? bv->cap * 2 : 2; bv->c = realloc(bv->c, bv->cap * sizeof(Chunk)); }
    bv->c[bv->n].beg = g_chunk_beg; bv->c[bv->n].end = end_vo; bv->n++;
}
static void idx_add(const Meta *m, uint64_t vo0, uint64_t vo1) {
    RefIdx *ri = &g_idx[m->ref];
    if (!ri->bins) { ri->bins = calloc(37450, sizeof(BinV)); ri->used = 1; ri->off_beg = vo0; }
    if (m->ref != g_last_ref || m->bin != g_last_bin) { idx_close_chunk(vo0); g_last_ref = m->ref; g_last_bin = m->bin; g_chunk_beg = vo0; }
    ri->off_end = vo1; ri->n_mapped++;
    uint32_t w0 = (uint32_t)m->beg >> 14, w1 = (uint32_t)(m->end - 1) >> 14;
    if (w1 + 1 > ri->caplin) { uint32_t nc = ri->caplin ? ri->caplin : 64; while (nc < w1 + 1) nc *= 2; ri->lin = realloc(ri->lin, nc * sizeof(uint64_t)); memset(ri->lin + ri->caplin, 0, (nc - ri->caplin) * sizeof(uint64_t)); ri->caplin = nc; }
    for (uint32_t w = w0; w <= w1; w++) if (ri->lin[w] == 0) ri->lin[w] = vo0;
    if (w1 + 1 > ri->nlin) ri->nlin = w1 + 1;
}
static void write_bai(const char *path, uint64_t last_vo) {
    idx_close_chunk(last_vo);
    FILE *f = fopen(path, "wb"); if (!f) die("cannot write .bai");
    uint8_t b4[4], b8[8];
#define W32(v) do { put32(b4, (uint32_t)(v)); fwrite(b4, 1, 4, f); } while (0)
#define W64(v) do { put32(b8, (uint32_t)(v)); put32(b8 + 4, (uint32_t)((uint64_t)(v) >> 32)); fwrite(b8, 1, 8, f); } while (0)
    fwrite("BAI\1", 1, 4, f); W32(g_nref);
    for (int r = 0; r < g_nref; r++) {
        RefIdx *ri = &g_idx[r];
        if (!ri->used) { W32(0); W32(0); continue; }
        uint32_t nb = 0; for (int b = 0; b < 37450; b++) if (ri->bins[b].n) nb++;
        W32(nb + 1);
        for (int b = 0; b < 37450; b++) if (ri->bins[b].n) { W32(b); W32(ri->bins[b].n); for (uint32_t k = 0; k < ri->bins[b].n; k++) { W64(ri->bins[b].c[k].beg); W64(ri->bins[b].c[k].end); } }
        W32(37450); W32(2); W64(ri->off_beg); W64(ri->off_end); W64(ri->n_mapped); W64(0);   /* samtools-style metadata pseudo-bin */
        /* linear index: fill empty windows with the previous value, as samtools does */
        for (uint32_t w = 1; w < ri->nlin; w++) if (ri->lin[w] == 0) ri->lin[w] = ri->lin[w - 1];
        W32(ri->nlin); for (uint32_t w = 0; w < ri->nlin; w++) W64(ri->lin[w]);
    }
    W64(0);
    fclose(f);
}

int main(int argc, char **argv) {
    const char *out = NULL; uint64_t n_reads = 0, seed = 20; int nthreads = 8, level = 6, stored_every = 0; const char *preset = NULL;
    Ref *refs = NULL; int nref = 0;
    for (int i = 1; i < argc; i++) {
        if (!strcmp(argv[i], "-o") && i + 1 < argc) out = argv[++i];
        else if (!strcmp(argv[i], "-n") && i + 1 < argc) n_reads = strtoull(argv[++i], NULL, 10);
        else if (!strcmp(argv[i], "-s") && i + 1 < argc) seed = strtoull(argv[++i], NULL, 10);
        else if (!strcmp(argv[i], "-t") && i + 1 < argc) nthreads = atoi(argv[++i]);
        else if (!strcmp(argv[i], "-l") && i + 1 < argc) level = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--stored-every") && i + 1 < argc) stored_every = atoi(argv[++i]);
        else if (!strcmp(argv[i], "--pairs") && i + 1 < argc) g_pairs = strtoull(argv[++i], NULL, 10);
        else if (!strcmp(argv[i], "--preset") && i + 1 < argc) preset = argv[++i];
        else if (!strcmp(argv[i], "--samples") && i + 1 < argc) { g_nsamp = (uint32_t)strtoul(argv[++i], NULL, 10); if (g_nsamp < 1 || g_nsamp > 65534) die("--samples: 1 .. 65534"); }
        else if (!strcmp(argv[i], "--sample") && i + 1 < argc) { g_sample = argv[++i]; if (!*g_sample || strlen(g_sample) > 64 || strpbrk(g_sample, "\t\n")) die("--sample: a name of 1 .. 64 characters without tabs"); }
        else if (!strcmp(argv[i], "-r") && i + 1 < argc) { char *s = argv[++i], *c = strrchr(s, ':'); if (!c) die("bad -r name:len"); refs = realloc(refs, (nref + 1) * sizeof(Ref)); memset(&refs[nref], 0, sizeof(Ref)); snprintf(refs[nref].name, 64, "%.*s", (int)(c - s), s); refs[nref].len = (uint32_t)strtoul(c + 1, NULL, 10); nref++; }
        else die("usage: bamgen -o out.bam [-n reads] [-s seed] [-t threads] [-l level] [-r name:len]... [--preset chr20|wgs|tiny] [--stored-every K] [--pairs K] [--samples K | --sample NAME]");
    }
    if (g_sample && g_nsamp > 1) die("--sample names the one read group of a file: not with --samples");
    if (!out) die("-o required");
    if (preset && !strcmp(preset, "chr20")) { refs = calloc(1, sizeof(Ref)); strcpy(refs[0].name, "chr20"); refs[0].len = 64444167; nref = 1; if (!n_reads) n_reads = 12888833; }
    else if (preset && !strcmp(preset, "wgs")) { refs = calloc(24, sizeof(Ref)); for (int i = 0; i < 24; i++) { if (i < 22) snprintf(refs[i].name, 64, "chr%d", i + 1); else strcpy(refs[i].name, i == 22 ? "chrX" : "chrY"); refs[i].len = GRCH38[i]; } nref = 24; if (!n_reads) n_reads = 620000000ULL; }
    else if (preset && !strcmp(preset, "tiny")) { refs = calloc(3, sizeof(Ref)); strcpy(refs[0].name, "ctgA"); refs[0].len = 30000; strcpy(refs[1].name, "ctgB"); refs[1].len = 1000; strcpy(refs[2].name, "ctgC"); refs[2].len = 52000; nref = 3; if (!n_reads) n_reads = 5000; }
    if (!nref) die("no references (-r or --preset)");
    if (!n_reads) die("-n required");
    g_refs = refs; g_nref = nref; g_G = 0;
    for (int i = 0; i < nref; i++) { refs[i].lin0 = g_G; refs[i].usable = refs[i].len > 400 ? refs[i].len - 200 : 0; g_G += refs[i].usable; }
    /* refs with usable==0 get no reads: make lookup skip them by giving them zero width (binary search lands on the last ref with lin0 <= x) */
    if (!g_G) die("references too short");
    init_qual_tab();
    g_idx = calloc(nref, sizeof(RefIdx));

    FILE *fo = fopen(out, "wb"); if (!fo) die("cannot open output");
    /* header bytes */
    size_t hcap = 1 << 16, hl = 0; char *text = malloc(hcap);
    hl += snprintf(text + hl, hcap - hl, "@HD\tVN:1.6\tSO:coordinate\n");
    for (int i = 0; i < nref; i++) { if (hcap - hl < 256) { hcap *= 2; text = realloc(text, hcap); } hl += snprintf(text + hl, hcap - hl, "@SQ\tSN:%s\tLN:%u\n", refs[i].name, refs[i].len); }
    for (uint32_t k = 1; k <= g_nsamp; k++) {
        if (hcap - hl < 256) { hcap *= 2; text = realloc(text, hcap); }
        if (g_sample) hl += snprintf(text + hl, hcap - hl, "@RG\tID:%s\tSM:%s\tPL:ILLUMINA\n", g_sample, g_sample);
        else hl += snprintf(text + hl, hcap - hl, "@RG\tID:rg%u\tSM:S%u\tPL:ILLUMINA\n", k, k);
    }
    if (hcap - hl < 256) { hcap *= 2; text = realloc(text, hcap); }
    hl += snprintf(text + hl, hcap - hl, "@PG\tID:bamgen\tPN:bamgen\tCL:seed=%llu\n", (unsigned long long)seed);
    size_t hdr_len = 12 + hl; for (int i = 0; i < nref; i++) hdr_len += 8 + strlen(refs[i].name) + 1;
    uint8_t *hdr = malloc(hdr_len), *p = hdr;
    memcpy(p, "BAM\1", 4); put32(p + 4, (uint32_t)hl); memcpy(p + 8, text, hl); p += 8 + hl; put32(p, (uint32_t)nref); p += 4;
    for (int i = 0; i < nref; i++) { uint32_t ln = (uint32_t)strlen(refs[i].name) + 1; put32(p, ln); memcpy(p + 4, refs[i].name, ln); put32(p + 4 + ln, refs[i].len); p += 8 + ln; }

    /* stream state */
    size_t batch_reads = (size_t)CHUNK_READS * 64 * (size_t)nthreads; if (batch_reads > (1u << 21)) batch_reads = (1u << 21) / CHUNK_READS * CHUNK_READS;
    GenJob *jobs = calloc(nthreads, sizeof(GenJob)); pthread_t *th = calloc(nthreads, sizeof(pthread_t));
    uint8_t *stream = NULL; size_t scap = 0, slen = 0;           /* pending uncompressed bytes (carry + batch) */
    uint64_t stream_u0 = 0;                                      /* global u offset of stream[0] (always a multiple of BLK) */
    uint64_t *coff = NULL; size_t ncoff = 0, capcoff = 0;        /* compressed offset per block */
    uint64_t cpos = 0;
    Meta *pend = NULL; size_t npend = 0, cappend = 0, pend_head = 0;
    uint8_t *cbuf = NULL; uint32_t *clen = NULL; size_t cblocks_cap = 0;
    /* header goes first into the stream */
    scap = hdr_len + 1024; stream = malloc(scap); memcpy(stream, hdr, hdr_len); slen = hdr_len;
    uint64_t total_u = hdr_len;
    uint64_t done = 0; int final = 0;
    while (!final) {
        uint64_t nb = n_reads - done; if (nb > batch_reads) nb = batch_reads;
        /* split on chunk boundaries */
        uint64_t chunks = (nb + CHUNK_READS - 1) / CHUNK_READS, c0 = 0;
        for (int t = 0; t < nthreads; t++) {
            uint64_t c1 = chunks * (uint64_t)(t + 1) / (uint64_t)nthreads;
            jobs[t].first_read = done + c0 * CHUNK_READS; uint64_t e = done + c1 * CHUNK_READS; if (e > done + nb) e = done + nb;
            jobs[t].n_reads = e > jobs[t].first_read ? e - jobs[t].first_read : 0; jobs[t].total_reads = n_reads; jobs[t].seed = seed; c0 = c1;
            pthread_create(&th[t], NULL, gen_worker, &jobs[t]);
        }
        for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
        for (int t = 0; t < nthreads; t++) {
            if (slen + jobs[t].len > scap) { scap = (slen + jobs[t].len) * 3 / 2; stream = realloc(stream, scap); if (!stream) die("oom"); }
            memcpy(stream + slen, jobs[t].buf, jobs[t].len);
            for (size_t k = 0; k < jobs[t].nmeta; k++) { Meta m = jobs[t].meta[k]; m.u0 += total_u; m.u1 += total_u; if (npend == cappend) { cappend = cappend ? cappend * 2 : 1 << 16; pend = realloc(pend, cappend * sizeof(Meta)); } pend[npend++] = m; }
            slen += jobs[t].len; total_u += jobs[t].len;
        }
        done += nb; final = done >= n_reads;
        size_t nblk = final ? (slen + BLK - 1) / BLK : slen / BLK;
        if (nblk) {
            if (nblk > cblocks_cap) { cblocks_cap = nblk; cbuf = realloc(cbuf, nblk * 65536); clen = realloc(clen, nblk * sizeof(uint32_t)); if (!cbuf) die("oom"); }
            uint32_t last_len = final ? (uint32_t)(slen - (nblk - 1) * (size_t)BLK) : BLK;
            CompJob *cj = calloc(nthreads, sizeof(CompJob));
            for (int t = 0; t < nthreads; t++) { cj[t] = (CompJob){ stream, nblk, 0, nthreads, t, level, last_len, cbuf, clen, stored_every, ncoff }; pthread_create(&th[t], NULL, comp_worker, &cj[t]); }
            for (int t = 0; t < nthreads; t++) pthread_join(th[t], NULL);
            free(cj);
            for (size_t b = 0; b < nblk; b++) {
                if (ncoff == capcoff) { capcoff = capcoff ? capcoff * 2 : 1 << 16; coff = realloc(coff, capcoff * sizeof(uint64_t)); }
                coff[ncoff++] = cpos; if (fwrite(cbuf + b * 65536, 1, clen[b], fo) != clen[b]) die("write error"); cpos += clen[b];
            }
            size_t used = final ? slen : nblk * (size_t)BLK;
            memmove(stream, stream + used, slen - used); slen -= used; stream_u0 += used;
        }
        /* index records whose end voffset is known (end block written, or end == stream end at final) */
        uint64_t written_u = stream_u0;
        while (pend_head < npend) {
            Meta *m = &pend[pend_head];
            uint64_t b1 = m->u1 / BLK;
            if (!(b1 < ncoff || (final && m->u1 == total_u))) break;
            uint64_t vo0 = (coff[m->u0 / BLK] << 16) | (m->u0 % BLK);
            uint64_t vo1 = (b1 < ncoff) ? ((coff[b1] << 16) | (m->u1 % BLK)) : (cpos << 16);
            idx_add(m, vo0, vo1); pend_head++;
        }
        (void)written_u;
        if (pend_head > (1u << 20)) { memmove(pend, pend + pend_head, (npend - pend_head) * sizeof(Meta)); npend -= pend_head; pend_head = 0; }
    }
    static const uint8_t eof_blk[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    fwrite(eof_blk, 1, 28, fo); fclose(fo);
    char bai[4096]; snprintf(bai, sizeof bai, "%s.bai", out); write_bai(bai, cpos << 16);
    fprintf(stderr, "bamgen: %llu reads, %zu blocks, %llu uncompressed bytes, %llu compressed bytes\n", (unsigned long long)n_reads, ncoff, (unsigned long long)total_u, (unsigned long long)(cpos + 28));
    return 0;
}
