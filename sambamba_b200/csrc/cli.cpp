// cli.cpp -- `sambamba depth`-compatible host on top of libbdepth.so.
//
// Mirrors depth_main (sambamba/depth.d:1079-1245): same positional grammar (mode, then BAMs), same
// options (depth.d:1121-1143, :413-415, :712-714, :1015-1018), same stdout text, same stderr lines
// ("Processing reference #k (name)", "sambamba-depth: <msg>"), same exit codes (0 on usage, 1 on
// error).  The reference's host language is D, which this image cannot compile (SURVEY F1); the
// D binding that would replace this file is in sambamba_b200/d/bdepth.d and INTEGRATION.md.
//
// Not supported through the GPU path yet (rejected with a message, never silently wrong):
//   -F with back-references / look-around in regular expressions ; several BAM files together with -m ; `depth base` with more than 64
//   samples without --combined ; -m in a region / window run whose samples take several passes (more than 64 samples).
// Region and window modes take any number of samples: the library counts them a group at a time.
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/bdepth.h"

static void usage() {
    static const char* L[] = {
        "Usage: sambamba-depth region|window|base [options] input.bam  [input2.bam [...]]", "",
        "          All BAM files must be coordinate-sorted and indexed.", "",
        "          The tool has three modes: base, region, and window,",
        "          each name means per which unit to print the statistics.", "",
        "Common options:", "         -F, --filter=FILTER",
        "                    set custom filter for alignments; the default value is",
        "                    'mapping_quality > 0 and not duplicate and not failed_quality_control'",
        "         -o, --output-file=FILENAME", "                    output filename (by default /dev/stdout)",
        "         -t, --nthreads=NTHREADS", "                    maximum number of threads to use",
        "         -c, --min-coverage=MINCOVERAGE",
        "                    minimum mean coverage for output (default: 0 for region/window, 1 for base)",
        "         -C, --max-coverage=MAXCOVERAGE", "                    maximum mean coverage for output",
        "         -q, --min-base-quality=QUAL", "                    don't count bases with lower base quality",
        "         --combined", "                    output combined statistics for all samples",
        "         -a, --annotate", "                    add additional column of y/n instead of",
        "                    skipping records not satisfying the criteria",
        "         -m, --fix-mate-overlaps", "                    detect overlaps of mate reads and handle them on per-base basis",
        "base subcommand options:", "         -L, --regions=FILENAME|REGION",
        "                    list or regions of interest or a single region in form chr:beg-end (optional)",
        "         -z, --report-zero-coverage (DEPRECATED, use --min-coverage=0 instead)",
        "                    don't skip zero coverage bases", "region subcommand options:",
        "         -L, --regions=FILENAME|REGION",
        "                    list or regions of interest or a single region in form chr:beg-end (required)",
        "         -T, --cov-threshold=COVTHRESHOLD", "                    multiple thresholds can be provided,",
        "                    for each one an extra column will be added,", "                    the percentage of bases in the region",
        "                    where coverage is more than this value", "window subcommand options:",
        "         -w, --window-size=WINDOWSIZE", "                    breadth of the window, in bp (required)",
        "         --overlap=OVERLAP", "                    overlap of successive windows, in bp (default is 0)",
        "         -T, --cov-threshold=COVTHRESHOLD", "                    same meaning as in 'region' subcommand"};
    for (const char* l : L) fprintf(stderr, "%s\n", l);
}

struct Args { std::vector<std::string> v; };
// std.getopt-like extraction (caseSensitive, passThrough, no bundling): "-x VAL", "-xVAL", "-x=VAL", "--long VAL", "--long=VAL"
static int opt_take(Args& a, const char* lng, char sht, bool has_val, std::vector<std::string>* vals) {
    int found = 0;
    for (size_t i = 1; i < a.v.size();) {
        const std::string& s = a.v[i]; size_t consumed = 0; std::string v;
        if (s == "--") break;
        if (s.size() > 2 && s[0] == '-' && s[1] == '-' && lng) {
            size_t ln = strlen(lng);
            if (!s.compare(2, ln, lng) && (s.size() == 2 + ln || s[2 + ln] == '=')) {
                if (!has_val) { if (s.size() == 2 + ln) consumed = 1; }
                else if (s.size() > 2 + ln) { v = s.substr(3 + ln); consumed = 1; }
                else if (i + 1 < a.v.size()) { v = a.v[i + 1]; consumed = 2; }
                else return -1;
            }
        } else if (s.size() >= 2 && s[0] == '-' && s[1] != '-' && sht && s[1] == sht) {
            if (!has_val) { if (s.size() == 2) consumed = 1; }
            else if (s.size() > 2 && s[2] == '=') { v = s.substr(3); consumed = 1; }
            else if (s.size() > 2) { v = s.substr(2); consumed = 1; }
            else if (i + 1 < a.v.size()) { v = a.v[i + 1]; consumed = 2; }
            else return -1;
        }
        if (consumed) { found++; if (has_val && vals) vals->push_back(v); a.v.erase(a.v.begin() + i, a.v.begin() + i + consumed); }
        else i++;
    }
    return found;
}

struct Out {
    FILE* f = nullptr; std::vector<char> buf; size_t n = 0;
    Out() { buf.resize(4 << 20); }
    void flush() { if (n) fwrite(buf.data(), 1, n, f); n = 0; }
    inline void room(size_t k) { if (n + k > buf.size()) flush(); }
    inline void str(const char* s, size_t l) { room(l); memcpy(&buf[n], s, l); n += l; }
    inline void lit(const char* s) { str(s, strlen(s)); }
    inline void ch(char c) { room(1); buf[n++] = c; }
    inline void u64(uint64_t v) { room(24); char t[24]; int k = 0; do { t[k++] = (char)('0' + v % 10); v /= 10; } while (v); while (k) buf[n++] = t[--k]; }
    void g(float v) { room(48); n += (size_t)snprintf(&buf[n], 48, "%g", (double)v); }   // D write(float) == %g
};

static bool is_white(char c) { return c == ' ' || c == '\t' || c == '\r' || c == '\n' || c == '\v' || c == '\f'; }

struct BedIv { std::string chr; long beg, end; };
// sambamba/utils/common/bed.d:59-97.  returns false if the file cannot be read / parsed (caller falls back to parseRegion)
static bool bed_read(const std::string& path, std::vector<BedIv>& ivs, std::vector<std::string>& lines) {
    FILE* f = fopen(path.c_str(), "rb"); if (!f) return false;
    std::string txt; char b[65536]; size_t k; while ((k = fread(b, 1, sizeof b, f)) > 0) txt.append(b, k); fclose(f);
    size_t p = 0;
    while (p <= txt.size()) {
        size_t e = txt.find('\n', p); if (e == std::string::npos) e = txt.size();
        std::vector<std::string> fs; size_t q = p;
        while (q < e) { while (q < e && is_white(txt[q])) q++; if (q >= e) break; size_t s = q; while (q < e && !is_white(txt[q])) q++; fs.push_back(txt.substr(s, q - s)); }
        if (fs.size() >= 2) {
            long v[2] = {0, 0};
            for (size_t j = 1; j < std::min<size_t>(fs.size(), 3); j++) { char* endp; v[j - 1] = strtol(fs[j].c_str(), &endp, 10); if (*endp || endp == fs[j].c_str()) return false; }
            long beg = v[0], end = fs.size() >= 3 ? v[1] : v[0] + 1;
            if (beg == end) end = beg + 1;
            if (beg < end) ivs.push_back({fs[0], beg, end});
            lines.push_back(txt.substr(p, e - p));
        }
        p = e + 1;
    }
    return true;
}
// BioD/bio/core/region.d (region.rl:29-35): ref[:beg[-end]] with ',' separators, 1-based closed -> 0-based half-open
static void parse_region_string(const std::string& s, std::string& ref, uint32_t& beg, uint32_t& end) {
    beg = 0; end = UINT32_MAX; size_t c = std::string::npos;
    for (size_t t = 0; t < s.size(); t++) if (s[t] == ':') {
        size_t q = t + 1; bool ok = q < s.size() && isdigit((unsigned char)s[q]);
        while (q < s.size() && (isdigit((unsigned char)s[q]) || s[q] == ',')) q++;
        if (ok && q < s.size() && s[q] == '-') { q++; if (!(q < s.size() && isdigit((unsigned char)s[q]))) ok = false; while (q < s.size() && (isdigit((unsigned char)s[q]) || s[q] == ',')) q++; }
        if (ok && q == s.size()) { c = t; break; }
    }
    if (c == std::string::npos) { ref = s; return; }
    ref = s.substr(0, c); long v = 0; size_t q = c + 1;
    while (q < s.size() && s[q] != '-') { if (s[q] != ',') v = v * 10 + (s[q] - '0'); q++; }
    beg = (uint32_t)(v - 1);
    if (q < s.size() && s[q] == '-') { q++; v = 0; while (q < s.size()) { if (s[q] != ',') v = v * 10 + (s[q] - '0'); q++; } end = (uint32_t)v; }
}

struct Ctx {
    bdepth_t* h = nullptr; Out out; int mode = 0;
    double min_cov = 0, max_cov = 1e50; bool combined = false, annotate = false;
    std::vector<std::string> ref_names; std::vector<std::string> samples;
    std::vector<uint32_t> thr;
    // region mode
    std::vector<std::string> raw_lines; bool window_mode = false;
    int last_ref_announced = -2;
};

// std.getopt hands the option text to std.conv.to!T, whose exceptions end depth_main with "sambamba-depth: <message>" and exit code 1
// (depth.d:1236-1243): a value that is no number of the option's type is an error, not a zero.
static bool conv_unsigned(const std::string& s, unsigned long long maxv, const char* type, unsigned long long& out, std::string& err) {
    if (s.empty()) { err = std::string("Unexpected end of input when converting from type string to type ") + type; return false; }
    unsigned long long v = 0;
    for (char ch : s) {
        if (ch < '0' || ch > '9') { err = std::string("Unexpected '") + ch + "' when converting from type string to type " + type; return false; }
        if (v > (maxv - (unsigned)(ch - '0')) / 10) { err = "Conversion positive overflow"; return false; }      // (maxv < 2^64 - 9 for every caller)
        v = v * 10 + (unsigned)(ch - '0');
    }
    out = v; return true;
}
static bool conv_double(const std::string& s, double& out, std::string& err) {
    if (s.empty()) { err = "Unexpected end of input when converting from type string to type double"; return false; }
    char* end = nullptr; double v = strtod(s.c_str(), &end);
    if (end == s.c_str() || *end || s[0] == ' ' || s[0] == '\t') { err = "no digits seen"; return false; }
    out = v; return true;
}

static int base_tile_cb(void* user, const bdepth_tile* t) {
    Ctx& c = *(Ctx*)user; Out& o = c.out;
    const std::string& name = c.ref_names[t->ref_id];
    const uint32_t S = t->n_samples;
    for (uint32_t i = 0; i < t->len; i++) {
        // does any sample have a column here?  (min_cov > 0: positions without any read print nothing, depth.d:568-572)
        uint64_t any = 0;
        for (uint32_t si = 0; si < S; si++) for (int p = 0; p < 7; p++) any |= t->counts[(size_t)si * t->sample_stride + (size_t)p * t->stride + i];
        if (!any && c.min_cov > 0) continue;
        for (uint32_t si = 0; si < S; si++) {
            const uint32_t* P = t->counts + (size_t)si * t->sample_stride + i;
            uint64_t a = P[0], cc = P[t->stride], g = P[2 * (size_t)t->stride], tt = P[3 * (size_t)t->stride], n = P[4 * (size_t)t->stride], d = P[5 * (size_t)t->stride], s = P[6 * (size_t)t->stride];
            uint64_t total = a + cc + g + tt + n + d + s;
            // depth.d:539-541: row printed iff min_cov <= COV <= max_cov (or -a); a failing sample ends the position
            // (`return`, not `continue`: the remaining samples are dropped -- SURVEY quirk 2)
            bool ok = (double)total >= c.min_cov && (double)total <= c.max_cov;
            if (!ok && !c.annotate) break;
            o.str(name.data(), name.size()); o.ch('\t'); o.u64((uint64_t)t->start + i); o.ch('\t'); o.u64(total);
            o.ch('\t'); o.u64(a); o.ch('\t'); o.u64(cc); o.ch('\t'); o.u64(g); o.ch('\t'); o.u64(tt); o.ch('\t'); o.u64(d); o.ch('\t'); o.u64(s);
            if (!c.combined) { const std::string& sn = c.samples[si]; o.ch('\t'); o.str(sn.data(), sn.size()); }
            if (c.annotate) { o.ch('\t'); o.ch(!any ? (c.min_cov > 0 ? 'n' : 'y') : (ok ? 'y' : 'n')); }
            o.ch('\n');
        }
    }
    return 0;
}

static int text_cb(void* user, const char* text, size_t len) {
    Ctx& c = *(Ctx*)user; c.out.flush();
    return fwrite(text, 1, len, c.out.f) == len ? 0 : 1;
}

static int stat_cb(void* user, const bdepth_region_stat* s, uint64_t idx) {
    Ctx& c = *(Ctx*)user; Out& o = c.out;
    uint32_t length = s->end - s->start;
    float mean_cov = (float)s->n_bases / (float)length;                       // depth.d:851
    bool ok = (double)mean_cov >= c.min_cov && (double)mean_cov <= c.max_cov;
    if (!ok && !c.annotate) return 0;
    if (c.window_mode) { const std::string& nm = c.ref_names[s->ref_id]; o.str(nm.data(), nm.size()); o.ch('\t'); o.u64(s->start); o.ch('\t'); o.u64(s->end); o.ch('\t'); }
    else { std::string l = c.raw_lines[idx]; while (!l.empty() && is_white(l.back())) l.pop_back(); o.str(l.data(), l.size()); o.ch('\t'); }
    o.u64(s->n_reads); o.ch('\t'); o.g(mean_cov);
    for (size_t j = 0; j < c.thr.size(); j++) {
        float pct = (float)s->cov_ge[j] * 100 / (float)length;                   // depth.d:861
        if (c.thr[j] == 0) pct = 100.0f;
        o.ch('\t'); o.g(pct);
    }
    if (!c.combined) { const std::string& sn = c.samples[s->sample_id]; o.ch('\t'); o.str(sn.data(), sn.size()); }
    if (c.annotate) { o.ch('\t'); o.ch(ok ? 'y' : 'n'); }
    o.ch('\n');
    return 0;
}

static void region_header(Ctx& c, size_t n_before) {      // depth.d:643-659
    static const char* def[3] = {"chrom", "chromStart", "chromEnd"};
    Out& o = c.out; o.lit("# ");
    for (size_t k = 0; k < std::min<size_t>(n_before, 3); k++) { o.str(def[k], strlen(def[k])); o.ch('\t'); }
    for (size_t k = 3; k < n_before; k++) { o.ch('F'); o.u64(k); o.ch('\t'); }
    o.lit("readCount\tmeanCoverage");
    for (uint32_t t : c.thr) { o.lit("\tpercentage"); o.u64(t); }
    if (!c.combined) o.lit("\tsampleName");
    if (c.annotate) o.lit("\tmeanCovWithinBounds");
    o.ch('\n'); o.flush(); fflush(o.f);
}

// `sambamba index input.bam [output.bai]` (index_main, sambamba/index.d:56-130) with the index built on the GPU (bdepth_build_index):
// -t / -p are accepted, -c (check bins) and -F (FASTA) are not offered.  Errors as "sambamba-index: <msg>", exit code 1.
static int index_main(Args& a) {
    a.v.erase(a.v.begin() + 1);
    std::vector<std::string> v;
    opt_take(a, "nthreads", 't', true, &v); opt_take(a, "show-progress", 'p', false, nullptr);
    if (a.v.size() != 2 && a.v.size() != 3) {
        fprintf(stderr, "Usage: sambamba-index [OPTIONS] <input.bam> [output_file]\n\n\tCreates index for a BAM file\n\nOptions: -t, --nthreads=NTHREADS\n               accepted for compatibility (the index is built on the GPU)\n         -p, --show-progress\n               accepted for compatibility\n");
        return 0;
    }
    const std::string in = a.v[1], out = a.v.size() > 2 ? a.v[2] : in + ".bai";
    bdepth_t* h = nullptr;
    if (bdepth_open(in.c_str(), 0, &h)) { fprintf(stderr, "sambamba-index: %s\n", bdepth_last_error(nullptr)); return 1; }
    int64_t n = bdepth_build_index(h, nullptr, 0);
    if (n < 0) { fprintf(stderr, "sambamba-index: %s\n", bdepth_last_error(h)); bdepth_close(h); return 1; }
    std::vector<uint8_t> buf((size_t)n);
    if (bdepth_build_index(h, buf.data(), (uint64_t)n) != n) { fprintf(stderr, "sambamba-index: %s\n", bdepth_last_error(h)); bdepth_close(h); return 1; }
    bdepth_close(h);
    FILE* f = fopen(out.c_str(), "wb");
    if (!f || fwrite(buf.data(), 1, buf.size(), f) != buf.size() || fclose(f) != 0) { fprintf(stderr, "sambamba-index: Cannot open file `%s' in mode `wb'\n", out.c_str()); return 1; }
    return 0;
}

int main(int argc, char** argv) {
    // accept both `sambamba-depth-b200 base ...` and `sambamba-depth-b200 depth base ...`
    Args a; for (int i = 0; i < argc; i++) a.v.push_back(argv[i]);
    if (a.v.size() > 1 && a.v[1] == "depth") a.v.erase(a.v.begin() + 1);
    if (a.v.size() > 1 && a.v[1] == "index") return index_main(a);
    if (a.v.size() < 3) { usage(); return 0; }
    Ctx c;
    if (a.v[1] == "base") c.mode = 0; else if (a.v[1] == "region") c.mode = 1; else if (a.v[1] == "window") c.mode = 2; else { usage(); return 0; }
    if (c.mode == 0) c.min_cov = 1;
    a.v.erase(a.v.begin());      // args = args[1 .. $] : a.v[0] is now the mode
    std::string err;
    auto die = [&](const std::string& m) { c.out.flush(); fprintf(stderr, "sambamba-depth: %s\n", m.c_str()); return 1; };
    std::vector<std::string> v; std::string query; bool has_query = false; std::string out_fn, bed_fn; bool has_bed = false; int min_bq = 0; bool fix_mates = false;
    if (opt_take(a, "filter", 'F', true, &v) > 0) { query = v.back(); has_query = true; } v.clear();
    if (opt_take(a, "output-filename", 'o', true, &v) > 0) out_fn = v.back();
    v.clear();
    opt_take(a, "nthreads", 't', true, &v); v.clear();                                      // accepted for compatibility (its value is not looked at)
    std::string cerr_; unsigned long long uv = 0;
    if (opt_take(a, "min-coverage", 'c', true, &v) > 0 && !conv_double(v.back(), c.min_cov, cerr_)) return die(cerr_);
    v.clear();
    if (opt_take(a, "max-coverage", 'C', true, &v) > 0 && !conv_double(v.back(), c.max_cov, cerr_)) return die(cerr_);
    v.clear();
    if (opt_take(a, "min-base-quality", 'q', true, &v) > 0) { if (!conv_unsigned(v.back(), 255, "ubyte", uv, cerr_)) return die(cerr_); min_bq = (int)uv; }      // ubyte min_base_quality, depth.d:280
    v.clear();
    if (opt_take(a, "annotate", 'a', false, nullptr) > 0) c.annotate = true;
    if (opt_take(a, "combined", 0, false, nullptr) > 0) c.combined = true;
    if (opt_take(a, "fix-mate-overlaps", 'm', false, nullptr) > 0) fix_mates = true;
    const bool build_index = opt_take(a, "build-index", 0, false, nullptr) > 0;      // not a sambamba option: index un-indexed input on the GPU instead of refusing it
    c.out.f = out_fn.empty() ? stdout : fopen(out_fn.c_str(), "w+");
    if (!c.out.f) return die("Cannot open file `" + out_fn + "' in mode `w+'");
    if (c.mode != 2 && opt_take(a, "regions", 'L', true, &v) > 0) { bed_fn = v.back(); has_bed = true; } v.clear();
    if (c.mode == 1 && !has_bed) { fprintf(stderr, "BED file or a region must be provided in region mode\n"); return 1; }
    // printer.init
    bool report_zero = false; uint32_t window = 0, overlap = 0;
    if (c.mode == 0) {
        if (opt_take(a, "report-zero-coverage", 'z', false, nullptr) > 0) report_zero = true;
        if (report_zero) c.min_cov = 0;
        c.out.lit("REF\tPOS\tCOV\tA\tC\tG\tT\tDEL\tREFSKIP");
        if (!c.combined) c.out.lit("\tSAMPLE");
        if (c.annotate) c.out.lit("\tFLAG");
        c.out.ch('\n');
    } else {
        if (c.mode == 2) {
            if (opt_take(a, "window-size", 'w', true, &v) > 0) { if (!conv_unsigned(v.back(), 0xFFFFFFFFFFFFFFF0ull, "ulong", uv, cerr_)) return die(cerr_); if (uv > 0xFFFFFFFFull) return die("window sizes of 2^32 and more are not supported"); window = (uint32_t)uv; }
    v.clear();
            if (opt_take(a, "overlap", 0, true, &v) > 0) { if (!conv_unsigned(v.back(), 0xFFFFFFFFFFFFFFF0ull, "ulong", uv, cerr_)) return die(cerr_); overlap = uv > 0xFFFFFFFFull ? 0xFFFFFFFFu : (uint32_t)uv; }
    v.clear();
        }
        opt_take(a, "cov-threshold", 'T', true, &v); for (auto& s : v) { if (!conv_unsigned(s, 0xFFFFFFFFull, "uint", uv, cerr_)) return die(cerr_); c.thr.push_back((uint32_t)uv); }
    v.clear();
        if (c.mode == 2) {
            if (!(window > 0)) return die("positive window size must be specified");
            if (!(overlap < window)) return die("specified overlap is larger than window size");
        }
    }
    int mapq_gt = 0; uint32_t flag_reject = 0x600;
    if (a.v.size() < 2) return die("no input BAM given");
    const std::string bam_path = a.v[1];
    if (c.mode == 2) { c.window_mode = true; }

    // with -L only the header and the BGZF members inside the regions' BAI chunks are looked at (a run that turns out to
    // need the whole file frames the rest itself)
    int rc = has_bed ? bdepth_open_lazy(bam_path.c_str(), 0, &c.h) : bdepth_open(bam_path.c_str(), 0, &c.h);
    if (rc) return die(bdepth_last_error(nullptr));
    for (size_t fi = 2; fi < a.v.size(); fi++) if (bdepth_add_input(c.h, a.v[fi].c_str())) return die(bdepth_last_error(c.h));      // new MultiBamReader(bam_filenames), depth.d:1162-1163
    if (!bdepth_is_coordinate_sorted(c.h)) return die("All files must be coordinate-sorted");
    if (!bdepth_has_index(c.h) && build_index && a.v.size() == 2) { if (bdepth_build_index(c.h, nullptr, 0) < 0) return die(bdepth_last_error(c.h)); }
    if (!bdepth_has_index(c.h)) return die("All files must be indexed");
    int nref = bdepth_n_ref(c.h);
    for (int i = 0; i < nref; i++) c.ref_names.push_back(bdepth_ref_name(c.h, i));
    for (int i = 0; i < bdepth_n_samples(c.h); i++) c.samples.push_back(bdepth_sample_name(c.h, i));
    bdepth_set_combined(c.h, c.combined ? 1 : 0);
    bdepth_set_filter(c.h, mapq_gt, flag_reject);
    if (has_query && bdepth_set_filter_query(c.h, query.c_str())) return die(bdepth_last_error(c.h));      // createFilterFromQuery, depth.d:1159
    bdepth_set_min_baseq(c.h, (uint32_t)min_bq);
    bdepth_set_fix_mates(c.h, fix_mates ? 1 : 0);
    auto find_ref = [&](const std::string& n) { for (int i = 0; i < nref; i++) if (c.ref_names[i] == n) return i; return -1; };
    if (c.mode == 2) region_header(c, 3);

    std::vector<bdepth_region> regs;
    if (has_bed) {
        std::vector<BedIv> ivs; std::vector<std::string> lines;
        if (bed_read(bed_fn, ivs, lines)) {
            for (auto& iv : ivs) { int id = find_ref(iv.chr); if (id < 0) continue; regs.push_back({(uint32_t)id, (uint32_t)iv.beg, (uint32_t)iv.end}); }
            if (c.mode == 1) { if (lines.empty()) return die("empty BED file"); c.raw_lines = lines; size_t nf = 0; { bool in = false; for (char ch : lines[0]) { if (!is_white(ch)) { if (!in) { nf++; in = true; } } else in = false; } } region_header(c, nf); }
        } else {
            std::string ref; uint32_t beg, end; parse_region_string(bed_fn, ref, beg, end);
            int id = find_ref(ref);
            if (id < 0) return die("couldn't open file " + bed_fn + " or find reference " + ref);
            if (end == UINT32_MAX) end = bdepth_ref_length(c.h, id);
            regs.push_back({(uint32_t)id, beg, end});
            if (c.mode == 1) { c.raw_lines = {ref + "\t" + std::to_string(beg) + "\t" + std::to_string(end)}; region_header(c, 3); }
        }
    }
    if (c.mode == 0) {
        if (has_bed) {
            // no region at all, or none that holds a position (a region string the wrong way round, one that begins behind its reference's end):
            // no read overlaps it, no row is required -- the header is all the reference prints (an empty region list would mean "everything" to the library)
            bool any = false;
            for (auto& g : regs) any |= g.start < g.end && g.start < bdepth_ref_length(c.h, (int)g.ref_id);
            if (!any) { c.out.flush(); bdepth_close(c.h); return 0; }
            bdepth_set_regions(c.h, regs.data(), regs.size());
        }
        // rows are formatted on the GPU (one counter set, or one row per sample and position); base_tile_cb is the host-side
        // formatter a caller of bdepth_run_base would use
        if (c.combined || c.samples.size() <= 64) { bdepth_text_opts to{c.min_cov, c.max_cov, c.annotate ? 1 : 0}; rc = bdepth_run_base_text(c.h, &to, text_cb, &c); }
        else rc = bdepth_run_base(c.h, base_tile_cb, &c);
    } else if (c.mode == 1) {
        rc = bdepth_run_regions(c.h, regs.data(), regs.size(), c.thr.data(), c.thr.size(), stat_cb, &c);
    } else {
        rc = bdepth_run_windows(c.h, window, overlap, c.thr.data(), c.thr.size(), stat_cb, &c);
    }
    if (rc) return die(bdepth_last_error(c.h));
    for (int i = 0; i < nref; i++) if (bdepth_ref_has_reads(c.h, i)) fprintf(stderr, "Processing reference #%d (%s)\n", i + 1, c.ref_names[i].c_str());
    c.out.flush(); fflush(c.out.f); if (!out_fn.empty()) fclose(c.out.f);
    bdepth_close(c.h);
    return 0;
}
