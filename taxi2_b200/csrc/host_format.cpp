// Host-side batch formatter and subset aggregator for the result files either side of the hot
// path (SURVEY.md 8f-1 / 8f-3).  Pure C++ (no CUDA): once the distances come off the GPU at
// millions of pairs per second, the reference's per-value `str.format` + generator `.send`
// writers (distances.py:95-186, versus_all.py:278-350) and its per-pair dict aggregation
// (versus_all.py:57-95, 623-645) would dominate the task by orders of magnitude.
//
// Byte-for-byte contract: rows are "\t".join(fields) + "\n" (handlers.py:219-227); floats are
// printf-formatted with the C equivalent of the Python format spec (both are correctly rounded, so
// "{:.4f}" and "%.4f" agree); undefined values print the `missing` marker.  The aggregation adds
// the values in the reference's row-major order, so the fp64 sums are bit-identical.
#include "../../include/taxi2_b200.h"

#include <algorithm>
#include <fcntl.h>
#include <unistd.h>
#include <sys/types.h>
#include <climits>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

namespace {

struct Table {
    const char* bytes;
    const int64_t* off;
    void append(std::string& out, int64_t k) const { out.append(bytes + off[k], (size_t)(off[k + 1] - off[k])); }
};

// "%.Nf" (N <= 9) / "%f": the formats the tasks use by default.  -1 = something else (snprintf).
inline int fixed_decimals(const char* fmt)
{
    if (fmt[0] != '%') return -1;
    if (fmt[1] == 'f' && fmt[2] == 0) return 6;
    if (fmt[1] != '.' || fmt[2] < '0' || fmt[2] > '9' || fmt[3] != 'f' || fmt[4] != 0) return -1;
    return fmt[2] - '0';
}

// v formatted like printf("%.{decimals}f") -- the correctly rounded decimal (ties to even on the
// EXACT binary value, which is what both glibc and Python's format do) -- by integer arithmetic:
// v = m * 2^e exactly, so v * 10^d = (m * 10^d) >> -e with the remainder deciding the rounding.
// ~15 ns instead of ~300 ns for snprintf; distances are written by the hundred million.
inline bool append_fixed(std::string& out, double v, int decimals)
{
    static const uint64_t kPow10[10] = {1ULL, 10ULL, 100ULL, 1000ULL, 10000ULL, 100000ULL, 1000000ULL, 10000000ULL, 100000000ULL, 1000000000ULL};
    uint64_t bits;
    std::memcpy(&bits, &v, sizeof bits);
    const bool negative = (bits >> 63) != 0;
    const int exponent = (int)((bits >> 52) & 0x7FF);
    uint64_t mant = bits & ((1ULL << 52) - 1);
    if (exponent == 0x7FF) return false;
    int e2;
    if (exponent == 0) e2 = -1074;
    else { mant |= 1ULL << 52; e2 = exponent - 1075; }
    if (e2 > 0) return false;                                      // |v| >= 2^53: leave it to snprintf
    unsigned __int128 scaled = (unsigned __int128)mant * kPow10[decimals];   // < 2^83
    unsigned __int128 q;
    const int shift = -e2;
    if (shift == 0) q = scaled;
    else if (shift >= 100) q = 0;                                   // far below half a unit of the last decimal
    else {
        q = scaled >> shift;
        const unsigned __int128 rem = scaled & ((((unsigned __int128)1) << shift) - 1), half = ((unsigned __int128)1) << (shift - 1);
        if (rem > half || (rem == half && (q & 1))) q += 1;
    }
    if (q >> 64) return false;
    // q = the value in units of the last decimal: its low `decimals` digits are the fraction, the rest the
    // whole part (at least one digit) -- peeled off from the right, no division by a run-time power of ten
    uint64_t digits = (uint64_t)q;
    char buf[48];
    int at = (int)sizeof buf;
    for (int k = 0; k < decimals; ++k) { buf[--at] = (char)('0' + digits % 10); digits /= 10; }
    if (decimals) buf[--at] = '.';
    do { buf[--at] = (char)('0' + digits % 10); digits /= 10; } while (digits);
    if (negative) buf[--at] = '-';
    out.append(buf + at, sizeof buf - (size_t)at);
    return true;
}

struct ValueFormat {
    const char* fmt;
    int decimals;
    explicit ValueFormat(const char* f) : fmt(f), decimals(fixed_decimals(f)) {}
};

inline void append_value(std::string& out, double v, bool undefined, double scale, const ValueFormat& vf, const char* missing)
{
    if (undefined || std::isnan(v) || std::isinf(v)) { out += missing; return; }
    const double x = v * scale;
    if (vf.decimals >= 0 && append_fixed(out, x, vf.decimals)) return;
    char buf[64];
    const int n = std::snprintf(buf, sizeof buf, vf.fmt, x);
    out.append(buf, (size_t)std::max(0, std::min<int>(n, (int)sizeof buf - 1)));
}

// run fn(row_begin, row_end, out) over row chunks on `threads` threads, then write the chunks in order
template <class Fn> int format_rows(const char* path, int32_t nx, int32_t threads, Fn fn)
{
    if (threads <= 0) threads = (int32_t)std::max(1u, std::thread::hardware_concurrency());
    threads = std::max(1, std::min<int32_t>(threads, std::max(1, nx)));
    std::vector<std::string> chunks((size_t)threads);
    std::vector<std::thread> pool;
    const int32_t per = (nx + threads - 1) / threads;
    for (int32_t t = 0; t < threads; ++t) {
        const int32_t b = t * per, e = std::min(nx, b + per);
        if (b >= e) break;
        if (threads == 1) fn(b, e, chunks[(size_t)t]);
        else pool.emplace_back([&, b, e, t] { fn(b, e, chunks[(size_t)t]); });
    }
    for (auto& th : pool) th.join();
    // append the chunks in order; the page-cache copy of hundreds of megabytes is itself worth
    // spreading over the threads, so every chunk is written at its own offset with pwrite
    const int fd = ::open(path, O_WRONLY | O_CREAT, 0644);
    if (fd < 0) return TAXI_E_ARG;
    off_t at = ::lseek(fd, 0, SEEK_END);
    if (at < 0) { ::close(fd); return TAXI_E_ARG; }
    std::vector<off_t> offsets(chunks.size());
    for (size_t t = 0; t < chunks.size(); ++t) { offsets[t] = at; at += (off_t)chunks[t].size(); }
    std::vector<int> ok(chunks.size(), 1);
    auto put = [&](size_t t) {
        const char* data = chunks[t].data();
        size_t left = chunks[t].size();
        off_t pos = offsets[t];
        while (left) {
            const ssize_t n = ::pwrite(fd, data, left, pos);
            if (n <= 0) { ok[t] = 0; return; }
            data += n; left -= (size_t)n; pos += n;
        }
    };
    std::vector<std::thread> writers;
    for (size_t t = 0; t < chunks.size(); ++t) {
        if (chunks[t].empty()) continue;
        if (chunks.size() == 1) put(t);
        else writers.emplace_back(put, t);
    }
    for (auto& th : writers) th.join();
    const bool all_ok = std::all_of(ok.begin(), ok.end(), [](int v) { return v != 0; });
    return (::close(fd) == 0 && all_ok) ? TAXI_OK : TAXI_E_ARG;
}

}  // namespace

extern "C" {

// Row layout segments of taxi_format_pairs
enum { SEG_X0 = 0, SEG_X1, SEG_X2, SEG_X3, SEG_Y0, SEG_Y1, SEG_Y2, SEG_Y3, SEG_SCORES, SEG_COMPARISON };

int taxi_format_pairs(const char* path, const int32_t* segments, int32_t nsegments,
                      const char* const* xbytes, const int64_t* const* xoff,
                      const char* const* ybytes, const int64_t* const* yoff,
                      int32_t x0, int32_t nx, int32_t ny,
                      const double* metrics, const uint8_t* undefined,
                      const int32_t* columns, int32_t ncolumns, double scale,
                      const char* float_format, const char* missing,
                      const int32_t* xgenus, const int32_t* xspecies, const int32_t* ygenus, const int32_t* yspecies,
                      const char* const* type_labels, int32_t threads)
{
    if (!path || !segments || nsegments <= 0 || nx < 0 || ny < 0 || !metrics || !float_format || !missing) return TAXI_E_ARG;
    const ValueFormat vf(float_format);
    // bytes of one row, estimated from the tables (y entries on average, x entries of the block's first row):
    // reserving the right amount up front saves the reallocation copies of chunks of hundreds of megabytes
    size_t row_bytes = 2;
    for (int32_t s = 0; s < nsegments; ++s) {
        const int seg = segments[s];
        if (seg >= SEG_X0 && seg <= SEG_X3 && nx > 0) row_bytes += (size_t)(xoff[seg][x0 + 1] - xoff[seg][x0]) + 8;
        else if (seg >= SEG_Y0 && seg <= SEG_Y3 && ny > 0) row_bytes += (size_t)((yoff[seg - SEG_Y0][ny] - yoff[seg - SEG_Y0][0]) / ny) + 2;
        else if (seg == SEG_SCORES) row_bytes += (size_t)ncolumns * 12;
        else row_bytes += 16;
    }
    auto fn = [&](int32_t b, int32_t e, std::string& out) {
        out.reserve((size_t)(e - b) * (size_t)ny * row_bytes);
        for (int32_t i = b; i < e; ++i) {
            for (int32_t j = 0; j < ny; ++j) {
                const size_t p = (size_t)i * ny + j;
                const bool undef = undefined && undefined[p];
                for (int32_t s = 0; s < nsegments; ++s) {
                    if (s) out += '\t';
                    const int seg = segments[s];
                    if (seg >= SEG_X0 && seg <= SEG_X3) Table{xbytes[seg], xoff[seg]}.append(out, x0 + i);
                    else if (seg >= SEG_Y0 && seg <= SEG_Y3) Table{ybytes[seg - SEG_Y0], yoff[seg - SEG_Y0]}.append(out, j);
                    else if (seg == SEG_SCORES) {
                        for (int32_t c = 0; c < ncolumns; ++c) {
                            if (c) out += '\t';
                            append_value(out, metrics[p * 4 + columns[c]], undef, scale, vf, missing);
                        }
                    } else if (seg == SEG_COMPARISON) {
                        // versus_all.py:262-275: None when a partition is absent, else "same subset?"
                        const int sg = xgenus ? (xgenus[x0 + i] == ygenus[j] ? 1 : 0) : -1;
                        const int ss = xspecies ? (xspecies[x0 + i] == yspecies[j] ? 1 : 0) : -1;
                        int label;   // 0 Unknown, 1 IntraSpecies, 2 InterSpecies, 3 IntraGenus, 4 InterGenus
                        if (sg < 0) label = ss < 0 ? 0 : (ss ? 1 : 2);
                        else if (sg == 0) label = 4;
                        else label = ss < 0 ? 3 : (ss ? 1 : 2);
                        out += type_labels[label];
                    }
                }
                out += '\n';
            }
        }
    };
    return format_rows(path, nx, threads, fn);
}

// n values as text, tab separated, into the caller's buffer: the float formatting of the subset
// statistics files (versus_all.py:143-249), whose S^2 cells are formatted in one call per column.
// Returns the bytes written, or -(bytes needed) when `capacity` is too small.
int64_t taxi_format_values(const double* values, int64_t n, const uint8_t* undefined, double scale,
                           const char* float_format, const char* missing, char* out, int64_t capacity)
{
    if (!values || n < 0 || !float_format || !missing || !out) return TAXI_E_ARG;
    const ValueFormat vf(float_format);
    std::string text;
    text.reserve((size_t)n * 8);
    for (int64_t k = 0; k < n; ++k) {
        if (k) text += '\t';
        append_value(text, values[k], undefined && undefined[k], scale, vf, missing);
    }
    if ((int64_t)text.size() > capacity) return -(int64_t)text.size();
    std::memcpy(out, text.data(), text.size());
    return (int64_t)text.size();
}

// One row per x: id, then one value per y (DistanceHandler.Matrix rows, distances.py:183-186)
int taxi_format_matrix(const char* path, const char* xid_bytes, const int64_t* xid_off, int32_t x0, int32_t nx, int32_t ny,
                       const double* metrics, const uint8_t* undefined, int32_t column, double scale,
                       const char* float_format, const char* missing, int32_t threads)
{
    if (!path || !xid_bytes || !xid_off || nx < 0 || ny < 0 || !metrics || column < 0 || column > 3) return TAXI_E_ARG;
    const Table ids{xid_bytes, xid_off};
    const ValueFormat vf(float_format);
    auto fn = [&](int32_t b, int32_t e, std::string& out) {
        out.reserve((size_t)(e - b) * (size_t)ny * 8);
        for (int32_t i = b; i < e; ++i) {
            ids.append(out, x0 + i);
            for (int32_t j = 0; j < ny; ++j) {
                const size_t p = (size_t)i * ny + j;
                out += '\t';
                append_value(out, metrics[p * 4 + column], undefined && undefined[p], scale, vf, missing);
            }
            out += '\n';
        }
    };
    return format_rows(path, nx, threads, fn);
}

// A gapped string holds one latin-1 byte per symbol (the sequences went in as str.encode("latin-1"));
// the file holds the UTF-8 text of that str, as the Python handler writes it: bytes 0x80-0xFF take two.
static void append_latin1_as_utf8(std::string& out, const uint8_t* s, size_t len)
{
    for (size_t k = 0; k < len; ++k) {
        const uint8_t c = s[k];
        if (c < 0x80) {
            out += (char)c;
        } else {
            out += (char)(0xC0 | (c >> 6));
            out += (char)(0x80 | (c & 0x3F));
        }
    }
}

// SequencePairHandler.Formatted records (pairs.py:51-97) for the nx*ny pairs of a row block, pair
// p = (x0 + p / ny, p % ny): "idx / idy", aligned x, the match pattern ('|' equal and not a gap, '-'
// either is a gap, '.' otherwise; one character per symbol), aligned y; records are separated by one
// empty line, so every record but the file's first is preceded by "\n".  The gapped strings are the
// right-aligned slots taxi_align_strings fills: pair p occupies [aln_start[p], aln_off[p + 1]).
int taxi_format_aligned_pairs(const char* path, int32_t first_record,
                              const char* xid_bytes, const int64_t* xid_off, const char* yid_bytes, const int64_t* yid_off,
                              int32_t x0, int32_t nx, int32_t ny,
                              const uint8_t* aln_x, const uint8_t* aln_y, const int64_t* aln_start, const int64_t* aln_off,
                              int32_t threads)
{
    if (!path || !xid_bytes || !xid_off || !yid_bytes || !yid_off || nx < 0 || ny < 0 || !aln_x || !aln_y || !aln_start || !aln_off)
        return TAXI_E_ARG;
    const Table xids{xid_bytes, xid_off}, yids{yid_bytes, yid_off};
    auto fn = [&](int32_t b, int32_t e, std::string& out) {
        size_t need = 0;
        for (int64_t p = (int64_t)b * ny; p < (int64_t)e * ny; ++p) need += 3 * (size_t)(aln_off[p + 1] - aln_start[p]) + 48;
        out.reserve(need);
        for (int32_t i = b; i < e; ++i) {
            for (int32_t j = 0; j < ny; ++j) {
                const int64_t p = (int64_t)i * ny + j;
                if (p > 0 || !first_record) out += '\n';
                xids.append(out, x0 + i);
                out += " / ";
                yids.append(out, j);
                out += '\n';
                const uint8_t* ax = aln_x + aln_start[p];
                const uint8_t* ay = aln_y + aln_start[p];
                const size_t len = (size_t)(aln_off[p + 1] - aln_start[p]);
                uint8_t high = 0;   // any byte >= 0x80 in either string: the UTF-8 path
                for (size_t k = 0; k < len; ++k) high |= ax[k] | ay[k];
                const bool ascii = high < 0x80;
                if (ascii) out.append(reinterpret_cast<const char*>(ax), len);
                else append_latin1_as_utf8(out, ax, len);
                out += '\n';
                const size_t at = out.size();
                out.resize(at + len);
                // '-' where either side is a gap, '|' where the symbols agree, '.' otherwise: written without
                // branches over raw pointers so that the compiler turns it into byte-wise SIMD compares / selects
                char* __restrict__ pat = &out[at];
                for (size_t k = 0; k < len; ++k) {
                    const uint8_t a = ax[k], c = ay[k];
                    const uint8_t gap = (uint8_t)-(uint8_t)((a == '-') | (c == '-')), eq = (uint8_t)-(uint8_t)(a == c);
                    const uint8_t base = (uint8_t)(('|' & eq) | ('.' & (uint8_t)~eq));
                    pat[k] = (char)(('-' & gap) | (base & (uint8_t)~gap));
                }
                out += '\n';
                if (ascii) out.append(reinterpret_cast<const char*>(ay), len);
                else append_latin1_as_utf8(out, ay, len);
                out += '\n';
            }
        }
    };
    return format_rows(path, nx, threads, fn);
}

// SimpleAggregator state per (subset_x, subset_y) for one metric column (versus_all.py:57-95):
// sum / min / max / n over the defined values in row-major order, plus the order in which the keys
// first appeared (the reference's dicts iterate in insertion order).  Subset ids are 0..nsub-1, with
// one id reserved by the caller for "not in the partition".
int taxi_aggregate_subsets(const double* metrics, const uint8_t* undefined, int32_t x0, int32_t nx, int32_t ny,
                           int32_t column, double scale, const int32_t* xsubset, const int32_t* ysubset, int32_t nsub,
                           double* sum, double* vmin, double* vmax, int64_t* count, int64_t* first_seen, int64_t* next_order)
{
    if (!metrics || !xsubset || !ysubset || !sum || !vmin || !vmax || !count || !first_seen || !next_order) return TAXI_E_ARG;
    for (int32_t i = 0; i < nx; ++i) {
        const int64_t sx = xsubset[x0 + i];
        for (int32_t j = 0; j < ny; ++j) {
            const size_t p = (size_t)i * ny + j;
            const int64_t k = sx * nsub + ysubset[j];
            if (first_seen[k] < 0) first_seen[k] = (*next_order)++;
            double v = metrics[p * 4 + column];
            if ((undefined && undefined[p]) || std::isnan(v) || std::isinf(v)) continue;
            v *= scale;
            sum[k] += v;
            if (v < vmin[k]) vmin[k] = v;
            if (v > vmax[k]) vmax[k] = v;
            count[k] += 1;
        }
    }
    return TAXI_OK;
}

// subsets/<partition>/linear/{pairs,identity}.tsv (versus_all.py:143-205, 647-684): one row per selected key
// (subset_x, subset_y) in first-seen order -- the label of subset_x, the label of subset_y when with_query,
// then mean / min / max of every metric, "NA" where no distance was defined.  Rows are appended; the
// header stays in Python.  A partition of S subsets has up to S^2 keys: a million rows for a thousand
// species, formerly a dozen Python strings each.
int taxi_format_subset_rows(const char* path, const char* label_bytes, const int64_t* label_off,
                            const int32_t* kx, const int32_t* ky, const uint8_t* select, int64_t nkeys, int32_t with_query,
                            int32_t nmetrics, const double* const* mean, const double* const* vmin, const double* const* vmax,
                            const int64_t* const* count, const char* float_format, int32_t threads)
{
    if (!path || !label_bytes || !label_off || !kx || !ky || nkeys < 0 || nkeys > INT32_MAX || nmetrics < 0 || !float_format) return TAXI_E_ARG;
    if (nmetrics > 0 && (!mean || !vmin || !vmax || !count)) return TAXI_E_ARG;
    const Table labels{label_bytes, label_off};
    const ValueFormat vf(float_format);
    auto fn = [&](int32_t b, int32_t e, std::string& out) {
        out.reserve((size_t)(e - b) * (size_t)(24 + 24 * nmetrics));
        for (int32_t k = b; k < e; ++k) {
            if (select && !select[k]) continue;
            labels.append(out, kx[k]);
            if (with_query) { out += '\t'; labels.append(out, ky[k]); }
            for (int32_t m = 0; m < nmetrics; ++m) {
                const bool none = count[m][k] == 0;
                out += '\t'; append_value(out, none ? 0.0 : mean[m][k], none, 1.0, vf, "NA");
                out += '\t'; append_value(out, none ? 0.0 : vmin[m][k], none, 1.0, vf, "NA");
                out += '\t'; append_value(out, none ? 0.0 : vmax[m][k], none, 1.0, vf, "NA");
            }
            out += '\n';
        }
    };
    return format_rows(path, (int32_t)nkeys, threads, fn);
}

// subsets/<partition>/matricial/<metric>.tsv (versus_all.py:207-249): the keys in first-seen order cut into runs of
// equal subset_x (the reference flushes a matrix row whenever subset_x changes); the first run is preceded by the
// header (an empty cell, then its subset_y labels); a cell is t0 mean t1 min t2 max t3 -- the pieces of the
// statistics template around its three fields -- or "NA" where no distance was defined.  The whole file.
int taxi_format_subset_matrix(const char* path, const char* label_bytes, const int64_t* label_off,
                              const int32_t* kx, const int32_t* ky, int64_t nkeys,
                              const double* mean, const double* vmin, const double* vmax, const int64_t* count,
                              const char* float_format, const char* t0, const char* t1, const char* t2, const char* t3, int32_t threads)
{
    if (!path || !label_bytes || !label_off || !kx || !ky || nkeys < 0 || nkeys > INT32_MAX || !float_format || !t0 || !t1 || !t2 || !t3) return TAXI_E_ARG;
    if (nkeys > 0 && (!mean || !vmin || !vmax || !count)) return TAXI_E_ARG;
    const Table labels{label_bytes, label_off};
    const ValueFormat vf(float_format);
    std::vector<int64_t> starts;
    for (int64_t k = 0; k < nkeys; ++k) if (k == 0 || kx[k] != kx[k - 1]) starts.push_back(k);
    starts.push_back(nkeys);
    const int32_t nruns = (int32_t)starts.size() - 1;
    { const int fd = ::open(path, O_WRONLY | O_CREAT | O_TRUNC, 0644); if (fd < 0) return TAXI_E_ARG; ::close(fd); }
    if (nruns == 0) return TAXI_OK;
    auto fn = [&](int32_t b, int32_t e, std::string& out) {
        out.reserve((size_t)(starts[e] - starts[b]) * 40 + 64);
        for (int32_t r = b; r < e; ++r) {
            const int64_t lo = starts[r], hi = starts[r + 1];
            if (r == 0) {
                for (int64_t k = lo; k < hi; ++k) { out += '\t'; labels.append(out, ky[k]); }
                out += '\n';
            }
            labels.append(out, kx[lo]);
            for (int64_t k = lo; k < hi; ++k) {
                out += '\t';
                if (count[k] == 0) { out += "NA"; continue; }
                out += t0; append_value(out, mean[k], false, 1.0, vf, "NA");
                out += t1; append_value(out, vmin[k], false, 1.0, vf, "NA");
                out += t2; append_value(out, vmax[k], false, 1.0, vf, "NA");
                out += t3;
            }
            out += '\n';
        }
    };
    return format_rows(path, nruns, threads, fn);
}

}  // extern "C"
