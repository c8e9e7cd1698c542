// C-ABI of the taxi2_b200 library (see include/taxi2_b200.h): context, sequence residency,
// kernel dispatch, host<->device staging.  No CPU compute path exists in this file: every
// entry point that produces results launches a CUDA kernel or fails with TAXI_E_CUDA.
#include "../../include/taxi2_b200.h"

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include <cub/device/device_scan.cuh>

#include "common.cuh"
#include "count_planes.cuh"
#include "count_tc.cuh"
#include "gotoh_pair16.cuh"
#include "gotoh_warp.cuh"

using namespace taxi;

namespace {

thread_local std::string g_error;

int fail(int code, const char* fmt, ...)
{
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}

#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t e_ = (expr);                                                                \
        if (e_ != cudaSuccess)                                                                  \
            return fail(TAXI_E_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

template <class T> struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
    // grow-only; `slack` (in 1/8ths) over-allocates so that a slightly larger next request
    // (the next tile's sequences) does not cost a cudaFree + cudaMalloc pair
    cudaError_t reserve(size_t n, int slack = 0)
    {
        if (n <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; cap = 0;
        const size_t want = std::max<size_t>(n + n / 8 * (size_t)slack, 1);
        cudaError_t e = cudaMalloc(&p, want * sizeof(T));
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// page-locked host memory, grow-only; growing keeps the first `keep` elements (results gathered over
// several device blocks), and device-to-host copies into it run at the full link rate
template <class T> struct HostBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
    cudaError_t reserve(size_t n, size_t keep)
    {
        if (n <= cap) return cudaSuccess;
        const size_t want = std::max(n, cap + cap / 2);
        void* q = nullptr;
        cudaError_t e = cudaHostAlloc(&q, want * sizeof(T), cudaHostAllocPortable);
        if (e != cudaSuccess) return e;
        if (keep) std::memcpy(q, p, keep * sizeof(T));
        if (p) cudaFreeHost(p);
        p = static_cast<T*>(q); cap = want;
        return cudaSuccess;
    }
    void release() { if (p) cudaFreeHost(p); p = nullptr; cap = 0; }
};

// Every entry point runs on its context's device and leaves the calling thread's current device
// as it found it (the caller may be torch, or another context's thread).
struct DeviceGuard {
    int prev = -1;
    cudaError_t err;
    explicit DeviceGuard(int device)
    {
        err = cudaGetDevice(&prev);
        if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
        else if (err == cudaSuccess) prev = -1;   // nothing to restore
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
#define ON_DEVICE(dev)                 \
    DeviceGuard device_guard_(dev);    \
    CUDA_TRY(device_guard_.err)

struct SeqSet {
    bool loaded = false;
    int32_t n = 0;
    int32_t maxlen = 0;
    int64_t total = 0;
    std::vector<int64_t> off;       // host copy of offsets
    DevBuf<uint8_t> bytes;          // normalized ASCII (DP kernels compare code points)
    DevBuf<uint8_t> codes;          // 3-bit symbol codes for the packed fast path (valid if ctx->codebook_ok)
    DevBuf<int64_t> d_off;
    DevBuf<uint4> planes;           // [W][n] (b0, b1, R, G') per 32 columns (count_planes.cuh)
    DevBuf<int2> span;              // [n] first / last word with a real column
    // tensor-core operand rows of the alignment-free kernel (count_tc.cuh), built on first use
    DevBuf<int8_t> tcops;           // [n][8 * Lp]
    int32_t Lp = 0;                 // columns padded to TC_TILE
    bool tc_built = false;
    CUtensorMap tc_map;            // boxes of 128 rows
    CUtensorMap tc_map64;          // boxes of 64 rows (x role of the two-CTAs-per-SM geometry)
    int32_t W = 0;
};

}  // namespace

struct taxi_ctx {
    int device = 0;
    int sms = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    SeqSet set[2];
    ScoreSet sc{};
    int32_t raw_scores[TAXI_NSCORES]{};
    bool have_scores = false;
    // symbol codebook shared by both sets: A C G T N are fixed, up to two more symbols are
    // assigned in order of appearance; more than CODE_SYMBOLS (15) symbols disable the packed fast path
    int16_t codebook[256];
    int ncodes = 5;
    bool codebook_ok = true;
    DevBuf<uint8_t> d_codebook;
    int force_general = 0;          // option: always use the general int32 kernel
    int force_top = 0;              // option: packed kernel without the bottom-aligned variant
    int sort_columns = 1;           // option: visit the columns of a rectangle longest first when their lengths differ
    int no_coop = 0;                // option: never use the intra-task kernel for long pairs
    int metric_tables = 1;          // option: alignment-free kernels take JC / K2P from the fixed-point logarithm table where rows are short enough
    DevBuf<long long> lntab;        // ln k * 2^58, k = 0 .. 3 * LN_TABLE_COLS
    int tc_persistent = 0;          // option: persistent form of the tensor-core counting kernel (count_tc_persistent_kernel)
    int tc_tile_x = 128;            // option: x rows per tile of the tensor-core counting kernel (128: one CTA per SM, 64: two)
    int count_kernel = 0;           // option: alignment-free rectangles on 0 = whichever fits, 1 = popcount kernel, 2 = tensor-core kernel
    int last_kernel = 0;            // 0 = none, 32 = gotoh_warp (int32), 16 = gotoh_pair16
    // scratch
    DevBuf<uint8_t> trace;
    DevBuf<int32_t> bnd;
    DevBuf<unsigned long long> counter;
    DevBuf<int> status;
    DevBuf<int32_t> d_px, d_py, d_xrows, d_ycols, d_units;
    std::vector<int32_t> h_la, h_lb, h_units;   // pair-list calls: x / y length of every pair, warp units of the packed kernel
    DevBuf<int32_t> d_score, d_counts;
    DevBuf<double> d_metrics;
    DevBuf<uint8_t> d_alnx, d_alny;
    DevBuf<int64_t> d_alnoff, d_alnstart;
    DevBuf<long long> d_redo;
    DevBuf<int32_t> d_rscore, d_rcounts;   // results of the re-aligned mirrored pairs before they are scattered
    DevBuf<double> d_rmetrics;
    DevBuf<unsigned long long> d_redo_count;
    DevBuf<int32_t> d_argidx, d_bestcounts;
    DevBuf<double> d_argval, d_bestmetrics;
    // taxi_pairs_within: per-row counts and offsets of a block, the scan's scratch, and the held CSR
    // result (taxi_pairs_within_fetch), dropped by the next call that computes on this context
    DevBuf<int32_t> d_rowcnt, d_rowoff;
    DevBuf<uint8_t> d_scantmp;
    std::vector<int32_t> h_rowoff;
    HostBuf<int32_t> h_within_idx, h_within_counts;
    HostBuf<double> h_within_metrics;
    int64_t within_total = 0;
    bool within_held = false;
    // stats of the last call
    int64_t launches = 0, cells = 0;
    double kernel_ms = 0.0;
    int64_t last_redo = 0;          // pairs the last "both orientations" call had to re-align
};

namespace {

const SeqSet& yset(const taxi_ctx* c) { return c->set[1].loaded ? c->set[1] : c->set[0]; }

int check_ctx(const taxi_ctx* c, bool need_scores)
{
    if (!c) return fail(TAXI_E_ARG, "null context");
    if (!c->set[0].loaded) return fail(TAXI_E_ARG, "no sequences loaded (taxi_load_sequences)");
    if (need_scores && !c->have_scores) return fail(TAXI_E_ARG, "no scores set (taxi_set_scores)");
    return TAXI_OK;
}

// rows-per-lane variants compiled in; 32*H rows form one stripe
const int kH[] = {4, 8, 12, 16, 21, 24, 32};

int pick_H(int max_rows)
{
    // fewest wasted row slots over whole stripes; ties -> larger H (fewer shuffles per cell)
    int best = 32;
    long long best_slots = -1;
    for (int h : kH) {
        const long long sl = 32LL * h;
        const long long slots = (max_rows + sl - 1) / sl * sl;
        if (best_slots < 0 || slots < best_slots || (slots == best_slots && h > best)) { best = h; best_slots = slots; }
    }
    return best;
}

template <int H> cudaError_t occupancy(int* blocks_per_sm)
{
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, gotoh_warp_kernel<H>, GOTOH_WARPS_PER_BLOCK * 32, 0);
}

template <int H> void launch_gotoh(const AlignArgs& a, int grid, cudaStream_t st)
{
    gotoh_warp_kernel<H><<<grid, GOTOH_WARPS_PER_BLOCK * 32, 0, st>>>(a);
}

template <int H> void launch_coop(const AlignArgs& a, int grid, cudaStream_t st)
{
    gotoh_coop_kernel<H><<<grid, GOTOH_COOP_WARPS * 32, 0, st>>>(a);
}

struct Dispatch {
    int H;
    cudaError_t (*occ)(int*);
    void (*launch)(const AlignArgs&, int, cudaStream_t);
    int HB;
    void (*coop)(const AlignArgs&, int, cudaStream_t) = nullptr;   // intra-task variant (general kernel only)
};

const Dispatch kDispatch[] = {
    {4, occupancy<4>, launch_gotoh<4>, TraceGeom<4>::HB},     {8, occupancy<8>, launch_gotoh<8>, TraceGeom<8>::HB},
    {12, occupancy<12>, launch_gotoh<12>, TraceGeom<12>::HB}, {16, occupancy<16>, launch_gotoh<16>, TraceGeom<16>::HB},
    {21, occupancy<21>, launch_gotoh<21>, TraceGeom<21>::HB, launch_coop<21>}, {24, occupancy<24>, launch_gotoh<24>, TraceGeom<24>::HB, launch_coop<24>},
    {32, occupancy<32>, launch_gotoh<32>, TraceGeom<32>::HB, launch_coop<32>},
};

// bytes -> 3-bit symbol codes through the context codebook, in the padded per-sequence layout of
// code_offset(): one block per sequence (grid-stride), CODE_LEAD pad codes, the codes, one pad code
__global__ void encode_codes_kernel(const uint8_t* __restrict__ bytes, const int64_t* __restrict__ off, int32_t nseq,
                                    const uint8_t* __restrict__ book, uint8_t* __restrict__ out)
{
    __shared__ uint8_t lut[256];
    lut[threadIdx.x & 255] = book[threadIdx.x & 255];
    __syncthreads();
    for (int32_t seq = blockIdx.x; seq < nseq; seq += gridDim.x) {
        const int64_t o = off[seq];
        const int len = (int)(off[seq + 1] - o);
        uint8_t* dst = out + code_offset(o, seq) - CODE_LEAD;
        for (int k = threadIdx.x; k < len + CODE_PAD; k += blockDim.x)
            dst[k] = (k < CODE_LEAD || k == CODE_LEAD + len) ? (uint8_t)CODE_PADSYM : lut[bytes[o + k - CODE_LEAD]];
    }
}

template <int H, int MODE> cudaError_t occupancy16(int* blocks_per_sm)
{
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, gotoh_pair16_kernel<H, MODE>, PAIR16_WARPS_PER_BLOCK * 32, 0);
}

template <int H, int MODE> void launch_pair16(const AlignArgs& a, int grid, cudaStream_t st)
{
    gotoh_pair16_kernel<H, MODE><<<grid, PAIR16_WARPS_PER_BLOCK * 32, 0, st>>>(a);
}

template <int H> cudaError_t occupancy16s(int* blocks_per_sm)
{
    return cudaOccupancyMaxActiveBlocksPerMultiprocessor(blocks_per_sm, gotoh_pair16_kernel<H, 1, true>, PAIR16_WARPS_PER_BLOCK * 32, 0);
}

template <int H> void launch_pair16s(const AlignArgs& a, int grid, cudaStream_t st)
{
    gotoh_pair16_kernel<H, 1, true><<<grid, PAIR16_WARPS_PER_BLOCK * 32, 0, st>>>(a);
}

#define P16(H, M) {H, occupancy16<H, M>, launch_pair16<H, M>, Pair16Geom<H>::HB}
const Dispatch kDispatch16[] = {P16(8, 0), P16(12, 0), P16(16, 0), P16(21, 0), P16(24, 0), P16(32, 0)};
// bottom-aligned rows (needs internal extend == end extend and one spare row slot)
const Dispatch kDispatch16b[] = {P16(8, 1), P16(12, 1), P16(16, 1), P16(21, 1), P16(24, 1), P16(32, 1)};
// ... in several stripes, for x longer than one stripe
const Dispatch kDispatch16m[] = {P16(16, 2), P16(21, 2), P16(24, 2), P16(32, 2)};
#undef P16
// bottom-aligned, "both orientations" (the code of every cell also records Ix / Iy ties, the walk mirrors the result)
#define P16S(H) {H, occupancy16s<H>, launch_pair16s<H>, Pair16Geom<H, true>::HB}
const Dispatch kDispatch16s[] = {P16S(8), P16S(12), P16S(16), P16S(21), P16S(24), P16S(32)};
#undef P16S

// Packed 16-bit fast path: is it EXACT for this score set and these lengths?  (gotoh_pair16.cuh)
// dead_extra: largest difference between the x lengths of the two pairs of a warp unit (0 for
// rectangles).  *max_dead_out (optional) receives the largest dead_extra that would still fit.
bool fast16_eligible(const taxi_ctx* c, int max_rows, int max_cols, int dead_extra, Fast16* out, int* H_out, int* mode_out,
                     long long* max_dead_out = nullptr)
{
    if (c->force_general || !c->codebook_ok) return false;
    const int32_t* s = c->raw_scores;
    const int match = s[0], mm = s[1], io = s[2], ie = s[3], eo = s[4], ee = s[5];
    if (io == ie && eo == ee) return false;                 // Needleman-Wunsch order: general kernel
    if (match < mm || match < 0) return false;
    const int beta = match, D = match - mm;
    // every gap step must be a non-negative penalty in the transformed space S' = S - match*i
    const int gaps[4] = {io, ie, eo, ee};
    for (int g : gaps) if (g > 0) return false;
    // No co-optimal path may put a vertical gap next to a horizontal one: replacing runs
    // (Iy^a Ix^b) by min(a,b) diagonals plus one gap of |a-b| must be strictly better for every
    // a, b >= 1 and every end/internal typing of the two runs (worst case: all mismatches).
    const int O[2] = {io, eo}, E[2] = {ie, ee};
    for (int tx = 0; tx < 2; ++tx)
        for (int ty = 0; ty < 2; ++ty) {
            const int slope = E[tx] + E[ty] - mm;            // mm = min(match, mismatch) here
            if (slope > 0) return false;
            if (O[tx] + E[ty] - mm >= 0) return false;       // a > b
            if (O[ty] + E[tx] - mm >= 0) return false;       // b > a
            if (O[tx] + O[ty] - mm >= 0) return false;       // a == b
        }
    // geometry: one stripe when x fits (the bottom-aligned variant keeps the border row in a slot
    // of its own), else the multi-stripe bottom-aligned variant with the least wasted slots
    const bool bottom = (ie == ee) && !c->force_top;
    int H = 0, mode = bottom ? 1 : 0;
    long long R = 0;
    for (const auto& e : kDispatch16) if (32 * e.H >= max_rows + (bottom ? 1 : 0)) { H = e.H; R = 32LL * e.H; break; }
    if (!H) {
        if (!bottom) return false;
        mode = 2;
        for (const auto& e : kDispatch16m) {
            const long long sl = 32LL * e.H, slots = (max_rows + 1 + sl - 1) / sl * sl;
            if (R == 0 || slots < R || (slots == R && e.H > H)) { R = slots; H = e.H; }
        }
    }
    Fast16 f;
    f.D16 = 16 * D; f.beta = beta;
    if (D > 2000) return false;
    f.negD = 0u - (uint32_t)f.D16;
    f.class_lut[0] = f.class_lut[1] = 0x55555555u;   // unused codes and the pad: "missing"
    f.ascii[0] = f.ascii[1] = f.ascii[2] = f.ascii[3] = 0; f.has_gap_symbol = 0;
    for (int ch = 0; ch < 256; ++ch) {
        const int k = c->codebook[ch];
        if (k < 0 || k >= CODE_SYMBOLS) continue;
        f.class_lut[k >> 3] = (f.class_lut[k >> 3] & ~(0xFu << (4 * (k & 7)))) | ((uint32_t)base_class(ch) << (4 * (k & 7)));
        f.ascii[k >> 2] |= (uint32_t)ch << (8 * (k & 3));
        if (ch == '-') f.has_gap_symbol = 1;
    }
    f.PoX = 16 * (match - io); f.PeX = 16 * (match - ie); f.PeoX = 16 * (match - eo); f.PeeX = 16 * (match - ee);
    f.PoY = -16 * io; f.PeY = -16 * ie; f.PeoY = -16 * eo; f.PeeY = -16 * ee;
    // Range.  The best transformed value is 0 (all matches), so the bias sits at the top of the
    // window.  Lowest real value of the padded DP: a leading end gap to the diagonal followed by
    // mismatches -- linear in (i, j), so its extreme is at a corner -- plus one gap opening for the
    // Ix / Iy states.
    // Dead slots (bottom-aligned variants: the slots above row 0 of a pair, inside the lanes that
    // are live for the unit) idle below `neg`: the topmost one is fed the constant `neg` from
    // above, and every further one sits at most one vertical extension below its upper neighbour
    // (H >= Ix >= Ix(above) - extend; the M and Iy candidates are then within one mismatch / one
    // opening of that).  A pair has at most H - 1 dead slots of its own plus, when its partner in
    // the unit has a longer x, the difference of the two x lengths (dead_extra).  `neg` must keep
    // the whole dead band non-negative -- a value that wraps below 0 reappears at the top of the
    // unsigned window and beats every real score -- and below every reachable real value.
    // (bottom-aligned variants pad ABOVE row 0 with dead slots, so their DP has max_rows real rows;
    //  the top-aligned variant pads below row nA with rows that extend the DP and has no dead slots)
    if (mode != 0) R = max_rows;
    const long long C = max_cols;
    const long long pen_e = std::max({f.PeX, f.PeeX, f.PeY, f.PeeY});
    const long long pen_o = std::max({f.PoX, f.PeoX, f.PoY, f.PeoY});
    if (pen_o > 3000 || pen_e > 3000) return false;
    const long long m = std::min(R, C);
    const long long corner_v = f.PeoX + R * f.PeeX;                                   // (R, 0)
    const long long corner_h = f.PeoY + C * f.PeeY;                                   // (0, C)
    const long long corner_d = m * f.D16 + (R > C ? f.PeoX + (R - C) * f.PeeX : f.PeoY + (C - R) * f.PeeY);   // (R, C)
    const long long lower = std::max({corner_v, corner_h, corner_d}) + pen_o + pen_e;
    const long long dead_step = std::max<long long>({f.D16, f.PeX, f.PeeX, 16});
    const long long dead_fixed = pen_o + pen_e + f.D16 + 512 + 15;
    const long long bias = (65535 - 256) / 16 * 16;
    const long long room = bias - lower - 256;                                        // largest admissible neg
    if (max_dead_out) *max_dead_out = (mode == 0) ? (1LL << 40) : (room - dead_fixed) / dead_step - H;
    const long long neg = ((mode == 0 ? (long long)H : (long long)H + dead_extra) * dead_step + dead_fixed) / 16 * 16;
    if (neg > room) return false;
    f.dead_extra = dead_extra;
    f.bias = (int32_t)bias; f.neg = (int32_t)neg;
    *out = f; *H_out = H;
    *mode_out = mode;
    return true;
}

// Enqueue one alignment launch.  All pointers in `a` other than scratch are already device
// pointers.  max_rows / max_cols bound the lengths of the x / y sequences touched.
// Pair-list launches of the packed kernel: which two pairs share a warp.  Pairs are visited by
// decreasing x length (then y length), so the two pairs of a unit sweep about the same rows and
// columns and the longest units are handed out first; two neighbours share a unit only if their
// x lengths differ by at most `max_dead` (see fast16_eligible), else a pair runs alone.
// Returns the largest difference actually used.
int build_units(taxi_ctx* c, long long npairs, long long max_dead)
{
    std::vector<int32_t> order((size_t)npairs);
    for (long long k = 0; k < npairs; ++k) order[(size_t)k] = (int32_t)k;
    const std::vector<int32_t>& la = c->h_la;
    const std::vector<int32_t>& lb = c->h_lb;
    std::stable_sort(order.begin(), order.end(), [&](int32_t u, int32_t v) {
        return la[u] != la[v] ? la[u] > la[v] : lb[u] > lb[v];
    });
    c->h_units.clear();
    c->h_units.reserve((size_t)npairs + 1);
    int used = 0;
    for (long long k = 0; k < npairs;) {
        const int32_t p0 = order[(size_t)k];
        if (k + 1 < npairs && (long long)la[p0] - la[order[(size_t)k + 1]] <= max_dead) {
            const int32_t p1 = order[(size_t)k + 1];
            used = std::max(used, la[p0] - la[p1]);
            c->h_units.push_back(p0); c->h_units.push_back(p1);
            k += 2;
        } else {
            c->h_units.push_back(p0); c->h_units.push_back(p0);
            k += 1;
        }
    }
    return used;
}

// Enqueue one alignment launch.  All pointers in `a` other than scratch are already device
// pointers.  max_rows / max_cols bound the lengths of the x / y sequences touched.  Pair-list
// launches (a.px set) expect the lengths of every pair in c->h_la / c->h_lb (upload_pairs).
// sym: the caller wants the "both orientations" kernel (a.t_* / a.redo set); *sym_used tells whether this launch could
// provide it (packed, bottom-aligned, one stripe) -- if not, nothing is launched and the caller falls back.
int enqueue_align(taxi_ctx* c, AlignArgs a, int max_rows, int max_cols, bool record_start = true, bool reset_work = true,
                  bool sym = false, bool* sym_used = nullptr)
{
    Fast16 f16{};
    int H = 0;
    int mode = 0;
    long long max_dead = 0;
    bool fast = fast16_eligible(c, max_rows, max_cols, 0, &f16, &H, &mode, &max_dead);
    a.unit_pairs = nullptr;
    a.nunits = 0;
    if (fast && a.px) {
        if (a.npairs >= (1LL << 31)) return fail(TAXI_E_ARG, "pair list too long (%lld)", a.npairs);
        const int used = build_units(c, a.npairs, std::max<long long>(0, max_dead));
        if (used > 0 && mode != 0) {
            fast = fast16_eligible(c, max_rows, max_cols, used, &f16, &H, &mode);
            if (!fast) return fail(TAXI_E_RANGE, "internal: dead-band budget (%d) rejected", used);
        }
        CUDA_TRY(c->d_units.reserve(c->h_units.size(), 1));
        CUDA_TRY(cudaMemcpyAsync(c->d_units.p, c->h_units.data(), c->h_units.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));   // h_units may be rebuilt by the next call
        a.unit_pairs = c->d_units.p;
        a.nunits = (long long)(c->h_units.size() / 2);
    } else if (fast) {
        a.nunits = (a.npairs / a.ny) * (((long long)a.ny + 1) / 2);   // whole rows: npairs = rows * ny
    }
    if (!fast) H = pick_H(max_rows);
    // few long pairs: the intra-task kernel wants tall stripes (its variants are the 21 / 24 / 32-row ones)
    if (!fast && !c->no_coop && max_rows > 2 * 32 * 21 && a.npairs * 4 <= (long long)c->sms * 3 * GOTOH_WARPS_PER_BLOCK) {
        long long best = -1;
        for (int h : {21, 24, 32}) {
            const long long sl = 32LL * h, slots = (max_rows + sl - 1) / sl * sl;
            if (best < 0 || slots < best || (slots == best && h > H)) { best = slots; H = h; }
        }
    }
    const Dispatch* d = nullptr;
    if (sym) {
        const bool ok = fast && mode == 1 && !a.px;
        if (sym_used) *sym_used = ok;
        if (!ok) return TAXI_OK;
        for (const auto& e : kDispatch16s) if (e.H == H) d = &e;
    }
    else if (fast) {
        if (mode == 2) { for (const auto& e : kDispatch16m) if (e.H == H) d = &e; }
        else { for (const auto& e : (mode == 1 ? kDispatch16b : kDispatch16)) if (e.H == H) d = &e; }
    }
    else { for (const auto& e : kDispatch) if (e.H == H) d = &e; }
    // occupancy of each kernel variant is queried once per process (contexts of several devices
    // may run on several host threads: the cache is shared and locked)
    static std::map<const Dispatch*, int> occupancy_cache;
    static std::mutex occupancy_lock;
    int bps = 0;
    {
        std::lock_guard<std::mutex> guard(occupancy_lock);
        auto hit = occupancy_cache.find(d);
        if (hit != occupancy_cache.end()) bps = hit->second;
        else {
            CUDA_TRY(d->occ(&bps));
            occupancy_cache[d] = bps;
        }
    }
    if (bps < 1) return fail(TAXI_E_CUDA, "gotoh kernel does not fit on an SM");
    const long long SL = 32LL * H;
    const long long nstripes = fast ? (mode == 2 ? (max_rows + 1 + SL - 1) / SL : 1) : (max_rows + SL - 1) / SL;
    // Size the arena for the longest column sequence of the loaded set, not just of this launch:
    // growing it later means cudaFree + cudaMalloc of ~1 GB, a device-wide synchronisation that
    // costs tens to hundreds of milliseconds when several ranks share the driver.
    const long long arena_cols = (std::max<long long>(max_cols, yset(c).maxlen) + 255) / 128 * 128;   // + headroom for reloaded sets
    const long long per_warp = ((nstripes * (arena_cols + 31LL) * 32 * d->HB) + 255) / 256 * 256;
    const long long bnd_per_warp = 2LL * (arena_cols + 2);
    const long long work_units = fast ? a.nunits : a.npairs;
    c->last_kernel = sym ? 20 : (fast ? 16 + mode : 32);
    a.f16 = f16;
    // Intra-task kernel: long pairs (several stripes) that are too few to occupy the GPU one pair per
    // warp share a CTA each, the stripes of a pair pipelined over its warps (gotoh_coop_kernel).
    const bool coop = !fast && !c->no_coop && d->coop != nullptr && nstripes >= 2 && nstripes <= GOTOH_COOP_MAX_STRIPES &&
                      a.npairs * 4 <= (long long)c->sms * bps * GOTOH_WARPS_PER_BLOCK;
    // resident warps (CTAs for the intra-task kernel), capped by pairs and by a trace-arena budget of half the free memory
    long long warps = coop ? (long long)c->sms : (long long)c->sms * bps * GOTOH_WARPS_PER_BLOCK;
    size_t free_b = 0, total_b = 0;
    if ((long long)c->trace.cap >= warps * per_warp) free_b = 0;   // arena already large enough: no query
    else CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    const long long budget = std::max<long long>((long long)c->trace.cap, (long long)((free_b + c->trace.cap) / 2));
    if (per_warp > budget) return fail(TAXI_E_NOMEM, "one pair needs %lld B of traceback arena, only %lld B available", per_warp, budget);
    warps = std::min(warps, std::max(1LL, budget / per_warp));
    warps = std::min(warps, work_units);
    int grid = coop ? (int)std::max(warps, 1LL) : (int)((warps + GOTOH_WARPS_PER_BLOCK - 1) / GOTOH_WARPS_PER_BLOCK);
    grid = std::max(grid, 1);
    const long long gw = coop ? (long long)grid : (long long)grid * GOTOH_WARPS_PER_BLOCK;
    CUDA_TRY(c->trace.reserve((size_t)(gw * per_warp)));
    CUDA_TRY(c->bnd.reserve((size_t)(gw * bnd_per_warp * (coop ? nstripes : 1))));
    CUDA_TRY(c->counter.reserve(1));
    CUDA_TRY(cudaMemsetAsync(c->counter.p, 0, sizeof(unsigned long long), c->stream));
    a.coop_stripes = (int32_t)nstripes;
    if (coop) c->last_kernel = 33;
    a.sc = c->sc;
    a.trace = c->trace.p; a.trace_per_warp = per_warp;
    a.bnd = c->bnd.p; a.bnd_per_warp = bnd_per_warp;
    a.counter = c->counter.p; a.status = c->status.p;
    if (record_start) CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
    if (coop) d->coop(a, grid, c->stream);
    else d->launch(a, grid, c->stream);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
    c->launches += 1;
    return TAXI_OK;
}

int finish_align(taxi_ctx* c)
{
    ON_DEVICE(c->device);
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, c->ev0, c->ev1) == cudaSuccess) c->kernel_ms += ms;
    // the device-side error flag is sticky: kernels only ever set it, and it is cleared here, after
    // it has been read, so that a *_device launch enqueued before another cannot lose its error
    int st = 0;
    CUDA_TRY(cudaMemcpy(&st, c->status.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (st != 0) CUDA_TRY(cudaMemset(c->status.p, 0, sizeof(int)));
    if (st == TAXI_E_EMPTY) return fail(TAXI_E_EMPTY, "sequence has zero length");
    if (st != 0) return fail(st, "device status %d", st);
    return TAXI_OK;
}

int range_check(const taxi_ctx* c, int max_rows, int max_cols)
{
    long long m = 0;
    for (int k = 0; k < TAXI_NSCORES; ++k) m = std::max<long long>(m, std::llabs((long long)c->raw_scores[k]));
    // every DP value is bounded by (rows + cols + 2) * max|score|; it must survive the *64 scaling
    if ((max_rows + (long long)max_cols + 2) * m >= (1LL << 24))
        return fail(TAXI_E_RANGE, "scores x lengths exceed the exact int32 range of the DP");
    return TAXI_OK;
}

void fill_rect(AlignArgs& a, const taxi_ctx* c, int32_t x0, int32_t y0, int32_t ny, long long npairs)
{
    const SeqSet& X = c->set[0];
    const SeqSet& Y = yset(c);
    a.xb = X.bytes.p; a.xoff = X.d_off.p;
    a.yb = Y.bytes.p; a.yoff = Y.d_off.p;
    a.xc = X.codes.p; a.yc = Y.codes.p;
    a.px = a.py = nullptr; a.xrows = nullptr; a.ycols = nullptr;
    a.x0 = x0; a.y0 = y0; a.ny = ny; a.npairs = npairs;
}

bool has_empty(const SeqSet& s, int32_t i0, int32_t n)
{
    for (int32_t i = i0; i < i0 + n; ++i) if (s.off[i + 1] == s.off[i]) return true;
    return false;
}

int max_len_range(const SeqSet& s, int32_t i0, int32_t n)
{
    int m = 0;
    for (int32_t i = i0; i < i0 + n; ++i) m = std::max<int>(m, (int)(s.off[i + 1] - s.off[i]));
    return m;
}

long long cells_rect(const SeqSet& X, const SeqSet& Y, int32_t x0, int32_t nx, int32_t y0, int32_t ny)
{
    return (long long)(X.off[x0 + nx] - X.off[x0]) * (long long)(Y.off[y0 + ny] - Y.off[y0]);
}

int check_rect(const taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny)
{
    const SeqSet& X = c->set[0];
    const SeqSet& Y = yset(c);
    if (nx < 0 || ny < 0 || x0 < 0 || y0 < 0 || x0 + (long long)nx > X.n || y0 + (long long)ny > Y.n)
        return fail(TAXI_E_ARG, "rectangle [%d,+%d) x [%d,+%d) outside the loaded sets (%d x %d)", x0, nx, y0, ny, X.n, Y.n);
    return TAXI_OK;
}

int upload_pairs(taxi_ctx* c, const int32_t* px, const int32_t* py, int64_t n, int* max_rows, int* max_cols, long long* cells,
                 bool need_nonempty = true)
{
    const SeqSet& X = c->set[0];
    const SeqSet& Y = yset(c);
    int mr = 0, mc = 0;
    long long cc = 0;
    c->h_la.resize((size_t)n); c->h_lb.resize((size_t)n);
    for (int64_t k = 0; k < n; ++k) {
        if (px[k] < 0 || px[k] >= X.n || py[k] < 0 || py[k] >= Y.n)
            return fail(TAXI_E_ARG, "pair %lld = (%d, %d) outside the loaded sets", (long long)k, px[k], py[k]);
        const int la = (int)(X.off[px[k] + 1] - X.off[px[k]]), lb = (int)(Y.off[py[k] + 1] - Y.off[py[k]]);
        c->h_la[(size_t)k] = la; c->h_lb[(size_t)k] = lb;
        if (need_nonempty && (la == 0 || lb == 0))
            return fail(TAXI_E_EMPTY, "sequence has zero length (pair %lld)", (long long)k);
        mr = std::max(mr, la); mc = std::max(mc, lb);
        cc += (long long)la * lb;
    }
    CUDA_TRY(c->d_px.reserve((size_t)n));
    CUDA_TRY(c->d_py.reserve((size_t)n));
    CUDA_TRY(cudaMemcpyAsync(c->d_px.p, px, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->d_py.p, py, (size_t)n * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    *max_rows = mr; *max_cols = mc;
    if (cells) *cells = cc;
    return TAXI_OK;
}

int reserve_outputs(taxi_ctx* c, int64_t n, uint32_t flags)
{
    if (flags & TAXI_OUT_SCORE) CUDA_TRY(c->d_score.reserve((size_t)n));
    if (flags & TAXI_OUT_COUNTS) CUDA_TRY(c->d_counts.reserve((size_t)n * 4));
    if (flags & TAXI_OUT_METRICS) CUDA_TRY(c->d_metrics.reserve((size_t)n * 4));
    return TAXI_OK;
}

int download_outputs(taxi_ctx* c, int64_t n, uint32_t flags, int32_t* score, int32_t* counts, double* metrics)
{
    if ((flags & TAXI_OUT_SCORE) && score)
        CUDA_TRY(cudaMemcpyAsync(score, c->d_score.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if ((flags & TAXI_OUT_COUNTS) && counts)
        CUDA_TRY(cudaMemcpyAsync(counts, c->d_counts.p, (size_t)n * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if ((flags & TAXI_OUT_METRICS) && metrics)
        CUDA_TRY(cudaMemcpyAsync(metrics, c->d_metrics.p, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    return TAXI_OK;
}

// at the start of every host-facing compute call; a new computation also drops the held pairs_within result
void reset_stats(taxi_ctx* c) { c->launches = 0; c->cells = 0; c->kernel_ms = 0.0; c->within_held = false; }

}  // namespace

extern "C" {

const char* taxi_last_error(void) { return g_error.c_str(); }

int taxi_abi_version(void) { return 1; }

int taxi_device_count(void)
{
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int taxi_ctx_create(int device, taxi_ctx** out)
{
    if (!out) return fail(TAXI_E_ARG, "null out pointer");
    *out = nullptr;
    int n = 0;
    CUDA_TRY(cudaGetDeviceCount(&n));
    if (device < 0 || device >= n) return fail(TAXI_E_CUDA, "CUDA device %d not present (%d visible)", device, n);
    ON_DEVICE(device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(TAXI_E_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device, prop.major, prop.minor);
    taxi_ctx* c = new (std::nothrow) taxi_ctx();
    if (!c) return fail(TAXI_E_NOMEM, "out of host memory");
    c->device = device;
    c->sms = prop.multiProcessorCount;
    cudaError_t e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&c->ev1);
    if (e == cudaSuccess) e = c->status.reserve(1);
    if (e == cudaSuccess) e = cudaMemset(c->status.p, 0, sizeof(int));
    if (e == cudaSuccess) {
        // ln k in fixed point for the table form of the metric epilogue (common.cuh); long double carries 64 bits
        std::vector<long long> tab(LN_TABLE_SIZE, 0);
        for (int k = 1; k < LN_TABLE_SIZE; ++k) tab[k] = (long long)llroundl(logl((long double)k) * 0x1p58L);
        e = c->lntab.reserve(LN_TABLE_SIZE);
        if (e == cudaSuccess) e = cudaMemcpy(c->lntab.p, tab.data(), LN_TABLE_SIZE * sizeof(long long), cudaMemcpyHostToDevice);
    }
    if (e != cudaSuccess) { taxi_ctx_destroy(c); return fail(TAXI_E_CUDA, "stream/event creation failed: %s", cudaGetErrorString(e)); }
    *out = c;
    return TAXI_OK;
}

void taxi_ctx_destroy(taxi_ctx* c)
{
    if (!c) return;
    DeviceGuard device_guard_(c->device);
    cudaStreamSynchronize(c->stream);
    for (auto& s : c->set) { s.bytes.release(); s.codes.release(); s.d_off.release(); s.planes.release(); s.span.release(); s.tcops.release(); }
    c->d_codebook.release(); c->lntab.release();
    c->trace.release(); c->bnd.release(); c->counter.release(); c->status.release();
    c->d_px.release(); c->d_py.release(); c->d_xrows.release(); c->d_ycols.release(); c->d_units.release(); c->d_score.release(); c->d_counts.release(); c->d_metrics.release();
    c->d_alnx.release(); c->d_alny.release(); c->d_alnoff.release(); c->d_alnstart.release();
    c->d_redo.release(); c->d_redo_count.release(); c->d_rscore.release(); c->d_rcounts.release(); c->d_rmetrics.release(); c->d_argidx.release(); c->d_argval.release(); c->d_bestcounts.release(); c->d_bestmetrics.release();
    c->d_rowcnt.release(); c->d_rowoff.release(); c->d_scantmp.release();
    c->h_within_idx.release(); c->h_within_counts.release(); c->h_within_metrics.release();
    cudaEventDestroy(c->ev0); cudaEventDestroy(c->ev1);
    cudaStreamDestroy(c->stream);
    delete c;
}

int taxi_set_scores(taxi_ctx* c, const int32_t s[TAXI_NSCORES])
{
    if (!c || !s) return fail(TAXI_E_ARG, "null argument");
    for (int k = 0; k < TAXI_NSCORES; ++k) {
        if (std::abs((long long)s[k]) > (1 << 20)) return fail(TAXI_E_RANGE, "score %d out of range", s[k]);
        c->raw_scores[k] = s[k];
    }
    ScoreSet& sc = c->sc;
    sc.match = s[0] * 64; sc.mismatch = s[1] * 64;
    sc.io = s[2] * 64; sc.ie = s[3] * 64; sc.eo = s[4] * 64; sc.ee = s[5] * 64;
    // Biopython picks Needleman-Wunsch when every open == extend, else Gotoh; their path
    // generators visit co-optimal predecessors in different orders (DESIGN.md, "tie-breaking").
    const bool gotoh = !(s[2] == s[3] && s[4] == s[5]);
    if (gotoh) { sc.pM = 3; sc.pX = 2; sc.pY = 1; }
    else       { sc.pM = 1; sc.pX = 2; sc.pY = 3; }
    sc.tagM = sc.pM * TAG_REP; sc.tagX = sc.pX * TAG_REP; sc.tagY = sc.pY * TAG_REP;
    c->have_scores = true;
    return TAXI_OK;
}

int taxi_load_sequences(taxi_ctx* c, int set, const uint8_t* bytes, const int64_t* offsets, int32_t n)
{
    if (!c || (set != 0 && set != 1) || !offsets || n < 0) return fail(TAXI_E_ARG, "bad argument");
    ON_DEVICE(c->device);
    SeqSet& s = c->set[set];
    s.loaded = false;
    s.off.assign(offsets, offsets + n + 1);
    if (s.off[0] != 0) return fail(TAXI_E_ARG, "offsets[0] must be 0");
    s.maxlen = 0;
    for (int32_t i = 0; i < n; ++i) {
        if (s.off[i + 1] < s.off[i]) return fail(TAXI_E_ARG, "offsets must be non-decreasing");
        s.maxlen = std::max<int32_t>(s.maxlen, (int32_t)(s.off[i + 1] - s.off[i]));
    }
    s.n = n;
    s.total = s.off[n];
    if (s.total > 0 && !bytes) return fail(TAXI_E_ARG, "null bytes");
    CUDA_TRY(s.bytes.reserve((size_t)s.total + 16, 1));
    CUDA_TRY(s.d_off.reserve((size_t)n + 1, 1));
    if (s.total) CUDA_TRY(cudaMemcpyAsync(s.bytes.p, bytes, (size_t)s.total, cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(s.d_off.p, s.off.data(), ((size_t)n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    // symbol codebook (host scan, O(total)); a new row set starts a new codebook
    if (set == 0) {
        for (auto& v : c->codebook) v = -1;
        const char* fixed = "ACGTN";
        for (int k = 0; k < 5; ++k) c->codebook[(unsigned char)fixed[k]] = (int16_t)k;
        c->ncodes = 5;
        c->codebook_ok = true;
    }
    for (int64_t k = 0; k < s.total && c->codebook_ok; ++k) {
        if (c->codebook[bytes[k]] < 0) {
            if (c->ncodes >= CODE_SYMBOLS) c->codebook_ok = false;
            else c->codebook[bytes[k]] = (int16_t)c->ncodes++;
        }
    }
    if (c->codebook_ok) {
        uint8_t book[256];
        for (int k = 0; k < 256; ++k) book[k] = (uint8_t)(c->codebook[k] < 0 ? CODE_PADSYM : c->codebook[k]);
        CUDA_TRY(c->d_codebook.reserve(256));
        CUDA_TRY(cudaMemcpyAsync(c->d_codebook.p, book, 256, cudaMemcpyHostToDevice, c->stream));
        CUDA_TRY(cudaStreamSynchronize(c->stream));  // `book` is a stack buffer
        CUDA_TRY(s.codes.reserve((size_t)s.total + (size_t)CODE_PAD * (size_t)std::max(n, 1) + 16, 1));
        if (n > 0) {
            encode_codes_kernel<<<(unsigned)std::min<int32_t>(n, 8192), 256, 0, c->stream>>>(s.bytes.p, s.d_off.p, n, c->d_codebook.p, s.codes.p);
            CUDA_TRY(cudaGetLastError());
        }
        // a symbol first seen in set 1 extends the book: set 0 was encoded with the older book,
        // which is still right for every symbol set 0 contains
    }
    s.tc_built = false;
    s.W = std::max(1, ((s.maxlen + 31) / 32 + COUNT_G - 1) / COUNT_G) * COUNT_G;   // whole carry-save groups
    CUDA_TRY(s.planes.reserve((size_t)std::max(n, 1) * s.W, 1));
    CUDA_TRY(s.span.reserve((size_t)std::max(n, 1), 1));
    if (n > 0) {
        const long long total = (long long)n * s.W;
        pack_planes_kernel<<<(unsigned)((total + 255) / 256), 256, 0, c->stream>>>(s.bytes.p, s.d_off.p, n, s.W, s.planes.p);
        CUDA_TRY(cudaGetLastError());
        clip_gaps_kernel<<<(unsigned)((n + 127) / 128), 128, 0, c->stream>>>(n, s.W, s.planes.p, s.span.p);
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    s.loaded = true;
    if (set == 0) c->set[1].loaded = false;  // a new row set serves as both until set 1 is loaded again
    return TAXI_OK;
}

int taxi_sync(taxi_ctx* c)
{
    if (!c) return fail(TAXI_E_ARG, "null context");
    return finish_align(c);
}

int taxi_align_rect_device(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                           int32_t* d_score, int32_t* d_counts, double* d_metrics)
{
    int rc = check_ctx(c, true);
    if (rc) return rc;
    c->within_held = false;
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    ON_DEVICE(c->device);
    const long long npairs = (long long)nx * ny;
    if (npairs == 0) return TAXI_OK;
    if (has_empty(c->set[0], x0, nx) || has_empty(yset(c), y0, ny))
        return fail(TAXI_E_EMPTY, "sequence has zero length");
    const int mr = max_len_range(c->set[0], x0, nx), mc = max_len_range(yset(c), y0, ny);
    if ((rc = range_check(c, mr, mc))) return rc;
    AlignArgs a{};
    fill_rect(a, c, x0, y0, ny, npairs);
    a.score = (flags & TAXI_OUT_SCORE) ? d_score : nullptr;
    a.counts = (flags & TAXI_OUT_COUNTS) ? d_counts : nullptr;
    a.metrics = (flags & TAXI_OUT_METRICS) ? d_metrics : nullptr;
    c->cells += cells_rect(c->set[0], yset(c), x0, nx, y0, ny);

    // Columns of unequal length: a warp sweeps max(len_y) columns for its two pairs, so pairing a
    // short column with a long one idles half the lanes' work.  Columns are visited longest first
    // (stable), which pairs similar lengths and hands the longest units out first.
    {
        const SeqSet& Y = yset(c);
        int lo = INT32_MAX, hi = 0;
        for (int32_t j = y0; j < y0 + ny; ++j) {
            const int len = (int)(Y.off[j + 1] - Y.off[j]);
            lo = std::min(lo, len); hi = std::max(hi, len);
        }
        if (c->sort_columns && ny > 2 && hi - lo > hi / 16) {
            std::vector<int32_t> cols((size_t)ny);
            for (int32_t j = 0; j < ny; ++j) cols[(size_t)j] = y0 + j;
            std::stable_sort(cols.begin(), cols.end(), [&](int32_t u, int32_t v) {
                return Y.off[u + 1] - Y.off[u] > Y.off[v + 1] - Y.off[v];
            });
            CUDA_TRY(c->d_ycols.reserve((size_t)ny, 1));
            CUDA_TRY(cudaMemcpyAsync(c->d_ycols.p, cols.data(), cols.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));   // `cols` is a host vector about to go out of scope
            a.ycols = c->d_ycols.p;
        }
    }

    // Mixed lengths (BASELINE config C5).  The packed kernel keeps 32*H row slots per stripe, so a
    // rectangle whose rows differ a lot in length wastes slots.  Rows are therefore grouped by the
    // kernel geometry that wastes the fewest slots for them -- one stripe of H = 8..32 rows per
    // lane, or several stripes of H = 16..32 above 1023 bp -- and every group gets its own launch
    // over a row list (longest rows first); results still land in the rectangle's row-major positions.
    {
        const SeqSet& X = c->set[0];
        const bool bottom = (c->raw_scores[3] == c->raw_scores[5]) && !c->force_top;
        constexpr int K = (int)(sizeof(kDispatch16) / sizeof(kDispatch16[0]));
        constexpr int M = (int)(sizeof(kDispatch16m) / sizeof(kDispatch16m[0]));
        std::vector<int32_t> rows[K + M];
        int maxlen[K + M] = {0};
        for (int32_t i = x0; i < x0 + nx; ++i) {
            const int len = (int)(X.off[i + 1] - X.off[i]);
            int k = 0;
            while (k < K && 32 * kDispatch16[k].H - (bottom ? 1 : 0) < len) ++k;
            if (k == K) {   // several stripes: same rule as fast16_eligible (fewest slots, ties -> larger H)
                long long best = 0;
                for (int m = 0; m < M; ++m) {
                    const long long sl = 32LL * kDispatch16m[m].H, slots = (len + 1 + sl - 1) / sl * sl;
                    if (best == 0 || slots <= best) { best = slots; k = K + m; }
                }
            }
            rows[k].push_back(i);
            maxlen[k] = std::max(maxlen[k], len);
        }
        // fold small groups (a launch should have enough pairs to fill the GPU): one-stripe groups
        // into the next larger geometry, multi-stripe groups into the fullest multi-stripe group
        const long long min_pairs = 8LL * c->sms * 24;
        auto fold = [&](int from, int to) {
            rows[to].insert(rows[to].end(), rows[from].begin(), rows[from].end());
            maxlen[to] = std::max(maxlen[to], maxlen[from]);
            rows[from].clear();
        };
        for (int k = 0; k < K - 1; ++k)
            if (!rows[k].empty() && (long long)rows[k].size() * ny < min_pairs) fold(k, k + 1);
        int fullest = K;
        for (int k = K; k < K + M; ++k) if (rows[k].size() > rows[fullest].size()) fullest = k;
        for (int k = K; k < K + M; ++k)
            if (k != fullest && !rows[k].empty() && (long long)rows[k].size() * ny < min_pairs) fold(k, fullest);
        int groups = 0;
        for (int k = 0; k < K + M; ++k) groups += !rows[k].empty();
        Fast16 f16{};
        int H = 0, mode = 0;
        if (groups > 1 && !c->force_general && fast16_eligible(c, std::min(mr, 32 * 32 - 1), mc, 0, &f16, &H, &mode)) {
            std::vector<int32_t> all;
            all.reserve((size_t)nx);
            for (int k = K + M - 1; k >= 0; --k) {   // the expensive groups first
                std::stable_sort(rows[k].begin(), rows[k].end(), [&](int32_t u, int32_t v) {
                    return X.off[u + 1] - X.off[u] > X.off[v + 1] - X.off[v];
                });
                all.insert(all.end(), rows[k].begin(), rows[k].end());
            }
            CUDA_TRY(c->d_xrows.reserve((size_t)nx, 1));
            CUDA_TRY(cudaMemcpyAsync(c->d_xrows.p, all.data(), all.size() * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
            CUDA_TRY(cudaStreamSynchronize(c->stream));   // `all` is a host vector about to go out of scope
            size_t at = 0;
            bool first = true;
            for (int k = K + M - 1; k >= 0; --k) {
                if (rows[k].empty()) continue;
                AlignArgs ak = a;
                ak.xrows = c->d_xrows.p + at;
                ak.npairs = (long long)rows[k].size() * ny;
                if ((rc = enqueue_align(c, ak, maxlen[k], mc, first, first))) return rc;
                at += rows[k].size();
                first = false;
            }
            c->last_kernel = 48;   // several launches: rows split by length
            return TAXI_OK;
        }
    }
    return enqueue_align(c, a, mr, mc);
}

// results of a re-aligned list of mirrored pairs -> their transposed positions
__global__ void scatter_redo_kernel(const long long* __restrict__ redo, long long n, int32_t nx, int32_t ny,
                                    const int32_t* __restrict__ score, const int32_t* __restrict__ counts, const double* __restrict__ metrics,
                                    int32_t* __restrict__ t_score, int32_t* __restrict__ t_counts, double* __restrict__ t_metrics)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const long long p = redo[k], t = (p % ny) * (long long)nx + p / ny;
    if (t_score) t_score[t] = score[k];
    if (t_counts) *reinterpret_cast<int4*>(t_counts + 4 * t) = *reinterpret_cast<const int4*>(counts + 4 * k);
    if (t_metrics) {
        reinterpret_cast<double2*>(t_metrics + 4 * t)[0] = reinterpret_cast<const double2*>(metrics + 4 * k)[0];
        reinterpret_cast<double2*>(t_metrics + 4 * t)[1] = reinterpret_cast<const double2*>(metrics + 4 * k)[1];
    }
}

// AlignArgs with the roles of the two sets exchanged: rows from the y set, columns from the x set
void fill_swapped(AlignArgs& a, const taxi_ctx* c)
{
    const SeqSet& X = c->set[0];
    const SeqSet& Y = yset(c);
    a.xb = Y.bytes.p; a.xoff = Y.d_off.p; a.xc = Y.codes.p;
    a.yb = X.bytes.p; a.yoff = X.d_off.p; a.yc = X.codes.p;
    a.px = a.py = nullptr; a.xrows = nullptr; a.ycols = nullptr;
}

// Host-facing rectangles of any size: the device-side result buffers hold at most kChunkPairs
// pairs, so a large rectangle (BASELINE C3 is 2.5e9 ordered pairs = 120 GB of results) is walked
// in blocks of whole rows, each downloaded into its place of the caller's arrays.
constexpr long long kChunkPairs = 1LL << 24;
// the alignment-free kernel needs no traceback arena and runs ~7000x more pairs per second: larger blocks (6.4 GB of results)
constexpr long long kCountChunkPairs = 1LL << 27;

int taxi_align_rect(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                    int32_t* out_score, int32_t* out_counts, double* out_metrics)
{
    int rc = check_ctx(c, true);
    if (rc) return rc;
    reset_stats(c);
    const long long npairs = (long long)nx * ny;
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    if (npairs == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    const int32_t rows = (int32_t)std::max<long long>(1, std::min<long long>(nx, kChunkPairs / ny));
    if ((rc = reserve_outputs(c, (long long)rows * ny, flags))) return rc;
    for (int32_t r0 = 0; r0 < nx; r0 += rows) {
        const int32_t nr = std::min(rows, nx - r0);
        const long long at = (long long)r0 * ny, n = (long long)nr * ny;
        if ((rc = taxi_align_rect_device(c, x0 + r0, nr, y0, ny, flags, c->d_score.p, c->d_counts.p, c->d_metrics.p))) return rc;
        if ((rc = download_outputs(c, n, flags, out_score ? out_score + at : nullptr, out_counts ? out_counts + 4 * at : nullptr,
                                   out_metrics ? out_metrics + 4 * at : nullptr))) return rc;
        if ((rc = finish_align(c))) return rc;
    }
    return TAXI_OK;
}

// Both orientations of a rectangle: (x, y) into d_* ([nx][ny]) and (y, x) into t_* ([ny][nx]).
// The DP of (y, x) is the transpose of the DP of (x, y) (the six scores treat the two sequences
// alike); only the choice between Ix and Iy at equal score differs, and the "both orientations"
// kernel notes on the traced path whether such a choice was ever made.  Pairs without one (99.3 % of
// COI barcodes) get their mirrored result for free; the others are re-aligned the other way round.
// Synchronous (the list of pairs to re-align is read back).  Falls back to two ordinary launches
// when the packed bottom-aligned kernel is not eligible or the rows need several geometries.
int taxi_align_rect_both_device(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                                int32_t* d_score, int32_t* d_counts, double* d_metrics,
                                int32_t* t_score, int32_t* t_counts, double* t_metrics)
{
    int rc = check_ctx(c, true);
    if (rc) return rc;
    c->within_held = false;
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    ON_DEVICE(c->device);
    const long long npairs = (long long)nx * ny;
    if (npairs == 0) return TAXI_OK;
    const SeqSet& X = c->set[0];
    const SeqSet& Y = yset(c);
    if (has_empty(X, x0, nx) || has_empty(Y, y0, ny)) return fail(TAXI_E_EMPTY, "sequence has zero length");
    const int mr = max_len_range(X, x0, nx), mc = max_len_range(Y, y0, ny);
    if ((rc = range_check(c, mr, mc))) return rc;
    int lo = INT32_MAX;
    for (int32_t i = x0; i < x0 + nx; ++i) lo = std::min<int>(lo, (int)(X.off[i + 1] - X.off[i]));
    AlignArgs a{};
    fill_rect(a, c, x0, y0, ny, npairs);
    a.nx = nx;
    a.score = (flags & TAXI_OUT_SCORE) ? d_score : nullptr;
    a.counts = (flags & TAXI_OUT_COUNTS) ? d_counts : nullptr;
    a.metrics = (flags & TAXI_OUT_METRICS) ? d_metrics : nullptr;
    a.t_score = (flags & TAXI_OUT_SCORE) ? t_score : nullptr;
    a.t_counts = (flags & TAXI_OUT_COUNTS) ? t_counts : nullptr;
    a.t_metrics = (flags & TAXI_OUT_METRICS) ? t_metrics : nullptr;
    CUDA_TRY(c->d_redo.reserve((size_t)npairs, 1));
    CUDA_TRY(c->d_redo_count.reserve(1));
    CUDA_TRY(cudaMemsetAsync(c->d_redo_count.p, 0, sizeof(unsigned long long), c->stream));
    a.redo = c->d_redo.p; a.redo_count = c->d_redo_count.p;
    bool sym_used = false;
    // rows of very different length would be split over several kernel geometries: leave those to the ordinary path
    if (lo * 2 > mr && (rc = enqueue_align(c, a, mr, mc, true, true, true, &sym_used))) return rc;
    if (!sym_used) {
        // fallback: two ordinary launches, the second with the roles of the sets exchanged
        c->last_redo = 0;
        if ((rc = taxi_align_rect_device(c, x0, nx, y0, ny, flags, d_score, d_counts, d_metrics))) return rc;
        if ((rc = finish_align(c))) return rc;
        AlignArgs b{};
        fill_swapped(b, c);
        b.x0 = y0; b.y0 = x0; b.ny = nx; b.npairs = npairs;
        b.score = a.t_score; b.counts = a.t_counts; b.metrics = a.t_metrics;
        c->cells += cells_rect(X, Y, x0, nx, y0, ny);
        if ((rc = enqueue_align(c, b, mc, mr))) return rc;
        return finish_align(c);
    }
    c->cells += cells_rect(X, Y, x0, nx, y0, ny);
    if ((rc = finish_align(c))) return rc;
    unsigned long long nredo = 0;
    CUDA_TRY(cudaMemcpy(&nredo, c->d_redo_count.p, sizeof nredo, cudaMemcpyDeviceToHost));
    c->last_redo = (int64_t)nredo;
    if (nredo == 0) return TAXI_OK;
    // re-align the orientation-sensitive pairs as (y, x): rows from the y set, columns from the x set
    std::vector<long long> redo((size_t)nredo);
    CUDA_TRY(cudaMemcpy(redo.data(), c->d_redo.p, (size_t)nredo * sizeof(long long), cudaMemcpyDeviceToHost));
    std::sort(redo.begin(), redo.end());                       // launch order independent of the atomics
    std::vector<int32_t> px((size_t)nredo), py((size_t)nredo);
    c->h_la.resize((size_t)nredo); c->h_lb.resize((size_t)nredo);
    int rmr = 0, rmc = 0;
    long long cells = 0;
    for (size_t k = 0; k < redo.size(); ++k) {
        const int32_t xi = x0 + (int32_t)(redo[k] / ny), yi = y0 + (int32_t)(redo[k] % ny);
        px[k] = yi; py[k] = xi;
        c->h_la[k] = (int32_t)(Y.off[yi + 1] - Y.off[yi]);
        c->h_lb[k] = (int32_t)(X.off[xi + 1] - X.off[xi]);
        rmr = std::max(rmr, c->h_la[k]); rmc = std::max(rmc, c->h_lb[k]);
        cells += (long long)c->h_la[k] * c->h_lb[k];
    }
    CUDA_TRY(cudaMemcpyAsync(c->d_redo.p, redo.data(), (size_t)nredo * sizeof(long long), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(c->d_px.reserve((size_t)nredo, 1));
    CUDA_TRY(c->d_py.reserve((size_t)nredo, 1));
    CUDA_TRY(cudaMemcpyAsync(c->d_px.p, px.data(), (size_t)nredo * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaMemcpyAsync(c->d_py.p, py.data(), (size_t)nredo * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));                // the host vectors go out of scope below
    CUDA_TRY(c->d_rscore.reserve((size_t)nredo, 1));
    CUDA_TRY(c->d_rcounts.reserve((size_t)nredo * 4, 1));
    CUDA_TRY(c->d_rmetrics.reserve((size_t)nredo * 4, 1));
    AlignArgs b{};
    fill_swapped(b, c);
    b.px = c->d_px.p; b.py = c->d_py.p; b.ny = 1; b.npairs = (long long)nredo;
    b.score = c->d_rscore.p; b.counts = c->d_rcounts.p; b.metrics = c->d_rmetrics.p;
    c->cells += cells;
    if ((rc = enqueue_align(c, b, rmr, rmc))) return rc;
    scatter_redo_kernel<<<(unsigned)((nredo + 255) / 256), 256, 0, c->stream>>>(c->d_redo.p, (long long)nredo, nx, ny, c->d_rscore.p, c->d_rcounts.p,
                                                                                  c->d_rmetrics.p, a.t_score, a.t_counts, a.t_metrics);
    CUDA_TRY(cudaGetLastError());
    c->last_kernel = 20;
    return finish_align(c);
}

// Host-facing form: (x, y) results into out_* with a row stride of ld_xy pairs, (y, x) results into
// tout_* with a row stride of ld_yx pairs (so a tile and its mirror can be written straight into
// their places of one big matrix); walked in blocks of whole rows like taxi_align_rect.
int taxi_align_rect_both(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                         int32_t* out_score, int32_t* out_counts, double* out_metrics, int64_t ld_xy,
                         int32_t* tout_score, int32_t* tout_counts, double* tout_metrics, int64_t ld_yx)
{
    int rc = check_ctx(c, true);
    if (rc) return rc;
    reset_stats(c);
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    if ((long long)nx * ny == 0) return TAXI_OK;
    if (ld_xy < ny || ld_yx < nx) return fail(TAXI_E_ARG, "row strides smaller than the rows");
    ON_DEVICE(c->device);
    const int32_t rows = (int32_t)std::max<long long>(1, std::min<long long>(nx, kChunkPairs / ny));
    const long long chunk = (long long)rows * ny;
    if ((rc = reserve_outputs(c, 2 * chunk, flags))) return rc;     // second half: the mirrored block
    int64_t redo_total = 0;
    for (int32_t r0 = 0; r0 < nx; r0 += rows) {
        const int32_t nr = std::min(rows, nx - r0);
        const long long n = (long long)nr * ny;
        int32_t* ds = c->d_score.p; int32_t* dc = c->d_counts.p; double* dm = c->d_metrics.p;
        int32_t* ts = ds ? ds + chunk : nullptr; int32_t* tc = dc ? dc + 4 * chunk : nullptr; double* tm = dm ? dm + 4 * chunk : nullptr;
        if ((rc = taxi_align_rect_both_device(c, x0 + r0, nr, y0, ny, flags, ds, dc, dm, ts, tc, tm))) return rc;
        redo_total += c->last_redo;
        auto copy2d = [&](void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t height) {
            return cudaMemcpy2DAsync(dst, dpitch, src, spitch, width, height, cudaMemcpyDeviceToHost, c->stream);
        };
        if ((flags & TAXI_OUT_SCORE) && out_score) CUDA_TRY(copy2d(out_score + (size_t)r0 * ld_xy, ld_xy * 4, ds, (size_t)ny * 4, (size_t)ny * 4, nr));
        if ((flags & TAXI_OUT_COUNTS) && out_counts) CUDA_TRY(copy2d(out_counts + 4 * (size_t)r0 * ld_xy, ld_xy * 16, dc, (size_t)ny * 16, (size_t)ny * 16, nr));
        if ((flags & TAXI_OUT_METRICS) && out_metrics) CUDA_TRY(copy2d(out_metrics + 4 * (size_t)r0 * ld_xy, ld_xy * 32, dm, (size_t)ny * 32, (size_t)ny * 32, nr));
        if ((flags & TAXI_OUT_SCORE) && tout_score) CUDA_TRY(copy2d(tout_score + r0, ld_yx * 4, ts, (size_t)nr * 4, (size_t)nr * 4, ny));
        if ((flags & TAXI_OUT_COUNTS) && tout_counts) CUDA_TRY(copy2d(tout_counts + 4 * (size_t)r0, ld_yx * 16, tc, (size_t)nr * 16, (size_t)nr * 16, ny));
        if ((flags & TAXI_OUT_METRICS) && tout_metrics) CUDA_TRY(copy2d(tout_metrics + 4 * (size_t)r0, ld_yx * 32, tm, (size_t)nr * 32, (size_t)nr * 32, ny));
        CUDA_TRY(cudaStreamSynchronize(c->stream));
        (void)n;
    }
    c->last_redo = redo_total;
    return TAXI_OK;
}

int taxi_align_pairs(taxi_ctx* c, const int32_t* px, const int32_t* py, int64_t npairs, uint32_t flags,
                     int32_t* out_score, int32_t* out_counts, double* out_metrics)
{
    int rc = check_ctx(c, true);
    if (rc) return rc;
    reset_stats(c);
    if (npairs < 0 || (npairs > 0 && (!px || !py))) return fail(TAXI_E_ARG, "bad pair list");
    if (npairs == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    int mr = 0, mc = 0;
    long long cells = 0;
    if ((rc = upload_pairs(c, px, py, npairs, &mr, &mc, &cells))) return rc;
    if ((rc = range_check(c, mr, mc))) return rc;
    if ((rc = reserve_outputs(c, npairs, flags))) return rc;
    AlignArgs a{};
    fill_rect(a, c, 0, 0, 1, npairs);
    a.px = c->d_px.p; a.py = c->d_py.p;
    a.score = (flags & TAXI_OUT_SCORE) ? c->d_score.p : nullptr;
    a.counts = (flags & TAXI_OUT_COUNTS) ? c->d_counts.p : nullptr;
    a.metrics = (flags & TAXI_OUT_METRICS) ? c->d_metrics.p : nullptr;
    c->cells += cells;
    if ((rc = enqueue_align(c, a, mr, mc))) return rc;
    if ((rc = download_outputs(c, npairs, flags, out_score, out_counts, out_metrics))) return rc;
    return finish_align(c);
}

int taxi_alignment_capacity(taxi_ctx* c, const int32_t* px, const int32_t* py, int64_t npairs, int64_t* aln_offsets)
{
    int rc = check_ctx(c, false);
    if (rc) return rc;
    if (npairs < 0 || !aln_offsets || (npairs > 0 && (!px || !py))) return fail(TAXI_E_ARG, "bad argument");
    const SeqSet& X = c->set[0];
    const SeqSet& Y = yset(c);
    aln_offsets[0] = 0;
    for (int64_t k = 0; k < npairs; ++k) {
        if (px[k] < 0 || px[k] >= X.n || py[k] < 0 || py[k] >= Y.n)
            return fail(TAXI_E_ARG, "pair %lld outside the loaded sets", (long long)k);
        aln_offsets[k + 1] = aln_offsets[k] + (X.off[px[k] + 1] - X.off[px[k]]) + (Y.off[py[k] + 1] - Y.off[py[k]]);
    }
    return TAXI_OK;
}

int taxi_align_strings_metrics(taxi_ctx* c, const int32_t* px, const int32_t* py, int64_t npairs,
                               const int64_t* aln_offsets, uint8_t* out_x, uint8_t* out_y, int64_t* aln_start,
                               uint32_t flags, int32_t* out_score, int32_t* out_counts, double* out_metrics)
{
    int rc = check_ctx(c, true);
    if (rc) return rc;
    reset_stats(c);
    if (npairs < 0 || (npairs > 0 && (!px || !py || !aln_offsets || !out_x || !out_y || !aln_start)))
        return fail(TAXI_E_ARG, "bad argument");
    if (npairs == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    int mr = 0, mc = 0;
    long long cells = 0;
    if ((rc = upload_pairs(c, px, py, npairs, &mr, &mc, &cells))) return rc;
    if ((rc = range_check(c, mr, mc))) return rc;
    const int64_t total = aln_offsets[npairs];
    CUDA_TRY(c->d_alnx.reserve((size_t)total + 16));
    CUDA_TRY(c->d_alny.reserve((size_t)total + 16));
    CUDA_TRY(c->d_alnoff.reserve((size_t)npairs + 1));
    CUDA_TRY(c->d_alnstart.reserve((size_t)npairs));
    if (!out_score) flags &= ~(uint32_t)TAXI_OUT_SCORE;
    if (!out_counts) flags &= ~(uint32_t)TAXI_OUT_COUNTS;
    if (!out_metrics) flags &= ~(uint32_t)TAXI_OUT_METRICS;
    if ((rc = reserve_outputs(c, npairs, flags))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->d_alnoff.p, aln_offsets, ((size_t)npairs + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, c->stream));
    AlignArgs a{};
    fill_rect(a, c, 0, 0, 1, npairs);
    a.px = c->d_px.p; a.py = c->d_py.p;
    a.score = (flags & TAXI_OUT_SCORE) ? c->d_score.p : nullptr;
    a.counts = (flags & TAXI_OUT_COUNTS) ? c->d_counts.p : nullptr;
    a.metrics = (flags & TAXI_OUT_METRICS) ? c->d_metrics.p : nullptr;
    a.aln_x = c->d_alnx.p; a.aln_y = c->d_alny.p; a.aln_off = c->d_alnoff.p; a.aln_start = c->d_alnstart.p;
    c->cells += cells;
    if ((rc = enqueue_align(c, a, mr, mc))) return rc;
    CUDA_TRY(cudaMemcpyAsync(out_x, c->d_alnx.p, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(out_y, c->d_alny.p, (size_t)total, cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaMemcpyAsync(aln_start, c->d_alnstart.p, (size_t)npairs * sizeof(int64_t), cudaMemcpyDeviceToHost, c->stream));
    if ((rc = download_outputs(c, npairs, flags, out_score, out_counts, out_metrics))) return rc;
    return finish_align(c);
}

int taxi_align_strings(taxi_ctx* c, const int32_t* px, const int32_t* py, int64_t npairs,
                       const int64_t* aln_offsets, uint8_t* out_x, uint8_t* out_y, int64_t* aln_start,
                       int32_t* out_score)
{
    return taxi_align_strings_metrics(c, px, py, npairs, aln_offsets, out_x, out_y, aln_start,
                                      out_score ? TAXI_OUT_SCORE : 0u, out_score, nullptr, nullptr);
}

// ---- tensor-core operands of the alignment-free kernel -------------------------------------------
constexpr size_t kTcMaxOperandBytes = (size_t)8 << 30;   // per set; beyond it rectangles stay on the popcount kernel

size_t tc_operand_bytes(const SeqSet& s)
{
    const size_t Lp = (size_t)(s.W * 32 + TC_TILE - 1) / TC_TILE * TC_TILE;
    return (size_t)std::max(s.n, 1) * TC_ROW_SEGMENTS * Lp;
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int ensure_tc_operands(taxi_ctx* c, SeqSet& s)
{
    if (s.tc_built) return TAXI_OK;
    static EncodeTiledFn encode = nullptr;
    static std::mutex encode_lock;
    {
        std::lock_guard<std::mutex> guard(encode_lock);
        if (!encode) {
            void* fn = nullptr;
            cudaDriverEntryPointQueryResult qres;
            CUDA_TRY(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
            if (!fn || qres != cudaDriverEntryPointSuccess) return fail(TAXI_E_CUDA, "cuTensorMapEncodeTiled is not available in this driver");
            encode = (EncodeTiledFn)fn;
        }
    }
    s.Lp = (s.W * 32 + TC_TILE - 1) / TC_TILE * TC_TILE;
    const size_t row = (size_t)TC_ROW_SEGMENTS * s.Lp;
    CUDA_TRY(s.tcops.reserve((size_t)std::max(s.n, 1) * row, 1));
    if (s.n > 0) {
        const long long threads = (long long)s.n * (s.Lp / 4);
        tc_operands_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, c->stream>>>(s.planes.p, s.n, s.W, s.Lp, s.tcops.p);
        CUDA_TRY(cudaGetLastError());
    }
    cuuint64_t dims[2] = {(cuuint64_t)row, (cuuint64_t)std::max(s.n, 1)};
    cuuint64_t strides[1] = {(cuuint64_t)row};
    cuuint32_t estr[2] = {1, 1};
    // boxes of 128 bytes of K x 128 rows (the y role, and the x role of the one-CTA-per-SM geometry) or 64 rows (x role, two CTAs per SM)
    for (int half = 0; half < 2; ++half) {
        cuuint32_t box[2] = {(cuuint32_t)TC_TILE, (cuuint32_t)(half ? TC_TILE / 2 : TC_TILE)};
        const CUresult r = encode(half ? &s.tc_map64 : &s.tc_map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, s.tcops.p, dims, strides, box, estr,
                                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) return fail(TAXI_E_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
    }
    s.tc_built = true;
    return TAXI_OK;
}

static int enqueue_count(taxi_ctx* c, CountArgs a)
{
    const SeqSet& X = c->set[0];
    const SeqSet& Y = yset(c);
    a.x = Planes{X.planes.p, X.span.p, X.W, X.n};
    a.y = Planes{Y.planes.p, Y.span.p, Y.W, Y.n};
    // one decision per job (it depends on the loaded sets only), so every kernel and every tile of a sharded
    // job computes JC / K2P the same way
    a.lntab = (c->metric_tables && std::min(X.W, Y.W) * 32 <= LN_TABLE_COLS) ? c->lntab.p : nullptr;
    if (a.px) {
        CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
        const long long blocks = (a.npairs + 255) / 256;
        count_pairs_kernel<<<(unsigned)blocks, 256, 0, c->stream>>>(a);
        CUDA_TRY(cudaGetLastError());
        CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
        c->launches += 1;
        c->last_kernel = 8;
        return TAXI_OK;
    }
    const int W = std::min(X.W, Y.W);
    // tensor-core kernel (count_tc.cuh): rectangles of at least a few tiles whose rows fit the operand layout
    if (c->count_kernel != 1) {
        const long long tiles = (long long)((a.nx + TC_TILE - 1) / TC_TILE) * ((a.ny + TC_TILE - 1) / TC_TILE);
        const bool fits = tc_operand_bytes(X) <= kTcMaxOperandBytes && tc_operand_bytes(Y) <= kTcMaxOperandBytes &&
                          (a.nx + 63) / 64 <= 65535;
        if (fits && (c->count_kernel == 2 || tiles >= 2LL * c->sms)) {
            int rc = ensure_tc_operands(c, c->set[0]);
            if (rc == TAXI_OK && c->set[1].loaded) rc = ensure_tc_operands(c, c->set[1]);
            if (rc) return rc;
            const SeqSet& XX = c->set[0];
            const SeqSet& YY = yset(c);
            a.slab = 0;
            CountTcArgs t{a, std::min(XX.Lp, YY.Lp), XX.Lp, YY.Lp};
            if (c->tc_persistent) {
                // one CTA per SM walking a static tile list, contraction of the next tile under the epilogue of this one
                const int ntiles = ((a.ny + TC_TILE - 1) / TC_TILE) * ((a.nx + TCP_TX - 1) / TCP_TX);
                CUDA_TRY(cudaFuncSetAttribute(count_tc_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TCP_SMEM));
                CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
                count_tc_persistent_kernel<<<std::min(ntiles, c->sms), TCP_THREADS, TCP_SMEM, c->stream>>>(XX.tc_map64, YY.tc_map, t);
                CUDA_TRY(cudaGetLastError());
                CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
                c->launches += 1;
                c->last_kernel = 9;
                return TAXI_OK;
            }
            const bool wide = c->tc_tile_x == 128;
            const int tx = wide ? 128 : 64;
            dim3 grid((unsigned)(((a.ny + TC_TILE - 1) / TC_TILE) * ((a.nx + tx - 1) / tx)));   // one-dimensional: count_tc_kernel orders the tiles itself
            if (wide) CUDA_TRY(cudaFuncSetAttribute(count_tc_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcGeom<128>::SMEM));
            else CUDA_TRY(cudaFuncSetAttribute(count_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TcGeom<64>::SMEM));
            CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
            if (wide) count_tc_kernel<128><<<grid, TcGeom<128>::THREADS, TcGeom<128>::SMEM, c->stream>>>(XX.tc_map, YY.tc_map, t);
            else count_tc_kernel<64><<<grid, TcGeom<64>::THREADS, TcGeom<64>::SMEM, c->stream>>>(XX.tc_map64, YY.tc_map, t);
            CUDA_TRY(cudaGetLastError());
            CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
            c->launches += 1;
            c->last_kernel = 9;
            return TAXI_OK;
        }
        if (c->count_kernel == 2) return fail(TAXI_E_RANGE, "sequences too long for the tensor-core counting kernel");
    }
    c->last_kernel = 8;
    // x rows per block: as many as fit ~64 KB of shared memory (three blocks per SM), at most COUNT_SLAB
    const size_t row_bytes = (size_t)W * sizeof(uint4);
    if (row_bytes > 200 * 1024) return fail(TAXI_E_RANGE, "sequences too long for the alignment-free kernel (%d words per plane)", W);
    a.slab = (int32_t)std::max<size_t>(1, std::min<size_t>(COUNT_SLAB, (64 * 1024) / row_bytes));
    const size_t smem = (size_t)a.slab * row_bytes;
    CUDA_TRY(cudaFuncSetAttribute(count_rect_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    // grid.y is limited to 65535 slabs: taller rectangles go in several launches
    const int32_t rows_per_launch = 65535 * a.slab;
    CUDA_TRY(cudaEventRecord(c->ev0, c->stream));
    for (int32_t r0 = 0; r0 < a.nx; r0 += rows_per_launch) {
        CountArgs part = a;
        part.x0 = a.x0 + r0;
        part.nx = std::min(rows_per_launch, a.nx - r0);
        if (part.counts) part.counts += 4LL * r0 * a.ny;
        if (part.metrics) part.metrics += 4LL * r0 * a.ny;
        dim3 grid((unsigned)((a.ny + COUNT_TY - 1) / COUNT_TY), (unsigned)((part.nx + a.slab - 1) / a.slab));
        count_rect_kernel<<<grid, COUNT_TY, smem, c->stream>>>(part);
        CUDA_TRY(cudaGetLastError());
        c->launches += 1;
    }
    CUDA_TRY(cudaEventRecord(c->ev1, c->stream));
    return TAXI_OK;
}

int taxi_count_rect_device(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                           int32_t* d_counts, double* d_metrics)
{
    int rc = check_ctx(c, false);
    if (rc) return rc;
    c->within_held = false;
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    const long long npairs = (long long)nx * ny;
    if (npairs == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    CountArgs a{};
    a.px = a.py = nullptr; a.x0 = x0; a.y0 = y0; a.nx = nx; a.ny = ny; a.npairs = npairs;
    a.counts = (flags & TAXI_OUT_COUNTS) ? d_counts : nullptr;
    a.metrics = (flags & TAXI_OUT_METRICS) ? d_metrics : nullptr;
    // the kernels write a pair's counts with one 128-bit and its metrics with one 256-bit store
    if (((uintptr_t)a.counts & 15) || ((uintptr_t)a.metrics & 31)) return fail(TAXI_E_ARG, "d_counts must be 16-byte and d_metrics 32-byte aligned");
    return enqueue_count(c, a);
}

int taxi_count_rect(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                    int32_t* out_counts, double* out_metrics)
{
    int rc = check_ctx(c, false);
    if (rc) return rc;
    reset_stats(c);
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    const long long npairs = (long long)nx * ny;
    if (npairs == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    flags &= ~(uint32_t)TAXI_OUT_SCORE;
    const int32_t rows = (int32_t)std::max<long long>(1, std::min<long long>(nx, kCountChunkPairs / ny));
    if ((rc = reserve_outputs(c, (long long)rows * ny, flags))) return rc;
    for (int32_t r0 = 0; r0 < nx; r0 += rows) {
        const int32_t nr = std::min(rows, nx - r0);
        const long long at = (long long)r0 * ny, n = (long long)nr * ny;
        if ((rc = taxi_count_rect_device(c, x0 + r0, nr, y0, ny, flags, c->d_counts.p, c->d_metrics.p))) return rc;
        if ((rc = download_outputs(c, n, flags, nullptr, out_counts ? out_counts + 4 * at : nullptr,
                                   out_metrics ? out_metrics + 4 * at : nullptr))) return rc;
        if ((rc = finish_align(c))) return rc;
    }
    return TAXI_OK;
}

int taxi_count_pairs(taxi_ctx* c, const int32_t* px, const int32_t* py, int64_t npairs, uint32_t flags,
                     int32_t* out_counts, double* out_metrics)
{
    int rc = check_ctx(c, false);
    if (rc) return rc;
    reset_stats(c);
    if (npairs < 0 || (npairs > 0 && (!px || !py))) return fail(TAXI_E_ARG, "bad pair list");
    if (npairs == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    int mr = 0, mc = 0;
    if ((rc = upload_pairs(c, px, py, npairs, &mr, &mc, nullptr, false))) return rc;
    if ((rc = reserve_outputs(c, npairs, flags & ~TAXI_OUT_SCORE))) return rc;
    CountArgs a{};
    a.px = c->d_px.p; a.py = c->d_py.p; a.npairs = npairs; a.ny = 1;
    a.counts = (flags & TAXI_OUT_COUNTS) ? c->d_counts.p : nullptr;
    a.metrics = (flags & TAXI_OUT_METRICS) ? c->d_metrics.p : nullptr;
    if ((rc = enqueue_count(c, a))) return rc;
    if ((rc = download_outputs(c, npairs, flags & ~TAXI_OUT_SCORE, nullptr, out_counts, out_metrics))) return rc;
    return finish_align(c);
}

// the four metrics of n count tuples {same, transitions, transversions, gap columns}: the epilogue every kernel
// ends with, on its own (one thread per tuple)
__global__ void metrics_from_counts_kernel(const int32_t* __restrict__ counts, long long n, const long long* __restrict__ lntab,
                                           double* __restrict__ out)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int4 c = *reinterpret_cast<const int4*>(counts + 4 * k);
    double m[4];
    // the table covers the logarithm arguments of tuples with at most LN_TABLE_COLS compared columns
    if (lntab && c.x >= 0 && c.y >= 0 && c.z >= 0 && (long long)c.x + c.y + c.z <= LN_TABLE_COLS)
        metrics_from_counts_table(c.x, c.y, c.z, c.w, m, [&](int i) { return __ldg(lntab + i); });
    else metrics_from_counts(c.x, c.y, c.z, c.w, m);
    reinterpret_cast<double2*>(out + 4 * k)[0] = make_double2(m[0], m[1]);
    reinterpret_cast<double2*>(out + 4 * k)[1] = make_double2(m[2], m[3]);
}

int taxi_metrics_from_counts(taxi_ctx* c, const int32_t* counts, int64_t n, int32_t form, double* out_metrics)
{
    int rc = check_ctx(c, false);
    if (rc) return rc;
    c->within_held = false;
    if (n < 0 || (n > 0 && (!counts || !out_metrics)) || (form != 0 && form != 1)) return fail(TAXI_E_ARG, "bad count tuples / form");
    if (n == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    if ((rc = reserve_outputs(c, n, TAXI_OUT_COUNTS | TAXI_OUT_METRICS))) return rc;
    CUDA_TRY(cudaMemcpyAsync(c->d_counts.p, counts, (size_t)n * 4 * sizeof(int32_t), cudaMemcpyHostToDevice, c->stream));
    metrics_from_counts_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(c->d_counts.p, (long long)n, form ? c->lntab.p : nullptr, c->d_metrics.p);
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(out_metrics, c->d_metrics.p, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return TAXI_OK;
}

int taxi_argmin_rows_device(taxi_ctx* c, const double* d_metrics, int32_t nx, int32_t ny, int32_t metric,
                            int32_t* out_index_host, double* out_value_host)
{
    if (!c || !d_metrics || nx < 0 || ny <= 0 || metric < 0 || metric > 3 || !out_index_host)
        return fail(TAXI_E_ARG, "bad argument");
    c->within_held = false;
    if (nx == 0) return TAXI_OK;
    ON_DEVICE(c->device);
    CUDA_TRY(c->d_argidx.reserve((size_t)nx));
    CUDA_TRY(c->d_argval.reserve((size_t)nx));
    const int wpb = 8;
    argmin_rows_kernel<<<(nx + wpb - 1) / wpb, wpb * 32, 0, c->stream>>>(d_metrics, nx, ny, metric, c->d_argidx.p, c->d_argval.p);
    CUDA_TRY(cudaGetLastError());
    c->launches += 1;
    CUDA_TRY(cudaMemcpyAsync(out_index_host, c->d_argidx.p, (size_t)nx * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
    if (out_value_host)
        CUDA_TRY(cudaMemcpyAsync(out_value_host, c->d_argval.p, (size_t)nx * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    return TAXI_OK;
}

int taxi_best_rows(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, int32_t metric, int32_t align,
                   int32_t* out_index, double* out_metrics, int32_t* out_counts)
{
    int rc = check_ctx(c, align != 0);
    if (rc) return rc;
    reset_stats(c);
    if (metric < 0 || metric > 3 || !out_index) return fail(TAXI_E_ARG, "bad argument");
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    if (nx == 0) return TAXI_OK;
    if (ny == 0) return fail(TAXI_E_ARG, "no columns to reduce over");
    const long long chunk = align ? kChunkPairs : kCountChunkPairs;
    if (ny > chunk) return fail(TAXI_E_ARG, "too many columns for one device block (%d > %lld)", ny, chunk);
    ON_DEVICE(c->device);
    const int32_t rows = (int32_t)std::max<long long>(1, std::min<long long>(nx, chunk / ny));
    const uint32_t flags = TAXI_OUT_COUNTS | TAXI_OUT_METRICS;
    if ((rc = reserve_outputs(c, (long long)rows * ny, flags))) return rc;
    CUDA_TRY(c->d_argidx.reserve((size_t)rows));
    CUDA_TRY(c->d_bestmetrics.reserve((size_t)rows * 4));
    CUDA_TRY(c->d_bestcounts.reserve((size_t)rows * 4));
    for (int32_t r0 = 0; r0 < nx; r0 += rows) {
        const int32_t nr = std::min(rows, nx - r0);
        if (align) rc = taxi_align_rect_device(c, x0 + r0, nr, y0, ny, flags, nullptr, c->d_counts.p, c->d_metrics.p);
        else rc = taxi_count_rect_device(c, x0 + r0, nr, y0, ny, flags, c->d_counts.p, c->d_metrics.p);
        if (rc) return rc;
        const int wpb = 8;
        best_rows_kernel<<<(nr + wpb - 1) / wpb, wpb * 32, 0, c->stream>>>(c->d_metrics.p, c->d_counts.p, nr, ny, metric, y0,
                                                                            c->d_argidx.p, c->d_bestmetrics.p, c->d_bestcounts.p);
        CUDA_TRY(cudaGetLastError());
        c->launches += 1;
        CUDA_TRY(cudaMemcpyAsync(out_index + r0, c->d_argidx.p, (size_t)nr * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        if (out_metrics)
            CUDA_TRY(cudaMemcpyAsync(out_metrics + 4 * (size_t)r0, c->d_bestmetrics.p, (size_t)nr * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        if (out_counts)
            CUDA_TRY(cudaMemcpyAsync(out_counts + 4 * (size_t)r0, c->d_bestcounts.p, (size_t)nr * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        if ((rc = finish_align(c))) return rc;
    }
    return TAXI_OK;
}

int taxi_best_rows_k(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, int32_t metric, int32_t align,
                     int32_t k, int32_t* out_index, double* out_metrics, int32_t* out_counts)
{
    int rc = check_ctx(c, align != 0);
    if (rc) return rc;
    reset_stats(c);
    if (metric < 0 || metric > 3 || !out_index) return fail(TAXI_E_ARG, "bad argument");
    if (k < 1 || k > BEST_K_MAX) return fail(TAXI_E_ARG, "k = %d outside 1..%d", k, BEST_K_MAX);
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    if (nx == 0) return TAXI_OK;
    if (ny == 0) return fail(TAXI_E_ARG, "no columns to reduce over");
    const long long chunk = align ? kChunkPairs : kCountChunkPairs;
    if (ny > chunk) return fail(TAXI_E_ARG, "too many columns for one device block (%d > %lld)", ny, chunk);
    ON_DEVICE(c->device);
    // a block's selected lists (rows x k slots, k may exceed ny) stay within the block size, like its results (rows x ny pairs)
    const int32_t rows = (int32_t)std::max<long long>(1, std::min<long long>(nx, chunk / std::max(ny, k)));
    const uint32_t flags = TAXI_OUT_COUNTS | TAXI_OUT_METRICS;
    if ((rc = reserve_outputs(c, (long long)rows * ny, flags))) return rc;
    const size_t kept = (size_t)rows * k;
    CUDA_TRY(c->d_argidx.reserve(kept));
    CUDA_TRY(c->d_bestmetrics.reserve(kept * 4));
    CUDA_TRY(c->d_bestcounts.reserve(kept * 4));
    for (int32_t r0 = 0; r0 < nx; r0 += rows) {
        const int32_t nr = std::min(rows, nx - r0);
        if (align) rc = taxi_align_rect_device(c, x0 + r0, nr, y0, ny, flags, nullptr, c->d_counts.p, c->d_metrics.p);
        else rc = taxi_count_rect_device(c, x0 + r0, nr, y0, ny, flags, c->d_counts.p, c->d_metrics.p);
        if (rc) return rc;
        const int wpb = 8;
        best_k_rows_kernel<<<(nr + wpb - 1) / wpb, wpb * 32, 0, c->stream>>>(c->d_metrics.p, c->d_counts.p, nr, ny, metric, k, y0,
                                                                              c->d_argidx.p, c->d_bestmetrics.p, c->d_bestcounts.p);
        CUDA_TRY(cudaGetLastError());
        c->launches += 1;
        const size_t at = (size_t)r0 * k, n = (size_t)nr * k;
        CUDA_TRY(cudaMemcpyAsync(out_index + at, c->d_argidx.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        if (out_metrics)
            CUDA_TRY(cudaMemcpyAsync(out_metrics + 4 * at, c->d_bestmetrics.p, n * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
        if (out_counts)
            CUDA_TRY(cudaMemcpyAsync(out_counts + 4 * at, c->d_bestcounts.p, n * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        if ((rc = finish_align(c))) return rc;
    }
    return TAXI_OK;
}

int taxi_pairs_within(taxi_ctx* c, int32_t x0, int32_t nx, int32_t y0, int32_t ny, int32_t metric, int32_t align,
                      double threshold, double scale, int32_t skip_self, int64_t* out_row_ptr, int64_t* out_total)
{
    int rc = check_ctx(c, align != 0);
    if (rc) return rc;
    reset_stats(c);
    if (metric < 0 || metric > 3 || !out_row_ptr || !out_total) return fail(TAXI_E_ARG, "bad argument");
    if (std::isnan(threshold)) return fail(TAXI_E_ARG, "threshold is NaN");
    if (!std::isfinite(scale) || !(scale > 0.0)) return fail(TAXI_E_ARG, "scale %g is not finite and positive", scale);
    if (skip_self && c->set[1].loaded) return fail(TAXI_E_ARG, "skip_self needs set 0 as both sets, and set 1 is loaded");
    if ((rc = check_rect(c, x0, nx, y0, ny))) return rc;
    out_row_ptr[0] = 0;
    *out_total = 0;
    if (nx == 0) {
        c->within_total = 0;
        c->within_held = true;
        return TAXI_OK;
    }
    if (ny == 0) return fail(TAXI_E_ARG, "no columns to select from");
    const long long chunk = align ? kChunkPairs : kCountChunkPairs;
    if (ny > chunk) return fail(TAXI_E_ARG, "too many columns for one device block (%d > %lld)", ny, chunk);
    ON_DEVICE(c->device);
    const int32_t rows = (int32_t)std::max<long long>(1, std::min<long long>(nx, chunk / ny));
    const uint32_t flags = TAXI_OUT_COUNTS | TAXI_OUT_METRICS;
    if ((rc = reserve_outputs(c, (long long)rows * ny, flags))) return rc;
    CUDA_TRY(c->d_rowcnt.reserve((size_t)rows + 1));
    CUDA_TRY(c->d_rowoff.reserve((size_t)rows + 1));
    size_t scan_bytes = 0;
    CUDA_TRY(cub::DeviceScan::ExclusiveSum(nullptr, scan_bytes, c->d_rowcnt.p, c->d_rowoff.p, rows + 1, c->stream));
    CUDA_TRY(c->d_scantmp.reserve(scan_bytes));
    c->h_rowoff.resize((size_t)rows + 1);
    WithinArgs a{};
    a.ny = ny; a.metric = metric; a.threshold = threshold; a.scale = scale; a.skip_self = skip_self != 0;
    const int wpb = 8;
    int64_t total = 0;
    for (int32_t r0 = 0; r0 < nx; r0 += rows) {
        const int32_t nr = std::min(rows, nx - r0);
        if (align) rc = taxi_align_rect_device(c, x0 + r0, nr, y0, ny, flags, nullptr, c->d_counts.p, c->d_metrics.p);
        else rc = taxi_count_rect_device(c, x0 + r0, nr, y0, ny, flags, c->d_counts.p, c->d_metrics.p);
        if (rc) return rc;
        a.metrics = c->d_metrics.p; a.counts = c->d_counts.p; a.nx = nr; a.self0 = x0 + r0 - y0;
        const int grid = (nr + wpb - 1) / wpb;
        within_count_kernel<<<grid, wpb * 32, 0, c->stream>>>(a, c->d_rowcnt.p);
        CUDA_TRY(cudaGetLastError());
        // one count past the last row: the exclusive scan of nr + 1 counts ends in the block total
        CUDA_TRY(cudaMemsetAsync(c->d_rowcnt.p + nr, 0, sizeof(int32_t), c->stream));
        CUDA_TRY(cub::DeviceScan::ExclusiveSum(c->d_scantmp.p, scan_bytes, c->d_rowcnt.p, c->d_rowoff.p, nr + 1, c->stream));
        CUDA_TRY(cudaMemcpyAsync(c->h_rowoff.data(), c->d_rowoff.p, ((size_t)nr + 1) * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        c->launches += 2;
        // also completes the previous block's downloads into the held arrays before they may grow
        if ((rc = finish_align(c))) return rc;
        // a block holds at most kCountChunkPairs = 2^27 pairs, so its offsets fit in int32
        const int32_t n = c->h_rowoff[(size_t)nr];
        for (int32_t r = 0; r < nr; ++r) out_row_ptr[(size_t)r0 + r + 1] = total + c->h_rowoff[(size_t)r + 1];
        if (n > 0) {
            CUDA_TRY(c->d_argidx.reserve((size_t)n, 1));
            CUDA_TRY(c->d_bestmetrics.reserve((size_t)n * 4, 1));
            CUDA_TRY(c->d_bestcounts.reserve((size_t)n * 4, 1));
            const size_t kept = (size_t)total, need = (size_t)total + n;
            CUDA_TRY(c->h_within_idx.reserve(need, kept));
            CUDA_TRY(c->h_within_metrics.reserve(need * 4, kept * 4));
            CUDA_TRY(c->h_within_counts.reserve(need * 4, kept * 4));
            within_write_kernel<<<grid, wpb * 32, 0, c->stream>>>(a, c->d_rowoff.p, y0, c->d_argidx.p, c->d_bestmetrics.p, c->d_bestcounts.p);
            CUDA_TRY(cudaGetLastError());
            c->launches += 1;
            CUDA_TRY(cudaMemcpyAsync(c->h_within_idx.p + kept, c->d_argidx.p, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(cudaMemcpyAsync(c->h_within_metrics.p + 4 * kept, c->d_bestmetrics.p, (size_t)n * 4 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
            CUDA_TRY(cudaMemcpyAsync(c->h_within_counts.p + 4 * kept, c->d_bestcounts.p, (size_t)n * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, c->stream));
        }
        total += n;
    }
    CUDA_TRY(cudaStreamSynchronize(c->stream));
    c->within_total = total;
    c->within_held = true;
    *out_total = total;
    return TAXI_OK;
}

int taxi_pairs_within_fetch(taxi_ctx* c, int32_t* out_index, double* out_metrics, int32_t* out_counts)
{
    if (!c) return fail(TAXI_E_ARG, "null context");
    if (!c->within_held) return fail(TAXI_E_ARG, "no taxi_pairs_within result is held (a later call computed on this context, or none ran)");
    const size_t n = (size_t)c->within_total;
    if (n == 0) return TAXI_OK;
    if (!out_index) return fail(TAXI_E_ARG, "null out_index");
    std::memcpy(out_index, c->h_within_idx.p, n * sizeof(int32_t));
    if (out_metrics) std::memcpy(out_metrics, c->h_within_metrics.p, n * 4 * sizeof(double));
    if (out_counts) std::memcpy(out_counts, c->h_within_counts.p, n * 4 * sizeof(int32_t));
    return TAXI_OK;
}

void* taxi_host_alloc(int64_t bytes)
{
    void* p = nullptr;
    if (bytes <= 0) return nullptr;
    if (cudaHostAlloc(&p, (size_t)bytes, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); fail(TAXI_E_NOMEM, "cudaHostAlloc(%lld) failed", (long long)bytes); return nullptr; }
    return p;
}

void taxi_host_free(void* p) { if (p) cudaFreeHost(p); }

int taxi_set_option(taxi_ctx* c, const char* key, int value)
{
    if (!c || !key) return fail(TAXI_E_ARG, "null argument");
    if (std::strcmp(key, "force_general") == 0) { c->force_general = value; return TAXI_OK; }
    if (std::strcmp(key, "force_top") == 0) { c->force_top = value; return TAXI_OK; }
    if (std::strcmp(key, "sort_columns") == 0) { c->sort_columns = value; return TAXI_OK; }
    if (std::strcmp(key, "count_kernel") == 0) { c->count_kernel = value; return TAXI_OK; }
    if (std::strcmp(key, "metric_tables") == 0) { c->metric_tables = value; return TAXI_OK; }
    if (std::strcmp(key, "tc_persistent") == 0) { c->tc_persistent = value; return TAXI_OK; }
    if (std::strcmp(key, "tc_tile_x") == 0) {
        if (value != 64 && value != 128) return fail(TAXI_E_ARG, "tc_tile_x must be 64 or 128");
        c->tc_tile_x = value;
        return TAXI_OK;
    }
    if (std::strcmp(key, "no_coop") == 0) { c->no_coop = value; return TAXI_OK; }
    return fail(TAXI_E_ARG, "unknown option %s", key);
}

int taxi_last_kernel(taxi_ctx* c) { return c ? c->last_kernel : 0; }

int64_t taxi_last_redo(taxi_ctx* c) { return c ? c->last_redo : 0; }

int taxi_last_stats(taxi_ctx* c, int64_t* launches, int64_t* cells, double* kernel_ms)
{
    if (!c) return fail(TAXI_E_ARG, "null context");
    if (launches) *launches = c->launches;
    if (cells) *cells = c->cells;
    if (kernel_ms) *kernel_ms = c->kernel_ms;
    return TAXI_OK;
}

}  // extern "C"
