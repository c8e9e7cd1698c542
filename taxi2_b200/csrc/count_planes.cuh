// Alignment-free mode (params.pairs.align = False): per-pair same / transition / transversion /
// gap-column counts straight from pre-aligned sequences, bit-sliced.
//
// Replaces calc.seq_distances_{p,p_gaps,jukes_cantor,kimura2p} applied to the raw strings
// (reference: src/itaxotools/taxi2/distances.py:319-348, called from versus_all.py:546-552 when
// versus_all.py:522-530 skipped normalisation and alignment).
//
// The packer turns every sequence into four bit planes of 32 columns per word, stored as ONE
// uint4 per (word, sequence), sequence fastest ([W][n]), so a warp whose threads hold consecutive
// sequences fetches all four planes of a word with one coalesced 128-bit load:
//   .x = b0, .y = b1 : 2-bit nucleotide (A=00 G=01 C=10 T=11; a transition flips only b0)
//   .z = R           : "real" mask (A/C/G/T)
//   .w = G'          : gap mask ('-'), restricted to the sequence's OWN real span (first..last
//                      real column).  The distances only look at columns between the first and
//                      the last column where BOTH sequences are real; a '-' outside a sequence's
//                      own span can never lie in there, so dropping it at pack time removes the
//                      leading / trailing pad of pre-aligned rows from the per-pair work.
// Columns past a sequence's end have R = G' = 0, which is exactly "truncate to the shorter".
// W is padded to a multiple of COUNT_G words (zero words).
//
// Per pair and word: 7 LOP3 build the four column masks (both-real, transversion, transition,
// gap column).  POPC issues at 16 lanes/clk/SM on sm_100 (tools/int_peak.cu: a quarter of LOP3),
// so four popcounts per word would bound the kernel; the masks of COUNT_G = 5 consecutive words
// go through two carry-save adders per quantity first (4 LOP3) and only 3 words are popcounted
// (weights 1, 2, 2): 10.2 LOP3 + 2.4 POPC + 1.6 IADD per word, the two pipes about balanced.
// The trim rule needs no per-word bookkeeping: gap columns are counted over the whole row and the
// few that precede the first / follow the last both-real column are subtracted afterwards by a
// scan that starts at the first word where both sequences have real columns (normally it looks
// at one word per end).
#pragma once
#include "common.cuh"

namespace taxi {

constexpr int COUNT_G = 5;       // words per carry-save group

struct Planes {
    const uint4* w;      // [W][nseq]: (b0, b1, R, G') of 32 columns
    const int2* span;    // [nseq]: first / last word that holds a real column (first > last: none)
    int32_t W;           // words per sequence, a multiple of COUNT_G
    int32_t nseq;
    __device__ __forceinline__ uint4 at(int word, int seq) const { return __ldg(w + (size_t)word * nseq + seq); }
};

// one thread per (sequence, word): bytes -> raw planes (G still holds every '-').  Consecutive
// threads take consecutive sequences so the plane words are written coalesced; the byte reads of
// a warp are scattered, but this runs once per load (O(N*L)) and is not on the O(N^2) path.
__global__ void pack_planes_kernel(const uint8_t* __restrict__ bytes, const int64_t* __restrict__ off,
                                   int32_t nseq, int32_t W, uint4* __restrict__ out)
{
    const int64_t gid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t total = (int64_t)nseq * W;
    if (gid >= total) return;
    const int w = (int)(gid / nseq), seq = (int)(gid % nseq);
    const int64_t o = off[seq];
    const int len = (int)(off[seq + 1] - o);
    uint32_t b0 = 0, b1 = 0, R = 0, G = 0;
    const int base = w * 32;
#pragma unroll 4
    for (int k = 0; k < 32; ++k) {
        const int pos = base + k;
        if (pos < len) {
            const int c = base_class((int)bytes[o + pos]);
            if (c < 4) { R |= 1u << k; b0 |= (uint32_t)(c & 1) << k; b1 |= (uint32_t)(c >> 1) << k; }
            else if (c == 4) G |= 1u << k;
        }
    }
    out[(size_t)w * nseq + seq] = make_uint4(b0, b1, R, G);
}

// one thread per sequence: find its real span, clip the gap plane to it, record the span words
__global__ void clip_gaps_kernel(int32_t nseq, int32_t W, uint4* __restrict__ planes, int2* __restrict__ span)
{
    const int seq = blockIdx.x * blockDim.x + threadIdx.x;
    if (seq >= nseq) return;
    int first = -1, last = -1;   // columns
    for (int w = 0; w < W; ++w) {
        const uint32_t R = planes[(size_t)w * nseq + seq].z;
        if (R) {
            if (first < 0) first = w * 32 + __ffs(R) - 1;
            last = w * 32 + 31 - __clz(R);
        }
    }
    for (int w = 0; w < W; ++w) {
        uint4* p = planes + (size_t)w * nseq + seq;
        uint32_t keep = 0;
        if (first >= 0 && w >= first / 32 && w <= last / 32) {
            keep = 0xffffffffu;
            if (w == first / 32) keep &= 0xffffffffu << (first % 32);
            if (w == last / 32) keep &= 0xffffffffu >> (31 - last % 32);
        }
        const uint32_t G = p->w;
        if ((G & keep) != G) p->w = G & keep;
    }
    span[seq] = first < 0 ? make_int2(W, -1) : make_int2(first / 32, last / 32);
}

struct CountArgs {
    Planes x, y;
    const int32_t* px; const int32_t* py;   // explicit list or nullptr (rect)
    int32_t x0, y0, nx, ny;
    int32_t slab;                           // rect mode: x rows staged in shared memory per block (<= COUNT_SLAB)
    long long npairs;
    int32_t* counts;   // [npairs][4] or nullptr
    double* metrics;   // [npairs][4] or nullptr
    const long long* lntab;   // ln k in fixed point (common.cuh: metrics_from_counts_table) or nullptr: floating-point form
};

// carry-save adder over three bit vectors: s = bit sum, c = carries (weight 2)
__device__ __forceinline__ void csa(uint32_t& s, uint32_t& c, uint32_t a, uint32_t b, uint32_t d)
{
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(s) : "r"(a), "r"(b), "r"(d));
    asm("lop3.b32 %0, %1, %2, %3, 0xE8;" : "=r"(c) : "r"(a), "r"(b), "r"(d));
}

// popcount of five mask words with three POPCs: ones += popc(s2); twos += popc(c1) + popc(c2)
__device__ __forceinline__ void add5(int& ones, int& twos, const uint32_t m[COUNT_G])
{
    uint32_t s1, c1, s2, c2;
    csa(s1, c1, m[0], m[1], m[2]);
    csa(s2, c2, s1, m[3], m[4]);
    ones += __popc(s2);
    twos += __popc(c1) + __popc(c2);
}

// unweighted partial counts of one pair: value = ones + 2 * twos
struct CountAcc {
    int n1, n2, v1, v2, s1, s2, g1, g2;   // both-real, transversions, transitions, gap columns
    __device__ __forceinline__ void init() { n1 = n2 = v1 = v2 = s1 = s2 = g1 = g2 = 0; }
    __device__ __forceinline__ void group(const uint4 x[COUNT_G], const uint4 y[COUNT_G])
    {
        uint32_t both[COUNT_G], tv[COUNT_G], ts[COUNT_G], gp[COUNT_G];
#pragma unroll
        for (int k = 0; k < COUNT_G; ++k) {
            const uint32_t d0 = x[k].x ^ y[k].x, d1 = x[k].y ^ y[k].y;
            both[k] = x[k].z & y[k].z;
            tv[k] = both[k] & d1;
            ts[k] = both[k] & d0 & ~d1;
            gp[k] = (x[k].w & y[k].z) | (x[k].z & y[k].w);
        }
        add5(n1, n2, both);
        add5(v1, v2, tv);
        add5(s1, s2, ts);
        add5(g1, g2, gp);
    }
};

// Gap columns that lie before the first / after the last both-real column of a pair (they were
// counted with the rest and do not belong to the distance).  `xat(w)` / `yat(w)` fetch a word.
template <class FX, class FY>
__device__ __forceinline__ int gaps_outside_trim(FX xat, FY yat, int2 sx, int2 sy)
{
    const int w0 = max(sx.x, sy.x), w1 = min(sx.y, sy.y);   // no both-real column outside [w0, w1]
    int out = 0;
    for (int w = w0; w <= w1; ++w) {
        const uint4 x = xat(w), y = yat(w);
        const uint32_t both = x.z & y.z, g = (x.w & y.z) | (x.z & y.w);
        if (both) { out += __popc(g & ((both & (0u - both)) - 1u)); break; }   // below the lowest both-real bit
        out += __popc(g);
    }
    for (int w = w1; w >= w0; --w) {
        const uint4 x = xat(w), y = yat(w);
        const uint32_t both = x.z & y.z, g = (x.w & y.z) | (x.z & y.w);
        if (both) { out += __popc(g & ~(0xffffffffu >> __clz(both))); break; }      // above the highest both-real bit
        out += __popc(g);
    }
    // words < w0 and > w1: one of the two sequences has no real column there, and its clipped gap
    // plane is empty outside its span, so neither term of the gap mask can be set
    return out;
}

// shared_tab: the table staged in shared memory by the caller (tensor-core kernels, STAGED: they never read it
// through L1, and leaving that path out keeps their unrolled epilogues a third smaller), else it is read through L1
template <bool STAGED = false>
__device__ __forceinline__ void store_pair(const CountArgs& a, long long p, int n, int tv, int ts, int gap, const long long* shared_tab = nullptr)
{
    const int same = n - tv - ts;
    if (a.counts) __stcs(reinterpret_cast<int4*>(a.counts + 4 * p), make_int4(same, ts, tv, gap));   // streamed out once
    if (a.metrics) {
        double m[4];
        if (shared_tab) metrics_from_counts_table(same, ts, tv, gap, m, [&](int k) { return shared_tab[k]; });
        else if (!STAGED && a.lntab) metrics_from_counts_table(same, ts, tv, gap, m, [&](int k) { return __ldg(a.lntab + k); });
        else metrics_from_counts(same, ts, tv, gap, m);
        // one 256-bit store per pair (STG.256, sm_100): every lane writes a whole 32-byte sector.  Results stream
        // out once, gigabytes per launch: evict-first in L2, so that they do not push out the operand rows / planes
        // every tile re-reads (the policy exists for 256-bit stores only)
        asm volatile("st.global.L1::no_allocate.L2::evict_first.v4.f64 [%0], {%1, %2, %3, %4};" :: "l"(a.metrics + 4 * p), "d"(m[0]), "d"(m[1]), "d"(m[2]), "d"(m[3]) : "memory");
    }
}

// Rectangle mode.  A block owns COUNT_TY consecutive y columns (one per thread) and walks the x
// rows of its slab in register tiles of COUNT_RX: the y words of a thread are loaded once per
// tile and word group (coalesced 128-bit loads) and reused for COUNT_RX pairs whose x words come
// from shared memory as 128-bit warp broadcasts.  Results are written coalesced, 16 B + 32 B per pair.
constexpr int COUNT_TY = 256;
constexpr int COUNT_RX = 4;
constexpr int COUNT_SLAB = 64;   // x rows staged in shared memory per block (fewer when the sequences are long)

__global__ void __launch_bounds__(COUNT_TY, 3) count_rect_kernel(const CountArgs a)
{
    extern __shared__ uint4 xs[];   // [slab][W]
    const int W = min(a.x.W, a.y.W);
    const int yj = blockIdx.x * COUNT_TY + threadIdx.x;          // column inside the rectangle
    const int xbase = blockIdx.y * a.slab;                       // first row of the slab
    const int rows = min(a.slab, a.nx - xbase);
    for (int k = threadIdx.x; k < rows * W; k += COUNT_TY) {
        const int r = k / W, w = k % W;
        xs[k] = a.x.at(w, a.x0 + xbase + r);
    }
    __syncthreads();
    if (yj >= a.ny) return;
    const int ys = a.y0 + yj;
    const int2 sy = __ldg(a.y.span + ys);
    for (int g = 0; g < rows; g += COUNT_RX) {
        CountAcc acc[COUNT_RX];
#pragma unroll
        for (int k = 0; k < COUNT_RX; ++k) acc[k].init();
        for (int w = 0; w < W; w += COUNT_G) {
            uint4 y[COUNT_G];
#pragma unroll
            for (int q = 0; q < COUNT_G; ++q) y[q] = a.y.at(w + q, ys);
#pragma unroll
            for (int k = 0; k < COUNT_RX; ++k) {
                // rows past the slab's end repeat its last row (discarded below): no branch in the hot loop
                const uint4* xw = xs + (size_t)min(g + k, rows - 1) * W + w;
                uint4 x[COUNT_G];
#pragma unroll
                for (int q = 0; q < COUNT_G; ++q) x[q] = xw[q];
                acc[k].group(x, y);
            }
        }
#pragma unroll
        for (int k = 0; k < COUNT_RX; ++k) {
            if (g + k >= rows) break;
            const CountAcc& c = acc[k];
            const int n = c.n1 + 2 * c.n2;
            int gap = c.g1 + 2 * c.g2;
            const int row = xbase + g + k;
            if (n > 0 && gap > 0) {
                const uint4* xw = xs + (size_t)(g + k) * W;
                gap -= gaps_outside_trim([&](int w) { return xw[w]; }, [&](int w) { return a.y.at(w, ys); },
                                         __ldg(a.x.span + a.x0 + row), sy);
            }
            store_pair(a, (long long)row * a.ny + yj, n, c.v1 + 2 * c.v2, c.s1 + 2 * c.s2, n > 0 ? gap : 0);
        }
    }
}

// Explicit pair list: one thread per pair.
__global__ void __launch_bounds__(256) count_pairs_kernel(const CountArgs a)
{
    const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= a.npairs) return;
    const int xi = a.px[p], yi = a.py[p];
    const int W = min(a.x.W, a.y.W);
    CountAcc c;
    c.init();
    for (int w = 0; w < W; w += COUNT_G) {
        uint4 x[COUNT_G], y[COUNT_G];
#pragma unroll
        for (int q = 0; q < COUNT_G; ++q) { x[q] = a.x.at(w + q, xi); y[q] = a.y.at(w + q, yi); }
        c.group(x, y);
    }
    const int n = c.n1 + 2 * c.n2;
    int gap = c.g1 + 2 * c.g2;
    if (n > 0 && gap > 0) {
        // spans may reach past the shorter set's width: clamp to the common words
        int2 sx = __ldg(a.x.span + xi), sy = __ldg(a.y.span + yi);
        sx.y = min(sx.y, W - 1); sy.y = min(sy.y, W - 1);
        gap -= gaps_outside_trim([&](int w) { return a.x.at(w, xi); }, [&](int w) { return a.y.at(w, yi); }, sx, sy);
    }
    store_pair(a, p, n, c.v1 + 2 * c.v2, c.s1 + 2 * c.s2, n > 0 ? gap : 0);
}

// versus_reference.py:184-188 / decontaminate.py:258-264: first minimum per query row, NaN skipped.
// One warp per row; ties resolve to the smallest column index.
__global__ void argmin_rows_kernel(const double* __restrict__ metrics, int32_t nx, int32_t ny, int32_t metric,
                                   int32_t* __restrict__ out_idx, double* __restrict__ out_val)
{
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= nx) return;
    double best = __longlong_as_double(0x7ff0000000000000LL);  // +inf
    int bidx = 0x7fffffff;
    for (int c = lane; c < ny; c += 32) {
        const double v = metrics[((size_t)row * ny + c) * 4 + metric];
        if (v == v && (v < best || (v == best && c < bidx))) { best = v; bidx = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_down_sync(TAXI_FULL_MASK, best, o);
        const int oi = __shfl_down_sync(TAXI_FULL_MASK, bidx, o);
        if (oi != 0x7fffffff && (bidx == 0x7fffffff || ov < best || (ov == best && oi < bidx))) { best = ov; bidx = oi; }
    }
    if (lane == 0) {
        out_idx[row] = (bidx == 0x7fffffff) ? -1 : bidx;
        out_val[row] = (bidx == 0x7fffffff) ? __longlong_as_double(0x7ff8000000000000LL) : best;
    }
}

// Same reduction, returning the whole winning pair: index (offset by col0, -1 = no defined
// distance in the row), its four metrics and its four counts -- what VersusReference needs per
// query (versus_reference.py:119-129,184-188), so the nx x ny matrix never leaves the device.
__global__ void best_rows_kernel(const double* __restrict__ metrics, const int32_t* __restrict__ counts, int32_t nx, int32_t ny,
                                 int32_t metric, int32_t col0, int32_t* __restrict__ out_idx, double* __restrict__ out_metrics,
                                 int32_t* __restrict__ out_counts)
{
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= nx) return;
    double best = __longlong_as_double(0x7ff0000000000000LL);  // +inf
    int bidx = 0x7fffffff;
    for (int c = lane; c < ny; c += 32) {
        const double v = metrics[((size_t)row * ny + c) * 4 + metric];
        if (v == v && (v < best || (v == best && c < bidx))) { best = v; bidx = c; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const double ov = __shfl_xor_sync(TAXI_FULL_MASK, best, o);
        const int oi = __shfl_xor_sync(TAXI_FULL_MASK, bidx, o);
        if (oi != 0x7fffffff && (bidx == 0x7fffffff || ov < best || (ov == best && oi < bidx))) { best = ov; bidx = oi; }
    }
    const bool none = bidx == 0x7fffffff;
    if (lane == 0) out_idx[row] = none ? -1 : col0 + bidx;
    if (lane < 4) {
        const size_t at = ((size_t)row * ny + (none ? 0 : bidx)) * 4 + lane;
        out_metrics[(size_t)row * 4 + lane] = none ? __longlong_as_double(0x7ff8000000000000LL) : metrics[at];
        if (counts && out_counts) out_counts[(size_t)row * 4 + lane] = none ? 0 : counts[at];
    }
}

// The k closest references of every query: per row the k smallest keys (value of metric column
// `metric`, column index) in ascending order -- for k = 1 the winner of best_rows_kernel.  NaN is
// never ranked; a row with fewer than k defined values ends in slots of index -1, NaN metrics and
// zero counts.  Out: [nx][k] indices (offset by col0), [nx][k][4] metrics and counts.
//
// One warp per row.  The sorted list lives in registers: lane l holds slots l and 32 + l (the
// second only when k > 32), empty slots (+inf, BEST_K_NONE), above every real key.  tau is the
// k-th key.  The warp reads BEST_K_STEPS x 32 columns at a time (loads in flight together), a
// ballot per 32 picks the lanes whose key is below tau, and each of those few is inserted by the
// whole warp: a rank from one ballot per slot set, a shift by one lane, tau re-read.  After the
// first k columns of a barcode row insertions are rare.  The key is a total order, so the list
// does not depend on the order in which candidates arrive.  No shared memory at any k; 46
// registers (sm_100a) allow 40 of 64 warps per SM, and capping them at 32 spills.
constexpr int BEST_K_MAX = 64;
constexpr int BEST_K_STEPS = 4;
constexpr int BEST_K_NONE = 0x7fffffff;

__device__ __forceinline__ bool key_less(double v, int c, double tv, int tc) { return v < tv || (v == tv && c < tc); }

__global__ void best_k_rows_kernel(const double* __restrict__ metrics, const int32_t* __restrict__ counts, int32_t nx, int32_t ny,
                                   int32_t metric, int32_t k, int32_t col0, int32_t* __restrict__ out_idx,
                                   double* __restrict__ out_metrics, int32_t* __restrict__ out_counts)
{
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= nx) return;
    const double inf = __longlong_as_double(0x7ff0000000000000LL), nan = __longlong_as_double(0x7ff8000000000000LL);
    const bool two = k > 32;                  // warp-uniform: the second slot set is in use
    double v0 = inf, v1 = inf;
    int c0 = BEST_K_NONE, c1 = BEST_K_NONE;
    double tv = inf;
    int tc = BEST_K_NONE;
    const double* m = metrics + (size_t)row * ny * 4 + metric;
    for (int base = 0; base < ny; base += 32 * BEST_K_STEPS) {
        double v[BEST_K_STEPS];
#pragma unroll
        for (int u = 0; u < BEST_K_STEPS; ++u) {
            const int c = base + 32 * u + lane;
            v[u] = c < ny ? m[(size_t)c * 4] : nan;
        }
#pragma unroll
        for (int u = 0; u < BEST_K_STEPS; ++u) {
            const int first = base + 32 * u;
            unsigned cand = __ballot_sync(TAXI_FULL_MASK, v[u] == v[u] && key_less(v[u], first + lane, tv, tc));
            while (cand) {
                const int src = __ffs(cand) - 1;
                cand &= cand - 1;
                const double cv = __shfl_sync(TAXI_FULL_MASK, v[u], src);
                const int cc = first + src;
                if (!key_less(cv, cc, tv, tc)) continue;      // tau has fallen since the ballot
                int pos = __popc(__ballot_sync(TAXI_FULL_MASK, key_less(v0, c0, cv, cc)));
                if (two) pos += __popc(__ballot_sync(TAXI_FULL_MASK, key_less(v1, c1, cv, cc)));
                // slot s takes slot s - 1 above the new key's rank
                const double u0 = __shfl_up_sync(TAXI_FULL_MASK, v0, 1);
                const int d0 = __shfl_up_sync(TAXI_FULL_MASK, c0, 1);
                if (two) {
                    const double top = __shfl_sync(TAXI_FULL_MASK, v0, 31);
                    const int ctop = __shfl_sync(TAXI_FULL_MASK, c0, 31);
                    const double u1 = __shfl_up_sync(TAXI_FULL_MASK, v1, 1);
                    const int d1 = __shfl_up_sync(TAXI_FULL_MASK, c1, 1);
                    const int s = 32 + lane;
                    if (s == pos) { v1 = cv; c1 = cc; }
                    else if (s > pos) { v1 = lane ? u1 : top; c1 = lane ? d1 : ctop; }
                }
                if (lane == pos) { v0 = cv; c0 = cc; }
                else if (lane > pos) { v0 = u0; c0 = d0; }
                const int kl = (k - 1) & 31;
                tv = __shfl_sync(TAXI_FULL_MASK, two ? v1 : v0, kl);
                tc = __shfl_sync(TAXI_FULL_MASK, two ? c1 : c0, kl);
            }
        }
    }
    const size_t o = (size_t)row * k;
    if (lane < k) out_idx[o + lane] = c0 == BEST_K_NONE ? -1 : col0 + c0;
    if (lane + 32 < k) out_idx[o + 32 + lane] = c1 == BEST_K_NONE ? -1 : col0 + c1;
    // the winners' four metrics and counts: 8 slots x 4 values per pass, one row's output written contiguously
    for (int t0 = 0; t0 < 4 * k; t0 += 32) {
        const int t = t0 + lane, s = t >> 2;
        const int c = __shfl_sync(TAXI_FULL_MASK, t0 >= 128 ? c1 : c0, s & 31);   // slots of one pass share a set
        if (t >= 4 * k) continue;
        const bool none = c == BEST_K_NONE;
        const size_t at = ((size_t)row * ny + (none ? 0 : c)) * 4 + (t & 3);
        out_metrics[4 * o + t] = none ? nan : metrics[at];
        if (counts && out_counts) out_counts[4 * o + t] = none ? 0 : counts[at];
    }
}

// Pairs within a distance (taxi_pairs_within): column c of row r is selected iff its value v of
// metric column `metric` satisfies v * scale <= threshold -- one fp64 multiply, then the compare, so
// NaN is never selected -- and, with skip_self, c is not the row's own column r + self0.  Two
// passes over the block compact the selection into CSR in row-major pair order: within_count_kernel
// counts per row, an exclusive scan of the counts gives every row its first slot, and
// within_write_kernel writes each selected pair there.  No atomics: the output is deterministic.
struct WithinArgs {
    const double* metrics;   // [nx][ny][4] of the device block
    const int32_t* counts;   // [nx][ny][4]
    int32_t nx, ny, metric;
    double threshold, scale;
    int32_t self0;           // skip_self: row r's own column is r + self0
    int32_t skip_self;
};

constexpr int WITHIN_STEPS = 4;   // 32-column strides of the metric column in flight per warp

__device__ __forceinline__ bool within_pair(const WithinArgs& a, double v, int c, int self)
{
    return v * a.scale <= a.threshold && c != self;
}

// One warp per row, WITHIN_STEPS x 32 columns per iteration (the loads issued together); a ballot
// per 32 columns, counted with popc.  row_count[r] = selected columns of row r.
__global__ void within_count_kernel(const WithinArgs a, int32_t* __restrict__ row_count)
{
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= a.nx) return;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const double* m = a.metrics + (size_t)row * a.ny * 4 + a.metric;
    const int self = a.skip_self ? row + a.self0 : -1;
    int n = 0;
    for (int base = 0; base < a.ny; base += 32 * WITHIN_STEPS) {
        double v[WITHIN_STEPS];
#pragma unroll
        for (int u = 0; u < WITHIN_STEPS; ++u) {
            const int c = base + 32 * u + lane;
            v[u] = c < a.ny ? m[(size_t)c * 4] : nan;
        }
#pragma unroll
        for (int u = 0; u < WITHIN_STEPS; ++u)
            n += __popc(__ballot_sync(TAXI_FULL_MASK, within_pair(a, v[u], base + 32 * u + lane, self)));
    }
    if (lane == 0) row_count[row] = n;
}

// One warp per row again, same reads.  Row r's pairs go to slots row_off[r] .. row_off[r + 1]: per
// 32 columns one ballot, and a selected lane's slot is the row's running offset plus the selected
// lanes below it.  Each selected pair writes its column (offset by col0), its four metrics as one
// 256-bit store and its four counts as one 128-bit store.  A row stops reading once its last slot
// is written.
__global__ void within_write_kernel(const WithinArgs a, const int32_t* __restrict__ row_off, int32_t col0,
                                    int32_t* __restrict__ out_idx, double* __restrict__ out_metrics,
                                    int32_t* __restrict__ out_counts)
{
    const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= a.nx) return;
    const double nan = __longlong_as_double(0x7ff8000000000000LL);
    const double* m = a.metrics + (size_t)row * a.ny * 4 + a.metric;
    const int self = a.skip_self ? row + a.self0 : -1;
    const unsigned below = (1u << lane) - 1u;
    int at = row_off[row];
    const int end = row_off[row + 1];
    for (int base = 0; base < a.ny && at < end; base += 32 * WITHIN_STEPS) {
        double v[WITHIN_STEPS];
#pragma unroll
        for (int u = 0; u < WITHIN_STEPS; ++u) {
            const int c = base + 32 * u + lane;
            v[u] = c < a.ny ? m[(size_t)c * 4] : nan;
        }
#pragma unroll
        for (int u = 0; u < WITHIN_STEPS; ++u) {
            const int c = base + 32 * u + lane;
            const bool sel = within_pair(a, v[u], c, self);
            const unsigned mask = __ballot_sync(TAXI_FULL_MASK, sel);
            if (sel) {
                const size_t slot = (size_t)at + __popc(mask & below);
                const size_t p = (size_t)row * a.ny + c;
                out_idx[slot] = col0 + c;
                double r0, r1, r2, r3;
                asm volatile("ld.global.nc.v4.f64 {%0, %1, %2, %3}, [%4];" : "=d"(r0), "=d"(r1), "=d"(r2), "=d"(r3) : "l"(a.metrics + 4 * p));
                asm volatile("st.global.L1::no_allocate.L2::evict_first.v4.f64 [%0], {%1, %2, %3, %4};" :: "l"(out_metrics + 4 * slot), "d"(r0), "d"(r1), "d"(r2), "d"(r3) : "memory");
                __stcs(reinterpret_cast<int4*>(out_counts + 4 * slot), __ldg(reinterpret_cast<const int4*>(a.counts + 4 * p)));
            }
            at += __popc(mask);
        }
    }
}

}  // namespace taxi
