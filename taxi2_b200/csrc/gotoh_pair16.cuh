// Fast path of the global affine-gap aligner: packed 16-bit DP, TWO pairs per warp.
//
// Same results as gotoh_warp.cuh (Biopython's first alignment + fused distance counts), for the
// score sets and lengths where three simplifications are provably exact (checked on the host in
// taxi_abi.cu: fast16_eligible()):
//
//  1. 16-bit cells.  Each 32-bit register holds the same DP cell of two different pairs (low
//     half = pair A, high half = pair B), so every VIMNMX3/VIADDMNMX (.U16x2) advances two
//     cells.  Values are kept unsigned below a bias near the top of the 16-bit range, in the
//     transformed score space S' = S - match*i: a matching column costs 0, a mismatch
//     match-mismatch, a vertical gap step match-g, a horizontal one -g -- every step is a
//     non-negative penalty, the value of a perfect match stays at the bias, and plain 32-bit
//     subtractions never borrow between the halves.  Anchoring the maximum (instead of the
//     mismatch) keeps the window at ~2*max(len) score units, so sequences up to ~1 800 bp fit.
//  2. Restricted recurrence.  When no co-optimal path can contain a vertical gap adjacent to a
//     horizontal one (true for TaxI2's default scores; the host proves it per score set), the
//     Ix<->Iy transitions of Biopython's recurrence can be dropped without changing the first
//     alignment.  Ix and Iy then have two candidate predecessors instead of three.
//  3. Tagged maxima with disjoint tag fields: candidates of H carry their priority in bits 0-1,
//     the M-candidate of Ix sets bit 2, the M-candidate of Iy sets bit 3.  Ties resolve in
//     Biopython's order (M before Ix before Iy) inside the max itself, and the 4-bit trace code
//     of a cell is a single three-input OR of the values that arrive at it.
//
// Rows = x (<= 32*H, single stripe), lane l owns rows [l*H, l*H+H); columns stream one per step.
#pragma once
#include <type_traits>

#include "common.cuh"

namespace taxi {

constexpr uint32_t F16_CLEAN = 0xFFF0FFF0u;

__device__ __forceinline__ uint32_t pack16(uint32_t lo, uint32_t hi) { return (lo & 0xFFFFu) | (hi << 16); }

__device__ __forceinline__ uint32_t lop3_or3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xFE;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

__device__ __forceinline__ uint32_t lop3_xor_or(uint32_t a, uint32_t b, uint32_t c)
{
    // (a ^ b) | c : (0xF0 ^ 0xCC) | 0xAA = 0xBE
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xBE;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

__device__ __forceinline__ uint32_t lop3_xor3(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0x96;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

// bits of a where c is set, bits of b elsewhere: (0xF0 & 0xAA) | (0xCC & 0x55) = 0xE4
__device__ __forceinline__ uint32_t lop3_mux(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(r) : "r"(a), "r"(b), "r"(c));
    return r;
}

__device__ __forceinline__ uint32_t lop3_and_or(uint32_t a, uint32_t mask, uint32_t c)
{
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xEA;" : "=r"(r) : "r"(a), "r"(mask), "r"(c));
    return r;
}

// Row symbol codes of the two pairs as diag_candidate() wants them: (-code) mod 2^16 per half
// (low half = pair A, high half = pair B).
__device__ __forceinline__ uint32_t row_codes(uint32_t c0, uint32_t c1) { return pack16(0u - c0, 0u - c1); }

// Diagonal candidate of a cell: H(i-1, j-1) minus the mismatch penalty, for both pairs at once.
// na2 holds the negated row codes (row_codes()), b2 the column codes, pair A in the low half and
// pair B in the high half.  The packed add of VIADDMNMX.U16x2 wraps per half, so na + b is zero
// exactly where the codes agree, and min(na + b, 1) is the 0 / 1 mismatch flag in one alu
// instruction (min(a ^ b, 1) before: LOP3 + VIMNMX, 2.3 % slower on C3).  One IMAD
// folds the multiplication by the penalty into the subtraction -- it runs on the fma pipe, off the
// alu pipe that bounds this kernel, and off the row-to-row dependency chain.  Works for any of the
// 16 symbol codes and any penalty.
__device__ __forceinline__ uint32_t diag_candidate(uint32_t Hd, uint32_t na2, uint32_t b2, uint32_t negD)
{
    const uint32_t ne = __viaddmin_u16x2(na2, b2, 0x00010001u);
    return ne * negD + Hd;
}

template <int H, bool SYM = false> struct Pair16Geom {
    static constexpr int WORDS = (H + 1) / 2;                 // trace words per (lane, step): 2 rows x 2 pairs each
    // SYM: one more word, the "no orientation-sensitive tie" bits of the lane's row groups (one bit per two rows
    // and pair; for H = 21 it takes the padding the 16-byte alignment leaves anyway)
    static constexpr int HB = ((WORDS + (SYM ? 1 : 0)) * 4 + 15) / 16 * 16;     // bytes per (lane, step)
    static constexpr int GROUPS = (H + 1) / 2;                // SYM: row groups per lane (bit GROUPS-1-q of a half = group q)
};

// Warp-parallel first-path traceback over the 4-bit codes.  An iteration looks at the next 32
// cells the path would visit if it stayed in its state (diagonal for M, one row / one column for
// Ix / Iy), follows it to the first cell that hands over to another state, and accounts for the
// cells visited.  The walks of the two pairs a warp has just aligned advance in lockstep: both
// windows' loads are issued before either is consumed.
//
// The walk is the only serial part of a pair and every one of its instructions competes with the
// DP loops of the two other warps of the scheduler (DESIGN.md 3.2: skipping it is worth 10 %), so
// it is written for instruction count: symbol codes and a class table instead of ASCII
// classification, per-lane partial counts that are summed once at the end, window validity from
// (i, j) instead of a ballot, and the gap-column bookkeeping reduced to what the state allows.
// (Measured and dropped: fetching the two neighbouring diagonals so that one-column gaps stay in
// one iteration -- 41 -> 25 iterations per 650 bp pair, same speed; prefetching the next
// straight-ahead window -- 2 % slower.)
struct Walk {
    const uint8_t* x; const uint8_t* y;   // symbol codes of the two sequences
    long long p;                          // pair index (outputs)
    int i, j, state;                      // current cell and state (0 = M, 1 = Ix, 2 = Iy)
    int half, off;                        // which 16-bit half of the arena; row -> slot offset
    int stride;                           // steps per stripe in the arena (multi-stripe kernel)
    int n, same, ts;                      // per-lane partial counts (both-real, identical, transitions)
    int gapc, pend;                       // warp-uniform: gap columns inside / after the both-real span so far
    bool seen;
    bool sens;                            // SYM: a tie between Ix and Iy was decided on the path: (y, x) may align differently
    int64_t wpos;                         // write cursor of the gapped strings
    int score;
    int tb, ca, cb;                       // the window element this lane holds: traceback code, x / y symbol codes
    bool entered;                         // SYM: the current cell was entered in its H state (start, or after a diagonal move)
};

// address of the traceback code of cell (ii, jj); MULTI = arena with several stripes
template <int H, bool MULTI, bool SYM = false>
__device__ __forceinline__ const uint8_t* trace_addr(const Walk& w, const uint8_t* trace, int l0, int ii, int jj)
{
    constexpr int HB = Pair16Geom<H, SYM>::HB;
    const int slot = w.off + ii - 1;   // row -> register slot (top-aligned: off = 0)
    int st = 0, q = slot;
    if (MULTI) { st = slot / (32 * H); q = slot % (32 * H); }
    const int l = q / H, r = q % H;
    const int first = (st == 0) ? l0 : 0;                  // only the first stripe starts at a later lane
    return trace + ((size_t)(st * w.stride + jj - 1 + l - first) * 32 + l) * HB + 2 * r + w.half;
}

template <int H, bool MULTI, bool SYM = false>
__device__ __forceinline__ void walk_fetch(const AlignArgs& a, Walk& w, int lane, const uint8_t* trace, int l0)
{
    const int di = (w.state != 2), dj = (w.state != 1);
    const int ii = w.i - lane * di, jj = w.j - lane * dj;
    w.tb = 0; w.ca = 0; w.cb = 0;
    if (SYM && w.entered && w.state == 1 && w.i > 0 && w.j > 0) {
        // Orientation.  The path of (y, x) is the transpose of this one unless the winner of H at a cell the
        // path enters in its H state (the end cell, the cell after every diagonal move) is Ix with Iy at the
        // same score: Biopython prefers Ix; transposed, the roles swap.  The aligner left one bit per group of
        // two rows, lane and column: clear if such a tie exists in the group (warp-uniform, rare: one load).
        constexpr int HB = Pair16Geom<H, true>::HB, WORDS = Pair16Geom<H, true>::WORDS, GROUPS = Pair16Geom<H, true>::GROUPS;
        const int slot = w.off + w.i - 1, l = slot / H, r = slot % H;
        const uint8_t* at = trace + ((size_t)(w.j - 1 + l - l0) * 32 + l) * HB + 4 * WORDS;
        TAXI_CHECK(a, at >= trace && at + 4 <= trace + a.trace_per_warp, 6);
        const uint32_t bits = __ldcg(reinterpret_cast<const uint32_t*>(at));
        if (!((bits >> (16 * w.half + GROUPS - 1 - (r >> 1))) & 1u)) w.sens = true;
    }
    if (w.i > 0 && w.j > 0 && ii >= 1 && jj >= 1) {
        const uint8_t* at = trace_addr<H, MULTI, SYM>(w, trace, l0, ii, jj);
        TAXI_CHECK(a, at >= trace && at < trace + a.trace_per_warp, 1);
        w.tb = (int)__ldcg(at);
        w.ca = (int)__ldg(w.x + ii - 1);
        w.cb = (int)__ldg(w.y + jj - 1);
    }
}

template <bool SYM = false>
__device__ __forceinline__ void walk_advance(Walk& w, const AlignArgs& a, int lane)
{
    if (!(w.i > 0 && w.j > 0)) return;   // warp-uniform
    const int state = w.state, tb = w.tb;
    const int di = (state != 2), dj = (state != 1);
    // cells of the window that exist: a prefix of the lanes
    const int nvalid = min(32, min(di ? w.i : 32, dj ? w.j : 32));
    // state I would hand over to if the path reaches my cell in `state`
    int ns;
    if (state == 0) ns = 3 - (tb & 3);            // 3 -> M, 2 -> Ix, 1 -> Iy
    else if (state == 1) ns = (tb & 4) ? 0 : 1;   // Ix: opened from M, or extended
    else ns = (tb & 8) ? 0 : 2;                   // Iy
    const unsigned cont = __ballot_sync(TAXI_FULL_MASK, ns == state);
    const int V = min(__ffs(~cont | 0x80000000u), nvalid);   // cells visited: up to and including the first hand-over
    const int next = __shfl_sync(TAXI_FULL_MASK, ns, V - 1);
    if (SYM) w.entered = (state == 0);   // the next cell is entered in its H state after a diagonal move (walk_fetch looks)
    const bool mine = lane < V;
    const unsigned visited = 0xffffffffu >> (32 - V);
    const Fast16& f = a.f16;
    if (state == 0) {
        const int ka = code_class(f, w.ca), kb = code_class(f, w.cb);
        const bool both = (ka | kb) < 4;
        const int d = ka ^ kb;
        w.n += (mine && both);
        w.same += (mine && both && d == 0);
        w.ts += (mine && both && d == 1);
        const unsigned bm = __ballot_sync(TAXI_FULL_MASK, both) & visited;
        if (!a.f16.has_gap_symbol) {   // aligned columns hold no gap: only the both-real span moves
            if (bm) { w.gapc += w.seen ? w.pend : 0; w.pend = 0; w.seen = true; }
        } else {                       // '-' inside a sequence: a column of '-' against a base counts as a gap column
            const unsigned gm = __ballot_sync(TAXI_FULL_MASK, (ka == 4) != (kb == 4) && (ka < 4 || kb < 4)) & visited;
            if (bm) {
                const int fb = __ffs(bm) - 1, lb = 31 - __clz(bm);
                const unsigned below = (1u << fb) - 1u;
                const unsigned upto = (lb == 31) ? 0xffffffffu : ((2u << lb) - 1u);
                if (w.seen) w.gapc += w.pend + __popc(gm & below);
                w.gapc += __popc(gm & upto & ~below);
                w.pend = __popc(gm & ~upto);
                w.seen = true;
            } else {
                w.pend += __popc(gm);
            }
        }
    } else {
        // a gap run: every column whose symbol is a base is a gap column, pending until the next both-real column
        const int k = code_class(f, state == 1 ? w.ca : w.cb);
        w.pend += __popc(__ballot_sync(TAXI_FULL_MASK, k < 4) & visited);
    }
    if (a.aln_x != nullptr && mine) {
        TAXI_CHECK(a, w.wpos - 1 - lane >= a.aln_off[w.p] && w.wpos - 1 - lane < a.aln_off[w.p + 1], 2);
        a.aln_x[w.wpos - 1 - lane] = (state == 2) ? (uint8_t)'-' : code_ascii(f, w.ca);
        a.aln_y[w.wpos - 1 - lane] = (state == 1) ? (uint8_t)'-' : code_ascii(f, w.cb);
    }
    w.wpos -= V;
    w.i -= V * di; w.j -= V * dj;
    w.state = next;
}

template <bool SYM = false>
__device__ __forceinline__ void walk_finish(Walk& w, const AlignArgs& a, int lane)
{
    if (a.aln_x != nullptr) {
        TAXI_CHECK(a, w.wpos - w.i - w.j >= a.aln_off[w.p] && w.wpos <= a.aln_off[w.p + 1], 3);
        // leading end gap: whatever is left of x (vertical) or y (horizontal)
        for (int k = lane; k < w.i; k += 32) {
            a.aln_x[w.wpos - 1 - k] = code_ascii(a.f16, (int)__ldg(w.x + w.i - 1 - k));
            a.aln_y[w.wpos - 1 - k] = '-';
        }
        w.wpos -= w.i;
        for (int k = lane; k < w.j; k += 32) {
            a.aln_x[w.wpos - 1 - k] = '-';
            a.aln_y[w.wpos - 1 - k] = code_ascii(a.f16, (int)__ldg(w.y + w.j - 1 - k));
        }
        w.wpos -= w.j;
        if (lane == 0) a.aln_start[w.p] = w.wpos;
    }
    const int n = (int)__reduce_add_sync(TAXI_FULL_MASK, (unsigned)w.n);
    const int same = (int)__reduce_add_sync(TAXI_FULL_MASK, (unsigned)w.same);
    const int ts = (int)__reduce_add_sync(TAXI_FULL_MASK, (unsigned)w.ts);
    const int tv = n - same - ts;
    if (lane != 0) return;
    if (a.score) a.score[w.p] = w.score;
    if (a.counts) *reinterpret_cast<int4*>(a.counts + 4 * w.p) = make_int4(same, ts, tv, w.gapc);
    double m[4];
    if (a.metrics || (SYM && a.t_metrics)) metrics_from_counts(same, ts, tv, w.gapc, m);
    if (a.metrics) {
        double2* dst = reinterpret_cast<double2*>(a.metrics + 4 * w.p);
        dst[0] = make_double2(m[0], m[1]);
        dst[1] = make_double2(m[2], m[3]);
    }
    if (SYM) {
        // the mirrored pair (y, x): same score, counts and metrics, at the transposed position -- unless the
        // path was orientation-sensitive, in which case the host re-aligns (y, x) on its own
        if (w.sens) {
            const unsigned long long k = atomicAdd(a.redo_count, 1ULL);
            TAXI_CHECK(a, k < (unsigned long long)a.npairs, 4);
            a.redo[k] = w.p;
        } else {
            const long long t = (w.p % a.ny) * (long long)a.nx + w.p / a.ny;
            TAXI_CHECK(a, t >= 0 && t < a.npairs && w.p / a.ny < a.nx, 5);
            if (a.t_score) a.t_score[t] = w.score;
            if (a.t_counts) *reinterpret_cast<int4*>(a.t_counts + 4 * t) = make_int4(same, ts, tv, w.gapc);
            if (a.t_metrics) {
                double2* dst = reinterpret_cast<double2*>(a.t_metrics + 4 * t);
                dst[0] = make_double2(m[0], m[1]);
                dst[1] = make_double2(m[2], m[3]);
            }
        }
    }
}

__device__ __forceinline__ Walk walk_start(const AlignArgs& a, long long p, const uint8_t* x, const uint8_t* y, int nA, int nB,
                                           int half, int off, uint32_t fin, int beta, int bias, int stride = 0)
{
    Walk w;
    w.x = x; w.y = y; w.p = p; w.i = nA; w.j = nB; w.state = 3 - (int)(fin & 3u);
    w.half = half; w.off = off; w.stride = stride;
    w.n = w.same = w.ts = w.gapc = w.pend = 0; w.seen = false; w.sens = false;
    w.wpos = a.aln_x != nullptr ? a.aln_off[p + 1] : 0;
    w.score = ((int)(fin & 0xFFF0u) - bias) / 16 + beta * nA;
    w.tb = w.ca = w.cb = 0;
    w.entered = true;
    return w;
}

template <int H, bool MULTI, bool SYM = false>
__device__ __forceinline__ void traceback_two(const AlignArgs& a, int lane, const uint8_t* trace, int l0, Walk& wa, Walk& wb, bool second)
{
    if (!second) { wb.i = 0; wb.j = 0; }
    while ((wa.i > 0 && wa.j > 0) || (wb.i > 0 && wb.j > 0)) {
        walk_fetch<H, MULTI, SYM>(a, wa, lane, trace, l0);
        walk_fetch<H, MULTI, SYM>(a, wb, lane, trace, l0);
        walk_advance<SYM>(wa, a, lane);
        walk_advance<SYM>(wb, a, lane);
    }
    walk_finish<SYM>(wa, a, lane);
    if (second) walk_finish<SYM>(wb, a, lane);
}

struct PairRef {
    const uint8_t* xc; const uint8_t* yc;   // 3-bit codes (DP, traceback counts, gapped strings via Fast16::ascii_*)
    int nA, nB;
    long long out;                          // index of this pair's results
};

__device__ __forceinline__ PairRef pair_ref(const AlignArgs& a, long long p)
{
    const PairIndex pi = pair_index(a, p);
    const int xi = pi.xi, yi = pi.yi;
    const int64_t xo = a.xoff[xi], yo = a.yoff[yi];
    PairRef r;
    r.out = pi.out;
    r.xc = a.xc + code_offset(xo, xi); r.yc = a.yc + code_offset(yo, yi);
    r.nA = (int)(a.xoff[xi + 1] - xo);
    r.nB = (int)(a.yoff[yi + 1] - yo);
    return r;
}

template <int H>
__device__ __forceinline__ void align_two(const AlignArgs& a, long long p0, long long p1, int lane, uint8_t* trace)
{
    constexpr int HB = Pair16Geom<H>::HB;
    constexpr int WORDS = Pair16Geom<H>::WORDS;
    const Fast16& f = a.f16;
    const PairRef A = pair_ref(a, p0), B = pair_ref(a, p1);
    const int nBmax = max(A.nB, B.nB), nAmax = max(A.nA, B.nA);
    const int nlive = (nAmax + H - 1) / H;
    const bool live = lane < nlive;
    const int nsteps = nBmax + nlive - 1;
    const int itop = lane * H + 1;

    uint32_t a2[H], Hl[H], Yn[H], ncYM[H], cYY[H];
#pragma unroll
    for (int r = 0; r < H; ++r) {
        const int i = itop + r;
        const uint32_t c0 = (i <= A.nA) ? (uint32_t)__ldg(A.xc + min(i, A.nA) - 1) : CODE_PADSYM;
        const uint32_t c1 = (i <= B.nA) ? (uint32_t)__ldg(B.xc + min(i, B.nA) - 1) : CODE_PADSYM;
        a2[r] = row_codes(c0, c1);
        const uint32_t xb = (uint32_t)f.bias - f.PeoX - (uint32_t)(i - 1) * f.PeeX + 2u;   // Ix(i,0), tagged as state Ix
        Hl[r] = pack16(xb, xb);
        Yn[r] = pack16((uint32_t)f.neg, (uint32_t)f.neg);                                        // no Ix->Iy: Iy(i,1) opens from M only
        const int yo0 = (i == A.nA) ? f.PeoY : f.PoY, yo1 = (i == B.nA) ? f.PeoY : f.PoY;
        const int ye0 = (i == A.nA) ? f.PeeY : f.PeY, ye1 = (i == B.nA) ? f.PeeY : f.PeY;
        ncYM[r] = pack16((uint32_t)(5 - yo0), (uint32_t)(5 - yo1));   // M(tag 3) -> Iy candidate with bit 3 set
        cYY[r] = pack16((uint32_t)(ye0 + 1), (uint32_t)(ye1 + 1));    // Iy(tag 1) -> Iy candidate with clean tag
    }
    uint32_t Hd_saved;
    if (itop == 1) Hd_saved = pack16((uint32_t)f.bias + 3u, (uint32_t)f.bias + 3u);   // (0,0): state M
    else {
        const uint32_t v = (uint32_t)f.bias - f.PeoX - (uint32_t)(itop - 2) * f.PeeX + 2u;
        Hd_saved = pack16(v, v);
    }
    const int llA = (A.nA - 1) / H, rlA = (A.nA - 1) % H;
    const int llB = (B.nA - 1) / H, rlB = (B.nA - 1) % H;
    uint32_t outX = 0, outH = 0, finA = 0, finB = 0;
    uint8_t* tbase = trace + (size_t)lane * HB;

    // The sweep runs in up to three segments so that H(nA, nB) of each pair can be picked up
    // right after the step that produces it (the other pair may keep the registers busy for
    // more columns), without any capture logic inside the hot loop.
    const int tA = A.nB - 1 + llA, tB = B.nB - 1 + llB;   // steps that produce the two end cells
    int t = 0;
#pragma unroll 1
    for (int seg = 0; seg < 3; ++seg) {
        const int tend = (seg == 0) ? min(tA, tB) + 1 : (seg == 1 ? max(tA, tB) + 1 : nsteps);
        for (; t < tend; ++t) {
            const int j = t - lane + 1;
            uint32_t rX = __shfl_up_sync(TAXI_FULL_MASK, outX, 1);
            uint32_t rH = __shfl_up_sync(TAXI_FULL_MASK, outH, 1);
            const bool active = live && j >= 1 && j <= nBmax;
            if (lane == 0 && active) {
                // row 0: only Iy is alive (leading end gap); nothing can open Ix from it
                const uint32_t y0 = (uint32_t)f.bias - f.PeoY - (uint32_t)(j - 1) * f.PeeY + 1u;
                rH = pack16(y0, y0);
                rX = pack16((uint32_t)f.neg, (uint32_t)f.neg);
            }
            if (active) {
                const uint32_t b0 = (j <= A.nB) ? (uint32_t)__ldg(A.yc + j - 1) : CODE_PADSYM;
                const uint32_t b1 = (j <= B.nB) ? (uint32_t)__ldg(B.yc + j - 1) : CODE_PADSYM;
                const uint32_t b2 = b0 | (b1 << 16);
                const int xo0 = (j == A.nB) ? f.PeoX : f.PoX, xo1 = (j == B.nB) ? f.PeoX : f.PoX;
                const int xe0 = (j == A.nB) ? f.PeeX : f.PeX, xe1 = (j == B.nB) ? f.PeeX : f.PeX;
                const uint32_t ncXM = pack16((uint32_t)(1 - xo0), (uint32_t)(1 - xo1));  // M(tag 3) -> Ix candidate with bit 2 set
                const uint32_t cXX = pack16((uint32_t)(xe0 + 2), (uint32_t)(xe1 + 2));   // Ix(tag 2) -> clean
                uint32_t Hd = Hd_saved, Xin = rX;
                uint32_t tw[WORDS];
                uint32_t tprev = 0;
#pragma unroll
                for (int r = 0; r < H; ++r) {
                    const uint32_t Mr = diag_candidate(Hd, a2[r], b2, f.negD);
                    const uint32_t Yin = Yn[r];
                    const uint32_t tc = lop3_or3(Mr, Xin, Yin);                   // 4-bit trace code per half (+ score bits above)
                    const uint32_t Mt = lop3_and_or(Mr, F16_CLEAN, 0x00030003u);
                    const uint32_t Xt = lop3_and_or(Xin, F16_CLEAN, 0x00020002u);
                    const uint32_t Yt = lop3_and_or(Yin, F16_CLEAN, 0x00010001u);
                    Hd = Hl[r];
                    Hl[r] = __vimax3_u16x2(Mt, Xt, Yt);
                    Xin = __viaddmax_u16x2(Mt, ncXM, Xt - cXX);
                    Yn[r] = __viaddmax_u16x2(Mt, ncYM[r], Yt - cYY[r]);
                    if (r & 1) tw[r >> 1] = __byte_perm(tprev, tc, 0x6420);
                    else if (r == H - 1) tw[r >> 1] = __byte_perm(tc, 0u, 0x6420);
                    tprev = tc;
                }
                outX = Xin;
                outH = Hl[H - 1];
                Hd_saved = rH;
                uint4* dst = reinterpret_cast<uint4*>(tbase + (size_t)t * 32 * HB);
                TAXI_CHECK(a, reinterpret_cast<uint8_t*>(dst) >= trace && reinterpret_cast<uint8_t*>(dst) + HB <= trace + a.trace_per_warp, 4);
#pragma unroll
                for (int k = 0; k < HB / 16; ++k) {
                    uint32_t w[4];
#pragma unroll
                    for (int q = 0; q < 4; ++q) w[q] = (4 * k + q < WORDS) ? tw[4 * k + q] : 0u;
                    __stcg(dst + k, make_uint4(w[0], w[1], w[2], w[3]));
                }
            }
        }
        if (t - 1 == tA && lane == llA) {
#pragma unroll
            for (int r = 0; r < H; ++r) finA = (r == rlA) ? (Hl[r] & 0xFFFFu) : finA;
        }
        if (t - 1 == tB && lane == llB) {
#pragma unroll
            for (int r = 0; r < H; ++r) finB = (r == rlB) ? (Hl[r] >> 16) : finB;
        }
    }
    finA = __shfl_sync(TAXI_FULL_MASK, finA, llA);
    finB = __shfl_sync(TAXI_FULL_MASK, finB, llB);
    __syncwarp();

    Walk wa = walk_start(a, A.out, A.xc, A.yc, A.nA, A.nB, 0, 0, finA, f.beta, f.bias);
    Walk wb = walk_start(a, B.out, B.xc, B.yc, B.nA, B.nB, 1, 0, finB, f.beta, f.bias);
    traceback_two<H, false>(a, lane, trace, 0, wa, wb, p1 != p0);
}

// Bottom-aligned variant: the rows of each pair are shifted (per half) so that row nA always sits
// in the last register slot of lane 31.  The only rows with special (end-gap) constants are then
// row nA -- a fixed slot -- and the border row 0, which is kept as an ordinary row whose Iy chain
// reproduces the leading end gap by itself (requires internal extend == end extend, checked on
// the host).  No per-row constant registers are needed; dead slots above row 0 idle at "minus
// infinity".
// SYM: besides the codes, one bit per group of two rows says whether H is won there by Ix with Iy at the same
// score -- the one decision that differs when the pair is aligned the other way round; see walk_fetch.
template <int H, bool SYM = false>
__device__ __forceinline__ void align_two_bottom(const AlignArgs& a, long long p0, long long p1, int lane, uint8_t* trace)
{
    constexpr int HB = Pair16Geom<H, SYM>::HB;
    constexpr int WORDS = Pair16Geom<H, SYM>::WORDS;
    constexpr int SL = 32 * H;
    const Fast16& f = a.f16;
    const PairRef A = pair_ref(a, p0), B = pair_ref(a, p1);
    const int offA = SL - A.nA, offB = SL - B.nA;        // slot of row 1; row 0 sits in slot off-1
    const int l0 = (min(offA, offB) - 1) / H;            // first lane that holds a row >= 0
    const int nBmax = max(A.nB, B.nB);
    const int nsteps = nBmax + (31 - l0);
    const bool live = lane >= l0;
    const uint32_t NEG2 = pack16((uint32_t)f.neg, (uint32_t)f.neg);

    auto col0_H = [&](int i) -> uint32_t {   // H(i, 0): Ix border for i >= 1, M(0,0) for i == 0, dead above
        if (i >= 1) return (uint32_t)f.bias - f.PeoX - (uint32_t)(i - 1) * f.PeeX + 2u;
        return i == 0 ? (uint32_t)f.bias + 3u : (uint32_t)f.neg;
    };

    uint32_t a2[H], Hl[H], Yn[H];
#pragma unroll
    for (int r = 0; r < H; ++r) {
        const int s = lane * H + r;
        const int iA = s - offA + 1, iB = s - offB + 1;
        const uint32_t c0 = (iA >= 1) ? (uint32_t)__ldg(A.xc + max(iA, 1) - 1) : CODE_PADSYM;
        const uint32_t c1 = (iB >= 1) ? (uint32_t)__ldg(B.xc + max(iB, 1) - 1) : CODE_PADSYM;
        a2[r] = row_codes(c0, c1);
        Hl[r] = pack16(col0_H(iA), col0_H(iB));
        // Iy(i, 1): only row 0 has one (the leading end gap, opened from M(0,0)); no Ix->Iy elsewhere
        const uint32_t y0 = (uint32_t)f.bias - f.PeoY + 8u;
        Yn[r] = pack16(iA == 0 ? y0 : (uint32_t)f.neg, iB == 0 ? y0 : (uint32_t)f.neg);
    }
    const int itA = lane * H - offA, itB = lane * H - offB;   // row above my top slot
    uint32_t Hd_saved = pack16(col0_H(itA), col0_H(itB));
    // Iy constants: internal everywhere except the very last slot (row nA of both pairs).  The
    // "subtract a packed non-negative constant" steps are written as x + (-c) with a full 32-bit
    // negation of the packed constant (no borrow can cross the halves, see the header comment).
    const uint32_t ncYMi = pack16((uint32_t)(5 - f.PoY), (uint32_t)(5 - f.PoY));
    const uint32_t cYYi = 0u - pack16((uint32_t)(f.PeY + 1), (uint32_t)(f.PeY + 1));
    const uint32_t ncYMl = (lane == 31) ? pack16((uint32_t)(5 - f.PeoY), (uint32_t)(5 - f.PeoY)) : ncYMi;
    const uint32_t cYYl = (lane == 31) ? 0u - pack16((uint32_t)(f.PeeY + 1), (uint32_t)(f.PeeY + 1)) : cYYi;
    const uint32_t ncXMi = pack16((uint32_t)(1 - f.PoX), (uint32_t)(1 - f.PoX));
    const uint32_t cXXi = 0u - pack16((uint32_t)(f.PeX + 2), (uint32_t)(f.PeX + 2));

    uint32_t outX = NEG2, outH = NEG2, finA = 0, finB = 0;
    uint8_t* tbase = trace + (size_t)lane * HB;
    const int tA = A.nB - 1 + (31 - l0), tB = B.nB - 1 + (31 - l0);   // steps at which lane 31 finishes column nB

    // Symbols of y travel down the lanes with the wavefront: lane l at step t works on the column
    // lane l-1 had at step t-1, so one SHFL.UP hands it over.  Lane l0 starts a new column (t + 1)
    // every step and takes it from a chunk of 32 packed columns that the warp loads together once
    // every 32 steps, one chunk ahead (lane k: column 32m + k + 1; past the end of a sequence the
    // clamp lands on the pad code behind it).
    auto load_chunk = [&](int t0) -> uint32_t {
        const int jj = t0 + lane + 1;
        return (uint32_t)__ldg(A.yc + min(jj, A.nB + 1) - 1) | ((uint32_t)__ldg(B.yc + min(jj, B.nB + 1) - 1) << 16);
    };
    uint32_t chunk = 0, next_chunk = load_chunk(0), b2 = 0;

    // One column step.  STEADY: every lane from l0 on is inside the matrix and none is at either
    // pair's last column, so there is no activity test and no end-column constant.  Lanes below
    // l0 then compute on garbage (their results are neither stored nor read: lane l0 takes
    // "minus infinity" from above whatever lane l0 - 1 holds), which costs no issue slot.
    int t = 0;
    auto step = [&](auto steady) {
        constexpr bool STEADY = decltype(steady)::value;
        const uint32_t next_b = __shfl_sync(TAXI_FULL_MASK, chunk, t);   // lane t mod 32: column t + 1
        b2 = __shfl_up_sync(TAXI_FULL_MASK, b2, 1);
        uint32_t rX = __shfl_up_sync(TAXI_FULL_MASK, outX, 1);
        uint32_t rH = __shfl_up_sync(TAXI_FULL_MASK, outH, 1);
        if (lane == l0) { b2 = next_b; rX = NEG2; rH = NEG2; }   // nothing above slot l0 * H holds a row >= 0
        const int j = t - (lane - l0) + 1;
        if (STEADY || (live && j >= 1 && j <= nBmax)) {
            uint32_t ncXM = ncXMi, cXX = cXXi;
            if (!STEADY && (j == A.nB || j == B.nB)) {   // a vertical gap in a pair's last column is an end gap
                const int xo0 = (j == A.nB) ? f.PeoX : f.PoX, xo1 = (j == B.nB) ? f.PeoX : f.PoX;
                const int xe0 = (j == A.nB) ? f.PeeX : f.PeX, xe1 = (j == B.nB) ? f.PeeX : f.PeX;
                ncXM = pack16((uint32_t)(1 - xo0), (uint32_t)(1 - xo1));
                cXX = 0u - pack16((uint32_t)(xe0 + 2), (uint32_t)(xe1 + 2));
            }
            uint32_t Xin = rX;
            uint32_t tw[WORDS];
            uint32_t tprev = 0;
            uint32_t Mr = diag_candidate(Hd_saved, a2[0], b2, f.negD);
            uint32_t ties = 0, zprev = 0;   // SYM
#pragma unroll
            for (int r = 0; r < H; ++r) {
                uint32_t Mr_next = 0;
                if (r + 1 < H) Mr_next = diag_candidate(Hl[r], a2[r + 1], b2, f.negD);   // needs H(i, j-1) before it is overwritten
                const uint32_t Yin = Yn[r];
                const uint32_t tc = lop3_or3(Mr, Xin, Yin);
                const uint32_t Mt = lop3_and_or(Mr, F16_CLEAN, 0x00030003u);
                const uint32_t Xt = lop3_and_or(Xin, F16_CLEAN, 0x00020002u);
                const uint32_t Yt = lop3_and_or(Yin, F16_CLEAN, 0x00010001u);
                Hl[r] = __vimax3_u16x2(Mt, Xt, Yt);
                if constexpr (SYM) {
                    // H ^ Iy ^ 3 is zero per half exactly where H holds Ix's value (tag 2) and Iy the same score
                    // (tag 1).  min3 over the two rows of a group and 1 gives "no such tie in the group", shifted
                    // into the lane's bit string on the fma pipe: 2 LOP3 + VIMNMX3 + IMAD per two row pairs.
                    const uint32_t z = lop3_xor3(Hl[r], Yt, 0x00030003u);
                    if (r & 1) ties = ties * 2u + __vimin3_u16x2(zprev, z, 0x00010001u);
                    else if (r == H - 1) ties = ties * 2u + __vminu2(z, 0x00010001u);
                    zprev = z;
                }
                Xin = __viaddmax_u16x2(Mt, ncXM, Xt + cXX);
                Yn[r] = __viaddmax_u16x2(Mt, (r == H - 1) ? ncYMl : ncYMi, Yt + ((r == H - 1) ? cYYl : cYYi));
                if (r & 1) tw[r >> 1] = __byte_perm(tprev, tc, 0x6420);
                else if (r == H - 1) tw[r >> 1] = __byte_perm(tc, 0u, 0x6420);
                tprev = tc;
                Mr = Mr_next;
            }
            outX = Xin;
            outH = Hl[H - 1];
            Hd_saved = rH;
            if (STEADY && !live) return;
            uint4* dst = reinterpret_cast<uint4*>(tbase + (size_t)t * 32 * HB);
            TAXI_CHECK(a, reinterpret_cast<uint8_t*>(dst) >= trace && reinterpret_cast<uint8_t*>(dst) + HB <= trace + a.trace_per_warp, 4);
#pragma unroll
            for (int k = 0; k < HB / 16; ++k) {
                uint32_t w[4];
#pragma unroll
                for (int q = 0; q < 4; ++q) w[q] = (4 * k + q < WORDS) ? tw[4 * k + q] : ((SYM && 4 * k + q == WORDS) ? ties : 0u);
                __stcg(dst + k, make_uint4(w[0], w[1], w[2], w[3]));
            }
        }
    };
    auto run = [&](int tend, auto steady) {
        while (t < tend) {
            if ((t & 31) == 0) { chunk = next_chunk; next_chunk = load_chunk(t + 32); }
            const int cend = min(tend, (t | 31) + 1);
#pragma unroll 1
            for (; t < cend; ++t) step(steady);
        }
    };

    // Five segments: the fill (lanes still starting), the steady state, and three more so that
    // H(nA, nB) of each pair can be picked up right after the step that produces it (the other
    // pair may keep the registers busy for more columns) without any capture logic in a loop.
    const int tfill = 31 - l0;                                   // lane 31 starts column 1
    const int tsteady = max(tfill, min(A.nB, B.nB) - 1);         // lane l0 reaches the first last column
#pragma unroll 1
    for (int seg = 0; seg < 5; ++seg) {
        if (seg == 1) run(tsteady, std::true_type{});
        else run(seg == 0 ? tfill : seg == 2 ? min(tA, tB) + 1 : seg == 3 ? max(tA, tB) + 1 : nsteps, std::false_type{});
        if (t - 1 == tA) finA = Hl[H - 1] & 0xFFFFu;
        if (t - 1 == tB) finB = Hl[H - 1] >> 16;
    }
    finA = __shfl_sync(TAXI_FULL_MASK, finA, 31);
    finB = __shfl_sync(TAXI_FULL_MASK, finB, 31);
    __syncwarp();

    Walk wa = walk_start(a, A.out, A.xc, A.yc, A.nA, A.nB, 0, offA, finA, f.beta, f.bias);
    Walk wb = walk_start(a, B.out, B.xc, B.yc, B.nA, B.nB, 1, offB, finB, f.beta, f.bias);
    traceback_two<H, false, SYM>(a, lane, trace, l0, wa, wb, p1 != p0);
}

// Multi-stripe form of the bottom-aligned variant for x longer than 32*H - 1: the slots are cut
// into stripes of 32*H that are swept one after the other; the bottom slot of a stripe hands its
// Ix / H values to the top slot of the next through a small per-warp boundary buffer (two packed
// words per column).  Kept as a separate instantiation so the single-stripe hot loop stays lean.
template <int H>
__device__ __forceinline__ void align_two_bottom_multi(const AlignArgs& a, long long p0, long long p1, int lane, uint8_t* trace,
                                                       uint32_t* bnd)
{
    constexpr int HB = Pair16Geom<H>::HB;
    constexpr int WORDS = Pair16Geom<H>::WORDS;
    constexpr int SL = 32 * H;
    const Fast16& f = a.f16;
    const PairRef A = pair_ref(a, p0), B = pair_ref(a, p1);
    const int nstripes = (max(A.nA, B.nA) + 1 + SL - 1) / SL;   // rows 0..nA of the longer pair
    const int total = nstripes * SL;
    const int offA = total - A.nA, offB = total - B.nA;
    const int l0 = (min(offA, offB) - 1) / H;                   // < 32 by construction
    const int nBmax = max(A.nB, B.nB);
    const int stride = nBmax + 31;
    const uint32_t NEG2 = pack16((uint32_t)f.neg, (uint32_t)f.neg);

    auto col0_H = [&](int i) -> uint32_t {
        if (i >= 1) return (uint32_t)f.bias - f.PeoX - (uint32_t)(i - 1) * f.PeeX + 2u;
        return i == 0 ? (uint32_t)f.bias + 3u : (uint32_t)f.neg;
    };
    const uint32_t ncYMi = pack16((uint32_t)(5 - f.PoY), (uint32_t)(5 - f.PoY));
    const uint32_t cYYi = 0u - pack16((uint32_t)(f.PeY + 1), (uint32_t)(f.PeY + 1));
    const uint32_t ncXMi = pack16((uint32_t)(1 - f.PoX), (uint32_t)(1 - f.PoX));
    const uint32_t cXXi = 0u - pack16((uint32_t)(f.PeX + 2), (uint32_t)(f.PeX + 2));
    uint32_t finA = 0, finB = 0;

    for (int st = 0; st < nstripes; ++st) {
        const bool last = st + 1 == nstripes;
        const int first_lane = (st == 0) ? l0 : 0;
        const bool live = lane >= first_lane;
        const int nsteps = nBmax + (31 - first_lane);
        uint32_t a2[H], Hl[H], Yn[H];
#pragma unroll
        for (int r = 0; r < H; ++r) {
            const int s = st * SL + lane * H + r;
            const int iA = s - offA + 1, iB = s - offB + 1;
            const uint32_t c0 = (iA >= 1) ? (uint32_t)__ldg(A.xc + max(iA, 1) - 1) : CODE_PADSYM;
            const uint32_t c1 = (iB >= 1) ? (uint32_t)__ldg(B.xc + max(iB, 1) - 1) : CODE_PADSYM;
        a2[r] = row_codes(c0, c1);
            Hl[r] = pack16(col0_H(iA), col0_H(iB));
            const uint32_t y0 = (uint32_t)f.bias - f.PeoY + 8u;
            Yn[r] = pack16(iA == 0 ? y0 : (uint32_t)f.neg, iB == 0 ? y0 : (uint32_t)f.neg);
        }
        const int itA = st * SL + lane * H - offA, itB = st * SL + lane * H - offB;
        uint32_t Hd_saved = pack16(col0_H(itA), col0_H(itB));
        const bool end_slot = last && lane == 31;
        const uint32_t ncYMl = end_slot ? pack16((uint32_t)(5 - f.PeoY), (uint32_t)(5 - f.PeoY)) : ncYMi;
        const uint32_t cYYl = end_slot ? 0u - pack16((uint32_t)(f.PeeY + 1), (uint32_t)(f.PeeY + 1)) : cYYi;
        uint32_t outX = NEG2, outH = NEG2;
        uint8_t* tbase = trace + ((size_t)st * stride * 32 + lane) * HB;
        const int tA = last ? A.nB - 1 + (31 - first_lane) : -2, tB = last ? B.nB - 1 + (31 - first_lane) : -2;
        int t = 0;
        // the y symbols of a column and, for the top slot of a later stripe, the values the previous
        // stripe left in the boundary buffer are fetched one step ahead, so that their latency hides
        // behind a whole step (the pad codes around every sequence make the symbol fetch a clamp)
        uint32_t nb0 = CODE_PADSYM, nb1 = CODE_PADSYM, nbX = NEG2, nbH = NEG2;
        auto fetch_next = [&](int jj) {
            nb0 = (uint32_t)__ldg(A.yc + min(jj, A.nB + 1) - 1);
            nb1 = (uint32_t)__ldg(B.yc + min(jj, B.nB + 1) - 1);
            if (lane == 0 && st > 0) {   // lane 0: jj >= 1
                TAXI_CHECK(a, jj >= 0 && 2LL * jj + 1 < a.bnd_per_warp, 6);
                nbX = __ldcg(bnd + 2 * jj); nbH = __ldcg(bnd + 2 * jj + 1);
            }
        };
        fetch_next(0 - (lane - first_lane) + 1);
#pragma unroll 1
        for (int seg = 0; seg < 3; ++seg) {
            const int tend = !last ? (seg == 2 ? nsteps : 0) : ((seg == 0) ? min(tA, tB) + 1 : (seg == 1 ? max(tA, tB) + 1 : nsteps));
            for (; t < tend; ++t) {
                const int j = t - (lane - first_lane) + 1;
                uint32_t rX = __shfl_up_sync(TAXI_FULL_MASK, outX, 1);
                uint32_t rH = __shfl_up_sync(TAXI_FULL_MASK, outH, 1);
                const bool active = live && j >= 1 && j <= nBmax;
                const uint32_t b0 = nb0, b1 = nb1;
                if (lane == 0) {
                    if (st == 0 || !active) { rX = NEG2; rH = NEG2; }
                    else { rX = nbX; rH = nbH; }
                }
                fetch_next(j + 1);
                if (active) {
                    const uint32_t b2 = b0 | (b1 << 16);
                    uint32_t ncXM = ncXMi, cXX = cXXi;
                    if (j == A.nB || j == B.nB) {
                        const int xo0 = (j == A.nB) ? f.PeoX : f.PoX, xo1 = (j == B.nB) ? f.PeoX : f.PoX;
                        const int xe0 = (j == A.nB) ? f.PeeX : f.PeX, xe1 = (j == B.nB) ? f.PeeX : f.PeX;
                        ncXM = pack16((uint32_t)(1 - xo0), (uint32_t)(1 - xo1));
                        cXX = 0u - pack16((uint32_t)(xe0 + 2), (uint32_t)(xe1 + 2));
                    }
                    uint32_t Xin = rX;
                    uint32_t tw[WORDS];
                    uint32_t tprev = 0;
                    uint32_t Mr = diag_candidate(Hd_saved, a2[0], b2, f.negD);
#pragma unroll
                    for (int r = 0; r < H; ++r) {
                        uint32_t Mr_next = 0;
                        if (r + 1 < H) Mr_next = diag_candidate(Hl[r], a2[r + 1], b2, f.negD);
                        const uint32_t Yin = Yn[r];
                        const uint32_t tc = lop3_or3(Mr, Xin, Yin);
                        const uint32_t Mt = lop3_and_or(Mr, F16_CLEAN, 0x00030003u);
                        const uint32_t Xt = lop3_and_or(Xin, F16_CLEAN, 0x00020002u);
                        const uint32_t Yt = lop3_and_or(Yin, F16_CLEAN, 0x00010001u);
                        Hl[r] = __vimax3_u16x2(Mt, Xt, Yt);
                        Xin = __viaddmax_u16x2(Mt, ncXM, Xt + cXX);
                        Yn[r] = __viaddmax_u16x2(Mt, (r == H - 1) ? ncYMl : ncYMi, Yt + ((r == H - 1) ? cYYl : cYYi));
                        if (r & 1) tw[r >> 1] = __byte_perm(tprev, tc, 0x6420);
                        else if (r == H - 1) tw[r >> 1] = __byte_perm(tc, 0u, 0x6420);
                        tprev = tc;
                        Mr = Mr_next;
                    }
                    outX = Xin;
                    outH = Hl[H - 1];
                    Hd_saved = rH;
                    uint4* dst = reinterpret_cast<uint4*>(tbase + (size_t)t * 32 * HB);
                    TAXI_CHECK(a, reinterpret_cast<uint8_t*>(dst) >= trace && reinterpret_cast<uint8_t*>(dst) + HB <= trace + a.trace_per_warp, 5);
#pragma unroll
                    for (int k = 0; k < HB / 16; ++k) {
                        uint32_t w[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) w[q] = (4 * k + q < WORDS) ? tw[4 * k + q] : 0u;
                        __stcg(dst + k, make_uint4(w[0], w[1], w[2], w[3]));
                    }
                    if (lane == 31 && !last) {   // hand the stripe's bottom slot to the next stripe
                        TAXI_CHECK(a, j >= 0 && 2LL * j + 1 < a.bnd_per_warp, 7);
                        __stcg(bnd + 2 * j, outX);
                        __stcg(bnd + 2 * j + 1, outH);
                    }
                }
            }
            if (last && t - 1 == tA) finA = Hl[H - 1] & 0xFFFFu;
            if (last && t - 1 == tB) finB = Hl[H - 1] >> 16;
        }
        __syncwarp();
    }
    finA = __shfl_sync(TAXI_FULL_MASK, finA, 31);
    finB = __shfl_sync(TAXI_FULL_MASK, finB, 31);
    __syncwarp();

    Walk wa = walk_start(a, A.out, A.xc, A.yc, A.nA, A.nB, 0, offA, finA, f.beta, f.bias, stride);
    Walk wb = walk_start(a, B.out, B.xc, B.yc, B.nA, B.nB, 1, offB, finB, f.beta, f.bias, stride);
    traceback_two<H, true>(a, lane, trace, l0, wa, wb, p1 != p0);
}

#ifndef PAIR16_WPB
#define PAIR16_WPB 4
#endif
#ifndef PAIR16_MIN_BLOCKS
#define PAIR16_MIN_BLOCKS 3   // 168 registers: measured best (fewer blocks or forced spills are both slower)
#endif
constexpr int PAIR16_WARPS_PER_BLOCK = PAIR16_WPB;

// MODE 0: top-aligned rows; 1: bottom-aligned rows; 2: bottom-aligned, several stripes (long x)
// Three blocks of four warps (168 registers) is the measured optimum for the 21-row kernel; the
// taller / multi-stripe instantiations need more registers and run two blocks per SM.
template <int H, int MODE, bool SYM = false>
__global__ void __launch_bounds__(PAIR16_WARPS_PER_BLOCK * 32, (H >= 32) ? 2 : PAIR16_MIN_BLOCKS)
gotoh_pair16_kernel(const AlignArgs a)
{
    const int lane = threadIdx.x & 31;
    const long long gw = (long long)blockIdx.x * PAIR16_WARPS_PER_BLOCK + (threadIdx.x >> 5);
    uint8_t* trace = a.trace + gw * a.trace_per_warp;
    uint32_t* bnd = reinterpret_cast<uint32_t*>(a.bnd + gw * a.bnd_per_warp);
    const unsigned long long units = (unsigned long long)a.nunits;
    const unsigned long long upr = ((unsigned long long)a.ny + 1ULL) / 2ULL;   // rect mode: units per row
    for (;;) {
        unsigned long long u = 0;
        if (lane == 0) u = atomicAdd(a.counter, 1ULL);
        u = __shfl_sync(TAXI_FULL_MASK, u, 0);
        if (u >= units) break;
        long long p0, p1;
        if (a.unit_pairs) {
            p0 = a.unit_pairs[2 * u]; p1 = a.unit_pairs[2 * u + 1];
        } else {
            const unsigned long long row = u / upr, cu = u % upr;
            p0 = (long long)(row * (unsigned long long)a.ny + 2ULL * cu);
            p1 = (2ULL * cu + 1ULL < (unsigned long long)a.ny) ? p0 + 1 : p0;
        }
        if constexpr (MODE == 2) align_two_bottom_multi<H>(a, p0, p1, lane, trace, bnd);
        else if constexpr (MODE == 1) align_two_bottom<H, SYM>(a, p0, p1, lane, trace);
        else align_two<H>(a, p0, p1, lane, trace);
        (void)bnd;
        __syncwarp();
    }
}

}  // namespace taxi
