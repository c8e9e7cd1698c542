/*
 * taxi_oracle.c -- CPU restatement of the TaxI2 pairwise-distance hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing in the product package (taxi2_b200/) may
 * import, link or execute this file; only tests/, __graft_entry__.smoke() and
 * bench.py's cpu_baseline / --impl reference legs use it, as the checker.
 *
 * What it restates (file:line relative to /root/reference):
 *   - src/itaxotools/taxi2/align.py:72-157   PairwiseAligner.Biopython.align():
 *       Bio.Align.PairwiseAligner(**scores).align(x, y)[0] in global mode, then
 *       _format_pretty() -> two equal-length gapped strings ('-' for gaps).
 *     The DP itself lives in the third-party C extension
 *       biopython==1.85 (requirements.txt:2), Bio/Align/_pairwisealigner.c,
 *     which is NOT under /root/reference and is not installable here.  Its
 *     published algorithm is restated below: algorithm selection (Needleman-Wunsch
 *     when every open==extend, else 3-state Gotoh with Ix<->Iy transitions), double
 *     scores with an epsilon for ties, a per-cell bitmask of ALL co-optimal
 *     predecessors, and the path generator's "first path" rule
 *     (Gotoh: end state and every predecessor chosen in the order M, Ix, Iy;
 *      NW: horizontal, then vertical, then diagonal).
 *   - src/itaxotools/taxi2/distances.py:319-348  DistanceMetric.{Uncorrected,
 *       UncorrectedWithGaps,JukesCantor,Kimura2P}._calculate() ->
 *       itaxotools-calculate-distances==0.1.1 (Rust, requirements.txt:14), also
 *       absent; rules reconstructed from tests/test_distances/metrics.tsv and
 *       tests/test_distances.py:515-521.
 *
 * PARITY STATUS.  The scoring model is pinned by the 53 known-answer cases of
 * tests/test_align.py:49-203 and the counting/trimming model by the 26x4+3 cases of
 * tests/test_distances (all reproduced: tests/test_oracle_golden.py).  The
 * tie-breaking ORDER among co-optimal alignments is "parity unpinned": the
 * reference tests accept any co-optimal answer; only tests/test_align.py:184-187
 * (comment) distinguishes Ix-before-Iy.  No Biopython binary exists in this image to
 * pin it further.
 */
#include <float.h>
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <pthread.h>
#include <unistd.h>

#define TAXI_OK 0
#define TAXI_E_EMPTY (-2)   /* Biopython raises ValueError on a zero-length sequence */
#define TAXI_E_NOMEM (-3)

/* score vector layout == Scores.defaults order, align.py:20-27 */
enum { S_MATCH = 0, S_MISMATCH, S_INT_OPEN, S_INT_EXT, S_END_OPEN, S_END_EXT };

/* co-optimal predecessor bitmasks */
#define B_M 1
#define B_X 2 /* Ix: vertical move, consumes a[i], '-' in the second string */
#define B_Y 4 /* Iy: horizontal move, consumes b[j], '-' in the first string  */
#define B_H 1 /* NW: horizontal */
#define B_V 2 /* NW: vertical   */
#define B_D 4 /* NW: diagonal   */

static const double EPS = 1e-6; /* Bio.Align.PairwiseAligner default epsilon */

int taxi_oracle_uses_gotoh(const double sc[6])
{
    /* all six open/extend pairs (target+query x left/internal/right) collapse to two in
       TaxI2, because align.py:75 only sets the internal_* / end_* shorthands */
    return !(sc[S_INT_OPEN] == sc[S_INT_EXT] && sc[S_END_OPEN] == sc[S_END_EXT]);
}

/* pick all maxima of three candidates with Biopython's epsilon rule */
static inline double pick3(double c0, double c1, double c2, unsigned char* bits)
{
    double best = c0;
    unsigned char t = 1;
    if (c1 > best + EPS) { best = c1; t = 2; }
    else if (c1 > best - EPS) t |= 2;
    if (c2 > best + EPS) { best = c2; t = 4; }
    else if (c2 > best - EPS) t |= 4;
    *bits = t;
    return best;
}

static int emit_path(const uint8_t* a, const uint8_t* b, const unsigned char* moves, int nmoves,
                     uint8_t* out_a, uint8_t* out_b)
{
    /* moves[] was collected end -> start; walk it backwards (align.py:101-145 semantics) */
    int i = 0, j = 0, k = 0;
    for (int m = nmoves - 1; m >= 0; --m, ++k) {
        switch (moves[m]) {
        case 'D': out_a[k] = a[i++]; out_b[k] = b[j++]; break;
        case 'V': out_a[k] = a[i++]; out_b[k] = '-'; break;
        default:  out_a[k] = '-'; out_b[k] = b[j++]; break;
        }
    }
    return k;
}

static int align_nw(const uint8_t* a, int nA, const uint8_t* b, int nB, const double sc[6],
                    uint8_t* out_a, uint8_t* out_b, int32_t* out_len, double* out_score)
{
    const double g_in = sc[S_INT_EXT], g_end = sc[S_END_EXT];
    const size_t W = (size_t)nB + 1;
    unsigned char* T = (unsigned char*)malloc((size_t)(nA + 1) * W);
    double* row = (double*)malloc(W * sizeof(double));
    unsigned char* moves = (unsigned char*)malloc((size_t)nA + nB + 1);
    if (!T || !row || !moves) { free(T); free(row); free(moves); return TAXI_E_NOMEM; }
    T[0] = 0;
    row[0] = 0.0;
    for (int j = 1; j <= nB; ++j) { row[j] = g_end * j; T[j] = B_H; }
    for (int i = 1; i <= nA; ++i) {
        double diag = row[0];
        row[0] = g_end * i;
        T[i * W] = B_V;
        const double hgap = (i == nA) ? g_end : g_in;
        for (int j = 1; j <= nB; ++j) {
            const double vgap = (j == nB) ? g_end : g_in;
            double score = diag + (a[i - 1] == b[j - 1] ? sc[S_MATCH] : sc[S_MISMATCH]);
            unsigned char t = B_D;
            double c = row[j - 1] + hgap;
            if (c > score + EPS) { score = c; t = B_H; }
            else if (c > score - EPS) t |= B_H;
            c = row[j] + vgap;
            if (c > score + EPS) { score = c; t = B_V; }
            else if (c > score - EPS) t |= B_V;
            diag = row[j];
            row[j] = score;
            T[i * W + j] = t;
        }
    }
    *out_score = row[nB];
    int i = nA, j = nB, n = 0;
    for (;;) {
        unsigned char t = T[i * W + j];
        if (t & B_H) { moves[n++] = 'H'; --j; }
        else if (t & B_V) { moves[n++] = 'V'; --i; }
        else if (t & B_D) { moves[n++] = 'D'; --i; --j; }
        else break;
    }
    *out_len = emit_path(a, b, moves, n, out_a, out_b);
    free(T); free(row); free(moves);
    return TAXI_OK;
}

static int align_gotoh(const uint8_t* a, int nA, const uint8_t* b, int nB, const double sc[6],
                       uint8_t* out_a, uint8_t* out_b, int32_t* out_len, double* out_score)
{
    const double NEG = -DBL_MAX;
    const size_t W = (size_t)nB + 1;
    const size_t cells = (size_t)(nA + 1) * W;
    unsigned char* TM = (unsigned char*)malloc(cells);
    unsigned char* TX = (unsigned char*)malloc(cells);
    unsigned char* TY = (unsigned char*)malloc(cells);
    double* M = (double*)malloc(3 * W * sizeof(double));
    unsigned char* moves = (unsigned char*)malloc((size_t)nA + nB + 1);
    if (!TM || !TX || !TY || !M || !moves) {
        free(TM); free(TX); free(TY); free(M); free(moves);
        return TAXI_E_NOMEM;
    }
    double* X = M + W;
    double* Y = X + W;
    /* borders: only Iy is alive on row 0, only Ix on column 0 */
    M[0] = 0.0; X[0] = NEG; Y[0] = NEG;
    TM[0] = TX[0] = TY[0] = 0;
    for (int j = 1; j <= nB; ++j) {
        M[j] = NEG; X[j] = NEG;
        Y[j] = sc[S_END_OPEN] + sc[S_END_EXT] * (j - 1);
        TM[j] = 0; TX[j] = 0; TY[j] = (j == 1) ? B_M : B_Y;
    }
    for (int i = 1; i <= nA; ++i) {
        double dM = M[0], dX = X[0], dY = Y[0];
        M[0] = NEG; Y[0] = NEG;
        X[0] = sc[S_END_OPEN] + sc[S_END_EXT] * (i - 1);
        TM[i * W] = 0; TY[i * W] = 0; TX[i * W] = (i == 1) ? B_M : B_X;
        /* a horizontal gap on the last row is an end gap */
        const double yo = (i == nA) ? sc[S_END_OPEN] : sc[S_INT_OPEN];
        const double ye = (i == nA) ? sc[S_END_EXT] : sc[S_INT_EXT];
        for (int j = 1; j <= nB; ++j) {
            /* a vertical gap in the last column is an end gap */
            const double xo = (j == nB) ? sc[S_END_OPEN] : sc[S_INT_OPEN];
            const double xe = (j == nB) ? sc[S_END_EXT] : sc[S_INT_EXT];
            const size_t at = i * W + j;
            double best = pick3(dM, dX, dY, &TM[at]);
            dM = M[j]; dX = X[j]; dY = Y[j];   /* (i-1, j): next column's diagonal */
            const double newM = best + (a[i - 1] == b[j - 1] ? sc[S_MATCH] : sc[S_MISMATCH]);
            const double newX = pick3(dM + xo, dX + xe, dY + xo, &TX[at]);
            M[j] = newM;
            X[j] = newX;
            Y[j] = pick3(M[j - 1] + yo, X[j - 1] + yo, Y[j - 1] + ye, &TY[at]);
        }
    }
    /* end state: best of the three; states below the best are not end points */
    const size_t end = (size_t)nA * W + nB;
    double best = M[nB];
    if (X[nB] > best) best = X[nB];
    if (Y[nB] > best) best = Y[nB];
    *out_score = best;
    int state;
    if (!(M[nB] < best - EPS) && TM[end]) state = B_M;
    else if (!(X[nB] < best - EPS) && TX[end]) state = B_X;
    else state = B_Y;
    int i = nA, j = nB, n = 0;
    while (i > 0 || j > 0) {
        unsigned char t;
        const size_t at = (size_t)i * W + j;
        if (state == B_M) { t = TM[at]; moves[n++] = 'D'; --i; --j; }
        else if (state == B_X) { t = TX[at]; moves[n++] = 'V'; --i; }
        else { t = TY[at]; moves[n++] = 'H'; --j; }
        if (t & B_M) state = B_M;
        else if (t & B_X) state = B_X;
        else if (t & B_Y) state = B_Y;
        else break;
    }
    *out_len = emit_path(a, b, moves, n, out_a, out_b);
    free(TM); free(TX); free(TY); free(M); free(moves);
    return TAXI_OK;
}

/* align.py:151-157.  out_a/out_b must hold nA+nB bytes each. */
int taxi_oracle_align(const uint8_t* a, int32_t nA, const uint8_t* b, int32_t nB, const double sc[6],
                      uint8_t* out_a, uint8_t* out_b, int32_t* out_len, double* out_score)
{
    if (nA <= 0 || nB <= 0) return TAXI_E_EMPTY;
    if (taxi_oracle_uses_gotoh(sc))
        return align_gotoh(a, nA, b, nB, sc, out_a, out_b, out_len, out_score);
    return align_nw(a, nA, b, nB, sc, out_a, out_b, out_len, out_score);
}

/* ---- distances ------------------------------------------------------------------------- */

/* 0..3 = A,G,C,T (bit1 = pyrimidine, so a transition flips only bit0); 4 = gap; 5 = missing */
static inline int base_class(uint8_t c)
{
    switch (c) {
    case 'A': case 'a': return 0;
    case 'G': case 'g': return 1;
    case 'C': case 'c': return 2;
    case 'T': case 't': return 3;
    case '-': return 4;
    default: return 5;
    }
}

/*
 * distances.py:319-348 -> calc.seq_distances_*: one scan of two (aligned) strings.
 * counts = {same, transitions, transversions, internal gap columns}; the scan is
 * trimmed to [first, last] column where BOTH symbols are A/C/G/T; unequal lengths are
 * truncated to the shorter.  Returns 1 when at least one such column exists, else 0.
 */
int taxi_oracle_count(const uint8_t* x, int64_t nx, const uint8_t* y, int64_t ny, int32_t counts[4])
{
    const int64_t n = nx < ny ? nx : ny;
    int64_t first = -1, last = -1;
    counts[0] = counts[1] = counts[2] = counts[3] = 0;
    for (int64_t k = 0; k < n; ++k) {
        if (base_class(x[k]) < 4 && base_class(y[k]) < 4) {
            if (first < 0) first = k;
            last = k;
        }
    }
    if (first < 0) return 0;
    for (int64_t k = first; k <= last; ++k) {
        const int cx = base_class(x[k]), cy = base_class(y[k]);
        if (cx < 4 && cy < 4) {
            if (cx == cy) counts[0]++;
            else if ((cx ^ cy) == 1) counts[1]++;
            else counts[2]++;
        } else if ((cx == 4 && cy < 4) || (cy == 4 && cx < 4)) {
            counts[3]++;
        }
    }
    return 1;
}

/* out = {p, p-gaps, jc, k2p}; NaN where the reference yields None (distances.py:290-292) */
void taxi_oracle_metrics(const int32_t counts[4], double out[4])
{
    const double same = counts[0], ts = counts[1], tv = counts[2], gap = counts[3];
    const double n = same + ts + tv;
    if (!(n > 0)) { out[0] = out[1] = out[2] = out[3] = NAN; return; }
    const double p = (ts + tv) / n;
    out[0] = p;
    out[1] = (ts + tv + gap) / (n + gap);
    const double P = ts / n, Q = tv / n;
    double jc = -0.75 * log(1.0 - 4.0 * p / 3.0);
    double k2p = -0.5 * log((1.0 - 2.0 * P - Q) * sqrt(1.0 - 2.0 * Q));
    out[2] = isfinite(jc) ? jc + 0.0 : NAN;   /* +0.0 folds -0.0 into +0.0 */
    out[3] = isfinite(k2p) ? k2p + 0.0 : NAN;
}

/* taxi_oracle_metrics of n count tuples (counts int32[n][4] -> out double[n][4]) */
void taxi_oracle_metrics_batch(const int32_t* counts, int64_t n, double* out)
{
    for (int64_t k = 0; k < n; ++k) taxi_oracle_metrics(counts + 4 * k, out + 4 * k);
}

/*
 * The whole per-pair path of versus_all.py:527-552 for a list of pairs:
 * align (Biopython restatement) -> 4 counts -> 4 metrics.  Used as the CPU baseline
 * ("port") and as the parity checker for the CUDA batch entry points.
 * seqs/offsets: concatenated normalized sequences; pair p = (px[p], py[p]).
 * Any output pointer may be NULL.  threads<=0 -> all host threads (pthreads, dynamic chunks).
 */
typedef struct {
    const uint8_t* seqs; const int64_t* offsets; const int32_t* px; const int32_t* py;
    int64_t npairs; const double* sc;
    int32_t* out_score; int32_t* out_counts; double* out_metrics; int32_t* out_alnlen;
    int64_t next;      /* next unclaimed chunk start (atomic) */
    int status;
} job_t;

enum { CHUNK = 8 };

static void* worker(void* arg)
{
    job_t* job = (job_t*)arg;
    uint8_t* ba = NULL; uint8_t* bb = NULL; size_t cap = 0;
    for (;;) {
        const int64_t p0 = __atomic_fetch_add(&job->next, (int64_t)CHUNK, __ATOMIC_RELAXED);
        if (p0 >= job->npairs) break;
        const int64_t p1 = p0 + CHUNK < job->npairs ? p0 + CHUNK : job->npairs;
        for (int64_t p = p0; p < p1; ++p) {
            const int64_t ox = job->offsets[job->px[p]], oy = job->offsets[job->py[p]];
            const int32_t nA = (int32_t)(job->offsets[job->px[p] + 1] - ox);
            const int32_t nB = (int32_t)(job->offsets[job->py[p] + 1] - oy);
            if ((size_t)(nA + nB) > cap) {
                cap = (size_t)(nA + nB) * 2 + 64;
                ba = (uint8_t*)realloc(ba, cap); bb = (uint8_t*)realloc(bb, cap);
            }
            int32_t len = 0; double score = 0.0;
            int rc = taxi_oracle_align(job->seqs + ox, nA, job->seqs + oy, nB, job->sc, ba, bb, &len, &score);
            if (rc != TAXI_OK) { __atomic_store_n(&job->status, rc, __ATOMIC_RELAXED); continue; }
            int32_t c[4];
            taxi_oracle_count(ba, len, bb, len, c);
            if (job->out_score) job->out_score[p] = (int32_t)llround(score);
            if (job->out_alnlen) job->out_alnlen[p] = len;
            if (job->out_counts) memcpy(job->out_counts + 4 * p, c, sizeof c);
            if (job->out_metrics) taxi_oracle_metrics(c, job->out_metrics + 4 * p);
        }
    }
    free(ba); free(bb);
    return NULL;
}

/*
 * Alignment-free mode for a list of pairs (params.pairs.align = False, versus_all.py:522-530):
 * the four calc.seq_distances_* scans on the raw strings (distances.py:319-348), truncated to the
 * shorter one.  Same threading as the aligned batch.
 */
typedef struct {
    const uint8_t* seqs; const int64_t* offsets; const int32_t* px; const int32_t* py;
    int64_t npairs; int32_t* out_counts; double* out_metrics; int64_t next;
} count_job_t;

static void* count_worker(void* arg)
{
    count_job_t* job = (count_job_t*)arg;
    for (;;) {
        const int64_t p0 = __atomic_fetch_add(&job->next, (int64_t)256, __ATOMIC_RELAXED);
        if (p0 >= job->npairs) break;
        const int64_t p1 = p0 + 256 < job->npairs ? p0 + 256 : job->npairs;
        for (int64_t p = p0; p < p1; ++p) {
            const int64_t ox = job->offsets[job->px[p]], oy = job->offsets[job->py[p]];
            int32_t c[4];
            taxi_oracle_count(job->seqs + ox, job->offsets[job->px[p] + 1] - ox, job->seqs + oy, job->offsets[job->py[p] + 1] - oy, c);
            if (job->out_counts) memcpy(job->out_counts + 4 * p, c, sizeof c);
            if (job->out_metrics) taxi_oracle_metrics(c, job->out_metrics + 4 * p);
        }
    }
    return NULL;
}

int taxi_oracle_max_threads(void);

int taxi_oracle_count_pairs(const uint8_t* seqs, const int64_t* offsets, const int32_t* px, const int32_t* py,
                            int64_t npairs, int32_t threads, int32_t* out_counts, double* out_metrics)
{
    count_job_t job = { seqs, offsets, px, py, npairs, out_counts, out_metrics, 0 };
    if (threads <= 0) threads = taxi_oracle_max_threads();
    if (threads > 256) threads = 256;
    if (threads == 1) { count_worker(&job); return TAXI_OK; }
    pthread_t tid[256];
    int started = 0;
    for (int t = 0; t < threads; ++t)
        if (pthread_create(&tid[started], NULL, count_worker, &job) == 0) ++started;
    if (!started) count_worker(&job);
    for (int t = 0; t < started; ++t) pthread_join(tid[t], NULL);
    return TAXI_OK;
}

int taxi_oracle_max_threads(void)
{
    long n = sysconf(_SC_NPROCESSORS_ONLN);
    return n > 0 ? (int)n : 1;
}

int taxi_oracle_align_count_pairs(const uint8_t* seqs, const int64_t* offsets,
                                  const int32_t* px, const int32_t* py, int64_t npairs,
                                  const double sc[6], int32_t threads,
                                  int32_t* out_score, int32_t* out_counts, double* out_metrics,
                                  int32_t* out_alnlen)
{
    job_t job = { seqs, offsets, px, py, npairs, sc, out_score, out_counts, out_metrics, out_alnlen, 0, TAXI_OK };
    if (threads <= 0) threads = taxi_oracle_max_threads();
    if (threads > 256) threads = 256;
    if (threads == 1) { worker(&job); return job.status; }
    pthread_t tid[256];
    int started = 0;
    for (int t = 0; t < threads; ++t)
        if (pthread_create(&tid[started], NULL, worker, &job) == 0) ++started;
    if (!started) worker(&job);
    for (int t = 0; t < started; ++t) pthread_join(tid[t], NULL);
    return job.status;
}
