/*
 * taxi2_b200.h -- C ABI of the B200-native TaxI2 pairwise-distance path.
 *
 * This is the drop-in boundary: plain pointers and sizes, no torch / CUDA types.  Every entry
 * point replaces one of the two un-vendored native dependencies the reference calls on its hot
 * path (citations relative to /root/reference/src/itaxotools/taxi2/):
 *
 *   Bio.Align.PairwiseAligner(**scores).align(x, y)[0] + _format_pretty   align.py:75,151-157
 *   calc.seq_distances_{p,p_gaps,jukes_cantor,kimura2p}(x, y)            distances.py:323-347
 *
 * All functions return 0 on success or a negative taxi_status; taxi_last_error() gives the text.
 * No exceptions cross the ABI.  Undefined distances are NaN in fp64 outputs (the Python side maps
 * them to None exactly as DistanceMetric._is_number does, distances.py:290-292).
 * There is NO CPU fallback: without a CUDA device every compute entry point fails with
 * TAXI_E_CUDA.
 */
#ifndef TAXI2_B200_H
#define TAXI2_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    TAXI_OK = 0,
    TAXI_E_ARG = -1,      /* bad argument */
    TAXI_E_EMPTY = -2,    /* zero-length sequence in a pair (Biopython raises ValueError) */
    TAXI_E_NOMEM = -3,
    TAXI_E_CUDA = -4,     /* CUDA runtime error / no device */
    TAXI_E_RANGE = -5     /* scores or lengths outside what the integer DP represents exactly */
} taxi_status;

typedef struct taxi_ctx taxi_ctx; /* one per (process, device); a context is not thread-safe, but contexts of
                                     different devices may be driven by different host threads concurrently */

/* Scores.defaults order (align.py:20-27): match, mismatch, internal open, internal extend,
   end open, end extend.  Integer scores only (Scores is dict[str,int], align.py:17). */
#define TAXI_NSCORES 6

/* output-selection flags */
#define TAXI_OUT_SCORE   1u
#define TAXI_OUT_COUNTS  2u   /* int32[4] per pair: same, transitions, transversions, gap columns */
#define TAXI_OUT_METRICS 4u   /* double[4] per pair: p, p-gaps, jc, k2p (NaN = undefined)        */

const char* taxi_last_error(void);
int taxi_abi_version(void);
int taxi_device_count(void);

int taxi_ctx_create(int device, taxi_ctx** out);
void taxi_ctx_destroy(taxi_ctx* ctx);

/* Replaces the kwargs of BioPairwiseAligner(**scores), align.py:75. */
int taxi_set_scores(taxi_ctx* ctx, const int32_t scores[TAXI_NSCORES]);

/*
 * Encoder/packer: uploads `n` normalized sequences (Sequence.normalize(), sequences.py:20-25)
 * given as concatenated bytes + offsets[n+1], and keeps them resident in HBM as
 *   - 1 byte/base class codes for the DP kernels, and
 *   - 32-column bit planes (2-bit nucleotide + "real" mask + gap mask) for the counting kernel.
 * set = 0 is the row/query set (x), set = 1 the column/reference set (y).  Loading set 0 discards
 * any previous set 1 and makes set 0 serve as both (versusAll); load set 1 afterwards for
 * query x reference work (versusReference).
 */
int taxi_load_sequences(taxi_ctx* ctx, int set, const uint8_t* bytes, const int64_t* offsets, int32_t n);

/*
 * Align + count + metrics for an explicit pair list (x index into set 0, y index into set 1).
 * Replaces, per pair:  aligner.align(x, y)[0] -> _format_pretty -> 4 x calc.seq_distances_*.
 * Host output buffers (any may be NULL if its flag is clear): score int32[n], counts int32[4n],
 * metrics double[4n].  Host<->device copies happen inside the call.
 */
int taxi_align_pairs(taxi_ctx* ctx, const int32_t* px, const int32_t* py, int64_t npairs, uint32_t flags,
                     int32_t* out_score, int32_t* out_counts, double* out_metrics);

/*
 * Same for the rectangle [x0, x0+nx) x [y0, y0+ny) of SequencePairs.fromProduct (pairs.py:23-25),
 * row-major: pair p = (x0 + p / ny, y0 + p % ny).  Outputs are host buffers of nx*ny entries.
 * Any size: the rectangle is walked in blocks of whole rows (at most 2^24 pairs of device-side
 * results at a time), each block downloaded into its place.
 */
int taxi_align_rect(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                    int32_t* out_score, int32_t* out_counts, double* out_metrics);

/*
 * Device-resident variant used for kernel-only timing and by callers that keep results in HBM:
 * the out_* arguments are DEVICE pointers (e.g. torch tensors' data_ptr()), nothing is copied.
 * The work is enqueued on the context's stream; taxi_sync() waits for it.
 */
int taxi_align_rect_device(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                           int32_t* d_score, int32_t* d_counts, double* d_metrics);
int taxi_sync(taxi_ctx* ctx);

/*
 * Both orientations of a rectangle from (almost) one alignment per unordered pair: versusAll aligns
 * (x, y) AND (y, x) (versus_all.py:746).  d_* receive the nx x ny results of (x, y), t_* the ny x nx
 * results of (y, x) (all device pointers).  The dynamic programme of (y, x) is the transpose of that
 * of (x, y); the first alignment differs only where Ix and Iy tie on the traced path, which the kernel
 * detects -- those pairs (taxi_last_redo() of them, 0.7 % of COI barcodes) are re-aligned the other
 * way round, the rest mirror their result.  Bit-identical to two taxi_align_rect_device calls.
 * Synchronous.
 */
int taxi_align_rect_both_device(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                                int32_t* d_score, int32_t* d_counts, double* d_metrics,
                                int32_t* t_score, int32_t* t_counts, double* t_metrics);
/* Host buffers: (x, y) results with a row stride of ld_xy pairs, (y, x) results with a row stride of
   ld_yx pairs -- a tile and its mirror can be written straight into their places of one matrix. */
int taxi_align_rect_both(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                         int32_t* out_score, int32_t* out_counts, double* out_metrics, int64_t ld_xy,
                         int32_t* tout_score, int32_t* tout_counts, double* tout_metrics, int64_t ld_yx);
int64_t taxi_last_redo(taxi_ctx* ctx);

/*
 * Gapped strings (align.py:151-157 return value).  aln_offsets[npairs+1] are exclusive prefix
 * sums of the capacities len(x)+len(y) (computed by taxi_alignment_capacity); each alignment is
 * written right-aligned inside its slot of out_x / out_y and aln_start[p] receives the index of
 * its first byte, so alignment p is out_x[aln_start[p] : aln_offsets[p+1]].
 */
int taxi_alignment_capacity(taxi_ctx* ctx, const int32_t* px, const int32_t* py, int64_t npairs,
                            int64_t* aln_offsets);
int taxi_align_strings(taxi_ctx* ctx, const int32_t* px, const int32_t* py, int64_t npairs,
                       const int64_t* aln_offsets, uint8_t* out_x, uint8_t* out_y, int64_t* aln_start,
                       int32_t* out_score);
/*
 * Same launch, with the distance counts / metrics of taxi_align_pairs as well: what a task needs
 * when it writes aligned pairs AND distances (versus_all.py:527-552 aligns once and feeds both
 * writers from that one alignment).  Any of out_score / out_counts / out_metrics may be NULL.
 */
int taxi_align_strings_metrics(taxi_ctx* ctx, const int32_t* px, const int32_t* py, int64_t npairs,
                               const int64_t* aln_offsets, uint8_t* out_x, uint8_t* out_y, int64_t* aln_start,
                               uint32_t flags, int32_t* out_score, int32_t* out_counts, double* out_metrics);

/*
 * Alignment-free mode (params.pairs.align = False, versus_all.py:522-530): per-pair counts and
 * metrics straight from the loaded (pre-aligned) sequences.  Replaces calc.seq_distances_* applied
 * to the raw strings (distances.py:323-347).  Rectangles of a few hundred thousand pairs and more
 * run as an int8 contraction on the tensor cores (tcgen05 + TMA + TMEM, count_tc.cuh) with the
 * trim rule and the fp64 metrics fused into its epilogue; pair lists, small rectangles and rows
 * too long for its operand layout run on the bit-sliced XOR/popcount kernel (count_planes.cuh).
 * Same results either way (option "count_kernel").  Device pointers: d_counts 16-byte, d_metrics
 * 32-byte aligned (a pair's four metrics leave as one 256-bit store).
 */
int taxi_count_rect(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                    int32_t* out_counts, double* out_metrics);
int taxi_count_rect_device(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, uint32_t flags,
                           int32_t* d_counts, double* d_metrics);
int taxi_count_pairs(taxi_ctx* ctx, const int32_t* px, const int32_t* py, int64_t npairs, uint32_t flags,
                     int32_t* out_counts, double* out_metrics);

/*
 * Best match per query row (versus_reference.py:184-188, decontaminate.py:258-264): first minimum
 * of metric column `metric` (0..3) over each row of an nx x ny metrics matrix (device pointer,
 * 4 doubles per pair); NaN never wins.  out_index[x] = -1 when the whole row is undefined.
 */
/*
 * The metric formulas on their own (distances.py:319-348 applied to counts instead of strings): n tuples
 * {same, transitions, transversions, internal gap columns} -> {p, p-gaps, jc, k2p} per tuple, NaN where the
 * reference yields None.  form 0: the floating-point form every aligner epilogue uses (operation for
 * operation the reference's formulas); form 1: the table form of the alignment-free kernels (ln k in fixed
 * point; tuples of more than 2048 compared columns fall back to form 0).  Host pointers.
 */
int taxi_metrics_from_counts(taxi_ctx* ctx, const int32_t* counts, int64_t n, int32_t form, double* out_metrics);
int taxi_argmin_rows_device(taxi_ctx* ctx, const double* d_metrics, int32_t nx, int32_t ny, int32_t metric,
                            int32_t* out_index_host, double* out_value_host);

/*
 * versusReference at scale (BASELINE config C4): for every query row x0..x0+nx the best match over
 * the reference columns [y0, y0+ny) -- alignment (align != 0) or alignment-free counting of the
 * rectangle in device-resident blocks, first minimum of metric column `metric` per row, and the
 * whole winning pair: out_index[x] = its column (index into set 1; -1 = the row has no defined
 * distance), out_metrics[x][4], out_counts[x][4] (either may be NULL).  Only the winners leave the
 * device.  Column ranges of the same rows computed by different calls (or devices) are combined
 * on the host: smaller value wins, ties go to the smaller column index.
 */
int taxi_best_rows(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, int32_t metric, int32_t align,
                   int32_t* out_index, double* out_metrics, int32_t* out_counts);

/*
 * The k closest references of every query row (1 <= k <= 64; anything else is TAXI_E_ARG): the same
 * blocks as taxi_best_rows, with the k smallest keys (value of metric column `metric`, column index)
 * of each row selected on the device in ascending order -- smaller value first, equal values by the
 * smaller column.  NaN is never ranked.  Row x's slots are out_index[x*k .. x*k+k), out_metrics and
 * out_counts [x*k + r][4] (either may be NULL); a row with fewer than k defined values ends in slots
 * of index -1, NaN metrics and zero counts.  k = 1 gives taxi_best_rows' results bit for bit.
 * Column ranges of the same rows from different calls merge on the host: the k smallest keys of
 * both lists, undefined slots last.
 */
int taxi_best_rows_k(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, int32_t metric, int32_t align,
                     int32_t k, int32_t* out_index, double* out_metrics, int32_t* out_counts);

/*
 * Every pair within a distance: the same blocks as taxi_best_rows, with the pairs of each block
 * selected and compacted on the device.  Pair (x, y) is selected iff its value v of metric column
 * `metric` is not NaN and v * scale <= threshold, one fp64 multiply (scale 100 restates a
 * percentage threshold exactly as the tasks' `d * 100 <= similarity`); threshold = +inf selects
 * every defined pair.  A NaN threshold, or a scale that is not finite and positive, is TAXI_E_ARG.
 * skip_self != 0 drops the pairs (i, i) of set 0 against itself (TAXI_E_ARG with set 1 loaded).
 * The result is CSR in row-major pair order: out_row_ptr (host int64[nx + 1]) and *out_total, the
 * number of selected pairs; row x's pairs are entries out_row_ptr[x] .. out_row_ptr[x + 1], in
 * ascending reference index.  It does not depend on block size or scheduling.  ny = 0 and ny
 * above one device block are TAXI_E_ARG.
 * The pairs themselves stay held by the context until the next call that computes on it, and
 * taxi_pairs_within_fetch copies them out: out_index[total] (column, an index into set 1),
 * out_metrics[total][4], out_counts[total][4] (either may be NULL).  Fetching with no result held
 * is TAXI_E_ARG.
 */
int taxi_pairs_within(taxi_ctx* ctx, int32_t x0, int32_t nx, int32_t y0, int32_t ny, int32_t metric, int32_t align,
                      double threshold, double scale, int32_t skip_self, int64_t* out_row_ptr, int64_t* out_total);
int taxi_pairs_within_fetch(taxi_ctx* ctx, int32_t* out_index, double* out_metrics, int32_t* out_counts);

/*
 * Host-side batch formatter and subset aggregator (no GPU involved; taxi2_b200/csrc/host_format.cpp)
 * for the result files of the tasks: replaces the per-value `str.format` + `.send` writers
 * (distances.py:95-186, 244-279; versus_all.py:278-350) and the per-pair dict aggregation
 * (versus_all.py:57-95, 623-645).  All functions APPEND rows to `path` (the caller writes the
 * header line); `metrics` is the block-local [nx][ny][4] fp64 array of an align/count call,
 * `undefined` an optional [nx][ny] mask forcing the missing marker (versus_all.py:549-552),
 * `float_format` a printf format equivalent to the Python spec ("{:.4f}" -> "%.4f").
 *
 * taxi_format_pairs: one row per pair, fields joined by tabs in the order given by `segments`:
 * 0..3 = x string table k, 4..7 = y string table k-4 (tables = concatenated bytes + offsets, x
 * tables are indexed by x0 + row), 8 = the selected metric columns, 9 = the comparison type derived
 * from the genus / species subset ids (NULL = no partition; labels in ComparisonType order).
 */
int taxi_format_pairs(const char* path, const int32_t* segments, int32_t nsegments,
                      const char* const* xbytes, const int64_t* const* xoff,
                      const char* const* ybytes, const int64_t* const* yoff,
                      int32_t x0, int32_t nx, int32_t ny,
                      const double* metrics, const uint8_t* undefined,
                      const int32_t* columns, int32_t ncolumns, double scale,
                      const char* float_format, const char* missing,
                      const int32_t* xgenus, const int32_t* xspecies, const int32_t* ygenus, const int32_t* yspecies,
                      const char* const* type_labels, int32_t threads);
/* DistanceHandler.Matrix rows: x id, then one value of metric `column` per y. */
int taxi_format_matrix(const char* path, const char* xid_bytes, const int64_t* xid_off, int32_t x0, int32_t nx, int32_t ny,
                       const double* metrics, const uint8_t* undefined, int32_t column, double scale,
                       const char* float_format, const char* missing, int32_t threads);
/*
 * SequencePairHandler.Formatted records (pairs.py:51-97) of the nx*ny pairs of a row block,
 * appended to `path`: "idx / idy", aligned x, match pattern, aligned y, records separated by an
 * empty line (first_record != 0: the file is still empty).  aln_* are the arrays
 * taxi_align_strings filled for these pairs in row-major order.
 */
int taxi_format_aligned_pairs(const char* path, int32_t first_record,
                              const char* xid_bytes, const int64_t* xid_off, const char* yid_bytes, const int64_t* yid_off,
                              int32_t x0, int32_t nx, int32_t ny,
                              const uint8_t* aln_x, const uint8_t* aln_y, const int64_t* aln_start, const int64_t* aln_off,
                              int32_t threads);
/* n doubles as tab-separated text in the caller's buffer (the S^2 cells of the subset statistics files,
   versus_all.py:143-249); returns the bytes written or -(bytes needed) if `capacity` is too small. */
int64_t taxi_format_values(const double* values, int64_t n, const uint8_t* undefined, double scale,
                           const char* float_format, const char* missing, char* out, int64_t capacity);
/* SimpleAggregator state (sum, min, max, n, first-seen order) per (subset_x, subset_y), row-major order. */
int taxi_aggregate_subsets(const double* metrics, const uint8_t* undefined, int32_t x0, int32_t nx, int32_t ny,
                           int32_t column, double scale, const int32_t* xsubset, const int32_t* ysubset, int32_t nsub,
                           double* sum, double* vmin, double* vmax, int64_t* count, int64_t* first_seen, int64_t* next_order);

/*
 * The subset statistics files of versusAll (subsets/<partition>/linear/{pairs,identity}.tsv and
 * matricial/<metric>.tsv; versus_all.py:143-249, 647-684) from the arrays of taxi_aggregate_subsets, gathered
 * in first-seen key order: kx / ky = subset ids of a key (indices into the label table), mean / min / max /
 * count per metric in that order.  _rows appends one row per selected key (headers stay in Python),
 * _matrix writes a whole matrix file (runs of equal kx are its rows; t0..t3 are the pieces of the statistics
 * template around {mean}, {min}, {max}).  "NA" where count is 0.
 */
int taxi_format_subset_rows(const char* path, const char* label_bytes, const int64_t* label_off,
                            const int32_t* kx, const int32_t* ky, const uint8_t* select, int64_t nkeys, int32_t with_query,
                            int32_t nmetrics, const double* const* mean, const double* const* vmin, const double* const* vmax,
                            const int64_t* const* count, const char* float_format, int32_t threads);
int taxi_format_subset_matrix(const char* path, const char* label_bytes, const int64_t* label_off,
                              const int32_t* kx, const int32_t* ky, int64_t nkeys,
                              const double* mean, const double* vmin, const double* vmax, const int64_t* count,
                              const char* float_format, const char* t0, const char* t1, const char* t2, const char* t3, int32_t threads);

/*
 * Page-locked host buffers for the host-facing calls above: results land in them with an
 * asynchronous DMA instead of a staged pageable copy.  Plain malloc'ed buffers work too.
 */
void* taxi_host_alloc(int64_t bytes);
void taxi_host_free(void* p);

/*
 * Options: "force_general" = 1 routes every alignment through the general int32 kernel
 * (the packed 16-bit fast path is only taken when it is provably exact for the score set and
 * lengths; this switch exists so tests can compare the two); "force_top" = 1 keeps the packed
 * kernel on its top-aligned variant; "sort_columns" = 0 stops rectangle calls from visiting
 * columns of unequal length longest first (a scheduling choice only: results and their
 * positions are the same either way).  taxi_last_kernel() reports which kernel the last alignment
 * call used: 32 = gotoh_warp (int32), 16 = gotoh_pair16 top-aligned, 17 = gotoh_pair16
 * bottom-aligned, 18 = gotoh_pair16 bottom-aligned in several stripes (x longer than 1023),
 * 48 = a rectangle whose rows were grouped by length into several launches; after an alignment-free
 * call: 8 = popcount kernel, 9 = tensor-core kernel.  "count_kernel" = 1 / 2 forces the popcount /
 * the tensor-core kernel for alignment-free rectangles (0 = whichever fits; tests compare the two).
 * 33 = gotoh_warp's intra-task variant (few pairs spanning several stripes: one pair per CTA, its
 * stripes pipelined over the warps); "no_coop" = 1 keeps such launches on the one-pair-per-warp kernel.
 */
int taxi_set_option(taxi_ctx* ctx, const char* key, int value);
int taxi_last_kernel(taxi_ctx* ctx);

/* Telemetry of the last align call: kernels launched, DP cells, device milliseconds. */
int taxi_last_stats(taxi_ctx* ctx, int64_t* launches, int64_t* cells, double* kernel_ms);

#ifdef __cplusplus
}
#endif
#endif /* TAXI2_B200_H */
