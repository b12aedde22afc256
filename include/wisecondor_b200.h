/*
 * wisecondor_b200 - C ABI of the B200-native WISECONDOR hot path (libwisecondor_b200.so).
 *
 * The reference (VUmcCGP/wisecondor) has no FFI: its hot path is a set of Python functions in wisetools.py /
 * triarray.py called from wisecondor.py's tool functions.  Each entry point below replaces the body of one of
 * those functions; the citation after each declaration is the reference interface it stands in for
 * (file:line under /root/reference).  INTEGRATION.md shows the ctypes binding a maintainer of the reference
 * would add.
 *
 * Conventions
 *   - plain C types only; every pointer is either a DEVICE pointer (suffix _d) or a HOST pointer (suffix _h);
 *   - every function returns 0 on success or a negative wc_status; wc_last_error() gives the text;
 *   - work is enqueued on the cudaStream_t passed as `stream` (a void*; NULL = legacy default stream);
 *     functions documented as "synchronous" wait for their own work before returning;
 *   - nothing here falls back to the CPU: without a CUDA device every compute entry point fails with
 *     WC_ERR_CUDA.
 */
#ifndef WISECONDOR_B200_H
#define WISECONDOR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct wc_ctx wc_ctx;

typedef enum wc_status {
    WC_OK = 0,
    WC_ERR_ARG = -1,      /* bad argument */
    WC_ERR_CUDA = -2,     /* CUDA runtime / driver error, or no device */
    WC_ERR_NOMEM = -3,    /* device allocation failed */
    WC_ERR_INTERNAL = -4  /* invariant violated (please report) */
} wc_status;

/* One segmentation call, the tuple the reference's TriArr.segmentTri returns (triarray.py:78):
 * (value, (x, y)) with inclusive cleaned-bin coordinates inside the chromosome. */
typedef struct wc_call {
    int32_t sample;   /* index into the batch */
    int32_t chrom;    /* 0-based index into the chromosome list given to wc_segment_batch */
    int32_t x;        /* first cleaned bin of the run */
    int32_t y;        /* last cleaned bin of the run (inclusive) */
    double z;         /* Stouffer z of the run */
} wc_call;

/* ---- context ------------------------------------------------------------------------------------------ */
/* Create a context bound to CUDA device `device`.  Returns NULL on failure (see wc_last_error). */
wc_ctx* wc_create(int device);
void wc_destroy(wc_ctx* ctx);
const char* wc_last_error(void);
/* Library version string and number of SMs of the bound device (0 if none). */
const char* wc_version(void);
int wc_sm_count(const wc_ctx* ctx);
/* Device-time (ms, CUDA events on `stream`) of the named phases of the most recent call:
 * which: 0 = centre+norms (K4), 1 = distance+streaming top-k (K5), 2 = exact re-score/finalise (K6),
 *        3 = exhaustive fallback rows, 4 = z-score passes (K8), 5 = segmentation (K9), 6 = test sample prep (K7),
 *        7 = PCA bin means + Gram matrix (K2), 8 = the first (threshold) pass of a symmetric K5, part of 1,
 *        9 = the symmetric pass of a sharded search, part of 1.  Phases of asynchronous calls are read lazily (this call waits). */
double wc_last_phase_ms(wc_ctx* ctx, int which);
/* Counters of the most recent calls: which: 0 = kernel launches of wc_newref_topk, 1 = its rows sent to the exhaustive
 * fallback, 2 = tiles of the plain search, 3 = tiles computed (fewer: symmetric search), 4 = CTAs launched for K5, 5 = kernel launches of
 * the last wc_zscore_batch, 6 = of the last wc_segment_batch, 7 = of the last wc_newref_prep;
 * 16 + p = (bin, sample) pairs that z-score pass p of the last wc_zscore_batch computed (synchronises). */
long long wc_last_counter(const wc_ctx* ctx, int which);

/* Raw device buffers for hosts without an allocator of their own (the command line runs without PyTorch this way;
 * library users normally pass pointers of their own tensors).  Copies are synchronous on the legacy default stream. */
int wc_device_count(void);
void* wc_dev_alloc(wc_ctx* ctx, size_t bytes);                 /* NULL on failure */
int wc_dev_free(wc_ctx* ctx, void* p);
int wc_copy_h2d(wc_ctx* ctx, void* dst_d, const void* src_h, size_t bytes);
int wc_copy_d2h(wc_ctx* ctx, void* dst_h, const void* src_d, size_t bytes);
int wc_dev_sync(wc_ctx* ctx);                                  /* cudaDeviceSynchronize on the context's device */

/* Debug aid, host only (no device, no context): the symmetric search's tile lists and CTA schedule for the 128-bin
 * blocks of rank `rank` of `world` (1/frac of the block pairs in the first pass; `grid` CTAs, `group` CTAs per row block
 * in rounds when rounds_on).  out: [nb, b0, b1, nA, nB, piecesA, piecesB, 0][off_a][off_b][list_a][list_b][pieces: cta,
 * row block, q0, q1, step]...[skip_lo nb][skip_n nb]; *used = ints needed.  The CPU tests check that every block pair
 * that holds a bin pair of different chromosomes reaches both of its blocks exactly once. */
int wc_debug_sym_plan(int N, const int* chrom_bins_h, int nchrom, int frac, int world, int rank, int grid, int group,
                      int rounds_on, int* out, long long out_ints, long long* used);

/* Debug aid: enable (1) / disable (0) per-CTA cycle counters in the distance kernel and copy the counters of the
 * most recent search to out_h (grid x 8 int64: total, wait-on-TMA, epilogue, prune, tiles, prunes, emitted by
 * thread 0, reserved).  Returns the number of CTAs copied, or a negative wc_status. */
int wc_debug_profile(wc_ctx* ctx, int enable, long long* out_h, int max_ctas);

/* Tuning knobs.  Results never depend on them.
 *   "k5_sym"    whole-matrix searches contract every unordered pair of bin blocks once (symmetric search): 0 = off (plain
 *               search), f in 2..64 = on, with 1/f of the block pairs computed in the first (threshold) pass.  Default 8.
 *   "k5_group"  CTAs sharing a row block per scheduling round (0 = automatic), "k5_stages" TMA ring depth (0 = automatic),
 *   "k5_lag"    chunks (0..4) by which half of the distance kernel's MMA warps trail the other half,
 *   "k5_f16"    the FILTER of the distance kernel (the exact fp64 re-score that decides the result is the same for all):
 *               0 = fp64 contraction on DMMA, 1 = fp16 on mma.sync, 2 = fp16 on tcgen05 with TMEM accumulators (default),
 *   "k5_pivots" 1 = pivot pass before the search proper with the tcgen05 filter (default), 0 = none,
 *   "k6_split"  the exact re-score: 1 = select -> streaming re-score on bulk copies -> rank (default; needs an even number
 *               of samples), 0 = one fused kernel; "k6_chunk" samples per bulk copy, "k6_warps" consumer warps per SM,
 *               "k6_prod" producer warps per consumer warp (0 = defaults 100 / 4 / 2), "k6_g4" 1 = candidate rows four per
 *               TMA request (tile::gather4) instead of one bulk copy each (default 0: measured no faster),
 *   "k6_select" 1 = streaming two-level histogram select (default: no limit on a row's candidate entries), 0 = entries
 *               held in shared memory + bisection (rows with more than 1024 entries: CTA-per-row select),
 *   "k6_parts"  wc_newref_topk_host only: row ranges (1..16, default 4) the last stage runs in; every finished range but the
 *               last is copied to the host while the next one is re-scored. */
int wc_set_option(wc_ctx* ctx, const char* key, double value);

/* Debug: searches that run the tcgen05 filter (k5_f16 = 2) also store every filter distance they compute into
 * out_d[(i - row_begin) * ld + j] (DEVICE float, caller-owned).  NULL switches it off.  Used by the tests that measure the
 * filter's error against the margin its exactness argument assumes. */
int wc_debug_filter_scores(wc_ctx* ctx, float* out_d, int ld);
/* debug: K5t's pivot selection alone - the R bins of smallest fp32 norm (ties by bin), sorted by bin; device pointers */
int wc_debug_pivot_select(wc_ctx* ctx, const float* n32_d, int N, int R, int* ids_d);

/* ABI version of this header; wc_abi_version() returns the one the library was built from (the binding refuses a mismatch). */
#define WC_ABI_VERSION 3
int wc_abi_version(void);

/* ---- newref: reference-bin search --------------------------------------------------------------------- */
/* Replaces getReference + getRefForBins (wisetools.py:364-398, 298-325) for target rows
 * [row_begin, row_end) - the rows wisetools.getPart (wisetools.py:358-361) hands one part.
 *   corrected_d  DEVICE  N x S float64, bin-major C order (row = bin, S contiguous): the `correctedData` of
 *                        the prep npz (wisecondor.py:106)
 *   chrom_bins_h HOST    nchrom masked bins per chromosome (`maskedChromBins`, wisecondor.py:93); sum == N
 *   refsize              `selectRefAmount` / -refsize (wisecondor.py:379), 1..384 (larger: wc_newref_topk_wide)
 *   idx_d        DEVICE  (row_end-row_begin) x refsize int32: positions in the other-chromosome concatenation
 *   dist_d       DEVICE  (row_end-row_begin) x refsize float64: squared distances, ascending
 * Rows are the first `refsize` candidates ordered by (distance, index); unfilled slots hold -1 / 1e10.
 * Distances are re-scored in the reference's operation order (sequential over samples, separately rounded
 * subtract/multiply/add) and are bit-identical to the reference's.  Synchronous. */
int wc_newref_topk(wc_ctx* ctx, const double* corrected_d, int N, int S, const int* chrom_bins_h, int nchrom,
                   int row_begin, int row_end, int refsize, int32_t* idx_d, double* dist_d, void* stream);

/* Largest refsize wc_newref_topk_wide accepts. */
#define WC_WIDE_REFSIZE_MAX 4096

/* The same search for 1 <= refsize <= WC_WIDE_REFSIZE_MAX, with the arguments and output contract of wc_newref_topk
 * (larger refsize: WC_ERR_ARG before any memory is touched).  Computes every distance of a chunk of target rows exactly,
 * in the reference's operation order, then selects and ranks each row; chunks of a multiple of 128 rows whose distances
 * take at most 1 GiB of device memory.  Phases: 1 = distances, 2 = select + rank; counter 0 = kernel launches,
 * 2 = rows per chunk.  Synchronous. */
int wc_newref_topk_wide(wc_ctx* ctx, const double* corrected_d, int N, int S, const int* chrom_bins_h, int nchrom,
                        int row_begin, int row_end, int refsize, int32_t* idx_d, double* dist_d, void* stream);

/* Same call with HOST buffers (copies in and out inside the call): the form toolNewrefPart
 * (wisecondor.py:111-132) would bind. */
int wc_newref_topk_host(wc_ctx* ctx, const double* corrected_h, int N, int S, const int* chrom_bins_h,
                        int nchrom, int row_begin, int row_end, int refsize, int32_t* idx_h, double* dist_h);

/* ---- newref on several GPUs: sharded symmetric search ------------------------------------------------------------
 * Replaces the `newrefpart` fan-out + `newrefpost` concatenation (wisecondor.py:111-158) when all parts run on the GPUs of
 * one node: since d(i, j) = d(j, i), every unordered pair of 128-bin blocks is contracted ONCE in the whole job and serves
 * both bins.  Rank r of `world` (one process per GPU, each holding the whole corrected matrix) owns nb/world consecutive
 * blocks of bins: it computes the tiles whose row block it owns and finalises its own bins.  Call order on every rank:
 *   wc_newref_shard_dims    sizes of the exchange buffers (out6: rows_per, in_cap, thr_len, row0, row1, nb)
 *   wc_newref_shard_begin   K4 + threshold pass; writes thr_d[thr_len] (u64 keys; the owned bins' thresholds)
 *   -> all-reduce MIN of thr_d over the ranks, read as int64 (all real keys are negative int64, padding is 0)
 *   wc_newref_shard_sweep   symmetric pass; fills in_key_d / in_j_d [world*rows_per][in_cap], in_cnt_d [world*rows_per]:
 *                           what this rank's tiles found for EVERY bin on their column side
 *   -> all-to-all of the three arrays in `world` equal splits of rows_per bins (split o goes to rank o)
 *   wc_newref_shard_finish  exact re-score / ranking of the bins [row0, row1): idx_d, dist_d (row1-row0) x refsize, as
 *                           wc_newref_topk writes them; recv_* = the all-to-all's outputs.  Synchronous.
 * The caller gathers the ranks' rows (they are consecutive and ordered by rank).  Results are identical to
 * wc_newref_topk over the same rows.  All pointers DEVICE except chrom_bins_h. */
int wc_newref_shard_dims(const wc_ctx* ctx, int N, int refsize, int world, int rank, long long* out6);
int wc_newref_shard_begin(wc_ctx* ctx, const double* corrected_d, int N, int S, const int* chrom_bins_h, int nchrom,
                          int refsize, int rank, int world, unsigned long long* thr_d, void* stream);
int wc_newref_shard_sweep(wc_ctx* ctx, unsigned long long* thr_d, unsigned long long* in_key_d, int* in_j_d,
                          int* in_cnt_d, void* stream);
int wc_newref_shard_finish(wc_ctx* ctx, const unsigned long long* recv_key_d, const int* recv_j_d, const int* recv_cnt_d,
                           int32_t* idx_d, double* dist_d, void* stream);

/* ---- newref: normalisation, mask, PCA residual ------------------------------------------------------------ */
/* Together these replace toNumpyArray (wisetools.py:240-264) and trainPCA (wisetools.py:89-101) as called from
 * toolNewrefPrep (wisecondor.py:91-96).  counts_d: DEVICE S x Nraw int32, one row per sample = its autosomal count
 * arrays concatenated (all samples must have equal chromosome lengths, as wisetools.py:250 requires). */

/* mask_d (DEVICE Nraw uint8) = sumPerBin > 0 (wisetools.py:259-260): some sample has a read in the bin. */
int wc_newref_mask(wc_ctx* ctx, const int32_t* counts_d, int S, int Nraw, uint8_t* mask_d, void* stream);

/* masked_d (DEVICE N x S float64, bin-major) = counts / per-sample total at the masked-in bins masked_raw_d
 * (wisetools.py:255-256, 261). */
int wc_newref_normalize(wc_ctx* ctx, const int32_t* counts_d, int S, int Nraw, const int32_t* masked_raw_d, int N,
                        double* masked_d, void* stream);

/* First half of PCA(n_components).fit (wisetools.py:90-92): mean_d (DEVICE N) = per-bin mean over samples (numpy's
 * summation order: bit-identical to pca.mean_), gram_d (DEVICE S x S) = Xc^T Xc of the centred matrix.  The caller
 * takes the top eigenpairs of gram_d on the host (numpy/scipy LAPACK; S is 600..2000). */
int wc_pca_gram(wc_ctx* ctx, const double* masked_d, int N, int S, double* mean_d, double* gram_d, void* stream);

/* Second half + transform / inverse_transform / divide (wisetools.py:94-96): eigvec_d DEVICE S x ncomp (columns =
 * eigenvectors of the Gram matrix, largest first), sigma_h HOST ncomp singular values (sqrt of the eigenvalues).
 * components_d DEVICE ncomp x N (pca.components_, sign not normalised), corrected_d DEVICE N x S (bin-major:
 * `correctedData`, wisecondor.py:106). */
int wc_pca_apply(wc_ctx* ctx, const double* masked_d, int N, int S, const double* mean_d, const double* eigvec_d,
                 const double* sigma_h, int ncomp, double* components_d, double* corrected_d, void* stream);

/* ---- test: batched sample preparation, within-sample z-scores, Stouffer segmentation ------------------------ */
/* Layout: the batch's corrected values are T[bin][sample] with leading dimension ldb (a multiple of 32, >= B). */

/* Once per reference: replaces the per-bin `index[distances[i] < cutoff]` selection and the other-chromosome
 * concatenation trySample rebuilds per chromosome (wisetools.py:420-424).
 *   indexes_d/distances_d DEVICE N x k: the reference npz's `indexes`, `distances` (wisecondor.py:164-165)
 *   cutoff                getOptimalCutoff's value (wisetools.py:328-336; sample independent, host numpy)
 *   table_d  DEVICE N x wc_table_stride(k) int32: table[i][0..count[i]) = GLOBAL masked-bin ids of bin i's usable
 *            reference bins, in stored order (rows are padded to a multiple of 4 entries for 16-byte loads)
 *   count_d  DEVICE N int32
 *   rev_off_d DEVICE N+1 int32, rev_idx_d DEVICE N x wc_table_stride(k) int32: the reverse table (CSR) - for every bin
 *            the bins that use it as a reference bin; lets the later passes of wc_zscore_batch touch only what a
 *            newly marked bin can change
 * k (the npz's refsize) may be any value >= 1 with N x wc_table_stride(k) < 2^31 (k <= 37 260 at 50 kb, 7 452 at
 * 10 kb); larger values are refused with WC_ERR_ARG before any memory is touched. */
int wc_table_stride(int k);
int wc_test_table(wc_ctx* ctx, const int32_t* indexes_d, const double* distances_d, int N, int k,
                  const int* chrom_bins_h, int nchrom, double cutoff, int32_t* table_d, int32_t* count_d,
                  int32_t* rev_off_d, int32_t* rev_idx_d, void* stream);

/* Replaces toNumpyRefFormat + applyPCA (wisetools.py:267-278, 104-113) for B samples.
 *   counts_d     DEVICE B x Nraw int32: per sample the autosomal read counts, each chromosome zero-padded /
 *                truncated to the reference's `chromosome_sizes` (wisetools.py:270-272; the host does that and
 *                scaleSample, wisetools.py:220-237)
 *   masked_raw_d DEVICE N int32: raw position of every masked-in bin (np.flatnonzero(mask))
 *   pca_mean_d N, pca_components_d ncomp x N: the reference npz's PCA (wisecondor.py:168-169)
 *   test_d       DEVICE N x ldb float64 out: x / ((x - mean) C^T C + mean), sample-minor.  Asynchronous. */
int wc_test_prep(wc_ctx* ctx, const int32_t* counts_d, int B, int Nraw, const int32_t* masked_raw_d, int N,
                 const double* pca_mean_d, const double* pca_components_d, int ncomp, double* test_d, int ldb,
                 void* stream);

/* applyPCA alone (wisetools.py:104-113) on already normalised, masked vectors x_d (DEVICE B x N float64). */
int wc_apply_pca(wc_ctx* ctx, const double* x_d, int B, int N, const double* pca_mean_d,
                 const double* pca_components_d, int ncomp, double* test_d, int ldb, void* stream);

/* Replaces repeatTest / trySample (wisetools.py:438-448, 407-435) for B samples: `repeats` passes, bins with
 * abs(z) >= z_threshold are marked -1 between passes and stop serving as reference values.
 *   z_d, r_d DEVICE B x N float64 (sample-major), refsizes_d DEVICE B x N int32: resultsZ, resultsR, refSizes of
 *   the last pass;  asdef_d DEVICE B float64: stdDevSum / stdDevNum.  Bit-identical to the reference (numpy's
 *   summation order).  copy_init_d (DEVICE N x ldb, or NULL = test_d) is trySample's `testCopy`: the values the
 *   reference bins are gathered from in the first pass, -1 where already marked.  k: the table's refsize, as given
 *   to wc_test_table (any k >= 1 with N x wc_table_stride(k) < 2^31; above 512 the wide-refsize kernels run).
 *   Asynchronous. */
int wc_zscore_batch(wc_ctx* ctx, const double* test_d, const double* copy_init_d, int N, int B, int ldb,
                    const int32_t* table_d, const int32_t* count_d, const int32_t* rev_off_d, const int32_t* rev_idx_d,
                    int k, double z_threshold, int repeats, double* z_d, double* r_d, int32_t* refsizes_d,
                    double* asdef_d, void* stream);

/* Replaces the chromosome loop of toolTest (wisecondor.py:233-238): fillTriMin / fillTri (wisetools.py:466-487) +
 * TriArr.segmentTri (triarray.py:59-84) on the bins with refsizes >= minrefbins (wisecondor.py:215-218), for the
 * chromosomes listed (0-based) in chromosomes_h.
 *   r_d, mineffectsize  -mineffectsize (wisecondor.py:460): when > 0, a run only counts if abs(median(R) - 1) >=
 *                  mineffectsize (r_d = DEVICE B x N resultsR); 0 = plain fillTri, r_d may be NULL
 *   cwz_d          DEVICE B x nsel float64: zTriangle.getValue(0, n-1) (wisecondor.py:237)
 *   cleaned_bins_d DEVICE B x nsel int32: kept bins of each listed chromosome (`cleanedBins`, wisecondor.py:220-222)
 *   calls_d        DEVICE B x max_calls wc_call, ncalls_d DEVICE B int32: unordered; sort by (chrom, x)
 * Non-finite z of a kept bin (reference sigma 0) gives the NaN / inf calls numpy's argmax/argmin give the reference, with
 * and without the effect-size filter (a NaN ratio fails the median test of every run that holds it, wisetools.py:483).
 * Synchronous. */
int wc_segment_batch(wc_ctx* ctx, const double* z_d, const double* r_d, const int32_t* refsizes_d, int N, int B,
                     const int* chrom_bins_h, int nchrom, const int* chromosomes_h, int nsel, int minrefbins,
                     double z_threshold, double mineffectsize, int min_search, double* cwz_d,
                     int32_t* cleaned_bins_d, wc_call* calls_d, int32_t* ncalls_d, int max_calls, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* WISECONDOR_B200_H */
