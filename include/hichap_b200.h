/*
 * hichap_b200.h -- C ABI of libhichap_b200.so: the B200 (sm_100a) implementation of the
 * hot path of HiCHap's `matrix` stage (reference: HiCHap/matrixBuilding.py).
 *
 * The reference is pure Python and has no FFI of its own; its boundary for this path is the
 * set of Python callables in HiCHap/matrixBuilding.py plus the `cooler balance` command line.
 * Each entry point below names the reference code (file:line, relative to the reference
 * root) whose arithmetic it replaces.  The Python mirror of those callables lives in
 * hichap_master_b200/matrixBuilding.py and binds this ABI with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - Every pointer is a DEVICE pointer unless its name starts with `h_` (host).  The caller
 *     owns all memory; the library borrows it for the duration of the (stream-ordered) call.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - Return value: 0 = success, negative = error; hc_last_error() returns the message of the
 *     last failing call on the calling thread.
 *   - Dense matrices are int32 row-major with leading dimension `ld` (elements, multiple of 4,
 *     rows 16-byte aligned); a "dense batch" is one buffer holding several such matrices,
 *     described by three small device tables (element offset, side n, ld per matrix).
 *   - No CPU fallback exists: every entry point launches CUDA kernels.
 */
#ifndef HICHAP_B200_H
#define HICHAP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HC_OK 0
#define HC_ERR_CUDA (-1)
#define HC_ERR_ARG (-2)
#define HC_ERR_NCCL (-3)
#define HC_ERR_UNSUPPORTED (-4)

#define HC_ABI_VERSION 2

int hc_version(void);
/* Optional, once per device: keep the library's stream-ordered scratch cached between calls. */
int hc_init(void);
/* Bytes the library's stream-ordered pool (the default cudaMallocAsync pool, kept by hc_init) holds without using them. */
int64_t hc_mempool_free_bytes(void);
const char* hc_last_error(void);
/* Number of kernels this library has launched in this process (bench.py's `gpu_launches`). */
int64_t hc_launch_count(void);

/* ------------------------------------------------------------------------------------------
 * (a) Valid-pair binning into dense integer tiles.
 * Pairs are columnar int32 (chromosome index into the sorted chromosome table, fragment
 * mid-point); a chromosome index < 0 means "filtered out" (matrixBuilding.py:577-580).
 * `mark` (nullable) is 0=Both 1=R1 2=R2 3=other (matrixBuilding.py:1133, :1274, :1290).
 * ---------------------------------------------------------------------------------------- */
#define HC_BIN_SYM_ALL 0   /* every pair, symmetric:  M[b1][b2]++ and, if b1!=b2, M[b2][b1]++ */
#define HC_BIN_SYM_BOTH 1  /* only mark==Both, symmetric (matrixBuilding.py:1131-1161)        */
#define HC_BIN_ONESIDED 2  /* only mark!=Both: R1 -> M[b1][b2]++, else M[b2][b1]++ (:1295-1301) */

/* Per-chromosome ("local") matrices: replaces the loop at matrixBuilding.py:595-603 (and
 * :844-852, :1153-1161, :1191-1199, :1295-1301, :1409-1415).  Only pairs with c1==c2 count;
 * bin = pos / res.  Pairs whose bin falls outside the matrix are counted into *oob (nullable)
 * instead of being applied (the reference would raise IndexError). */
int hc_bin_pairs_local(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                       const uint8_t* mark, int64_t npairs, int32_t res, int32_t mode,
                       int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                       const int32_t* mat_ld, int32_t nchrom, unsigned long long* oob,
                       void* stream);

/* Same result as hc_bin_pairs_local for the SYMMETRIC modes when the matrices are symmetric on
 * entry (e.g. freshly zeroed), with most updates resolved in L2: only the upper triangle is
 * updated, pairs fewer than band_width bins apart go to a compact nbins x band_width accumulator
 * (work: hc_bin_band_work_bytes) that stays L2-resident, then the band is merged into the tiles
 * and the upper triangle mirrored.  bin_off: device int64[nchrom+1] concatenated bin offsets;
 * h_mat_n: host copy of the sides; band_width: power of two in [32, 1024]. */
int64_t hc_bin_band_work_bytes(int64_t nbins, int32_t band_width);
int hc_bin_pairs_local_banded(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                              const uint8_t* mark, int64_t npairs, int32_t res, int32_t mode,
                              int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                              const int32_t* mat_ld, const int64_t* bin_off, int32_t nchrom,
                              const int32_t* h_mat_n, int32_t band_width, unsigned long long* oob,
                              void* work, void* stream);

/* The same three phases, separately callable, so that a caller can accumulate pairs chunk by chunk
 * while later chunks are still crossing PCIe (the reference reads the whole bed stream before it has
 * a matrix, matrixBuilding.py:573-592): begin zeroes the band; accumulate may be called any number of
 * times (chrom_is_u8 != 0: c1/c2 are uint8 columns, 255 = filtered, 4-byte aligned; else int32 columns);
 * finish merges the band into the tiles and mirrors the upper triangle. */
int hc_bin_band_begin(void* work, int64_t nbins, int32_t band_width, void* stream);
int hc_bin_band_accumulate(const void* c1, const int32_t* p1, const void* c2, const int32_t* p2,
                           const uint8_t* mark, int64_t npairs, int32_t chrom_is_u8, int32_t res, int32_t mode,
                           int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                           const int32_t* mat_ld, const int64_t* bin_off, int32_t nchrom,
                           int32_t band_width, unsigned long long* oob, void* work, void* stream);
int hc_bin_band_finish(int32_t* mats, const int64_t* mat_off, const int32_t* mat_n, const int32_t* mat_ld,
                       const int64_t* bin_off, int32_t nchrom, const int32_t* h_mat_n, int32_t band_width,
                       void* work, void* stream);

/* Inter-chromosomal imputation on the genome-wide haplotype matrix: replaces the per-line loops of
 * matrixBuilding.py:1302-1378 (M_M file, own_is_p = 0) and :1416-1492 (P_P file, own_is_p = 1), bug for
 * bug.  Only lines with mark != Both and c1 != c2 act.  `un` (total x total, leading dimension ld) is the
 * UN-imputed matrix the vote reads; `imp` receives the +1s.  start_m / start_p: device int64[nchrom]
 * first bins of the maternal / paternal copy of each chromosome.  half_width = Imputation_region // res;
 * nb_i / nb_j: device int32[npts] window indices of GetNeighborhoodIndex (:721-732).
 * last_qualifying (nullable, device, initialised to -1 by the caller): atomic max of the index of lines
 * that passed the window bounds checks -- for the M_M file it identifies the window the reference
 * leaves in `M_M_sub`, which its P_P R1 branch then reads (:1448).  For the P_P file the caller passes
 * that window's disc sum in stale_sum (stale_state 0), or stale_state 1 / 2 when the reference would
 * raise NameError / IndexError at the first such line; *stale_needed (device int32, zeroed by the caller)
 * is then set if one exists. */
int hc_impute_inter(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                    const uint8_t* mark, int64_t npairs, int32_t res, const int64_t* start_m,
                    const int64_t* start_p, int32_t nchrom, int32_t own_is_p, const int32_t* un,
                    int32_t* imp, int32_t total, int64_t ld, int32_t half_width, const int32_t* nb_i,
                    const int32_t* nb_j, int32_t npts, int64_t imputation_min, double imputation_ratio,
                    int32_t stale_state, int64_t stale_sum, long long* last_qualifying,
                    int32_t* stale_needed, void* stream);

/* Chromosome-id columns may cross PCIe as uint8 (255 = filtered chromosome): widen to the int32
 * columns the binning entry points take (255 -> -1). */
int hc_widen_u8_i32(const uint8_t* src, int32_t* dst, int64_t n, void* stream);

/* dst[i] += src[i]: replicate merge of dense tiles (matrixBuilding.py:1700-1719). */
int hc_add_i32(int32_t* dst, const int32_t* src, int64_t n, void* stream);

/* Genome-wide ("whole") matrix: replaces matrixBuilding.py:582-592 (and :831-841, :1144-1151,
 * :1182-1189, :1217-1221, :1239-1243, :1285-1293).  bin1 = p1/res + start1[c1],
 * bin2 = p2/res + start2[c2]; start tables are device int64[nchrom].  HC_BIN_ONESIDED only
 * applies cis pairs (c1==c2); the inter-chromosomal one-sided branch is the reference's
 * neighbourhood imputation, which is outside this library (SURVEY.md section 8f). */
int hc_bin_pairs_whole(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                       const uint8_t* mark, int64_t npairs, int32_t res, int32_t mode,
                       const int64_t* start1, const int64_t* start2, int32_t nchrom,
                       int32_t* M, int32_t total, int64_t ld, unsigned long long* oob,
                       void* stream);

/* Dense -> sparse marshalling: replaces np.triu/np.nonzero at matrixBuilding.py:489-503 and
 * :515-521.  Two calls: count (writes row_ptr[nrows+1], exclusive prefix sum, row-major order)
 * then extract (bin1, bin2 block-local; val).  triu=1 keeps col>=row only.
 * `is_f64` selects int32 (0) or float64 (1) element type for M / val. */
int hc_dense_nonzero_count(const void* M, int64_t ld, int32_t nrows, int32_t ncols, int32_t triu,
                           int32_t is_f64, int64_t* row_ptr, void* stream);
int hc_dense_nonzero_extract(const void* M, int64_t ld, int32_t nrows, int32_t ncols, int32_t triu,
                             int32_t is_f64, const int64_t* row_ptr, int32_t* bin1, int32_t* bin2,
                             void* val, void* stream);

/* The same marshalling for EVERY matrix of a dense batch in two launches, producing the
 * reference's record layout directly: records[i] = {int64 bin1, int64 bin2, float64 IF} (24 B,
 * the S_dtype of matrixBuilding.py:460-461), upper triangle, row-major; the records of matrix p
 * are the contiguous range [row_ptr[bin_off[p]], row_ptr[bin_off[p+1]]).  row_ptr: nbins+1. */
int hc_dense_batch_triu_count(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                              const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                              int64_t nbins, int64_t* row_ptr, void* stream);
int hc_dense_batch_triu_records(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                                int64_t nbins, const int64_t* row_ptr, void* records, void* stream);

/* ------------------------------------------------------------------------------------------
 * (b) ICE balancing == `cooler balance --ignore-diags K [--cis-only]`
 * (call sites matrixBuilding.py:708, :713, :1537, :1542, :1761, :1766; arithmetic restated in
 * oracle/cooler_ice.py from cooler.balance.balance_cooler).
 * ---------------------------------------------------------------------------------------- */
typedef struct hc_ice_params {
    double tol;            /* 1e-5 */
    double mad_max;        /* 5    */
    int32_t min_nnz;       /* 10   */
    int32_t min_count;     /* 0    */
    int32_t ignore_diags;  /* HiCHap passes 1 */
    int32_t max_iters;     /* 200  */
    int32_t rescale_marginals; /* 1 */
    int32_t poll_every;    /* host polls the device-side done counter every this many launches */
} hc_ice_params;

/* Filter marginals of a dense batch of symmetric matrices (one balancing problem per matrix,
 * bins concatenated: problem p owns bias[bin_off[p] .. bin_off[p+1])).  Writes, per bin, the
 * number of non-zero off-band pixels (nnz_marg) and their sum (marg, as float64).
 * Replaces the two pre-iteration marginalisations of balance_cooler. */
int hc_ice_dense_marginals(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                           const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                           int32_t ignore_diags, double* nnz_marg, double* marg, void* stream);

/* Bin filters -> initial bias (1 = keep, 0 = masked): min_nnz, min_count, then MAD-max on
 * log-marginals normalised by the per-chromosome median (chrom_off: device int64[nchrom+1]
 * over the concatenated bins).  `marg` is modified in place (divided by the chromosome
 * medians) exactly as cooler does.  `work` must hold 2*nbins doubles. */
int hc_ice_filter_bins(const double* nnz_marg, double* marg, int64_t nbins,
                       const int64_t* chrom_off, int32_t nchrom, const hc_ice_params* h_params,
                       double* bias, double* work, void* stream);

/* Per-problem results of a balancing run (device array of nprob of these). */
typedef struct hc_ice_result {
    double scale;      /* mean of the non-zero marginals at the last iteration (NaN if empty) */
    double var;        /* their population variance                                           */
    int32_t iters;     /* iterations executed                                                 */
    int32_t converged; /* var < tol                                                           */
} hc_ice_result;

/* Host-side record of one balancing run. */
typedef struct hc_ice_run_info {
    int32_t launches; /* kernels launched by the call (iterations + finalise)                  */
    float loop_ms;    /* device time of the iteration loop (CUDA events on `stream`)           */
    int32_t packed;   /* dense: 1 when the loop streamed the uint8 + overflow encoding; CSR: 2 = column-blocked */
    float pack_ms;    /* dense: device time of building that encoding (once per call)          */
    int64_t overflow_cells; /* dense, packed: cells whose weighted count exceeds 255; CSR, packed == 2 (column-blocked
                               4-byte entries): stored entries incl. segment padding                              */
    float stream_full_ms;   /* dense, HC_ICE_TIME_KERNEL=1: mean duration of a stream-kernel launch  */
    int32_t stream_full_launches; /* ... over this many launches in which every problem was active */
} hc_ice_run_info;

/* Iterate every problem of the dense batch to convergence, independently (own loop, scale and
 * early exit -- cooler's _balance_cisonly; one problem == _balance_genomewide).
 * bias: in = initial bias from the filters, out = final weights (NaN for masked bins, divided
 * by sqrt(scale) when rescale_marginals).  All scratch is stream-ordered and library-owned (ABI v1 took a
 * `work` pointer here that was never used; v2 drops it).  The reduction over the
 * marginals, the bias update, the rescale and the convergence test all run on the device
 * (stream kernel + per-chromosome update kernel, replayed as a CUDA graph); the host only polls a
 * done counter.  By default the tiles are first re-encoded into uint8 + an overflow list (exact; a
 * quarter of the bytes per iteration; HC_ICE_PACKED=0 streams the int32 tiles instead) in stream-ordered
 * scratch of 1 byte per tile element.  Every mat_ld must be a multiple of 128 elements (512-byte rows). */
int hc_ice_dense_balance(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                         const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                         const int32_t* h_mat_n, const hc_ice_params* h_params, double* bias,
                         hc_ice_result* results, hc_ice_run_info* h_info, void* stream);

/* ------------------------------------------------------------------------------------------
 * (a') Sort path: pairs -> keys -> radix sort -> reduce-by-key -> SYMMETRIC CSR (both triangles
 * stored) with integer counts.  Replaces the dense accumulation of matrixBuilding.py:559-603
 * where the dense matrix is infeasible (genome-wide 10 kb / 5 kb).  The reference's
 * upper-triangular records (matrixBuilding.py:489-503) are the col >= row subset.
 * ---------------------------------------------------------------------------------------- */

/* key = (row << col_bits) | col with row/col = pos/res + start[chrom]; every off-diagonal pair
 * yields two keys (row,col) and (col,row), a diagonal pair one; dropped pairs (filtered
 * chromosome, or trans when cis_only) yield the padding key ~0.  keys: 2*npairs entries.
 * *n_valid (device) receives the number of real keys; *oob counts out-of-range pairs.
 * start: device int64[nchrom]; chrom_bins: device int32[nchrom] (bins per chromosome). */
int hc_pairs_to_keys(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                     int64_t npairs, int32_t res, const int64_t* start, const int32_t* chrom_bins,
                     int32_t nchrom, int32_t cis_only, int32_t col_bits, unsigned long long* keys,
                     unsigned long long* n_valid, unsigned long long* oob, void* stream);

/* LSD radix sort of 64-bit keys on bits [begin_bit, end_bit), 8 bits per pass, onesweep style
 * (one histogram pass + one read/write of the keys per digit, decoupled look-back).
 * keys/tmp: n-element ping-pong buffers; *h_result_in_tmp = 1 when the sorted keys are in tmp.
 * work: hc_sort_work_bytes(n) bytes.  Stream-ordered, no host synchronisation. */
int64_t hc_sort_work_bytes(int64_t n);
int hc_sort_keys_u64(unsigned long long* keys, unsigned long long* tmp, int64_t n, int32_t begin_bit,
                     int32_t end_bit, void* work, int32_t* h_result_in_tmp, void* stream);

/* Reduce-by-key over the sorted keys: count distinct keys among the first *n_valid (device)
 * -> *h_nnz (synchronises the stream), then emit row_ptr[nrows+1], col[nnz], cnt[nnz] for the
 * row block [row0, row0+nrows) that all keys belong to (row_ptr is indexed by local row).
 * work: hc_csr_work_bytes(nkeys) (kept between the two calls); ukey/upos: nnz-element scratch. */
int64_t hc_csr_work_bytes(int64_t nkeys);
int hc_csr_count(const unsigned long long* sorted_keys, int64_t nkeys, const unsigned long long* n_valid,
                 void* work, int64_t* h_nnz, void* stream);
int hc_csr_emit(const unsigned long long* sorted_keys, int64_t nkeys, const unsigned long long* n_valid,
                const void* work, int64_t nnz, int32_t col_bits, int64_t row0, int64_t nrows,
                unsigned long long* ukey,
                int64_t* upos, int64_t* row_ptr, int32_t* col, int32_t* cnt, void* stream);

/* One key per pair (the default sort path).  A 64-bit ENTRY is
 *   (row << (col_bits + cnt_bits)) | (col << cnt_bits) | count,   2*col_bits + cnt_bits <= 63.
 * hc_pairs_to_entries writes one entry per pair: its upper-triangle cell (row <= col) with count 1, or the padding
 * key ~0 for a dropped pair (npairs entries; *n_valid, *oob as in hc_pairs_to_keys).  After hc_sort_keys_u64 on the
 * bits [cnt_bits, cnt_bits + 2*col_bits (+1 when nbins is a power of two)):
 *   hc_entries_count     distinct cells among the first *n_valid entries -> *h_nuniq (synchronises);
 *   hc_entries_reduce    out[nuniq] = one entry per cell; unit != 0: count = run length (all inputs carry 1),
 *                        unit == 0: the counts of a run are added (merging lists received from other ranks).
 *                        *h_overflow = 1 when a count needs more than cnt_bits bits (synchronises);
 *   hc_entries_transpose lo[n] = the off-diagonal cells with row and col swapped (padding key for diagonal cells),
 *                        *n_lo (device) = number of real ones.  `up` is ordered by (row, col), so lo is already
 *                        ordered by its minor key: ONE stable sort over the new row bits
 *                        [cnt_bits + col_bits, cnt_bits + 2*col_bits (+1)) orders it;
 *   hc_entries_to_csr    symmetric CSR of the rows [row0, row0+nrows): row r = lower entries | upper entries.
 *                        lo == NULL: `up` holds every entry of those rows (a row-block shard after the exchange).
 * Replaces the same reference lines as hc_pairs_to_keys (matrixBuilding.py:559-603). */
int hc_pairs_to_entries(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                        int64_t npairs, int32_t res, const int64_t* start, const int32_t* chrom_bins,
                        int32_t nchrom, int32_t cis_only, int32_t col_bits, int32_t cnt_bits,
                        unsigned long long* entries, unsigned long long* n_valid, unsigned long long* oob,
                        void* stream);
int hc_entries_count(const unsigned long long* sorted, int64_t n, const unsigned long long* n_valid,
                     int32_t cnt_bits, void* work /* hc_csr_work_bytes(n) */, int64_t* h_nuniq, void* stream);
int hc_entries_reduce(const unsigned long long* sorted, int64_t n, const unsigned long long* n_valid,
                      const void* work, int64_t nuniq, int32_t cnt_bits, int32_t unit, int64_t* upos /* nuniq */,
                      unsigned long long* out, int32_t* d_overflow, int32_t* h_overflow, void* stream);
/* The default reduction: after hc_entries_count (whose `work` keeps the scanned per-tile head counts), ONE pass writes
 * out[nuniq] and, when lo != NULL, the swapped list of hc_entries_transpose (lo[nuniq], *n_lo) as well. */
int hc_entries_emit(const unsigned long long* sorted, int64_t n, const unsigned long long* n_valid, const void* work,
                    int64_t nuniq, int32_t col_bits, int32_t cnt_bits, int32_t unit, unsigned long long* out,
                    unsigned long long* lo, unsigned long long* n_lo, int32_t* d_overflow, int32_t* h_overflow, void* stream);
int hc_entries_transpose(const unsigned long long* up, int64_t n, int32_t col_bits, int32_t cnt_bits,
                         unsigned long long* lo, unsigned long long* n_lo, void* stream);
/* Directed entries of the allelic haplotype matrices: two slots per pair (entries[2*npairs], 16-byte aligned), cis pairs
 * of an M_M or P_P bed routed through `start` (the M or P offsets of the concatenated haplotype bins).  A Both pair
 * (mark 0) gives (b1, b2) and, off the diagonal, (b2, b1) -- the cells of HC_BIN_SYM_BOTH; with `onesided`, an R1 pair
 * (mark 1) gives (b1, b2) and a pair with any other non-zero mark (b2, b1) -- the cells of HC_BIN_ONESIDED
 * (matrixBuilding.py:1153-1161, :1295-1301).  Unused slots hold the padding key.  *n_valid and *oob are ADDED to (not
 * reset), so the two beds can fill the two halves of one buffer.  Sorted on 2*col_bits bits and reduced with
 * hc_entries_count / hc_entries_emit, the entries give the rows of a general (asymmetric) CSR; the swapped list of
 * hc_entries_emit, re-sorted on its row bits, gives its transpose without the diagonal. */
int hc_pairs_to_directed_entries(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                                 const uint8_t* mark, int64_t npairs, int32_t res, const int64_t* start,
                                 const int32_t* chrom_bins, int32_t nchrom, int32_t onesided, int32_t col_bits,
                                 int32_t cnt_bits, unsigned long long* entries, unsigned long long* n_valid,
                                 unsigned long long* oob, void* stream);
int64_t hc_entries_csr_work_bytes(int64_t nrows);
int hc_entries_to_csr(const unsigned long long* up, int64_t n_up, const unsigned long long* lo,
                      const unsigned long long* n_lo, int32_t col_bits, int32_t cnt_bits, int64_t row0,
                      int64_t nrows, void* work, int64_t* row_ptr, int32_t* col, int32_t* cnt, void* stream);

/* Upper-triangular (bin1, bin2, count) records of the symmetric CSR in row-major order
 * (WholeMatrixToSparseDict's output layout before the per-chromosome split): count fills
 * out_ptr[nrows+1] (exclusive scan), then emit. */
int hc_csr_upper_count(const int64_t* row_ptr, const int32_t* col, int64_t row0, int64_t nrows,
                       int64_t* out_ptr, void* stream);
int hc_csr_upper_emit(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0,
                      int64_t nrows, const int64_t* out_ptr, int32_t* bin1, int32_t* bin2, int32_t* val, void* stream);

/* ICE on the symmetric CSR.  The local rows [row0, row0+nloc) may be a row block of a matrix
 * sharded over several GPUs; marg / nnz_marg / bias are FULL-length vectors.
 * hc_ice_csr_marginals writes the filter marginals of the local rows at their global positions
 * (zero the vectors first when they will be allreduced). */
int hc_ice_csr_marginals(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0,
                         int64_t nloc, int32_t ignore_diags, double* nnz_marg, double* marg,
                         void* stream);

/* Balance to convergence.  By default the CSR is first re-encoded (once per call, stream-ordered scratch of ~4 B per
 * stored entry) into column blocks of 8192 bins with 4-byte entries so that the bias of a block is staged in shared
 * memory (cp.async.bulk) instead of being gathered from L2, and the whole iteration -- stream kernel, marginal
 * reduction, the NCCL allreduce, cluster update kernel -- is replayed as a CUDA graph (HC_CSR_BLOCKED=0 or a count
 * beyond 19 bits: row-major gather kernel).  One problem per [bin_off[p], bin_off[p+1]) range: one range =
 * genome-wide; per-chromosome ranges on cis-only keys = `--cis-only`).  bias: in = initial
 * bias from hc_ice_filter_bins, out = final weights.  nccl_comm: NULL on one GPU, otherwise a
 * communicator from hc_nccl_comm_init -- the marginal vector is then allreduced in-stream once
 * per iteration and every rank applies the same O(n) update.  work: hc_ice_csr_work_bytes. */
int64_t hc_ice_csr_work_bytes(int64_t nbins, int32_t nprob);
int hc_ice_csr_balance(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0,
                       int64_t nloc, const int64_t* bin_off, int32_t nprob, const int64_t* h_bin_off,
                       const hc_ice_params* h_params, double* bias, void* work, hc_ice_result* results,
                       hc_ice_run_info* h_info, void* nccl_comm, void* stream);

/* NCCL plumbing (libnccl.so.2 resolved with dlopen at first use). h_id128: 128-byte host buffer. */
int hc_nccl_available(void);
int hc_nccl_unique_id(void* h_id128);
int hc_nccl_comm_init(const void* h_id128, int32_t nranks, int32_t rank, void** h_comm);
int hc_nccl_comm_destroy(void* comm);
int hc_nccl_allreduce_sum_f64(void* comm, double* buf, int64_t count, void* stream);

/* ------------------------------------------------------------------------------------------
 * (c) Two-step allelic correction (matrixBuilding.py:984-1023 TwoStepCorrection, with
 * Gap_defined :915-929, Trans2symmetry :945-979, Correct_VC :780-790).
 * ---------------------------------------------------------------------------------------- */

/* Row sums (int64) and non-zero counts (int32) of an int32 matrix view.  Replaces the row
 * loops at matrixBuilding.py:904-912 and :994-995. */
int hc_rowstats_i32(const int32_t* M, int64_t ld, int32_t nrows, int32_t ncols, int64_t* rowsum,
                    int32_t* rownnz, void* stream);

#define HC_GAP_PERCENTILE 0 /* Gap_defined: min(percentile(cov[cov!=0], 25), 0.2)  (:915-929) */
#define HC_GAP_FIXED 1      /* Gap_definedLowRes: 0.1                               (:742-753) */

/* O(n) part of the correction, on device: coverage -> gap rows of MM and PM, SNP-density
 * factor alpha = (rowsum MM + rowsum PM) / (rowsum TM + 1), normalised by its max over the
 * non-gap rows, zeros -> 1, floored at its 20th percentile (matrixBuilding.py:989-1005).
 * gap_union=1: non-gap = NonGap(MM) | NonGap(PM) (TwoStepCorrection); gap_union=0 with
 * nnz_b == NULL: gaps from matrix A only (GenomeWideMatrixCorrection :872-885, where A is the
 * traditional block).  Outputs: alpha[n]; gap flags (uint8[n]) and ascending index lists with
 * counts ngap[2].  work: 2*n doubles. */
int hc_twostep_alpha(const int64_t* rowsum_t, const int64_t* rowsum_m, const int64_t* rowsum_p,
                     const int32_t* nnz_a, const int32_t* nnz_b, int32_t n, int32_t ncols,
                     int32_t gap_mode, double* alpha, uint8_t* gapflag_a, uint8_t* gapflag_b,
                     int32_t* gapidx_a, int32_t* gapidx_b, int32_t* ngap, double* work,
                     void* stream);

/* Fused  X / alpha[:,None] -> Trans2symmetry -> Correct_VC(2/3) -> rescale to the raw mean
 * for ONE int32 matrix X (n x n, leading dimension ld).  gapflag == NULL or *h_ngap == 0
 * selects the reference's "no gap rows" rule (S_ij + S_ji, matrixBuilding.py:948-952 and
 * Trans2symmetryLowRes :770-776); otherwise both-gap -> max, else mean.  out is float64
 * n x n with leading dimension ld_out.  work: hc_twostep_work_bytes(n) bytes. */
int64_t hc_twostep_work_bytes(int32_t n);
int hc_twostep_correct(const int32_t* X, int64_t ld, int32_t n, const double* alpha,
                       const uint8_t* gapflag, int32_t has_gap, const int64_t* rowsum_x,
                       double* out, int64_t ld_out, void* work, void* stream);

/* IntraChromMatrixCorrection (matrixBuilding.py:1026-1041) for a whole batch in one call, no host
 * round trip: T = nchrom traditional matrices, H = 2*nchrom haplotype matrices (all maternal, then all
 * paternal) of the same sides, both as dense batches (device tables + host copies h_*).  Outputs:
 * out (fp64; matrix k of H at h_out_off[k], row-major n x n), alpha (per T bin), gapflag and gapidx (per
 * H bin; ascending gap rows of matrix k at gapidx[h_hbin[k] ...]), ngap[2*nchrom] ordered (M_c, P_c).
 * work: hc_twostep_batch_work_bytes(t_nbins, h_nbins, max_n). */
int64_t hc_twostep_batch_work_bytes(int64_t t_nbins, int64_t h_nbins, int32_t max_n);
int hc_twostep_batch(const int32_t* tmats, const int64_t* t_off, const int32_t* t_n, const int32_t* t_ld,
                     const int64_t* t_bin_off, const int32_t* hmats, const int64_t* h_off, const int32_t* h_n,
                     const int32_t* h_ld, const int64_t* h_bin_off, int32_t nchrom, const int32_t* h_sizes,
                     const int64_t* h_hoff, const int32_t* h_hld, const int64_t* h_tbin, const int64_t* h_hbin,
                     double* out, const int64_t* h_out_off, double* alpha, uint8_t* gapflag, int32_t* gapidx,
                     int32_t* ngap, void* work, void* stream);

/* hc_twostep_batch on CSR matrices, for local resolutions whose dense tiles would not fit: memory O(nnz + n).
 * T: symmetric CSR (row_ptr, cnt) of the nchrom traditional matrices over t_nbins concatenated bins (t_bin_off,
 * device, nchrom+1).  X: general CSR (row_ptr int64, col int32 = global bin, cnt int32; rows column-sorted) of the
 * 2*nchrom imputed haplotype matrices (all maternal, then all paternal; h_bin_off, device, 2*nchrom+1; h_nbins =
 * 2*t_nbins).  XT: the transpose of X in the same layout (its diagonal is not read).  Same arithmetic as the dense
 * batch: row sums and coverage (non-zeros of the asymmetric X), gaps / alpha by the same kernel (bit-exact gaps),
 * Trans2symmetry on the union pattern of X and XT, Correct_VC(2/3) with the row sum for the column sum, RF =
 * sum(X) / sum(Cor).  Outputs: alpha, gapflag, gapidx, ngap as hc_twostep_batch; rec_ptr[h_nbins+1] the offsets of
 * every row's records; records: 24-byte (int64 bin1, int64 bin2, float64 IF) upper-triangle records of every matrix,
 * chromosome-local bins, row-major, matrix k starting at rec_ptr[h_bin_off[k]] -- room for nnz(X) + nnz(XT) records;
 * *h_nrec the number written (synchronises; the only host round trip).
 * work: hc_twostep_csr_batch_work_bytes(t_nbins, h_nbins, nchrom). */
int64_t hc_twostep_csr_batch_work_bytes(int64_t t_nbins, int64_t h_nbins, int32_t nchrom);
int hc_twostep_csr_batch(const int64_t* t_row_ptr, const int32_t* t_cnt, const int64_t* x_row_ptr, const int32_t* x_col,
                         const int32_t* x_cnt, const int64_t* xt_row_ptr, const int32_t* xt_col, const int32_t* xt_cnt,
                         const int64_t* t_bin_off, const int64_t* h_bin_off, int32_t nchrom, int64_t t_nbins,
                         int64_t h_nbins, double* alpha, uint8_t* gapflag, int32_t* gapidx, int32_t* ngap,
                         int64_t* rec_ptr, void* records, int64_t* h_nrec, void* work, void* stream);

/* The reference's own building blocks, separately callable (SURVEY.md section 8b keeps Correct_VC(X, alpha)
 * among the signatures; hc_twostep_correct fuses all of them for the int32 tiles).  Float64 matrices,
 * row-major with leading dimension ld.
 *   hc_rownnz_f64          non-zero entries per row: Coverage_M = 1 - zeros/len (matrixBuilding.py:904-912);
 *                          integer matrices use hc_rowstats_i32.
 *   hc_gap_rows            coverage[n], gap flags and the ascending gap-row list from the per-row non-zero
 *                          counts: Gap_defined (:915-929, HC_GAP_PERCENTILE) / Gap_definedLowRes (:742-753,
 *                          HC_GAP_FIXED).  Non_Gap_Defined (:932-943) is the complement (gapflag == 0).
 *   hc_trans2symmetry_f64  Trans2symmetry (:945-979): gapflag == NULL -> S_ij + S_ji (also
 *                          Trans2symmetryLowRes :770-776); else both rows gaps -> max, otherwise mean; the
 *                          diagonal is copied.  out must not alias S.
 *   hc_correct_vc_f64      Correct_VC (:780-790): x / (colsum^alpha [None,:] * rowsum^alpha [:,None]), zero
 *                          sums -> 1.  work: hc_correct_vc_work_bytes(nrows, ncols). */
int hc_rownnz_f64(const double* M, int64_t ld, int32_t nrows, int32_t ncols, int32_t* rownnz, void* stream);
int hc_gap_rows(const int32_t* rownnz, int32_t n, int32_t ncols, int32_t gap_mode, double* coverage,
                uint8_t* gapflag, int32_t* gapidx, int32_t* ngap, void* stream);
int hc_trans2symmetry_f64(const double* S, int64_t ld, int32_t n, const uint8_t* gapflag, double* out,
                          int64_t ld_out, void* stream);
int64_t hc_correct_vc_work_bytes(int32_t nrows, int32_t ncols);
int hc_correct_vc_f64(const double* X, int64_t ld, int32_t nrows, int32_t ncols, double alpha, double* out,
                      int64_t ld_out, void* work, void* stream);

/* ------------------------------------------------------------------------------------------
 * First downstream consumers of the stage's outputs (SURVEY.md section 8f row 4; HiCHap/StructureFind.py).
 * Float64 matrices are row-major n x n with leading dimension ld.
 *   hc_balance_apply_i32         out = nan_to_num(count * w_i * w_j): what cooler.matrix(balance=True).fetch() +
 *                                np.nan_to_num hand to CallPeaks (StructureFind.py:2005-2007)
 *   hc_colnnz_f64                non-zero entries per COLUMN: Distance_Decay's own gap rule (:216-221)
 *   hc_distance_sums_f64         dsum[d] = sum of M[i][j], |i-j| = d, column j not flagged (both triangles): the
 *                                bincount of Distance_Decay (:225-253); the O(n) gap normalisation stays on the host
 *   hc_observed_expected_f64     M[i][j] / decline[|i-j|] where M != 0 (Get_PCA :321-326)
 *   hc_directionality_index_f64  Get_DI (:804-840): chitest = 0 t-test flavour, 1 chi-square flavour
 * ---------------------------------------------------------------------------------------- */
int hc_balance_apply_i32(const int32_t* M, int64_t ld, int32_t n, const double* weight, double* out, int64_t ld_out,
                         void* stream);
int hc_colnnz_f64(const double* M, int64_t ld, int32_t n, int32_t* colnnz, void* stream);
int hc_distance_sums_f64(const double* M, int64_t ld, int32_t n, const uint8_t* gapflag, double* dsum, void* stream);
int hc_observed_expected_f64(const double* M, int64_t ld, int32_t n, const double* decline, double* out, int64_t ld_out,
                             void* stream);
int hc_directionality_index_f64(const double* M, int64_t ld, int32_t n, const uint8_t* gapflag, const int32_t* window_bin,
                                int32_t chitest, double* di, void* stream);

/* ------------------------------------------------------------------------------------------
 * Valid-pair text ingest (host, multithreaded; SURVEY.md section 8f row 1): parses the 23-column
 * *_Valid.bed (layout 0: chromosomes in columns 1 and 8, fragment mid-points in columns 6 and 13;
 * matrixBuilding.py:573-586) or the 4/5-column allelic beds (layout 1: c1 p1 c2 p2 [mark];
 * :822-834, :1131-1141) of several files in order (the reference pipes `cat`, :307-313), with the
 * reference's `lstrip('chr')` character-set strip and chromosome filter (:360, :577).
 * chrom_names[i]: stripped name of chromosome index i; filter_names: the `chroms` list ("#" =
 * numeric labels; nfilter = 0 keeps all).  Dropped lines are omitted.  hc_ingest_parse returns the
 * number of kept pairs; hc_ingest_fetch (same host thread) copies the columns out and frees them.
 * Errors: HC_ERR_ARG with hc_last_error() "KeyError: <chrom>" (passes the filter but is not in the
 * genome table), "ValueError: ..." or "IOError: ...". */
int hc_ingest_parse(const char* const* h_paths, int32_t npaths, int32_t layout,
                    const char* const* h_chrom_names, int32_t nchrom,
                    const char* const* h_filter_names, int32_t nfilter, int32_t nthreads,
                    int64_t* h_npairs);
int hc_ingest_fetch(int32_t* h_c1, int32_t* h_p1, int32_t* h_c2, int32_t* h_p2, uint8_t* h_mark);

#ifdef __cplusplus
}
#endif
#endif /* HICHAP_B200_H */
