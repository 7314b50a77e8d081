// SURVEY.md section 8(f) row 4: the first downstream consumers of the matrix stage's outputs -- the weight vector and
// the (corrected) matrices -- in HiCHap/StructureFind.py:
//   balanced matrix       cooler.matrix(balance=True).fetch(chrom) + np.nan_to_num   (StructureFind.py:2005-2007)
//   Distance_Decay        mean contact per genomic distance with gap columns removed (:201-272)
//   observed / expected   the O/E matrix Get_PCA builds from that curve               (:321-329)
//   Get_DI                directionality index, t-test or chi-square flavour          (:804-840)
// Streaming kernels over dense tiles, and the same four over a canonical CSR (CSC for Get_DI, which reads columns) for
// the resolutions whose dense matrix does not fit; every floating-point reduction has a fixed order (deterministic).
#include <math.h>
#include "hc_common.cuh"

namespace {

// out[i][j] = nan_to_num(M[i][j] * w[i] * w[j]); NaN weights (filtered bins) give NaN products -> 0
__global__ void __launch_bounds__(256)
balance_apply_kernel(const int32_t* __restrict__ M, int64_t ld, int n, const double* __restrict__ w,
                     double* __restrict__ out, int64_t ld_out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= n) return;
    const double wi = w[i], v = (double)M[(int64_t)i * ld + j] * wi * w[j];      // (count * w_i) * w_j, cooler's order
    double r = v;
    if (isnan(v)) r = 0.0;
    else if (isinf(v)) r = v > 0 ? 1.7976931348623157e308 : -1.7976931348623157e308;   // np.nan_to_num
    out[(int64_t)i * ld_out + j] = r;
}

// non-zero count per COLUMN (Distance_Decay's gap rule looks at columns, StructureFind.py:218)
__global__ void __launch_bounds__(256)
colnnz_f64_kernel(const double* __restrict__ M, int64_t ld, int n, int32_t* __restrict__ colnnz) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    int c = 0;
    for (int i = 0; i < n; ++i) c += (M[(int64_t)i * ld + j] != 0.0);
    colnnz[j] = c;
}

// one warp per distance d: sum of M[i][j] over |i - j| == d with column j not a gap (both triangles), fixed order
__global__ void __launch_bounds__(256)
distance_sum_kernel(const double* __restrict__ M, int64_t ld, int n, const uint8_t* __restrict__ gap,
                    double* __restrict__ dsum) {
    const int d = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (d >= n) return;
    double s = 0.0;
    for (int i = lane; i + d < n; i += 32) {
        const int j = i + d;
        if (!gap[j]) s += M[(int64_t)i * ld + j];            // entry (i, j): column j
        if (d > 0 && !gap[i]) s += M[(int64_t)j * ld + i];   // entry (j, i): column i
    }
    s = warp_sum(s);
    if (lane == 0) dsum[d] = s;
}

// OE[i][j] = M[i][j] / decline[|i - j|] where M != 0 (decline has no zeros: the caller replaced them, :318-319)
__global__ void __launch_bounds__(256)
oe_kernel(const double* __restrict__ M, int64_t ld, int n, const double* __restrict__ decline, double* __restrict__ out,
          int64_t ld_out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j >= n) return;
    const double v = M[(int64_t)i * ld + j];
    out[(int64_t)i * ld_out + j] = v != 0.0 ? v / decline[i > j ? i - j : j - i] : 0.0;
}

// one thread per bin (the windows are a few tens of bins)
__global__ void __launch_bounds__(128)
di_kernel(const double* __restrict__ M, int64_t ld, int n, const uint8_t* __restrict__ gap,
          const int32_t* __restrict__ window_bin, int chitest, double* __restrict__ di) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int w = window_bin[j];
    double bias = 0.0;
    if (!gap[j] && w >= 1 && j >= w && j <= n - w - 1) {
        double up_sum = 0.0, down_sum = 0.0;
        for (int t = 1; t <= w; ++t) { up_sum += M[(int64_t)(j - t) * ld + j]; down_sum += M[(int64_t)(j + t) * ld + j]; }
        if (!chitest) {
            const double um = up_sum / w, dm = down_sum / w;
            const double den = (double)w * (double)(w - 1);
            double uq = 0.0, dq = 0.0;
            for (int t = 1; t <= w; ++t) {
                const double a = M[(int64_t)(j - t) * ld + j] - um, b = M[(int64_t)(j + t) * ld + j] - dm;
                uq += a * a / den; dq += b * b / den;
            }
            const double s = sqrt(uq + dq);
            if (s != 0.0) bias = (dm - um) / s;               // NaN when w == 1 (0/0), as NumPy gives the reference
        } else {
            const double e = (up_sum + down_sum) / 2.0;
            if (up_sum != down_sum && e != 0.0) {
                const double dd = down_sum - up_sum;
                bias = dd / fabs(dd) * ((up_sum - e) * (up_sum - e) / e + (down_sum - e) * (down_sum - e) / e);
            }
        }
    }
    di[j] = bias;
}

// ---- the same consumers on a canonical CSR (rows column-sorted, no duplicate cells, no explicit zeros), for the
// resolutions whose n x n matrix does not fit: O(nnz + n) bytes instead of O(n^2).  Row-parallel kernels use one warp
// per row with lane-strided (coalesced) entries.

// balance_apply_kernel per stored entry: the same expression, so the values are bit-identical
__global__ void __launch_bounds__(256)
balance_apply_csr_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                         const int32_t* __restrict__ cnt, int n, const double* __restrict__ w, double* __restrict__ out) {
    const int i = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    const double wi = w[i];
    for (int64_t e = row_ptr[i] + lane; e < row_ptr[i + 1]; e += 32) {
        const double v = (double)cnt[e] * wi * w[col[e]];
        double r = v;
        if (isnan(v)) r = 0.0;
        else if (isinf(v)) r = v > 0 ? 1.7976931348623157e308 : -1.7976931348623157e308;
        out[e] = r;
    }
}

// stored entries per column; integer counts, so the atomics leave the result order-independent
__global__ void __launch_bounds__(256)
colnnz_csr_kernel(const int32_t* __restrict__ col, int64_t nnz, int32_t* __restrict__ colnnz) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < nnz; e += (int64_t)gridDim.x * blockDim.x)
        atomicAdd(colnnz + col[e], 1);
}

// key of entry e = (|i - j| << idx_bits) | e, or distance n (past every real one) when column j is a gap
__global__ void __launch_bounds__(256)
distance_keys_csr_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, int n,
                         const uint8_t* __restrict__ gap, int idx_bits, unsigned long long* __restrict__ keys) {
    const int i = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    for (int64_t e = row_ptr[i] + lane; e < row_ptr[i + 1]; e += 32) {
        const int j = col[e];
        const unsigned long long d = gap[j] ? (unsigned)n : (unsigned)(i > j ? i - j : j - i);
        keys[e] = (d << idx_bits) | (unsigned long long)e;
    }
}

__device__ __forceinline__ int64_t lower_bound_key(const unsigned long long* __restrict__ k, int64_t nnz,
                                                   unsigned long long x) {
    int64_t lo = 0, hi = nnz;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (k[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// one warp per distance d over the keys sorted by distance (entry order kept within a distance: the sort is stable):
// lane-strided sum of the entries' values, then warp_sum -- a fixed order, so repeated calls are bit-identical
__global__ void __launch_bounds__(256)
distance_segsum_kernel(const unsigned long long* __restrict__ keys, int64_t nnz, int idx_bits,
                       const double* __restrict__ val, int n, double* __restrict__ dsum) {
    const int d = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (d >= n) return;
    const int64_t b = lower_bound_key(keys, nnz, (unsigned long long)d << idx_bits);
    const int64_t e = lower_bound_key(keys, nnz, (unsigned long long)(d + 1) << idx_bits);
    const unsigned long long mask = (1ull << idx_bits) - 1;
    double s = 0.0;
    for (int64_t k = b + lane; k < e; k += 32) s += val[keys[k] & mask];
    s = warp_sum(s);
    if (lane == 0) dsum[d] = s;
}

// oe_kernel per stored entry (stored entries are non-zero): bit-identical values
__global__ void __launch_bounds__(256)
oe_csr_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const double* __restrict__ val,
              int n, const double* __restrict__ decline, double* __restrict__ out) {
    const int i = (int)((blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (i >= n) return;
    for (int64_t e = row_ptr[i] + lane; e < row_ptr[i + 1]; e += 32) {
        const int j = col[e];
        out[e] = val[e] / decline[i > j ? i - j : j - i];
    }
}

// di_kernel on the column-compressed matrix: column j's rows are sorted, so the cells j - t (t = 1..w) are met walking
// down from the last row < j and the cells j + t walking up from the first row > j; a missing cell reads 0.0.  The
// loops and the arithmetic are di_kernel's, term for term, so the result is bit-identical to it.
__global__ void __launch_bounds__(128)
di_csc_kernel(const int64_t* __restrict__ col_ptr, const int32_t* __restrict__ row, const double* __restrict__ val,
              int n, const uint8_t* __restrict__ gap, const int32_t* __restrict__ window_bin, int chitest,
              double* __restrict__ di) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int w = window_bin[j];
    double bias = 0.0;
    if (!gap[j] && w >= 1 && j >= w && j <= n - w - 1) {
        const int64_t cb = col_ptr[j], ce = col_ptr[j + 1];
        int64_t lo = cb, hi = ce;                                  // first stored row >= j
        while (lo < hi) { const int64_t mid = (lo + hi) >> 1; if (row[mid] < j) lo = mid + 1; else hi = mid; }
        const int64_t up0 = lo - 1, dn0 = (lo < ce && row[lo] == j) ? lo + 1 : lo;
        double up_sum = 0.0, down_sum = 0.0;
        int64_t pu = up0, pd = dn0;
        for (int t = 1; t <= w; ++t) {
            const double a = (pu >= cb && row[pu] == j - t) ? val[pu--] : 0.0;
            const double b = (pd < ce && row[pd] == j + t) ? val[pd++] : 0.0;
            up_sum += a; down_sum += b;
        }
        if (!chitest) {
            const double um = up_sum / w, dm = down_sum / w;
            const double den = (double)w * (double)(w - 1);
            double uq = 0.0, dq = 0.0;
            pu = up0; pd = dn0;
            for (int t = 1; t <= w; ++t) {
                const double mu = (pu >= cb && row[pu] == j - t) ? val[pu--] : 0.0;
                const double md = (pd < ce && row[pd] == j + t) ? val[pd++] : 0.0;
                const double a = mu - um, b = md - dm;
                uq += a * a / den; dq += b * b / den;
            }
            const double s = sqrt(uq + dq);
            if (s != 0.0) bias = (dm - um) / s;               // NaN when w == 1 (0/0), as in di_kernel
        } else {
            const double e = (up_sum + down_sum) / 2.0;
            if (up_sum != down_sum && e != 0.0) {
                const double dd = down_sum - up_sum;
                bias = dd / fabs(dd) * ((up_sum - e) * (up_sum - e) / e + (down_sum - e) * (down_sum - e) / e);
            }
        }
    }
    di[j] = bias;
}

inline unsigned warp_per_item_blocks(int64_t items) { return (unsigned)((items * 32 + 255) / 256); }

inline int bit_width(int64_t x) { int b = 0; while (x >> b) ++b; return b; }   // bits of x (0 for 0)

inline int64_t align256(int64_t b) { return (b + 255) / 256 * 256; }

}  // namespace

extern "C" int hc_balance_apply_i32(const int32_t* M, int64_t ld, int32_t n, const double* weight, double* out,
                                    int64_t ld_out, void* stream) {
    HC_REQUIRE(n > 0 && ld >= n && ld_out >= n && M && weight && out, "arguments");
    balance_apply_kernel<<<dim3((n + 255) / 256, n), 256, 0, (cudaStream_t)stream>>>(M, ld, n, weight, out, ld_out);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_colnnz_f64(const double* M, int64_t ld, int32_t n, int32_t* colnnz, void* stream) {
    HC_REQUIRE(n > 0 && ld >= n && M && colnnz, "arguments");
    colnnz_f64_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(M, ld, n, colnnz);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_distance_sums_f64(const double* M, int64_t ld, int32_t n, const uint8_t* gapflag, double* dsum,
                                    void* stream) {
    HC_REQUIRE(n > 0 && ld >= n && M && gapflag && dsum, "arguments");
    distance_sum_kernel<<<(unsigned)(((int64_t)n * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(M, ld, n, gapflag, dsum);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_observed_expected_f64(const double* M, int64_t ld, int32_t n, const double* decline, double* out,
                                        int64_t ld_out, void* stream) {
    HC_REQUIRE(n > 0 && ld >= n && ld_out >= n && M && decline && out, "arguments");
    oe_kernel<<<dim3((n + 255) / 256, n), 256, 0, (cudaStream_t)stream>>>(M, ld, n, decline, out, ld_out);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_directionality_index_f64(const double* M, int64_t ld, int32_t n, const uint8_t* gapflag,
                                           const int32_t* window_bin, int32_t chitest, double* di, void* stream) {
    HC_REQUIRE(n > 0 && ld >= n && M && gapflag && window_bin && di, "arguments");
    di_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(M, ld, n, gapflag, window_bin, chitest, di);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_balance_apply_csr_i32(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int32_t n,
                                        const double* weight, double* out, void* stream) {
    HC_REQUIRE(n > 0 && row_ptr && weight, "arguments");   // col / cnt / out may be NULL when nnz == 0
    balance_apply_csr_kernel<<<warp_per_item_blocks(n), 256, 0, (cudaStream_t)stream>>>(row_ptr, col, cnt, n, weight, out);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_colnnz_csr(const int32_t* col, int64_t nnz, int32_t n, int32_t* colnnz, void* stream) {
    HC_REQUIRE(n > 0 && nnz >= 0 && (col || nnz == 0) && colnnz, "arguments");
    cudaStream_t s = (cudaStream_t)stream;
    HC_CUDA(cudaMemsetAsync(colnnz, 0, sizeof(int32_t) * n, s));
    if (nnz == 0) return HC_OK;
    const int64_t blocks = (nnz + 255) / 256, cap = (int64_t)hc_num_sms() * 16;
    colnnz_csr_kernel<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, s>>>(col, nnz, colnnz);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

// work: the keys and the sort's ping-pong buffer (8 bytes per entry each), then the sort's own scratch
extern "C" int64_t hc_distance_sums_csr_work_bytes(int64_t nnz) {
    return 2 * align256(8 * (nnz > 0 ? nnz : 1)) + hc_sort_work_bytes(nnz);
}

extern "C" int hc_distance_sums_csr_f64(const int64_t* row_ptr, const int32_t* col, const double* val, int64_t nnz,
                                        int32_t n, const uint8_t* gapflag, double* dsum, void* work, void* stream) {
    HC_REQUIRE(n > 0 && nnz >= 0 && row_ptr && (nnz == 0 || (col && val)) && gapflag && dsum && work, "arguments");
    const int idx_bits = bit_width(nnz > 0 ? nnz - 1 : 0), d_bits = bit_width(n);   // distance n marks a gap column
    HC_REQUIRE(idx_bits + d_bits <= 64, "nnz * 2n needs more than 64 key bits");
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long* keys = reinterpret_cast<unsigned long long*>(work);
    unsigned long long* tmp = reinterpret_cast<unsigned long long*>((char*)work + align256(8 * (nnz > 0 ? nnz : 1)));
    void* sort_work = (char*)tmp + align256(8 * (nnz > 0 ? nnz : 1));
    distance_keys_csr_kernel<<<warp_per_item_blocks(n), 256, 0, s>>>(row_ptr, col, n, gapflag, idx_bits, keys);
    HC_LAUNCH_CHECK();
    int32_t in_tmp = 0;
    const int rc = hc_sort_keys_u64(keys, tmp, nnz, idx_bits, idx_bits + d_bits, sort_work, &in_tmp, stream);
    if (rc != HC_OK) return rc;
    distance_segsum_kernel<<<warp_per_item_blocks(n), 256, 0, s>>>(in_tmp ? tmp : keys, nnz, idx_bits, val, n, dsum);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_observed_expected_csr_f64(const int64_t* row_ptr, const int32_t* col, const double* val, int32_t n,
                                            const double* decline, double* out, void* stream) {
    HC_REQUIRE(n > 0 && row_ptr && decline, "arguments");   // col / val / out may be NULL when nnz == 0
    oe_csr_kernel<<<warp_per_item_blocks(n), 256, 0, (cudaStream_t)stream>>>(row_ptr, col, val, n, decline, out);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_directionality_index_csc_f64(const int64_t* col_ptr, const int32_t* row, const double* val, int32_t n,
                                               const uint8_t* gapflag, const int32_t* window_bin, int32_t chitest,
                                               double* di, void* stream) {
    HC_REQUIRE(n > 0 && col_ptr && gapflag && window_bin && di, "arguments");   // row / val may be NULL when nnz == 0
    di_csc_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(col_ptr, row, val, n, gapflag, window_bin, chitest, di);
    HC_LAUNCH_CHECK();
    return HC_OK;
}
