// (b) ICE balancing on the symmetric CSR (genome-wide matrices too large for dense tiles; also
// per-chromosome problems when the keys were built cis-only).  Same algorithm as hc_ice.cu
// (cooler balance restated in oracle/cooler_ice.py); call sites matrixBuilding.py:708, :1537, :1761.
//
// Per iteration:  stream kernel (one warp per row: gather bias[col], fp64 FMA with the int
// count, warp-shuffle reduce, one store per row)  ->  [one NCCL allreduce of the marginal
// vector when the matrix is row-block sharded across GPUs]  ->  three small grid kernels that
// reduce mean / variance over the non-zero marginals, update the bias and test convergence,
// all on the device.  The host only polls a done counter.
//
// Roofline: HBM-bound; this layout streams 8 B per stored entry, 2 entries per upper-triangle
// pixel => 16*Z + 24*n bytes per iteration against SURVEY's algorithmic 8*Z + 24*n.
#include <math.h>
#include <stdlib.h>
#include <vector>
#include "hc_common.cuh"

int hc_nccl_allreduce_f64(void* comm, const double* send, double* recv, size_t count, cudaStream_t s);  // hc_nccl.cu
// hc_ice_csrb.cu: the column-blocked encoding (default); returns +1 when a count does not fit its 19 bits
int hc_ice_csr_balance_blocked(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0, int64_t nloc,
                               const int64_t* bin_off, int32_t nprob, const int64_t* h_bin_off, const hc_ice_params* P,
                               double* bias, hc_ice_result* results, hc_ice_run_info* h_info, void* nccl_comm,
                               cudaStream_t caller);

namespace {

constexpr int STAT_SLICES = 32;
constexpr int STAT_THREADS = 256;

struct CsrView {
    const int64_t* row_ptr;  // local: nloc + 1
    const int32_t* col;
    const int32_t* cnt;
    long long row0;          // global index of local row 0
    long long nloc;
};

__device__ __forceinline__ double csr_band_weight(long long c, long long r, int kd) {
    const long long d = c - r;
    if (d == 0) return kd == 0 ? 2.0 : 0.0;
    return (d < kd && d > -kd) ? 0.0 : 1.0;
}

__device__ __forceinline__ int find_problem(const int64_t* __restrict__ bin_off, int nprob, long long r) {
    int lo = 0, hi = nprob - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (bin_off[mid] <= r) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// FILTER: nnz / sum marginals (bias == 1).  Otherwise marg[r] = b[r] * sum_c w(r,c) cnt b[c].
template <bool FILTER>
__global__ void __launch_bounds__(256)
ice_csr_stream_kernel(CsrView A, const double* __restrict__ bias, int kd, const int64_t* __restrict__ bin_off,
                      int nprob, const int32_t* __restrict__ done_at, int k, double* __restrict__ marg,
                      double* __restrict__ nnz_marg) {
    const int lane = threadIdx.x & 31;
    const long long warp0 = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const long long nwarps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long rl = warp0; rl < A.nloc; rl += nwarps) {
        const long long r = A.row0 + rl;
        if (!FILTER) {
            const int p = nprob > 1 ? find_problem(bin_off, nprob, r) : 0;
            const int d = done_at[p];
            if (d != 0 && d < k) continue;   // this chromosome converged in an earlier iteration
        }
        const long long e0 = A.row_ptr[rl], e1 = A.row_ptr[rl + 1];
        double acc0 = 0.0, acc1 = 0.0;
        long long s = 0;
        int nz = 0;
        auto one = [&](int c, int v, double& acc) {
            const double w = csr_band_weight(c, r, kd);
            if (FILTER) { s += (long long)(w * v); nz += (v != 0) ? (int)w : 0; }
            else acc = fma(w * (double)v, __ldg(bias + c), acc);
        };
        // head: up to 3 entries until the entry index is a multiple of 4 (16-byte aligned vectors)
        const long long head = min((long long)((4 - (e0 & 3)) & 3), e1 - e0);
        if (lane < head) one(__ldg(A.col + e0 + lane), __ldg(A.cnt + e0 + lane), acc0);
        const long long eb = e0 + head;
        const long long nvec = (e1 - eb) >> 2;
        // software pipeline: the (col, cnt) vectors of the next step are requested before the bias
        // gathers of the current step are issued, so the two dependent latencies overlap
        long long v = lane;
        int4 c0 = make_int4(0, 0, 0, 0), k0 = c0, c1 = c0, k1 = c0;
        bool h0 = v < nvec, h1 = v + 32 < nvec;
        if (h0) { c0 = ld_stream_v4(A.col + eb + 4 * v); k0 = ld_stream_v4(A.cnt + eb + 4 * v); }
        if (h1) { c1 = ld_stream_v4(A.col + eb + 4 * (v + 32)); k1 = ld_stream_v4(A.cnt + eb + 4 * (v + 32)); }
        while (h0) {
            const long long vn = v + 64;
            const bool n0 = vn < nvec, n1 = vn + 32 < nvec;
            int4 d0 = make_int4(0, 0, 0, 0), q0 = d0, d1 = d0, q1 = d0;
            if (n0) { d0 = ld_stream_v4(A.col + eb + 4 * vn); q0 = ld_stream_v4(A.cnt + eb + 4 * vn); }
            if (n1) { d1 = ld_stream_v4(A.col + eb + 4 * (vn + 32)); q1 = ld_stream_v4(A.cnt + eb + 4 * (vn + 32)); }
            one(c0.x, k0.x, acc0); one(c0.y, k0.y, acc1); one(c0.z, k0.z, acc0); one(c0.w, k0.w, acc1);
            if (h1) { one(c1.x, k1.x, acc0); one(c1.y, k1.y, acc1); one(c1.z, k1.z, acc0); one(c1.w, k1.w, acc1); }
            c0 = d0; k0 = q0; c1 = d1; k1 = q1; h0 = n0; h1 = n1; v = vn;
        }
        const long long et = eb + (nvec << 2);   // tail: fewer than 4 entries
        if (et + lane < e1) one(__ldg(A.col + et + lane), __ldg(A.cnt + et + lane), acc1);
        if (FILTER) {
            s = warp_sum_ll(s);
            nz = warp_sum_i(nz);
            if (lane == 0) { marg[r] = (double)s; nnz_marg[r] = (double)nz; }
        } else {
            const double acc = warp_sum(acc0 + acc1);
            if (lane == 0) marg[r] = bias[r] * acc;
        }
    }
}

// ---- per-iteration statistics and update (grid = (STAT_SLICES, nprob)) ---------------------
struct StatArgs {
    const int64_t* bin_off; int nprob;
    const double* marg; double* bias;
    double* part_sum; long long* part_cnt; double* part_var;  // [nprob][STAT_SLICES]
    int32_t* done_at; int32_t* n_done; hc_ice_result* results;
    double tol; int max_iters; int k;
};

__device__ __forceinline__ bool stat_active(const StatArgs& a, int p) {
    const int d = a.done_at[p];
    return d == 0 || d >= a.k;
}

__device__ __forceinline__ void slice_range(const StatArgs& a, int p, long long* lo, long long* hi) {
    const long long b0 = a.bin_off[p], n = a.bin_off[p + 1] - b0;
    *lo = b0 + n * blockIdx.x / gridDim.x;
    *hi = b0 + n * (blockIdx.x + 1) / gridDim.x;
}

__global__ void __launch_bounds__(STAT_THREADS) ice_stat_sum_kernel(StatArgs a) {
    __shared__ double red[32];
    __shared__ long long redll[32];
    const int p = blockIdx.y;
    if (!stat_active(a, p)) return;
    long long lo, hi;
    slice_range(a, p, &lo, &hi);
    double s = 0.0;
    long long c = 0;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const double m = a.marg[i];
        if (m != 0.0) { s += m; ++c; }
    }
    s = block_sum(s, red);
    c = block_sum_ll(c, redll);
    if (threadIdx.x == 0) { a.part_sum[p * gridDim.x + blockIdx.x] = s; a.part_cnt[p * gridDim.x + blockIdx.x] = c; }
}

__device__ __forceinline__ void problem_mean(const StatArgs& a, int p, double* mean, long long* cnt) {
    double s = 0.0;
    long long c = 0;
    for (int i = 0; i < (int)gridDim.x; ++i) { s += a.part_sum[p * gridDim.x + i]; c += a.part_cnt[p * gridDim.x + i]; }
    *cnt = c;
    *mean = c ? s / (double)c : 0.0;
}

__global__ void __launch_bounds__(STAT_THREADS) ice_stat_var_kernel(StatArgs a) {
    __shared__ double red[32];
    const int p = blockIdx.y;
    if (!stat_active(a, p)) return;
    double mean;
    long long cnt;
    problem_mean(a, p, &mean, &cnt);
    long long lo, hi;
    slice_range(a, p, &lo, &hi);
    double v = 0.0;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const double m = a.marg[i];
        if (m != 0.0) { const double d = m - mean; v += d * d; }
    }
    v = block_sum(v, red);
    if (threadIdx.x == 0) a.part_var[p * gridDim.x + blockIdx.x] = v;
}

__global__ void __launch_bounds__(STAT_THREADS) ice_stat_update_kernel(StatArgs a) {
    const int p = blockIdx.y;
    if (!stat_active(a, p)) return;
    double mean;
    long long cnt;
    problem_mean(a, p, &mean, &cnt);
    long long lo, hi;
    slice_range(a, p, &lo, &hi);
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (cnt == 0) {   // cooler: bias = NaN, scale = NaN, var = 0, stop
        for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) a.bias[i] = nan;
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            hc_ice_result r; r.scale = nan; r.var = 0.0; r.iters = a.k; r.converged = 1;
            a.results[p] = r; a.done_at[p] = a.k; atomicAdd(a.n_done, 1);
        }
        return;
    }
    double var = 0.0;
    for (int i = 0; i < (int)gridDim.x; ++i) var += a.part_var[p * gridDim.x + i];
    var /= (double)cnt;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        double m = a.marg[i] / mean;
        if (m == 0.0) m = 1.0;
        a.bias[i] = a.bias[i] / m;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        hc_ice_result r; r.scale = mean; r.var = var; r.iters = a.k; r.converged = var < a.tol;
        a.results[p] = r;
        if (var < a.tol || a.k >= a.max_iters) { a.done_at[p] = a.k; atomicAdd(a.n_done, 1); }
    }
}

__global__ void __launch_bounds__(256)
ice_csr_finalize_kernel(const int64_t* __restrict__ bin_off, int nprob, const hc_ice_result* __restrict__ results,
                        int rescale, double* bias) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= bin_off[nprob]) return;
    const int p = nprob > 1 ? find_problem(bin_off, nprob, g) : 0;
    const hc_ice_result r = results[p];
    double b = bias[g];
    if (!isnan(r.scale)) {
        if (b == 0.0) b = __longlong_as_double(0x7ff8000000000000ll);
        if (rescale) b = b / sqrt(r.scale);
    } else b = __longlong_as_double(0x7ff8000000000000ll);
    bias[g] = b;
}

int stream_grid() { return hc_num_sms() * 8; }

}  // namespace

// Filter marginals of the local rows [row0, row0+nloc): writes marg / nnz_marg at the GLOBAL
// row positions of the full-length vectors (zero the vectors first when they will be
// allreduced across row-block shards).
extern "C" int hc_ice_csr_marginals(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0,
                                    int64_t nloc, int32_t ignore_diags, double* nnz_marg, double* marg,
                                    void* stream) {
    HC_REQUIRE(nloc >= 0 && row0 >= 0 && ignore_diags >= 0, "sizes");
    if (nloc == 0) return HC_OK;
    CsrView A{row_ptr, col, cnt, row0, nloc};
    ice_csr_stream_kernel<true><<<stream_grid(), 256, 0, (cudaStream_t)stream>>>(A, nullptr, ignore_diags, nullptr, 1,
                                                                              nullptr, 0, marg, nnz_marg);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int64_t hc_ice_csr_work_bytes(int64_t nbins, int32_t nprob) {
    return (int64_t)sizeof(double) * (2 * nbins + 3ll * nprob * STAT_SLICES) + sizeof(int32_t) * (nprob + 4ll) + 64;
}

// Balance to convergence.  bias: full-length vector (in: initial bias from the filters; out:
// final weights), identical on every rank.  h_bin_off: host copy of bin_off (nprob+1).
// nccl_comm: NULL for a single GPU; otherwise the marginal vector is allreduced in-stream each
// iteration (every rank then performs the same O(n) update redundantly -- no broadcast).
extern "C" int hc_ice_csr_balance(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0,
                                  int64_t nloc, const int64_t* bin_off, int32_t nprob, const int64_t* h_bin_off,
                                  const hc_ice_params* P, double* bias, void* work, hc_ice_result* results,
                                  hc_ice_run_info* h_info, void* nccl_comm, void* stream) {
    HC_REQUIRE(nprob > 0 && h_bin_off != nullptr && P != nullptr && nloc >= 0, "arguments");
    HC_REQUIRE(P->max_iters >= 1 && P->ignore_diags >= 0, "max_iters>=1, ignore_diags>=0");
    cudaStream_t s = (cudaStream_t)stream;
    const long long nbins = h_bin_off[nprob];
    if (h_info) { h_info->launches = 0; h_info->loop_ms = 0.f; h_info->packed = 0; h_info->pack_ms = 0.f; h_info->overflow_cells = 0; h_info->stream_full_ms = 0.f; h_info->stream_full_launches = 0; }
    if (nbins == 0) return HC_OK;
    {
        // default: column-blocked 4-byte entries with the bias block staged in shared memory (hc_ice_csrb.cu);
        // HC_CSR_BLOCKED=0 (A/B) or a count beyond 19 bits -> the row-major gather kernel below
        bool blocked = true;
        if (const char* e = getenv("HC_CSR_BLOCKED")) blocked = atoi(e) != 0;
        if (blocked) {
            const int r = hc_ice_csr_balance_blocked(row_ptr, col, cnt, row0, nloc, bin_off, nprob, h_bin_off, P, bias, results,
                                                     h_info, nccl_comm, s);
            if (r <= 0) return r;
        }
    }

    double* marg = reinterpret_cast<double*>(work);
    // sharded: the stream kernel writes the local rows of marg_local (zero elsewhere, zeroed once)
    // and the allreduce sums the ranks' vectors into marg; single GPU: both are the same buffer
    double* marg_local = nccl_comm ? marg + nbins : marg;
    double* part_sum = marg + 2 * nbins;
    double* part_var = part_sum + (size_t)nprob * STAT_SLICES;
    long long* part_cnt = reinterpret_cast<long long*>(part_var + (size_t)nprob * STAT_SLICES);
    int32_t* done_at = reinterpret_cast<int32_t*>(part_cnt + (size_t)nprob * STAT_SLICES);
    int32_t* n_done = done_at + nprob;
    HC_CUDA(cudaMemsetAsync(marg, 0, sizeof(double) * 2 * nbins, s));
    HC_CUDA(cudaMemsetAsync(done_at, 0, sizeof(int32_t) * (nprob + 1), s));

    // empty problems (no bins) are done from the start
    int nonempty = 0;
    {
        std::vector<hc_ice_result> h_res(nprob);
        bool any_empty = false;
        for (int p = 0; p < nprob; ++p) {
            h_res[p].scale = NAN; h_res[p].var = 0.0; h_res[p].iters = 0; h_res[p].converged = 1;
            if (h_bin_off[p + 1] > h_bin_off[p]) ++nonempty; else any_empty = true;
        }
        if (any_empty) {
            HC_CUDA(cudaMemcpyAsync(results, h_res.data(), sizeof(hc_ice_result) * nprob, cudaMemcpyHostToDevice, s));
            HC_CUDA(cudaStreamSynchronize(s));
        }
    }
    // problems without bins must not count as active in the kernels: mark them done at iteration 0 -> use -1
    // (done_at != 0 && done_at < k holds for every k >= 1)
    {
        std::vector<int32_t> h_done(nprob, 0);
        bool any = false;
        for (int p = 0; p < nprob; ++p) if (h_bin_off[p + 1] == h_bin_off[p]) { h_done[p] = -1; any = true; }
        if (any) {
            HC_CUDA(cudaMemcpyAsync(done_at, h_done.data(), sizeof(int32_t) * nprob, cudaMemcpyHostToDevice, s));
            HC_CUDA(cudaStreamSynchronize(s));
        }
    }

    CsrView A{row_ptr, col, cnt, row0, nloc};
    StatArgs st;
    st.bin_off = bin_off; st.nprob = nprob; st.marg = marg; st.bias = bias;
    st.part_sum = part_sum; st.part_cnt = part_cnt; st.part_var = part_var;
    st.done_at = done_at; st.n_done = n_done; st.results = results;
    st.tol = P->tol; st.max_iters = P->max_iters;
    const dim3 sgrid(STAT_SLICES, nprob);

    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    if (h_info) { cudaEventCreate(&ev0); cudaEventCreate(&ev1); cudaEventRecord(ev0, s); }
    const int poll = P->poll_every > 0 ? P->poll_every : 8;
    int launches = 0, h_done = 0, rc = HC_OK;
    for (int k = 1; k <= P->max_iters; ++k) {
        if (nloc > 0) {
            ice_csr_stream_kernel<false><<<stream_grid(), 256, 0, s>>>(A, bias, P->ignore_diags, bin_off, nprob, done_at,
                                                                     k, marg_local, nullptr);
            hc_count_launch(); ++launches;
        }
        if (nccl_comm) {
            rc = hc_nccl_allreduce_f64(nccl_comm, marg_local, marg, (size_t)nbins, s);
            if (rc != HC_OK) break;
        }
        st.k = k;
        ice_stat_sum_kernel<<<sgrid, STAT_THREADS, 0, s>>>(st);
        ice_stat_var_kernel<<<sgrid, STAT_THREADS, 0, s>>>(st);
        ice_stat_update_kernel<<<sgrid, STAT_THREADS, 0, s>>>(st);
        hc_count_launch(3); launches += 3;
        if (k % poll == 0 || k == P->max_iters) {
            cudaError_t e = hc_read_small(&h_done, n_done, sizeof(int32_t), s);
            if (e != cudaSuccess) { hc_set_error("hc_ice_csr_balance: %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; break; }
            if (h_done >= nonempty) break;
        }
    }
    if (h_info && ev0) cudaEventRecord(ev1, s);
    if (rc == HC_OK) {
        ice_csr_finalize_kernel<<<(unsigned)((nbins + 255) / 256), 256, 0, s>>>(bin_off, nprob, results,
                                                                               P->rescale_marginals, bias);
        hc_count_launch(); ++launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { hc_set_error("hc_ice_csr_balance: %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; }
    }
    cudaError_t e = cudaStreamSynchronize(s);
    if (rc == HC_OK && e != cudaSuccess) { hc_set_error("hc_ice_csr_balance: %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; }
    if (h_info) {
        h_info->launches = launches;
        if (ev0 && e == cudaSuccess) cudaEventElapsedTime(&h_info->loop_ms, ev0, ev1);
        if (ev0) { cudaEventDestroy(ev0); cudaEventDestroy(ev1); }
    }
    return rc;
}
