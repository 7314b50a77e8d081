// (b) ICE balancing on dense symmetric int32 tiles  ==  `cooler balance --ignore-diags K [--cis-only]`
// (HiCHap call sites: matrixBuilding.py:708, :713, :1537, :1542, :1761, :1766; algorithm restated
// in oracle/cooler_ice.py from cooler.balance.balance_cooler).
//
// One iteration of EVERY problem (chromosome) of the batch = two launches:
//   stream kernel: persistent warps draw row-group work items from a global queue and compute
//       marg[r] = b[r] * sum_j w(r,j) A[r][j] b[j]   (fp64, warp-shuffle reduction, one store per row);
//   update kernel (one CTA per chromosome): mean / variance of the fresh marginals over the non-zero bins,
//       b <- b / (marg / mean), convergence test var < tol, bookkeeping -- all on the device.
// The whole loop is one launch of a CUDA graph (a WHILE node that the last update CTA of an iteration ends), and the
// update kernel also drops converged chromosomes from the work list: nothing goes back to the host inside the loop.
//
// Two encodings of the matrix for the stream kernel:
//   * int32 tiles as they are (ice_dense_stream_kernel): 4*N^2 bytes per iteration per chromosome, fp64 FMAs;
//   * packed (default, ice_q8_mma_kernel): the tiles are re-encoded ONCE per call into uint8
//     min(w*count, 255) (w = cooler's pixel weight: ignored diagonals become 0) plus a per-row overflow
//     list (col, w*count - 255) for the few cells above 254 -- Hi-C counts are small except next to the
//     diagonal -- so an iteration streams N^2 + 8*overflow bytes, a quarter of the int32 traffic, and the
//     active chromosomes start to fit the 126 MB L2 as the others converge.  A quarter of the bytes means four
//     times the cells per second, and an fp64 FMA per cell then runs out of issue slots (measured: 6 warp
//     instructions per 32 cells, 63 % issue utilisation at half the HBM roofline, profiles/r1h).  So the
//     row sums are computed EXACTLY in integers on the tensor cores instead: the bias vector is held as
//     64-bit fixed point relative to the chromosome's largest bias (every fp64 bias within 2^11 of it is
//     represented exactly), split into 8 unsigned byte planes, and one
//     mma.sync.m16n8k32.u8.u8.s32 multiplies a 16-row x 32-column tile of counts with the 8 planes of those
//     32 columns -- 512 cells per instruction; the 8 int32 plane sums of a row are recombined in fp64.
//     This is not a GEMM reshaped to chase tensor FLOPs (the tensor pipe idles): it removes the per-cell
//     instructions so that the kernel is a pure HBM stream.
#include <cooperative_groups.h>
#include <vector>
#include <algorithm>
#include <math.h>
#include <stdlib.h>
#include "hc_common.cuh"
#include "hc_select.cuh"

namespace {

__device__ __forceinline__ double band_weight(int j, int r, int kd) {
    // pixel weight under cooler's _zero_diags + _marginalize on upper-triangular pixels:
    // |i-j| < ignore_diags -> dropped; a kept diagonal pixel (ignore_diags == 0) counts twice
    const int d = j - r;
    if (d == 0) return kd == 0 ? 2.0 : 0.0;
    return (d < kd && d > -kd) ? 0.0 : 1.0;
}

// ---------------------------------------------------------------------------------------
// filter marginals: per bin, count and sum of kept pixels
// ---------------------------------------------------------------------------------------
// one warp per global bin, grid-stride: the number of bins is read here, so the host launches without waiting for it
__global__ void __launch_bounds__(256)
ice_dense_marginals_kernel(const int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off,
                           const int32_t* __restrict__ mat_n, const int32_t* __restrict__ mat_ld,
                           const int64_t* __restrict__ bin_off, int nprob, int kd,
                           double* __restrict__ nnz_marg, double* __restrict__ marg) {
    const int lane = threadIdx.x & 31;
    const int64_t nbins = bin_off[nprob], nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; g < nbins; g += nwarps) {
        int p = 0;
        while (p + 1 < nprob && bin_off[p + 1] <= g) ++p;
        const int r = (int)(g - bin_off[p]), n = mat_n[p];
        const int64_t ld = mat_ld[p];
        const int32_t* row = mats + mat_off[p] + (int64_t)r * ld;
        const int nvec = (int)(ld >> 2);
        long long s = 0;
        int c = 0;
        for (int v = lane; v < nvec; v += 32) {
            const int4 a = ld_stream_v4(row + 4 * v);
            const int j = 4 * v;
            const int x[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                if (j + e < n) {
                    const double w = band_weight(j + e, r, kd);
                    s += (long long)(w * x[e]);
                    c += (x[e] != 0) ? (int)w : 0;
                }
            }
        }
        s = warp_sum_ll(s);
        c = warp_sum_i(c);
        if (lane == 0) { marg[g] = (double)s; nnz_marg[g] = (double)c; }
    }
}

// ---------------------------------------------------------------------------------------
// bin filters
// ---------------------------------------------------------------------------------------
// grid = nchrom.  bias <- 1, then min_nnz / min_count masks; marg[lo:hi] /= median(marg[lo:hi][>0])
__global__ void __launch_bounds__(1024)
ice_filter_chrom_kernel(const double* __restrict__ nnz_marg, double* __restrict__ marg,
                        const int64_t* __restrict__ chrom_off, int min_nnz, int min_count, int do_mad,
                        double* __restrict__ bias) {
    __shared__ HcSelectSmem sm;
    const int64_t lo = chrom_off[blockIdx.x], hi = chrom_off[blockIdx.x + 1];
    const long long n = hi - lo;
    double* m = marg + lo;
    long long cnt = 0;
    for (long long i = threadIdx.x; i < n; i += blockDim.x) {
        double b = 1.0;
        if (min_nnz > 0 && nnz_marg[lo + i] < (double)min_nnz) b = 0.0;
        if (min_count != 0 && m[i] < (double)min_count) b = 0.0;
        bias[lo + i] = b;
        cnt += (m[i] > 0.0);
    }
    if (!do_mad) return;
    cnt = block_sum_ll(cnt, sm.redll);
    const double med = block_median([&](long long i) { return m[i]; }, [&](long long i) { return m[i] > 0.0; },
                                    n, cnt, &sm);
    __syncthreads();
    for (long long i = threadIdx.x; i < n; i += blockDim.x) m[i] = m[i] / med;
}

// single CTA.  logs of the positive normalised marginals -> median, MAD -> cutoff -> mask
__global__ void __launch_bounds__(1024)
ice_filter_mad_kernel(const double* __restrict__ marg, int64_t nbins, double mad_max,
                      double* __restrict__ bias, double* __restrict__ work) {
    __shared__ HcSelectSmem sm;
    double* lg = work;           // log(marg) where marg > 0
    double* dev = work + nbins;  // |lg - median|
    long long cnt = 0;
    for (long long i = threadIdx.x; i < nbins; i += blockDim.x) {
        const double v = marg[i];
        const bool ok = v > 0.0;  // false for NaN
        lg[i] = ok ? log(v) : 0.0;
        cnt += ok;
    }
    cnt = block_sum_ll(cnt, sm.redll);
    auto valid = [&](long long i) { return marg[i] > 0.0; };
    const double med = block_median([&](long long i) { return lg[i]; }, valid, nbins, cnt, &sm);
    __syncthreads();
    for (long long i = threadIdx.x; i < nbins; i += blockDim.x) dev[i] = fabs(lg[i] - med);
    __syncthreads();
    const double mad = block_median([&](long long i) { return dev[i]; }, valid, nbins, cnt, &sm);
    const double cutoff = exp(med - mad_max * mad);
    for (long long i = threadIdx.x; i < nbins; i += blockDim.x)
        if (marg[i] < cutoff) bias[i] = 0.0;
}

// ---- the same filter over the whole grid -------------------------------------------------
// One CTA streaming 2 x 8 radix passes over all bins is latency-bound (0.5 ms at 62 k bins, ~3 ms at 304 k).  Here every
// pass is one grid-wide launch: CTAs histogram their share into shared memory, add it to a global histogram, and the
// last CTA to finish picks the digit (last-block pattern) -- ~20 short launches whatever the number of bins.
struct MadState {
    unsigned long long prefix, mask;    // radix-select state: keys with (key & mask) == prefix are still candidates
    long long k;                        // rank of the wanted key among the candidates
    long long count;                    // valid (positive-marginal) bins
    long long le;                       // keys <= the selected key
    unsigned long long nxt;             // smallest key above the selected key
    unsigned int done;                  // CTAs that finished the current launch
    unsigned int pad;
    unsigned int hist[256];
    double result[2];                   // median of the log-marginals, median absolute deviation
};
constexpr unsigned long long MAD_INVALID = ~0ull;    // not the key of any finite value
constexpr int MAD_THREADS = 256;

__device__ __forceinline__ long long mad_median_rank(long long count) { return (count & 1) ? count / 2 : count / 2 - 1; }

// last-block pattern: true in every thread of the CTA that finishes last
__device__ __forceinline__ bool mad_last_cta(MadState* st, int* flag_s) {
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned int t = atomicAdd(&st->done, 1u);
        *flag_s = (t == gridDim.x - 1);
        if (*flag_s) st->done = 0;
    }
    __syncthreads();
    const bool last = *flag_s != 0;
    if (last) __threadfence();
    return last;
}

// stage 0: keys of log(marg) for marg > 0 (lg keeps the logs); stage 1: keys of |lg - median|
template <int STAGE>
__global__ void __launch_bounds__(MAD_THREADS)
mad_keys_kernel(const double* __restrict__ marg, long long n, double* __restrict__ lg, unsigned long long* __restrict__ keys,
                MadState* st) {
    __shared__ long long red[32];
    const double med = STAGE ? *reinterpret_cast<volatile double*>(&st->result[0]) : 0.0;
    long long cnt = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const double v = marg[i];
        const bool ok = v > 0.0;            // false for NaN
        unsigned long long key = MAD_INVALID;
        if (STAGE == 0) {
            const double l = ok ? log(v) : 0.0;
            lg[i] = l;
            if (ok) key = f64_key(l);
        } else if (ok) {
            key = f64_key(fabs(__dadd_rn(lg[i], -med)));
        }
        keys[i] = key;
        cnt += ok;
    }
    if (STAGE == 0) {
        cnt = block_sum_ll(cnt, red);
        if (threadIdx.x == 0 && cnt) atomicAdd(reinterpret_cast<unsigned long long*>(&st->count), (unsigned long long)cnt);
    }
}

// one 8-bit digit of the radix select (shift = 56, 48, .. 0)
__global__ void __launch_bounds__(MAD_THREADS)
mad_select_pass_kernel(const unsigned long long* __restrict__ keys, long long n, int shift, MadState* st) {
    __shared__ unsigned int hist[256];
    __shared__ int flag_s;
    const long long count = *reinterpret_cast<volatile long long*>(&st->count);
    if (count == 0) return;
    const bool first = shift == 56;
    const unsigned long long prefix = first ? 0ull : *reinterpret_cast<volatile unsigned long long*>(&st->prefix);
    const unsigned long long mask = first ? 0ull : *reinterpret_cast<volatile unsigned long long*>(&st->mask);
    hist[threadIdx.x] = 0;
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long base = (long long)blockIdx.x * blockDim.x + threadIdx.x; base < n; base += 4 * stride) {
        unsigned long long key[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { const long long i = base + u * stride; key[u] = i < n ? keys[i] : MAD_INVALID; }
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (key[u] != MAD_INVALID && (key[u] & mask) == prefix) atomicAdd(&hist[(key[u] >> shift) & 255ull], 1u);
    }
    __syncthreads();
    if (hist[threadIdx.x]) atomicAdd(&st->hist[threadIdx.x], hist[threadIdx.x]);
    if (!mad_last_cta(st, &flag_s)) return;
    // the last CTA: warp 0 finds the digit that holds rank k (lane l owns digits 8l .. 8l+7)
    if (threadIdx.x < 32) {
        const int lane = threadIdx.x;
        long long k = first ? mad_median_rank(count) : *reinterpret_cast<volatile long long*>(&st->k);
        unsigned int h[8];
        long long s = 0;
#pragma unroll
        for (int e = 0; e < 8; ++e) { h[e] = __ldcg(&st->hist[8 * lane + e]); s += h[e]; }
        long long incl = s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        long long run = incl - s;
        if (k >= run && k < incl) {
            int digit = 8 * lane + 7;
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                if (k < run + h[e]) { digit = 8 * lane + e; break; }
                if (e < 7) run += h[e];
            }
            st->prefix = prefix | ((unsigned long long)digit << shift);
            st->mask = mask | (0xffull << shift);
            st->k = k - run;
            if (shift == 0) { st->le = 0; st->nxt = MAD_INVALID; }
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) st->hist[8 * lane + e] = 0;
    }
}

// neighbours of the selected key -> the median (NumPy: mean of the two middle values for an even count)
template <int STAGE>
__global__ void __launch_bounds__(MAD_THREADS)
mad_median_kernel(const unsigned long long* __restrict__ keys, long long n, MadState* st) {
    __shared__ long long red[32];
    __shared__ unsigned long long redu[32];
    __shared__ int flag_s;
    const long long count = *reinterpret_cast<volatile long long*>(&st->count);
    if (count == 0) {
        if (blockIdx.x == 0 && threadIdx.x == 0) st->result[STAGE] = __longlong_as_double(0x7ff8000000000000ll);
        return;
    }
    const unsigned long long klo = *reinterpret_cast<volatile unsigned long long*>(&st->prefix);
    long long le = 0;
    unsigned long long nxt = MAD_INVALID;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned long long key = keys[i];
        if (key == MAD_INVALID) continue;
        if (key <= klo) ++le; else if (key < nxt) nxt = key;
    }
    le = block_sum_ll(le, red);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_xor_sync(0xffffffffu, nxt, o);
        nxt = other < nxt ? other : nxt;
    }
    if ((threadIdx.x & 31) == 0) redu[threadIdx.x >> 5] = nxt;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < MAD_THREADS / 32; ++w) nxt = redu[w] < nxt ? redu[w] : nxt;
        if (le) atomicAdd(reinterpret_cast<unsigned long long*>(&st->le), (unsigned long long)le);
        atomicMin(&st->nxt, nxt);
    }
    if (!mad_last_cta(st, &flag_s)) return;
    if (threadIdx.x == 0) {
        const long long k = mad_median_rank(count);
        const long long le_all = *reinterpret_cast<volatile long long*>(&st->le);
        const unsigned long long nxt_all = *reinterpret_cast<volatile unsigned long long*>(&st->nxt);
        const double lo = key_f64(klo);
        double hi = lo;
        if (k + 1 < count && le_all < k + 2) hi = key_f64(nxt_all);
        st->result[STAGE] = (count & 1) ? lo : __dmul_rn(__dadd_rn(lo, hi), 0.5);
    }
}

__global__ void __launch_bounds__(MAD_THREADS)
mad_apply_kernel(const double* __restrict__ marg, long long n, double mad_max, const MadState* __restrict__ st,
                 double* __restrict__ bias) {
    const double cutoff = exp(__dadd_rn(st->result[0], -__dmul_rn(mad_max, st->result[1])));
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        if (marg[i] < cutoff) bias[i] = 0.0;
}

// ---------------------------------------------------------------------------------------
// the fused iteration
// ---------------------------------------------------------------------------------------
struct IceDenseArgs {
    const int32_t* mats; const int64_t* mat_off; const int32_t* mat_n; const int32_t* mat_ld;
    const int64_t* pad_off;     // start of each problem in the padded (ld-strided, 128 B aligned) vectors
    const int32_t* item_prob; const int32_t* item_row0; const int32_t* item_nrows;   // work items (~equal bytes)
    const unsigned int* nitems; unsigned int* queue;   // global work queue: warps draw items until it runs dry
    int32_t* iter;              // iteration counter, advanced on the device (the loop is replayed as a CUDA graph)
    double* bias;               // padded layout; updated in place by the update kernel
    double* marg;               // padded layout; fresh marginals of this iteration
    hc_ice_result* results; int32_t* done; int32_t* n_done;
    double tol; int kd; int max_iters; int nprob;
    unsigned int queue_start;   // number of warps of the stream kernel: items below it are pre-assigned
    // packed encoding (ice_q8_mma_kernel)
    const uint8_t* q8; const int64_t* q_off;    // 512-byte tiles (16 rows x 32 columns in A-fragment order), [strip][k-tile]
    uint8_t* digits; int32_t* dig_exp;          // byte planes of the fixed-point bias in B-fragment order (8 B per column); exponent
    const int4* desc; int kseg;                 // packed items: 4 x int4 descriptors (see ice_q8_mma_kernel); a row group is split
                                                // along K into segments of kseg k-tiles
    double* part; int nseg_max; long long npad; // partial row sums part[(k0 / kseg) * npad + pad_off + row], summed by the update kernel
    const int64_t* ovf_ptr; const int32_t* ovf_col; const int32_t* ovf_val;   // per global row: cells with w*count > 255
    int packed;
    // loop control on the device (ice_iteration_end): the last update CTA of an iteration rewrites the live work list when
    // a chromosome has converged, and sets the condition of the graph's WHILE node
    int nonempty;               // chromosomes with at least one bin: the loop ends when n_done reaches it
    unsigned int* upd_cnt;      // update CTAs that finished the current launch
    int32_t* changed;           // a chromosome converged in the current iteration
    const int32_t* rng;         // chromosomes, largest first: [nprob] chromosome | [nprob] first item | [nprob] item end
    int32_t* rng_off;           // [nprob] their offsets in the live work list
    const int32_t* full_row0; const int32_t* full_nrows;   // int32 kernel: the full list of items that the live list filters
    cudaGraphConditionalHandle cond; int has_cond;         // has_cond == 0: plain launches, the host polls n_done
    int loop_end;               // this update launch ends a graph body (or a plain-launch iteration): runs ice_iteration_end
};

// one column chunk (128 columns, 4 per lane) of RG rows: acc[q] += sum_j w * A[rq][j] * b[j]
template <int RG>
__device__ __forceinline__ void consume_chunk(const int4 (&a)[RG], const double* __restrict__ b, int j, int jc,
                                              int rg, int kd, int kspan, double (&acc)[RG]) {
    const double2 b01 = *reinterpret_cast<const double2*>(b + j);        // through L1: reused by every row
    const double2 b23 = *reinterpret_cast<const double2*>(b + j + 2);
    const bool band = jc <= rg + RG - 1 + kspan && jc + 127 >= rg - kspan;   // warp-uniform
#pragma unroll
    for (int q = 0; q < RG; ++q) {
        double x0 = (double)a[q].x, x1 = (double)a[q].y, x2 = (double)a[q].z, x3 = (double)a[q].w;
        if (band) {
            const int r = rg + q;
            x0 *= band_weight(j, r, kd); x1 *= band_weight(j + 1, r, kd);
            x2 *= band_weight(j + 2, r, kd); x3 *= band_weight(j + 3, r, kd);
        }
        acc[q] = fma(x0, b01.x, acc[q]); acc[q] = fma(x1, b01.y, acc[q]);
        acc[q] = fma(x2, b23.x, acc[q]); acc[q] = fma(x3, b23.y, acc[q]);
    }
}

// Streaming half of an iteration: marg[r] = b[r] * sum_j w(r,j) A[r][j] b[j] for every row of every
// unconverged chromosome.  Persistent warps draw row-group items (~48 KB each) from a global queue,
// so the launch stays balanced however the chromosomes differ in size; the next item is drawn
// before the current one is processed, hiding the atomic's latency behind the row loads.
template <int RG, int U, int MINB>
__global__ void __launch_bounds__(256, MINB)
ice_dense_stream_kernel(IceDenseArgs A) {
    const int lane = threadIdx.x & 31;
    const int kd = A.kd, kspan = kd > 0 ? kd - 1 : 0;
    const unsigned nitems = *A.nitems;
    // the first item of a warp is its global index (4736 simultaneous draws on one address would serialise
    // the start of every launch); the queue counter is re-armed to the warp count by the update kernel
    unsigned item = 0;
    if (lane == 0) {
        item = (blockIdx.x * 256u + threadIdx.x) >> 5;
        if (item == 0) atomicAdd(A.iter, 1);       // exactly one warp per launch owns index 0: it opens iteration k
    }
    item = __shfl_sync(0xffffffffu, item, 0);
    while (item < nitems) {
        unsigned next = 0;
        if (lane == 0) next = atomicAdd(A.queue, 1u);
        const int p = A.item_prob[item];
        if (!A.done[p]) {
            const int ld = A.mat_ld[p];            // multiple of 128: every 128-column chunk is full
            const int nchunk = ld >> 7;
            const int64_t lo = A.pad_off[p];
            const int32_t* mat = A.mats + A.mat_off[p];
            const double* __restrict__ b = A.bias + lo;
            double* mout = A.marg + lo;
            const int r0 = A.item_row0[item], r1 = r0 + A.item_nrows[item];
            for (int rg = r0; rg < r1; rg += RG) {
                const int nr = min(RG, r1 - rg);
                const int32_t* base = mat + (int64_t)rg * ld + 4 * lane;
                int roff[RG];                      // ragged last group: re-read the last valid row, discard below
#pragma unroll
                for (int q = 0; q < RG; ++q) roff[q] = min(q, nr - 1) * ld;
                double acc[RG];
#pragma unroll
                for (int q = 0; q < RG; ++q) acc[q] = 0.0;
                int c0 = 0;
                for (; c0 + U <= nchunk; c0 += U) {   // RG x U independent 128-bit streaming loads in flight per lane
                    int4 a[U][RG];
#pragma unroll
                    for (int u = 0; u < U; ++u)
#pragma unroll
                        for (int q = 0; q < RG; ++q) a[u][q] = ld_stream_v4(base + roff[q] + (c0 + u) * 128);
#pragma unroll
                    for (int u = 0; u < U; ++u)
                        consume_chunk<RG>(a[u], b, (c0 + u) * 128 + 4 * lane, (c0 + u) * 128, rg, kd, kspan, acc);
                }
                for (; c0 < nchunk; ++c0) {
                    int4 a[RG];
#pragma unroll
                    for (int q = 0; q < RG; ++q) a[q] = ld_stream_v4(base + roff[q] + c0 * 128);
                    consume_chunk<RG>(a, b, c0 * 128 + 4 * lane, c0 * 128, rg, kd, kspan, acc);
                }
#pragma unroll
                for (int q = 0; q < RG; ++q) {
                    const double sacc = warp_sum(acc[q]);
                    if (lane == 0 && q < nr) mout[rg + q] = b[rg + q] * sacc;
                }
            }
        }
        item = __shfl_sync(0xffffffffu, next, 0);
    }
}

// ---------------------------------------------------------------------------------------
// packed encoding: uint8 tiles + overflow list
// ---------------------------------------------------------------------------------------
// weighted count of cell (r, j): ignored diagonals 0, a kept main diagonal twice (see band_weight)
__device__ __forceinline__ long long weighted_count(int v, int j, int r, int kd) {
    const int d = j - r;
    if (d == 0) return kd == 0 ? 2ll * v : 0ll;
    return (d < kd && d > -kd) ? 0ll : (long long)v;
}

// Tile order of the packed matrix.  A chromosome is cut into strips of 16 rows and k-tiles of 32 columns; tile
// (strip s, k-tile t) is the 512 bytes at q_off[p] + (s * KT + t) * 512, and lane l's 16 bytes of it are exactly
// its A fragment of mma.sync.m16n8k32 (row-major u8): with g = l / 4, c = 4 * (l % 4)
//   word 0: row g,     columns c .. c+3        word 1: row g + 8, columns c .. c+3
//   word 2: row g,     columns 16+c .. 16+c+3  word 3: row g + 8, columns 16+c .. 16+c+3
// so one coalesced 128-bit load per lane feeds one MMA.  Rows past n (last strip) are zero.
__global__ void __launch_bounds__(256)
ice_pack_tiles_kernel(const int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off,
                      const int32_t* __restrict__ mat_n, const int32_t* __restrict__ mat_ld,
                      const int64_t* __restrict__ q_off, const int64_t* __restrict__ strip_off,
                      const int64_t* __restrict__ bin_off, int nprob, int kd, uint8_t* __restrict__ q8,
                      unsigned long long* __restrict__ ovf_cnt, int32_t* __restrict__ ovf_lo, int32_t* __restrict__ ovf_hi) {
    // blockIdx.x / warp -> strip (strip_off = prefix of strips per chromosome); blockIdx.y -> group of 8 k-tiles
    const int64_t gs = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (gs >= strip_off[nprob]) return;
    int p = 0;
    while (p + 1 < nprob && strip_off[p + 1] <= gs) ++p;
    const int sidx = (int)(gs - strip_off[p]), n = mat_n[p], ld = mat_ld[p], KT = ld >> 5;
    const int32_t* M = mats + mat_off[p];
    uint8_t* out = q8 + q_off[p] + (int64_t)sidx * KT * 512 + 16 * lane;
    const int g = lane >> 2, c = 4 * (lane & 3);
    const int ra = sidx * 16 + g, rb = ra + 8;
    const int64_t grow = bin_off[p] + sidx * 16;
    for (int t = 8 * blockIdx.y; t < min(KT, 8 * (int)blockIdx.y + 8); ++t) {
        uint32_t w[4];
#pragma unroll
        for (int h = 0; h < 4; ++h) {
            const int r = (h & 1) ? rb : ra, j0 = t * 32 + ((h & 2) ? 16 : 0) + c;
            uint32_t word = 0;
            if (r < n) {
                const int4 a = ld_stream_v4(M + (int64_t)r * ld + j0);
                const int x[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const long long wc = (j0 + e < n) ? weighted_count(x[e], j0 + e, r, kd) : 0ll;
                    if (wc > 255) {      // rare: a few cells next to the diagonal
                        const int64_t gr = grow + (r - sidx * 16);
                        atomicAdd(ovf_cnt + gr, 1ull);
                        atomicMin(ovf_lo + gr, j0 + e);
                        atomicMax(ovf_hi + gr, j0 + e);
                    }
                    word |= (uint32_t)(wc > 255 ? 255 : (wc < 0 ? 0 : wc)) << (8 * e);
                }
            }
            w[h] = word;
        }
        *reinterpret_cast<uint4*>(out + (int64_t)t * 512) = make_uint4(w[0], w[1], w[2], w[3]);
    }
}

// Byte planes of the bias of one chromosome, in B-fragment order of mma.sync.m16n8k32 (col-major u8, 32 x 8):
// k-tile t owns 256 bytes; lane l = 4 * plane + (column % 16) / 4 holds word (column / 16) whose byte
// (column % 4) is the digit.  Fixed point: F = floor(b * 2^(64 - E)) with 2^E above the chromosome's largest
// bias; plane 0 is the most significant byte.  Called by all threads of a CTA (one CTA per chromosome).
__device__ __forceinline__ void ice_store_digits(const double (&bv)[4], int j4, double pow2, uint32_t* __restrict__ dw) {
    unsigned long long F[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) F[e] = bv[e] > 0.0 ? __double2ull_rn(bv[e] * pow2) : 0ull;     // pow2 = 2^(64 - E): exact scaling; b < 2^E and b has 53 bits, so the product is <= 2^64 - 2^11
    const int t = j4 >> 5, cc = j4 & 31, sub = (cc & 15) >> 2, reg = cc >> 4;
#pragma unroll
    for (int pl = 0; pl < 8; ++pl) {
        const int sh = 8 * (7 - pl);
        const uint32_t word = (uint32_t)((F[0] >> sh) & 255ull) | ((uint32_t)((F[1] >> sh) & 255ull) << 8) |
                              ((uint32_t)((F[2] >> sh) & 255ull) << 16) | ((uint32_t)((F[3] >> sh) & 255ull) << 24);
        dw[t * 64 + (pl * 4 + sub) * 2 + reg] = word;
    }
}

__device__ __forceinline__ double block_max(double v, double* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t = fmax(t, red[w]);
    return t;
}

// exponent E with 2^E above the largest bias, and 2^(64 - E)
__device__ __forceinline__ int digits_exponent(double mx, double* pow2) {
    // mx is a finite normal number here (biases are O(1)); its exponent field gives floor(log2 mx)
    const int E = (mx > 1.0e-300 && mx < 1.0e300) ? (int)((__double_as_longlong(mx) >> 52) & 0x7ff) - 1023 + 1 : 0;
    *pow2 = __longlong_as_double((long long)(1023 + 64 - E) << 52);
    return E;
}

__device__ void ice_write_digits(const double* __restrict__ bw, int n, int ld, uint8_t* __restrict__ dig,
                                 int32_t* __restrict__ exp_out, double* red) {
    double mx = 0.0;
    for (int j = threadIdx.x; j < n; j += blockDim.x) mx = fmax(mx, bw[j]);
    mx = block_max(mx, red);
    double pow2;
    const int E = digits_exponent(mx, &pow2);
    if (threadIdx.x == 0) *exp_out = E;
    uint32_t* dw = reinterpret_cast<uint32_t*>(dig);
    for (int j4 = threadIdx.x * 4; j4 < ld; j4 += blockDim.x * 4) {      // 4 consecutive columns -> one word per plane
        double bv[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) bv[e] = (j4 + e < n) ? bw[j4 + e] : 0.0;
        ice_store_digits(bv, j4, pow2, dw);
    }
}

__global__ void __launch_bounds__(1024) ice_digits_kernel(IceDenseArgs A) {
    __shared__ double red[32];
    const int p = blockIdx.x;
    const int n = A.mat_n[p];
    if (n == 0) return;
    const int64_t lo = A.pad_off[p];
    ice_write_digits(A.bias + lo, n, A.mat_ld[p], A.digits + 8 * lo, A.dig_exp + p, red);
}

// exclusive scan of the per-row overflow counts, in place, total -> ptr[n]: per-block sums (1024 rows per block),
// a single-CTA scan of those, then a local rescan with the block's offset
__global__ void __launch_bounds__(256) ice_ovf_blocksum_kernel(const int64_t* __restrict__ ptr, int64_t n, int64_t* __restrict__ bsum) {
    __shared__ long long redll[8];
    const int64_t base = (int64_t)blockIdx.x * 1024;
    long long s = 0;
    for (int i = threadIdx.x; i < 1024; i += 256) if (base + i < n) s += ptr[base + i];
    s = block_sum_ll(s, redll);
    if (threadIdx.x == 0) bsum[blockIdx.x] = s;
}
__global__ void __launch_bounds__(1024) ice_ovf_scan_blocks_kernel(int64_t* __restrict__ bsum, int nb) {
    __shared__ long long sh[1024];
    long long run = 0;
    for (int b0 = 0; b0 < nb; b0 += 1024) {
        const int i = b0 + threadIdx.x;
        long long v = i < nb ? bsum[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {       // Hillis-Steele inclusive scan
            const long long t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < nb) bsum[i] = run + sh[threadIdx.x] - v;     // exclusive
        run += sh[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) bsum[nb] = run;
}
__global__ void __launch_bounds__(256) ice_ovf_scan_kernel(int64_t* __restrict__ ptr, int64_t n, const int64_t* __restrict__ bsum, int nb) {
    __shared__ long long wsum[8];
    const int64_t base = (int64_t)blockIdx.x * 1024 + 4 * threadIdx.x;
    long long v[4], t = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) { v[e] = base + e < n ? ptr[base + e] : 0; t += v[e]; }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long inc = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
    if (lane == 31) wsum[wid] = inc;
    __syncthreads();
    long long off = bsum[blockIdx.x] + inc - t;
    for (int w = 0; w < wid; ++w) off += wsum[w];
#pragma unroll
    for (int e = 0; e < 4; ++e) { if (base + e < n) ptr[base + e] = off; off += v[e]; }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) ptr[n] = bsum[nb];
}

// pass 2 (one warp per global row): the overflow cells of the row, in column order, from the span pass 1 found
__global__ void __launch_bounds__(256)
ice_pack_ovf_kernel(const int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off,
                    const int32_t* __restrict__ mat_n, const int32_t* __restrict__ mat_ld,
                    const int64_t* __restrict__ bin_off, int nprob, int kd, const int64_t* __restrict__ ovf_ptr,
                    const int32_t* __restrict__ ovf_lo, const int32_t* __restrict__ ovf_hi,
                    int32_t* __restrict__ ovf_col, int32_t* __restrict__ ovf_val, long long cap, IceDenseArgs A,
                    int32_t* __restrict__ abort_flag) {
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (ovf_ptr[bin_off[nprob]] > cap) {
        // more overflow cells than the arrays hold: write none, mark every chromosome done so that the loop streams
        // nothing, and leave the caller's bias alone (ice_finalize_kernel); the host grows the arrays and runs again
        if (g == 0 && lane == 0) {
            *abort_flag = 1;
            for (int p = 0; p < nprob; ++p) A.done[p] = 1;
            *A.n_done = A.nonempty;
        }
        return;
    }
    if (g >= bin_off[nprob]) return;
    int64_t out = ovf_ptr[g];
    if (ovf_ptr[g + 1] == out) return;
    int p = 0;
    while (p + 1 < nprob && bin_off[p + 1] <= g) ++p;
    const int r = (int)(g - bin_off[p]);
    const int32_t* row = mats + mat_off[p] + (int64_t)r * mat_ld[p];
    const int hi = ovf_hi[g];
    for (int j0 = ovf_lo[g]; j0 <= hi; j0 += 32) {
        const int j = j0 + lane;
        const long long w = j <= hi ? weighted_count(row[j], j, r, kd) : 0ll;
        const unsigned m = __ballot_sync(0xffffffffu, w > 255);
        if (w > 255) {
            const int64_t at = out + __popc(m & ((1u << lane) - 1u));
            ovf_col[at] = j;
            ovf_val[at] = (int32_t)(w - 255);
        }
        out += __popc(m);
    }
}

__device__ __forceinline__ void mma_u8(int (&c)[4], const int4& a, const uint2& b) {
    asm volatile("mma.sync.aligned.m16n8k32.row.col.s32.u8.u8.s32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+r"(c[0]), "+r"(c[1]), "+r"(c[2]), "+r"(c[3])
                 : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y));
}

// Streaming half of an iteration on the packed encoding.  Same work distribution as the int32 kernel (persistent
// warps, global queue of items; a row group is one strip of 16 rows).  Per k-tile a lane issues one 128-bit
// streaming load (its A fragment), one 64-bit load of the bias planes (B fragment, through L1) and one MMA;
// Q8_U k-tiles are in flight.  C fragment: lane l holds, for rows g and g + 8 (g = l / 4), the int32 sums of
// planes 2 * (l % 4) and 2 * (l % 4) + 1 -- folded into fp64 with the planes' weights, reduced over the 4 lanes
// of the group, scaled by 2^(E - 64), plus the row's overflow cells in fp64.
// 16 k-tiles in flight per lane at 2 CTAs/SM (16 warps/SM): the fastest of the variants measured on B200.
constexpr int Q8_U = 16, Q8_MINB = 2;
__global__ void __launch_bounds__(256, Q8_MINB)
ice_q8_mma_kernel(IceDenseArgs A) {
    const int lane = threadIdx.x & 31;
    const int g = lane >> 2, t4 = lane & 3;
    // weights of this lane's two planes: 2^(8 * (7 - plane)), exact
    const double w_even = __longlong_as_double((long long)(1023 + 8 * (7 - 2 * t4)) << 52);
    const double w_odd = __longlong_as_double((long long)(1023 + 8 * (6 - 2 * t4)) << 52);
    const unsigned nitems = *A.nitems;
    // An item = one strip x one K segment, described by 4 x int4 the host precomputed:
    //   d0 = tile byte offset (int64) | index of the item's first partial sum (int64)
    //   d1 = byte offset of the segment's bias planes (int64) | global row of the first row (int64)
    //   d2 = chromosome, offset of the chromosome in the padded vectors, (unused), rows
    //   d3 = k-tiles in the segment, segment index, (k-tiles per strip, unused), (unused)
    // Items 0..W-1 are pre-assigned to the W warps; the rest are drawn from the global queue.  The descriptor
    // of the NEXT item is fetched while the current one is processed, and the draw after that is in flight too,
    // so no item starts with a chain of dependent L2 reads.
    unsigned cur = (blockIdx.x * 256u + threadIdx.x) >> 5;
    unsigned nxt = 0;
    if (lane == 0) {
        nxt = atomicAdd(A.queue, 1u);
        if (cur == 0) atomicAdd(A.iter, 1);       // exactly one warp per launch owns index 0: it opens iteration k
    }
    int4 d0 = make_int4(0, 0, 0, 0), d1 = d0, d2 = d0, d3 = d0;
    // (A.item_prob is the list of live item ids here: the descriptors stay put, the host only re-uploads that list)
    if (cur < nitems) {
        const int4* dp = A.desc + 4 * (int64_t)A.item_prob[cur];
        d0 = __ldg(dp); d1 = __ldg(dp + 1); d2 = __ldg(dp + 2); d3 = __ldg(dp + 3);
    }
    nxt = __shfl_sync(0xffffffffu, nxt, 0);
    while (cur < nitems) {
        unsigned drawn = 0;
        if (lane == 0) drawn = atomicAdd(A.queue, 1u);
        int4 e0 = make_int4(0, 0, 0, 0), e1 = e0, e2 = e0, e3 = e0;
        if (nxt < nitems) {
            const int4* dp = A.desc + 4 * (int64_t)A.item_prob[nxt];
            e0 = __ldg(dp); e1 = __ldg(dp + 1); e2 = __ldg(dp + 2); e3 = __ldg(dp + 3);
        }
        const int p = d2.x;
        if (!A.done[p]) {
            const int64_t tile_off = ((int64_t)(uint32_t)d0.x) | ((int64_t)d0.y << 32);
            const int64_t part_base = ((int64_t)(uint32_t)d0.z) | ((int64_t)d0.w << 32);
            const int64_t dig_off = ((int64_t)(uint32_t)d1.x) | ((int64_t)d1.y << 32);
            const int64_t grow = ((int64_t)(uint32_t)d1.z) | ((int64_t)d1.w << 32);
            const int nrows = d2.w, nk = d3.x, seg = d3.y;
            const uint8_t* qp = A.q8 + tile_off + 16 * lane;
            const uint8_t* dig = A.digits + dig_off + 8 * lane;
            const double* __restrict__ b = A.bias + d2.y;
            const double scale = __longlong_as_double((long long)(1023 + A.dig_exp[p] - 64) << 52);   // 2^(E - 64)
            double* pout = A.part + part_base;
            int c[4] = {0, 0, 0, 0};
            for (int t = 0; t < nk; t += Q8_U) {       // nk <= 1024: the int32 plane sums cannot overflow
                int4 a[Q8_U];
                uint2 bf[Q8_U];
#pragma unroll
                for (int u = 0; u < Q8_U; ++u) {
                    const int tt = min(t + u, nk - 1);
                    a[u] = ld_stream_v4(reinterpret_cast<const int32_t*>(qp + (int64_t)tt * 512));
                    bf[u] = t + u < nk ? *reinterpret_cast<const uint2*>(dig + (int64_t)tt * 256) : make_uint2(0u, 0u);
                }
#pragma unroll
                for (int u = 0; u < Q8_U; ++u) mma_u8(c, a[u], bf[u]);
            }
            const int ra = g, rb = g + 8;
            double va = ((double)c[0] * w_even + (double)c[1] * w_odd) * scale;
            double vb = ((double)c[2] * w_even + (double)c[3] * w_odd) * scale;
            if (seg == 0) {      // the first segment of a row also carries its overflow cells
                if (ra < nrows) {
                    const int64_t x0 = A.ovf_ptr[grow + ra], x1 = A.ovf_ptr[grow + ra + 1];
                    for (int64_t e = x0 + t4; e < x1; e += 4) va = fma((double)A.ovf_val[e], b[A.ovf_col[e]], va);
                }
                if (rb < nrows) {
                    const int64_t x0 = A.ovf_ptr[grow + rb], x1 = A.ovf_ptr[grow + rb + 1];
                    for (int64_t e = x0 + t4; e < x1; e += 4) vb = fma((double)A.ovf_val[e], b[A.ovf_col[e]], vb);
                }
            }
            va += __shfl_xor_sync(0xffffffffu, va, 1); va += __shfl_xor_sync(0xffffffffu, va, 2);
            vb += __shfl_xor_sync(0xffffffffu, vb, 1); vb += __shfl_xor_sync(0xffffffffu, vb, 2);
            if (t4 == 0) {
                if (ra < nrows) pout[ra] = va;
                if (rb < nrows) pout[rb] = vb;
            }
        }
        cur = nxt; d0 = e0; d1 = e1; d2 = e2; d3 = e3;
        nxt = __shfl_sync(0xffffffffu, drawn, 0);
    }
}

__device__ __forceinline__ void ice_mark_done(const IceDenseArgs& A, int p) {
    A.done[p] = 1;
    atomicAdd(A.n_done, 1);
    *A.changed = 1;
}

// The live work list after a convergence: the items of the chromosomes still running, in the order of A.rng (largest
// first), and their number.  Run by the whole last CTA of an update launch, when every other CTA has finished.
__device__ void ice_compact_items(const IceDenseArgs& A) {
    __shared__ int wsum[32];
    __shared__ int total_s;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5, nprob = A.nprob;
    if (threadIdx.x == 0) total_s = 0;
    __syncthreads();
    for (int i0 = 0; i0 < nprob; i0 += blockDim.x) {      // exclusive scan of the live item counts
        const int i = i0 + threadIdx.x;
        const int cnt = i < nprob && !__ldcg(A.done + A.rng[i]) ? A.rng[2 * nprob + i] - A.rng[nprob + i] : 0;
        int inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += t; }
        if (lane == 31) wsum[wid] = inc;
        __syncthreads();
        int off = total_s;
        for (int w = 0; w < wid; ++w) off += wsum[w];
        if (i < nprob) A.rng_off[i] = off + inc - cnt;
        __syncthreads();
        if (threadIdx.x == blockDim.x - 1) total_s = off + inc;
        __syncthreads();
    }
    int32_t* prob = const_cast<int32_t*>(A.item_prob);
    int32_t* row0 = const_cast<int32_t*>(A.item_row0);
    int32_t* nrows = const_cast<int32_t*>(A.item_nrows);
    for (int i = wid; i < nprob; i += nw) {                // one warp per chromosome
        const int p = A.rng[i];
        if (__ldcg(A.done + p)) continue;
        const int lo = A.rng[nprob + i], m = A.rng[2 * nprob + i] - lo, off = A.rng_off[i];
        for (int j = lane; j < m; j += 32) {
            if (A.packed) { prob[off + j] = lo + j; continue; }      // packed: descriptor ids
            prob[off + j] = p; row0[off + j] = A.full_row0[lo + j]; nrows[off + j] = A.full_nrows[lo + j];
        }
    }
    if (threadIdx.x == 0) { *const_cast<unsigned int*>(A.nitems) = (unsigned)total_s; *A.changed = 0; }
}

// Tail of the update launch that ends a graph body: the last CTA to finish compacts the work list if a chromosome
// converged, and decides whether the graph's WHILE node runs another body -- so the loop needs no host round trip.
__device__ void ice_iteration_end(const IceDenseArgs& A) {
    __shared__ int last_s;
    if (!A.loop_end) return;    // within a graph body the stream kernel skips the items of converged chromosomes
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        const unsigned t = atomicAdd(A.upd_cnt, 1u);
        last_s = t == gridDim.x - 1;
        if (last_s) *A.upd_cnt = 0;
    }
    __syncthreads();
    if (!last_s) return;
    __threadfence();
    if (*reinterpret_cast<volatile int32_t*>(A.changed)) ice_compact_items(A);
    if (threadIdx.x == 0 && A.has_cond) {
        const int k = *reinterpret_cast<volatile int32_t*>(A.iter);
        const int nd = *reinterpret_cast<volatile int32_t*>(A.n_done);
        cudaGraphSetConditional(A.cond, nd < A.nonempty && k < A.max_iters ? 1u : 0u);
    }
}

// Vector half of an iteration (grid = one CTA per chromosome): mean / variance of the fresh
// marginals over the non-zero bins, bias update b /= marg/mean (in place), convergence test,
// scale / iteration bookkeeping -- all on the device.
__device__ __forceinline__ void ice_dense_update(const IceDenseArgs& A) {
    __shared__ double red[32];
    __shared__ long long redll[32];
    const int p = blockIdx.x;
    const int k = *A.iter;                                // opened by this iteration's stream kernel
    if (p == 0 && threadIdx.x == 0) *A.queue = A.queue_start;   // re-arm the work queue for the next iteration
    if (A.done[p] || k > A.max_iters) return;
    const int n = A.mat_n[p];
    if (n == 0) return;
    const int64_t lo = A.pad_off[p];
    double* m_in = A.marg + lo;
    double* bw = A.bias + lo;
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (A.packed && n <= 8 * (int)blockDim.x) {
        // packed encoding, register-resident: thread t owns columns 4t..4t+3 (and 4096+4t.. for the second half):
        // one round of loads (partial sums + bias), everything else in registers, one round of stores
        const int nseg = ((A.mat_ld[p] >> 5) + A.kseg - 1) / A.kseg;
        const int ld = A.mat_ld[p];
        const double* part = A.part + lo;
        double m[8], bb[8];
        double s = 0.0;
        long long c = 0;
        // all loads of the thread are issued before the first use: 4 consecutive columns per half = two 16-byte loads
        // per segment (the padded vectors are 128-byte aligned and ld entries long: no bound check needed below ld)
        const int ja = 4 * threadIdx.x, jb = 4 * (int)blockDim.x + 4 * threadIdx.x;
        const bool ina = ja < ld, inb = jb < ld;
#pragma unroll
        for (int i = 0; i < 8; ++i) m[i] = 0.0;
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (q < nseg) {
                const double* pq = part + (int64_t)q * A.npad;
                if (ina) {
                    const double2 x = *reinterpret_cast<const double2*>(pq + ja), y = *reinterpret_cast<const double2*>(pq + ja + 2);
                    m[0] += x.x; m[1] += x.y; m[2] += y.x; m[3] += y.y;
                }
                if (inb) {
                    const double2 x = *reinterpret_cast<const double2*>(pq + jb), y = *reinterpret_cast<const double2*>(pq + jb + 2);
                    m[4] += x.x; m[5] += x.y; m[6] += y.x; m[7] += y.y;
                }
            }
        }
        for (int q = 8; q < nseg; ++q) {        // more than 8 segments: rare (kseg is chosen so that it does not happen)
            const double* pq = part + (int64_t)q * A.npad;
#pragma unroll
            for (int e = 0; e < 4; ++e) { if (ina) m[e] += pq[ja + e]; if (inb) m[4 + e] += pq[jb + e]; }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) bb[i] = 0.0;
        if (ina) {
            const double2 x = *reinterpret_cast<const double2*>(bw + ja), y = *reinterpret_cast<const double2*>(bw + ja + 2);
            bb[0] = x.x; bb[1] = x.y; bb[2] = y.x; bb[3] = y.y;
        }
        if (inb) {
            const double2 x = *reinterpret_cast<const double2*>(bw + jb), y = *reinterpret_cast<const double2*>(bw + jb + 2);
            bb[4] = x.x; bb[5] = x.y; bb[6] = y.x; bb[7] = y.y;
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int j = (i < 4 ? ja : jb) + (i & 3);
            m[i] = j < n ? bb[i] * m[i] : 0.0;          // rows past n of the last strip hold no partial sums
            if (j >= n) bb[i] = 0.0;
            if (m[i] != 0.0) { s += m[i]; ++c; }
        }
        s = block_sum(s, red);
        c = block_sum_ll(c, redll);
        if (c == 0) {   // nothing left to balance: cooler sets bias = NaN, scale = NaN, var = 0
            if (threadIdx.x == 0) {
                hc_ice_result r; r.scale = nan; r.var = 0.0; r.iters = k; r.converged = 1;
                A.results[p] = r; ice_mark_done(A, p);
            }
            return;
        }
        const double mean = s / (double)c;
        double v = 0.0, mx = 0.0;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            if (m[i] != 0.0) { const double d = m[i] - mean; v += d * d; }
            double q = m[i] / mean;
            if (q == 0.0) q = 1.0;
            bb[i] = bb[i] / q;
            mx = fmax(mx, bb[i]);
        }
        const double var = block_sum(v, red) / (double)c;
        mx = block_max(mx, red);
        double pow2;
        const int E = digits_exponent(mx, &pow2);
        uint32_t* dw = reinterpret_cast<uint32_t*>(A.digits + 8 * lo);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int j4 = h * 4 * (int)blockDim.x + 4 * threadIdx.x;
            if (j4 < ld) {
                double bv[4];
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    bv[e] = bb[4 * h + e];
                    if (j4 + e < n) { bw[j4 + e] = bv[e]; m_in[j4 + e] = m[4 * h + e]; }
                }
                ice_store_digits(bv, j4, pow2, dw);
            }
        }
        if (threadIdx.x == 0) {
            A.dig_exp[p] = E;
            hc_ice_result r; r.scale = mean; r.var = var; r.iters = k; r.converged = var < A.tol;
            A.results[p] = r;
            if (var < A.tol || k >= A.max_iters) { ice_mark_done(A, p); }
        }
        return;
    }
    double s = 0.0;
    long long c = 0;
    if (A.packed) {      // marg[r] = b[r] * (sum of the row's K-segment partial sums, in segment order)
        const int nseg = ((A.mat_ld[p] >> 5) + A.kseg - 1) / A.kseg;
        const double* part = A.part + lo;
        for (int j = threadIdx.x; j < n; j += blockDim.x) {
            double t = 0.0;
            for (int q = 0; q < nseg; ++q) t += part[(int64_t)q * A.npad + j];
            m_in[j] = bw[j] * t;
        }
    }
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        const double m = m_in[j];
        if (m != 0.0) { s += m; ++c; }
    }
    s = block_sum(s, red);
    c = block_sum_ll(c, redll);
    if (c == 0) {   // nothing left to balance: cooler sets bias = NaN, scale = NaN, var = 0
        if (threadIdx.x == 0) {
            hc_ice_result r; r.scale = nan; r.var = 0.0;
            r.iters = k; r.converged = 1;
            A.results[p] = r; ice_mark_done(A, p);
        }
        return;
    }
    const double mean = s / (double)c;
    double v = 0.0;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        const double m = m_in[j];
        if (m != 0.0) { const double d = m - mean; v += d * d; }
    }
    const double var = block_sum(v, red) / (double)c;
    for (int j = threadIdx.x; j < n; j += blockDim.x) {
        double m = m_in[j] / mean;
        if (m == 0.0) m = 1.0;
        bw[j] = bw[j] / m;
    }
    if (threadIdx.x == 0) {
        hc_ice_result r; r.scale = mean; r.var = var; r.iters = k; r.converged = var < A.tol;
        A.results[p] = r;
        if (var < A.tol || k >= A.max_iters) { ice_mark_done(A, p); }
    }
    if (A.packed) {      // the stream kernel reads the bias as byte planes
        __syncthreads();
        ice_write_digits(bw, n, A.mat_ld[p], A.digits + 8 * lo, A.dig_exp + p, red);
    }
}
__global__ void __launch_bounds__(1024)
ice_dense_update_kernel(IceDenseArgs A) {
    ice_dense_update(A);
    ice_iteration_end(A);
}

// The same update for the packed encoding when every chromosome has at most 8192 padded columns: a thread-block
// CLUSTER of 8 CTAs x 256 threads per chromosome, 4 consecutive columns per thread, everything in registers,
// the three chromosome-wide reductions (sum / count, variance, max) through distributed shared memory.  The
// single-CTA kernel above spends ~25 us per iteration on this (latency: six block barriers, 16 fp64 divisions and
// 450 KB through one SM); that is a third of an iteration once the matrix pass takes ~50 us.
constexpr int UPD_CLUSTER = 8;
__device__ __forceinline__ void ice_q8_update_cluster(const IceDenseArgs& A) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double red[8];
    __shared__ long long redll[8];
    __shared__ double sh_sum, sh_var, sh_max;
    __shared__ long long sh_cnt;
    const int p = blockIdx.x / UPD_CLUSTER, rank = (int)cluster.block_rank();
    const int k = *A.iter;
    if (blockIdx.x == 0 && threadIdx.x == 0) *A.queue = A.queue_start;
    if (A.done[p] || k > A.max_iters) return;       // uniform over the cluster
    const int n = A.mat_n[p];
    if (n == 0) return;
    const int64_t lo = A.pad_off[p];
    const int ld = A.mat_ld[p];
    double* m_in = A.marg + lo;
    double* bw = A.bias + lo;
    const int nseg = ((ld >> 5) + A.kseg - 1) / A.kseg;
    const double* part = A.part + lo;
    const int j4 = 4 * (rank * 256 + (int)threadIdx.x);
    const bool in = j4 < ld;
    double m[4] = {0.0, 0.0, 0.0, 0.0}, bb[4] = {0.0, 0.0, 0.0, 0.0};
    if (in) {
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            if (q < nseg) {
                const double* pq = part + (int64_t)q * A.npad + j4;
                const double2 x = *reinterpret_cast<const double2*>(pq), y = *reinterpret_cast<const double2*>(pq + 2);
                m[0] += x.x; m[1] += x.y; m[2] += y.x; m[3] += y.y;
            }
        }
        for (int q = 8; q < nseg; ++q) {
            const double* pq = part + (int64_t)q * A.npad + j4;
#pragma unroll
            for (int e = 0; e < 4; ++e) m[e] += pq[e];
        }
        const double2 x = *reinterpret_cast<const double2*>(bw + j4), y = *reinterpret_cast<const double2*>(bw + j4 + 2);
        bb[0] = x.x; bb[1] = x.y; bb[2] = y.x; bb[3] = y.y;
    }
    double s = 0.0;
    long long c = 0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        m[e] = (j4 + e < n) ? bb[e] * m[e] : 0.0;      // rows past n of the last strip hold no partial sums
        if (j4 + e >= n) bb[e] = 0.0;
        if (m[e] != 0.0) { s += m[e]; ++c; }
    }
    s = block_sum(s, red);
    c = block_sum_ll(c, redll);
    if (threadIdx.x == 0) { sh_sum = s; sh_cnt = c; }
    cluster.sync();
    s = 0.0; c = 0;
#pragma unroll
    for (int r = 0; r < UPD_CLUSTER; ++r) {       // rank order: every CTA gets the same bits
        s += *cluster.map_shared_rank(&sh_sum, r);
        c += *cluster.map_shared_rank(&sh_cnt, r);
    }
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (c == 0) {   // nothing left to balance: cooler sets bias = NaN, scale = NaN, var = 0
        if (rank == 0 && threadIdx.x == 0) {
            hc_ice_result r; r.scale = nan; r.var = 0.0; r.iters = k; r.converged = 1;
            A.results[p] = r; ice_mark_done(A, p);
        }
        cluster.sync();      // nobody leaves while its shared memory may still be read
        return;
    }
    const double mean = s / (double)c;
    double v = 0.0, mx = 0.0;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        if (m[e] != 0.0) { const double d = m[e] - mean; v += d * d; }
        double q = m[e] / mean;
        if (q == 0.0) q = 1.0;
        bb[e] = bb[e] / q;
        mx = fmax(mx, bb[e]);
    }
    v = block_sum(v, red);
    mx = block_max(mx, red);
    if (threadIdx.x == 0) { sh_var = v; sh_max = mx; }
    cluster.sync();
    v = 0.0; mx = 0.0;
#pragma unroll
    for (int r = 0; r < UPD_CLUSTER; ++r) {
        v += *cluster.map_shared_rank(&sh_var, r);
        mx = fmax(mx, *cluster.map_shared_rank(&sh_max, r));
    }
    const double var = v / (double)c;
    double pow2;
    const int E = digits_exponent(mx, &pow2);
    if (in) {
#pragma unroll
        for (int e = 0; e < 4; ++e)
            if (j4 + e < n) { bw[j4 + e] = bb[e]; m_in[j4 + e] = m[e]; }
        ice_store_digits(bb, j4, pow2, reinterpret_cast<uint32_t*>(A.digits + 8 * lo));
    }
    if (rank == 0 && threadIdx.x == 0) {
        A.dig_exp[p] = E;
        hc_ice_result r; r.scale = mean; r.var = var; r.iters = k; r.converged = var < A.tol;
        A.results[p] = r;
        if (var < A.tol || k >= A.max_iters) { ice_mark_done(A, p); }
    }
    cluster.sync();          // keep every CTA's shared memory alive until the remote reads are done
}
__global__ void __cluster_dims__(UPD_CLUSTER, 1, 1) __launch_bounds__(256)
ice_q8_update_cluster_kernel(IceDenseArgs A) {
    ice_q8_update_cluster(A);
    ice_iteration_end(A);
}

// user bias (concatenated bins) <-> padded internal layout
__global__ void __launch_bounds__(256)
ice_pad_bias_kernel(const int64_t* __restrict__ bin_off, const int64_t* __restrict__ pad_off, int nprob,
                    const double* __restrict__ bias, double* __restrict__ padded) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= bin_off[nprob]) return;
    int p = 0;
    while (p + 1 < nprob && bin_off[p + 1] <= g) ++p;
    padded[pad_off[p] + (g - bin_off[p])] = bias[g];
}

// final weights: bias==0 -> NaN; divide by sqrt(scale) when rescaling (cooler balance_cooler tail)
__global__ void __launch_bounds__(256)
ice_finalize_kernel(const int64_t* __restrict__ bin_off, const int64_t* __restrict__ pad_off, int nprob,
                    const hc_ice_result* __restrict__ results, int rescale, const double* __restrict__ padded,
                    double* __restrict__ bias, const int32_t* __restrict__ abort_flag) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= bin_off[nprob] || *abort_flag) return;
    int p = 0;
    while (p + 1 < nprob && bin_off[p + 1] <= g) ++p;
    const hc_ice_result r = results[p];
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    double b = padded[pad_off[p] + (g - bin_off[p])];
    if (isnan(r.scale)) b = nan;
    else {
        if (b == 0.0) b = nan;
        if (rescale) b = b / sqrt(r.scale);
    }
    bias[g] = b;
}

// timing events of one balancing call, released on every exit path
struct EventPair {
    cudaEvent_t a = nullptr, b = nullptr;
    void create() { cudaEventCreate(&a); cudaEventCreate(&b); }
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

typedef void (*StreamKernel)(IceDenseArgs);
struct StreamVariant { StreamKernel fn; int rg, minb; };
// int32 kernel, tuned on B200 (profiles/): RG rows share the bias loads; RG*U 128-bit loads in flight per lane.
// <4,2,4> is the fastest per byte (5.5 TB/s on C2, profiles/r1c_ice_variants_v3.log); the others keep every
// resident warp busy when the batch has few rows.
const StreamVariant kVariants[] = {
    {ice_dense_stream_kernel<4, 2, 4>, 4, 4},
    {ice_dense_stream_kernel<2, 2, 4>, 2, 4},
    {ice_dense_stream_kernel<1, 4, 4>, 1, 4},
};
// packed kernel: an item is one strip of 16 rows
const StreamVariant kQ8 = {ice_q8_mma_kernel, 16, Q8_MINB};

// Everything of hc_ice_dense_balance that depends only on the launch shape, kept between calls (per host thread and
// device): the host tables (work-item descriptors, padded offsets) and their device copies, every scratch buffer, and
// the instantiated graph of the iteration loop.  Each pointer in A is owned here, so the graph's kernel nodes are the
// same for every call of the shape and a repeated call neither builds nor uploads anything.
struct IceDenseCache {
    // key
    int packed = -1, nprob = 0, kseg = 0, cluster = 0, timed = 0, kd = 0, max_iters = 0;
    StreamKernel fn = nullptr;
    double tol = 0.0;
    const void* mats = nullptr; const void* mat_off = nullptr;   // int32 kernel only: it streams the caller's tiles
    std::vector<int32_t> n, ld;
    // device memory of the shape (one allocation)
    unsigned char* mem = nullptr;
    IceDenseArgs A;
    int32_t* state = nullptr;          // per-call state, reset from `pristine` at the start of every call
    const int32_t* pristine = nullptr;
    size_t state_ints = 0;
    int64_t* ovf_ptr = nullptr; int64_t* qoff = nullptr; int64_t* strip = nullptr; int32_t* lo = nullptr; int32_t* hi = nullptr;
    int32_t* abort_flag = nullptr;
    int64_t nbins = 0, strips = 0;
    int kt_max = 0, grid = 0;
    // overflow cells (packed encoding): grow-only capacity, kept across shapes
    int32_t* ovf = nullptr;
    long long ovf_cap = 0;
    // the iteration loop as one graph: first iteration, then a WHILE node over the same two kernels
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    cudaEvent_t ev[2] = {nullptr, nullptr};    // around the first stream launch (HC_ICE_TIME_KERNEL=1)
    long long* mbox = nullptr;                 // pinned: [0] overflow cells, [1] iterations (int32) of the last call
    void drop_graph() {
        if (exec) cudaGraphExecDestroy(exec);
        if (graph) cudaGraphDestroy(graph);
        exec = nullptr; graph = nullptr;
    }
    void drop() {
        drop_graph();
        if (mem) cudaFree(mem);
        mem = nullptr; packed = -1; n.clear(); ld.clear();
    }
};

}  // namespace

extern "C" int hc_ice_dense_marginals(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                      const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                                      int32_t ignore_diags, double* nnz_marg, double* marg, void* stream) {
    HC_REQUIRE(nprob > 0 && ignore_diags >= 0, "nprob>0, ignore_diags>=0");
    // grid-stride over the bins (count read on the device): no wait for the binning that precedes this call
    ice_dense_marginals_kernel<<<(unsigned)hc_num_sms() * 8, 256, 0, (cudaStream_t)stream>>>(
        mats, mat_off, mat_n, mat_ld, bin_off, nprob, ignore_diags, nnz_marg, marg);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_ice_filter_bins(const double* nnz_marg, double* marg, int64_t nbins, const int64_t* chrom_off,
                                  int32_t nchrom, const hc_ice_params* P, double* bias, double* work, void* stream) {
    HC_REQUIRE(nbins >= 0 && nchrom > 0 && P != nullptr, "nbins>=0, nchrom>0, params");
    if (nbins == 0) return HC_OK;
    const int do_mad = P->mad_max > 0.0;
    ice_filter_chrom_kernel<<<nchrom, 1024, 0, (cudaStream_t)stream>>>(nnz_marg, marg, chrom_off, P->min_nnz,
                                                                      P->min_count, do_mad, bias);
    HC_LAUNCH_CHECK();
    if (do_mad) {
        // small problems (one chromosome, a few thousand bins): the single-CTA kernel is one ~20 us launch, the grid-wide
        // select ~20 launches of ~4 us each; HC_ICE_MAD_SINGLE=1 / 0 forces either
        const char* e_single = getenv("HC_ICE_MAD_SINGLE");
        const bool single = e_single ? atoi(e_single) != 0 : nbins < 8192;
        if (single) {
            ice_filter_mad_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(marg, nbins, P->mad_max, bias, work);
            HC_LAUNCH_CHECK();
            return HC_OK;
        }
        cudaStream_t s = (cudaStream_t)stream;
        // the 1 KB select state lives in a per-thread buffer that is kept between calls: a stream-ordered allocation here was
        // carved out of the default pool's largest free block and cost the next multi-MB request of another call fresh mappings
        struct MadCache { MadState* p = nullptr; int dev = -1; cudaStream_t last = nullptr; bool used = false; };
        static thread_local MadCache mc;
        int dev = 0;
        HC_CUDA(cudaGetDevice(&dev));
        if (mc.p == nullptr || mc.dev != dev) {
            if (mc.p) { cudaFree(mc.p); mc.p = nullptr; }
            HC_CUDA(cudaMalloc(reinterpret_cast<void**>(&mc.p), sizeof(MadState)));
            mc.dev = dev; mc.used = false;
        }
        if (mc.used && mc.last != s) HC_CUDA(cudaStreamSynchronize(mc.last));     // the previous call ran on another stream
        mc.last = s; mc.used = true;
        MadState* st = mc.p;
        HC_CUDA(cudaMemsetAsync(st, 0, sizeof(MadState), s));
        double* lg = work;
        unsigned long long* keys = reinterpret_cast<unsigned long long*>(work + nbins);
        long long grid = (nbins + MAD_THREADS * 4 - 1) / (MAD_THREADS * 4);
        const long long cap = 2ll * hc_num_sms();
        if (grid > cap) grid = cap;
        const unsigned g = (unsigned)grid;
        mad_keys_kernel<0><<<g, MAD_THREADS, 0, s>>>(marg, nbins, lg, keys, st);
        for (int shift = 56; shift >= 0; shift -= 8) mad_select_pass_kernel<<<g, MAD_THREADS, 0, s>>>(keys, nbins, shift, st);
        mad_median_kernel<0><<<g, MAD_THREADS, 0, s>>>(keys, nbins, st);
        mad_keys_kernel<1><<<g, MAD_THREADS, 0, s>>>(marg, nbins, lg, keys, st);
        for (int shift = 56; shift >= 0; shift -= 8) mad_select_pass_kernel<<<g, MAD_THREADS, 0, s>>>(keys, nbins, shift, st);
        mad_median_kernel<1><<<g, MAD_THREADS, 0, s>>>(keys, nbins, st);
        mad_apply_kernel<<<g, MAD_THREADS, 0, s>>>(marg, nbins, P->mad_max, st, bias);
        HC_LAUNCH_CHECK();
    }
    return HC_OK;
}


extern "C" int hc_ice_dense_balance(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                    const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                                    const int32_t* h_mat_n, const hc_ice_params* P, double* bias,
                                    hc_ice_result* results, hc_ice_run_info* h_info, void* stream) {
    HC_REQUIRE(nprob > 0 && h_mat_n != nullptr && P != nullptr, "nprob>0, h_mat_n, params");
    HC_REQUIRE(P->max_iters >= 1 && P->ignore_diags >= 0, "max_iters>=1, ignore_diags>=0");
    int64_t nbins = 0;
    for (int p = 0; p < nprob; ++p) {
        HC_REQUIRE(h_mat_n[p] >= 0, "matrix side");
        nbins += h_mat_n[p];
    }
    if (h_info) { h_info->launches = 0; h_info->loop_ms = 0.f; h_info->packed = 0; h_info->pack_ms = 0.f; h_info->overflow_cells = 0; h_info->stream_full_ms = 0.f; h_info->stream_full_launches = 0; }
    if (nbins == 0) return HC_OK;
    // The iteration loop is a CUDA graph, which cannot be captured or launched on the legacy default stream: run on a
    // private stream ordered after the caller's stream (the call synchronises before returning, so the caller's later
    // work is ordered after it).
    static thread_local cudaStream_t private_stream[64] = {nullptr};
    int dev = 0;
    HC_CUDA(cudaGetDevice(&dev));
    HC_REQUIRE(dev >= 0 && dev < 64, "device index");
    if (!private_stream[dev]) HC_CUDA(cudaStreamCreateWithFlags(&private_stream[dev], cudaStreamNonBlocking));
    cudaStream_t s = private_stream[dev];
    {
        cudaEvent_t e_in;
        HC_CUDA(cudaEventCreateWithFlags(&e_in, cudaEventDisableTiming));
        HC_CUDA(cudaEventRecord(e_in, (cudaStream_t)stream));
        HC_CUDA(cudaStreamWaitEvent(s, e_in, 0));
        cudaEventDestroy(e_in);
    }

    // HC_ICE_PACKED=0: stream the int32 tiles instead of the uint8 + overflow encoding (the reference path that the
    // tests compare the packed kernel against)
    bool packed = true;
    if (const char* e = getenv("HC_ICE_PACKED")) packed = atoi(e) != 0;
    // int32 kernel: 4 rows per warp step is the fastest per byte, but a warp item is at least RG rows; when the
    // batch is small (one large chromosome per GPU in the 8-way sharded run) fewer rows per item keep
    // every resident warp busy
    StreamVariant V = kQ8;
    if (!packed) {
        const int64_t warps = (int64_t)hc_num_sms() * 4 * 8;
        V = kVariants[nbins / 4 >= warps + warps / 4 ? 0 : (nbins / 2 >= warps + warps / 4 ? 1 : 2)];   // <4,2,4> | <2,2,4> | <1,4,4>
    }
    const int item_kb = 32;   // int32 kernel: bytes of matrix per work item, small enough that the last item is a short tail
    // packed kernel: an item is one strip x kseg k-tiles (of 32 columns): rows are split along K so that items stay
    // small (16 rows of chr1 are 100 KB) -- the per-segment partial row sums are added up by the update kernel
    int kseg = 48;
    if (packed) {       // small batches (one chromosome per GPU): shorter segments keep every resident warp busy
        const int64_t warps = (int64_t)hc_num_sms() * V.minb * 8;
        for (;;) {
            int64_t items = 0;
            for (int p = 0; p < nprob; ++p) items += (int64_t)((h_mat_n[p] + V.rg - 1) / V.rg) * (((h_mat_n[p] + 127) / 128 * 4 + kseg - 1) / kseg);
            if (items >= 4 * warps || kseg <= 16) break;
            kseg -= 16;
        }
    }

    // padded internal vectors: problem p owns [pad_off[p], pad_off[p] + ld_p), 128-byte aligned, so the
    // kernel can read the bias of any 4-column group with two aligned 16-byte loads and never
    // needs a column bound check (matrix padding columns are zero, padded bias entries are zero)
    // (the one wait of a call on the device: the leading dimensions exist only in device memory)
    std::vector<int32_t> h_ld(nprob);
    HC_CUDA(hc_read_small(h_ld.data(), mat_ld, sizeof(int32_t) * nprob, s));
    for (int p = 0; p < nprob; ++p) {
        if (h_ld[p] < h_mat_n[p] || (h_ld[p] & 127) != 0) {
            hc_set_error("hc_ice_dense_balance: ld must be >= n and a multiple of 128 elements (matrix %d: n=%d ld=%d)",
                         p, h_mat_n[p], h_ld[p]);
            return HC_ERR_ARG;
        }
    }
    // update kernel: the 8-CTA cluster version needs every chromosome to fit 8 x 256 x 4 padded columns
    bool cluster_update = packed;
    for (int p = 0; p < nprob; ++p) cluster_update = cluster_update && h_ld[p] <= UPD_CLUSTER * 256 * 4;
    // HC_ICE_TIME_KERNEL=1 (set by bench.py): the stream-kernel launch of the first iteration, in which every
    // chromosome is active, is bracketed by a pair of events (event-record nodes in the graph), so that its duration
    // can be read back separately from the update kernel and the launch gaps
    const bool timed = h_info != nullptr && getenv("HC_ICE_TIME_KERNEL") != nullptr && atoi(getenv("HC_ICE_TIME_KERNEL")) != 0;

    static thread_local IceDenseCache caches[64];
    IceDenseCache& C = caches[dev];
    if (!C.mbox) HC_CUDA(cudaHostAlloc(reinterpret_cast<void**>(&C.mbox), 2 * sizeof(long long), cudaHostAllocDefault));
    if (timed)
        for (auto& e : C.ev) if (e == nullptr) HC_CUDA(cudaEventCreate(&e));
    const bool hit = C.mem != nullptr && C.packed == (int)packed && C.nprob == nprob && C.kseg == kseg && C.fn == V.fn &&
                     C.cluster == (int)cluster_update && C.timed == (int)timed && C.kd == P->ignore_diags &&
                     C.max_iters == P->max_iters && C.tol == P->tol && C.mats == (packed ? nullptr : (const void*)mats) &&
                     C.mat_off == (packed ? nullptr : (const void*)mat_off) &&
                     std::equal(h_mat_n, h_mat_n + nprob, C.n.begin(), C.n.end()) && C.ld == h_ld;
    if (!hit) {
        // ---- a new launch shape: host tables, device buffers ---------------------------------------
        C.drop();
        std::vector<int64_t> h_pad(nprob + 1, 0);
        for (int p = 0; p < nprob; ++p) h_pad[p + 1] = h_pad[p] + h_ld[p];
        const int64_t npad = h_pad[nprob];
        int nseg_max = 1, kt_max = 0, nonempty = 0;
        for (int p = 0; p < nprob; ++p) {
            nseg_max = std::max(nseg_max, ((h_ld[p] >> 5) + kseg - 1) / kseg);
            kt_max = std::max(kt_max, h_ld[p] >> 5);
            nonempty += h_mat_n[p] > 0;
        }
        // work items, largest chromosomes first.  Packed: the descriptors of every item (4 x int4 each, see
        // ice_q8_mma_kernel); int32: row groups of ~item_kb KB, a multiple of RG rows each (chromosome, first row, rows).
        // The items of the chromosome at position i of `order` are [rng_lo[i], rng_hi[i]) of the full list; the live
        // list (item_prob ...) is the full list less the converged chromosomes, rewritten on the device.
        std::vector<int> order(nprob);
        for (int p = 0; p < nprob; ++p) order[p] = p;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return h_mat_n[a] > h_mat_n[b]; });
        std::vector<int4> item_desc;
        std::vector<int32_t> full_prob, full_row0, full_nrows, rng(3 * (size_t)nprob + 3 * (size_t)nprob, 0);
        std::vector<int64_t> h_q(2 * (size_t)nprob + 1, 0);     // q_off[nprob] | strip_off[nprob+1]
        int64_t qbytes = 0, strips = 0;
        for (int p = 0; p < nprob; ++p) {
            h_q[p] = qbytes;
            h_q[nprob + p] = strips;
            const int64_t sp = (h_mat_n[p] + 15) / 16;
            qbytes += sp * 16 * h_ld[p];
            strips += sp;
        }
        h_q[2 * (size_t)nprob] = strips;
        auto lohi = [](int64_t v, int& a, int& b) { a = (int)(uint32_t)(v & 0xffffffffll); b = (int)(v >> 32); };
        int64_t binoff = 0;
        std::vector<int64_t> h_binoff(nprob + 1, 0);
        for (int p = 0; p < nprob; ++p) { h_binoff[p] = binoff; binoff += h_mat_n[p]; }
        for (int i = 0; i < nprob; ++i) {
            const int p = order[i], n = h_mat_n[p];
            rng[i] = p;
            rng[nprob + i] = (int)full_prob.size();
            if (packed) {
                const int KT = h_ld[p] >> 5;
                for (int r0 = 0; r0 < n; r0 += V.rg)
                    for (int k0 = 0; k0 < KT; k0 += kseg) {
                        int4 d0, d1, d2, d3;
                        lohi(h_q[p] + ((int64_t)(r0 / 16) * KT + k0) * 512, d0.x, d0.y);
                        lohi((int64_t)(k0 / kseg) * npad + h_pad[p] + r0, d0.z, d0.w);
                        lohi(8 * h_pad[p] + (int64_t)k0 * 256, d1.x, d1.y);
                        lohi(h_binoff[p] + r0, d1.z, d1.w);
                        d2 = make_int4(p, (int)h_pad[p], r0, std::min(V.rg, n - r0));
                        d3 = make_int4(std::min(kseg, KT - k0), k0 / kseg, KT, 0);
                        item_desc.push_back(d0); item_desc.push_back(d1); item_desc.push_back(d2); item_desc.push_back(d3);
                        full_prob.push_back((int)full_prob.size()); full_row0.push_back(0); full_nrows.push_back(0);
                    }
            } else if (n > 0) {
                int rows = (int)((int64_t)item_kb * 1024 / ((int64_t)h_ld[p] * 4));
                rows = std::max(V.rg, rows / V.rg * V.rg);
                for (int r0 = 0; r0 < n; r0 += rows) {
                    full_prob.push_back(p); full_row0.push_back(r0); full_nrows.push_back(std::min(rows, n - r0));
                }
            }
            rng[2 * nprob + i] = (int)full_prob.size();
        }
        for (int p = 0; p < nprob; ++p) { rng[4 * nprob + p] = h_mat_n[p]; rng[5 * nprob + p] = h_ld[p]; }   // mat_n | mat_ld
        const size_t M = full_prob.size();
        const int grid = hc_num_sms() * V.minb;    // persistent: every resident slot filled exactly once
        const unsigned int queue_start = (unsigned)grid * 8u;
        // per-call state: live items (3 x M) | done[nprob] | n_done | queue | iter | nitems | upd_cnt | changed | abort
        const size_t st = 3 * M + (size_t)nprob;
        const size_t S = st + 7;
        std::vector<int32_t> h_state(S, 0);
        std::copy(full_prob.begin(), full_prob.end(), h_state.begin());
        std::copy(full_row0.begin(), full_row0.end(), h_state.begin() + M);
        std::copy(full_nrows.begin(), full_nrows.end(), h_state.begin() + 2 * M);
        h_state[st + 1] = (int32_t)queue_start;
        h_state[st + 3] = (int32_t)M;
        std::vector<hc_ice_result> h_res(nprob);      // empty problems never get work: their result stays this one
        for (int p = 0; p < nprob; ++p) { h_res[p].scale = NAN; h_res[p].var = 0.0; h_res[p].iters = 0; h_res[p].converged = 1; }

        size_t off = 0;
        auto take = [&](size_t bytes) { const size_t o = off; off = (off + bytes + 255) & ~(size_t)255; return o; };
        const size_t ptr_bytes = ((size_t)nbins + 1 + 2 * (size_t)nprob + 1 + (size_t)((nbins + 1023) / 1024) + 1) * sizeof(int64_t);
        const size_t o_vec = take((2 * (size_t)npad + nprob + 1) * sizeof(double));     // bias | marg | pad_off (int64)
        const size_t o_q8 = take(packed ? (size_t)qbytes + 8 * (size_t)npad * (1 + (size_t)nseg_max) + 16 : 0);   // tiles | digits | part
        // ptr[nbins+1] | q_off[nprob] | strip_off[nprob+1] | bsum | lo[nbins] hi[nbins] exp[nprob] (int32)
        const size_t o_ptr = take(packed ? ptr_bytes + (2 * (size_t)nbins + nprob) * sizeof(int32_t) : 0);
        const size_t o_state = take(S * sizeof(int32_t));
        const size_t o_pristine = take(S * sizeof(int32_t));
        const size_t o_tab = take(rng.size() * sizeof(int32_t));
        const size_t o_desc = take(item_desc.size() * sizeof(int4));
        const size_t o_res = take((size_t)nprob * sizeof(hc_ice_result));
        HC_CUDA(cudaMalloc(reinterpret_cast<void**>(&C.mem), off));
        unsigned char* m = C.mem;
        IceDenseArgs A = {};
        A.bias = reinterpret_cast<double*>(m + o_vec);
        A.marg = A.bias + npad;
        int64_t* d_pad = reinterpret_cast<int64_t*>(A.bias + 2 * npad);
        A.pad_off = d_pad;
        C.state = reinterpret_cast<int32_t*>(m + o_state);
        C.pristine = reinterpret_cast<const int32_t*>(m + o_pristine);
        C.state_ints = S;
        int32_t* tab = reinterpret_cast<int32_t*>(m + o_tab);
        A.mats = packed ? nullptr : mats; A.mat_off = packed ? nullptr : mat_off;
        A.mat_n = tab + 4 * nprob; A.mat_ld = tab + 5 * nprob;
        A.item_prob = C.state; A.item_row0 = C.state + M; A.item_nrows = C.state + 2 * M;
        A.done = C.state + 3 * M;
        A.n_done = C.state + st;
        A.queue = reinterpret_cast<unsigned int*>(C.state + st + 1);
        A.iter = C.state + st + 2;
        A.nitems = reinterpret_cast<const unsigned int*>(C.state + st + 3);
        A.upd_cnt = reinterpret_cast<unsigned int*>(C.state + st + 4);
        A.changed = C.state + st + 5;
        C.abort_flag = C.state + st + 6;
        A.results = reinterpret_cast<hc_ice_result*>(m + o_res);
        A.tol = P->tol; A.kd = P->ignore_diags; A.max_iters = P->max_iters; A.nprob = nprob; A.queue_start = queue_start;
        A.packed = packed ? 1 : 0; A.kseg = kseg; A.nseg_max = nseg_max; A.npad = npad;
        A.nonempty = nonempty;
        A.rng = tab; A.rng_off = tab + 3 * nprob;
        A.full_row0 = C.pristine + M; A.full_nrows = C.pristine + 2 * M;
        A.loop_end = 1;
        if (packed) {
            uint8_t* q8 = m + o_q8;
            A.q8 = q8;
            A.digits = q8 + ((qbytes + 15) & ~15ll);
            A.part = reinterpret_cast<double*>(A.digits + 8 * (size_t)npad);
            C.ovf_ptr = reinterpret_cast<int64_t*>(m + o_ptr);
            C.qoff = C.ovf_ptr + nbins + 1;
            C.strip = C.qoff + nprob;
            C.lo = reinterpret_cast<int32_t*>(m + o_ptr + ptr_bytes);
            C.hi = C.lo + nbins;
            A.dig_exp = C.hi + nbins;
            A.q_off = C.qoff;
            A.ovf_ptr = C.ovf_ptr;
            A.desc = reinterpret_cast<const int4*>(m + o_desc);
            HC_CUDA(cudaMemcpyAsync(C.qoff, h_q.data(), h_q.size() * sizeof(int64_t), cudaMemcpyHostToDevice, s));
            HC_CUDA(cudaMemcpyAsync(m + o_desc, item_desc.data(), item_desc.size() * sizeof(int4), cudaMemcpyHostToDevice, s));
        }
        HC_CUDA(cudaMemcpyAsync(d_pad, h_pad.data(), (nprob + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        HC_CUDA(cudaMemcpyAsync(m + o_pristine, h_state.data(), S * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        HC_CUDA(cudaMemcpyAsync(tab, rng.data(), rng.size() * sizeof(int32_t), cudaMemcpyHostToDevice, s));
        HC_CUDA(cudaMemcpyAsync(A.results, h_res.data(), h_res.size() * sizeof(hc_ice_result), cudaMemcpyHostToDevice, s));
        HC_CUDA(cudaStreamSynchronize(s));      // the host tables go out of scope
        C.A = A;
        C.packed = packed; C.nprob = nprob; C.kseg = kseg; C.fn = V.fn; C.cluster = cluster_update; C.timed = timed;
        C.kd = P->ignore_diags; C.max_iters = P->max_iters; C.tol = P->tol;
        C.mats = A.mats; C.mat_off = A.mat_off;
        C.n.assign(h_mat_n, h_mat_n + nprob); C.ld = h_ld;
        C.nbins = nbins; C.strips = strips; C.kt_max = kt_max; C.grid = grid;
    }
    IceDenseArgs& A = C.A;
    if (packed && C.ovf == nullptr) {
        C.ovf_cap = std::max(4 * (long long)nbins, 1024ll);
        HC_CUDA(cudaMalloc(reinterpret_cast<void**>(&C.ovf), 2 * (size_t)C.ovf_cap * sizeof(int32_t)));
    }
    A.ovf_col = C.ovf; A.ovf_val = C.ovf ? C.ovf + C.ovf_cap : nullptr;
    // the bias vector (its byte planes for the packed kernel) is the only data that should live in L1
    cudaFuncSetAttribute(V.fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    auto launch_update = [&]() {
        if (C.cluster) ice_q8_update_cluster_kernel<<<nprob * UPD_CLUSTER, 256, 0, s>>>(A);
        else ice_dense_update_kernel<<<nprob, 1024, 0, s>>>(A);
    };
    // The loop as one graph: the first iteration (all chromosomes active; its stream launch bracketed by the timing
    // events), then a WHILE node whose body is ICE_BODY_ITERS iterations.  The condition is set by the last CTA of the
    // update launch that ends the first iteration and each body (ice_iteration_end, which also compacts the work list),
    // so the loop needs no host poll; iterations past the last convergence in a body find every chromosome done (about
    // 5 us each).  Measured on B200 (C2, 86 iterations): a body of one iteration costs ~2 us more per iteration than 4
    // or 8 (loop 5.61 ms against 5.47 / 5.44 ms).
    constexpr int ICE_BODY_ITERS = 4;
    auto build_graph = [&]() -> cudaError_t {
        cudaGraph_t g = nullptr;
        cudaError_t e = cudaGraphCreate(&g, 0);
        cudaGraphConditionalHandle h = 0;
        if (e == cudaSuccess) e = cudaGraphConditionalHandleCreate(&h, g, 1, cudaGraphCondAssignDefault);
        IceDenseArgs GA = A, GB = A;          // GB: the update launches inside a body that do not end it
        GA.cond = GB.cond = h; GA.has_cond = GB.has_cond = 1; GA.loop_end = 1; GB.loop_end = 0;
        void* args[1] = {&GA};
        void* args_mid[1] = {&GB};
        cudaKernelNodeParams ks = {}, ku = {};
        ks.func = reinterpret_cast<void*>(C.fn); ks.gridDim = dim3(C.grid); ks.blockDim = dim3(256); ks.kernelParams = args;
        ku.func = C.cluster ? reinterpret_cast<void*>(ice_q8_update_cluster_kernel) : reinterpret_cast<void*>(ice_dense_update_kernel);
        ku.gridDim = dim3(C.cluster ? nprob * UPD_CLUSTER : nprob); ku.blockDim = dim3(C.cluster ? 256 : 1024); ku.kernelParams = args;
        cudaKernelNodeParams ku_mid = ku;
        ku_mid.kernelParams = args_mid;
        cudaGraphNode_t prev = nullptr, node = nullptr;
        if (e == cudaSuccess && C.timed) { e = cudaGraphAddEventRecordNode(&node, g, nullptr, 0, C.ev[0]); prev = node; }
        if (e == cudaSuccess) { e = cudaGraphAddKernelNode(&node, g, prev ? &prev : nullptr, prev ? 1 : 0, &ks); prev = node; }
        if (e == cudaSuccess && C.timed) { e = cudaGraphAddEventRecordNode(&node, g, &prev, 1, C.ev[1]); prev = node; }
        if (e == cudaSuccess) { e = cudaGraphAddKernelNode(&node, g, &prev, 1, &ku); prev = node; }
        cudaGraphNodeParams cp = {};
        cp.type = cudaGraphNodeTypeConditional;
        cp.conditional.handle = h; cp.conditional.type = cudaGraphCondTypeWhile; cp.conditional.size = 1;
        if (e == cudaSuccess) e = cudaGraphAddNode(&node, g, &prev, 1, &cp);
        if (e == cudaSuccess) {
            cudaGraph_t body = cp.conditional.phGraph_out[0];
            cudaGraphNode_t bs = nullptr, bp = nullptr;
            for (int u = 0; u < ICE_BODY_ITERS && e == cudaSuccess; ++u) {
                e = cudaGraphAddKernelNode(&bs, body, bp ? &bp : nullptr, bp ? 1 : 0, &ks);
                if (e == cudaSuccess) e = cudaGraphAddKernelNode(&bp, body, &bs, 1, u + 1 < ICE_BODY_ITERS ? &ku_mid : &ku);
            }
        }
        if (e == cudaSuccess) e = cudaGraphInstantiate(&C.exec, g, 0);
        if (e != cudaSuccess) { if (g) cudaGraphDestroy(g); C.exec = nullptr; (void)cudaGetLastError(); return e; }
        C.graph = g;
        return cudaSuccess;
    };

    float loop_ms = 0.f, pack_ms = 0.f, stream_ms = 0.f;
    int iters = 0;
    long long novf = 0;
    for (;;) {      // twice only when the overflow cells outgrow their arrays
        HC_CUDA(cudaMemcpyAsync(C.state, C.pristine, C.state_ints * sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
        HC_CUDA(cudaMemsetAsync(A.bias, 0, 2 * (size_t)A.npad * sizeof(double), s));
        ice_pad_bias_kernel<<<(unsigned)((nbins + 255) / 256), 256, 0, s>>>(bin_off, A.pad_off, nprob, bias, A.bias);
        HC_LAUNCH_CHECK();

        // ---- packed encoding of the tiles (once per call) ------------------------------------------
        EventPair evp;
        if (packed) {
            if (h_info) { evp.create(); cudaEventRecord(evp.a, s); }
            HC_CUDA(cudaMemsetAsync(C.ovf_ptr, 0, ((size_t)nbins + 1) * sizeof(int64_t), s));
            HC_CUDA(cudaMemsetAsync(C.lo, 0x7f, (size_t)nbins * sizeof(int32_t), s));
            HC_CUDA(cudaMemsetAsync(C.hi, 0xff, (size_t)nbins * sizeof(int32_t), s));
            ice_pack_tiles_kernel<<<dim3((unsigned)((C.strips * 32 + 255) / 256), (unsigned)((C.kt_max + 7) / 8)), 256, 0, s>>>(
                mats, mat_off, mat_n, mat_ld, C.qoff, C.strip, bin_off, nprob, P->ignore_diags, const_cast<uint8_t*>(A.q8),
                reinterpret_cast<unsigned long long*>(C.ovf_ptr), C.lo, C.hi);
            HC_LAUNCH_CHECK();
            const int nb = (int)((nbins + 1023) / 1024);
            int64_t* d_bsum = C.strip + nprob + 1;       // nb + 1 entries behind the strip table
            ice_ovf_blocksum_kernel<<<nb, 256, 0, s>>>(C.ovf_ptr, nbins, d_bsum);
            HC_LAUNCH_CHECK();
            ice_ovf_scan_blocks_kernel<<<1, 1024, 0, s>>>(d_bsum, nb);
            HC_LAUNCH_CHECK();
            ice_ovf_scan_kernel<<<nb, 256, 0, s>>>(C.ovf_ptr, nbins, d_bsum, nb);
            HC_LAUNCH_CHECK();
            ice_pack_ovf_kernel<<<(unsigned)((nbins * 32 + 255) / 256), 256, 0, s>>>(
                mats, mat_off, mat_n, mat_ld, bin_off, nprob, P->ignore_diags, C.ovf_ptr, C.lo, C.hi,
                const_cast<int32_t*>(A.ovf_col), const_cast<int32_t*>(A.ovf_val), C.ovf_cap, A, C.abort_flag);
            HC_LAUNCH_CHECK();
            ice_digits_kernel<<<nprob, 1024, 0, s>>>(A);      // byte planes of the initial bias
            HC_LAUNCH_CHECK();
            if (evp.a) cudaEventRecord(evp.b, s);
        }

        if (!C.exec && build_graph() != cudaSuccess) C.exec = nullptr;   // plain launches below
        EventPair evl;                              // device time of the iteration loop, for the roofline
        if (h_info) { evl.create(); cudaEventRecord(evl.a, s); }
        cudaError_t e = cudaSuccess;
        if (C.exec) e = cudaGraphLaunch(C.exec, s);
        else {
            // without the graph: launch pairs, the host polls the done counter every `poll` iterations
            const int poll = P->poll_every > 0 ? P->poll_every : 8;
            for (int k0 = 0; k0 < P->max_iters && e == cudaSuccess; k0 += poll) {
                for (int i = 0; i < poll; ++i) {
                    if (k0 + i == 0 && C.timed) cudaEventRecord(C.ev[0], s);
                    C.fn<<<C.grid, 256, 0, s>>>(A);
                    if (k0 + i == 0 && C.timed) cudaEventRecord(C.ev[1], s);
                    launch_update();
                }
                int32_t nd = 0;
                e = hc_read_small(&nd, A.n_done, sizeof(int32_t), s);   // not a memcpy: see hc_read_small
                if (e == cudaSuccess && nd >= A.nonempty) break;
            }
        }
        if (evl.a) cudaEventRecord(evl.b, s);
        if (e == cudaSuccess) {
            ice_finalize_kernel<<<(unsigned)((nbins + 255) / 256), 256, 0, s>>>(bin_off, A.pad_off, nprob, A.results,
                                                                               P->rescale_marginals, A.bias, bias, C.abort_flag);
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaMemcpyAsync(results, A.results, (size_t)nprob * sizeof(hc_ice_result), cudaMemcpyDeviceToDevice, s);
        if (e == cudaSuccess && packed) e = cudaMemcpyAsync(C.mbox, C.ovf_ptr + nbins, sizeof(long long), cudaMemcpyDeviceToHost, s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(C.mbox + 1, A.iter, sizeof(int32_t), cudaMemcpyDeviceToHost, s);
        const cudaError_t es = cudaStreamSynchronize(s);
        if (e == cudaSuccess) e = es;
        if (e != cudaSuccess) { hc_set_error("hc_ice_dense_balance: %s", cudaGetErrorString(e)); return HC_ERR_CUDA; }
        iters = *reinterpret_cast<const int32_t*>(C.mbox + 1);
        novf = packed ? C.mbox[0] : 0;
        hc_count_launch(2 * iters + 1);
        if (h_info) {
            cudaEventElapsedTime(&loop_ms, evl.a, evl.b);
            if (evp.a) cudaEventElapsedTime(&pack_ms, evp.a, evp.b);
            if (C.timed && cudaEventElapsedTime(&stream_ms, C.ev[0], C.ev[1]) != cudaSuccess) { stream_ms = 0.f; (void)cudaGetLastError(); }
        }
        if (novf <= C.ovf_cap) break;
        // the overflow arrays were too small: nothing was streamed and the caller's bias is untouched; grow, run again
        cudaFree(C.ovf);
        C.ovf = nullptr;
        C.ovf_cap = novf + novf / 4;
        HC_CUDA(cudaMalloc(reinterpret_cast<void**>(&C.ovf), 2 * (size_t)C.ovf_cap * sizeof(int32_t)));
        A.ovf_col = C.ovf; A.ovf_val = C.ovf + C.ovf_cap;
        C.drop_graph();     // its kernel nodes hold the old pointers
    }
    if (h_info) {
        h_info->launches = 2 * iters + 1;
        h_info->loop_ms = loop_ms;
        h_info->packed = packed ? 1 : 0;
        h_info->overflow_cells = novf;
        h_info->stream_full_launches = stream_ms > 0.f ? 1 : 0;
        h_info->stream_full_ms = stream_ms;
        h_info->pack_ms = pack_ms;
    }
    return HC_OK;
}
