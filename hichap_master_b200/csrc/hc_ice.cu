// (b) ICE balancing on dense symmetric int32 tiles  ==  `cooler balance --ignore-diags K [--cis-only]`
// (HiCHap call sites: matrixBuilding.py:708, :713, :1537, :1542, :1761, :1766; algorithm restated
// in oracle/cooler_ice.py from cooler.balance.balance_cooler).
//
// One iteration of EVERY problem (chromosome) of the batch = two launches:
//   stream kernel: persistent warps draw row-group work items from a global queue and compute
//       marg[r] = b[r] * sum_j w(r,j) A[r][j] b[j]   (fp64, warp-shuffle reduction, one store per row);
//   update kernel (one CTA per chromosome): mean / variance of the fresh marginals over the non-zero bins,
//       b <- b / (marg / mean), convergence test var < tol, bookkeeping -- all on the device.
// `poll` iterations are captured once as a CUDA graph and replayed; nothing goes back to the host inside
// the loop except a done-counter poll through a pinned mailbox.
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
__global__ void __launch_bounds__(256)
ice_dense_marginals_kernel(const int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off,
                           const int32_t* __restrict__ mat_n, const int32_t* __restrict__ mat_ld,
                           const int64_t* __restrict__ bin_off, int nprob, int kd,
                           double* __restrict__ nnz_marg, double* __restrict__ marg) {
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;  // global bin == one warp
    const int lane = threadIdx.x & 31;
    if (g >= bin_off[nprob]) return;
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
    const int64_t* bin_off;
    const int64_t* ovf_ptr; const int32_t* ovf_col; const int32_t* ovf_val;   // per global row: cells with w*count > 255
    int packed;
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
                    int32_t* __restrict__ ovf_col, int32_t* __restrict__ ovf_val) {
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
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
// warps, global queue of row-group items; a row group is RS strips of 16 rows).  Per k-tile a lane issues RS
// 128-bit streaming loads (its A fragments), one 64-bit load of the bias planes (B fragment, through L1) and RS
// MMAs; U k-tiles are in flight.  C fragment: lane l holds, for rows g and g + 8 (g = l / 4), the int32 sums of
// planes 2 * (l % 4) and 2 * (l % 4) + 1 -- folded into fp64 with the planes' weights, reduced over the 4 lanes
// of the group, scaled by 2^(E - 64), plus the row's overflow cells in fp64.
template <int RS, int U, int MINB>
__global__ void __launch_bounds__(256, MINB)
ice_q8_mma_kernel(IceDenseArgs A) {
    const int lane = threadIdx.x & 31;
    const int g = lane >> 2, t4 = lane & 3;
    // weights of this lane's two planes: 2^(8 * (7 - plane)), exact
    const double w_even = __longlong_as_double((long long)(1023 + 8 * (7 - 2 * t4)) << 52);
    const double w_odd = __longlong_as_double((long long)(1023 + 8 * (6 - 2 * t4)) << 52);
    const unsigned nitems = *A.nitems;
    // An item = one row group (RS strips) x one K segment, described by 4 x int4 the host precomputed:
    //   d0 = tile byte offset (int64) | index of the item's first partial sum (int64)
    //   d1 = byte offset of the segment's bias planes (int64) | global row of the first row (int64)
    //   d2 = chromosome, offset of the chromosome in the padded vectors, (unused), rows
    //   d3 = k-tiles in the segment, segment index, k-tiles per strip, (unused)
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
            const int nrows = d2.w, nk = d3.x, seg = d3.y, KT = d3.z;
            const uint8_t* qp = A.q8 + tile_off + 16 * lane;
            const uint8_t* dig = A.digits + dig_off + 8 * lane;
            const double* __restrict__ b = A.bias + d2.y;
            const double scale = __longlong_as_double((long long)(1023 + A.dig_exp[p] - 64) << 52);   // 2^(E - 64)
            double* pout = A.part + part_base;
            const int ns = min(RS, (nrows + 15) >> 4);      // strips that exist
            const uint8_t* sp[RS];
#pragma unroll
            for (int s = 0; s < RS; ++s) sp[s] = qp + (int64_t)min(s, ns - 1) * KT * 512;
            int c[RS][4];
#pragma unroll
            for (int s = 0; s < RS; ++s) { c[s][0] = 0; c[s][1] = 0; c[s][2] = 0; c[s][3] = 0; }
            for (int t = 0; t < nk; t += U) {       // nk <= 1024: the int32 plane sums cannot overflow
                int4 a[U][RS];
                uint2 bf[U];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const int tt = min(t + u, nk - 1);
#pragma unroll
                    for (int s = 0; s < RS; ++s)
                        a[u][s] = ld_stream_v4(reinterpret_cast<const int32_t*>(sp[s] + (int64_t)tt * 512));
                    bf[u] = t + u < nk ? *reinterpret_cast<const uint2*>(dig + (int64_t)tt * 256) : make_uint2(0u, 0u);
                }
#pragma unroll
                for (int u = 0; u < U; ++u)
#pragma unroll
                    for (int s = 0; s < RS; ++s) mma_u8(c[s], a[u][s], bf[u]);
            }
#pragma unroll
            for (int s = 0; s < RS; ++s) {
                if (s < ns) {       // warp-uniform
                    const int ra = 16 * s + g, rb = ra + 8;
                    double va = ((double)c[s][0] * w_even + (double)c[s][1] * w_odd) * scale;
                    double vb = ((double)c[s][2] * w_even + (double)c[s][3] * w_odd) * scale;
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
            }
        }
        cur = nxt; d0 = e0; d1 = e1; d2 = e2; d3 = e3;
        nxt = __shfl_sync(0xffffffffu, drawn, 0);
    }
}

// Vector half of an iteration (grid = one CTA per chromosome): mean / variance of the fresh
// marginals over the non-zero bins, bias update b /= marg/mean (in place), convergence test,
// scale / iteration bookkeeping -- all on the device.
__global__ void __launch_bounds__(1024)
ice_dense_update_kernel(IceDenseArgs A) {
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
                A.results[p] = r; A.done[p] = 1; atomicAdd(A.n_done, 1);
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
            if (var < A.tol || k >= A.max_iters) { A.done[p] = 1; atomicAdd(A.n_done, 1); }
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
            A.results[p] = r; A.done[p] = 1; atomicAdd(A.n_done, 1);
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
        if (var < A.tol || k >= A.max_iters) { A.done[p] = 1; atomicAdd(A.n_done, 1); }
    }
    if (A.packed) {      // the stream kernel reads the bias as byte planes
        __syncthreads();
        ice_write_digits(bw, n, A.mat_ld[p], A.digits + 8 * lo, A.dig_exp + p, red);
    }
}

// The same update for the packed encoding when every chromosome has at most 8192 padded columns: a thread-block
// CLUSTER of 8 CTAs x 256 threads per chromosome, 4 consecutive columns per thread, everything in registers,
// the three chromosome-wide reductions (sum / count, variance, max) through distributed shared memory.  The
// single-CTA kernel above spends ~25 us per iteration on this (latency: six block barriers, 16 fp64 divisions and
// 450 KB through one SM); that is a third of an iteration once the matrix pass takes ~50 us.
constexpr int UPD_CLUSTER = 8;
__global__ void __cluster_dims__(UPD_CLUSTER, 1, 1) __launch_bounds__(256)
ice_q8_update_cluster_kernel(IceDenseArgs A) {
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
            A.results[p] = r; A.done[p] = 1; atomicAdd(A.n_done, 1);
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
        if (var < A.tol || k >= A.max_iters) { A.done[p] = 1; atomicAdd(A.n_done, 1); }
    }
    cluster.sync();          // keep every CTA's shared memory alive until the remote reads are done
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
                    double* __restrict__ bias) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= bin_off[nprob]) return;
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

// stream-ordered scratch and timing events of one balancing call, released on every exit path
struct Scratch {
    cudaStream_t s;
    std::vector<void*> ptrs;
    explicit Scratch(cudaStream_t st) : s(st) {}
    cudaError_t alloc(void** p, size_t bytes) {
        const cudaError_t e = cudaMallocAsync(p, bytes, s);
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
    ~Scratch() { for (void* p : ptrs) cudaFreeAsync(p, s); }
};
struct EventPair {
    cudaEvent_t a = nullptr, b = nullptr;
    void create() { cudaEventCreate(&a); cudaEventCreate(&b); }
    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
};

typedef void (*StreamKernel)(IceDenseArgs);
struct StreamVariant { StreamKernel fn; int rg, u, minb; };
// tuned on B200 (profiles/): RG rows share the bias loads; RG*U 128-bit loads in flight per lane
const StreamVariant kVariants[] = {
    {ice_dense_stream_kernel<4, 2, 4>, 4, 2, 4},   // default: 5.5 TB/s on C2 (profiles/r1c_ice_variants_v3.log)
    {ice_dense_stream_kernel<4, 2, 3>, 4, 2, 3},
    {ice_dense_stream_kernel<2, 2, 4>, 2, 2, 4},
    {ice_dense_stream_kernel<2, 4, 3>, 2, 4, 3},
    {ice_dense_stream_kernel<4, 4, 2>, 4, 4, 2},
    {ice_dense_stream_kernel<1, 4, 4>, 1, 4, 4},
};

// packed kernel: <RS strips of 16 rows per step, U k-tiles in flight, CTAs per SM>; .rg = rows per step
const StreamVariant kQ8Variants[] = {
    {ice_q8_mma_kernel<2, 4, 4>, 32, 4, 4},
    {ice_q8_mma_kernel<1, 4, 4>, 16, 4, 4},
    {ice_q8_mma_kernel<1, 8, 3>, 16, 8, 3},
    {ice_q8_mma_kernel<2, 4, 3>, 32, 4, 3},
    {ice_q8_mma_kernel<1, 8, 4>, 16, 8, 4},
    {ice_q8_mma_kernel<2, 8, 2>, 32, 8, 2},
    {ice_q8_mma_kernel<1, 16, 2>, 16, 16, 2},
    {ice_q8_mma_kernel<1, 12, 3>, 16, 12, 3},
};

}  // namespace

extern "C" int hc_ice_dense_marginals(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                      const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                                      int32_t ignore_diags, double* nnz_marg, double* marg, void* stream) {
    HC_REQUIRE(nprob > 0 && ignore_diags >= 0, "nprob>0, ignore_diags>=0");
    int64_t total = 0;
    HC_CUDA(hc_read_small(&total, bin_off + nprob, sizeof(int64_t), (cudaStream_t)stream));
    if (total == 0) return HC_OK;
    const int64_t blocks = (total * 32 + 255) / 256;
    ice_dense_marginals_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
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
    // The iteration loop is replayed as a CUDA graph, which cannot be captured on the legacy default
    // stream: run on a private stream ordered after the caller's stream (the call synchronises
    // before returning, so the caller's later work is ordered after it).
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

    // variant: 4 rows per warp step is the fastest per byte, but a warp item is at least RG rows; when the
    // batch is small (one large chromosome per GPU in the 8-way sharded run) fewer rows per item keep
    // every resident warp busy.  HC_ICE_VARIANT overrides (tuning).
    // HC_ICE_PACKED=0: stream the int32 tiles instead of the uint8 + overflow encoding
    bool packed = true;
    if (const char* e = getenv("HC_ICE_PACKED")) packed = atoi(e) != 0;
    int64_t total_rows = 0;
    for (int p = 0; p < nprob; ++p) total_rows += h_mat_n[p];
    StreamVariant V;
    if (packed) {
        int vi = -1;
        if (const char* e = getenv("HC_ICE_Q8_VARIANT")) vi = atoi(e);
        if (vi < 0 || vi >= (int)(sizeof(kQ8Variants) / sizeof(kQ8Variants[0]))) vi = 6;   // <1,16,2>: 16 warps/SM, 16 tiles in flight per lane
        V = kQ8Variants[vi];
    } else {
        int vi = -1;
        if (const char* e = getenv("HC_ICE_VARIANT")) vi = atoi(e);
        if (vi < 0 || vi >= (int)(sizeof(kVariants) / sizeof(kVariants[0]))) {
            const int64_t warps = (int64_t)hc_num_sms() * 4 * 8;
            vi = total_rows / 4 >= warps + warps / 4 ? 0 : (total_rows / 2 >= warps + warps / 4 ? 2 : 5);   // <4,2,4> | <2,2,4> | <1,4,4>
        }
        V = kVariants[vi];
    }
    int item_kb = 32;   // int32 kernel: bytes of matrix per work item, small enough that the last item is a short tail
    if (const char* e = getenv("HC_ICE_ITEM_KB")) item_kb = std::max(1, atoi(e));
    // packed kernel: an item is V.rg rows x kseg k-tiles (of 32 columns): rows are split along K so that items stay
    // small (16 rows of chr1 are 100 KB) -- the per-segment partial row sums are added up by the update kernel
    int kseg = 48;
    if (const char* e = getenv("HC_ICE_KSEG")) kseg = std::min(1024, std::max(4, atoi(e) / 4 * 4));
    else if (packed) {       // small batches (one chromosome per GPU): shorter segments keep every resident warp busy
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
    std::vector<int32_t> h_ld(nprob);
    HC_CUDA(hc_read_small(h_ld.data(), mat_ld, sizeof(int32_t) * nprob, s));
    std::vector<int64_t> h_pad(nprob + 1, 0);
    for (int p = 0; p < nprob; ++p) {
        if (h_ld[p] < h_mat_n[p] || (h_ld[p] & 127) != 0) {
            hc_set_error("hc_ice_dense_balance: ld must be >= n and a multiple of 128 elements (matrix %d: n=%d ld=%d)",
                         p, h_mat_n[p], h_ld[p]);
            return HC_ERR_ARG;
        }
        h_pad[p + 1] = h_pad[p] + h_ld[p];
    }
    const int64_t npad = h_pad[nprob];

    // ---- work items: RG-aligned row groups of ~item_kb KB, largest chromosomes first -----------
    std::vector<int32_t> h_done(nprob, 0);
    std::vector<int32_t> item_prob, item_row0, item_nrows;
    std::vector<int4> item_desc;       // packed kernel: 4 per item, built once
    bool desc_built = false;
    std::vector<int> desc_lo(nprob, 0), desc_hi(nprob, 0);
    std::vector<int64_t> h_qoff(nprob, 0), h_binoff(nprob + 1, 0);
    if (packed) {
        int64_t qb = 0;
        for (int p = 0; p < nprob; ++p) {
            h_qoff[p] = qb;
            qb += (int64_t)((h_mat_n[p] + 15) / 16) * 16 * h_ld[p];
            h_binoff[p + 1] = h_binoff[p] + h_mat_n[p];
        }
    }
    int nseg_max = 1;
    for (int p = 0; p < nprob; ++p) nseg_max = std::max(nseg_max, ((h_ld[p] >> 5) + kseg - 1) / kseg);
    auto build_items = [&]() {
        item_prob.clear(); item_row0.clear(); item_nrows.clear();
        std::vector<int> order(nprob);
        for (int p = 0; p < nprob; ++p) order[p] = p;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return h_mat_n[a] > h_mat_n[b]; });
        for (int p : order) {
            const int n = h_mat_n[p];
            if (n == 0 || h_done[p]) continue;
            if (packed) {
                const int KT = h_ld[p] >> 5;
                auto lohi = [](int64_t v, int& a, int& b) { a = (int)(uint32_t)(v & 0xffffffffll); b = (int)(v >> 32); };
                if (desc_built) {      // later builds: only the list of live item ids changes
                    for (int id = desc_lo[p]; id < desc_hi[p]; ++id) { item_prob.push_back(id); item_row0.push_back(0); item_nrows.push_back(0); }
                    continue;
                }
                for (int r0 = 0; r0 < n; r0 += V.rg)
                    for (int k0 = 0; k0 < KT; k0 += kseg) {
                        item_prob.push_back((int)(item_desc.size() / 4)); item_row0.push_back(r0); item_nrows.push_back(std::min(V.rg, n - r0));
                        int4 d0, d1, d2, d3;
                        lohi(h_qoff[p] + ((int64_t)(r0 / 16) * KT + k0) * 512, d0.x, d0.y);
                        lohi((int64_t)(k0 / kseg) * npad + h_pad[p] + r0, d0.z, d0.w);
                        lohi(8 * h_pad[p] + (int64_t)k0 * 256, d1.x, d1.y);
                        lohi(h_binoff[p] + r0, d1.z, d1.w);
                        d2 = make_int4(p, (int)h_pad[p], r0, std::min(V.rg, n - r0));
                        d3 = make_int4(std::min(kseg, KT - k0), k0 / kseg, KT, 0);
                        item_desc.push_back(d0); item_desc.push_back(d1); item_desc.push_back(d2); item_desc.push_back(d3);
                    }
                continue;
            }
            int rows = (int)((int64_t)item_kb * 1024 / ((int64_t)h_ld[p] * 4));
            rows = std::max(V.rg, rows / V.rg * V.rg);
            for (int r0 = 0; r0 < n; r0 += rows) {
                item_prob.push_back(p); item_row0.push_back(r0); item_nrows.push_back(std::min(rows, n - r0));
            }
        }
    };
    build_items();
    const size_t max_items = item_prob.size();
    if (packed) {       // descriptor ids are positions in build order: remember each chromosome's id range
        desc_built = true;
        std::vector<int> cnt(nprob, 0);
        for (size_t i = 0; i < item_desc.size(); i += 4) cnt[item_desc[i + 2].x]++;
        // build order = chromosomes by decreasing size; ids are contiguous per chromosome in that order
        std::vector<int> order(nprob);
        for (int p = 0; p < nprob; ++p) order[p] = p;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return h_mat_n[a] > h_mat_n[b]; });
        int run = 0;
        for (int p : order) { desc_lo[p] = run; run += cnt[p]; desc_hi[p] = run; }
    }

    Scratch scratch(s);
    double* d_vec = nullptr;     // [npad] bias | [npad] marg | [nprob+1] pad_off (as int64)
    HC_CUDA(scratch.alloc((void**)&d_vec, (2 * (size_t)npad + nprob + 1) * sizeof(double)));
    double* biasp = d_vec;
    double* marg = d_vec + npad;
    int64_t* d_pad = reinterpret_cast<int64_t*>(d_vec + 2 * npad);
    HC_CUDA(cudaMemsetAsync(d_vec, 0, 2 * (size_t)npad * sizeof(double), s));
    HC_CUDA(cudaMemcpyAsync(d_pad, h_pad.data(), (nprob + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    ice_pad_bias_kernel<<<(unsigned)((nbins + 255) / 256), 256, 0, s>>>(bin_off, d_pad, nprob, bias, biasp);
    HC_LAUNCH_CHECK();

    // ---- packed encoding of the tiles (once per call) ------------------------------------------
    uint8_t* d_q8 = nullptr;           // tiles | digits (8 B per padded column) behind them
    int64_t* d_ovf_ptr = nullptr;      // [nbins+1] ptr | q_off[nprob] | strip_off[nprob+1] | lo[nbins] hi[nbins] exp[nprob] (int32)
    int32_t* d_ovf = nullptr;          // col[novf] | val[novf]
    uint8_t* d_digits = nullptr;
    double* d_part = nullptr;          // [npad][nseg_max] partial row sums
    int64_t* d_qoff = nullptr;
    int32_t* d_exp = nullptr;
    long long novf = 0;
    EventPair evp;
    cudaEvent_t& evp0 = evp.a;
    cudaEvent_t& evp1 = evp.b;
    if (packed) {
        if (h_info) { evp.create(); cudaEventRecord(evp0, s); }
        std::vector<int64_t> h_q(2 * (size_t)nprob + 1);     // q_off[nprob] | strip_off[nprob+1]
        int64_t qbytes = 0, strips = 0;
        for (int p = 0; p < nprob; ++p) {
            h_q[p] = qbytes;
            h_q[nprob + p] = strips;
            const int64_t sp = (h_mat_n[p] + 15) / 16;
            qbytes += sp * 16 * h_ld[p];
            strips += sp;
        }
        h_q[2 * (size_t)nprob] = strips;
        HC_CUDA(scratch.alloc((void**)&d_q8, (size_t)qbytes + 8 * (size_t)npad * (1 + (size_t)nseg_max) + 16));
        d_digits = d_q8 + ((qbytes + 15) & ~15ll);
        d_part = reinterpret_cast<double*>(d_digits + 8 * (size_t)npad);
        const size_t ptr_bytes = ((size_t)nbins + 1 + 2 * (size_t)nprob + 1 + (size_t)((nbins + 1023) / 1024) + 1) * sizeof(int64_t);
        HC_CUDA(scratch.alloc((void**)&d_ovf_ptr, ptr_bytes + (2 * (size_t)nbins + nprob) * sizeof(int32_t)));
        d_qoff = d_ovf_ptr + nbins + 1;
        int64_t* d_strip = d_qoff + nprob;
        int32_t* d_lo = reinterpret_cast<int32_t*>(reinterpret_cast<unsigned char*>(d_ovf_ptr) + ptr_bytes);
        int32_t* d_hi = d_lo + nbins;
        d_exp = d_hi + nbins;
        HC_CUDA(cudaMemcpyAsync(d_qoff, h_q.data(), h_q.size() * sizeof(int64_t), cudaMemcpyHostToDevice, s));
        HC_CUDA(cudaMemsetAsync(d_ovf_ptr, 0, ((size_t)nbins + 1) * sizeof(int64_t), s));
        HC_CUDA(cudaMemsetAsync(d_lo, 0x7f, (size_t)nbins * sizeof(int32_t), s));
        HC_CUDA(cudaMemsetAsync(d_hi, 0xff, (size_t)nbins * sizeof(int32_t), s));
        HC_CUDA(cudaStreamSynchronize(s));      // h_q goes out of scope
        int kt_max = 0;
        for (int p = 0; p < nprob; ++p) kt_max = std::max(kt_max, h_ld[p] >> 5);
        ice_pack_tiles_kernel<<<dim3((unsigned)((strips * 32 + 255) / 256), (unsigned)((kt_max + 7) / 8)), 256, 0, s>>>(
            mats, mat_off, mat_n, mat_ld, d_qoff, d_strip, bin_off, nprob, P->ignore_diags, d_q8,
            reinterpret_cast<unsigned long long*>(d_ovf_ptr), d_lo, d_hi);
        HC_LAUNCH_CHECK();
        {
            const int nb = (int)((nbins + 1023) / 1024);
            int64_t* d_bsum = d_strip + nprob + 1;       // nb + 1 entries behind the strip table
            ice_ovf_blocksum_kernel<<<nb, 256, 0, s>>>(d_ovf_ptr, nbins, d_bsum);
            HC_LAUNCH_CHECK();
            ice_ovf_scan_blocks_kernel<<<1, 1024, 0, s>>>(d_bsum, nb);
            HC_LAUNCH_CHECK();
            ice_ovf_scan_kernel<<<nb, 256, 0, s>>>(d_ovf_ptr, nbins, d_bsum, nb);
            HC_LAUNCH_CHECK();
        }
        HC_CUDA(hc_read_small(&novf, d_ovf_ptr + nbins, sizeof(long long), s));
        HC_CUDA(scratch.alloc((void**)&d_ovf, 2 * (size_t)std::max(novf, 1ll) * sizeof(int32_t)));
        if (novf > 0) {
            ice_pack_ovf_kernel<<<(unsigned)((nbins * 32 + 255) / 256), 256, 0, s>>>(
                mats, mat_off, mat_n, mat_ld, bin_off, nprob, P->ignore_diags, d_ovf_ptr, d_lo, d_hi, d_ovf, d_ovf + novf);
            HC_LAUNCH_CHECK();
        }
    }
    int32_t* d_tab = nullptr;    // 3 item tables | done[nprob] | n_done | queue | iter | nitems | pad to 16 B | item descriptors (packed)
    const size_t desc_at = (3 * max_items + (size_t)nprob + 4 + 3) & ~(size_t)3;
    const size_t tab_ints = desc_at + (packed ? 16 * max_items : 0);
    HC_CUDA(scratch.alloc((void**)&d_tab, tab_ints * sizeof(int32_t)));
    bool desc_uploaded = false;
    auto upload_items = [&]() -> cudaError_t {
        const size_t n = item_prob.size();
        const int32_t n32 = (int32_t)n;
        cudaError_t e = cudaMemcpyAsync(d_tab + 3 * max_items + nprob + 3, &n32, sizeof(int32_t), cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_tab, item_prob.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_tab + max_items, item_row0.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess) e = cudaMemcpyAsync(d_tab + 2 * max_items, item_nrows.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, s);
        if (e == cudaSuccess && packed && !desc_uploaded) {
            e = cudaMemcpyAsync(d_tab + desc_at, item_desc.data(), item_desc.size() * sizeof(int4), cudaMemcpyHostToDevice, s);
            desc_uploaded = true;
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(s);   // the host vectors may be rebuilt afterwards
        return e;
    };
    HC_CUDA(cudaMemsetAsync(d_tab + 3 * max_items, 0, ((size_t)nprob + 3) * sizeof(int32_t), s));
    HC_CUDA(upload_items());
    const int grid = hc_num_sms() * V.minb;    // persistent: every resident slot filled exactly once
    const unsigned int queue_start = (unsigned)grid * 8u;
    HC_CUDA(cudaMemcpyAsync(d_tab + 3 * max_items + nprob + 1, &queue_start, sizeof(unsigned int), cudaMemcpyHostToDevice, s));

    IceDenseArgs A;
    A.mats = mats; A.mat_off = mat_off; A.mat_n = mat_n; A.mat_ld = mat_ld; A.pad_off = d_pad;
    A.item_prob = d_tab; A.item_row0 = d_tab + max_items; A.item_nrows = d_tab + 2 * max_items;
    A.done = d_tab + 3 * max_items;
    A.n_done = A.done + nprob;
    A.queue = reinterpret_cast<unsigned int*>(A.n_done + 1);
    A.iter = A.n_done + 2;
    A.nitems = reinterpret_cast<const unsigned int*>(A.n_done + 3);
    A.bias = biasp; A.marg = marg; A.results = results;
    A.tol = P->tol; A.kd = P->ignore_diags; A.max_iters = P->max_iters; A.nprob = nprob; A.queue_start = queue_start;
    A.q8 = d_q8; A.q_off = d_qoff; A.digits = d_digits; A.dig_exp = d_exp; A.packed = packed ? 1 : 0;
    A.desc = reinterpret_cast<const int4*>(d_tab + desc_at); A.kseg = kseg; A.part = d_part; A.nseg_max = nseg_max; A.npad = npad;
    A.bin_off = bin_off; A.ovf_ptr = d_ovf_ptr; A.ovf_col = d_ovf; A.ovf_val = d_ovf ? d_ovf + novf : nullptr;
    if (packed) {
        ice_digits_kernel<<<nprob, 1024, 0, s>>>(A);      // byte planes of the initial bias
        HC_LAUNCH_CHECK();
        if (evp0) cudaEventRecord(evp1, s);
    }

    int nonempty = 0;
    for (int p = 0; p < nprob; ++p) nonempty += h_mat_n[p] > 0;
    if (nonempty != nprob) {   // empty problems never get work: give them a defined result
        std::vector<hc_ice_result> h_res(nprob);
        for (int p = 0; p < nprob; ++p) { h_res[p].scale = NAN; h_res[p].var = 0.0; h_res[p].iters = 0; h_res[p].converged = 1; }
        HC_CUDA(cudaMemcpyAsync(results, h_res.data(), sizeof(hc_ice_result) * nprob, cudaMemcpyHostToDevice, s));
        HC_CUDA(cudaStreamSynchronize(s));
    }
    // the bias vector (its byte planes for the packed kernel) is the only data that should live in L1
    const size_t smem = 0;
    cudaFuncSetAttribute(V.fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxL1);
    // update kernel: the 8-CTA cluster version needs every chromosome to fit 8 x 256 x 4 padded columns
    bool cluster_update = packed;
    for (int p = 0; p < nprob; ++p) cluster_update = cluster_update && h_ld[p] <= UPD_CLUSTER * 256 * 4;
    if (const char* e = getenv("HC_ICE_CLUSTER_UPDATE")) cluster_update = cluster_update && atoi(e) != 0;
    auto launch_update = [&]() {
        if (cluster_update) ice_q8_update_cluster_kernel<<<nprob * UPD_CLUSTER, 256, 0, s>>>(A);
        else ice_dense_update_kernel<<<nprob, 1024, 0, s>>>(A);
    };
    const int poll = P->poll_every > 0 ? P->poll_every : 8;
    int launches = 0, h_ndone = 0, seen_done = 0;
    int rc = HC_OK;
    // `poll` iterations (stream + update kernel each) captured once and replayed: the iteration index,
    // the work-list length and every convergence decision live in device memory, so the graph is static
    cudaGraphExec_t gexec = nullptr;
    bool use_graph = true;
    if (const char* e = getenv("HC_ICE_GRAPH")) use_graph = atoi(e) != 0;
    // HC_ICE_TIME_KERNEL=1 (set by bench.py): the first stream-kernel launch of every graph replay is bracketed by a pair
    // of events, so that its duration can be read back separately from the update kernel and the launch gaps (external
    // event-record nodes inside the graph; bracketing all 8 launches of a replay cost ~11 us per iteration)
    // The captured graph is kept between calls (per host thread): the next call with the same launch shape only
    // rewrites the kernel parameters of its nodes (cudaGraphExecKernelNodeSetParams) instead of capturing and
    // instantiating again -- ~0.4 ms of host time per call on C2.
    // HC_ICE_TIME_KERNEL=1 (set by bench.py): the first stream-kernel launch of every graph replay is bracketed by a pair
    // of events, so that its duration can be read back separately from the update kernel and the launch gaps (external
    // event-record nodes inside the graph; bracketing all 8 launches of a replay cost ~11 us per iteration)
    struct GraphCache {
        cudaGraphExec_t exec = nullptr;
        cudaGraph_t graph = nullptr;
        std::vector<cudaGraphNode_t> knodes;
        void* fn = nullptr;
        int grid = 0, poll = 0, nprob = 0, cluster = 0, timed = 0, dev = -1;
        cudaEvent_t ev[2] = {nullptr, nullptr};
        void drop() {
            if (exec) cudaGraphExecDestroy(exec);
            if (graph) cudaGraphDestroy(graph);
            exec = nullptr; graph = nullptr; knodes.clear();
        }
    };
    static thread_local GraphCache gc;
    const bool timed = h_info != nullptr && getenv("HC_ICE_TIME_KERNEL") != nullptr && atoi(getenv("HC_ICE_TIME_KERNEL")) != 0;
    struct { std::vector<cudaEvent_t> ev; } sev;
    if (timed) {
        for (auto& e : gc.ev) if (e == nullptr && cudaEventCreate(&e) != cudaSuccess) { e = nullptr; (void)cudaGetLastError(); }
        if (gc.ev[0] && gc.ev[1]) sev.ev.assign(gc.ev, gc.ev + 2);
    }
    double stream_ms_sum = 0.0;
    int stream_ms_n = 0;
    if (use_graph) {
        const bool hit = gc.exec != nullptr && gc.fn == (void*)V.fn && gc.grid == grid && gc.poll == poll && gc.nprob == nprob &&
                         gc.cluster == (int)cluster_update && gc.timed == (int)!sev.ev.empty() && gc.dev == dev;
        cudaError_t e = cudaSuccess;
        if (hit) {
            for (cudaGraphNode_t node : gc.knodes) {
                cudaKernelNodeParams kp;
                e = cudaGraphKernelNodeGetParams(node, &kp);
                void* args[1] = {&A};
                kp.kernelParams = args;
                if (e == cudaSuccess) e = cudaGraphExecKernelNodeSetParams(gc.exec, node, &kp);
                if (e != cudaSuccess) break;
            }
            if (e != cudaSuccess) { (void)cudaGetLastError(); gc.drop(); }
        } else gc.drop();               // another launch shape: capture again
        if (gc.exec == nullptr) {
            e = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal);
            if (e == cudaSuccess) {
                for (int i = 0; i < poll; ++i) {
                    if (i == 0 && !sev.ev.empty()) cudaEventRecordWithFlags(sev.ev[0], s, cudaEventRecordExternal);
                    V.fn<<<grid, 256, smem, s>>>(A);
                    if (i == 0 && !sev.ev.empty()) cudaEventRecordWithFlags(sev.ev[1], s, cudaEventRecordExternal);
                    launch_update();
                }
                e = cudaStreamEndCapture(s, &gc.graph);
            }
            if (e == cudaSuccess) e = cudaGraphInstantiate(&gc.exec, gc.graph, 0);
            if (e == cudaSuccess) {
                size_t nn = 0;
                e = cudaGraphGetNodes(gc.graph, nullptr, &nn);
                std::vector<cudaGraphNode_t> nodes(nn);
                if (e == cudaSuccess && nn) e = cudaGraphGetNodes(gc.graph, nodes.data(), &nn);
                for (size_t k = 0; e == cudaSuccess && k < nn; ++k) {
                    cudaGraphNodeType t;
                    e = cudaGraphNodeGetType(nodes[k], &t);
                    if (e == cudaSuccess && t == cudaGraphNodeTypeKernel) gc.knodes.push_back(nodes[k]);
                }
            }
            if (e != cudaSuccess) { gc.drop(); (void)cudaGetLastError(); }   // plain launches below
            else { gc.fn = (void*)V.fn; gc.grid = grid; gc.poll = poll; gc.nprob = nprob; gc.cluster = (int)cluster_update;
                   gc.timed = (int)!sev.ev.empty(); gc.dev = dev; }
        }
        gexec = gc.exec;
    }
    EventPair evl;                              // device time of the iteration loop, for the roofline
    cudaEvent_t& ev0 = evl.a;
    cudaEvent_t& ev1 = evl.b;
    if (h_info) { evl.create(); cudaEventRecord(ev0, s); }
    for (int k0 = 0; k0 < P->max_iters; k0 += poll) {
        cudaError_t e = cudaSuccess;
        if (gexec) e = cudaGraphLaunch(gexec, s);
        else for (int i = 0; i < poll; ++i) {
            if (i == 0 && !sev.ev.empty()) cudaEventRecord(sev.ev[0], s);
            V.fn<<<grid, 256, smem, s>>>(A);
            if (i == 0 && !sev.ev.empty()) cudaEventRecord(sev.ev[1], s);
            launch_update();
        }
        hc_count_launch(2 * poll);
        launches += 2 * poll;
        if (e == cudaSuccess) e = hc_read_small(&h_ndone, A.n_done, sizeof(int32_t), s);   // not a memcpy: see hc_read_small
        if (e == cudaSuccess && h_ndone == 0 && !sev.ev.empty()) {
            // no problem has finished yet: the bracketed launch streamed every matrix of the batch
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, sev.ev[0], sev.ev[1]) == cudaSuccess) { stream_ms_sum += ms; ++stream_ms_n; }
            else (void)cudaGetLastError();
        }
        if (e == cudaSuccess && h_ndone >= nonempty) break;
        if (e == cudaSuccess && h_ndone != seen_done) {
            // drop the converged chromosomes from the work list (their items would only be skipped)
            seen_done = h_ndone;
            e = hc_read_small(h_done.data(), A.done, sizeof(int32_t) * nprob, s);
            if (e == cudaSuccess) { build_items(); e = upload_items(); }
        }
        if (e != cudaSuccess) { hc_set_error("hc_ice_dense_balance: %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; break; }
    }
    if (h_info && ev0) cudaEventRecord(ev1, s);
    if (rc == HC_OK) {
        const int64_t blocks = (nbins + 255) / 256;
        ice_finalize_kernel<<<(unsigned)blocks, 256, 0, s>>>(bin_off, d_pad, nprob, results, P->rescale_marginals, biasp, bias);
        hc_count_launch();
        ++launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { hc_set_error("hc_ice_dense_balance: %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; }
    }
    cudaError_t e = cudaStreamSynchronize(s);
    if (rc == HC_OK && e != cudaSuccess) { hc_set_error("hc_ice_dense_balance: %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; }
    if (h_info) {
        h_info->launches = launches;
        if (ev0 && e == cudaSuccess) cudaEventElapsedTime(&h_info->loop_ms, ev0, ev1);
        h_info->packed = packed ? 1 : 0;
        h_info->overflow_cells = novf;
        h_info->stream_full_launches = stream_ms_n;
        h_info->stream_full_ms = stream_ms_n ? (float)(stream_ms_sum / stream_ms_n) : 0.f;
        if (evp0 && e == cudaSuccess) cudaEventElapsedTime(&h_info->pack_ms, evp0, evp1);
    }
    return rc;
}
