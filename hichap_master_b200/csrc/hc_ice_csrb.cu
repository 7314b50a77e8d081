// (b) ICE on the symmetric CSR, column-blocked encoding (default path of hc_ice_csr_balance).
// Same algorithm as hc_ice.cu / hc_ice_csr.cu (cooler balance restated in oracle/cooler_ice.py; HiCHap call
// sites matrixBuilding.py:708, :1537, :1761).
//
// Why: on the row-major CSR every stored entry gathers bias[col] (8 B) from L2 as a 32-byte sector.  On a
// genome-wide 10 kb matrix half of the entries are trans / far-cis singletons with effectively random columns,
// so an iteration moves 32 B of L2 traffic per 8 B entry and runs at the L2 gather rate (measured round 1:
// 2.4 TB/s of entries = 0.18 of the HBM roofline on SURVEY's 8Z + 24n bytes).
//
// Encoding (built once per call from the CSR, a pure permutation of runs):
//   * columns are cut into blocks of CB = 8192 bins; the bias of one block is 64 KB and is staged in shared
//     memory by ONE bulk asynchronous copy (cp.async.bulk -> mbarrier), so every gather becomes an LDS.64;
//   * an entry is 4 bytes: column within the block (13 bits) | weighted count (19 bits; cooler's pixel weight
//     already applied: ignored diagonals are 0, a kept main diagonal counts twice).  Both triangles are
//     stored, so an iteration streams 4 B x 2Z = SURVEY's 8Z algorithmic bytes and stays a pure row-wise
//     reduction (no atomics, deterministic);
//   * segment (cb, row) = the entries of `row` whose column lies in block cb, padded to a multiple of 4
//     entries (16-byte aligned 128-bit loads); segments are ordered (cb, row); seg_ptr is int64;
//   * a count that does not fit 19 bits makes the call fall back to the row-major kernel (hc_ice_csr.cu).
//
// Per iteration (all inside a replayed CUDA graph, nothing returns to the host except a done-counter poll):
//   csrb_stream_kernel  persistent CTAs draw items (one column block x a run of rows holding ~64 K entries)
//                       from a global queue; groups of 2 / 8 / 32 lanes reduce one segment each and store
//                       part[cb][row];
//   csrb_marg_kernel    marg[row] = bias[row] * sum_cb part[cb][row] (fixed order);
//   [ncclAllReduce of marg when the matrix is row-block sharded -- captured in the same graph]
//   csrb_update_kernel  one thread-block cluster per problem: mean / variance of the non-zero marginals
//                       through distributed shared memory, bias update, convergence test.
#include <cooperative_groups.h>
#include <math.h>
#include <stdlib.h>
#include <algorithm>
#include <vector>
#include "hc_common.cuh"
#include <chrono>

int hc_nccl_allreduce_f64(void* comm, const double* send, double* recv, size_t count, cudaStream_t s);  // hc_nccl.cu

namespace {

constexpr int CB_BITS = 13;
constexpr int CB = 1 << CB_BITS;            // bins per column block: 64 KB of fp64 bias
constexpr int CNT_BITS = 16;                // entry = (column within the block) * 8 in the low 16 bits | weighted count << 16
constexpr long long CNT_MAX = (1ll << CNT_BITS) - 1;
constexpr int ST_THREADS = 352;             // stream kernel: 3 CTAs x 352 threads x 64 KB per SM (<= 62 registers per thread)
constexpr int ST_MINB = 3;
constexpr int UPD_CLUSTER = 8;
constexpr int UPD_THREADS = 1024;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ long long band_wcount(long long c, long long r, int kd, int v) {
    const long long d = c - r;
    if (d == 0) return kd == 0 ? 2ll * v : 0ll;
    return (d < kd && d > -kd) ? 0ll : (long long)v;
}

__device__ __forceinline__ int find_problem(const int64_t* __restrict__ bin_off, int nprob, long long r) {
    int lo = 0, hi = nprob - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (bin_off[mid] <= r) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---------------------------------------------------------------------------------------
// build
// ---------------------------------------------------------------------------------------
// start[cb * nloc + rl] = index (into col/cnt) of the first entry of local row rl whose column block is >= cb.
// One warp per row; the columns of a row are sorted, so the lane that sees a block change writes the starts of
// every block in between.
__global__ void __launch_bounds__(256)
csrb_start_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, long long nloc, int nb,
                  int64_t* __restrict__ start) {
    const long long rl = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (rl >= nloc) return;
    const long long e0 = row_ptr[rl], e1 = row_ptr[rl + 1];
    for (long long e = e0 + lane; e < e1 + 1; e += 32) {      // e == e1: the sentinel past the last entry
        const int cbp = e == e0 ? -1 : (__ldg(col + e - 1) >> CB_BITS);
        const int cbe = e == e1 ? nb - 1 : (__ldg(col + e) >> CB_BITS);
        const int upto = e == e1 ? nb - 1 : cbe;
        for (int b = cbp + 1; b <= upto; ++b) start[(long long)b * nloc + rl] = e;
        (void)cbe;
    }
}

// seg_len (padded to a multiple of 4 entries) in (cb, row) order
__global__ void __launch_bounds__(256)
csrb_len_kernel(const int64_t* __restrict__ row_ptr, const int64_t* __restrict__ start, long long nloc, int nb,
                int64_t* __restrict__ seg_ptr) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nloc * nb) return;
    const long long cb = i / nloc, rl = i - cb * nloc;
    const long long s0 = start[i], s1 = cb + 1 < nb ? start[i + nloc] : row_ptr[rl + 1];
    seg_ptr[i] = (s1 - s0 + 3) & ~3ll;
}

// exclusive scan of int64 (in place), total -> v[n]: per-block sums (2048 per block), single-CTA scan of those, rescan
constexpr int SCAN_BLOCK = 2048;
__global__ void __launch_bounds__(256) csrb_scan_blocksum_kernel(const int64_t* __restrict__ v, long long n, int64_t* __restrict__ bsum) {
    __shared__ long long redll[8];
    const long long base = (long long)blockIdx.x * SCAN_BLOCK;
    long long s = 0;
    for (int i = threadIdx.x; i < SCAN_BLOCK; i += 256) if (base + i < n) s += v[base + i];
    s = block_sum_ll(s, redll);
    if (threadIdx.x == 0) bsum[blockIdx.x] = s;
}
__global__ void __launch_bounds__(1024) csrb_scan_blocks_kernel(int64_t* __restrict__ bsum, int nb) {
    __shared__ long long sh[1024];
    long long run = 0;
    for (int b0 = 0; b0 < nb; b0 += 1024) {
        const int i = b0 + threadIdx.x;
        const long long v = i < nb ? bsum[i] : 0;
        sh[threadIdx.x] = v;
        __syncthreads();
        for (int o = 1; o < 1024; o <<= 1) {
            const long long t = threadIdx.x >= o ? sh[threadIdx.x - o] : 0;
            __syncthreads();
            sh[threadIdx.x] += t;
            __syncthreads();
        }
        if (i < nb) bsum[i] = run + sh[threadIdx.x] - v;
        run += sh[1023];
        __syncthreads();
    }
    if (threadIdx.x == 0) bsum[nb] = run;
}
__global__ void __launch_bounds__(256) csrb_scan_apply_kernel(int64_t* __restrict__ v, long long n, const int64_t* __restrict__ bsum, int nb) {
    __shared__ long long wsum[8];
    const long long base = (long long)blockIdx.x * SCAN_BLOCK + 8 * threadIdx.x;
    long long x[8], t = 0;
#pragma unroll
    for (int e = 0; e < 8; ++e) { x[e] = base + e < n ? v[base + e] : 0; t += x[e]; }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    long long inc = t;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const long long u = __shfl_up_sync(0xffffffffu, inc, o); if (lane >= o) inc += u; }
    if (lane == 31) wsum[wid] = inc;
    __syncthreads();
    long long off = bsum[blockIdx.x] + inc - t;
    for (int w = 0; w < wid; ++w) off += wsum[w];
#pragma unroll
    for (int e = 0; e < 8; ++e) { if (base + e < n) v[base + e] = off; off += x[e]; }
    if (blockIdx.x == gridDim.x - 1 && threadIdx.x == 0) v[n] = bsum[nb];
}

// entries into their segments; overflow[0] is set when a weighted count does not fit CNT_BITS
__global__ void __launch_bounds__(256)
csrb_fill_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, const int32_t* __restrict__ cnt,
                 long long row0, long long nloc, int kd, const int64_t* __restrict__ start,
                 const int64_t* __restrict__ seg_ptr, uint32_t* __restrict__ ent, int32_t* __restrict__ overflow) {
    const long long rl = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (rl >= nloc) return;
    const long long e0 = row_ptr[rl], e1 = row_ptr[rl + 1], r = row0 + rl;
    bool ovf = false;
    for (long long e = e0 + lane; e < e1; e += 32) {
        const int c = __ldg(col + e);
        const long long i = (long long)(c >> CB_BITS) * nloc + rl;
        const long long wc = band_wcount(c, r, kd, __ldg(cnt + e));
        ovf |= wc > CNT_MAX || wc < 0;
        ent[seg_ptr[i] + (e - start[i])] = ((uint32_t)(c & (CB - 1)) << 3) | ((uint32_t)(wc & CNT_MAX) << 16);
    }
    if (__any_sync(0xffffffffu, ovf) && lane == 0) atomicExch(overflow, 1);
}

__global__ void csrb_flag_kernel(const int32_t* __restrict__ flag, double* __restrict__ out) {
    if (threadIdx.x == 0) out[0] = (flag != nullptr && *flag != 0) ? 1.0 : 0.0;
}

// seg_ptr at the block boundaries -> a small contiguous table the host reads (entries per column block)
__global__ void csrb_block_totals_kernel(const int64_t* __restrict__ seg_ptr, long long nloc, int nb, int64_t* __restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i <= nb) out[i] = seg_ptr[(long long)i * nloc];
}

// item k of column block cb covers the rows whose segments start in [base + k * target, base + (k + 1) * target):
// desc = {cb, first row, end row, log2 of the lane-group size}
__global__ void __launch_bounds__(256)
csrb_items_kernel(const int64_t* __restrict__ seg_ptr, long long nloc, int nb, const int32_t* __restrict__ item_first,
                  int nitems, long long target, int4 gthr, int4* __restrict__ desc) {
    const int it = blockIdx.x * blockDim.x + threadIdx.x;
    if (it >= nitems) return;
    int lo = 0, hi = nb - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (item_first[mid] <= it) lo = mid; else hi = mid - 1; }
    const int cb = lo, k = it - item_first[cb];
    const int64_t* sp = seg_ptr + (long long)cb * nloc;
    const long long base = sp[0];
    auto first_row_at = [&](long long off) {      // first row whose segment start is >= off
        long long a = 0, b = nloc;
        while (a < b) { const long long m = (a + b) >> 1; if (sp[m] < off) a = m + 1; else b = m; }
        return a;
    };
    const long long r0 = k == 0 ? 0 : first_row_at(base + (long long)k * target);
    const long long r1 = it + 1 == item_first[cb + 1] ? nloc : first_row_at(base + (long long)(k + 1) * target);
    const long long entries = sp[r1] - sp[r0];          // sp[nloc] is the next block's first segment (or the total)
    const long long rows = r1 > r0 ? r1 - r0 : 1;
    const long long avg = entries / rows;
    // lanes per segment: fewer lanes per segment = more segments (independent load chains) in flight per warp
    const int glog = avg >= gthr.w ? 5 : (avg >= gthr.z ? 4 : (avg >= gthr.y ? 3 : (avg >= gthr.x ? 2 : 1)));
    desc[it] = make_int4(cb, (int)r0, (int)r1, glog);
}

// ---------------------------------------------------------------------------------------
// iteration
// ---------------------------------------------------------------------------------------
struct CsrbArgs {
    const int64_t* seg_ptr; const uint32_t* ent; const int4* items; int nitems;
    long long nloc, row0; int nb;
    const double* bias_pad;          // [nb * CB], zero beyond nbins
    double* part;                    // [nb * nloc]
    unsigned int* queue;
    const int64_t* bin_off; int nprob; const int32_t* done_at; const int32_t* n_done; int nonempty;
};

// one entry: count (high 16 bits) times the staged bias at byte offset (low 16 bits).  The count becomes a double by
// being placed in the mantissa of 2^52 (one DADD, no conversion instruction).
__device__ __forceinline__ double csrb_term(unsigned e, const double* __restrict__ sb, double acc) {
    const double c = __hiloint2double(0x43300000, (int)(e >> 16)) - 4503599627370496.0;
    return fma(c, *reinterpret_cast<const double*>(reinterpret_cast<const unsigned char*>(sb) + (e & 0xffffu)), acc);
}
__device__ __forceinline__ void csrb_fma4(const int4& q, const double* __restrict__ sb, double& a0, double& a1) {
    a0 = csrb_term((unsigned)q.x, sb, a0);
    a1 = csrb_term((unsigned)q.y, sb, a1);
    a0 = csrb_term((unsigned)q.z, sb, a0);
    a1 = csrb_term((unsigned)q.w, sb, a1);
}

// One item: rows [r0, r1) of column block cb.  Groups of G lanes take rows round robin.  The segments are short (tens to
// a few hundred entries), so a row is a chain of two dependent loads (segment bounds -> entries) with little work
// behind it; the loop is therefore software-pipelined over rows: while row r is reduced, the first 128-bit vector of
// the group's next row is in flight and the bounds of the one after that are being fetched (ncu on the unpipelined
// version: long-scoreboard stalls dominate at 2.1 TB/s, profiles/r2c_ncu_csrb_stream_v1.json).
template <int G>
__device__ __forceinline__ void csrb_process_item(const CsrbArgs& A, const double* __restrict__ sb, int cb, int r0, int r1) {
    const int gl = threadIdx.x & (G - 1);
    const int gid = threadIdx.x / G, ng = blockDim.x / G;
    // the groups of one warp run different numbers of rows: shuffle only among the lanes of the own group
    const unsigned gmask = G == 32 ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1)));
    const int64_t* __restrict__ sp = A.seg_ptr + (long long)cb * A.nloc;
    const long long base4 = __ldg(sp + r0) >> 2;                 // 128-bit vector index of the item's first entry
    const int4* __restrict__ e4 = reinterpret_cast<const int4*>(A.ent) + base4;
    double* __restrict__ pout = A.part + (long long)cb * A.nloc;
    const int4 zero = make_int4(0, 0, 0, 0);
    int row = r0 + gid;
    int c0 = 0, c1 = 0, n0 = 0, n1 = 0, m0 = 0, m1 = 0;          // bounds (vectors, relative to base4) of this row, the next, the one after
    if (row < r1) { c0 = (int)((__ldg(sp + row) >> 2) - base4); c1 = (int)((__ldg(sp + row + 1) >> 2) - base4); }
    if (row + ng < r1) { n0 = (int)((__ldg(sp + row + ng) >> 2) - base4); n1 = (int)((__ldg(sp + row + ng + 1) >> 2) - base4); }
    int4 qc = (row < r1 && c0 + gl < c1) ? ld_stream_v4(reinterpret_cast<const int32_t*>(e4 + c0 + gl)) : zero;
    for (; row < r1; row += ng) {
        if (row + 2 * ng < r1) {
            m0 = (int)((__ldg(sp + row + 2 * ng) >> 2) - base4);
            m1 = (int)((__ldg(sp + row + 2 * ng + 1) >> 2) - base4);
        }
        const int4 qn = (row + ng < r1 && n0 + gl < n1) ? ld_stream_v4(reinterpret_cast<const int32_t*>(e4 + n0 + gl)) : zero;
        bool live = true;
        if (A.nprob > 1) live = A.done_at[find_problem(A.bin_off, A.nprob, A.row0 + row)] == 0;   // group-uniform
        if (live) {
            double a0 = 0.0, a1 = 0.0;
            csrb_fma4(qc, sb, a0, a1);                    // an absent vector is all zero: count 0 times sb[0]
            int v = c0 + gl + G;
            for (; v + G < c1; v += 2 * G) {              // two 128-bit loads in flight per lane
                const int4 q = ld_stream_v4(reinterpret_cast<const int32_t*>(e4 + v));
                const int4 u = ld_stream_v4(reinterpret_cast<const int32_t*>(e4 + v + G));
                csrb_fma4(q, sb, a0, a1);
                csrb_fma4(u, sb, a0, a1);
            }
            if (v < c1) {
                const int4 q = ld_stream_v4(reinterpret_cast<const int32_t*>(e4 + v));
                csrb_fma4(q, sb, a0, a1);
            }
            double acc = a0 + a1;
#pragma unroll
            for (int o = G / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(gmask, acc, o);
            if (gl == 0) pout[row] = acc;
        }
        c0 = n0; c1 = n1; n0 = m0; n1 = m1; qc = qn;
    }
}

__global__ void __launch_bounds__(ST_THREADS, ST_MINB)
csrb_stream_kernel(CsrbArgs A) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double* sb = reinterpret_cast<double*>(smem_raw);
    __shared__ __align__(8) unsigned long long mbar;
    __shared__ unsigned int item_s;
    if (*A.n_done >= A.nonempty) return;             // every problem converged: the rest of the replayed graph is idle
    if (threadIdx.x == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(&mbar)), "r"(1) : "memory");
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    uint32_t phase = 0;
    int staged = -1;
    for (;;) {
        if (threadIdx.x == 0) item_s = atomicAdd(A.queue, 1u);
        __syncthreads();                            // also: every warp is done with the previous item (and its bias block)
        const unsigned int it = item_s;
        __syncthreads();                            // item_s is rewritten at the top of the next round
        if (it >= (unsigned)A.nitems) break;
        const int4 d = __ldg(A.items + it);
        if (d.x != staged) {
            if (threadIdx.x == 0) {
                const uint32_t bytes = CB * (uint32_t)sizeof(double);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");     // generic-proxy reads of sb precede the async write
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(&mbar)), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                             :: "r"(smem_u32(sb)), "l"(A.bias_pad + (long long)d.x * CB), "r"(bytes), "r"(smem_u32(&mbar)) : "memory");
            }
            uint32_t done = 0;
            while (!done) {
                asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
                             : "=r"(done) : "r"(smem_u32(&mbar)), "r"(phase) : "memory");
            }
            phase ^= 1;
            staged = d.x;
        }
        if (d.w == 5) csrb_process_item<32>(A, sb, d.x, d.y, d.z);
        else if (d.w == 4) csrb_process_item<16>(A, sb, d.x, d.y, d.z);
        else if (d.w == 3) csrb_process_item<8>(A, sb, d.x, d.y, d.z);
        else if (d.w == 2) csrb_process_item<4>(A, sb, d.x, d.y, d.z);
        else csrb_process_item<2>(A, sb, d.x, d.y, d.z);
    }
}

struct VecArgs {
    const int64_t* bin_off; int nprob;
    long long nloc, row0, nbins; int nb;
    const double* part; double* bias_pad; double* marg_local; const double* marg;
    unsigned int* queue; int32_t* iter; int32_t* done_at; int32_t* n_done; int nonempty;
    hc_ice_result* results; double tol; int max_iters;
};

// marg_local[row] = bias[row] * sum over column blocks of part[cb][row], in block order; opens iteration k
__global__ void __launch_bounds__(256) csrb_marg_kernel(VecArgs a) {
    const long long rl = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (blockIdx.x == 0 && threadIdx.x == 0) { *a.queue = 0u; if (*a.n_done < a.nonempty) atomicAdd(a.iter, 1); }
    if (*a.n_done >= a.nonempty || rl >= a.nloc) return;
    const long long r = a.row0 + rl;
    if (a.nprob > 1 && a.done_at[find_problem(a.bin_off, a.nprob, r)] != 0) return;
    double s = 0.0;
    for (int cb = 0; cb < a.nb; ++cb) s += a.part[(long long)cb * a.nloc + rl];
    a.marg_local[r] = a.bias_pad[r] * s;
}

// single-GPU rank with no local rows still has to open the iteration
__global__ void csrb_open_iter_kernel(VecArgs a) {
    if (threadIdx.x == 0) { *a.queue = 0u; if (*a.n_done < a.nonempty) atomicAdd(a.iter, 1); }
}

// one cluster of UPD_CLUSTER CTAs per problem: mean / variance over the non-zero marginals, bias update, convergence
__global__ void __cluster_dims__(UPD_CLUSTER, 1, 1) __launch_bounds__(UPD_THREADS)
csrb_update_kernel(VecArgs a) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    __shared__ double red[32];
    __shared__ long long redll[32];
    __shared__ double sh_sum, sh_var;
    __shared__ long long sh_cnt;
    const int p = blockIdx.x / UPD_CLUSTER, rank = (int)cluster.block_rank();
    const int k = *a.iter;
    if (a.done_at[p] != 0 || k > a.max_iters) return;        // uniform over the cluster
    const long long b0 = a.bin_off[p], n = a.bin_off[p + 1] - b0;
    if (n == 0) return;
    const long long lo = b0 + n * rank / UPD_CLUSTER, hi = b0 + n * (rank + 1) / UPD_CLUSTER;
    double s = 0.0;
    long long c = 0;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const double m = a.marg[i];
        if (m != 0.0) { s += m; ++c; }
    }
    s = block_sum(s, red);
    c = block_sum_ll(c, redll);
    if (threadIdx.x == 0) { sh_sum = s; sh_cnt = c; }
    cluster.sync();
    s = 0.0; c = 0;
#pragma unroll
    for (int r = 0; r < UPD_CLUSTER; ++r) { s += *cluster.map_shared_rank(&sh_sum, r); c += *cluster.map_shared_rank(&sh_cnt, r); }
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    if (c == 0) {       // nothing left to balance: cooler sets bias = NaN, scale = NaN, var = 0
        for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) a.bias_pad[i] = nan;
        if (rank == 0 && threadIdx.x == 0) {
            hc_ice_result r; r.scale = nan; r.var = 0.0; r.iters = k; r.converged = 1;
            a.results[p] = r; a.done_at[p] = k; atomicAdd(a.n_done, 1);
        }
        cluster.sync();
        return;
    }
    const double mean = s / (double)c;
    double v = 0.0;
    for (long long i = lo + threadIdx.x; i < hi; i += blockDim.x) {
        const double m = a.marg[i];
        if (m != 0.0) { const double d = m - mean; v += d * d; }
        double q = m / mean;
        if (q == 0.0) q = 1.0;
        a.bias_pad[i] = a.bias_pad[i] / q;
    }
    v = block_sum(v, red);
    if (threadIdx.x == 0) sh_var = v;
    cluster.sync();
    v = 0.0;
#pragma unroll
    for (int r = 0; r < UPD_CLUSTER; ++r) v += *cluster.map_shared_rank(&sh_var, r);
    const double var = v / (double)c;
    if (rank == 0 && threadIdx.x == 0) {
        hc_ice_result r; r.scale = mean; r.var = var; r.iters = k; r.converged = var < a.tol;
        a.results[p] = r;
        if (var < a.tol || k >= a.max_iters) { a.done_at[p] = k; atomicAdd(a.n_done, 1); }
    }
    cluster.sync();          // keep every CTA's shared memory alive until the remote reads are done
}

__global__ void __launch_bounds__(256)
csrb_finalize_kernel(const int64_t* __restrict__ bin_off, int nprob, const hc_ice_result* __restrict__ results,
                     int rescale, const double* __restrict__ bias_pad, double* __restrict__ bias) {
    const long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= bin_off[nprob]) return;
    const int p = nprob > 1 ? find_problem(bin_off, nprob, g) : 0;
    const hc_ice_result r = results[p];
    double b = bias_pad[g];
    if (!isnan(r.scale)) {
        if (b == 0.0) b = __longlong_as_double(0x7ff8000000000000ll);
        if (rescale) b = b / sqrt(r.scale);
    } else b = __longlong_as_double(0x7ff8000000000000ll);
    bias[g] = b;
}

struct Scratch {
    cudaStream_t s;
    std::vector<void*> ptrs;
    explicit Scratch(cudaStream_t st) : s(st) {}
    cudaError_t alloc(void** p, size_t bytes) {
        const cudaError_t e = cudaMallocAsync(p, bytes ? bytes : 16, s);
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
    cudaError_t alloc_big(void** p, size_t bytes) {      // from the pool that only holds multi-GB blocks (hc_big_pool)
        cudaMemPool_t pool = hc_big_pool();
        if (!pool) return alloc(p, bytes);
        const cudaError_t e = cudaMallocFromPoolAsync(p, bytes ? bytes : 16, pool, s);
        if (e == cudaSuccess) ptrs.push_back(*p);
        return e;
    }
    void release(void* p) {
        for (auto& q : ptrs) if (q == p) { cudaFreeAsync(p, s); q = nullptr; }
    }
    ~Scratch() { for (void* p : ptrs) if (p) cudaFreeAsync(p, s); }
};

}  // namespace

// Returns HC_OK, an error, or +1 when the encoding cannot hold the counts (caller falls back to the row-major path).
int hc_ice_csr_balance_blocked(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0, int64_t nloc,
                               const int64_t* bin_off, int32_t nprob, const int64_t* h_bin_off, const hc_ice_params* P,
                               double* bias, hc_ice_result* results, hc_ice_run_info* h_info, void* nccl_comm,
                               cudaStream_t caller) {
    const long long nbins = h_bin_off[nprob];
    const int nb = (int)((nbins + CB - 1) / CB);
    // the loop is replayed as a CUDA graph, which cannot be captured on the legacy default stream: private stream
    // ordered after the caller's (the call synchronises before returning)
    static thread_local cudaStream_t private_stream[64] = {nullptr};
    int dev = 0;
    HC_CUDA(cudaGetDevice(&dev));
    HC_REQUIRE(dev >= 0 && dev < 64, "device index");
    if (!private_stream[dev]) HC_CUDA(cudaStreamCreateWithFlags(&private_stream[dev], cudaStreamNonBlocking));
    cudaStream_t s = private_stream[dev];
    {
        cudaEvent_t e_in;
        HC_CUDA(cudaEventCreateWithFlags(&e_in, cudaEventDisableTiming));
        HC_CUDA(cudaEventRecord(e_in, caller));
        HC_CUDA(cudaStreamWaitEvent(s, e_in, 0));
        cudaEventDestroy(e_in);
    }
    Scratch scratch(s);
    const bool trace = getenv("HC_DEBUG_MEM") != nullptr && atoi(getenv("HC_DEBUG_MEM")) != 0;
    auto t_last = std::chrono::steady_clock::now();
    auto tick = [&](const char* what) {
        if (!trace) return;
        cudaStreamSynchronize(s);
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[csrb] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    tick("enter");
    cudaEvent_t evb0 = nullptr, evb1 = nullptr, ev0 = nullptr, ev1 = nullptr;
    struct EvGuard { cudaEvent_t* e[4]; ~EvGuard() { for (auto p : e) if (*p) cudaEventDestroy(*p); } } evg{{&evb0, &evb1, &ev0, &ev1}};
    if (h_info) { cudaEventCreate(&evb0); cudaEventCreate(&evb1); cudaEventCreate(&ev0); cudaEventCreate(&ev1); cudaEventRecord(evb0, s); }

    // ---- encoding -----------------------------------------------------------------------------------------
    const long long nseg = (long long)nb * nloc;
    int64_t *d_start = nullptr, *d_seg = nullptr, *d_bsum = nullptr, *d_tot = nullptr;
    int32_t* d_flag = nullptr;
    uint32_t* d_ent = nullptr;
    long long total_ent = 0;
    std::vector<int64_t> h_tot(nb + 1, 0);
    if (nloc > 0) {
        const int nsb = (int)((nseg + SCAN_BLOCK - 1) / SCAN_BLOCK);
        // The entry buffer is by far the largest scratch block (3.9 GB on C4).  It is requested FIRST, with an upper bound on
        // its size (every non-empty segment pads at most 3 entries), and from a pool of its own (hc_big_pool): in the default
        // pool smaller requests -- of this call or of another one -- were carved out of the big free block, and the next big
        // request paid 30-200 ms for fresh mappings (profiles/r3d_c4ice.json; 238 instead of 59 ms inside bench.py).
        int64_t h_nnz = 0;
        HC_CUDA(hc_read_small(&h_nnz, row_ptr + nloc, sizeof(int64_t), s));
        const long long ent_cap = std::max(4ll, (long long)h_nnz + 3 * std::min<long long>(nseg, (long long)h_nnz));
        tick("read nnz");
        HC_CUDA(scratch.alloc_big((void**)&d_ent, sizeof(uint32_t) * (size_t)ent_cap));
        tick("alloc entries");
        HC_CUDA(scratch.alloc((void**)&d_start, sizeof(int64_t) * nseg));
        HC_CUDA(scratch.alloc((void**)&d_seg, sizeof(int64_t) * (nseg + 1)));      // + the total
        HC_CUDA(scratch.alloc((void**)&d_bsum, sizeof(int64_t) * (nsb + 1 + nb + 1) + 16));
        d_tot = d_bsum + nsb + 1;
        d_flag = reinterpret_cast<int32_t*>(d_tot + nb + 1);
        HC_CUDA(cudaMemsetAsync(d_flag, 0, sizeof(int32_t), s));
        csrb_start_kernel<<<(unsigned)((nloc * 32 + 255) / 256), 256, 0, s>>>(row_ptr, col, nloc, nb, d_start);
        HC_LAUNCH_CHECK();
        csrb_len_kernel<<<(unsigned)((nseg + 255) / 256), 256, 0, s>>>(row_ptr, d_start, nloc, nb, d_seg);
        HC_LAUNCH_CHECK();
        csrb_scan_blocksum_kernel<<<nsb, 256, 0, s>>>(d_seg, nseg, d_bsum);
        HC_LAUNCH_CHECK();
        csrb_scan_blocks_kernel<<<1, 1024, 0, s>>>(d_bsum, nsb);
        HC_LAUNCH_CHECK();
        csrb_scan_apply_kernel<<<nsb, 256, 0, s>>>(d_seg, nseg, d_bsum, nsb);
        HC_LAUNCH_CHECK();
        csrb_block_totals_kernel<<<(nb + 1 + 255) / 256, 256, 0, s>>>(d_seg, nloc, nb, d_tot);
        HC_LAUNCH_CHECK();
        HC_CUDA(hc_read_small(h_tot.data(), d_tot, sizeof(int64_t) * (nb + 1), s));
        tick("start/len/scan");
        total_ent = h_tot[nb];
        HC_REQUIRE(total_ent <= ent_cap, "internal: entry bound");
        HC_CUDA(cudaMemsetAsync(d_ent, 0, sizeof(uint32_t) * (size_t)std::max(total_ent, 4ll), s));
        csrb_fill_kernel<<<(unsigned)((nloc * 32 + 255) / 256), 256, 0, s>>>(row_ptr, col, cnt, row0, nloc, P->ignore_diags, d_start,
                                                                             d_seg, d_ent, d_flag);
        HC_LAUNCH_CHECK();
        tick("memset + fill");
        scratch.release(d_start);
        d_start = nullptr;
    }
    {
        // a count beyond 19 bits anywhere (on any rank: the ranks must take the same path, their allreduce
        // sequences differ) -> row-major kernel instead
        double* d_f = nullptr;
        HC_CUDA(scratch.alloc((void**)&d_f, 2 * sizeof(double)));
        csrb_flag_kernel<<<1, 32, 0, s>>>(d_flag, d_f);
        HC_LAUNCH_CHECK();
        if (nccl_comm) {
            const int r = hc_nccl_allreduce_f64(nccl_comm, d_f, d_f + 1, 1, s);
            if (r != HC_OK) return r;
        }
        double h_f = 0.0;
        HC_CUDA(hc_read_small(&h_f, nccl_comm ? d_f + 1 : d_f, sizeof(double), s));
        if (h_f != 0.0) return 1;
    }
    // ---- items: ~target entries each, never across a column block ------------------------------------------
    long long target = 64 * 1024;
    if (const char* e = getenv("HC_CSRB_ITEM_ENTRIES")) target = std::max(1024ll, atoll(e));
    const int grid = hc_num_sms() * ST_MINB;
    while (target > 4096 && total_ent / target < 8ll * grid) target >>= 1;     // small problems: enough items for every CTA
    std::vector<int32_t> h_first(nb + 1, 0);
    for (int b = 0; b < nb; ++b) {
        const long long e = h_tot[b + 1] - h_tot[b];
        h_first[b + 1] = h_first[b] + (int32_t)(e > 0 ? (e + target - 1) / target : 0);
    }
    const int nitems = h_first[nb];
    int4* d_items = nullptr;
    int32_t* d_first = nullptr;
    HC_CUDA(scratch.alloc((void**)&d_items, sizeof(int4) * (size_t)std::max(nitems, 1)));
    HC_CUDA(scratch.alloc((void**)&d_first, sizeof(int32_t) * (nb + 1)));
    HC_CUDA(cudaMemcpyAsync(d_first, h_first.data(), sizeof(int32_t) * (nb + 1), cudaMemcpyHostToDevice, s));
    // average segment length from which a segment gets 4 / 8 / 16 / 32 lanes (HC_CSRB_GTHR="a,b,c,d" overrides)
    int4 gthr = make_int4(8, 32, 128, 512);      // measured on C4 (profiles/README.md): flat between these and (20, 20, 192, 192)
    if (const char* e = getenv("HC_CSRB_GTHR")) {
        int a = 0, b = 0, c = 0, d = 0;
        if (sscanf(e, "%d,%d,%d,%d", &a, &b, &c, &d) == 4) gthr = make_int4(a, b, c, d);
    }
    if (nitems > 0) {
        csrb_items_kernel<<<(nitems + 255) / 256, 256, 0, s>>>(d_seg, nloc, nb, d_first, nitems, target, gthr, d_items);
        HC_LAUNCH_CHECK();
    }
    HC_CUDA(cudaStreamSynchronize(s));             // h_first goes out of use
    tick("flag + items");

    // ---- vectors and bookkeeping ---------------------------------------------------------------------------
    double* d_vec = nullptr;        // bias_pad[nb*CB] | marg[nbins] | marg_local[nbins] (sharded only)
    const size_t npad = (size_t)nb * CB;
    HC_CUDA(scratch.alloc((void**)&d_vec, sizeof(double) * (npad + 2 * (size_t)nbins)));
    double* bias_pad = d_vec;
    double* marg = d_vec + npad;
    double* marg_local = nccl_comm ? marg + nbins : marg;
    HC_CUDA(cudaMemsetAsync(d_vec, 0, sizeof(double) * (npad + 2 * (size_t)nbins), s));
    HC_CUDA(cudaMemcpyAsync(bias_pad, bias, sizeof(double) * (size_t)nbins, cudaMemcpyDeviceToDevice, s));
    double* d_part = nullptr;
    HC_CUDA(scratch.alloc((void**)&d_part, sizeof(double) * (size_t)std::max(nseg, 1ll)));
    HC_CUDA(cudaMemsetAsync(d_part, 0, sizeof(double) * (size_t)std::max(nseg, 1ll), s));
    int32_t* d_book = nullptr;      // done_at[nprob] | n_done | queue | iter
    HC_CUDA(scratch.alloc((void**)&d_book, sizeof(int32_t) * (nprob + 4)));
    std::vector<int32_t> h_book(nprob + 4, 0);
    std::vector<hc_ice_result> h_res(nprob);
    int nonempty = 0;
    for (int p = 0; p < nprob; ++p) {
        h_res[p].scale = NAN; h_res[p].var = 0.0; h_res[p].iters = 0; h_res[p].converged = 1;
        if (h_bin_off[p + 1] > h_bin_off[p]) ++nonempty; else h_book[p] = -1;     // problems without bins are done from the start
    }
    HC_CUDA(cudaMemcpyAsync(d_book, h_book.data(), sizeof(int32_t) * (nprob + 4), cudaMemcpyHostToDevice, s));
    HC_CUDA(cudaMemcpyAsync(results, h_res.data(), sizeof(hc_ice_result) * nprob, cudaMemcpyHostToDevice, s));
    HC_CUDA(cudaStreamSynchronize(s));
    tick("vectors + book");
    if (h_info && evb1) cudaEventRecord(evb1, s);

    CsrbArgs A;
    A.seg_ptr = d_seg; A.ent = d_ent; A.items = d_items; A.nitems = nitems; A.nloc = nloc; A.row0 = row0; A.nb = nb;
    A.bias_pad = bias_pad; A.part = d_part; A.queue = reinterpret_cast<unsigned int*>(d_book + nprob + 1);
    A.bin_off = bin_off; A.nprob = nprob; A.done_at = d_book; A.n_done = d_book + nprob; A.nonempty = nonempty;
    VecArgs V;
    V.bin_off = bin_off; V.nprob = nprob; V.nloc = nloc; V.row0 = row0; V.nbins = nbins; V.nb = nb; V.part = d_part;
    V.bias_pad = bias_pad; V.marg_local = marg_local; V.marg = marg; V.queue = A.queue; V.iter = d_book + nprob + 2;
    V.done_at = d_book; V.n_done = d_book + nprob; V.nonempty = nonempty; V.results = results; V.tol = P->tol; V.max_iters = P->max_iters;

    const size_t smem = (size_t)CB * sizeof(double);
    HC_CUDA(cudaFuncSetAttribute(csrb_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaFuncSetAttribute(csrb_stream_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    int rc = HC_OK;
    auto one_iteration = [&](cudaEvent_t t0, cudaEvent_t t1, unsigned flags) -> int {
        if (nloc > 0 && nitems > 0) {
            if (t0) cudaEventRecordWithFlags(t0, s, flags);
            csrb_stream_kernel<<<grid, ST_THREADS, smem, s>>>(A);
            if (t1) cudaEventRecordWithFlags(t1, s, flags);
            csrb_marg_kernel<<<(unsigned)((nloc + 255) / 256), 256, 0, s>>>(V);
        } else {
            csrb_open_iter_kernel<<<1, 32, 0, s>>>(V);
        }
        if (nccl_comm) {
            const int r = hc_nccl_allreduce_f64(nccl_comm, marg_local, marg, (size_t)nbins, s);
            if (r != HC_OK) return r;
        }
        csrb_update_kernel<<<nprob * UPD_CLUSTER, UPD_THREADS, 0, s>>>(V);
        return HC_OK;
    };
    const int poll = P->poll_every > 0 ? std::min(P->poll_every, 4) : 4;
    const int per_iter = (nloc > 0 && nitems > 0 ? 2 : 1) + 1;
    cudaEvent_t tk0 = nullptr, tk1 = nullptr;
    struct TkGuard { cudaEvent_t* a; cudaEvent_t* b; ~TkGuard() { if (*a) cudaEventDestroy(*a); if (*b) cudaEventDestroy(*b); } } tkg{&tk0, &tk1};
    if (h_info != nullptr && getenv("HC_ICE_TIME_KERNEL") != nullptr && atoi(getenv("HC_ICE_TIME_KERNEL")) != 0) {
        if (cudaEventCreate(&tk0) != cudaSuccess || cudaEventCreate(&tk1) != cudaSuccess) { tk0 = nullptr; tk1 = nullptr; (void)cudaGetLastError(); }
    }
    bool use_graph = true;
    if (const char* e = getenv("HC_ICE_GRAPH")) use_graph = atoi(e) != 0;
    cudaGraphExec_t gexec = nullptr;
    if (use_graph) {
        cudaGraph_t graph = nullptr;
        cudaError_t e = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal);
        if (e == cudaSuccess) {
            for (int i = 0; i < poll && rc == HC_OK; ++i)
                rc = one_iteration(i == 0 ? tk0 : nullptr, i == 0 ? tk1 : nullptr, cudaEventRecordExternal);
            e = cudaStreamEndCapture(s, &graph);
        }
        if (rc != HC_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e == cudaSuccess) e = cudaGraphInstantiate(&gexec, graph, 0);
        if (graph) cudaGraphDestroy(graph);
        if (e != cudaSuccess) { gexec = nullptr; (void)cudaGetLastError(); }
    }
    tick("graph capture");
    if (h_info && ev0) cudaEventRecord(ev0, s);
    int launches = 0, h_done = 0;
    double stream_ms_sum = 0.0;
    int stream_ms_n = 0;
    for (int k0 = 0; k0 < P->max_iters && rc == HC_OK; k0 += poll) {
        cudaError_t e = cudaSuccess;
        if (gexec) e = cudaGraphLaunch(gexec, s);
        else for (int i = 0; i < poll && rc == HC_OK; ++i) rc = one_iteration(i == 0 ? tk0 : nullptr, i == 0 ? tk1 : nullptr, cudaEventRecordDefault);
        if (rc != HC_OK) break;
        hc_count_launch(per_iter * poll);
        launches += per_iter * poll;
        if (e == cudaSuccess) e = cudaGetLastError();
        if (e == cudaSuccess) e = hc_read_small(&h_done, V.n_done, sizeof(int32_t), s);
        if (e == cudaSuccess && tk0 && nloc > 0 && nitems > 0) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, tk0, tk1) == cudaSuccess) { stream_ms_sum += ms; ++stream_ms_n; } else (void)cudaGetLastError();
        }
        if (e != cudaSuccess) { hc_set_error("hc_ice_csr_balance (blocked): %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; break; }
        if (h_done >= nonempty) break;
    }
    if (h_info && ev1) cudaEventRecord(ev1, s);
    if (gexec) cudaGraphExecDestroy(gexec);
    if (rc == HC_OK) {
        csrb_finalize_kernel<<<(unsigned)((nbins + 255) / 256), 256, 0, s>>>(bin_off, nprob, results, P->rescale_marginals, bias_pad, bias);
        hc_count_launch(); ++launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { hc_set_error("hc_ice_csr_balance (blocked): %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; }
    }
    cudaError_t e = cudaStreamSynchronize(s);
    if (rc == HC_OK && e != cudaSuccess) { hc_set_error("hc_ice_csr_balance (blocked): %s", cudaGetErrorString(e)); rc = HC_ERR_CUDA; }
    if (h_info) {
        h_info->launches = launches;
        h_info->packed = 2;                          // column-blocked 4-byte entries
        h_info->overflow_cells = total_ent;          // stored entries incl. padding: 4 B each streamed per iteration
        if (ev0 && e == cudaSuccess) cudaEventElapsedTime(&h_info->loop_ms, ev0, ev1);
        if (evb0 && e == cudaSuccess) cudaEventElapsedTime(&h_info->pack_ms, evb0, evb1);
        h_info->stream_full_launches = stream_ms_n;
        h_info->stream_full_ms = stream_ms_n ? (float)(stream_ms_sum / stream_ms_n) : 0.f;
    }
    return rc;
}
