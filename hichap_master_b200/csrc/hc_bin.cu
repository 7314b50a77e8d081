// (a) Valid-pair binning into dense int32 tiles + dense->sparse marshalling.
// Replaces the interpreted per-line loops of HiCHap/matrixBuilding.py:568-603 (traditional),
// :817-852 (traditional-in-allelic), :1131-1161 / :1169-1199 (M_M / P_P 'Both'),
// :1207-1243 (M_P / P_M), :1284-1301 / :1398-1415 (one-sided R1/R2), and the np.triu/np.nonzero
// marshalling at :457-524.
//
// Roofline: HBM-bound streaming read of the columnar pairs (16 B/pair, +1 B mark) with 128-bit
// loads; the += 1 updates are 32-bit RED atomics resolved in L2 (not HBM traffic).
#include <algorithm>
#include <stdlib.h>
#include "hc_common.cuh"

namespace {

constexpr int BIN_THREADS = 256;
constexpr int PAIRS_PER_THREAD = 4;  // one int4 per column per thread

struct PairCols {
    const int32_t* c1; const int32_t* p1; const int32_t* c2; const int32_t* p2; const uint8_t* mark;
};

__device__ __forceinline__ bool mode_accepts(int mode, int mk) {
    // HC_BIN_SYM_ALL: everything; SYM_BOTH: mark==Both only; ONESIDED: mark!=Both only
    return mode == HC_BIN_SYM_ALL || (mode == HC_BIN_SYM_BOTH ? mk == 0 : mk != 0);
}

template <bool WHOLE>
__device__ __forceinline__ void apply_pair(int c1, int p1, int c2, int p2, int mk, FastDiv res, int mode,
                                           int32_t* __restrict__ mats, const int64_t* __restrict__ t0,
                                           const int64_t* __restrict__ t1, const int32_t* __restrict__ mat_n,
                                           const int32_t* __restrict__ mat_ld, int nchrom, int64_t whole_ld,
                                           int32_t whole_n, unsigned long long* oob) {
    if (c1 < 0 || c2 < 0 || c1 >= nchrom || c2 >= nchrom) return;   // filtered chromosome
    if (!mode_accepts(mode, mk)) return;
    if ((!WHOLE || mode == HC_BIN_ONESIDED) && c1 != c2) return;     // cis only
    if (p1 < 0 || p2 < 0) { if (oob) atomicAdd(oob, 1ull); return; }
    int64_t b1 = fast_div((uint32_t)p1, res), b2 = fast_div((uint32_t)p2, res);
    int32_t* M;
    int64_t ld, n;
    if (WHOLE) {
        b1 += t0[c1]; b2 += t1[c2];
        M = mats; ld = whole_ld; n = whole_n;
    } else {
        M = mats + t0[c1]; ld = mat_ld[c1]; n = mat_n[c1];
    }
    if (b1 >= n || b2 >= n) { if (oob) atomicAdd(oob, 1ull); return; }
    if (mode == HC_BIN_ONESIDED) {
        // R1: row = first mate; anything else (R2): row = second mate  (matrixBuilding.py:1298-1301)
        if (mk == 1) atomicAdd(&M[b1 * ld + b2], 1); else atomicAdd(&M[b2 * ld + b1], 1);
    } else {
        atomicAdd(&M[b1 * ld + b2], 1);
        if (b1 != b2) atomicAdd(&M[b2 * ld + b1], 1);
    }
}

template <bool WHOLE>
__global__ void __launch_bounds__(BIN_THREADS)
bin_pairs_kernel(PairCols in, int64_t npairs, FastDiv res, int mode, int32_t* __restrict__ mats,
                 const int64_t* __restrict__ t0, const int64_t* __restrict__ t1,
                 const int32_t* __restrict__ mat_n, const int32_t* __restrict__ mat_ld, int nchrom,
                 int64_t whole_ld, int32_t whole_n, unsigned long long* oob) {
    const int64_t nvec = npairs / PAIRS_PER_THREAD;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += stride) {
        const int4 a = ld_stream_v4(in.c1 + 4 * v), b = ld_stream_v4(in.p1 + 4 * v);
        const int4 c = ld_stream_v4(in.c2 + 4 * v), d = ld_stream_v4(in.p2 + 4 * v);
        uint32_t mk4 = 0;
        if (in.mark) mk4 = *reinterpret_cast<const uint32_t*>(in.mark + 4 * v);
        apply_pair<WHOLE>(a.x, b.x, c.x, d.x, mk4 & 255, res, mode, mats, t0, t1, mat_n, mat_ld, nchrom, whole_ld, whole_n, oob);
        apply_pair<WHOLE>(a.y, b.y, c.y, d.y, (mk4 >> 8) & 255, res, mode, mats, t0, t1, mat_n, mat_ld, nchrom, whole_ld, whole_n, oob);
        apply_pair<WHOLE>(a.z, b.z, c.z, d.z, (mk4 >> 16) & 255, res, mode, mats, t0, t1, mat_n, mat_ld, nchrom, whole_ld, whole_n, oob);
        apply_pair<WHOLE>(a.w, b.w, c.w, d.w, (mk4 >> 24) & 255, res, mode, mats, t0, t1, mat_n, mat_ld, nchrom, whole_ld, whole_n, oob);
    }
    // ragged tail (< 4 pairs)
    if (blockIdx.x == 0 && threadIdx.x < (int)(npairs - nvec * PAIRS_PER_THREAD)) {
        const int64_t i = nvec * PAIRS_PER_THREAD + threadIdx.x;
        apply_pair<WHOLE>(in.c1[i], in.p1[i], in.c2[i], in.p2[i], in.mark ? in.mark[i] : 0, res, mode, mats, t0, t1,
                          mat_n, mat_ld, nchrom, whole_ld, whole_n, oob);
    }
}

int bin_grid(int64_t npairs) {
    int64_t nvec = (npairs + PAIRS_PER_THREAD - 1) / PAIRS_PER_THREAD;
    int64_t blocks = (nvec + BIN_THREADS - 1) / BIN_THREADS;
    int64_t cap = (int64_t)hc_num_sms() * 8;  // 8 resident CTAs of 256 threads per SM
    if (blocks > cap) blocks = cap;
    return blocks < 1 ? 1 : (int)blocks;
}

bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- dense -> sparse -------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
row_nonzero_count_kernel(const T* __restrict__ M, int64_t ld, int nrows, int ncols, int triu,
                         int64_t* __restrict__ row_cnt) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nrows) return;
    const T* row = M + (int64_t)warp * ld;
    int cnt = 0;
    for (int j = (triu ? warp : 0) + lane; j < ncols; j += 32) cnt += (row[j] != T(0));
    cnt = warp_sum_i(cnt);
    if (lane == 0) row_cnt[warp] = cnt;
}

// single-CTA exclusive scan of row_cnt[0..n) in place, total to row_cnt[n]
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(int64_t* __restrict__ v, int n) {
    __shared__ long long warp_tot[32];
    __shared__ long long carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int base = 0; base < n; base += 1024) {
        const int i = base + threadIdx.x;
        long long x = i < n ? v[i] : 0, incl = x;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            long long y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) warp_tot[wid] = incl;
        __syncthreads();
        long long woff = 0;
        for (int w = 0; w < wid; ++w) woff += warp_tot[w];
        const long long carry = carry_s;
        if (i < n) v[i] = carry + woff + incl - x;
        __syncthreads();
        if (threadIdx.x == 1023) carry_s = carry + woff + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) v[n] = carry_s;
}

template <typename T>
__global__ void __launch_bounds__(256)
row_nonzero_extract_kernel(const T* __restrict__ M, int64_t ld, int nrows, int ncols, int triu,
                           const int64_t* __restrict__ row_ptr, int32_t* __restrict__ bin1,
                           int32_t* __restrict__ bin2, T* __restrict__ val) {
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (warp >= nrows) return;
    const T* row = M + (int64_t)warp * ld;
    int64_t out = row_ptr[warp];
    const int j0 = triu ? warp : 0;
    for (int base = j0; base < ncols; base += 32) {   // ascending columns: row-major order
        const int j = base + lane;
        T x = j < ncols ? row[j] : T(0);
        const unsigned m = __ballot_sync(0xffffffffu, x != T(0));
        if (x != T(0)) {
            const int64_t o = out + __popc(m & ((1u << lane) - 1u));
            bin1[o] = warp; bin2[o] = j; val[o] = x;
        }
        out += __popc(m);
    }
}

__device__ __forceinline__ int batch_problem(const int64_t* __restrict__ bin_off, int nprob, int64_t g) {
    int lo = 0, hi = nprob - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (bin_off[mid] <= g) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// ---- banded binning: near-diagonal updates land in an L2-resident band accumulator --------
// The direct kernel above is bound by random DRAM read-modify-write: += 1 scattered over 1.2 GB of
// tiles misses L2 on almost every update (ncu, profiles/r1a: 31 GB of DRAM traffic for 6.4 GB of
// pairs, 13.7 ms).  Hi-C contacts concentrate near the diagonal (P(s) ~ 1/s), so here each pair
// updates only the UPPER triangle, and pairs whose bins are fewer than BW apart go to a compact
// band accumulator band[global_row][d] (nbins x BW int32: 39 MB at 40 kb with BW = 128) that
// stays resident in the 126 MB L2; only the far pairs touch the big tiles.  A merge pass adds
// the band into the tiles (coalesced 512-byte row segments) and a tile-transpose pass mirrors
// upper -> lower.  (A two-pass radix partition by chromosome / row block was measured first --
// profiles/r1c, r1d -- and lost to this single pass.)
struct BandArgs {
    PairCols in; long long npairs; FastDiv res; int mode; int nchrom;
    int32_t* mats; const int64_t* mat_off; const int32_t* mat_n; const int32_t* mat_ld;
    const int64_t* bin_off;              // global row offset of each chromosome
    int32_t* band; int bw_shift;         // band[(global_row << bw_shift) + d], d < (1 << bw_shift)
    unsigned long long* oob;
};

__device__ __forceinline__ void band_apply(const BandArgs& a, int c1, int p1, int c2, int p2, int mk,
                                           unsigned long long& my_oob, uint64_t keep) {
    if (c1 < 0 || c1 != c2 || c1 >= a.nchrom) return;
    if (!mode_accepts(a.mode, mk)) return;
    if (p1 < 0 || p2 < 0) { ++my_oob; return; }
    const uint32_t b1 = fast_div((uint32_t)p1, a.res), b2 = fast_div((uint32_t)p2, a.res), n = (uint32_t)a.mat_n[c1];
    if (b1 >= n || b2 >= n) { ++my_oob; return; }
    const uint32_t lo = min(b1, b2), d = max(b1, b2) - lo;
    if ((d >> a.bw_shift) == 0) red_add_s32_hint(a.band + (((a.bin_off[c1] + lo) << a.bw_shift) + d), 1, keep);
    else atomicAdd(a.mats + a.mat_off[c1] + (int64_t)lo * a.mat_ld[c1] + (lo + d), 1);
}

// U8: the chromosome columns are the uint8 columns a host parser ships over PCIe (255 = filtered,
// rejected by the c1 >= nchrom test), read 4 at a time as one word
template <bool U8>
__global__ void __launch_bounds__(BIN_THREADS) bin_pairs_band_kernel(BandArgs a) {
    const int64_t nvec = a.npairs / PAIRS_PER_THREAD;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long my_oob = 0;
    const uint64_t once = l2_policy_evict_first(), keep = l2_policy_evict_last();   // pairs stream through; the band stays
    const uint8_t* c1b = reinterpret_cast<const uint8_t*>(a.in.c1);
    const uint8_t* c2b = reinterpret_cast<const uint8_t*>(a.in.c2);
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += stride) {
        int4 c1, c2;
        if (U8) {
            const uint32_t w1 = *reinterpret_cast<const uint32_t*>(c1b + 4 * v), w2 = *reinterpret_cast<const uint32_t*>(c2b + 4 * v);
            c1 = make_int4(w1 & 255, (w1 >> 8) & 255, (w1 >> 16) & 255, w1 >> 24);
            c2 = make_int4(w2 & 255, (w2 >> 8) & 255, (w2 >> 16) & 255, w2 >> 24);
        } else {
            c1 = ld_stream_v4_hint(a.in.c1 + 4 * v, once);
            c2 = ld_stream_v4_hint(a.in.c2 + 4 * v, once);
        }
        const int4 p1 = ld_stream_v4_hint(a.in.p1 + 4 * v, once), p2 = ld_stream_v4_hint(a.in.p2 + 4 * v, once);
        uint32_t mk = 0;
        if (a.in.mark) mk = *reinterpret_cast<const uint32_t*>(a.in.mark + 4 * v);
        band_apply(a, c1.x, p1.x, c2.x, p2.x, mk & 255, my_oob, keep);
        band_apply(a, c1.y, p1.y, c2.y, p2.y, (mk >> 8) & 255, my_oob, keep);
        band_apply(a, c1.z, p1.z, c2.z, p2.z, (mk >> 16) & 255, my_oob, keep);
        band_apply(a, c1.w, p1.w, c2.w, p2.w, (mk >> 24) & 255, my_oob, keep);
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(a.npairs - nvec * PAIRS_PER_THREAD)) {
        const int64_t i = nvec * PAIRS_PER_THREAD + threadIdx.x;
        const int x = U8 ? (int)c1b[i] : a.in.c1[i], y = U8 ? (int)c2b[i] : a.in.c2[i];
        band_apply(a, x, a.in.p1[i], y, a.in.p2[i], a.in.mark ? a.in.mark[i] : 0, my_oob, keep);
    }
    if (a.oob) {
        my_oob = (unsigned long long)warp_sum_ll((long long)my_oob);
        if ((threadIdx.x & 31) == 0 && my_oob) atomicAdd(a.oob, my_oob);
    }
}

// ---- hot-diagonal variant: the hottest diagonals are counted in SHARED MEMORY ----------------------------------
// The banded kernel above is bound by the L2 atomic rate (~80 G RED/s measured: 400 M pairs = 5 ms).  Half of all
// Hi-C pairs fall on the first few diagonals (P(s) ~ 1/s), so every CTA keeps 16-bit counters for the diagonals
// d < d_hot of EVERY bin in its own 200 KB of shared memory (100 K counters: the main diagonal of the 75 918 bins of
// hg19 at 40 kb): a pair on a hot diagonal becomes one shared-memory atomic, and only the other pairs go to L2 (band)
// / DRAM (far pairs).  At the end of the launch every CTA adds its non-zero counters into the band.  A counter that
// reaches 0x8000 is drained into the band by the thread that saw it cross (only the 1024 threads of the CTA can add in
// between, so the 16-bit field never carries into its neighbour).
constexpr int HOT_THREADS = 1024;
constexpr int HOT_PER_CTA = 100 * 1024;          // 16-bit counters per CTA (200 KB of shared memory)
constexpr int HOT_MAX_D = 16;

template <bool U8>
__global__ void __launch_bounds__(HOT_THREADS, 1) bin_pairs_band_hot_kernel(BandArgs a) {
    extern __shared__ __align__(16) uint32_t hot[];          // HOT_PER_CTA / 2 words
    const long long nbins = a.bin_off[a.nchrom];
    const int d_hot = (int)min((long long)HOT_MAX_D, nbins > 0 ? (long long)HOT_PER_CTA / nbins : 0ll);
    for (int i = threadIdx.x; i < HOT_PER_CTA / 2; i += blockDim.x) hot[i] = 0u;
    __syncthreads();
    const int64_t nvec = a.npairs / PAIRS_PER_THREAD;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x;
    unsigned long long my_oob = 0;
    const uint64_t once = l2_policy_evict_first(), keep = l2_policy_evict_last();
    const uint8_t* c1b = reinterpret_cast<const uint8_t*>(a.in.c1);
    const uint8_t* c2b = reinterpret_cast<const uint8_t*>(a.in.c2);
    auto apply = [&](int c1, int p1, int c2, int p2, int mk) {
        if (c1 < 0 || c1 != c2 || c1 >= a.nchrom) return;
        if (!mode_accepts(a.mode, mk)) return;
        if (p1 < 0 || p2 < 0) { ++my_oob; return; }
        const uint32_t b1 = fast_div((uint32_t)p1, a.res), b2 = fast_div((uint32_t)p2, a.res), n = (uint32_t)a.mat_n[c1];
        if (b1 >= n || b2 >= n) { ++my_oob; return; }
        const uint32_t lo = min(b1, b2), d = max(b1, b2) - lo;
        const long long grow = a.bin_off[c1] + lo;
        if ((int)d < d_hot) {
            const unsigned idx = (unsigned)(grow * d_hot + d);
            uint32_t* w = hot + (idx >> 1);
            const unsigned sh = (idx & 1u) * 16u;
            const uint32_t old = atomicAdd(w, 1u << sh);
            if (((old >> sh) & 0xffffu) == 0x7fffu) {          // this add made it 0x8000: drain that much into the band
                atomicSub(w, 0x8000u << sh);
                red_add_s32_hint(a.band + ((grow << a.bw_shift) + d), 0x8000, keep);
            }
        } else if ((d >> a.bw_shift) == 0) red_add_s32_hint(a.band + ((grow << a.bw_shift) + d), 1, keep);
        else atomicAdd(a.mats + a.mat_off[c1] + (int64_t)lo * a.mat_ld[c1] + (lo + d), 1);
    };
    for (int64_t v = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += stride) {
        int4 c1, c2;
        if (U8) {
            const uint32_t w1 = *reinterpret_cast<const uint32_t*>(c1b + 4 * v), w2 = *reinterpret_cast<const uint32_t*>(c2b + 4 * v);
            c1 = make_int4(w1 & 255, (w1 >> 8) & 255, (w1 >> 16) & 255, w1 >> 24);
            c2 = make_int4(w2 & 255, (w2 >> 8) & 255, (w2 >> 16) & 255, w2 >> 24);
        } else {
            c1 = ld_stream_v4_hint(a.in.c1 + 4 * v, once);
            c2 = ld_stream_v4_hint(a.in.c2 + 4 * v, once);
        }
        const int4 p1 = ld_stream_v4_hint(a.in.p1 + 4 * v, once), p2 = ld_stream_v4_hint(a.in.p2 + 4 * v, once);
        uint32_t mk = 0;
        if (a.in.mark) mk = *reinterpret_cast<const uint32_t*>(a.in.mark + 4 * v);
        apply(c1.x, p1.x, c2.x, p2.x, mk & 255);
        apply(c1.y, p1.y, c2.y, p2.y, (mk >> 8) & 255);
        apply(c1.z, p1.z, c2.z, p2.z, (mk >> 16) & 255);
        apply(c1.w, p1.w, c2.w, p2.w, (mk >> 24) & 255);
    }
    if (blockIdx.x == 0 && threadIdx.x < (int)(a.npairs - nvec * PAIRS_PER_THREAD)) {
        const int64_t i = nvec * PAIRS_PER_THREAD + threadIdx.x;
        const int x = U8 ? (int)c1b[i] : a.in.c1[i], y = U8 ? (int)c2b[i] : a.in.c2[i];
        apply(x, a.in.p1[i], y, a.in.p2[i], a.in.mark ? a.in.mark[i] : 0);
    }
    __syncthreads();           // every add has landed; nobody touches the counters any more
    if (d_hot > 0) {
        for (int i = threadIdx.x; i < HOT_PER_CTA / 2; i += blockDim.x) {
            const uint32_t w = hot[i];
            if (w == 0u) continue;
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int v = (int)((w >> (16 * h)) & 0xffffu);
                if (v) {
                    const unsigned idx = 2u * i + h;
                    const long long grow = idx / d_hot;
                    const int d = (int)(idx - grow * d_hot);
                    if (grow < nbins) red_add_s32_hint(a.band + ((grow << a.bw_shift) + d), v, keep);
                }
            }
        }
    }
    if (a.oob) {
        my_oob = (unsigned long long)warp_sum_ll((long long)my_oob);
        if ((threadIdx.x & 31) == 0 && my_oob) atomicAdd(a.oob, my_oob);
    }
}

// tiles[r][r + d] += band[r][d]: one warp per global row, coalesced on both sides
__global__ void __launch_bounds__(256) band_merge_kernel(BandArgs a, int64_t nbins) {
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= nbins) return;
    const int p = batch_problem(a.bin_off, a.nchrom, g);
    const int r = (int)(g - a.bin_off[p]), n = a.mat_n[p], bw = 1 << a.bw_shift;
    int32_t* row = a.mats + a.mat_off[p] + (int64_t)r * a.mat_ld[p] + r;
    const int32_t* b = a.band + (g << a.bw_shift);
    for (int d = lane; d < bw && r + d < n; d += 32) {
        const int v = b[d];
        if (v) row[d] += v;
    }
}

constexpr int PART_MAX_BUCKETS = 256;   // (bounds the by-value table of the mirror kernel)

// lower = transpose(upper) for every matrix of the batch (32x32 tiles through shared memory)
struct MirrorTab { int nprob; int start[PART_MAX_BUCKETS + 1]; };   // prefix of T_p(T_p+1)/2 tile pairs per matrix

__global__ void __launch_bounds__(256)
mirror_upper_kernel(int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off, const int32_t* __restrict__ mat_n,
                    const int32_t* __restrict__ mat_ld, MirrorTab tab) {
    __shared__ int32_t t[32][33];
    int p = 0;
    {
        int lo = 0, hi = tab.nprob - 1;
        while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (tab.start[mid] <= (int)blockIdx.x) lo = mid; else hi = mid - 1; }
        p = lo;
    }
    const int n = mat_n[p];
    // destination tile (row block I, col block J), I >= J, enumerated row by row
    const int idx = blockIdx.x - tab.start[p];
    int I = (int)((sqrtf(8.0f * idx + 1.0f) - 1.0f) * 0.5f);
    while (I * (I + 1) / 2 > idx) --I;
    while ((I + 1) * (I + 2) / 2 <= idx) ++I;
    const int J = idx - I * (I + 1) / 2;
    int32_t* M = mats + mat_off[p];
    const int64_t ld = mat_ld[p];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 8 rows per pass
#pragma unroll
    for (int r = ty; r < 32; r += 8) {               // source tile (J, I): rows J*32.., cols I*32..
        const int sr = J * 32 + r, sc = I * 32 + tx;
        t[r][tx] = (sr < n && sc < n) ? M[(int64_t)sr * ld + sc] : 0;
    }
    __syncthreads();
#pragma unroll
    for (int r = ty; r < 32; r += 8) {
        const int dr = I * 32 + r, dc = J * 32 + tx;
        if (dr < n && dc < n && dr > dc) M[(int64_t)dr * ld + dc] = t[tx][r];
    }
}

// ---- whole batch at once: upper-triangular records in the reference's 24-byte layout ------
struct Rec24 { long long bin1; long long bin2; double IF; };   // matrixBuilding.py:460-461 S_dtype

__global__ void __launch_bounds__(256)
batch_triu_count_kernel(const int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off,
                        const int32_t* __restrict__ mat_n, const int32_t* __restrict__ mat_ld,
                        const int64_t* __restrict__ bin_off, int nprob, int64_t* __restrict__ row_cnt) {
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;   // one warp per (global) row
    const int lane = threadIdx.x & 31;
    if (g >= bin_off[nprob]) return;
    const int p = batch_problem(bin_off, nprob, g);
    const int r = (int)(g - bin_off[p]), n = mat_n[p];
    const int32_t* row = mats + mat_off[p] + (int64_t)r * mat_ld[p];
    int cnt = 0;
    for (int j = r + lane; j < n; j += 32) cnt += (row[j] != 0);
    cnt = warp_sum_i(cnt);
    if (lane == 0) row_cnt[g] = cnt;
}

__global__ void __launch_bounds__(256)
batch_triu_records_kernel(const int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off,
                          const int32_t* __restrict__ mat_n, const int32_t* __restrict__ mat_ld,
                          const int64_t* __restrict__ bin_off, int nprob, const int64_t* __restrict__ row_ptr,
                          Rec24* __restrict__ rec) {
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= bin_off[nprob]) return;
    const int p = batch_problem(bin_off, nprob, g);
    const int r = (int)(g - bin_off[p]), n = mat_n[p];
    const int32_t* row = mats + mat_off[p] + (int64_t)r * mat_ld[p];
    int64_t out = row_ptr[g];
    for (int base = r; base < n; base += 32) {
        const int j = base + lane;
        const int x = j < n ? row[j] : 0;
        const unsigned m = __ballot_sync(0xffffffffu, x != 0);
        if (x != 0) {
            Rec24 v; v.bin1 = r; v.bin2 = j; v.IF = (double)x;
            rec[out + __popc(m & ((1u << lane) - 1u))] = v;
        }
        out += __popc(m);
    }
}

// multi-CTA exclusive scan is not needed: bins are O(1e5); one CTA with a 64-bit carry
}  // namespace

extern "C" int hc_dense_batch_triu_count(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                         const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                                         int64_t nbins, int64_t* row_ptr, void* stream) {
    HC_REQUIRE(nprob > 0 && nbins >= 0, "nprob>0, nbins>=0");
    cudaStream_t s = (cudaStream_t)stream;
    if (nbins > 0) {
        const int64_t blocks = (nbins * 32 + 255) / 256;
        batch_triu_count_kernel<<<(unsigned)blocks, 256, 0, s>>>(mats, mat_off, mat_n, mat_ld, bin_off, nprob, row_ptr);
        HC_LAUNCH_CHECK();
    }
    HC_REQUIRE(nbins < (1ll << 31), "too many bins for the single-CTA scan");
    exclusive_scan_kernel<<<1, 1024, 0, s>>>(row_ptr, (int)nbins);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_dense_batch_triu_records(const int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                           const int32_t* mat_ld, const int64_t* bin_off, int32_t nprob,
                                           int64_t nbins, const int64_t* row_ptr, void* records, void* stream) {
    HC_REQUIRE(nprob > 0 && nbins >= 0, "nprob>0, nbins>=0");
    if (nbins == 0) return HC_OK;
    const int64_t blocks = (nbins * 32 + 255) / 256;
    batch_triu_records_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        mats, mat_off, mat_n, mat_ld, bin_off, nprob, row_ptr, reinterpret_cast<Rec24*>(records));
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_bin_pairs_local(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                                  const uint8_t* mark, int64_t npairs, int32_t res, int32_t mode, int32_t* mats,
                                  const int64_t* mat_off, const int32_t* mat_n, const int32_t* mat_ld,
                                  int32_t nchrom, unsigned long long* oob, void* stream) {
    HC_REQUIRE(npairs >= 0 && res > 0 && nchrom > 0, "npairs>=0, res>0, nchrom>0");
    HC_REQUIRE(mode >= HC_BIN_SYM_ALL && mode <= HC_BIN_ONESIDED, "mode");
    if (npairs == 0) return HC_OK;
    HC_REQUIRE(mode == HC_BIN_SYM_ALL || mark != nullptr, "mark column required for this mode");
    HC_REQUIRE(aligned16(c1) && aligned16(p1) && aligned16(c2) && aligned16(p2), "pair columns must be 16-byte aligned");
    HC_REQUIRE(mark == nullptr || (reinterpret_cast<uintptr_t>(mark) & 3u) == 0, "mark must be 4-byte aligned");
    PairCols in{c1, p1, c2, p2, mark};
    bin_pairs_kernel<false><<<bin_grid(npairs), BIN_THREADS, 0, (cudaStream_t)stream>>>(
        in, npairs, make_fast_div((uint32_t)res), mode, mats, mat_off, nullptr, mat_n, mat_ld, nchrom, 0, 0, oob);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

// Banded variant of hc_bin_pairs_local for the SYMMETRIC modes on matrices that are symmetric on
// entry (e.g. freshly zeroed): same result, most atomics resolved in L2.
extern "C" int64_t hc_bin_band_work_bytes(int64_t nbins, int32_t band_width) {
    return (int64_t)sizeof(int32_t) * (nbins > 0 ? nbins : 1) * band_width;
}

namespace {
int band_shift(int band_width) { int sh = 0; while ((1 << sh) < band_width) ++sh; return sh; }
bool band_width_ok(int bw) { return bw >= 32 && bw <= 1024 && (bw & (bw - 1)) == 0; }
}  // namespace

// The three phases of banded binning, separately callable so that pairs can be accumulated chunk by
// chunk while later chunks are still crossing PCIe: begin (zero the band) -> accumulate xN -> finish
// (merge the band into the tiles, mirror upper -> lower).
extern "C" int hc_bin_band_begin(void* work, int64_t nbins, int32_t band_width, void* stream) {
    HC_REQUIRE(nbins >= 0 && band_width_ok(band_width), "band_width: power of two in [32,1024]");
    if (nbins == 0) return HC_OK;
    HC_REQUIRE(work != nullptr, "work");
    HC_CUDA(cudaMemsetAsync(work, 0, sizeof(int32_t) * (size_t)nbins * band_width, (cudaStream_t)stream));
    return HC_OK;
}

extern "C" int hc_bin_band_accumulate(const void* c1, const int32_t* p1, const void* c2, const int32_t* p2,
                                      const uint8_t* mark, int64_t npairs, int32_t chrom_is_u8, int32_t res, int32_t mode,
                                      int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                      const int32_t* mat_ld, const int64_t* bin_off, int32_t nchrom,
                                      int32_t band_width, unsigned long long* oob, void* work, void* stream) {
    HC_REQUIRE(npairs >= 0 && res > 0 && nchrom > 0, "npairs>=0, res>0, nchrom>0");
    HC_REQUIRE(mode == HC_BIN_SYM_ALL || mode == HC_BIN_SYM_BOTH, "banded binning is for the symmetric modes");
    HC_REQUIRE(band_width_ok(band_width), "band_width: power of two in [32,1024]");
    HC_REQUIRE(!chrom_is_u8 || nchrom <= 255, "uint8 chromosome columns hold at most 255 chromosomes");
    if (npairs == 0) return HC_OK;
    HC_REQUIRE(mode == HC_BIN_SYM_ALL || mark != nullptr, "mark column required for this mode");
    HC_REQUIRE(aligned16(p1) && aligned16(p2), "position columns must be 16-byte aligned");
    if (chrom_is_u8) HC_REQUIRE(((reinterpret_cast<uintptr_t>(c1) | reinterpret_cast<uintptr_t>(c2)) & 3u) == 0, "uint8 chromosome columns must be 4-byte aligned");
    else HC_REQUIRE(aligned16(c1) && aligned16(c2), "pair columns must be 16-byte aligned");
    HC_REQUIRE(mark == nullptr || (reinterpret_cast<uintptr_t>(mark) & 3u) == 0, "mark must be 4-byte aligned");
    cudaStream_t s = (cudaStream_t)stream;
    BandArgs a;
    a.in = PairCols{reinterpret_cast<const int32_t*>(c1), p1, reinterpret_cast<const int32_t*>(c2), p2, mark};
    a.npairs = npairs; a.res = make_fast_div((uint32_t)res); a.mode = mode;
    a.nchrom = nchrom; a.mats = mats; a.mat_off = mat_off; a.mat_n = mat_n; a.mat_ld = mat_ld; a.bin_off = bin_off;
    a.band = reinterpret_cast<int32_t*>(work); a.oob = oob;
    a.bw_shift = band_shift(band_width);
    // large inputs: every CTA counts the hottest diagonals in 16-bit shared-memory counters of its own and drains them
    // into the band at the end (measured on C2: binning 5.50 -> 5.39 ms, step 12.92 -> 12.76 ms, twice in a row)
    if (npairs >= (1 << 20)) {
        auto kern = chrom_is_u8 ? bin_pairs_band_hot_kernel<true> : bin_pairs_band_hot_kernel<false>;
        const size_t smem = (size_t)HOT_PER_CTA * 2;
        HC_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<hc_num_sms(), HOT_THREADS, smem, s>>>(a);      // one CTA per SM
        HC_LAUNCH_CHECK();
        return HC_OK;
    }
    if (chrom_is_u8) bin_pairs_band_kernel<true><<<bin_grid(npairs), BIN_THREADS, 0, s>>>(a);
    else bin_pairs_band_kernel<false><<<bin_grid(npairs), BIN_THREADS, 0, s>>>(a);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_bin_band_finish(int32_t* mats, const int64_t* mat_off, const int32_t* mat_n, const int32_t* mat_ld,
                                  const int64_t* bin_off, int32_t nchrom, const int32_t* h_mat_n, int32_t band_width,
                                  void* work, void* stream) {
    HC_REQUIRE(nchrom > 0 && nchrom <= PART_MAX_BUCKETS && h_mat_n != nullptr, "at most 256 chromosomes; h_mat_n");
    HC_REQUIRE(band_width_ok(band_width), "band_width: power of two in [32,1024]");
    MirrorTab mtab;
    mtab.nprob = nchrom;
    mtab.start[0] = 0;
    int64_t nbins = 0;
    for (int p = 0; p < nchrom; ++p) {
        HC_REQUIRE(h_mat_n[p] >= 0, "matrix side");
        nbins += h_mat_n[p];
        const long long T = (h_mat_n[p] + 31) / 32;
        const long long nxt = mtab.start[p] + T * (T + 1) / 2;
        HC_REQUIRE(nxt < (1ll << 31), "too many tiles");
        mtab.start[p + 1] = (int)nxt;
    }
    if (nbins == 0) return HC_OK;
    cudaStream_t s = (cudaStream_t)stream;
    BandArgs a{};
    a.nchrom = nchrom; a.mats = mats; a.mat_off = mat_off; a.mat_n = mat_n; a.mat_ld = mat_ld; a.bin_off = bin_off;
    a.band = reinterpret_cast<int32_t*>(work);
    a.bw_shift = band_shift(band_width);
    band_merge_kernel<<<(unsigned)((nbins * 32 + 255) / 256), 256, 0, s>>>(a, nbins);
    HC_LAUNCH_CHECK();
    if (mtab.start[nchrom] > 0) {
        mirror_upper_kernel<<<mtab.start[nchrom], 256, 0, s>>>(mats, mat_off, mat_n, mat_ld, mtab);
        HC_LAUNCH_CHECK();
    }
    return HC_OK;
}

extern "C" int hc_bin_pairs_local_banded(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                                         const uint8_t* mark, int64_t npairs, int32_t res, int32_t mode,
                                         int32_t* mats, const int64_t* mat_off, const int32_t* mat_n,
                                         const int32_t* mat_ld, const int64_t* bin_off, int32_t nchrom,
                                         const int32_t* h_mat_n, int32_t band_width, unsigned long long* oob,
                                         void* work, void* stream) {
    HC_REQUIRE(nchrom > 0 && nchrom <= PART_MAX_BUCKETS && h_mat_n != nullptr, "at most 256 chromosomes; h_mat_n");
    int64_t nbins = 0;
    for (int p = 0; p < nchrom; ++p) nbins += h_mat_n[p] > 0 ? h_mat_n[p] : 0;
    if (npairs == 0 || nbins == 0) return HC_OK;
    int rc = hc_bin_band_begin(work, nbins, band_width, stream);
    if (rc == HC_OK) rc = hc_bin_band_accumulate(c1, p1, c2, p2, mark, npairs, 0, res, mode, mats, mat_off, mat_n, mat_ld,
                                                 bin_off, nchrom, band_width, oob, work, stream);
    if (rc == HC_OK) rc = hc_bin_band_finish(mats, mat_off, mat_n, mat_ld, bin_off, nchrom, h_mat_n, band_width, work, stream);
    return rc;
}

extern "C" int hc_bin_pairs_whole(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                                  const uint8_t* mark, int64_t npairs, int32_t res, int32_t mode,
                                  const int64_t* start1, const int64_t* start2, int32_t nchrom, int32_t* M,
                                  int32_t total, int64_t ld, unsigned long long* oob, void* stream) {
    HC_REQUIRE(npairs >= 0 && res > 0 && nchrom > 0 && total > 0 && ld >= total, "sizes");
    HC_REQUIRE(mode >= HC_BIN_SYM_ALL && mode <= HC_BIN_ONESIDED, "mode");
    if (npairs == 0) return HC_OK;
    HC_REQUIRE(mode == HC_BIN_SYM_ALL || mark != nullptr, "mark column required for this mode");
    HC_REQUIRE(aligned16(c1) && aligned16(p1) && aligned16(c2) && aligned16(p2), "pair columns must be 16-byte aligned");
    HC_REQUIRE(mark == nullptr || (reinterpret_cast<uintptr_t>(mark) & 3u) == 0, "mark must be 4-byte aligned");
    PairCols in{c1, p1, c2, p2, mark};
    bin_pairs_kernel<true><<<bin_grid(npairs), BIN_THREADS, 0, (cudaStream_t)stream>>>(
        in, npairs, make_fast_div((uint32_t)res), mode, M, start1, start2, nullptr, nullptr, nchrom, ld, total, oob);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_dense_nonzero_count(const void* M, int64_t ld, int32_t nrows, int32_t ncols, int32_t triu,
                                      int32_t is_f64, int64_t* row_ptr, void* stream) {
    HC_REQUIRE(nrows >= 0 && ncols >= 0 && ld >= ncols, "shape");
    cudaStream_t s = (cudaStream_t)stream;
    if (nrows > 0) {
        const int blocks = (nrows * 32 + 255) / 256;
        if (is_f64) row_nonzero_count_kernel<double><<<blocks, 256, 0, s>>>((const double*)M, ld, nrows, ncols, triu, row_ptr);
        else row_nonzero_count_kernel<int32_t><<<blocks, 256, 0, s>>>((const int32_t*)M, ld, nrows, ncols, triu, row_ptr);
        HC_LAUNCH_CHECK();
    }
    exclusive_scan_kernel<<<1, 1024, 0, s>>>(row_ptr, nrows);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_dense_nonzero_extract(const void* M, int64_t ld, int32_t nrows, int32_t ncols, int32_t triu,
                                        int32_t is_f64, const int64_t* row_ptr, int32_t* bin1, int32_t* bin2,
                                        void* val, void* stream) {
    HC_REQUIRE(nrows >= 0 && ncols >= 0 && ld >= ncols, "shape");
    if (nrows == 0) return HC_OK;
    cudaStream_t s = (cudaStream_t)stream;
    const int blocks = (nrows * 32 + 255) / 256;
    if (is_f64) row_nonzero_extract_kernel<double><<<blocks, 256, 0, s>>>((const double*)M, ld, nrows, ncols, triu, row_ptr, bin1, bin2, (double*)val);
    else row_nonzero_extract_kernel<int32_t><<<blocks, 256, 0, s>>>((const int32_t*)M, ld, nrows, ncols, triu, row_ptr, bin1, bin2, (int32_t*)val);
    HC_LAUNCH_CHECK();
    return HC_OK;
}
