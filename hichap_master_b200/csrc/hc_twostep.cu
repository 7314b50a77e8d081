// (c) Two-step allelic correction: matrixBuilding.py:984-1023 (TwoStepCorrection) with
// Coverage_M :904-912, Gap_defined :915-929, Gap_definedLowRes :742-753, Trans2symmetry :945-979,
// Trans2symmetryLowRes :770-776 and Correct_VC :780-790; also the building blocks of
// GenomeWideMatrixCorrection :857-901.
//
// Data flow for one haplotype matrix X (int32, n x n):
//   rowstats         : row sums + non-zero counts                      (reads X once)
//   twostep_alpha    : O(n) on one CTA: coverage -> gap rows, alpha, percentiles (radix select)
//   sym pass ROWSUM  : tile pairs (I,J)/(J,I): S = X/alpha[:,None]; Sym = f(S_ij, S_ji, gap);
//                      deterministic per-tile partial row sums          (reads X once)
//   vc_scale         : s = rowsum(Sym)^(2/3), 0 -> 1
//   sym pass TOTAL   : sum_ij Sym_ij / (s_i s_j)                        (reads X once)
//   sym pass WRITE   : out = RF * Sym_ij / (s_j s_i), RF = mean(X)/mean(Cor)  (reads X, writes fp64)
// The reference's 2*N^2 interpreted iterations in Trans2symmetry become the tile-pair passes.
// Roofline: HBM-bound, (4+4+4+4+8) N^2 = 24 N^2 bytes per haplotype matrix (+4 N^2 for TM).
#include <limits.h>
#include <math.h>
#include "hc_common.cuh"
#include <algorithm>
#include <string.h>
#include <vector>
#include "hc_select.cuh"

namespace {

constexpr int T = 64;          // tile side
constexpr int LDB = T + 1;     // padded leading dimension of the transposed-access tile
constexpr int TS_THREADS = 256;

// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
rowstats_kernel(const int32_t* __restrict__ M, int64_t ld, int nrows, int ncols, int vec_ok,
                int64_t* __restrict__ rowsum, int32_t* __restrict__ rownnz) {
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (r >= nrows) return;
    const int32_t* row = M + (int64_t)r * ld;
    long long s = 0;
    int c = 0;
    int done = 0;
    if (vec_ok) {
        const int nvec = ncols >> 2;
        for (int v = lane; v < nvec; v += 32) {
            const int4 a = ld_stream_v4(row + 4 * v);
            s += (long long)a.x + a.y + a.z + a.w;
            c += (a.x != 0) + (a.y != 0) + (a.z != 0) + (a.w != 0);
        }
        done = nvec << 2;
    }
    for (int j = done + lane; j < ncols; j += 32) { const int x = row[j]; s += x; c += (x != 0); }
    s = warp_sum_ll(s);
    c = warp_sum_i(c);
    if (lane == 0) { rowsum[r] = s; if (rownnz) rownnz[r] = c; }
}

// ---------------------------------------------------------------------------------------
struct AlphaArgs {
    const int64_t* rs_t; const int64_t* rs_m; const int64_t* rs_p;
    const int32_t* nnz_a; const int32_t* nnz_b;
    int n; int ncols; int gap_mode;
    double* alpha; uint8_t* gf_a; uint8_t* gf_b; int32_t* gi_a; int32_t* gi_b; int32_t* ngap;
    double* work;
    double q25, q20;
    // batched path (grid = nchrom): per-chromosome offsets into the concatenated vectors; NULL = single problem
    const int64_t* t_bin_off; const int64_t* h_bin_off; int nchrom;
};

__device__ void gap_rows(const int32_t* nnz, int n, int ncols, int gap_mode, double q25, double* cov,
                         uint8_t* gf, HcSelectSmem* sm) {
    long long cnt = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        // 1 - zeros/len, in the reference's operation order (matrixBuilding.py:909)
        const double v = __dadd_rn(1.0, -__ddiv_rn((double)(ncols - nnz[i]), (double)ncols));
        cov[i] = v;
        cnt += (v != 0.0);
    }
    __syncthreads();
    double thr = 0.1;
    if (gap_mode == HC_GAP_PERCENTILE) {
        cnt = block_sum_ll(cnt, sm->redll);
        thr = block_percentile([&](long long i) { return cov[i]; }, [&](long long i) { return cov[i] != 0.0; },
                               n, cnt, q25, sm);
        if (thr > 0.2) thr = 0.2;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) gf[i] = cov[i] < thr;
    __syncthreads();
}

// ordered compaction of flagged indices by one CTA
__device__ void compact_flags(const uint8_t* gf, int n, int32_t* idx, int32_t* count) {
    __shared__ int wtot[32];
    __shared__ int base_s;
    if (threadIdx.x == 0) base_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    for (int b0 = 0; b0 < n; b0 += blockDim.x) {
        const int i = b0 + threadIdx.x;
        const bool f = i < n && gf[i];
        const unsigned m = __ballot_sync(0xffffffffu, f);
        if (lane == 0) wtot[wid] = __popc(m);
        __syncthreads();
        int off = base_s;
        for (int w = 0; w < wid; ++w) off += wtot[w];
        if (f) idx[off + __popc(m & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < nw; ++w) t += wtot[w]; base_s += t; }
        __syncthreads();
    }
    if (threadIdx.x == 0) *count = base_s;
    __syncthreads();
}

__global__ void __launch_bounds__(1024) twostep_alpha_kernel(AlphaArgs a) {
    __shared__ HcSelectSmem sm;
    if (a.t_bin_off) {          // batched: chromosome c; M matrix c and P matrix nchrom + c of the haplotype batch
        const int c = blockIdx.x;
        const int64_t t0 = a.t_bin_off[c], m0 = a.h_bin_off[c], p0 = a.h_bin_off[a.nchrom + c];
        a.n = (int)(a.t_bin_off[c + 1] - t0);
        a.ncols = a.n;
        a.rs_t += t0; a.rs_m += m0; a.rs_p += p0; a.nnz_a += m0; a.nnz_b += p0;
        a.alpha += t0; a.gf_a += m0; a.gf_b += p0; a.gi_a += m0; a.gi_b += p0;
        a.ngap += 2 * c;
        a.work += 2 * t0;
        if (a.n == 0) return;
    }
    const int n = a.n;
    double* cov_a = a.work;
    double* cov_b = a.work + n;
    gap_rows(a.nnz_a, n, a.ncols, a.gap_mode, a.q25, cov_a, a.gf_a, &sm);
    compact_flags(a.gf_a, n, a.gi_a, a.ngap);
    const bool two = a.nnz_b != nullptr;
    if (two) {
        gap_rows(a.nnz_b, n, a.ncols, a.gap_mode, a.q25, cov_b, a.gf_b, &sm);
        compact_flags(a.gf_b, n, a.gi_b, a.ngap + 1);
    }
    // non-gap rows: NonGap(A) | NonGap(B)  ==  not (gap_a and gap_b)      (matrixBuilding.py:999)
    auto nongap = [&](long long i) { return two ? !(a.gf_a[i] && a.gf_b[i]) : !a.gf_a[i]; };
    double* al = a.alpha;
    double mx = -INFINITY;
    long long cnt = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const double v = __ddiv_rn((double)(a.rs_m[i] + a.rs_p[i]), (double)(a.rs_t[i] + 1));
        al[i] = v;
        if (nongap(i)) { mx = fmax(mx, v); ++cnt; }
    }
    cnt = block_sum_ll(cnt, sm.redll);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    __syncthreads();
    if ((threadIdx.x & 31) == 0) sm.red[threadIdx.x >> 5] = mx;
    __syncthreads();
    mx = sm.red[0];
    for (int w = 1; w < (int)(blockDim.x >> 5); ++w) mx = fmax(mx, sm.red[w]);
    __syncthreads();
    if (cnt == 0) mx = __longlong_as_double(0x7ff8000000000000ll);  // np.max of an empty selection has no value
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        double v = __ddiv_rn(al[i], mx);
        if (v == 0.0) v = 1.0;
        al[i] = v;
    }
    __syncthreads();
    const double thr = block_percentile([&](long long i) { return al[i]; }, nongap, n, cnt, a.q20, &sm);
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) if (al[i] < thr) al[i] = thr;
}

// ---------------------------------------------------------------------------------------
// tile-pair passes
// ---------------------------------------------------------------------------------------
enum { PASS_ROWSUM = 0, PASS_TOTAL = 1, PASS_WRITE = 2 };

struct SymArgs {
    const int32_t* X; int64_t ld; int n; int nT;
    const double* alpha; const uint8_t* gapflag; int has_gap;
    const int32_t* ngap_dev;   // batched path: has_gap = (*ngap_dev > 0), decided on the device (no host round trip)
    double* ra;           // [nT*T] 1 / alpha_i (0 beyond n)
    double* partial;      // [nT][nT*T] per-tile partial row sums of Sym
    double* rs;           // [nT*T] 1 / s_i  (s = rowsum^(2/3), 0 -> 1)
    double* cta_partial;  // [npairs]
    const double* scalars; // scalars[0] = RF
    double* out; int64_t ld_out;
};

__device__ __forceinline__ void tile_index(int idx, int nT, int* I, int* J) {
    // row-major enumeration of the upper triangle (I <= J)
    int i = (int)floor(((2.0 * nT + 1.0) - sqrt((2.0 * nT + 1.0) * (2.0 * nT + 1.0) - 8.0 * idx)) * 0.5);
    if (i < 0) i = 0;
    while (i > 0 && (long long)i * (2 * nT - i + 1) / 2 > idx) --i;
    while ((long long)(i + 1) * (2 * nT - i) / 2 <= idx) ++i;
    *I = i;
    *J = i + (idx - (int)((long long)i * (2 * nT - i + 1) / 2));
}

__device__ __forceinline__ void load_tile(const int32_t* __restrict__ X, int64_t ld, int n, int r0, int c0,
                                          int32_t* dst, int ldd) {
    // 64 rows x 16 int4; thread t loads (row = t/16 + 16a, vec = t%16)
    const int v = threadIdx.x & 15, rr = threadIdx.x >> 4;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int r = rr + 16 * a, gi = r0 + r, gc = c0 + 4 * v;
        int4 x = make_int4(0, 0, 0, 0);
        if (gi < n && gc < (int)ld) x = ld_stream_v4(X + (int64_t)gi * ld + gc);
        int32_t* d = dst + r * ldd + 4 * v;
        d[0] = gc < n ? x.x : 0; d[1] = gc + 1 < n ? x.y : 0; d[2] = gc + 2 < n ? x.z : 0; d[3] = gc + 3 < n ? x.w : 0;
    }
}

// 64 x 64 tile: fast path for tiles that lie inside the matrix (128-bit shared-memory stores, no bound checks)
__device__ __forceinline__ void load_tile_fast(const int32_t* __restrict__ X, int64_t ld, int r0, int c0, int32_t* dst, int ldd) {
    const int v = threadIdx.x & 15, rr = threadIdx.x >> 4;
    int4 x[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) x[a] = ld_stream_v4(X + (int64_t)(r0 + rr + 16 * a) * ld + c0 + 4 * v);
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        int32_t* d = dst + (rr + 16 * a) * ldd + 4 * v;
        if ((ldd & 3) == 0) *reinterpret_cast<int4*>(d) = x[a];
        else { d[0] = x[a].x; d[1] = x[a].y; d[2] = x[a].z; d[3] = x[a].w; }
    }
}

// The per-cell work of a tile pair.  Everything that depends only on the row or only on the column (1 / alpha, the gap
// flag, 1 / s) is staged once per tile in shared memory / registers; cells outside the matrix are zero in the staged
// tiles and have 1 / alpha = 0, so they need no test.  (The first version evaluated bounds, flags and the 1 / alpha
// loads per cell: 31 thread instructions per cell, issue-bound at 2.6 TB/s -- profiles/r1d_ncu_secondary_raw.csv.)
// DIAG: the tile pair is a diagonal tile (I == J: one tile, read at both orientations, leading dimension T); otherwise the
// transposed operand is the padded copy of tile (J, I) -- compile-time so that the inner loop carries neither the diagonal
// test nor a run-time leading dimension (the ROWSUM / TOTAL passes are issue-bound)
template <int PASS, bool GAP, bool DIAG>
__device__ __forceinline__ void sym_pass_body(const SymArgs& a, int I, int J, int r0, int c0, const int32_t* sA, const int32_t* tB,
                                              const double* vr, const double* vc, double* sV, double (*colred)[T], double* red,
                                              int cta) {
    constexpr int ldb = DIAG ? T : LDB;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;   // 8 warps; a warp covers one tile row at a time
    // per-column values of this thread's two columns
    double raj[2], rsj[2];
    bool gj[2];
#pragma unroll
    for (int b = 0; b < 2; ++b) {
        const int c = tx + 32 * b;
        raj[b] = vc[c];
        rsj[b] = PASS != PASS_ROWSUM ? vc[T + c] : 0.0;
        gj[b] = GAP ? vc[2 * T + c] != 0.0 : false;
    }
    double val[8][2];
    double rs8[8];
    double colp[2] = {0.0, 0.0};
    double tot = 0.0;
    const int64_t np = (int64_t)a.nT * T;
#pragma unroll
    for (int ai = 0; ai < 8; ++ai) {
        const int r = ty + 8 * ai;
        const double rai = vr[r];
        const double rsi = PASS != PASS_ROWSUM ? vr[T + r] : 0.0;
        const bool gi = GAP ? vr[2 * T + r] != 0.0 : false;
        double rsum = 0.0;
#pragma unroll
        for (int b = 0; b < 2; ++b) {
            const int c = tx + 32 * b;
            const double sij = i32_to_f64(sA[r * T + c]) * rai;
            const double sji = i32_to_f64(tB[c * ldb + r]) * raj[b];
            double sym;
            if (GAP) sym = (gi && gj[b]) ? fmax(sij, sji) : (sij + sji) * 0.5;
            else sym = sij + sji;
            if (DIAG && r == c) sym = sij;
            if (PASS == PASS_ROWSUM) { rsum += sym; colp[b] += sym; }
            else {
                const double cor = sym * (rsi * rsj[b]);
                if (PASS == PASS_TOTAL) tot += cor; else val[ai][b] = cor;
            }
        }
        if (PASS == PASS_ROWSUM) rs8[ai] = rsum;
    }
    if (PASS == PASS_ROWSUM) {
        // the eight row sums of the warp in one halving butterfly (9 exchanges instead of 8 x 5): after the three halving steps a
        // lane holds the partial of row ai = (lane >> 2) & 7 bit-reversed as below, two plain steps finish it
        {
            const bool h4 = tx & 16, h3 = tx & 8, h2 = tx & 4;
            double w4[4], w2[2], w1;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const double mine = h4 ? rs8[i + 4] : rs8[i], other = h4 ? rs8[i] : rs8[i + 4];
                w4[i] = mine + __shfl_xor_sync(0xffffffffu, other, 16);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const double mine = h3 ? w4[i + 2] : w4[i], other = h3 ? w4[i] : w4[i + 2];
                w2[i] = mine + __shfl_xor_sync(0xffffffffu, other, 8);
            }
            {
                const double mine = h2 ? w2[1] : w2[0], other = h2 ? w2[0] : w2[1];
                w1 = mine + __shfl_xor_sync(0xffffffffu, other, 4);
            }
            w1 += __shfl_xor_sync(0xffffffffu, w1, 2);
            w1 += __shfl_xor_sync(0xffffffffu, w1, 1);
            if ((tx & 3) == 0) {
                const int ai = (h4 ? 4 : 0) + (h3 ? 2 : 0) + (h2 ? 1 : 0);
                a.partial[(int64_t)J * np + r0 + ty + 8 * ai] = w1;            // rows of block I, other block J
            }
        }
        if (!DIAG) {
            colred[ty][tx] = colp[0]; colred[ty][tx + 32] = colp[1];
            __syncthreads();
            if (threadIdx.x < T) {
                double s = 0.0;
#pragma unroll
                for (int w = 0; w < 8; ++w) s += colred[w][threadIdx.x];
                a.partial[(int64_t)I * np + c0 + threadIdx.x] = s;           // rows of block J, other block I
            }
        }
    } else if (PASS == PASS_TOTAL) {
        const double s = block_sum(tot, red);
        if (threadIdx.x == 0) a.cta_partial[cta] = DIAG ? s : 2.0 * s;
    } else {
        const double rf = a.scalars[0];
        if (!DIAG) __syncthreads();          // sV aliases sA / sB: every thread is done reading them
#pragma unroll
        for (int ai = 0; ai < 8; ++ai) {
            const int r = ty + 8 * ai, gi = r0 + r;
#pragma unroll
            for (int b = 0; b < 2; ++b) {
                const int c = tx + 32 * b, gjj = c0 + c;
                const double v = rf * val[ai][b];
                if (gi < a.n && gjj < a.n) a.out[(int64_t)gi * a.ld_out + gjj] = v;
                if (!DIAG) sV[c * LDB + r] = v;
            }
        }
        if (!DIAG) {
            __syncthreads();
#pragma unroll
            for (int ai = 0; ai < 8; ++ai) {
                const int c = ty + 8 * ai, gjj = c0 + c;   // row of the mirrored tile
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    const int r = tx + 32 * b, gi = r0 + r;
                    if (gi < a.n && gjj < a.n) a.out[(int64_t)gjj * a.ld_out + gi] = sV[c * LDB + r];
                }
            }
        }
    }
}

// one tile pair (`cta` = its index in the row-major enumeration of the upper triangle) of one matrix
template <int PASS>
__device__ __forceinline__ void sym_pass_run(SymArgs a, int cta) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    int32_t* sA = reinterpret_cast<int32_t*>(smem_raw);     // [T][T]    tile (I,J)
    int32_t* sB = sA + T * T;                               // [T][LDB]  tile (J,I)
    double* sV = reinterpret_cast<double*>(smem_raw);      // PASS_WRITE: [T][LDB] staged mirror tile, written over the two
                                                           // input tiles once every thread holds its cells in registers
                                                           // (33 KB instead of 66 KB per CTA: 36 % -> 50+ % occupancy)
    __shared__ double colred[8][T];
    __shared__ double red[32];
    __shared__ double vr[3 * T], vc[3 * T];                 // per row / per column of the tile: 1/alpha, 1/s, gap flag

    if (a.ngap_dev) a.has_gap = *a.ngap_dev > 0;
    int I, J;
    tile_index(cta, a.nT, &I, &J);
    const int r0 = I * T, c0 = J * T;
    const bool inside = r0 + T <= a.n && c0 + T <= a.n && c0 + T <= (int)a.ld && r0 + T <= (int)a.ld;
    if (inside) {
        load_tile_fast(a.X, a.ld, r0, c0, sA, T);
        if (I != J) load_tile_fast(a.X, a.ld, c0, r0, sB, LDB);
    } else {
        load_tile(a.X, a.ld, a.n, r0, c0, sA, T);
        if (I != J) load_tile(a.X, a.ld, a.n, c0, r0, sB, LDB);
    }
    if (threadIdx.x < 2 * T) {          // ra / rs are zero-padded up to nT * T entries (recip_alpha_kernel, vc_scale_kernel)
        const int t = threadIdx.x & (T - 1);
        const int gidx = (threadIdx.x < T ? r0 : c0) + t;
        double* v = threadIdx.x < T ? vr : vc;
        v[t] = a.ra[gidx];
        v[T + t] = PASS != PASS_ROWSUM ? (gidx < a.n ? a.rs[gidx] : 0.0) : 0.0;
        v[2 * T + t] = (a.has_gap && gidx < a.n && a.gapflag[gidx]) ? 1.0 : 0.0;
    }
    __syncthreads();
    if (I != J) {
        if (a.has_gap) sym_pass_body<PASS, true, false>(a, I, J, r0, c0, sA, sB, vr, vc, sV, colred, red, cta);
        else sym_pass_body<PASS, false, false>(a, I, J, r0, c0, sA, sB, vr, vc, sV, colred, red, cta);
    } else {
        if (a.has_gap) sym_pass_body<PASS, true, true>(a, I, J, r0, c0, sA, sA, vr, vc, sV, colred, red, cta);
        else sym_pass_body<PASS, false, true>(a, I, J, r0, c0, sA, sA, vr, vc, sV, colred, red, cta);
    }
}

template <int PASS>
__global__ void __launch_bounds__(TS_THREADS, PASS == PASS_WRITE ? 4 : 5) sym_pass_kernel(SymArgs a) { sym_pass_run<PASS>(a, (int)blockIdx.x); }

// ---- all matrices of a batch in one launch per pass -------------------------------------------
// (46 matrices x 6 dependent launches, most of them small, cost 1.1 ms of launch-latency chains out of 5.8 ms --
// profiles/r2s_c3_launches.csv; the matrices are independent, so every pass runs over the tile pairs of all of them.)
struct SymBatch {
    const SymArgs* mats;          // device array, one entry per matrix
    const int* pair_off;          // [nmat+1] prefix of the tile-pair counts
    const int64_t* const* rowsum; // [nmat] row sums of the input matrix (for the rescale factor)
    int nmat;
};

__device__ __forceinline__ int batch_find(const int* __restrict__ off, int nmat, int x) {
    int lo = 0, hi = nmat;        // largest k with off[k] <= x
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (off[mid] <= x) lo = mid; else hi = mid; }
    return lo;
}

template <int PASS>
__global__ void __launch_bounds__(TS_THREADS, PASS == PASS_WRITE ? 4 : 5) sym_pass_batch_kernel(SymBatch b) {
    const int k = batch_find(b.pair_off, b.nmat, (int)blockIdx.x);
    sym_pass_run<PASS>(b.mats[k], (int)blockIdx.x - b.pair_off[k]);
}

__device__ __forceinline__ void recip_alpha_run(const SymArgs& a, int i) {
    if (i < a.nT * T) a.ra[i] = i < a.n ? 1.0 / a.alpha[i] : 0.0;
}
__global__ void __launch_bounds__(256) recip_alpha_kernel(SymArgs a) { recip_alpha_run(a, blockIdx.x * blockDim.x + threadIdx.x); }
__global__ void __launch_bounds__(256) recip_alpha_batch_kernel(SymBatch b) {        // grid.y = matrix
    recip_alpha_run(b.mats[blockIdx.y], blockIdx.x * blockDim.x + threadIdx.x);
}

// s_i = (sum_K partial[K][i])^(2/3), zeros -> 1; store the reciprocal
__device__ __forceinline__ void vc_scale_run(const SymArgs& a, int i) {
    const int64_t np = (int64_t)a.nT * T;
    if (i >= np) return;
    double s = 0.0;
    if (i < a.n) for (int K = 0; K < a.nT; ++K) s += a.partial[(int64_t)K * np + i];
    s = pow(s, 2.0 / 3.0);
    if (s == 0.0) s = 1.0;
    a.rs[i] = 1.0 / s;
}
__global__ void __launch_bounds__(256) vc_scale_kernel(SymArgs a) { vc_scale_run(a, blockIdx.x * blockDim.x + threadIdx.x); }
__global__ void __launch_bounds__(256) vc_scale_batch_kernel(SymBatch b) { vc_scale_run(b.mats[blockIdx.y], blockIdx.x * blockDim.x + threadIdx.x); }

// RF = mean(X) / mean(Cor)
__device__ __forceinline__ void vc_rescale_factor_run(const double* __restrict__ cta_partial, int npairs,
                                                      const int64_t* __restrict__ rowsum_x, int n, double* __restrict__ scalars) {
    __shared__ double red[32];
    __shared__ long long redll[32];
    double t = 0.0;
    for (int i = threadIdx.x; i < npairs; i += blockDim.x) t += cta_partial[i];
    t = block_sum(t, red);
    long long sx = 0;
    for (int i = threadIdx.x; i < n; i += blockDim.x) sx += rowsum_x[i];
    sx = block_sum_ll(sx, redll);
    if (threadIdx.x == 0) {
        const double cells = (double)n * (double)n;
        const double mean_x = (double)sx / cells, mean_cor = t / cells;
        scalars[0] = mean_x / mean_cor;
        scalars[1] = mean_x;
        scalars[2] = mean_cor;
    }
}
__global__ void __launch_bounds__(1024)
vc_rescale_factor_kernel(const double* __restrict__ cta_partial, int npairs, const int64_t* __restrict__ rowsum_x,
                         int n, double* __restrict__ scalars) {
    vc_rescale_factor_run(cta_partial, npairs, rowsum_x, n, scalars);
}
__global__ void __launch_bounds__(1024) vc_rescale_factor_batch_kernel(SymBatch b) {      // one CTA per matrix
    const SymArgs& a = b.mats[blockIdx.x];
    vc_rescale_factor_run(a.cta_partial, b.pair_off[blockIdx.x + 1] - b.pair_off[blockIdx.x], b.rowsum[blockIdx.x], a.n,
                          const_cast<double*>(a.scalars));
}

// row sums + non-zero counts of every matrix of a batch (one warp per global row)
__global__ void __launch_bounds__(256)
rowstats_batch_kernel(const int32_t* __restrict__ mats, const int64_t* __restrict__ mat_off, const int32_t* __restrict__ mat_n,
                      const int32_t* __restrict__ mat_ld, const int64_t* __restrict__ bin_off, int nprob,
                      int64_t* __restrict__ rowsum, int32_t* __restrict__ rownnz) {
    const int64_t g = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= bin_off[nprob]) return;
    int lo = 0, hi = nprob - 1;
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (bin_off[mid] <= g) lo = mid; else hi = mid - 1; }
    const int p = lo, r = (int)(g - bin_off[p]);
    const int32_t* row = mats + mat_off[p] + (int64_t)r * mat_ld[p];
    const int nvec = mat_ld[p] >> 2;            // padding columns are zero
    long long s = 0;
    int c = 0;
    for (int v = lane; v < nvec; v += 32) {
        const int4 a = ld_stream_v4(row + 4 * v);
        s += (long long)a.x + a.y + a.z + a.w;
        c += (a.x != 0) + (a.y != 0) + (a.z != 0) + (a.w != 0);
    }
    s = warp_sum_ll(s);
    c = warp_sum_i(c);
    if (lane == 0) { rowsum[g] = s; if (rownnz) rownnz[g] = c; }
}

struct TwoStepWork { double* partial; double* rs; double* ra; double* cta_partial; double* scalars; };

TwoStepWork carve(void* work, int n) {
    const int64_t nT = (n + T - 1) / T, np = nT * T, npairs = nT * (nT + 1) / 2;
    TwoStepWork w;
    w.partial = reinterpret_cast<double*>(work);
    w.rs = w.partial + nT * np;
    w.ra = w.rs + np;
    w.cta_partial = w.ra + np;
    w.scalars = w.cta_partial + npairs;
    return w;
}

}  // namespace

extern "C" int hc_rowstats_i32(const int32_t* M, int64_t ld, int32_t nrows, int32_t ncols, int64_t* rowsum,
                               int32_t* rownnz, void* stream) {
    HC_REQUIRE(nrows >= 0 && ncols >= 0 && ld >= ncols, "shape");
    if (nrows == 0) return HC_OK;
    const int vec_ok = ((reinterpret_cast<uintptr_t>(M) & 15u) == 0) && ((ld & 3) == 0);
    const int blocks = (int)(((int64_t)nrows * 32 + 255) / 256);
    rowstats_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(M, ld, nrows, ncols, vec_ok, rowsum, rownnz);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_twostep_alpha(const int64_t* rowsum_t, const int64_t* rowsum_m, const int64_t* rowsum_p,
                                const int32_t* nnz_a, const int32_t* nnz_b, int32_t n, int32_t ncols,
                                int32_t gap_mode, double* alpha, uint8_t* gapflag_a, uint8_t* gapflag_b,
                                int32_t* gapidx_a, int32_t* gapidx_b, int32_t* ngap, double* work, void* stream) {
    HC_REQUIRE(n > 0 && ncols > 0, "n>0, ncols>0");
    HC_REQUIRE(gap_mode == HC_GAP_PERCENTILE || gap_mode == HC_GAP_FIXED, "gap_mode");
    HC_REQUIRE(nnz_a && gapflag_a && gapidx_a && ngap && alpha && work, "null pointer");
    HC_REQUIRE(nnz_b == nullptr || (gapflag_b && gapidx_b), "second gap outputs");
    AlphaArgs a;
    a.rs_t = rowsum_t; a.rs_m = rowsum_m; a.rs_p = rowsum_p; a.nnz_a = nnz_a; a.nnz_b = nnz_b;
    a.n = n; a.ncols = ncols; a.gap_mode = gap_mode;
    a.alpha = alpha; a.gf_a = gapflag_a; a.gf_b = gapflag_b; a.gi_a = gapidx_a; a.gi_b = gapidx_b; a.ngap = ngap;
    a.work = work;
    a.t_bin_off = nullptr; a.h_bin_off = nullptr; a.nchrom = 0;
    a.q25 = 25.0 / 100.0;  // np.percentile divides q by 100 first
    a.q20 = 20.0 / 100.0;
    twostep_alpha_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(a);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int64_t hc_twostep_work_bytes(int32_t n) {
    const int64_t nT = (n + T - 1) / T, np = nT * T, npairs = nT * (nT + 1) / 2;
    return (int64_t)sizeof(double) * (nT * np + 2 * np + npairs + 8);
}

extern "C" int hc_twostep_correct(const int32_t* X, int64_t ld, int32_t n, const double* alpha,
                                  const uint8_t* gapflag, int32_t has_gap, const int64_t* rowsum_x, double* out,
                                  int64_t ld_out, void* work, void* stream) {
    HC_REQUIRE(n > 0 && ld >= n && (ld & 3) == 0 && ld_out >= n, "shape (ld multiple of 4)");
    HC_REQUIRE((reinterpret_cast<uintptr_t>(X) & 15u) == 0, "X must be 16-byte aligned");
    HC_REQUIRE(!has_gap || gapflag != nullptr, "gapflag required when has_gap");
    cudaStream_t s = (cudaStream_t)stream;
    const int nT = (n + T - 1) / T;
    const int64_t npairs64 = (int64_t)nT * (nT + 1) / 2;
    HC_REQUIRE(npairs64 < (1ll << 31), "matrix too large");
    const int npairs = (int)npairs64;
    TwoStepWork w = carve(work, n);
    SymArgs a;
    a.X = X; a.ld = ld; a.n = n; a.nT = nT; a.alpha = alpha; a.gapflag = gapflag; a.has_gap = has_gap ? 1 : 0;
    a.ngap_dev = nullptr;
    a.partial = w.partial; a.rs = w.rs; a.ra = w.ra; a.cta_partial = w.cta_partial; a.scalars = w.scalars;
    a.out = out; a.ld_out = ld_out;
    const size_t smem_tiles = (size_t)(T * T + T * LDB) * sizeof(int32_t);
    const size_t smem_write = std::max(smem_tiles, (size_t)T * LDB * sizeof(double));
    HC_CUDA(cudaFuncSetAttribute(sym_pass_kernel<PASS_WRITE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_write));
    recip_alpha_kernel<<<(nT * T + 255) / 256, 256, 0, s>>>(a);
    HC_LAUNCH_CHECK();
    sym_pass_kernel<PASS_ROWSUM><<<npairs, TS_THREADS, smem_tiles, s>>>(a);
    HC_LAUNCH_CHECK();
    vc_scale_kernel<<<(nT * T + 255) / 256, 256, 0, s>>>(a);
    HC_LAUNCH_CHECK();
    sym_pass_kernel<PASS_TOTAL><<<npairs, TS_THREADS, smem_tiles, s>>>(a);
    HC_LAUNCH_CHECK();
    vc_rescale_factor_kernel<<<1, 1024, 0, s>>>(w.cta_partial, npairs, rowsum_x, n, w.scalars);
    HC_LAUNCH_CHECK();
    sym_pass_kernel<PASS_WRITE><<<npairs, TS_THREADS, smem_write, s>>>(a);
    HC_LAUNCH_CHECK();
    return HC_OK;
}


// ---- whole-batch driver: IntraChromMatrixCorrection (matrixBuilding.py:1026-1041) in one call -----
// T: nchrom traditional matrices; H: 2*nchrom haplotype matrices (all maternal, then all paternal),
// same sides.  Everything is enqueued on `stream` with no host round trip: the gap decisions
// (`has_gap`) are read by the tile kernels from the device counters.  Outputs: out (fp64, matrix k of H
// at h_out_off[k], row-major n x n), alpha (per T bin), gapflag / gapidx (per H bin), ngap[2*nchrom]
// ordered (M_c, P_c) per chromosome.
extern "C" int64_t hc_twostep_batch_work_bytes(int64_t t_nbins, int64_t h_nbins, int32_t max_n) {
    return (int64_t)sizeof(int64_t) * (t_nbins + h_nbins) + (int64_t)sizeof(int32_t) * h_nbins + (int64_t)sizeof(double) * 2 * t_nbins +
           hc_twostep_work_bytes(max_n) + 256;
}

extern "C" int hc_twostep_batch(const int32_t* tmats, const int64_t* t_off, const int32_t* t_n, const int32_t* t_ld,
                                const int64_t* t_bin_off, const int32_t* hmats, const int64_t* h_off,
                                const int32_t* h_n, const int32_t* h_ld, const int64_t* h_bin_off, int32_t nchrom,
                                const int32_t* h_sizes, const int64_t* h_hoff, const int32_t* h_hld,
                                const int64_t* h_tbin, const int64_t* h_hbin, double* out, const int64_t* h_out_off,
                                double* alpha, uint8_t* gapflag, int32_t* gapidx, int32_t* ngap, void* work,
                                void* stream) {
    HC_REQUIRE(nchrom > 0 && h_sizes && h_hoff && h_hld && h_tbin && h_hbin && h_out_off, "arguments");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t t_nbins = h_tbin[nchrom], h_nbins = h_hbin[2 * nchrom];
    int max_n = 0;
    for (int c = 0; c < nchrom; ++c) max_n = h_sizes[c] > max_n ? h_sizes[c] : max_n;
    if (t_nbins == 0) return HC_OK;
    // scratch: row sums of T and H, nnz of H, alpha work, per-matrix two-step work
    int64_t* rs_t = reinterpret_cast<int64_t*>(work);
    int64_t* rs_h = rs_t + t_nbins;
    double* awork = reinterpret_cast<double*>(rs_h + h_nbins);
    int32_t* nz_h = reinterpret_cast<int32_t*>(awork + 2 * t_nbins);
    void* mwork = reinterpret_cast<void*>((reinterpret_cast<uintptr_t>(nz_h + h_nbins) + 255) & ~(uintptr_t)255);

    rowstats_batch_kernel<<<(unsigned)((t_nbins * 32 + 255) / 256), 256, 0, s>>>(tmats, t_off, t_n, t_ld, t_bin_off, nchrom, rs_t, nullptr);
    HC_LAUNCH_CHECK();
    rowstats_batch_kernel<<<(unsigned)((h_nbins * 32 + 255) / 256), 256, 0, s>>>(hmats, h_off, h_n, h_ld, h_bin_off, 2 * nchrom, rs_h, nz_h);
    HC_LAUNCH_CHECK();
    AlphaArgs a;
    a.rs_t = rs_t; a.rs_m = rs_h; a.rs_p = rs_h; a.nnz_a = nz_h; a.nnz_b = nz_h; a.n = 0; a.ncols = 0;
    a.gap_mode = HC_GAP_PERCENTILE; a.alpha = alpha; a.gf_a = gapflag; a.gf_b = gapflag; a.gi_a = gapidx; a.gi_b = gapidx;
    a.ngap = ngap; a.work = awork; a.q25 = 25.0 / 100.0; a.q20 = 20.0 / 100.0;
    a.t_bin_off = t_bin_off; a.h_bin_off = h_bin_off; a.nchrom = nchrom;
    twostep_alpha_kernel<<<nchrom, 1024, 0, s>>>(a);
    HC_LAUNCH_CHECK();

    // per-matrix descriptors and scratch (stream-ordered allocation, released before returning); every pass is ONE launch
    // over the tile pairs of all matrices
    std::vector<SymArgs> mats;
    std::vector<int> pair_off(1, 0);
    std::vector<const int64_t*> rowsum;
    int64_t scratch_bytes = 0;
    int max_np = 0;
    for (int k = 0; k < 2 * nchrom; ++k) {
        const int c = k % nchrom, n = h_sizes[c];
        if (n == 0) continue;
        scratch_bytes += (hc_twostep_work_bytes(n) + 255) & ~(int64_t)255;
    }
    const size_t desc_bytes = ((sizeof(SymArgs) + sizeof(int) + sizeof(void*)) * (size_t)(2 * nchrom + 1) + 255) & ~(size_t)255;
    unsigned char* scratch = nullptr;
    HC_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&scratch), (size_t)scratch_bytes + desc_bytes + 256, s));
    unsigned char* cur = scratch + desc_bytes;
    for (int k = 0; k < 2 * nchrom; ++k) {
        const int c = k % nchrom, hap = k / nchrom, n = h_sizes[c];
        if (n == 0) continue;
        const int nT = (n + T - 1) / T;
        const int64_t npairs64 = (int64_t)nT * (nT + 1) / 2;
        if ((int64_t)pair_off.back() + npairs64 >= (1ll << 31)) { cudaFreeAsync(scratch, s); HC_REQUIRE(false, "batch too large"); }
        TwoStepWork w = carve(cur, n);
        cur += (hc_twostep_work_bytes(n) + 255) & ~(int64_t)255;
        SymArgs g;
        g.X = hmats + h_hoff[k]; g.ld = h_hld[k]; g.n = n; g.nT = nT;
        g.alpha = alpha + h_tbin[c]; g.gapflag = gapflag + h_hbin[k]; g.has_gap = 0; g.ngap_dev = ngap + 2 * c + hap;
        g.partial = w.partial; g.rs = w.rs; g.ra = w.ra; g.cta_partial = w.cta_partial; g.scalars = w.scalars;
        g.out = out + h_out_off[k]; g.ld_out = n;
        mats.push_back(g);
        pair_off.push_back(pair_off.back() + (int)npairs64);
        rowsum.push_back(rs_h + h_hbin[k]);
        max_np = nT * T > max_np ? nT * T : max_np;
    }
    const int nmat = (int)mats.size();
    if (nmat > 0) {
        // descriptors: [SymArgs x nmat][rowsum pointers x nmat][pair_off x (nmat+1)], one staged upload
        std::vector<unsigned char> stage(desc_bytes, 0);
        size_t o_rows = sizeof(SymArgs) * (size_t)nmat;
        size_t o_pair = o_rows + sizeof(void*) * (size_t)nmat;
        memcpy(stage.data(), mats.data(), sizeof(SymArgs) * (size_t)nmat);
        memcpy(stage.data() + o_rows, rowsum.data(), sizeof(void*) * (size_t)nmat);
        memcpy(stage.data() + o_pair, pair_off.data(), sizeof(int) * (size_t)(nmat + 1));
        HC_CUDA(cudaMemcpyAsync(scratch, stage.data(), desc_bytes, cudaMemcpyHostToDevice, s));   // pageable source: staged before return
        SymBatch b;
        b.mats = reinterpret_cast<const SymArgs*>(scratch);
        b.rowsum = reinterpret_cast<const int64_t* const*>(scratch + o_rows);
        b.pair_off = reinterpret_cast<const int*>(scratch + o_pair);
        b.nmat = nmat;
        const size_t smem_tiles = (size_t)(T * T + T * LDB) * sizeof(int32_t);
        const size_t smem_write = std::max(smem_tiles, (size_t)T * LDB * sizeof(double));
        HC_CUDA(cudaFuncSetAttribute(sym_pass_batch_kernel<PASS_WRITE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_write));
        const dim3 vgrid((unsigned)((max_np + 255) / 256), (unsigned)nmat);
        const unsigned total_pairs = (unsigned)pair_off.back();
        recip_alpha_batch_kernel<<<vgrid, 256, 0, s>>>(b);
        sym_pass_batch_kernel<PASS_ROWSUM><<<total_pairs, TS_THREADS, smem_tiles, s>>>(b);
        vc_scale_batch_kernel<<<vgrid, 256, 0, s>>>(b);
        sym_pass_batch_kernel<PASS_TOTAL><<<total_pairs, TS_THREADS, smem_tiles, s>>>(b);
        vc_rescale_factor_batch_kernel<<<(unsigned)nmat, 1024, 0, s>>>(b);
        sym_pass_batch_kernel<PASS_WRITE><<<total_pairs, TS_THREADS, smem_write, s>>>(b);
        hc_count_launch(6);
    }
    HC_CUDA(cudaFreeAsync(scratch, s));
    HC_CUDA(cudaGetLastError());
    return HC_OK;
}


// =========================================================================================
// The same correction on CSR matrices: local resolutions of allelic mode whose dense tiles would not fit (10 kb / 5 kb).
// Every step needs only per-row vectors and a per-cell rule, so it runs on the non-zeros: memory O(nnz + n).
//   T  : symmetric CSR of the nchrom traditional matrices over their concatenated bins (t_bin_off)
//   X  : general CSR of the 2*nchrom imputed haplotype matrices (all maternal, then all paternal; h_bin_off), global
//        column indices, rows column-sorted;  XT: its transpose, same layout (diagonal entries, if any, are not read)
// Passes, each one launch over all matrices:
//   csr_rowstats (T, X)  row sums (int64); non-zero counts of X -- coverage counts the non-zeros of the asymmetric matrix
//   twostep_alpha        the dense path's kernel: coverage -> gaps, alpha, percentiles (gaps are bit-exact)
//   sym ROWSUM           row i of Sym = merge of row i of X and row i of XT with S = X / alpha[:, None] and the rule of
//                        Trans2symmetry; s_i = rowsum(Sym)_i^(2/3), 0 -> 1 (the row sum stands in for the column sum)
//   sym TOTAL            per row: sum_j Sym_ij / (s_i s_j), and the number of non-zero upper-triangle cells (j >= i)
//   scan, rescale        record offsets; RF = mean(X) / mean(Cor) per matrix (the n^2 cancels)
//   sym EMIT             upper-triangle records (bin1, bin2, IF) in chromosome-local bins, row-major
// One thread merges one row: haplotype rows hold tens of cells at 10 kb, so a row is a short serial merge.
// =========================================================================================
namespace {

enum { CSR_ROWSUM = 0, CSR_TOTAL = 1, CSR_EMIT = 2 };

struct Rec24 { long long bin1; long long bin2; double IF; };   // matrixBuilding.py:460-461 S_dtype

struct SymCsrArgs {
    const int64_t* x_ptr; const int32_t* x_col; const int32_t* x_cnt;
    const int64_t* xt_ptr; const int32_t* xt_col; const int32_t* xt_cnt;
    const int64_t* t_bin_off; const int64_t* h_bin_off; int nchrom; int64_t h_nbins;
    const double* alpha; const uint8_t* gapflag; const int32_t* ngap;
    double* rsinv;          // [h_nbins] 1 / s_i
    double* rowtot;         // [h_nbins] per-row sum of Cor
    const double* scalars;  // [2*nchrom][4]: RF, mean(X), mean(Cor)
    int64_t* rec_ptr;       // [h_nbins + 1] upper-cell counts, then their exclusive scan
    Rec24* rec;
};

// row sums (+ non-zero counts) of a CSR, one warp per row
__global__ void __launch_bounds__(256)
csr_rowstats_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ cnt, int64_t nrows,
                    int64_t* __restrict__ rowsum, int32_t* __restrict__ rownnz) {
    const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= nrows) return;
    long long s = 0;
    int c = 0;
    for (int64_t e = row_ptr[r] + lane; e < row_ptr[r + 1]; e += 32) { const int x = cnt[e]; s += x; c += (x != 0); }
    s = warp_sum_ll(s);
    c = warp_sum_i(c);
    if (lane == 0) { rowsum[r] = s; if (rownnz) rownnz[r] = c; }
}

template <int PASS>
__global__ void __launch_bounds__(256) sym_csr_kernel(SymCsrArgs a) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.h_nbins) return;
    int lo = 0, hi = 2 * a.nchrom - 1;                 // matrix of the row: largest k with h_bin_off[k] <= g
    while (lo < hi) { const int mid = (lo + hi + 1) >> 1; if (a.h_bin_off[mid] <= g) lo = mid; else hi = mid - 1; }
    const int k = lo, c = k % a.nchrom, hap = k / a.nchrom;
    const int64_t base = a.h_bin_off[k], tb = a.t_bin_off[c] - base;     // alpha of global bin j: alpha[tb + j]
    const bool has_gap = a.ngap[2 * c + hap] > 0;
    const double rai = 1.0 / a.alpha[tb + g];
    const bool gi = has_gap && a.gapflag[g];
    const double rsi = PASS != CSR_ROWSUM ? a.rsinv[g] : 0.0;
    const double rf = PASS == CSR_EMIT ? a.scalars[4 * k] : 0.0;
    int64_t pa = a.x_ptr[g], pb = a.xt_ptr[g], o = PASS == CSR_EMIT ? a.rec_ptr[g] : 0;
    const int64_t ea = a.x_ptr[g + 1], eb = a.xt_ptr[g + 1];
    double acc = 0.0;
    long long upper = 0;
    while (pa < ea || pb < eb) {
        const int ja = pa < ea ? a.x_col[pa] : INT_MAX, jb = pb < eb ? a.xt_col[pb] : INT_MAX;
        const int j = ja < jb ? ja : jb;
        const int xij = ja == j ? a.x_cnt[pa++] : 0;
        const int xji = jb == j ? a.xt_cnt[pb++] : 0;
        const double sij = i32_to_f64(xij) * rai;
        double sym;
        if (j == g) sym = sij;                         // the diagonal is S_ii
        else {
            const double sji = i32_to_f64(xji) * (1.0 / a.alpha[tb + j]);
            if (has_gap) sym = (gi && a.gapflag[j]) ? fmax(sij, sji) : (sij + sji) * 0.5;
            else sym = sij + sji;
        }
        if (PASS == CSR_ROWSUM) { acc += sym; continue; }
        const double cor = sym * (rsi * a.rsinv[j]);
        const bool keep = j >= g && sym != 0.0;        // the non-zeros of the dense upper triangle
        if (PASS == CSR_TOTAL) { acc += cor; upper += keep; }
        else if (keep) {
            Rec24 r; r.bin1 = g - base; r.bin2 = j - base; r.IF = rf * cor;
            a.rec[o++] = r;
        }
    }
    if (PASS == CSR_ROWSUM) {
        double s = pow(acc, 2.0 / 3.0);
        if (s == 0.0) s = 1.0;
        a.rsinv[g] = 1.0 / s;
    } else if (PASS == CSR_TOTAL) {
        a.rowtot[g] = acc;
        a.rec_ptr[g] = upper;
    }
}

// RF of matrix blockIdx.x from its row totals of Cor and its row sums of X (one CTA per matrix)
__global__ void __launch_bounds__(1024) csr_rescale_factor_kernel(SymCsrArgs a, const int64_t* __restrict__ rowsum_x) {
    const int k = blockIdx.x;
    const int64_t base = a.h_bin_off[k];
    const int n = (int)(a.h_bin_off[k + 1] - base);
    if (n == 0) return;
    vc_rescale_factor_run(a.rowtot + base, n, rowsum_x + base, n, const_cast<double*>(a.scalars) + 4 * k);
}

}  // namespace

extern "C" int64_t hc_twostep_csr_batch_work_bytes(int64_t t_nbins, int64_t h_nbins, int32_t nchrom) {
    return (int64_t)sizeof(int64_t) * (t_nbins + h_nbins) + (int64_t)sizeof(double) * (2 * t_nbins + 2 * h_nbins + 8 * (int64_t)nchrom) +
           (int64_t)sizeof(int32_t) * h_nbins + 256;
}

extern "C" int hc_twostep_csr_batch(const int64_t* t_row_ptr, const int32_t* t_cnt, const int64_t* x_row_ptr, const int32_t* x_col,
                                    const int32_t* x_cnt, const int64_t* xt_row_ptr, const int32_t* xt_col, const int32_t* xt_cnt,
                                    const int64_t* t_bin_off, const int64_t* h_bin_off, int32_t nchrom, int64_t t_nbins,
                                    int64_t h_nbins, double* alpha, uint8_t* gapflag, int32_t* gapidx, int32_t* ngap,
                                    int64_t* rec_ptr, void* records, int64_t* h_nrec, void* work, void* stream) {
    HC_REQUIRE(nchrom > 0 && t_nbins >= 0 && h_nbins == 2 * t_nbins && h_nrec != nullptr, "sizes (h_nbins = 2 t_nbins)");
    HC_REQUIRE(t_row_ptr && x_row_ptr && xt_row_ptr && t_bin_off && h_bin_off && alpha && gapflag && gapidx && ngap && rec_ptr &&
               records && work, "null pointer");      // col / cnt arrays of an empty CSR may be NULL
    HC_REQUIRE(h_nbins < (1ll << 31), "column indices are int32");
    cudaStream_t s = (cudaStream_t)stream;
    *h_nrec = 0;
    if (t_nbins == 0) return HC_OK;
    int64_t* rs_t = reinterpret_cast<int64_t*>(work);
    int64_t* rs_h = rs_t + t_nbins;
    double* awork = reinterpret_cast<double*>(rs_h + h_nbins);
    double* rsinv = awork + 2 * t_nbins;
    double* rowtot = rsinv + h_nbins;
    double* scalars = rowtot + h_nbins;
    int32_t* nz_h = reinterpret_cast<int32_t*>(scalars + 8 * (int64_t)nchrom);

    csr_rowstats_kernel<<<(unsigned)((t_nbins * 32 + 255) / 256), 256, 0, s>>>(t_row_ptr, t_cnt, t_nbins, rs_t, nullptr);
    HC_LAUNCH_CHECK();
    csr_rowstats_kernel<<<(unsigned)((h_nbins * 32 + 255) / 256), 256, 0, s>>>(x_row_ptr, x_cnt, h_nbins, rs_h, nz_h);
    HC_LAUNCH_CHECK();
    AlphaArgs aa;
    aa.rs_t = rs_t; aa.rs_m = rs_h; aa.rs_p = rs_h; aa.nnz_a = nz_h; aa.nnz_b = nz_h; aa.n = 0; aa.ncols = 0;
    aa.gap_mode = HC_GAP_PERCENTILE; aa.alpha = alpha; aa.gf_a = gapflag; aa.gf_b = gapflag; aa.gi_a = gapidx; aa.gi_b = gapidx;
    aa.ngap = ngap; aa.work = awork; aa.q25 = 25.0 / 100.0; aa.q20 = 20.0 / 100.0;
    aa.t_bin_off = t_bin_off; aa.h_bin_off = h_bin_off; aa.nchrom = nchrom;
    twostep_alpha_kernel<<<nchrom, 1024, 0, s>>>(aa);
    HC_LAUNCH_CHECK();

    SymCsrArgs a;
    a.x_ptr = x_row_ptr; a.x_col = x_col; a.x_cnt = x_cnt; a.xt_ptr = xt_row_ptr; a.xt_col = xt_col; a.xt_cnt = xt_cnt;
    a.t_bin_off = t_bin_off; a.h_bin_off = h_bin_off; a.nchrom = nchrom; a.h_nbins = h_nbins;
    a.alpha = alpha; a.gapflag = gapflag; a.ngap = ngap; a.rsinv = rsinv; a.rowtot = rowtot; a.scalars = scalars;
    a.rec_ptr = rec_ptr; a.rec = reinterpret_cast<Rec24*>(records);
    const unsigned rows = (unsigned)((h_nbins + 255) / 256);
    sym_csr_kernel<CSR_ROWSUM><<<rows, 256, 0, s>>>(a);
    HC_LAUNCH_CHECK();
    sym_csr_kernel<CSR_TOTAL><<<rows, 256, 0, s>>>(a);
    HC_LAUNCH_CHECK();
    if (hc_exclusive_scan_i64(rec_ptr, h_nbins, s) != HC_OK) return HC_ERR_CUDA;
    csr_rescale_factor_kernel<<<(unsigned)(2 * nchrom), 1024, 0, s>>>(a, rs_h);
    HC_LAUNCH_CHECK();
    sym_csr_kernel<CSR_EMIT><<<rows, 256, 0, s>>>(a);
    HC_LAUNCH_CHECK();
    HC_CUDA(cudaMemcpyAsync(h_nrec, rec_ptr + h_nbins, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    HC_CUDA(cudaStreamSynchronize(s));
    return HC_OK;
}


// =========================================================================================
// Standalone building blocks with the reference's own granularity (SURVEY.md section 8b lists
// Correct_VC(X, alpha) among the signatures to keep; TwoStepCorrection above fuses all of them).
// These work on float64 matrices -- what the reference functions receive in TwoStepCorrection
// (MM / alpha[:,None] is float) -- and on any rectangular shape where the reference allows one.
// =========================================================================================
namespace {

// non-zero count per row of a float64 matrix: Coverage_M / Gap_defined (matrixBuilding.py:904-929)
__global__ void __launch_bounds__(256)
rownnz_f64_kernel(const double* __restrict__ M, int64_t ld, int nrows, int ncols, int32_t* __restrict__ rownnz) {
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (r >= nrows) return;
    const double* row = M + (int64_t)r * ld;
    int c = 0;
    for (int j = lane; j < ncols; j += 32) c += (row[j] != 0.0);     // NaN != 0 -> counted, as (i == 0).sum() does
    c = warp_sum_i(c);
    if (lane == 0) rownnz[r] = c;
}

// coverage -> gap flags -> ascending gap index list, one CTA (same code path as twostep_alpha_kernel)
__global__ void __launch_bounds__(1024)
gap_rows_kernel(const int32_t* __restrict__ nnz, int n, int ncols, int gap_mode, double q25, double* __restrict__ cov,
                uint8_t* __restrict__ gf, int32_t* __restrict__ gi, int32_t* __restrict__ ngap) {
    __shared__ HcSelectSmem sm;
    gap_rows(nnz, n, ncols, gap_mode, q25, cov, gf, &sm);
    compact_flags(gf, n, gi, ngap);
}

// Trans2symmetry (matrixBuilding.py:945-979) / Trans2symmetryLowRes (:770-776) on a float64 matrix:
// 32 x 32 output tile per CTA; the mirrored input tile is read coalesced and transposed through shared memory
__global__ void __launch_bounds__(256)
trans2sym_f64_kernel(const double* __restrict__ S, int64_t ld, int n, const uint8_t* __restrict__ gapflag,
                     double* __restrict__ out, int64_t ld_out) {
    __shared__ double tb[32][33];
    const int r0 = blockIdx.y * 32, c0 = blockIdx.x * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int rr = c0 + ty + 8 * a, cc = r0 + tx;          // tile (J, I)
        tb[ty + 8 * a][tx] = (rr < n && cc < n) ? S[(int64_t)rr * ld + cc] : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        const int i = r0 + ty + 8 * a, j = c0 + tx;
        if (i < n && j < n) {
            const double sij = S[(int64_t)i * ld + j], sji = tb[tx][ty + 8 * a];
            double v;
            if (i == j) v = sij;
            else if (gapflag == nullptr) v = sij + sji;
            else if (gapflag[i] && gapflag[j]) v = fmax(sij, sji);
            else v = (sij + sji) / 2.0;
            out[(int64_t)i * ld_out + j] = v;
        }
    }
}

// Correct_VC (matrixBuilding.py:780-790): row sums (one warp per row, fixed order)
__global__ void __launch_bounds__(256)
rowsum_f64_kernel(const double* __restrict__ X, int64_t ld, int nrows, int ncols, double* __restrict__ rs) {
    const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (r >= nrows) return;
    const double* row = X + (int64_t)r * ld;
    double s = 0.0;
    for (int j = lane; j < ncols; j += 32) s += row[j];
    s = warp_sum(s);
    if (lane == 0) rs[r] = s;
}
// column sums: partial sums over chunks of 128 rows (coalesced across columns), then a fixed-order reduction
constexpr int VC_ROWS = 128;
__global__ void __launch_bounds__(256)
colsum_partial_f64_kernel(const double* __restrict__ X, int64_t ld, int nrows, int ncols, double* __restrict__ part) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= ncols) return;
    const int r0 = blockIdx.y * VC_ROWS, r1 = min(nrows, r0 + VC_ROWS);
    double s = 0.0;
    for (int r = r0; r < r1; ++r) s += X[(int64_t)r * ld + j];
    part[(int64_t)blockIdx.y * ncols + j] = s;
}
// s = sum^alpha, zeros -> 1
__global__ void __launch_bounds__(256)
vc_pow_kernel(double* __restrict__ rs, int nrows, const double* __restrict__ part, int nchunks, int ncols,
              double* __restrict__ cs, double alpha) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < nrows) {
        double s = pow(rs[i], alpha);
        if (s == 0.0) s = 1.0;
        rs[i] = s;
    } else if (i - nrows < ncols) {
        const int j = i - nrows;
        double s = 0.0;
        for (int k = 0; k < nchunks; ++k) s += part[(int64_t)k * ncols + j];
        s = pow(s, alpha);
        if (s == 0.0) s = 1.0;
        cs[j] = s;
    }
}
__global__ void __launch_bounds__(256)
vc_apply_f64_kernel(const double* __restrict__ X, int64_t ld, int nrows, int ncols, const double* __restrict__ rs,
                    const double* __restrict__ cs, double* __restrict__ out, int64_t ld_out) {
    const int j = blockIdx.x * blockDim.x + threadIdx.x, i = blockIdx.y;
    if (j < ncols && i < nrows) out[(int64_t)i * ld_out + j] = X[(int64_t)i * ld + j] / (cs[j] * rs[i]);
}

}  // namespace

extern "C" int hc_rownnz_f64(const double* M, int64_t ld, int32_t nrows, int32_t ncols, int32_t* rownnz, void* stream) {
    HC_REQUIRE(nrows >= 0 && ncols >= 0 && ld >= ncols && rownnz != nullptr, "shape");
    if (nrows == 0) return HC_OK;
    rownnz_f64_kernel<<<(unsigned)(((int64_t)nrows * 32 + 255) / 256), 256, 0, (cudaStream_t)stream>>>(M, ld, nrows, ncols, rownnz);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_gap_rows(const int32_t* rownnz, int32_t n, int32_t ncols, int32_t gap_mode, double* coverage,
                           uint8_t* gapflag, int32_t* gapidx, int32_t* ngap, void* stream) {
    HC_REQUIRE(n > 0 && ncols > 0 && rownnz && coverage && gapflag && gapidx && ngap, "arguments");
    HC_REQUIRE(gap_mode == HC_GAP_PERCENTILE || gap_mode == HC_GAP_FIXED, "gap_mode");
    gap_rows_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(rownnz, n, ncols, gap_mode, 25.0 / 100.0, coverage, gapflag, gapidx, ngap);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_trans2symmetry_f64(const double* S, int64_t ld, int32_t n, const uint8_t* gapflag, double* out,
                                     int64_t ld_out, void* stream) {
    HC_REQUIRE(n > 0 && ld >= n && ld_out >= n && S != nullptr && out != nullptr && S != out, "shape / aliasing");
    const dim3 grid((n + 31) / 32, (n + 31) / 32);
    trans2sym_f64_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(S, ld, n, gapflag, out, ld_out);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int64_t hc_correct_vc_work_bytes(int32_t nrows, int32_t ncols) {
    const int64_t nchunks = (nrows + VC_ROWS - 1) / VC_ROWS;
    return (int64_t)sizeof(double) * ((int64_t)nrows + ncols + nchunks * ncols + 8);
}

extern "C" int hc_correct_vc_f64(const double* X, int64_t ld, int32_t nrows, int32_t ncols, double alpha, double* out,
                                 int64_t ld_out, void* work, void* stream) {
    HC_REQUIRE(nrows > 0 && ncols > 0 && ld >= ncols && ld_out >= ncols && X && out && work, "arguments");
    cudaStream_t s = (cudaStream_t)stream;
    const int nchunks = (nrows + VC_ROWS - 1) / VC_ROWS;
    double* rs = reinterpret_cast<double*>(work);
    double* cs = rs + nrows;
    double* part = cs + ncols;
    rowsum_f64_kernel<<<(unsigned)(((int64_t)nrows * 32 + 255) / 256), 256, 0, s>>>(X, ld, nrows, ncols, rs);
    HC_LAUNCH_CHECK();
    colsum_partial_f64_kernel<<<dim3((ncols + 255) / 256, nchunks), 256, 0, s>>>(X, ld, nrows, ncols, part);
    HC_LAUNCH_CHECK();
    vc_pow_kernel<<<(nrows + ncols + 255) / 256, 256, 0, s>>>(rs, nrows, part, nchunks, ncols, cs, alpha);
    HC_LAUNCH_CHECK();
    vc_apply_f64_kernel<<<dim3((ncols + 255) / 256, nrows), 256, 0, s>>>(X, ld, nrows, ncols, rs, cs, out, ld_out);
    HC_LAUNCH_CHECK();
    return HC_OK;
}
