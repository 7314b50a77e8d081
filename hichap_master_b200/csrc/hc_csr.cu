// (a) sort path: valid pairs -> (row, col) bin keys -> radix sort (hc_sort.cu) -> run-length
// reduce-by-key -> SYMMETRIC CSR with integer counts (both triangles stored, so an ICE
// iteration is a pure row-wise segmented reduction: no atomics, deterministic, and each rank
// of a row-block-sharded matrix owns complete marginals for its rows).
// Replaces the dense np.zeros((Sum,Sum)) accumulation of matrixBuilding.py:559-603 where the
// dense matrix is infeasible (genome-wide 10 kb / 5 kb: 738 GB / 2.95 TB as int64).
// The reference's upper-triangular (bin1, bin2, count) records (matrixBuilding.py:489-503)
// are the col >= row subset of this CSR (hc_csr_upper_records).
#include "hc_common.cuh"
#include <algorithm>

namespace {

constexpr unsigned long long PAD_KEY = ~0ull;
constexpr int RLE_THREADS = 256;
constexpr int RLE_ITEMS = 16;
constexpr int RLE_TILE = RLE_THREADS * RLE_ITEMS;

// ---- pairs -> keys ---------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pairs_to_keys_kernel(const int32_t* __restrict__ c1, const int32_t* __restrict__ p1, const int32_t* __restrict__ c2,
                     const int32_t* __restrict__ p2, long long npairs, FastDiv res,
                     const int64_t* __restrict__ start, const int32_t* __restrict__ chrom_bins, int nchrom,
                     int cis_only, int col_bits, unsigned long long* __restrict__ keys,
                     unsigned long long* __restrict__ n_valid, unsigned long long* __restrict__ oob) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned long long local_valid = 0, local_oob = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npairs; i += stride) {
        unsigned long long k0 = PAD_KEY, k1 = PAD_KEY;
        const int a = c1[i], b = c2[i];
        if (a >= 0 && b >= 0 && a < nchrom && b < nchrom && (!cis_only || a == b)) {
            const int x = p1[i], y = p2[i];
            const long long ba = x >= 0 ? (long long)fast_div((uint32_t)x, res) : -1;
            const long long bb = y >= 0 ? (long long)fast_div((uint32_t)y, res) : -1;
            if (ba < 0 || bb < 0 || ba >= chrom_bins[a] || bb >= chrom_bins[b]) {
                ++local_oob;
            } else {
                const unsigned long long r = (unsigned long long)(ba + start[a]);
                const unsigned long long c = (unsigned long long)(bb + start[b]);
                k0 = (r << col_bits) | c;
                if (r != c) k1 = (c << col_bits) | r;
                local_valid += (r != c) ? 2 : 1;
            }
        }
        keys[2 * i] = k0;
        keys[2 * i + 1] = k1;
    }
    local_valid = (unsigned long long)warp_sum_ll((long long)local_valid);
    local_oob = (unsigned long long)warp_sum_ll((long long)local_oob);
    if ((threadIdx.x & 31) == 0) {
        if (local_valid) atomicAdd(n_valid, local_valid);
        if (local_oob && oob) atomicAdd(oob, local_oob);
    }
}

// ---- run-length reduce-by-key ------------------------------------------------------------
// heads per tile (a head = first key of a run of equal keys; padding keys sort last and are
// cut off by n_valid)
__global__ void __launch_bounds__(RLE_THREADS)
rle_count_kernel(const unsigned long long* __restrict__ keys, const unsigned long long* __restrict__ n_valid_p,
                 int64_t* __restrict__ tile_heads) {
    __shared__ long long red[32];
    const long long m = (long long)*n_valid_p;
    const long long base = (long long)blockIdx.x * RLE_TILE;
    long long c = 0;
    for (int j = threadIdx.x; j < RLE_TILE; j += RLE_THREADS) {
        const long long i = base + j;
        if (i < m) c += (i == 0) || (keys[i] != keys[i - 1]);
    }
    c = block_sum_ll(c, red);
    if (threadIdx.x == 0) tile_heads[blockIdx.x] = c;
}

// single-CTA exclusive scan (in place), total appended at v[n]
__global__ void __launch_bounds__(1024) csr_exclusive_scan_kernel(int64_t* __restrict__ v, long long n) {
    __shared__ long long warp_tot[32];
    __shared__ long long carry_s;
    if (threadIdx.x == 0) carry_s = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (long long base = 0; base < n; base += 1024) {
        const long long i = base + threadIdx.x;
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

// unique keys + head positions, in sorted order.  Block-local ordered compaction.
__global__ void __launch_bounds__(RLE_THREADS)
rle_emit_kernel(const unsigned long long* __restrict__ keys, const unsigned long long* __restrict__ n_valid_p,
                const int64_t* __restrict__ tile_off, unsigned long long* __restrict__ ukey,
                int64_t* __restrict__ upos) {
    __shared__ int wtot[RLE_THREADS / 32];
    __shared__ long long run_s;
    const long long m = (long long)*n_valid_p;
    const long long base = (long long)blockIdx.x * RLE_TILE;
    if (threadIdx.x == 0) run_s = tile_off[blockIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int j0 = 0; j0 < RLE_TILE; j0 += RLE_THREADS) {   // consecutive threads = consecutive keys
        const long long i = base + j0 + threadIdx.x;
        unsigned long long k = 0;
        bool head = false;
        if (i < m) { k = keys[i]; head = (i == 0) || (k != keys[i - 1]); }
        const unsigned b = __ballot_sync(0xffffffffu, head);
        if (lane == 0) wtot[wid] = __popc(b);
        __syncthreads();
        long long off = run_s;
        for (int w = 0; w < wid; ++w) off += wtot[w];
        if (head) { const long long u = off + __popc(b & ((1u << lane) - 1u)); ukey[u] = k; upos[u] = i; }
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < RLE_THREADS / 32; ++w) t += wtot[w]; run_s += t; }
        __syncthreads();
    }
}

// (col, count) per unique key and the row pointer
__global__ void __launch_bounds__(256)
csr_finish_kernel(const unsigned long long* __restrict__ ukey, const int64_t* __restrict__ upos, long long nnz,
                  const unsigned long long* __restrict__ n_valid_p, int col_bits, long long row0, long long nrows,
                  int64_t* __restrict__ row_ptr, int32_t* __restrict__ col, int32_t* __restrict__ cnt) {
    const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nnz) {
        if (u == nnz && nnz == 0) for (long long r = 0; r <= nrows; ++r) row_ptr[r] = 0;   // empty matrix
        return;
    }
    const unsigned long long k = ukey[u];
    const long long row = (long long)(k >> col_bits) - row0;
    col[u] = (int32_t)(k & ((1ull << col_bits) - 1ull));
    const long long next = (u + 1 < nnz) ? upos[u + 1] : (long long)*n_valid_p;
    cnt[u] = (int32_t)(next - upos[u]);
    const long long prev_row = u == 0 ? -1 : (long long)(ukey[u - 1] >> col_bits) - row0;
    for (long long r = prev_row + 1; r <= row; ++r) row_ptr[r] = u;     // rows (prev_row, row] start here
    if (u == nnz - 1) for (long long r = row + 1; r <= nrows; ++r) row_ptr[r] = nnz;
}

// upper-triangular records of the symmetric CSR (col >= row), row-major: count then emit
__global__ void __launch_bounds__(256)
csr_upper_count_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col, long long row0,
                       long long nrows, int64_t* __restrict__ out_cnt) {
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= nrows) return;
    int c = 0;
    for (long long e = row_ptr[r] + lane; e < row_ptr[r + 1]; e += 32) c += col[e] >= r + row0;
    c = warp_sum_i(c);
    if (lane == 0) out_cnt[r] = c;
}

__global__ void __launch_bounds__(256)
csr_upper_emit_kernel(const int64_t* __restrict__ row_ptr, const int32_t* __restrict__ col,
                      const int32_t* __restrict__ cnt, long long row0, long long nrows,
                      const int64_t* __restrict__ out_ptr,
                      int32_t* __restrict__ bin1, int32_t* __restrict__ bin2, int32_t* __restrict__ val) {
    const long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (r >= nrows) return;
    long long out = out_ptr[r];
    const long long e1 = row_ptr[r + 1];
    for (long long e0 = row_ptr[r]; e0 < e1; e0 += 32) {
        const long long e = e0 + lane;
        const bool keep = e < e1 && col[e] >= r + row0;
        const unsigned b = __ballot_sync(0xffffffffu, keep);
        if (keep) {
            const long long o = out + __popc(b & ((1u << lane) - 1u));
            bin1[o] = (int32_t)(r + row0); bin2[o] = col[e]; val[o] = cnt[e];
        }
        out += __popc(b);
    }
}


// =========================================================================================
// One key per pair ("entries"): a 64-bit entry is  (row << (col_bits + cnt_bits)) | (col << cnt_bits) | count.
// A pair contributes ONE entry of its upper-triangle cell (row <= col, count 1); after the sort and the
// reduce-by-key the unique upper cells carry their counts in the low bits.  The lower triangle is the same list
// with row and col swapped: it is already ordered by its new minor key, so a stable LSD sort over the new row
// bits alone (3 digit passes over the unique cells instead of 5 passes over a second key per pair) orders it, and
// the symmetric CSR is the row-wise concatenation lower part | upper part of the two lists.
// =========================================================================================
__device__ __forceinline__ unsigned long long pair_entry(int a, int x, int b, int y, FastDiv res, const int64_t* __restrict__ start,
                                                        const int32_t* __restrict__ chrom_bins, int nchrom, int cis_only,
                                                        int col_bits, int cnt_bits, unsigned long long& n_valid,
                                                        unsigned long long& n_oob) {
    if (a < 0 || b < 0 || a >= nchrom || b >= nchrom || (cis_only && a != b)) return PAD_KEY;
    const long long ba = x >= 0 ? (long long)fast_div((uint32_t)x, res) : -1;
    const long long bb = y >= 0 ? (long long)fast_div((uint32_t)y, res) : -1;
    if (ba < 0 || bb < 0 || ba >= chrom_bins[a] || bb >= chrom_bins[b]) { ++n_oob; return PAD_KEY; }
    const unsigned long long r = (unsigned long long)(ba + start[a]);
    const unsigned long long c = (unsigned long long)(bb + start[b]);
    const unsigned long long lo = r < c ? r : c, hi = r < c ? c : r;
    ++n_valid;
    return (((lo << col_bits) | hi) << cnt_bits) | 1ull;
}

// VEC: four pairs per thread and trip through 128-bit loads (64 B of loads in flight per thread; one pair per trip left the
// kernel at 2.5 TB/s); needs 16-byte aligned columns, checked by the launcher.
template <bool VEC>
__global__ void __launch_bounds__(256)
pairs_to_entries_kernel(const int32_t* __restrict__ c1, const int32_t* __restrict__ p1, const int32_t* __restrict__ c2,
                        const int32_t* __restrict__ p2, long long npairs, FastDiv res,
                        const int64_t* __restrict__ start, const int32_t* __restrict__ chrom_bins, int nchrom,
                        int cis_only, int col_bits, int cnt_bits, unsigned long long* __restrict__ entries,
                        unsigned long long* __restrict__ n_valid, unsigned long long* __restrict__ oob) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long local_valid = 0, local_oob = 0;
    long long done = 0;
    if (VEC) {
        const long long nvec = npairs >> 2;
        for (long long v = t; v < nvec; v += stride) {
            const int4 a = ld_stream_v4(c1 + 4 * v), x = ld_stream_v4(p1 + 4 * v), b = ld_stream_v4(c2 + 4 * v), y = ld_stream_v4(p2 + 4 * v);
            ulonglong2 e0, e1;
            e0.x = pair_entry(a.x, x.x, b.x, y.x, res, start, chrom_bins, nchrom, cis_only, col_bits, cnt_bits, local_valid, local_oob);
            e0.y = pair_entry(a.y, x.y, b.y, y.y, res, start, chrom_bins, nchrom, cis_only, col_bits, cnt_bits, local_valid, local_oob);
            e1.x = pair_entry(a.z, x.z, b.z, y.z, res, start, chrom_bins, nchrom, cis_only, col_bits, cnt_bits, local_valid, local_oob);
            e1.y = pair_entry(a.w, x.w, b.w, y.w, res, start, chrom_bins, nchrom, cis_only, col_bits, cnt_bits, local_valid, local_oob);
            reinterpret_cast<ulonglong2*>(entries)[2 * v] = e0;
            reinterpret_cast<ulonglong2*>(entries)[2 * v + 1] = e1;
        }
        done = nvec << 2;
    }
    for (long long i = done + t; i < npairs; i += stride)
        entries[i] = pair_entry(c1[i], p1[i], c2[i], p2[i], res, start, chrom_bins, nchrom, cis_only, col_bits, cnt_bits,
                                local_valid, local_oob);
    local_valid = (unsigned long long)warp_sum_ll((long long)local_valid);
    local_oob = (unsigned long long)warp_sum_ll((long long)local_oob);
    if ((threadIdx.x & 31) == 0) {
        if (local_valid) atomicAdd(n_valid, local_valid);
        if (local_oob && oob) atomicAdd(oob, local_oob);
    }
}

// Directed entries of the allelic haplotype matrices (cis pairs of an M_M or P_P bed).  Same cells as the tile updates of
// hc_bin.cu: a Both pair (mark 0) counts at (b1, b2) and, off the diagonal, at (b2, b1) -- HC_BIN_SYM_BOTH; with `onesided`, an
// R1 pair (mark 1) counts at (b1, b2) and a pair with any other non-zero mark at (b2, b1) -- HC_BIN_ONESIDED.  Two entry slots
// per pair; an unused slot holds the padding key.
__device__ __forceinline__ void directed_entries(int a, int x, int b, int y, int mk, FastDiv res, const int64_t* __restrict__ start,
                                                 const int32_t* __restrict__ chrom_bins, int nchrom, int onesided, int col_bits,
                                                 int cnt_bits, unsigned long long& e0, unsigned long long& e1,
                                                 unsigned long long& n_valid, unsigned long long& n_oob) {
    e0 = e1 = PAD_KEY;
    if (a < 0 || b < 0 || a >= nchrom || b >= nchrom) return;          // filtered chromosome
    if (mk != 0 && !onesided) return;
    if (a != b) return;                                                // cis only
    if (x < 0 || y < 0) { ++n_oob; return; }
    const long long ba = fast_div((uint32_t)x, res), bb = fast_div((uint32_t)y, res);
    if (ba >= chrom_bins[a] || bb >= chrom_bins[a]) { ++n_oob; return; }
    const unsigned long long r = (unsigned long long)(ba + start[a]), c = (unsigned long long)(bb + start[a]);
    const unsigned long long rc = (((r << col_bits) | c) << cnt_bits) | 1ull, cr = (((c << col_bits) | r) << cnt_bits) | 1ull;
    if (mk == 0) { e0 = rc; if (r != c) e1 = cr; }
    else e0 = mk == 1 ? rc : cr;
    n_valid += 1 + (e1 != PAD_KEY);
}

__global__ void __launch_bounds__(256)
pairs_to_directed_entries_kernel(const int32_t* __restrict__ c1, const int32_t* __restrict__ p1, const int32_t* __restrict__ c2,
                                 const int32_t* __restrict__ p2, const uint8_t* __restrict__ mark, long long npairs, FastDiv res,
                                 const int64_t* __restrict__ start, const int32_t* __restrict__ chrom_bins, int nchrom,
                                 int onesided, int col_bits, int cnt_bits, unsigned long long* __restrict__ entries,
                                 unsigned long long* __restrict__ n_valid, unsigned long long* __restrict__ oob) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    unsigned long long local_valid = 0, local_oob = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < npairs; i += stride) {
        ulonglong2 e;
        directed_entries(c1[i], p1[i], c2[i], p2[i], mark[i], res, start, chrom_bins, nchrom, onesided, col_bits, cnt_bits, e.x, e.y,
                         local_valid, local_oob);
        reinterpret_cast<ulonglong2*>(entries)[i] = e;
    }
    local_valid = (unsigned long long)warp_sum_ll((long long)local_valid);
    local_oob = (unsigned long long)warp_sum_ll((long long)local_oob);
    if ((threadIdx.x & 31) == 0) {
        if (local_valid) atomicAdd(n_valid, local_valid);
        if (local_oob && oob) atomicAdd(oob, local_oob);
    }
}

// heads per tile on the cell bits (entry >> cnt_bits)
__global__ void __launch_bounds__(RLE_THREADS)
ent_count_kernel(const unsigned long long* __restrict__ ent, const unsigned long long* __restrict__ n_valid_p,
                 int cnt_bits, int64_t* __restrict__ tile_heads) {
    __shared__ long long red[32];
    const long long m = (long long)*n_valid_p;
    const long long base = (long long)blockIdx.x * RLE_TILE;
    long long c = 0;
    for (int j = threadIdx.x; j < RLE_TILE; j += RLE_THREADS) {
        const long long i = base + j;
        if (i < m) c += (i == 0) || ((ent[i] >> cnt_bits) != (ent[i - 1] >> cnt_bits));
    }
    c = block_sum_ll(c, red);
    if (threadIdx.x == 0) tile_heads[blockIdx.x] = c;
}

// position of every head, in order (block-local ordered compaction, like rle_emit_kernel)
__global__ void __launch_bounds__(RLE_THREADS)
ent_heads_kernel(const unsigned long long* __restrict__ ent, const unsigned long long* __restrict__ n_valid_p,
                 int cnt_bits, const int64_t* __restrict__ tile_off, int64_t* __restrict__ upos) {
    __shared__ int wtot[RLE_THREADS / 32];
    __shared__ long long run_s;
    const long long m = (long long)*n_valid_p;
    const long long base = (long long)blockIdx.x * RLE_TILE;
    if (threadIdx.x == 0) run_s = tile_off[blockIdx.x];
    __syncthreads();
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    for (int j0 = 0; j0 < RLE_TILE; j0 += RLE_THREADS) {
        const long long i = base + j0 + threadIdx.x;
        bool head = false;
        if (i < m) head = (i == 0) || ((ent[i] >> cnt_bits) != (ent[i - 1] >> cnt_bits));
        const unsigned b = __ballot_sync(0xffffffffu, head);
        if (lane == 0) wtot[wid] = __popc(b);
        __syncthreads();
        long long off = run_s;
        for (int w = 0; w < wid; ++w) off += wtot[w];
        if (head) upos[off + __popc(b & ((1u << lane) - 1u))] = i;
        __syncthreads();
        if (threadIdx.x == 0) { int t = 0; for (int w = 0; w < RLE_THREADS / 32; ++w) t += wtot[w]; run_s += t; }
        __syncthreads();
    }
}

// one reduced entry per run.  unit != 0: every input count is 1, so the run length is the count; otherwise the
// counts of the run are added (runs are then short: at most one entry per contributing rank).
__global__ void __launch_bounds__(256)
ent_reduce_kernel(const unsigned long long* __restrict__ ent, const int64_t* __restrict__ upos, long long nuniq,
                  const unsigned long long* __restrict__ n_valid_p, int cnt_bits, int unit,
                  unsigned long long* __restrict__ out, int32_t* __restrict__ overflow) {
    const long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (u >= nuniq) return;
    const long long p0 = upos[u], p1 = (u + 1 < nuniq) ? upos[u + 1] : (long long)*n_valid_p;
    const unsigned long long mask = (1ull << cnt_bits) - 1ull;
    const unsigned long long e = ent[p0];
    unsigned long long cnt;
    if (unit) cnt = (unsigned long long)(p1 - p0);
    else { cnt = 0; for (long long p = p0; p < p1; ++p) cnt += ent[p] & mask; }
    if (cnt > mask) { atomicOr(overflow, 1); cnt = mask; }
    out[u] = (e & ~mask) | cnt;
}

// ---- reduce (+ transpose) in one pass over the sorted entries, given the scanned per-tile head counts ---------------
// A warp owns 16 x 32 consecutive entries (item k of a lane = entry wbase + 32 k + lane: coalesced).  Head flags come from
// ballots; a head's run ends at the next head, found in the 16 ballot masks (backward sweep) or, for the last head of the
// warp's chunk, by a galloping + binary search in the sorted array (a hot diagonal cell holds thousands of pairs).  The
// head writes the reduced entry -- and, when `lo` is given, the swapped one -- at tile_off + rank: no list of head
// positions is written or read back (that list cost 3.8 GB each way, and the look-back version of the head scan sat at a
// barrier for 60 % of its samples: profiles/r2z_ncu_heads_scan_v1.json).
template <bool UNIT, bool LOWER>
__global__ void __launch_bounds__(RLE_THREADS)
ent_emit_kernel(const unsigned long long* __restrict__ ent, const unsigned long long* __restrict__ n_valid_p, int cnt_bits,
                const int64_t* __restrict__ tile_off, unsigned long long* __restrict__ out, unsigned long long* __restrict__ lo,
                int col_bits, unsigned long long* __restrict__ n_lo, int32_t* __restrict__ overflow) {
    __shared__ int wtot[RLE_THREADS / 32];
    const long long m = (long long)*n_valid_p;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long wbase = (long long)blockIdx.x * RLE_TILE + (long long)wid * (32 * RLE_ITEMS);
    const long long wend = wbase + 32 * RLE_ITEMS;
    const unsigned long long vmask = (1ull << cnt_bits) - 1ull;
    unsigned long long e[RLE_ITEMS];
#pragma unroll
    for (int k = 0; k < RLE_ITEMS; ++k) {
        const long long i = wbase + 32 * k + lane;
        e[k] = i < m ? ent[i] : 0ull;
    }
    // the entry before the chunk and the 32 entries behind it (the run of the chunk's last head usually ends there)
    unsigned long long carry = (lane == 0 && wbase > 0 && wbase < m) ? ent[wbase - 1] >> cnt_bits : 0ull;
    const unsigned long long beyond = wend + lane < m ? ent[wend + lane] >> cnt_bits : ~0ull;
    unsigned bal[RLE_ITEMS];
    int cnt = 0;
#pragma unroll
    for (int k = 0; k < RLE_ITEMS; ++k) {
        const long long i = wbase + 32 * k + lane;
        const unsigned long long c = e[k] >> cnt_bits;
        unsigned long long prev = __shfl_up_sync(0xffffffffu, c, 1);
        if (lane == 0) prev = carry;
        bal[k] = __ballot_sync(0xffffffffu, i < m && (i == 0 || c != prev));
        carry = __shfl_sync(0xffffffffu, c, 31);         // after the loop: the cell of the chunk's last entry
        cnt += __popc(bal[k]);
    }
    // where the run of the chunk's LAST head ends (warp-uniform): the first entry behind the chunk with another cell
    long long chunk_run_end;
    {
        const unsigned differs = __ballot_sync(0xffffffffu, beyond != carry);     // entries past m count as different
        if (wend >= m) chunk_run_end = m;
        else if (differs) chunk_run_end = wend + (__ffs(differs) - 1);
        else {                                             // a long run (hot diagonal cell): gallop, then bisect
            long long known = wend + 31, q = known + 1, step = 32;
            while (q < m && (ent[q] >> cnt_bits) == carry) { known = q; q += step; step <<= 1; }
            long long hi = q < m ? q : m;
            while (hi - known > 1) {
                const long long mid = known + ((hi - known) >> 1);
                if ((ent[mid] >> cnt_bits) == carry) known = mid; else hi = mid;
            }
            chunk_run_end = hi;
        }
    }
    if (lane == 0) wtot[wid] = cnt;
    __syncthreads();
    long long o = tile_off[blockIdx.x];
#pragma unroll
    for (int w = 0; w < RLE_THREADS / 32; ++w) if (w < wid) o += wtot[w];
    o += cnt;                                            // one past the warp's last head; the sweep below runs backward
    const unsigned gt = lane == 31 ? 0u : (0xffffffffu << (lane + 1));
    long long next_head = chunk_run_end;                 // end of a run that no later head of the chunk closes
    long long kept = 0;
    const unsigned long long cmask = (1ull << col_bits) - 1ull;
#pragma unroll
    for (int k = RLE_ITEMS - 1; k >= 0; --k) {
        o -= __popc(bal[k]);
        if ((bal[k] >> lane) & 1u) {
            const long long i = wbase + 32 * k + lane;
            const unsigned long long cell = e[k] >> cnt_bits;
            const unsigned above = bal[k] & gt;
            const long long end = above ? wbase + 32 * k + (__ffs(above) - 1) : next_head;
            unsigned long long c;
            if (UNIT) c = (unsigned long long)(end - i);
            else { c = e[k] & vmask; for (long long q = i + 1; q < end; ++q) c += ent[q] & vmask; }
            if (c > vmask) { atomicOr(overflow, 1); c = vmask; }
            const long long u = o + __popc(bal[k] & ((1u << lane) - 1u));
            out[u] = (cell << cnt_bits) | c;
            if (LOWER) {
                const unsigned long long r = cell >> col_bits, cc = cell & cmask;
                const bool off = r != cc;
                lo[u] = off ? ((((cc << col_bits) | r) << cnt_bits) | c) : PAD_KEY;
                kept += off;
            }
        }
        if (bal[k]) next_head = wbase + 32 * k + (__ffs(bal[k]) - 1);
    }
    if (LOWER) {
        kept = warp_sum_ll(kept);
        if (lane == 0 && kept) atomicAdd(n_lo, (unsigned long long)kept);
    }
}

// swapped copy of the off-diagonal cells; a diagonal cell becomes the padding key (sorts last)
__global__ void __launch_bounds__(256)
ent_transpose_kernel(const unsigned long long* __restrict__ up, long long n, int col_bits, int cnt_bits,
                     unsigned long long* __restrict__ lo, unsigned long long* __restrict__ n_lo) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    const unsigned long long cmask = (1ull << col_bits) - 1ull, vmask = (1ull << cnt_bits) - 1ull;
    long long kept = 0;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < n; u += stride) {
        const unsigned long long e = up[u];
        const unsigned long long r = e >> (col_bits + cnt_bits), c = (e >> cnt_bits) & cmask;
        const bool off = r != c;
        lo[u] = off ? ((((c << col_bits) | r) << cnt_bits) | (e & vmask)) : PAD_KEY;
        kept += off;
    }
    kept = warp_sum_ll(kept);
    if ((threadIdx.x & 31) == 0 && kept) atomicAdd(n_lo, (unsigned long long)kept);
}

// ptr[r] = index of the first entry whose row is >= row0 + r, r in [0, nrows]; *n_p entries (device) or n when n_p == 0.
// One binary search per row over the sorted entries (~30 dependent L2 reads, all rows in parallel) instead of a pass over
// every entry: 0.05 ms instead of 1.0 ms at 483 M entries.
__global__ void __launch_bounds__(256)
ent_row_ptr_kernel(const unsigned long long* __restrict__ ent, const unsigned long long* __restrict__ n_p, long long n_host,
                   int row_shift, long long row0, long long nrows, int64_t* __restrict__ ptr) {
    const long long n = n_p ? (long long)*n_p : n_host;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x; r <= nrows; r += stride) {
        const unsigned long long want = (unsigned long long)(row0 + r);
        long long lo = 0, hi = n;                        // first index in [0, n] with row >= want
        while (lo < hi) {
            const long long mid = lo + ((hi - lo) >> 1);
            if ((ent[mid] >> row_shift) < want) lo = mid + 1; else hi = mid;
        }
        ptr[r] = lo;
    }
}

__global__ void __launch_bounds__(256)
ent_row_ptr_sum_kernel(const int64_t* __restrict__ a, const int64_t* __restrict__ b, long long n1, int64_t* __restrict__ out) {
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < n1) out[r] = a[r] + (b ? b[r] : 0);
}

// row r of the CSR = lower entries of row r (cols < r, ascending) followed by its upper entries (cols >= r)
__global__ void __launch_bounds__(256)
ent_scatter_kernel(const unsigned long long* __restrict__ ent, const unsigned long long* __restrict__ n_p, long long n_host,
                   int col_bits, int cnt_bits, long long row0, const int64_t* __restrict__ other_ptr, int other_next,
                   int32_t* __restrict__ col, int32_t* __restrict__ cnt) {
    const long long n = n_p ? (long long)*n_p : n_host;
    const long long stride = (long long)gridDim.x * blockDim.x;
    const unsigned long long cmask = (1ull << col_bits) - 1ull, vmask = (1ull << cnt_bits) - 1ull;
    for (long long u = (long long)blockIdx.x * blockDim.x + threadIdx.x; u < n; u += stride) {
        const unsigned long long e = ent[u];
        const long long r = (long long)(e >> (col_bits + cnt_bits)) - row0;
        const long long dst = u + (other_ptr ? other_ptr[r + other_next] : 0);
        col[dst] = (int32_t)((e >> cnt_bits) & cmask);
        cnt[dst] = (int32_t)(e & vmask);
    }
}

}  // namespace

extern "C" int hc_pairs_to_keys(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                                int64_t npairs, int32_t res, const int64_t* start, const int32_t* chrom_bins,
                                int32_t nchrom, int32_t cis_only, int32_t col_bits, unsigned long long* keys,
                                unsigned long long* n_valid, unsigned long long* oob, void* stream) {
    HC_REQUIRE(npairs >= 0 && res > 0 && nchrom > 0 && col_bits > 0 && col_bits <= 31, "sizes");
    HC_CUDA(cudaMemsetAsync(n_valid, 0, sizeof(unsigned long long), (cudaStream_t)stream));
    if (npairs == 0) return HC_OK;
    long long blocks = (npairs + 255) / 256;
    const long long cap = (long long)hc_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    pairs_to_keys_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        c1, p1, c2, p2, npairs, make_fast_div((uint32_t)res), start, chrom_bins, nchrom, cis_only, col_bits, keys, n_valid, oob);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int64_t hc_csr_work_bytes(int64_t nkeys) {
    const int64_t tiles = (nkeys + RLE_TILE - 1) / RLE_TILE;
    return (int64_t)sizeof(int64_t) * (tiles + 2);
}

// Number of distinct keys among the first *n_valid sorted keys -> *h_nnz (synchronises).
// work: hc_csr_work_bytes(nkeys); keeps the scanned per-tile offsets for hc_csr_emit.
extern "C" int hc_csr_count(const unsigned long long* sorted_keys, int64_t nkeys,
                            const unsigned long long* n_valid, void* work, int64_t* h_nnz, void* stream) {
    HC_REQUIRE(nkeys >= 0 && h_nnz != nullptr, "nkeys>=0, h_nnz");
    cudaStream_t s = (cudaStream_t)stream;
    int64_t* tile_heads = reinterpret_cast<int64_t*>(work);
    const long long tiles = (nkeys + RLE_TILE - 1) / RLE_TILE;
    *h_nnz = 0;
    if (tiles == 0) return HC_OK;
    rle_count_kernel<<<(unsigned)tiles, RLE_THREADS, 0, s>>>(sorted_keys, n_valid, tile_heads);
    HC_LAUNCH_CHECK();
    csr_exclusive_scan_kernel<<<1, 1024, 0, s>>>(tile_heads, tiles);
    HC_LAUNCH_CHECK();
    HC_CUDA(cudaMemcpyAsync(h_nnz, tile_heads + tiles, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    HC_CUDA(cudaStreamSynchronize(s));
    return HC_OK;
}

// Emit the CSR of rows [row0, row0+nrows) (every key's row must lie in that range; row_ptr is
// indexed by LOCAL row).  ukey/upos: nnz-element scratch (the free ping-pong buffer of the sort is
// large enough for both).  row_ptr: nrows+1; col, cnt: nnz.
extern "C" int hc_csr_emit(const unsigned long long* sorted_keys, int64_t nkeys, const unsigned long long* n_valid,
                           const void* work, int64_t nnz, int32_t col_bits, int64_t row0, int64_t nrows,
                           unsigned long long* ukey, int64_t* upos, int64_t* row_ptr, int32_t* col, int32_t* cnt,
                           void* stream) {
    HC_REQUIRE(nkeys >= 0 && nnz >= 0 && nrows >= 0, "sizes");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t* tile_off = reinterpret_cast<const int64_t*>(work);
    const long long tiles = (nkeys + RLE_TILE - 1) / RLE_TILE;
    if (nnz > 0) {
        rle_emit_kernel<<<(unsigned)tiles, RLE_THREADS, 0, s>>>(sorted_keys, n_valid, tile_off, ukey, upos);
        HC_LAUNCH_CHECK();
    }
    const long long blocks = (nnz + 1 + 255) / 256;
    csr_finish_kernel<<<(unsigned)blocks, 256, 0, s>>>(ukey, upos, nnz, n_valid, col_bits, row0, nrows, row_ptr, col, cnt);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

// Upper-triangular (bin1, bin2, count) records (global bins) of the local rows [row0, row0+nrows)
// of a symmetric CSR, row-major.
// Two calls like hc_dense_nonzero_*: count fills out_ptr[nrows+1] (exclusive scan), then emit.
extern "C" int hc_csr_upper_count(const int64_t* row_ptr, const int32_t* col, int64_t row0, int64_t nrows,
                                  int64_t* out_ptr, void* stream) {
    HC_REQUIRE(nrows >= 0, "nrows");
    cudaStream_t s = (cudaStream_t)stream;
    if (nrows > 0) {
        const long long blocks = (nrows * 32 + 255) / 256;
        csr_upper_count_kernel<<<(unsigned)blocks, 256, 0, s>>>(row_ptr, col, row0, nrows, out_ptr);
        HC_LAUNCH_CHECK();
    }
    csr_exclusive_scan_kernel<<<1, 1024, 0, s>>>(out_ptr, nrows);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int hc_csr_upper_emit(const int64_t* row_ptr, const int32_t* col, const int32_t* cnt, int64_t row0,
                                 int64_t nrows, const int64_t* out_ptr, int32_t* bin1, int32_t* bin2, int32_t* val, void* stream) {
    HC_REQUIRE(nrows >= 0, "nrows");
    if (nrows == 0) return HC_OK;
    const long long blocks = (nrows * 32 + 255) / 256;
    csr_upper_emit_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(row_ptr, col, cnt, row0, nrows, out_ptr,
                                                                             bin1, bin2, val);
    HC_LAUNCH_CHECK();
    return HC_OK;
}


// ---- one key per pair: entries -----------------------------------------------------------
extern "C" int hc_pairs_to_entries(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                                   int64_t npairs, int32_t res, const int64_t* start, const int32_t* chrom_bins,
                                   int32_t nchrom, int32_t cis_only, int32_t col_bits, int32_t cnt_bits,
                                   unsigned long long* entries, unsigned long long* n_valid, unsigned long long* oob,
                                   void* stream) {
    HC_REQUIRE(npairs >= 0 && res > 0 && nchrom > 0 && col_bits > 0 && cnt_bits > 0 && cnt_bits <= 31 &&
               2 * col_bits + cnt_bits <= 63, "sizes");
    HC_CUDA(cudaMemsetAsync(n_valid, 0, sizeof(unsigned long long), (cudaStream_t)stream));
    if (npairs == 0) return HC_OK;
    long long blocks = (npairs / 4 + 255) / 256 + 1;
    const long long cap = (long long)hc_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    const bool vec = ((reinterpret_cast<uintptr_t>(c1) | reinterpret_cast<uintptr_t>(p1) | reinterpret_cast<uintptr_t>(c2) |
                       reinterpret_cast<uintptr_t>(p2) | reinterpret_cast<uintptr_t>(entries)) & 15) == 0;
    if (vec)
        pairs_to_entries_kernel<true><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            c1, p1, c2, p2, npairs, make_fast_div((uint32_t)res), start, chrom_bins, nchrom, cis_only, col_bits, cnt_bits,
            entries, n_valid, oob);
    else
        pairs_to_entries_kernel<false><<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
            c1, p1, c2, p2, npairs, make_fast_div((uint32_t)res), start, chrom_bins, nchrom, cis_only, col_bits, cnt_bits,
            entries, n_valid, oob);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

// Two entries per pair (entries: 2*npairs, 16-byte aligned); *n_valid and *oob are ADDED to, so that the M_M and P_P beds can
// fill the two halves of one buffer.
extern "C" int hc_pairs_to_directed_entries(const int32_t* c1, const int32_t* p1, const int32_t* c2, const int32_t* p2,
                                            const uint8_t* mark, int64_t npairs, int32_t res, const int64_t* start,
                                            const int32_t* chrom_bins, int32_t nchrom, int32_t onesided, int32_t col_bits,
                                            int32_t cnt_bits, unsigned long long* entries, unsigned long long* n_valid,
                                            unsigned long long* oob, void* stream) {
    HC_REQUIRE(npairs >= 0 && res > 0 && nchrom > 0 && col_bits > 0 && cnt_bits > 0 && cnt_bits <= 31 &&
               2 * col_bits + cnt_bits <= 63, "sizes");
    HC_REQUIRE(n_valid != nullptr, "n_valid");
    if (npairs == 0) return HC_OK;
    HC_REQUIRE(mark != nullptr, "mark column required");
    HC_REQUIRE((reinterpret_cast<uintptr_t>(entries) & 15) == 0, "entries must be 16-byte aligned");
    long long blocks = (npairs + 255) / 256;
    const long long cap = (long long)hc_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    pairs_to_directed_entries_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
        c1, p1, c2, p2, mark, npairs, make_fast_div((uint32_t)res), start, chrom_bins, nchrom, onesided ? 1 : 0, col_bits, cnt_bits,
        entries, n_valid, oob);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

int hc_exclusive_scan_i64(int64_t* v, long long n, cudaStream_t s) {
    csr_exclusive_scan_kernel<<<1, 1024, 0, s>>>(v, n);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

// Distinct cells among the first *n_valid sorted entries -> *h_nuniq (synchronises).  work: hc_csr_work_bytes(n).
extern "C" int hc_entries_count(const unsigned long long* sorted, int64_t n, const unsigned long long* n_valid,
                                int32_t cnt_bits, void* work, int64_t* h_nuniq, void* stream) {
    HC_REQUIRE(n >= 0 && h_nuniq != nullptr && cnt_bits > 0 && cnt_bits < 64, "n>=0, h_nuniq, cnt_bits");
    cudaStream_t s = (cudaStream_t)stream;
    int64_t* tile_heads = reinterpret_cast<int64_t*>(work);
    const long long tiles = (n + RLE_TILE - 1) / RLE_TILE;
    *h_nuniq = 0;
    if (tiles == 0) return HC_OK;
    ent_count_kernel<<<(unsigned)tiles, RLE_THREADS, 0, s>>>(sorted, n_valid, cnt_bits, tile_heads);
    HC_LAUNCH_CHECK();
    csr_exclusive_scan_kernel<<<1, 1024, 0, s>>>(tile_heads, tiles);
    HC_LAUNCH_CHECK();
    HC_CUDA(cudaMemcpyAsync(h_nuniq, tile_heads + tiles, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    HC_CUDA(cudaStreamSynchronize(s));
    return HC_OK;
}

// Reduced entries out[nuniq] (count = run length when unit, else the sum of the run's counts).  upos: nuniq int64
// scratch.  *h_overflow = 1 when a count does not fit cnt_bits (synchronises).
extern "C" int hc_entries_reduce(const unsigned long long* sorted, int64_t n, const unsigned long long* n_valid,
                                 const void* work, int64_t nuniq, int32_t cnt_bits, int32_t unit, int64_t* upos,
                                 unsigned long long* out, int32_t* d_overflow, int32_t* h_overflow, void* stream) {
    HC_REQUIRE(n >= 0 && nuniq >= 0 && d_overflow != nullptr && h_overflow != nullptr, "sizes");
    cudaStream_t s = (cudaStream_t)stream;
    *h_overflow = 0;
    if (nuniq == 0) return HC_OK;
    const long long tiles = (n + RLE_TILE - 1) / RLE_TILE;
    HC_CUDA(cudaMemsetAsync(d_overflow, 0, sizeof(int32_t), s));
    ent_heads_kernel<<<(unsigned)tiles, RLE_THREADS, 0, s>>>(sorted, n_valid, cnt_bits, reinterpret_cast<const int64_t*>(work), upos);
    HC_LAUNCH_CHECK();
    ent_reduce_kernel<<<(unsigned)((nuniq + 255) / 256), 256, 0, s>>>(sorted, upos, nuniq, n_valid, cnt_bits, unit, out, d_overflow);
    HC_LAUNCH_CHECK();
    HC_CUDA(cudaMemcpyAsync(h_overflow, d_overflow, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    HC_CUDA(cudaStreamSynchronize(s));
    return HC_OK;
}

// The reduction in one pass after hc_entries_count (whose `work` holds the scanned per-tile head counts): out[nuniq], and --
// when lo != NULL -- the swapped list of hc_entries_transpose (lo[nuniq], *n_lo) from the same pass.
extern "C" int hc_entries_emit(const unsigned long long* sorted, int64_t n, const unsigned long long* n_valid, const void* work,
                               int64_t nuniq, int32_t col_bits, int32_t cnt_bits, int32_t unit, unsigned long long* out,
                               unsigned long long* lo, unsigned long long* n_lo, int32_t* d_overflow, int32_t* h_overflow,
                               void* stream) {
    HC_REQUIRE(n >= 0 && nuniq >= 0 && d_overflow != nullptr && h_overflow != nullptr && col_bits > 0 && cnt_bits > 0, "sizes");
    HC_REQUIRE(lo == nullptr || n_lo != nullptr, "n_lo");
    cudaStream_t s = (cudaStream_t)stream;
    *h_overflow = 0;
    if (lo) HC_CUDA(cudaMemsetAsync(n_lo, 0, sizeof(unsigned long long), s));
    if (nuniq == 0) return HC_OK;
    const long long tiles = (n + RLE_TILE - 1) / RLE_TILE;
    HC_CUDA(cudaMemsetAsync(d_overflow, 0, sizeof(int32_t), s));
    auto kern = unit ? (lo ? ent_emit_kernel<true, true> : ent_emit_kernel<true, false>)
                     : (lo ? ent_emit_kernel<false, true> : ent_emit_kernel<false, false>);
    kern<<<(unsigned)tiles, RLE_THREADS, 0, s>>>(sorted, n_valid, cnt_bits, reinterpret_cast<const int64_t*>(work), out, lo, col_bits,
                                                 n_lo, d_overflow);
    HC_LAUNCH_CHECK();
    HC_CUDA(cudaMemcpyAsync(h_overflow, d_overflow, sizeof(int32_t), cudaMemcpyDeviceToHost, s));
    HC_CUDA(cudaStreamSynchronize(s));
    return HC_OK;
}

// lo[n]: (col, row, count) of every off-diagonal cell of up[n], padding key for the diagonal ones; *n_lo (device)
// receives the number of real entries.  Sort lo on bits [cnt_bits + col_bits, cnt_bits + 2*col_bits (+1)) afterwards.
extern "C" int hc_entries_transpose(const unsigned long long* up, int64_t n, int32_t col_bits, int32_t cnt_bits,
                                    unsigned long long* lo, unsigned long long* n_lo, void* stream) {
    HC_REQUIRE(n >= 0 && col_bits > 0 && cnt_bits > 0, "sizes");
    cudaStream_t s = (cudaStream_t)stream;
    HC_CUDA(cudaMemsetAsync(n_lo, 0, sizeof(unsigned long long), s));
    if (n == 0) return HC_OK;
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)hc_num_sms() * 16;
    if (blocks > cap) blocks = cap;
    ent_transpose_kernel<<<(unsigned)blocks, 256, 0, s>>>(up, n, col_bits, cnt_bits, lo, n_lo);
    HC_LAUNCH_CHECK();
    return HC_OK;
}

extern "C" int64_t hc_entries_csr_work_bytes(int64_t nrows) { return (int64_t)sizeof(int64_t) * 2 * (nrows + 1); }

// CSR of the rows [row0, row0+nrows) from the upper list up[n_up] (row <= col, row-major) and the sorted lower list
// lo[*n_lo] (row > col, row-major); lo == NULL: `up` alone already holds every entry of the rows (row-block shards).
// row_ptr: nrows+1; col, cnt: n_up + *n_lo.  work: hc_entries_csr_work_bytes(nrows).
extern "C" int hc_entries_to_csr(const unsigned long long* up, int64_t n_up, const unsigned long long* lo,
                                 const unsigned long long* n_lo, int32_t col_bits, int32_t cnt_bits, int64_t row0,
                                 int64_t nrows, void* work, int64_t* row_ptr, int32_t* col, int32_t* cnt, void* stream) {
    HC_REQUIRE(n_up >= 0 && nrows >= 0 && col_bits > 0 && cnt_bits > 0, "sizes");
    HC_REQUIRE(lo == nullptr || n_lo != nullptr, "n_lo");
    cudaStream_t s = (cudaStream_t)stream;
    int64_t* up_ptr = reinterpret_cast<int64_t*>(work);
    int64_t* lo_ptr = up_ptr + (nrows + 1);
    const int row_shift = col_bits + cnt_bits;
    const long long cap = (long long)hc_num_sms() * 16;
    long long blocks = (std::max<long long>(n_up, nrows + 1) + 255) / 256;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    const unsigned rblocks = (unsigned)std::min<long long>(cap, (nrows + 1 + 255) / 256);
    ent_row_ptr_kernel<<<rblocks, 256, 0, s>>>(up, nullptr, n_up, row_shift, row0, nrows, up_ptr);
    HC_LAUNCH_CHECK();
    if (lo) {
        ent_row_ptr_kernel<<<rblocks, 256, 0, s>>>(lo, n_lo, 0, row_shift, row0, nrows, lo_ptr);
        HC_LAUNCH_CHECK();
    }
    ent_row_ptr_sum_kernel<<<(unsigned)((nrows + 1 + 255) / 256), 256, 0, s>>>(up_ptr, lo ? lo_ptr : nullptr, nrows + 1, row_ptr);
    HC_LAUNCH_CHECK();
    if (n_up > 0) {
        // an upper entry of row r sits after the lower entries of the rows <= r
        ent_scatter_kernel<<<(unsigned)blocks, 256, 0, s>>>(up, nullptr, n_up, col_bits, cnt_bits, row0, lo ? lo_ptr : nullptr, 1, col, cnt);
        HC_LAUNCH_CHECK();
    }
    if (lo) {
        // a lower entry of row r sits after the upper entries of the rows < r
        ent_scatter_kernel<<<(unsigned)blocks, 256, 0, s>>>(lo, n_lo, 0, col_bits, cnt_bits, row0, up_ptr, 0, col, cnt);
        HC_LAUNCH_CHECK();
    }
    return HC_OK;
}
