// Hand-written LSD radix sort (64-bit keys, keys only) in the "onesweep" style: one upfront
// histogram pass over all digits, then ONE kernel per 8-bit digit that ranks a tile in shared
// memory and resolves its global offsets with a decoupled look-back over earlier tiles -- every
// key is read once and written once per pass.  This is the sort of north_star kernel (a)
// ("radix sort plus reduce-by-key"); the keys are row*nbins+col bin pairs built by hc_csr.cu.
//
// Roofline: HBM-bound, 8*P (histogram) + passes*16*P bytes for P keys.
#include "hc_common.cuh"

namespace {

constexpr int RADIX_BITS = 8;
constexpr int RADIX = 1 << RADIX_BITS;
constexpr int MAX_PASSES = 8;
constexpr int SORT_THREADS = 512;
constexpr int SORT_ITEMS = 16;                        // keys per thread
constexpr int SORT_TILE = SORT_THREADS * SORT_ITEMS;
constexpr int SORT_MIN_BLOCKS = 2;                    // 64 registers/thread -> 2 CTAs (32 warps) per SM
constexpr int SORT_LOOKBACK = 8;                      // status words fetched per look-back step

__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" :: "l"(p), "l"(v) : "memory");
}

constexpr unsigned long long FLAG_AGG = 1ull << 62;
constexpr unsigned long long FLAG_INC = 2ull << 62;
constexpr unsigned long long FLAG_MASK = 3ull << 62;

// ---- upfront histogram of every digit --------------------------------------------------
__global__ void __launch_bounds__(512)
radix_histogram_kernel(const unsigned long long* __restrict__ keys, long long n, int begin_bit, int passes,
                       unsigned long long* __restrict__ ghist /*[passes][256]*/) {
    __shared__ unsigned int sh[MAX_PASSES][RADIX];
    for (int i = threadIdx.x; i < MAX_PASSES * RADIX; i += blockDim.x) (&sh[0][0])[i] = 0;
    __syncthreads();
    const long long stride = (long long)gridDim.x * blockDim.x;
    // bounded trip count per block keeps the 32-bit shared counters from overflowing
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const unsigned long long k = keys[i] >> begin_bit;
#pragma unroll
        for (int p = 0; p < MAX_PASSES; ++p)
            if (p < passes) atomicAdd(&sh[p][(k >> (RADIX_BITS * p)) & (RADIX - 1)], 1u);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < passes * RADIX; i += blockDim.x) {
        const unsigned int v = (&sh[0][0])[i];
        if (v) atomicAdd(&ghist[i], (unsigned long long)v);
    }
}

// exclusive scan of each pass's 256-bin histogram (one block per pass, 256 threads)
__global__ void __launch_bounds__(RADIX) radix_scan_kernel(unsigned long long* __restrict__ ghist) {
    __shared__ unsigned long long s[RADIX];
    unsigned long long* h = ghist + (size_t)blockIdx.x * RADIX;
    s[threadIdx.x] = h[threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long run = 0;
        for (int d = 0; d < RADIX; ++d) { const unsigned long long c = s[d]; s[d] = run; run += c; }
    }
    __syncthreads();
    h[threadIdx.x] = s[threadIdx.x];
}

// ---- one digit pass -------------------------------------------------------------------
// 512 threads x 16 keys per tile.  The tile size sets the length of the digit runs a tile writes (tile / 256 keys on a
// uniform digit): 128 B runs at 4096 keys, 256 B at 8192 -- the low-digit passes are bound by those scattered writes
// (measured 2.1 TB/s at 4096 against 3.3 TB/s for the top digit, whose 64 occupied bins give 512 B runs).  12 keys per
// thread at five CTAs of 256 threads per SM was measured too: 19.9 against 17.3 ms per 500 M keys.
struct SortSmem {
    unsigned long long keys[SORT_TILE];
    unsigned int warp_hist[SORT_THREADS / 32][RADIX];
    unsigned int tile_off[RADIX];       // exclusive scan of the tile's digit totals
    unsigned long long gbase[RADIX];    // global position of the tile's first key of each digit, minus tile_off
    unsigned int scan_tmp[RADIX / 32];
    unsigned int tile_id;
};

// Lanes of the warp that hold the same 8-bit digit.  MATCH.ANY does it in one instruction, but it runs on the address
// divergence unit at about one warp instruction per 60 cycles and SM: with 16 of them per thread the pass sat at 81 % ADU
// utilisation and 2.1 TB/s (profiles/r2r_ncu_onesweep_v2.json).  Eight ballots (ALU pipe) narrow the mask bit by bit.
__device__ __forceinline__ unsigned match_digit(unsigned d, bool ok) {
    unsigned m = __ballot_sync(0xffffffffu, ok);
#pragma unroll
    for (int b = 0; b < RADIX_BITS; ++b) {
        const bool bit = (d >> b) & 1u;
        const unsigned bal = __ballot_sync(0xffffffffu, bit);
        m &= bit ? bal : ~bal;
    }
    return m;
}

__global__ void __launch_bounds__(SORT_THREADS, SORT_MIN_BLOCKS)
radix_onesweep_kernel(const unsigned long long* __restrict__ in, unsigned long long* __restrict__ out, long long n,
                      int shift, const unsigned long long* __restrict__ digit_base /*[256]*/,
                      unsigned long long* status /*[num_tiles][256]*/, unsigned int* tile_counter) {
    constexpr int WARPS = SORT_THREADS / 32;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    SortSmem& sm = *reinterpret_cast<SortSmem*>(smem_raw);
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    if (tid == 0) sm.tile_id = atomicAdd(tile_counter, 1u);   // tiles are claimed in launch order
    for (int i = tid; i < WARPS * RADIX; i += SORT_THREADS) (&sm.warp_hist[0][0])[i] = 0;
    __syncthreads();
    const long long tile = sm.tile_id;
    const long long base = tile * SORT_TILE;
    const int valid = (int)min((long long)SORT_TILE, n - base);

    // warp-striped load keeps memory order == (warp, item, lane) order -> stable ranking
    unsigned long long key[SORT_ITEMS];
    unsigned int rank2[SORT_ITEMS / 2];    // ranks inside the warp's digit run (< 65536): two per register
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int j = w * (32 * SORT_ITEMS) + i * 32 + lane;
        key[i] = j < valid ? in[base + j] : ~0ull;
    }
    // Ranking: lanes holding the same digit are counted by their first lane in the warp's counter row.  (Two independent
    // half-chunk chains per warp, each with its own counter row, were measured slower: 18.7 vs 17.1 ms for 500 M keys.)
    const unsigned lt = (1u << lane) - 1u;
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int j = w * (32 * SORT_ITEMS) + i * 32 + lane;
        const bool ok = j < valid;
        const unsigned d = (unsigned)((key[i] >> shift) & (RADIX - 1));
        const unsigned m = match_digit(d, ok);          // padding lanes match nobody and count nowhere
        const int leader = __ffs(m) - 1;
        unsigned prev = 0;
        if (ok && lane == leader) {
            prev = sm.warp_hist[w][d];
            sm.warp_hist[w][d] = prev + __popc(m);
        }
        prev = __shfl_sync(0xffffffffu, prev, leader & 31);
        const unsigned rk = prev + __popc(m & lt);
        rank2[i >> 1] = (i & 1) ? (rank2[i >> 1] | (rk << 16)) : rk;
        __syncwarp();
    }
    __syncthreads();

    // per digit (threads 0..255): exclusive scan over warps, tile total -- published at once so that later tiles can add it
    unsigned total = 0;
    unsigned long long* my = status + tile * RADIX + tid;
    if (tid < RADIX) {
        unsigned run = 0;
#pragma unroll
        for (int ww = 0; ww < WARPS; ++ww) {
            const unsigned c = sm.warp_hist[ww][tid];
            sm.warp_hist[ww][tid] = run;
            run += c;
        }
        total = run;
        st_relaxed_u64(my, (tile == 0 ? FLAG_INC : FLAG_AGG) | total);
        // block exclusive scan of the digit totals -> position of each digit run inside the tile
        unsigned incl = total;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned y = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += y;
        }
        if (lane == 31) sm.scan_tmp[w] = incl;
        total = incl - total;      // exclusive inside the warp, for the moment
    }
    __syncthreads();
    if (tid < RADIX) {
        unsigned woff = 0;
        for (int ww = 0; ww < w; ++ww) woff += sm.scan_tmp[ww];
        sm.tile_off[tid] = woff + total;
    }
    __syncthreads();

    // reorder inside shared memory so the global writes are contiguous per digit run (the keys leave the registers
    // before the look-back needs them for its window)
#pragma unroll
    for (int i = 0; i < SORT_ITEMS; ++i) {
        const int j = w * (32 * SORT_ITEMS) + i * 32 + lane;
        if (j < valid) {
            const unsigned d = (unsigned)((key[i] >> shift) & (RADIX - 1));
            sm.keys[sm.tile_off[d] + sm.warp_hist[w][d] + ((rank2[i >> 1] >> (16 * (i & 1))) & 0xffffu)] = key[i];
        }
    }

    // decoupled look-back for digit `tid`: SORT_LOOKBACK status words are fetched at once and consumed in order (a walk of
    // one L2 round trip per predecessor is ~20 hops long at this tile rate)
    if (tid < RADIX) {
        unsigned long long excl = 0;
        if (tile != 0) {
            // the tile total again: next digit's offset minus this one's (the last digit: up to `valid`)
            const unsigned mine = (tid == RADIX - 1 ? (unsigned)valid : sm.tile_off[tid + 1]) - sm.tile_off[tid];
            long long t = tile - 1;
            bool found = false;
            while (!found) {
                unsigned long long v[SORT_LOOKBACK];
#pragma unroll
                for (int u = 0; u < SORT_LOOKBACK; ++u)
                    v[u] = (t - u >= 0) ? ld_relaxed_u64(status + (t - u) * RADIX + tid) : FLAG_INC;   // before tile 0: nothing
#pragma unroll
                for (int u = 0; u < SORT_LOOKBACK; ++u) {
                    if (!found) {
                        unsigned long long x = v[u];
                        while ((x & FLAG_MASK) == 0) x = ld_relaxed_u64(status + (t - u) * RADIX + tid);   // not published yet
                        excl += x & ~FLAG_MASK;
                        found = (x & FLAG_MASK) == FLAG_INC;
                    }
                }
                t -= SORT_LOOKBACK;
            }
            st_relaxed_u64(my, FLAG_INC | (excl + mine));
        }
        sm.gbase[tid] = digit_base[tid] + excl - sm.tile_off[tid];
    }
    __syncthreads();
    for (int j = tid; j < valid; j += SORT_THREADS) {
        const unsigned long long k = sm.keys[j];
        const unsigned d = (unsigned)((k >> shift) & (RADIX - 1));
        out[sm.gbase[d] + (unsigned)j] = k;
    }
}

}  // namespace

// Workspace layout (bytes): [passes*256 u64 histogram][16 B counters][num_tiles*256 u64 status]; the status array has
// room for one row per 4096 keys, twice the tiles of SORT_TILE keys
extern "C" int64_t hc_sort_work_bytes(int64_t n) {
    const int64_t tiles = (n + 4095) / 4096;
    return (int64_t)sizeof(unsigned long long) * (MAX_PASSES * RADIX + (tiles > 0 ? tiles : 1) * RADIX) + 64;
}

// Sorts keys[0..n) ascending on bits [begin_bit, end_bit).  `keys` and `tmp` are n-element
// device buffers used as a ping-pong pair; *h_result_in_tmp tells the caller where the sorted
// keys ended up (1 = tmp).  Stream-ordered; no host synchronisation.
extern "C" int hc_sort_keys_u64(unsigned long long* keys, unsigned long long* tmp, int64_t n, int32_t begin_bit,
                                int32_t end_bit, void* work, int32_t* h_result_in_tmp, void* stream) {
    HC_REQUIRE(n >= 0 && begin_bit >= 0 && end_bit <= 64 && begin_bit <= end_bit, "n>=0, 0<=begin<=end<=64");
    if (h_result_in_tmp) *h_result_in_tmp = 0;
    const int passes = (end_bit - begin_bit + RADIX_BITS - 1) / RADIX_BITS;
    if (n <= 1 || passes == 0) return HC_OK;
    HC_REQUIRE(passes <= MAX_PASSES, "too many digit passes");
    cudaStream_t s = (cudaStream_t)stream;
    unsigned long long* ghist = reinterpret_cast<unsigned long long*>(work);
    unsigned int* counter = reinterpret_cast<unsigned int*>(ghist + MAX_PASSES * RADIX);
    unsigned long long* status = ghist + MAX_PASSES * RADIX + 2;

    HC_CUDA(cudaMemsetAsync(ghist, 0, sizeof(unsigned long long) * MAX_PASSES * RADIX, s));
    {
        long long blocks = (n + 512 * 64 - 1) / (512 * 64);     // >= 64 keys per thread
        const long long cap = (long long)hc_num_sms() * 4;
        if (blocks > cap) blocks = cap;
        // 32-bit shared counters: a block sees at most n/blocks keys; split further if needed
        while (n / blocks >= (1ll << 31)) blocks *= 2;
        radix_histogram_kernel<<<(unsigned)blocks, 512, 0, s>>>(keys, n, begin_bit, passes, ghist);
        HC_LAUNCH_CHECK();
    }
    radix_scan_kernel<<<passes, RADIX, 0, s>>>(ghist);
    HC_LAUNCH_CHECK();

    const size_t smem = sizeof(SortSmem);
    const long long tiles = (n + SORT_TILE - 1) / SORT_TILE;
    HC_CUDA(cudaFuncSetAttribute(radix_onesweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    unsigned long long* src = keys;
    unsigned long long* dst = tmp;
    for (int p = 0; p < passes; ++p) {
        HC_CUDA(cudaMemsetAsync(counter, 0, 16 + sizeof(unsigned long long) * tiles * RADIX, s));
        radix_onesweep_kernel<<<(unsigned)tiles, SORT_THREADS, smem, s>>>(
            src, dst, n, begin_bit + RADIX_BITS * p, ghist + p * RADIX, status, counter);
        HC_LAUNCH_CHECK();
        unsigned long long* t = src; src = dst; dst = t;
    }
    if (h_result_in_tmp) *h_result_in_tmp = (src == tmp) ? 1 : 0;
    return HC_OK;
}
