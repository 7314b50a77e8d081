// Shared helpers for libhichap_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/hichap_b200.h"

void hc_set_error(const char* fmt, ...);
void hc_count_launch(int n = 1);
// synchronous small device->host read through a pinned mailbox (no copy engine; see hc_abi.cu)
cudaError_t hc_read_small(void* dst, const void* src, size_t bytes, cudaStream_t s);
cudaMemPool_t hc_big_pool(void);      // stream-ordered pool reserved for multi-GB scratch blocks (hc_abi.cu)
int hc_exclusive_scan_i64(int64_t* v, long long n, cudaStream_t s);   // single-CTA, in place, total to v[n] (hc_csr.cu)

#define HC_CUDA(call)                                                                       \
    do {                                                                                    \
        cudaError_t e_ = (call);                                                            \
        if (e_ != cudaSuccess) {                                                            \
            hc_set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #call,                 \
                         cudaGetErrorString(e_));                                           \
            return HC_ERR_CUDA;                                                             \
        }                                                                                   \
    } while (0)

#define HC_LAUNCH_CHECK()                                                                   \
    do {                                                                                    \
        hc_count_launch();                                                                  \
        HC_CUDA(cudaGetLastError());                                                        \
    } while (0)

#define HC_REQUIRE(cond, msg)                                                               \
    do {                                                                                    \
        if (!(cond)) {                                                                      \
            hc_set_error("%s:%d: invalid argument: %s", __FILE__, __LINE__, msg);           \
            return HC_ERR_ARG;                                                              \
        }                                                                                   \
    } while (0)

static inline int hc_num_sms() {
    static int sms = 0;
    if (sms == 0) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess ||
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sms <= 0)
            sms = 148;  // B200
    }
    return sms;
}

// Unsigned 32-bit division by a run-time invariant (bin = position / resolution) as a multiply-high
// and two shifts (Granlund & Montgomery, "Division by invariant integers using multiplication").
struct FastDiv { uint32_t m; int s1, s2; };
static inline FastDiv make_fast_div(uint32_t d) {
    int l = 0;
    while (l < 32 && (1ull << l) < d) ++l;                       // ceil(log2 d)
    FastDiv f;
    f.m = (uint32_t)(((1ull << 32) * ((1ull << l) - d)) / d + 1);
    f.s1 = l < 1 ? l : 1;
    f.s2 = l > 1 ? l - 1 : 0;
    return f;
}

// ---- device helpers ---------------------------------------------------------------------
__device__ __forceinline__ uint32_t fast_div(uint32_t n, FastDiv f) {
    const uint32_t t = __umulhi(f.m, n);
    return (t + ((n - t) >> f.s1)) >> f.s2;
}

// int32 -> double without the conversion pipe (I2F.F64 issues at a quarter of the FP64 FMA rate):
// place the biased integer in the mantissa of 2^52 and subtract 2^52 + 2^31 (exact for every int32)
__device__ __forceinline__ double i32_to_f64(int x) {
    return __hiloint2double(0x43300000, x ^ (int)0x80000000) - 4503601774854144.0;
}

__device__ __forceinline__ int4 ld_stream_v4(const int32_t* p) {
    // 128-bit streaming load: read-only path, do not allocate in L1 (data is touched once)
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// L2 eviction policies: streamed inputs should not displace a working set that other warps keep
// updating in L2 (the band accumulator of the binning kernel)
__device__ __forceinline__ uint64_t l2_policy_evict_first() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ int4 ld_stream_v4_hint(const int32_t* p, uint64_t policy) {
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0,%1,%2,%3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(policy));
    return r;
}
__device__ __forceinline__ void red_add_s32_hint(int32_t* p, int v, uint64_t policy) {
    asm volatile("red.global.add.L2::cache_hint.s32 [%0], %1, %2;" :: "l"(p), "r"(v), "l"(policy) : "memory");
}

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_sum_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum of doubles in a fixed order (deterministic); red must hold >= 32 doubles.
// Every thread receives the result.
__device__ __forceinline__ double block_sum(double v, double* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum(v);
    __syncthreads();  // protect red from a previous use
    if (lane == 0) red[wid] = v;
    __syncthreads();
    double t = 0.0;
    for (int w = 0; w < nw; ++w) t += red[w];
    return t;
}
__device__ __forceinline__ long long block_sum_ll(long long v, long long* red) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    v = warp_sum_ll(v);
    __syncthreads();
    if (lane == 0) red[wid] = v;
    __syncthreads();
    long long t = 0;
    for (int w = 0; w < nw; ++w) t += red[w];
    return t;
}

// Order-preserving map double -> uint64 (total order; NaNs sort high/low by sign bit).
__device__ __forceinline__ unsigned long long f64_key(double x) {
    unsigned long long b = (unsigned long long)__double_as_longlong(x);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(unsigned long long k) {
    unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}
