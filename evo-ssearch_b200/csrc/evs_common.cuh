// evs_common.cuh -- shared device helpers for libevs (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "libevs is written for sm_100a (B200) only"
#endif

namespace evs {

typedef unsigned long long u64;

// ---------------------------------------------------------------------------------------------
// Candidate keys.  A candidate is one (scan score, shard-local row) pair packed into 64 bits so
// that a plain unsigned compare realises the canonical order "higher score first, then lower
// row id": high word = order-preserving map of the fp32 score, low word = ~row.
// key 0 is "empty".  NaN scores map to 0 and never enter (faiss: heap_top < NaN is false).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t score_to_ordered(float s) {
    uint32_t u = __float_as_uint(s);
    uint32_t o = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
    return (s != s) ? 0u : o;
}
__device__ __forceinline__ float ordered_to_score(uint32_t o) {
    uint32_t u = (o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o;
    return __uint_as_float(u);
}
__device__ __forceinline__ u64 make_key(float s, uint32_t row) {
    uint32_t o = score_to_ordered(s);
    return o == 0u ? 0ull : (((u64)o << 32) | (u64)(0xFFFFFFFFu - row));
}
__device__ __forceinline__ uint32_t key_row(u64 key) { return 0xFFFFFFFFu - (uint32_t)(key & 0xFFFFFFFFull); }
__device__ __forceinline__ float key_score(u64 key) { return ordered_to_score((uint32_t)(key >> 32)); }

// order-preserving map of an fp64 score to u64 (for the final canonical ranking)
__device__ __forceinline__ u64 f64_to_ordered(double s) {
    u64 u = (u64)__double_as_longlong(s);
    return (u & 0x8000000000000000ull) ? ~u : (u | 0x8000000000000000ull);
}

__device__ __forceinline__ u64 umax64(u64 a, u64 b) { return a > b ? a : b; }

// ---------------------------------------------------------------------------------------------
// Warp-synchronous bitonic networks over a u64 array in shared memory, DESCENDING order.
// n is a power of two >= 64.  All 32 lanes of the calling warp must take part.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void cmpx_desc(u64* a, int i, int j, bool desc) {
    u64 x = a[i], y = a[j];
    bool swap = desc ? (x < y) : (x > y);
    if (swap) {
        a[i] = y;
        a[j] = x;
    }
}

// index of the lower element of compare-exchange pair t at distance `stride` (a power of two): insert a 0 bit at log2(stride)
__device__ __forceinline__ int bitonic_low(int t, int stride) { return ((t & ~(stride - 1)) << 1) | (t & (stride - 1)); }

// full sort: after the call a[0] >= a[1] >= ... >= a[n-1]
__device__ __forceinline__ void warp_bitonic_sort_desc(u64* a, int n, int lane) {
    for (int size = 2; size <= n; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncwarp();
            for (int t = lane; t < (n >> 1); t += 32) {
                const int i = bitonic_low(t, stride);
                cmpx_desc(a, i, i + stride, (i & size) == 0);
            }
        }
    }
    __syncwarp();
}

// a[0..n) is bitonic on entry -> sorted descending on exit
__device__ __forceinline__ void warp_bitonic_merge_desc(u64* a, int n, int lane) {
    for (int stride = n >> 1; stride > 0; stride >>= 1) {
        __syncwarp();
        for (int t = lane; t < (n >> 1); t += 32) {
            const int i = bitonic_low(t, stride);
            cmpx_desc(a, i, i + stride, true);
        }
    }
    __syncwarp();
}

// A[0..kp) and B[0..kp) sorted descending (B may live in global memory) -> A = top kp of the union,
// sorted descending.  max(A[i], B[kp-1-i]) is a bitonic sequence holding exactly the kp largest.
__device__ __forceinline__ void warp_merge_top(u64* A, const u64* B, int kp, int lane) {
    __syncwarp();
    for (int i = lane; i < kp; i += 32) A[i] = umax64(A[i], B[kp - 1 - i]);
    warp_bitonic_merge_desc(A, kp, lane);
}

// ---------------------------------------------------------------------------------------------
// CANON-32: the fixed-order fp64 inner product every final score is computed with (DESIGN.md,
// oracle/flat_ip_oracle.c).  One warp per (row, query) pair; every lane returns the same bits.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double canon32_dot(const float* __restrict__ x, const float* __restrict__ q, int d,
                                              int lane) {
    double acc = 0.0;
    for (int i = lane; i < d; i += 32) acc = fma((double)x[i], (double)q[i], acc);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc = acc + __shfl_xor_sync(0xffffffffu, acc, off);
    return acc;
}

// ---------------------------------------------------------------------------------------------
// mbarrier + bulk async copy (TMA engine, 1-D form: SASS UBLKCP) wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "EVS_WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra EVS_DONE_%=;\n\t"
        "bra EVS_WAIT_%=;\n\t"
        "EVS_DONE_%=:\n\t"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// global -> shared bulk copy, completion counted in bytes on `bar`.  dst/src 16-byte aligned,
// bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}

// 128-bit streaming global load that does not allocate in L1 (database rows are read once)
__device__ __forceinline__ float4 ldg_stream_f4(const float4* p) {
    float4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
                 : "l"(p));
    return r;
}
__device__ __forceinline__ uint2 ldg_stream_u2(const uint2* p) {
    uint2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
    return r;
}

}  // namespace evs
