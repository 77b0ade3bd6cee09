// evs_scan_launch.cuh -- launch wrappers of the GEMV scan kernels (evs_scan.cuh), shared by the translation units that
// instantiate them.  The kernels are split over several .cu files by element type and row width only to keep the build
// short (one file with every instantiation took four minutes of the five-minute clean build).
#pragma once
#include <string.h>

#include "evs_internal.h"
#include "evs_scan.cuh"

namespace evs {

#define EVS_LAUNCH_CHECK()                                  \
    do {                                                    \
        g_kernel_launches.fetch_add(1);                     \
        cudaError_t e__ = cudaGetLastError();               \
        if (e__ != cudaSuccess) return e__;                 \
    } while (0)

// opt a kernel in to more than 48 KB of dynamic shared memory once per (kernel, device): `table` is a per-kernel array
template <typename K>
static cudaError_t ensure_smem_optin(K kern, size_t smem, size_t (&table)[16]) {
    if (smem <= 48 * 1024) return cudaSuccess;
    int dev = 0;
    cudaGetDevice(&dev);
    size_t& have = table[dev & 15];
    if (smem <= have) return cudaSuccess;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e == cudaSuccess) have = smem;
    return e;
}

static ScanParams scan_params(const ScanArgs& a, const ScanPlan* plan) {
    ScanParams p;
    p.xb = a.xb;
    p.xs = a.xs;
    p.n = a.n;
    p.d = a.d;
    p.xq = a.xq;
    p.q0 = a.q0;
    p.lists = reinterpret_cast<u64*>(a.lists);
    p.kp = a.kp;
    p.tile_rows = plan->tile_rows;
    p.stages = plan->stages;
    p.lists_stride_q = plan->grid * a.kp;
    p.ticket = nullptr;
    p.next_chunk = nullptr;
    p.chunk_groups = 1;
    p.qmap = a.qmap;
    p.nactive = a.nactive;
    p.qcap = a.qcap;
    p.cta_clock = nullptr;
    return p;
}

// dynamic shared memory of the pool kernel: the warps' buffers or the finalise area, whichever is larger (the pool kernel
// re-scores up to pool_rescore_slots candidates at a time)
static size_t pool_smem_bytes(const ScanPlan* plan, const FinalizeParams& f) {
    const size_t fs = pool_finalize_smem_bytes(64, f.d, f.x.world * f.k) + 3 * (size_t)(pool_rescore_slots(f) - 64) * 8;
    const size_t bufs = (size_t)(plan->threads / 32) * 128 * 8;
    return fs > bufs ? fs : bufs;
}

template <typename T, int NQ, int NV>
static cudaError_t launch_scan_t(const ScanArgs& a, ScanPlan* plan, cudaStream_t st) {
    ScanParams p = scan_params(a, plan);
    if (plan->variant == 2) {
        if (a.fuse || a.nactive) return cudaErrorInvalidValue;  // the ring variant neither fuses nor re-runs
        auto kern = scan_ring_kernel<T, NQ, NV>;
        cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)plan->smem_bytes);
        kern<<<plan->grid, plan->threads, plan->smem_bytes, st>>>(p);
        EVS_LAUNCH_CHECK();
        return cudaSuccess;
    }
    FinalizeParams f;
    size_t smem = plan->smem_bytes;
    if constexpr (NQ == 1) {
        if (a.fuse != nullptr && a.pool != nullptr && a.kp == 64 && a.nactive == nullptr) {
            f = *a.fuse;
            p.cta_clock = a.cta_clock;
            if (a.next_chunk != nullptr && a.chunk_groups > 0) {
                p.next_chunk = a.next_chunk;
                p.chunk_groups = a.chunk_groups;
            }
            const size_t fs = pool_finalize_smem_bytes(64, f.d, f.x.world * f.k);
            smem = pool_smem_bytes(plan, f);
            if (a.small_fast_cap > 0) {  // small shard: keys by row, threshold from the chunk maxima (no buffers: only the finalise area)
                const int cap = a.small_fast_cap < POOL_SURV ? a.small_fast_cap : POOL_SURV;
                cudaError_t se;
                if (a.q_inline != nullptr) {  // host search: the query rides in the parameter block
                    if (a.d > EVS_SMALL_QUERY_MAX_D) return cudaErrorInvalidValue;
                    auto sk = scan_small_kernel<T, NV, true>;
                    static size_t optin_q[16] = {};
                    const size_t smem_q = small_query_smem_offset(64, f.d, f.x.world * f.k) + (size_t)a.d * 4;
                    se = ensure_smem_optin(sk, smem_q, optin_q);
                    if (se != cudaSuccess) return se;
                    SmallQuery qb;
                    memcpy(qb.v, a.q_inline, (size_t)a.d * 4);
                    se = launch_pdl(sk, dim3((unsigned)plan->grid), dim3((unsigned)plan->threads), smem_q, st, p, f, reinterpret_cast<u64*>(a.pool), cap, qb);
                } else {
                    auto sk = scan_small_kernel<T, NV, false>;
                    static size_t optin_s[16] = {};
                    se = ensure_smem_optin(sk, fs, optin_s);
                    if (se != cudaSuccess) return se;
                    se = launch_pdl(sk, dim3((unsigned)plan->grid), dim3((unsigned)plan->threads), fs, st, p, f, reinterpret_cast<u64*>(a.pool), cap, NoQuery{0});
                }
                g_kernel_launches.fetch_add(1);
                if (se != cudaSuccess) return se;
                return cudaGetLastError();
            }
            auto pk = scan_pool_kernel<T, NV>;
            static size_t optin_p[16] = {};
            cudaError_t oe = ensure_smem_optin(pk, smem, optin_p);
            if (oe != cudaSuccess) return oe;
            cudaError_t le = launch_pdl(pk, dim3((unsigned)plan->grid), dim3((unsigned)plan->threads), smem, st, p, f, reinterpret_cast<u64*>(a.pool));
            g_kernel_launches.fetch_add(1);
            if (le != cudaSuccess) return le;
            return cudaGetLastError();
        }
    }
    if (a.fuse != nullptr && NQ == 1 && a.ticket != nullptr) {
        f = *a.fuse;
        p.ticket = a.ticket;
        p.cta_clock = a.cta_clock;
        if (a.next_chunk != nullptr && a.chunk_groups > 0) {
            p.next_chunk = a.next_chunk;
            p.chunk_groups = a.chunk_groups;
        }
        const size_t fs = finalize_smem_bytes_host(f.L, f.kp, f.d);
        if (fs > smem) smem = fs;
    } else if (a.fuse != nullptr) {
        return cudaErrorInvalidValue;
    }
    auto kern = scan_direct_kernel<T, NQ, NV>;
    static size_t optin[16] = {};  // per instantiation
    cudaError_t oe = ensure_smem_optin(kern, smem, optin);
    if (oe != cudaSuccess) return oe;
    cudaError_t le = launch_pdl(kern, dim3((unsigned)plan->grid), dim3((unsigned)plan->threads), smem, st, p, f);
    g_kernel_launches.fetch_add(1);
    if (le != cudaSuccess) return le;
    return cudaGetLastError();
}

template <typename T, int NV>
static cudaError_t launch_scan_nq(const ScanArgs& a, ScanPlan* plan, cudaStream_t st) {
    switch (a.nq_pass) {
        case 1: return launch_scan_t<T, 1, NV>(a, plan, st);
        case 2: return launch_scan_t<T, 2, NV>(a, plan, st);
        case 3: return launch_scan_t<T, 3, NV>(a, plan, st);
        case 4: return launch_scan_t<T, 4, NV>(a, plan, st);
        default: return cudaErrorInvalidValue;
    }
}

template <typename T>
static cudaError_t launch_scan_generic(const ScanArgs& a, ScanPlan* plan, cudaStream_t st) {
    ScanParams p = scan_params(a, plan);
    if (a.fuse || a.nactive) return cudaErrorInvalidValue;
    for (int qi = 0; qi < a.nq_pass; qi++) {
        p.q0 = a.q0 + qi;
        scan_generic_kernel<T><<<plan->grid, plan->threads, plan->smem_bytes, st>>>(p);
        EVS_LAUNCH_CHECK();
    }
    return cudaSuccess;
}


// one entry point per translation unit (evs_scan_*.cu); `plan->nv` selects the instantiation
cudaError_t launch_scan_f32_narrow(const ScanArgs& a, ScanPlan* plan, cudaStream_t st);  // nv = 1, 2, 3
cudaError_t launch_scan_f32_512(const ScanArgs& a, ScanPlan* plan, cudaStream_t st);     // nv = 4 (d = 512)
cudaError_t launch_scan_f32_wide(const ScanArgs& a, ScanPlan* plan, cudaStream_t st);    // nv = 6, 8
cudaError_t launch_scan_bf16_narrow(const ScanArgs& a, ScanPlan* plan, cudaStream_t st); // nv = 1, 2
cudaError_t launch_scan_bf16_wide(const ScanArgs& a, ScanPlan* plan, cudaStream_t st);   // nv = 3, 4
cudaError_t launch_scan_i8(const ScanArgs& a, ScanPlan* plan, cudaStream_t st);          // nv = 1 .. 4, pool kernel only
cudaError_t launch_scan_generic_any(const ScanArgs& a, ScanPlan* plan, cudaStream_t st); // any d

}  // namespace evs
