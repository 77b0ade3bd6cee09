// evs_scan_i8.cu -- the pool kernel (evs_scan.cuh: scan_pool_kernel) over the int8 scan copy of the rows, NV = d / 256
// = 1 .. 4 (d = 256 .. 1024).  Only the fused single-query search scans this copy.
#include "evs_scan_launch.cuh"

namespace evs {

template <int NV>
static cudaError_t launch_pool_i8(const ScanArgs& a, ScanPlan* plan, cudaStream_t st) {
    if (a.fuse == nullptr || a.pool == nullptr || a.xs == nullptr || a.kp != 64 || a.nq_pass != 1 || a.nactive != nullptr ||
        a.small_fast_cap > 0 || plan->variant != 1)
        return cudaErrorInvalidValue;
    ScanParams p = scan_params(a, plan);
    const FinalizeParams f = *a.fuse;
    p.cta_clock = a.cta_clock;
    if (a.next_chunk != nullptr && a.chunk_groups > 0) {
        p.next_chunk = a.next_chunk;
        p.chunk_groups = a.chunk_groups;
    }
    const size_t smem = pool_smem_bytes(plan, f);
    auto pk = scan_pool_kernel<int8_t, NV>;
    static size_t optin[16] = {};
    cudaError_t oe = ensure_smem_optin(pk, smem, optin);
    if (oe != cudaSuccess) return oe;
    cudaError_t le = launch_pdl(pk, dim3((unsigned)plan->grid), dim3((unsigned)plan->threads), smem, st, p, f, reinterpret_cast<u64*>(a.pool));
    g_kernel_launches.fetch_add(1);
    if (le != cudaSuccess) return le;
    return cudaGetLastError();
}

cudaError_t launch_scan_i8(const ScanArgs& a, ScanPlan* plan, cudaStream_t st) {
    switch (plan->nv) {
        case 1: return launch_pool_i8<1>(a, plan, st);
        case 2: return launch_pool_i8<2>(a, plan, st);
        case 3: return launch_pool_i8<3>(a, plan, st);
        case 4: return launch_pool_i8<4>(a, plan, st);
        default: return cudaErrorInvalidValue;
    }
}

}  // namespace evs
