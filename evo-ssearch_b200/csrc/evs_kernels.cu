// evs_kernels.cu -- kernel definitions and launch wrappers of libevs (sm_100a).
//
//   scan launchers       score + fused top-k' selection               (evs_scan.cuh)
//   finalize_kernel      merge the per-CTA lists of one query, re-score the k' candidates in the
//                        canonical fp64 order, rank, emit (D,I) or a shard partial
//   merge_partials_kernel  G-way merge of shard partials after the NCCL all-gather, every k
//   merge_exchange_kernel  the same merge after the peer-store exchange, behind its wait protocol, every k (both rank
//                        with merge_rank, evs_finalize.cuh)
//   l2_normalize_kernel  oldapp.py:35/43/51, 128-bit coalesced, in place
//   f32_to_bf16_kernel   the one-time database layout kernel
//   synth_fill_kernel    counter-based synthetic embeddings (bit-identical to oracle/orc_synth_fill)
#include <float.h>

#include <atomic>

#include "evs_internal.h"
#include "evs_scan.cuh"
#include "evs_scan_launch.cuh"

namespace evs {

std::atomic<long long> g_kernel_launches{0};

// =============================================================================================
// finalize: one CTA per query around finalize_query (evs_finalize.cuh).  grid = nq, block = 1024 or 256.
// Launched with programmatic stream serialisation behind the scan: the prologue (the query widened to fp64 -- it does
// not come from the scan) overlaps the scan's tail; everything below the wait sees the scan's lists.
// Guard second phase (pred_slot != null): only the queries the first finalise queued are finalised again, from the
// lists of the exact re-run; every other CTA returns at once.
// =============================================================================================
__global__ void __launch_bounds__(1024) finalize_kernel(FinalizeParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const long long qi = blockIdx.x;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next kernel of the chain may get resident
    const u64* lists;
    if (p.pred_slot != nullptr) {
        asm volatile("griddepcontrol.wait;" ::: "memory");
        const int slot = p.pred_slot[qi];
        if (slot < 0 || slot >= p.guard_cap) return;  // certified by the first phase (the usual case): CTA-uniform
        lists = p.lists + (size_t)slot * p.L * p.kp;
        if (threadIdx.x == 0 && p.reruns) atomicAdd(p.reruns, 1ull);
        finalize_prologue(p, qi, smem_raw);
    } else {
        finalize_prologue(p, qi, smem_raw);
        asm volatile("griddepcontrol.wait;" ::: "memory");
        if (threadIdx.x == 0 && p.guard_slot) p.guard_slot[qi] = -1;  // overwritten below (barriers in between) if uncertified
        lists = p.lists + (size_t)qi * p.L * p.kp;
    }
    finalize_query(p, qi, lists, smem_raw);
}

// =============================================================================================
// publish: copy this shard's partial (scores[nq*k], ids[nq*k]) into its slot on EVERY rank over NVLink
// (peer stores, one flagged 32-byte entry per result: evs_internal.h).  Used when the partial was produced by a
// path that cannot write the slots itself (scans whose result the device guard may still overwrite, empty
// shard).  grid = any, block = 256.
// =============================================================================================
__global__ void __launch_bounds__(256) publish_partials_kernel(Exchange x, long long count, const double* __restrict__ scores,
                                                              const long long* __restrict__ ids) {
    asm volatile("griddepcontrol.wait;" ::: "memory");  // the partial is the preceding kernels' output
    const uint32_t flag = exchange_flag(x.seq);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x)
        exchange_store_entry(x, (size_t)e, scores[e], ids[e], flag);
}

// =============================================================================================
// poison: this rank could not run search `x.seq` (an allocation or a launch failed after its peers may already be waiting):
// every entry of its slot on every rank gets the sequence flag with bit 31 set, so that the peers' merges report the failure
// instead of waiting ~10 s or returning a result that silently misses this shard.  grid = any, block = 256.
// =============================================================================================
__global__ void publish_poison_kernel(Exchange x, long long count) {
    const uint32_t flag = exchange_flag(x.seq) | kExchangePoison;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < count; e += (long long)gridDim.x * blockDim.x)
        exchange_store_entry(x, (size_t)e, 0.0, -1, flag);
}

// =============================================================================================
// merge after the peer-store exchange: poll the entries of this search in the LOCAL gather buffer until every
// shard's have arrived, then rank the world*k partials of each query (exchange_merge).  grid = nq, block = 256 for
// k <= EVS_MAX_K (entries staged in shared memory), 1024 above (ranked in the gather buffer).
// Every rank runs this kernel on its own GPU; the entries are written by the other GPUs' finalise / publish kernels.
// A rank that never arrives (~10 s watchdog) or that reported failure (poisoned flag) makes the whole result
// padding (-FLT_MAX, -1) and sets *x.status (host-mapped): stale slots are never merged.
// =============================================================================================
__global__ void __launch_bounds__(1024) merge_exchange_kernel(Exchange x, int k, float* __restrict__ D, long long* __restrict__ I) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int s_nvalid, s_fail;
    if (threadIdx.x == 0) {
        s_nvalid = 0;
        s_fail = 0;
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");  // launched programmatically behind this rank's finalise / publish kernel
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    __syncthreads();
    if (k <= EVS_MAX_K) exchange_merge<true>(x, blockIdx.x, k, D, I, smem_raw, &s_fail, &s_nvalid);
    else exchange_merge<false>(x, blockIdx.x, k, D, I, smem_raw, &s_fail, &s_nvalid);
}

// =============================================================================================
// merge of shard partials: scores/ids laid out [part][nq][k].  k <= EVS_MAX_K: grid = nq, the query's nparts*k entries
// staged in shared memory and merged by merge_query.  Larger k (nparts*k*24 bytes outgrow shared memory): grid = (entry
// blocks, query stride), one thread per entry ranked straight from global memory by merge_rank; with the query spread over
// CTAs nothing counts the real entries, so the padding entries of part 0 rank themselves behind all of them and fill the
// slots [nvalid, k) (a later part's padding ranks behind part 0's k entries).  block = 256.
// =============================================================================================
__global__ void __launch_bounds__(256) merge_partials_kernel(int nparts, long long nq, int k,
                                                            const double* __restrict__ scores,
                                                            const long long* __restrict__ ids, long long part_stride,
                                                            float* __restrict__ D, long long* __restrict__ I) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int m = nparts * k;
    if (k <= EVS_MAX_K) {
        __shared__ int s_nvalid;
        const long long qi = blockIdx.x;
        const StagedParts staged(smem_raw, nparts, k);
        if (threadIdx.x == 0) s_nvalid = 0;
        for (int e = threadIdx.x; e < m; e += blockDim.x) {
            const size_t src = (size_t)(e / k) * part_stride + (size_t)qi * k + e % k;
            staged.put(e, scores[src], ids[src]);
        }
        __syncthreads();
        merge_query(staged, nparts, k, D + (size_t)qi * k, I + (size_t)qi * k, &s_nvalid);
        return;
    }
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m) return;
    const int part = e / k, r = e - part * k;
    // not unrolled: the unrolled loop's trip count costs a 64-bit division call and a spill
#pragma unroll 1
    for (long long qi = blockIdx.y; qi < nq; qi += gridDim.y) {
        const auto in_place = [&](int pp, int j) {
            const size_t o = (size_t)pp * part_stride + (size_t)qi * k + j;
            const double s = scores[o];
            return PartEntry{s, score_rank_key(s), ids[o]};
        };
        const PartEntry t = in_place(part, r);
        const bool pad = t.id < 0;
        if (pad && part > 0) continue;
        const int rank = merge_rank(in_place, nparts, k, part, r, pad ? 0ull : t.key, pad ? LLONG_MAX : t.id);
        if (rank < k) {
            D[(size_t)qi * k + rank] = pad ? -FLT_MAX : (float)t.score;
            I[(size_t)qi * k + rank] = pad ? -1 : t.id;
        }
    }
}

// =============================================================================================
// L2 normalise, in place.  One warp per row; the row is staged in shared memory as fp32 with
// 128-bit coalesced global loads, the sum of squares is taken in the CANON-32 order in fp64,
// norm = T(float(sqrt(sum))), out = T(float(x) / float(norm)); written back with 128-bit stores.
// =============================================================================================
template <typename T> __device__ __forceinline__ float to_f32(T v);
template <> __device__ __forceinline__ float to_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_f32<__half>(__half v) { return __half2float(v); }
template <> __device__ __forceinline__ float to_f32<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __half from_f32<__half>(float v) { return __float2half_rn(v); }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

template <typename T, bool VEC16>
__global__ void __launch_bounds__(256) l2_normalize_kernel(T* __restrict__ x, long long n, int d) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    float* stage = reinterpret_cast<float*>(smem_raw) + (size_t)warp * d;
    constexpr int EPV = 16 / sizeof(T);  // elements per 16-byte vector
    for (long long row = (long long)blockIdx.x * nwarps + warp; row < n; row += (long long)gridDim.x * nwarps) {
        T* xr = x + (size_t)row * d;
        if (VEC16) {
            const uint4* src = reinterpret_cast<const uint4*>(xr);
            for (int v = lane; v < d / EPV; v += 32) {
                uint4 raw = src[v];
                const T* e = reinterpret_cast<const T*>(&raw);
#pragma unroll
                for (int c = 0; c < EPV; c++) stage[v * EPV + c] = to_f32<T>(e[c]);
            }
        } else {
            for (int i = lane; i < d; i += 32) stage[i] = to_f32<T>(xr[i]);
        }
        __syncwarp();
        double acc = 0.0;
        for (int i = lane; i < d; i += 32) {
            double v = (double)stage[i];
            acc = fma(v, v, acc);
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) acc = acc + __shfl_xor_sync(0xffffffffu, acc, off);
        const float nrm = to_f32<T>(from_f32<T>((float)sqrt(acc)));
        if (VEC16) {
            uint4* dst = reinterpret_cast<uint4*>(xr);
            for (int v = lane; v < d / EPV; v += 32) {
                uint4 raw;
                T* e = reinterpret_cast<T*>(&raw);
#pragma unroll
                for (int c = 0; c < EPV; c++) e[c] = from_f32<T>(__fdiv_rn(stage[v * EPV + c], nrm));
                dst[v] = raw;
            }
        } else {
            for (int i = lane; i < d; i += 32) xr[i] = from_f32<T>(__fdiv_rn(stage[i], nrm));
        }
        __syncwarp();
    }
}

// fp32 rows whose length is a multiple of 128 (every CLIP width): the tuned form of the kernel above, same arithmetic.
//   * a warp takes TWO rows per step: both rows' 128-bit streaming loads (ld.global.cs) are in flight together and the
//     two fp64 chains interleave;
//   * the row stays in registers: shared memory is used only to transpose it into the CANON-32 order for the sum of squares
//     (lane l owns elements l, l+32, ...: 128-bit stores, conflict-free 32-bit loads); the quotients are computed from the
//     registers and written back with 128-bit stores;
//   * x / norm, correctly rounded, without the 16 MUFU.RCP + FCHK + slow-path calls per lane that __fdiv_rn expands to: the
//     reciprocal of the norm is taken once per row (__frcp_rn, correctly rounded) and every quotient is two Markstein
//     steps  q <- q + (x - q n) r  on FMAs (the first makes q faithful, the second correctly rounded), the sign of a zero
//     restored at the end.  That holds while nothing under- or overflows on the way: rows whose norm or whose non-zero
//     elements lie outside [2^-60, 2^60] (or hold inf / NaN) take __fdiv_rn instead (a warp-uniform branch per row).
//     tests/test_gpu_parity.py compares against the oracle's IEEE division bit for bit, extreme rows included.
// The first version (one row per warp, staged reads for the quotients too, __fdiv_rn) ran at 0.76x of the HBM roofline.
__device__ __forceinline__ float div_by_norm(float x, float n, float r) {
    float q = x * r;
    q = fmaf(fmaf(-q, n, x), r, q);
    q = fmaf(fmaf(-q, n, x), r, q);
    return __uint_as_float((__float_as_uint(q) & 0x7FFFFFFFu) | (__float_as_uint(x) & 0x80000000u));
}
// 1 when |x| is neither zero nor inside [2^-60, 2^60] (inf and NaN included)
__device__ __forceinline__ unsigned out_of_fast_range(float x) {
    const unsigned t = __float_as_uint(x) & 0x7FFFFFFFu;
    return (t != 0u && (t - 0x21800000u) > (0x5D800000u - 0x21800000u)) ? 1u : 0u;
}

template <int NV>
__global__ void __launch_bounds__(256) l2_normalize_f32_kernel(float* __restrict__ x, long long n) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    constexpr int D = 128 * NV;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    float* stage = reinterpret_cast<float*>(smem_raw) + (size_t)warp * 2 * D;
    const long long pairs = (n + 1) / 2;
    for (long long pr = (long long)blockIdx.x * nwarps + warp; pr < pairs; pr += (long long)gridDim.x * nwarps) {
        const long long r0 = 2 * pr;
        const bool two = r0 + 1 < n;
        float4* xa = reinterpret_cast<float4*>(x + (size_t)r0 * D);
        float4* xb = reinterpret_cast<float4*>(x + (size_t)(two ? r0 + 1 : r0) * D);  // odd tail: row r0 twice (stored once)
        float4 va[NV], vb[NV];
#pragma unroll
        for (int u = 0; u < NV; u++) va[u] = __ldcs(xa + lane + 32 * u);  // streaming, but coherent: the row is rewritten in place
#pragma unroll
        for (int u = 0; u < NV; u++) vb[u] = __ldcs(xb + lane + 32 * u);
        unsigned bad = 0u;
#pragma unroll
        for (int u = 0; u < NV; u++) {
            reinterpret_cast<float4*>(stage)[lane + 32 * u] = va[u];
            reinterpret_cast<float4*>(stage + D)[lane + 32 * u] = vb[u];
            bad |= out_of_fast_range(va[u].x) | out_of_fast_range(va[u].y) | out_of_fast_range(va[u].z) | out_of_fast_range(va[u].w);
            bad |= out_of_fast_range(vb[u].x) | out_of_fast_range(vb[u].y) | out_of_fast_range(vb[u].z) | out_of_fast_range(vb[u].w);
        }
        __syncwarp();
        double acca = 0.0, accb = 0.0;
#pragma unroll
        for (int j = 0; j < 4 * NV; j++) {
            const double wa = (double)stage[lane + 32 * j];
            const double wb = (double)stage[D + lane + 32 * j];
            acca = fma(wa, wa, acca);
            accb = fma(wb, wb, accb);
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            acca = acca + __shfl_xor_sync(0xffffffffu, acca, off);
            accb = accb + __shfl_xor_sync(0xffffffffu, accb, off);
        }
        const float na = (float)sqrt(acca), nb = (float)sqrt(accb);
        bad |= out_of_fast_range(na) | out_of_fast_range(nb) | (na == 0.f ? 1u : 0u) | (nb == 0.f ? 1u : 0u);
        if (!__any_sync(0xffffffffu, bad != 0u)) {
            const float ra = __frcp_rn(na), rb = __frcp_rn(nb);
#pragma unroll
            for (int u = 0; u < NV; u++) {
                float4 o;
                o.x = div_by_norm(va[u].x, na, ra);
                o.y = div_by_norm(va[u].y, na, ra);
                o.z = div_by_norm(va[u].z, na, ra);
                o.w = div_by_norm(va[u].w, na, ra);
                xa[lane + 32 * u] = o;
            }
            if (two) {
#pragma unroll
                for (int u = 0; u < NV; u++) {
                    float4 o;
                    o.x = div_by_norm(vb[u].x, nb, rb);
                    o.y = div_by_norm(vb[u].y, nb, rb);
                    o.z = div_by_norm(vb[u].z, nb, rb);
                    o.w = div_by_norm(vb[u].w, nb, rb);
                    xb[lane + 32 * u] = o;
                }
            }
        } else {  // extreme magnitudes, zero rows (x / 0), inf, NaN: IEEE division as it comes (operands re-read from the staging rows)
#pragma unroll 1
            for (int u = 0; u < (two ? 2 : 1) * NV; u++) {
                const bool second = u >= NV;
                const float nn = second ? nb : na;
                const int vi = lane + 32 * (second ? u - NV : u);
                const float4 v = reinterpret_cast<const float4*>(second ? stage + D : stage)[vi];
                float4 o;
                o.x = __fdiv_rn(v.x, nn);
                o.y = __fdiv_rn(v.y, nn);
                o.z = __fdiv_rn(v.z, nn);
                o.w = __fdiv_rn(v.w, nn);
                (second ? xb : xa)[vi] = o;
            }
        }
        __syncwarp();  // the staging rows are rewritten by the next pair
    }
}

// =============================================================================================
// fp32 -> bf16 (round to nearest even), 2 x 128-bit loads and 1 x 128-bit store per thread
// =============================================================================================
__global__ void __launch_bounds__(256) f32_to_bf16_kernel(const float* __restrict__ src, __nv_bfloat16* __restrict__ dst,
                                                         long long count) {
    const long long nvec = count / 8;
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += stride) {
        float4 a = ldg_stream_f4(reinterpret_cast<const float4*>(src) + 2 * v);
        float4 b = ldg_stream_f4(reinterpret_cast<const float4*>(src) + 2 * v + 1);
        __nv_bfloat162 o0 = __floats2bfloat162_rn(a.x, a.y), o1 = __floats2bfloat162_rn(a.z, a.w);
        __nv_bfloat162 o2 = __floats2bfloat162_rn(b.x, b.y), o3 = __floats2bfloat162_rn(b.z, b.w);
        uint4 out;
        out.x = *reinterpret_cast<uint32_t*>(&o0);
        out.y = *reinterpret_cast<uint32_t*>(&o1);
        out.z = *reinterpret_cast<uint32_t*>(&o2);
        out.w = *reinterpret_cast<uint32_t*>(&o3);
        reinterpret_cast<uint4*>(dst)[v] = out;
    }
    // tail (count not a multiple of 8)
    for (long long i = nvec * 8 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride)
        dst[i] = __float2bfloat16_rn(src[i]);
}

// fp16 / bf16 -> fp32 (exact), used by add_dev for half-precision encoder output (oldapp.py:86 astype)
template <typename T>
__global__ void __launch_bounds__(256) to_f32_kernel(const T* __restrict__ src, float* __restrict__ dst, long long count) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) dst[i] = to_f32<T>(src[i]);
}

// =============================================================================================
// row gather: dst[i][:] = src[ids[i]][:] (incremental re-index keeps the rows of unchanged files on the device).
// One warp per row, 128-bit copies when d % 4 == 0.
// =============================================================================================
__global__ void __launch_bounds__(256) gather_rows_kernel(const float* __restrict__ src, const long long* __restrict__ ids,
                                                         float* __restrict__ dst, long long n, int d) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
        const float* s = src + (size_t)ids[r] * d;
        float* o = dst + (size_t)r * d;
        if ((d & 3) == 0) {
            for (int i = lane; i < (d >> 2); i += 32) reinterpret_cast<float4*>(o)[i] = reinterpret_cast<const float4*>(s)[i];
        } else {
            for (int i = lane; i < d; i += 32) o[i] = s[i];
        }
    }
}

// =============================================================================================
// largest row norm of rows [0, n): one warp per row, fp32 sum of squares (an upper-bound estimate is all the
// certification needs: it is inflated by 1e-6 relative on use), atomicMax on the float bits (norms are >= 0, so the
// unsigned order of the bits is the numeric order).  NaN rows are ignored.
// =============================================================================================
// 1 when |x| is subnormal, infinite or NaN (zero and normal numbers: 0)
__device__ __forceinline__ unsigned is_special_f32(float x) {
    const unsigned t = __float_as_uint(x) & 0x7FFFFFFFu;
    return (t != 0u && (t - 0x00800000u) >= 0x7F000000u) ? 1u : 0u;
}
// With dst16 != null the same pass also writes the rows rounded to bf16 (RNE); an element that rounds to a bf16 infinity
// marks the index special.  With dst8 != null it writes the int8 scan copy: per row the scale s = max|x_i| / 127 (fp32) to
// scale8 and the codes c_i = rint(x_i / s) (|c_i| <= 127) to dst8, and raises *emax to the largest |x - s c|_2 of a row,
// summed in fp64 and rounded up: the bound the single-query scans of the copy are made exact with (evs_scan.cuh:
// scan_pool_kernel).  The codes take a second read of the row, which the first has just brought on chip.
__global__ void __launch_bounds__(256) row_norm_max_kernel(const float* __restrict__ rows, long long n, int d, float* __restrict__ max_norm,
                                                          unsigned* __restrict__ special, __nv_bfloat16* __restrict__ dst16,
                                                          signed char* __restrict__ dst8, float* __restrict__ scale8,
                                                          float* __restrict__ emax) {
    const int lane = threadIdx.x & 31;
    const long long warps = ((long long)gridDim.x * blockDim.x) >> 5;
    float best = 0.f;
    double ebest = 0.0;
    unsigned spec = 0u;
    auto to16 = [&](float v) {
        const __nv_bfloat16 h = __float2bfloat16_rn(v);
        spec |= (isinf(__bfloat162float(h)) && !isinf(v)) ? 1u : 0u;
        return h;
    };
    auto to8 = [&](float v, float sc, double& e2) {
        const float c = sc > 0.f ? fminf(fmaxf(rintf(__fdiv_rn(v, sc)), -127.f), 127.f) : 0.f;
        const double diff = (double)v - (double)sc * (double)c;  // s c exact in fp64
        e2 = fma(diff, diff, e2);
        return (int)c;
    };
    const bool vec = (d & 3) == 0;
    for (long long r = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < n; r += warps) {
        const float* x = rows + (size_t)r * d;
        float s = 0.f, amax = 0.f;
        double e2 = 0.0;
        if (vec) {
            for (int i = lane; i < (d >> 2); i += 32) {
                const float4 v = ldg_stream_f4(reinterpret_cast<const float4*>(x) + i);
                s = fmaf(v.x, v.x, s);
                s = fmaf(v.y, v.y, s);
                s = fmaf(v.z, v.z, s);
                s = fmaf(v.w, v.w, s);
                amax = fmaxf(amax, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
                spec |= is_special_f32(v.x) | is_special_f32(v.y) | is_special_f32(v.z) | is_special_f32(v.w);
                if (dst16) {
                    __nv_bfloat162 o0, o1;
                    o0.x = to16(v.x);
                    o0.y = to16(v.y);
                    o1.x = to16(v.z);
                    o1.y = to16(v.w);
                    uint2 o;
                    o.x = *reinterpret_cast<uint32_t*>(&o0);
                    o.y = *reinterpret_cast<uint32_t*>(&o1);
                    reinterpret_cast<uint2*>(dst16 + (size_t)r * d)[i] = o;
                }
            }
        } else {
            for (int i = lane; i < d; i += 32) {
                s = fmaf(x[i], x[i], s);
                amax = fmaxf(amax, fabsf(x[i]));
                spec |= is_special_f32(x[i]);
                if (dst16) dst16[(size_t)r * d + i] = to16(x[i]);
            }
        }
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, off);
            amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, off));
        }
        if (dst8) {
            const float sc = __fdiv_rn(amax, 127.f);  // (NaN rows: NaN scale; they mark the index special, whose searches scan fp32)
            if (lane == 0) scale8[r] = sc;
            if (vec) {
                for (int i = lane; i < (d >> 2); i += 32) {
                    const float4 v = reinterpret_cast<const float4*>(x)[i];
                    const unsigned o = ((unsigned)to8(v.x, sc, e2) & 255u) | (((unsigned)to8(v.y, sc, e2) & 255u) << 8) |
                                       (((unsigned)to8(v.z, sc, e2) & 255u) << 16) | (((unsigned)to8(v.w, sc, e2) & 255u) << 24);
                    reinterpret_cast<unsigned*>(dst8 + (size_t)r * d)[i] = o;
                }
            } else {
                for (int i = lane; i < d; i += 32) dst8[(size_t)r * d + i] = (signed char)to8(x[i], sc, e2);
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) e2 += __shfl_xor_sync(0xffffffffu, e2, off);
        }
        if (s == s) best = fmaxf(best, s);
        if (e2 > ebest) ebest = e2;  // (NaN rows mark the index special: its single-query searches scan the fp32 rows)
    }
    if (lane == 0 && best > 0.f) atomicMax(reinterpret_cast<unsigned*>(max_norm), __float_as_uint(sqrtf(best) * 1.000001f));
    if (spec && special) atomicOr(special, 1u);  // the index holds a subnormal / inf / NaN element: the finalise widens fp32 -> fp64 the slow exact way
    if (lane == 0 && emax && ebest > 0.0) atomicMax(reinterpret_cast<unsigned*>(emax), __float_as_uint(__double2float_ru(__dsqrt_ru(ebest))));
}

__global__ void fill_i32_kernel(int* __restrict__ p, long long count, int value) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) p[i] = value;
}

// =============================================================================================
// synthetic rows: value(seed, global row, col) -- same integer function as oracle/orc_synth_fill
// =============================================================================================
__device__ __forceinline__ u64 splitmix64(u64 z) {
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
__device__ __forceinline__ float synth_value(u64 hr, int col) {
    u64 h = splitmix64(hr + (u64)col);
    int s = (int)(h & 0xFFFF) + (int)((h >> 16) & 0xFFFF) + (int)((h >> 32) & 0xFFFF) + (int)((h >> 48) & 0xFFFF) - 131070;
    return (float)s;
}
// one thread per 4 consecutive columns (d % 4 == 0) or per element otherwise
__global__ void __launch_bounds__(256) synth_fill_kernel(float* __restrict__ out, long long n, int d, u64 seed,
                                                        long long row_base) {
    const u64 s0 = splitmix64(seed ^ 0xD1B54A32D192ED03ull);
    const long long stride = (long long)gridDim.x * blockDim.x;
    if ((d & 3) == 0) {
        const int vpr = d >> 2;
        const long long total = n * vpr;
        for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < total; v += stride) {
            long long r = v / vpr;
            int c = (int)(v % vpr) * 4;
            u64 hr = splitmix64(s0 + (u64)(r + row_base) * 0x2545F4914F6CDD1Dull);
            float4 o = make_float4(synth_value(hr, c), synth_value(hr, c + 1), synth_value(hr, c + 2),
                                   synth_value(hr, c + 3));
            reinterpret_cast<float4*>(out)[v] = o;
        }
    } else {
        const long long total = n * d;
        for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
            long long r = i / d;
            int c = (int)(i % d);
            u64 hr = splitmix64(s0 + (u64)(r + row_base) * 0x2545F4914F6CDD1Dull);
            out[i] = synth_value(hr, c);
        }
    }
}

// =============================================================================================
// launch wrappers
// =============================================================================================
static int clamp_grid(long long want, int cap) {
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

template <int NV>
static cudaError_t launch_l2_normalize_f32(float* x, long long n, int sm_count, cudaStream_t st) {
    const int threads = 256, nwarps = threads / 32;
    const size_t smem = (size_t)nwarps * 2 * 128 * NV * sizeof(float);
    static size_t optin[16] = {};
    cudaError_t oe = ensure_smem_optin(l2_normalize_f32_kernel<NV>, smem, optin);
    if (oe != cudaSuccess) return oe;
    int per_sm = (int)((200 * 1024) / (smem + 1024));
    if (per_sm > 6) per_sm = 6;
    if (per_sm < 1) per_sm = 1;
    const int grid = clamp_grid(((n + 1) / 2 + nwarps - 1) / nwarps, sm_count * per_sm);
    l2_normalize_f32_kernel<NV><<<grid, threads, smem, st>>>(x, n);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_l2_normalize(void* x, long long n, int d, int dtype, int sm_count, cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    if (dtype == EVS_F32 && d % 128 == 0 && (reinterpret_cast<uintptr_t>(x) % 16) == 0) {
        float* xf = reinterpret_cast<float*>(x);
        switch (d / 128) {  // 128 .. 1024: the CLIP widths (512, 768, 1024) and their neighbours
            case 1: return launch_l2_normalize_f32<1>(xf, n, sm_count, st);
            case 2: return launch_l2_normalize_f32<2>(xf, n, sm_count, st);
            case 3: return launch_l2_normalize_f32<3>(xf, n, sm_count, st);
            case 4: return launch_l2_normalize_f32<4>(xf, n, sm_count, st);
            case 5: return launch_l2_normalize_f32<5>(xf, n, sm_count, st);
            case 6: return launch_l2_normalize_f32<6>(xf, n, sm_count, st);
            case 8: return launch_l2_normalize_f32<8>(xf, n, sm_count, st);
            default: break;
        }
    }
    const int threads = 256, nwarps = threads / 32;
    size_t smem = (size_t)nwarps * d * sizeof(float);
    int grid = clamp_grid((n + nwarps - 1) / nwarps, sm_count * 8);
    const size_t esz = dtype == EVS_F32 ? 4 : 2;
    const bool vec = ((size_t)d * esz) % 16 == 0 && (reinterpret_cast<uintptr_t>(x) % 16) == 0;
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
#define EVS_NORM(T, V)                                                                                   \
    do {                                                                                                 \
        if (smem > 48 * 1024)                                                                            \
            cudaFuncSetAttribute(l2_normalize_kernel<T, V>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        l2_normalize_kernel<T, V><<<grid, threads, smem, st>>>(reinterpret_cast<T*>(x), n, d);          \
    } while (0)
    if (dtype == EVS_F32) { if (vec) EVS_NORM(float, true); else EVS_NORM(float, false); }
    else if (dtype == EVS_F16) { if (vec) EVS_NORM(__half, true); else EVS_NORM(__half, false); }
    else if (dtype == EVS_BF16) { if (vec) EVS_NORM(__nv_bfloat16, true); else EVS_NORM(__nv_bfloat16, false); }
    else return cudaErrorInvalidValue;
#undef EVS_NORM
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_f32_to_bf16(const float* src, void* dst, long long count, int sm_count, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    int grid = clamp_grid((count / 8 + 255) / 256, sm_count * 16);
    f32_to_bf16_kernel<<<grid, 256, 0, st>>>(src, reinterpret_cast<__nv_bfloat16*>(dst), count);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_to_f32(const void* src, int dtype, float* dst, long long count, int sm_count, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    int grid = clamp_grid((count + 255) / 256, sm_count * 16);
    if (dtype == EVS_F16) to_f32_kernel<__half><<<grid, 256, 0, st>>>(reinterpret_cast<const __half*>(src), dst, count);
    else if (dtype == EVS_BF16)
        to_f32_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>(reinterpret_cast<const __nv_bfloat16*>(src), dst, count);
    else return cudaErrorInvalidValue;
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_gather_rows(const float* src, const long long* ids_dev, float* dst, long long n, int d, int sm_count,
                               cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    int grid = clamp_grid((n * 32 + 255) / 256, sm_count * 16);
    gather_rows_kernel<<<grid, 256, 0, st>>>(src, ids_dev, dst, n, d);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_synth_fill(float* out, long long n, int d, unsigned long long seed, long long row_base, int sm_count,
                              cudaStream_t st) {
    if (n <= 0) return cudaSuccess;
    long long work = (d & 3) == 0 ? n * (d >> 2) : n * d;
    int grid = clamp_grid((work + 255) / 256, sm_count * 16);
    synth_fill_kernel<<<grid, 256, 0, st>>>(out, n, d, seed, row_base);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_merge_partials(int nparts, long long nq, int k, const double* scores, const long long* ids,
                                  long long part_stride, float* D, long long* I, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    if (k <= EVS_MAX_K) {
        const size_t smem = (size_t)nparts * k * 24;
        if (smem > 200 * 1024) return cudaErrorInvalidValue;
        if (smem > 48 * 1024)
            cudaFuncSetAttribute(merge_partials_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        merge_partials_kernel<<<(unsigned)nq, 256, smem, st>>>(nparts, nq, k, scores, ids, part_stride, D, I);
    } else {
        const unsigned gx = (unsigned)((nparts * k + 255) / 256);
        const unsigned gy = (unsigned)(nq < 65535 ? nq : 65535);
        merge_partials_kernel<<<dim3(gx, gy), 256, 0, st>>>(nparts, nq, k, scores, ids, part_stride, D, I);
    }
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_publish_partials(const Exchange& x, long long nq, int k, const double* scores, const long long* ids,
                                    cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    const long long count = nq * k;
    int grid = (int)((count + 255) / 256 < 64 ? (count + 255) / 256 : 64);
    publish_partials_kernel<<<grid, 256, 0, st>>>(x, count, scores, ids);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_publish_poison(const Exchange& x, cudaStream_t st) {
    const long long count = x.nq_total * x.k;
    if (count <= 0) return cudaSuccess;
    int grid = (int)((count + 255) / 256 < 64 ? (count + 255) / 256 : 64);
    publish_poison_kernel<<<grid, 256, 0, st>>>(x, count);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_merge_exchange(const Exchange& x, long long nq, int k, float* D, long long* I, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    if (x.world < 1 || x.world > 8) return cudaErrorInvalidValue;
    const bool staged = k <= EVS_MAX_K;
    const size_t smem = staged ? (size_t)x.world * k * 24 : 0;  // at most 8 * 112 * 24 bytes: no opt-in needed
    cudaError_t le = launch_pdl(merge_exchange_kernel, dim3((unsigned)nq), dim3(staged ? 256 : 1024), smem, st, x, k, D, I);
    g_kernel_launches.fetch_add(1);
    if (le != cudaSuccess) return le;
    return cudaGetLastError();
}

cudaError_t launch_row_norm_max(const float* rows, long long n, int d, float* max_norm, unsigned* special, int sm_count, cudaStream_t st,
                                void* dst16, signed char* dst8, float* scale8, float* emax) {
    if (n <= 0) return cudaSuccess;
    int grid = clamp_grid((n * 32 + 255) / 256, sm_count * 8);
    row_norm_max_kernel<<<grid, 256, 0, st>>>(rows, n, d, max_norm, special, reinterpret_cast<__nv_bfloat16*>(dst16), dst8, scale8, emax);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

cudaError_t launch_fill_i32(int* p, long long count, int value, cudaStream_t st) {
    if (count <= 0) return cudaSuccess;
    int grid = clamp_grid((count + 255) / 256, 64);
    fill_i32_kernel<<<grid, 256, 0, st>>>(p, count, value);
    EVS_LAUNCH_CHECK();
    return cudaSuccess;
}

size_t finalize_smem_bytes_host(int L, int kp, int d) { return finalize_smem_bytes(L, kp, d) + 16; }

cudaError_t launch_finalize(const FinalizeParams& p, long long nq, cudaStream_t st) {
    if (nq <= 0) return cudaSuccess;
    size_t smem = finalize_smem_bytes_host(p.L, p.kp, p.d);
    if (smem > 200 * 1024) return cudaErrorInvalidValue;
    static size_t optin[16] = {};
    cudaError_t oe = ensure_smem_optin(finalize_kernel, smem, optin);
    if (oe != cudaSuccess) return oe;
    // small batches: 1024 threads shorten the single CTA's critical path; large batches: 256 threads
    // so that several queries share an SM
    const int threads = nq <= 296 ? 1024 : 256;
    cudaError_t le = launch_pdl(finalize_kernel, dim3((unsigned)nq), dim3((unsigned)threads), smem, st, p);
    g_kernel_launches.fetch_add(1);
    if (le != cudaSuccess) return le;
    return cudaGetLastError();
}

// number of vectors per lane per row for the vectorised kernels (16 bytes; 8 bytes of int8 codes), 0 = use the generic
// kernel (int8: no scan)
static int vectors_per_lane(int d, int elem) {
    int unit = elem == SCAN_F32 ? 128 : 256;
    if (d % unit) return 0;
    int nv = d / unit;
    if (elem != SCAN_F32) return (nv >= 1 && nv <= 4) ? nv : 0;
    return (nv == 1 || nv == 2 || nv == 3 || nv == 4 || nv == 6 || nv == 8) ? nv : 0;
}

// Decide variant, grid, block and shared memory for a scan over `n` rows (does not launch).
cudaError_t plan_scan(long long n, int d, int elem, int kp, int nq_pass, int sm_count, const ScanTuning& tune,
                      ScanPlan* plan) {
    const int nv = vectors_per_lane(d, elem);
    const size_t esz = elem == SCAN_F32 ? 4 : (elem == SCAN_BF16 ? 2 : 1);
    plan->nv = nv;
    if (nv == 0 && elem == SCAN_I8) return cudaErrorInvalidValue;
    if (nv == 0) {
        plan->variant = 0;
        plan->threads = 256;
        plan->smem_bytes = (size_t)(plan->threads / 32) * 2 * kp * 8;
        plan->grid = clamp_grid((n + 7) / 8, sm_count * 4);
        plan->tile_rows = plan->stages = 0;
        return cudaSuccess;
    }
    int variant = tune.scan_variant ? tune.scan_variant : 1;
    if (variant == 2 && elem != SCAN_I8) {
        const int cw = 8;
        size_t row_bytes = (size_t)d * esz;
        int tr = tune.tile_rows > 0 ? tune.tile_rows : (int)(32768 / row_bytes);
        if (tr < 1) tr = 1;
        size_t sel = (size_t)cw * nq_pass * 2 * kp * 8;
        int stages = tune.stages > 0 ? tune.stages : 4;
        const size_t budget = 200 * 1024;
        while (stages > 2 && (size_t)stages * tr * row_bytes + sel + 2 * stages * 8 > budget) stages--;
        while (tr > 1 && (size_t)stages * tr * row_bytes + sel + 2 * stages * 8 > budget) tr--;
        size_t smem = (size_t)stages * tr * row_bytes + 2 * stages * 8 + sel;
        if (smem > budget) variant = 1;
        else {
            plan->variant = 2;
            plan->threads = 32 * (cw + 1);
            plan->tile_rows = tr;
            plan->stages = stages;
            plan->smem_bytes = smem;
            long long ntiles = (n + tr - 1) / tr;
            plan->grid = clamp_grid(ntiles, sm_count);
            return cudaSuccess;
        }
    }
    plan->variant = 1;
    plan->threads = 256;
    plan->tile_rows = plan->stages = 0;
    plan->smem_bytes = (size_t)(plan->threads / 32) * nq_pass * 2 * kp * 8;
    // measured on B200 at 10M x 512 (profiles/r01_tune_scan_*): fp32 rows peak at 2 CTAs/SM, bf16 rows
    // (half the bytes in flight per row) need 4; int8 rows hold two groups in registers (ScanOcc) and peak at 2
    // (profiles/int8_group_occupancy_sweep.jsonl)
    int per_sm = tune.ctas_per_sm > 0 ? tune.ctas_per_sm : (elem == SCAN_BF16 ? 4 : 2);
    long long groups = (n + 3) / 4;
    plan->grid = clamp_grid((groups + 7) / 8, sm_count * per_sm);
    return cudaSuccess;
}

size_t scan_pool_key_slots(size_t pool_words) { return pool_words > (size_t)POOL_HDR ? pool_words - (size_t)POOL_HDR : 0; }
size_t scan_pool_words(const ScanPlan& plan) { return (size_t)POOL_HDR + (size_t)plan.grid * (plan.threads / 32) * 128; }
size_t scan_pool_window_words() { return 3 * (size_t)POOL_CMAX; }

cudaError_t launch_scan(const ScanArgs& a, ScanPlan* plan, cudaStream_t st) {
    if (a.n <= 0) return cudaErrorInvalidValue;
    if (a.is_i8) return launch_scan_i8(a, plan, st);
    if (plan->nv == 0) return launch_scan_generic_any(a, plan, st);
    if (a.is_bf16) return plan->nv <= 2 ? launch_scan_bf16_narrow(a, plan, st) : launch_scan_bf16_wide(a, plan, st);
    if (plan->nv <= 3) return launch_scan_f32_narrow(a, plan, st);
    if (plan->nv == 4) return launch_scan_f32_512(a, plan, st);
    return launch_scan_f32_wide(a, plan, st);
}

}  // namespace evs
