// evs_large_k.cu -- exact search for EVS_MAX_K < k <= EVS_MAX_K_LARGE (option "max_k"; DESIGN.md section 2).
//
// The k <= 112 paths keep a fixed candidate list of k' = 64 or 128 keys per scan.  A large k takes a different shape,
// one pass of up to max_queries_per_pass(d) queries at a time, every kernel chained with programmatic serialisation:
//   1. lk_score_kernel      the fp32 GEMV of scan_direct_kernel (same loads, same row_scores arithmetic, same grid), but it
//                           writes every row's scan score as an order-preserving u32 key to S[q][row] (a warp collects 32
//                           rows and stores them with one 128-byte store) and builds a histogram of the keys' top 11 bits;
//   2. lk_select / lk_hist  radix select of s_(k), the exact k-th largest scan key (digits 11 + 11 + 10 bits; the later
//                           passes count only the keys that share the digits found so far); the cut is the key of
//                           score(s_(k)) - 2E rounded down, E = gemv_err_coef(d) |q| max|x| (every row, when the index has a
//                           subnormal / inf / NaN element or E is not finite);
//   3. lk_compact_kernel    every row whose key is >= the cut joins the candidate list C (one atomic per warp);
//   4. lk_rescore_kernel    grid-wide CANON-32 fp64 score of every candidate (canon32_dot_multi: the bits the finalise
//                           computes for the same row);
//   5. lk_rank_kernel       top k of C by (canonical desc, row asc): a shared-memory bitonic sort of up to LK_SORT keys,
//                           or -- larger C (ties, special data) -- a radix select of the k-th (score, row) pair first.
// Exact by construction: the k rows with the best scan scores all have exact scores >= s_(k) - E, so the exact k-th score
// is >= s_(k) - E and every row of the exact top k has a scan score >= s_(k) - 2E.
// Batches of 2..4 queries with k <= EVS_MAX_K over an int8 copy take the same kernels with lk_score_i8_kernel as step 1 and
// the copy's bound as E (plan_path in evs_api.cu).
#include <float.h>

#include <atomic>

#include "evs_internal.h"
#include "evs_scan.cuh"
#include "evs_scan_launch.cuh"

namespace evs {

constexpr int LK_SORT = 4096;  // candidates the rank kernel sorts in shared memory (>= EVS_MAX_K_LARGE)
static_assert(LK_SORT >= EVS_MAX_K_LARGE, "the rank kernel sorts the k selected candidates in shared memory");

__device__ __forceinline__ void lk_wait() {
    asm volatile("griddepcontrol.wait;" ::: "memory");
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// inverse of score_rank_key (canonical scores are never -0.0: the CANON-32 sum starts at +0.0)
__device__ __forceinline__ double rank_key_score(u64 o) {
    const u64 u = (o & 0x8000000000000000ull) ? (o & 0x7FFFFFFFFFFFFFFFull) : ~o;
    return __longlong_as_double((long long)u);
}

// add the block's digit histogram to the global one (zeroed before the pass)
__device__ __forceinline__ void lk_flush_hist(const unsigned* h, unsigned* g, int nbins) {
    for (int b = threadIdx.x; b < nbins; b += blockDim.x) {
        const unsigned v = h[b];
        if (v) atomicAdd(g + b, v);
    }
}

// ---------------------------------------------------------------------------------------------
// 1. score scan
// ---------------------------------------------------------------------------------------------
template <int NQ, int NV>
__global__ void __launch_bounds__(256, ScanOcc<float, NQ, NV>::value) lk_score_kernel(LargeKArgs a) {
    __shared__ unsigned h[NQ][LK_BINS];
    constexpr int QREGS = NQ * NV * 4;
    constexpr int RAW = (100 - QREGS) / (NV * 4);  // rows in flight per warp, sized like scan_direct_kernel's
    constexpr int RPG = RAW >= 4 ? 4 : RAW >= 2 ? 2 : 1;  // ... but a divisor of 32
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int i = threadIdx.x; i < NQ * LK_BINS; i += blockDim.x) (&h[0][0])[i] = 0u;
    lk_wait();
    __syncthreads();
    QueryRegs<float, NQ, NV> q;
    q.load(a.xq, 0, a.d, lane);
    const size_t row_vecs = (size_t)a.d / 4;
    const float4* base = reinterpret_cast<const float4*>(a.xb);
    const long long nblk = (a.n + 31) / 32;
    const long long total_warps = (long long)gridDim.x * nwarps;
    for (long long blk = (long long)blockIdx.x * nwarps + warp; blk < nblk; blk += total_warps) {
        const long long r0 = blk * 32;
        unsigned mine[NQ];
#pragma unroll
        for (int qi = 0; qi < NQ; qi++) mine[qi] = 0u;
#pragma unroll 1
        for (int g = 0; g < 32; g += RPG) {
            float4 raw[RPG][NV];
#pragma unroll
            for (int r = 0; r < RPG; r++) {
                const long long row = r0 + g + r < a.n ? r0 + g + r : a.n - 1;  // clamp: tail rows are re-read, not stored
                const float4* src = base + (size_t)row * row_vecs + lane;
#pragma unroll
                for (int j = 0; j < NV; j++) raw[r][j] = ldg_stream_f4(src + 32 * j);
            }
#pragma unroll
            for (int r = 0; r < RPG; r++) {
                float s[NQ];
                row_scores<float, NQ, NV>(raw[r], q, s);
#pragma unroll
                for (int qi = 0; qi < NQ; qi++) mine[qi] = lane == g + r ? score_to_ordered(s[qi]) : mine[qi];
            }
        }
        if (r0 + lane < a.n) {
#pragma unroll
            for (int qi = 0; qi < NQ; qi++) {
                a.S[(size_t)qi * a.npad + r0 + lane] = mine[qi];
                atomicAdd(&h[qi][mine[qi] >> 21], 1u);
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int qi = 0; qi < NQ; qi++) lk_flush_hist(h[qi], a.hist + (size_t)qi * LK_BINS, LK_BINS);
}

// any d: the arithmetic of scan_generic_kernel (one fp32 FMA chain per lane, then the butterfly); query blockIdx.y
__global__ void __launch_bounds__(256) lk_score_generic_kernel(LargeKArgs a) {
    __shared__ unsigned h[LK_BINS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const int qi = blockIdx.y;
    for (int i = threadIdx.x; i < LK_BINS; i += blockDim.x) h[i] = 0u;
    lk_wait();
    __syncthreads();
    const float* q = a.xq + (size_t)qi * a.d;
    const long long nblk = (a.n + 31) / 32;
    for (long long blk = (long long)blockIdx.x * nwarps + warp; blk < nblk; blk += (long long)gridDim.x * nwarps) {
        const long long r0 = blk * 32;
        unsigned mine = 0u;
        for (int r = 0; r < 32 && r0 + r < a.n; r++) {
            const float* x = a.xb + (size_t)(r0 + r) * a.d;
            float s = 0.f;
            for (int i = lane; i < a.d; i += 32) s = fmaf(__ldg(x + i), __ldg(q + i), s);
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
            if (lane == r) mine = score_to_ordered(s);
        }
        if (r0 + lane < a.n) {
            a.S[(size_t)qi * a.npad + r0 + lane] = mine;
            atomicAdd(&h[mine >> 21], 1u);
        }
    }
    __syncthreads();
    lk_flush_hist(h, a.hist + (size_t)qi * LK_BINS, LK_BINS);
}

// The int8 copy, NQ = LK_I8_NQ queries per pass (batches of 2..4 queries, k <= EVS_MAX_K; DESIGN.md section 2): the
// arithmetic of scan_pool_kernel<int8_t> -- the same query codes and split 16-bit IDP.4A chains, the exact integer I, the
// same wide-d fp64 combine and s~ = fl(fl(I) fl(s_q s_r)) -- so that its bound E holds for every key.  A group of R rows
// yields R * NQ (* 2 for wide d) lane sums, 32 in all: one halving reduction leaves lane l with value l, so every lane
// (every other lane for wide d) ends holding one (row, query) score.
template <int NQ, int NV>
struct I8Batch {
    static constexpr int W = NV <= 2 ? 1 : 2;  // values per (row, query): the int32 sum, or the h and l chains
    static constexpr int R = 32 / (NQ * W);    // rows per group
    static_assert(R >= 1 && R * NQ * W == 32, "one value per lane after the reduction");
    static constexpr int OCC = 2;              // CTAs of 256 threads per SM (128 registers)
};

template <int NQ, int NV>
__global__ void __launch_bounds__(256, I8Batch<NQ, NV>::OCC) lk_score_i8_kernel(LargeKArgs a) {
    extern __shared__ unsigned lk_i8_hist[];  // [NQ][LK_BINS]
    typedef I8Lane<NV> L;
    typedef I8Batch<NQ, NV> B;
    constexpr int R = B::R, W = B::W;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    for (int i = threadIdx.x; i < NQ * LK_BINS; i += blockDim.x) lk_i8_hist[i] = 0u;
    lk_wait();
    __syncthreads();
    // queries past the pass's last repeat it: their keys are never stored
    QueryRegs<int8_t, 1, NV> q[NQ];
#pragma unroll
    for (int qi = 0; qi < NQ; qi++) q[qi].load(a.xq, qi < a.nq_pass ? qi : a.nq_pass - 1, a.d, lane);
    const int pair = lane / W, my_r = pair / NQ, my_q = pair % NQ;
    const bool rep = (lane % W) == 0;
    float my_sq = q[0].sq;
#pragma unroll
    for (int qi = 1; qi < NQ; qi++) my_sq = my_q == qi ? q[qi].sq : my_sq;
    const int8_t* codes = reinterpret_cast<const int8_t*>(a.xi8);
    struct Group {
        unsigned w[R][L::WORDS];
        float sr;  // the scale of row my_r
    };
    auto load = [&](Group& b, long long g) {
        const long long r0 = g * R;
        b.sr = __ldg(a.xs8 + (r0 + my_r < a.n ? r0 + my_r : a.n - 1));
#pragma unroll
        for (int r = 0; r < R; r++) {
            const long long row = r0 + r < a.n ? r0 + r : a.n - 1;  // clamp: tail rows are re-read, not stored
            L::load(codes + (size_t)row * a.d, lane, b.w[r]);
        }
    };
    auto score = [&](const Group& b, long long g) {
        int v[32];
#pragma unroll
        for (int r = 0; r < R; r++)
#pragma unroll
            for (int qi = 0; qi < NQ; qi++) {
                int ih = 0, il = 0;
#pragma unroll
                for (int w = 0; w < L::WORDS; w++) {
                    ih = __dp4a((int)b.w[r][w], q[qi].h[w], ih);
                    il = __dp4a((int)b.w[r][w], q[qi].l[w], il);
                }
                if constexpr (W == 1) v[r * NQ + qi] = ih * 256 + il;
                else {
                    v[2 * (r * NQ + qi)] = ih;
                    v[2 * (r * NQ + qi) + 1] = il;
                }
            }
        i8_warp_sum<32>(v, lane);
        float fi;
        if constexpr (W == 1) fi = __int2float_rn(v[0]);
        else {  // even lanes hold the h sum, odd lanes the l sum of the same (row, query)
            const int o = __shfl_xor_sync(0xffffffffu, v[0], 1);
            fi = __double2float_rn(fma((double)(rep ? v[0] : o), 256.0, (double)(rep ? o : v[0])));
        }
        const float s = __fmul_rn(fi, __fmul_rn(my_sq, b.sr));
        const long long row = g * R + my_r;
        if (rep && row < a.n && my_q < a.nq_pass) {
            const unsigned key = score_to_ordered(s);
            a.S[(size_t)my_q * a.npad + row] = key;
            atomicAdd(&lk_i8_hist[my_q * LK_BINS + (key >> 21)], 1u);
        }
    };
    const long long ngroups = (a.n + R - 1) / R;
    const long long total_warps = (long long)gridDim.x * nwarps;
    long long g = (long long)blockIdx.x * nwarps + warp;
    // one group in registers per warp: the other warps of the SM keep the loads in flight (two resident CTAs)
    for (; g < ngroups; g += total_warps) {
        Group A;
        load(A, g);
        score(A, g);
    }
    __syncthreads();
    for (int qi = 0; qi < a.nq_pass && qi < NQ; qi++) lk_flush_hist(lk_i8_hist + qi * LK_BINS, a.hist + (size_t)qi * LK_BINS, LK_BINS);
}

// ---------------------------------------------------------------------------------------------
// 2. threshold: radix select of the k-th largest scan key
// ---------------------------------------------------------------------------------------------
// With the LK_BINS bins of `h` taken in descending order: the bin b with above(b) < krem <= above(b) + h[b], above(b) the
// count of the bins above it, into *digit / *above (*digit stays -1 when krem exceeds the total).  All 1024 threads.
__device__ __forceinline__ void lk_find_digit(const unsigned* h, unsigned krem, unsigned* s_warp, int* digit, unsigned* above) {
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
    const int b0 = LK_BINS - 1 - 2 * t, b1 = b0 - 1;
    const unsigned c0 = h[b0], c1 = h[b1];
    unsigned v = c0 + c1;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) {
        const unsigned u = __shfl_up_sync(0xffffffffu, v, off);
        if (lane >= off) v += u;
    }
    if (lane == 31) s_warp[warp] = v;
    __syncthreads();
    if (warp == 0) {
        unsigned w = s_warp[lane];
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const unsigned u = __shfl_up_sync(0xffffffffu, w, off);
            if (lane >= off) w += u;
        }
        s_warp[lane] = w;
    }
    __syncthreads();
    const unsigned before = (warp ? s_warp[warp - 1] : 0u) + v - (c0 + c1);
    if (before < krem && krem <= before + c0) {
        *digit = b0;
        *above = before;
    } else if (before + c0 < krem && krem <= before + c0 + c1) {
        *digit = b1;
        *above = before + c0;
    }
    __syncthreads();
}

// E of query qi over the fp32 rows: gemv_err_coef(d) |q| max|x|, |q| and max|x| inflated for their own roundings (max_norm is
// an fp32 sum of squares: within d 2^-24 of the truth), plus an absolute term for products that underflow in fp32.  All
// threads of the CTA; every thread returns E.
__device__ __noinline__ float lk_f32_bound(const LargeKArgs& a, int qi, double* s_q2) {
    const int t = threadIdx.x;
    double q2 = 0.0;
    for (int i = t; i < a.d; i += blockDim.x) {
        const double v = (double)a.xq[(size_t)qi * a.d + i];
        q2 = fma(v, v, q2);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) q2 += __shfl_xor_sync(0xffffffffu, q2, off);
    if ((t & 31) == 0) s_q2[t >> 5] = q2;
    __syncthreads();
    q2 = 0.0;
    for (int w = 0; w < 32; w++) q2 += s_q2[w];
    const double qn = sqrt(q2) * (1.0 + 0x1p-20), nx = (double)__ldg(a.max_norm) * (1.0 + 0x1p-7);
    double e = (double)a.err_coef * qn * nx * (1.0 + 0x1p-20) + 0x1p-120;
    if (!(qn * nx <= 0x1p126)) e = INFINITY;  // fp32 partial sums might overflow: every row is a candidate
    return __double2float_ru(e);
}
// ... over the int8 copy: i8_scan_bound of |q - q^| and |q^|, from the query codes every warp of the score scan derived
__device__ __noinline__ float lk_i8_bound(const LargeKArgs& a, int qi, double* s_dq2, double* s_qh2) {
    const int t = threadIdx.x;
    const float* q = a.xq + (size_t)qi * a.d;
    const float sq = i8_query_scale(q, a.d, t & 31);
    double dq2 = 0.0, qh2 = 0.0;
    for (int i = t; i < a.d; i += blockDim.x) {
        const double qh = (double)sq * (double)i8_query_code(q[i], sq);  // exact: 24 x 16 bits
        dq2 = fma((double)q[i] - qh, (double)q[i] - qh, dq2);
        qh2 = fma(qh, qh, qh2);
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        dq2 += __shfl_xor_sync(0xffffffffu, dq2, off);
        qh2 += __shfl_xor_sync(0xffffffffu, qh2, off);
    }
    if ((t & 31) == 0) {
        s_dq2[t >> 5] = dq2;
        s_qh2[t >> 5] = qh2;
    }
    __syncthreads();
    dq2 = 0.0;
    qh2 = 0.0;
    for (int w = 0; w < 32; w++) {
        dq2 += s_dq2[w];
        qh2 += s_qh2[w];
    }
    return i8_scan_bound(dq2, qh2, __ldg(a.max_norm), __ldg(a.emax));
}

// one CTA of 1024 threads per query; level 0 also derives E (lk_f32_bound, or lk_i8_bound for the int8 copy)
__global__ void __launch_bounds__(1024) lk_select_kernel(LargeKArgs a, int level) {
    __shared__ unsigned s_warp[32];
    __shared__ int s_digit;
    __shared__ unsigned s_above;
    __shared__ double s_q2[32], s_qh2[32];
    const int qi = blockIdx.x, t = threadIdx.x;
    lk_wait();
    LargeKQuery* st = a.st + qi;
    unsigned prefix = 0u, krem = (unsigned)a.k;
    if (level > 0) {
        if (__ldcg(&st->done)) return;  // CTA-uniform
        prefix = __ldcg(&st->prefix);
        krem = __ldcg(&st->krem);
    }
    if (t == 0) s_digit = -1;
    const float E = level > 0 ? __ldcg(&st->E) : a.xi8 ? lk_i8_bound(a, qi, s_q2, s_qh2) : lk_f32_bound(a, qi, s_q2);
    __syncthreads();
    const bool all = a.all_rows || !(2.f * E <= FLT_MAX);
    if (!all) lk_find_digit(a.hist + ((size_t)level * a.nq_pass + qi) * LK_BINS, krem, s_warp, &s_digit, &s_above);
    if (t != 0) return;
    unsigned cut = 0u, done = 0u;
    if (all || s_digit < 0) {  // special data, no finite bound, or at most k rows: every row is a candidate
        done = 1u;
    } else {
        prefix = (prefix << (level < 2 ? 11 : 10)) | (unsigned)s_digit;
        krem -= s_above;
        if (level == 2) {  // prefix = s_(k): the cut is the key of score(s_(k)) - 2E, rounded down
            done = 1u;
            cut = (unsigned)(key_lowered((u64)prefix << 32, 2.f * E) >> 32);
        }
    }
    if (level == 0) {
        st->ncand = 0u;
        st->best_excl = 0u;
        st->E = E;
    }
    st->prefix = prefix;
    st->krem = krem;
    st->cut = cut;
    st->done = done;
}

// digit histogram of level 1 (bits 20..10) or 2 (bits 9..0) over the keys that share the digits found so far
__global__ void __launch_bounds__(256) lk_hist_kernel(LargeKArgs a, int level) {
    __shared__ unsigned h[LK_BINS];
    const int qi = blockIdx.y;
    for (int i = threadIdx.x; i < LK_BINS; i += blockDim.x) h[i] = 0u;
    lk_wait();
    const LargeKQuery* st = a.st + qi;
    const unsigned done = __ldcg(&st->done), prefix = __ldcg(&st->prefix);
    if (done) return;  // CTA-uniform
    __syncthreads();
    const int hi = level == 1 ? 21 : 10, lo = level == 1 ? 10 : 0;
    const unsigned mask = level == 1 ? 2047u : 1023u;
    const unsigned* S = a.S + (size_t)qi * a.npad;
    const long long nvec = a.npad / 4;
    for (long long v = (long long)blockIdx.x * blockDim.x + threadIdx.x; v < nvec; v += (long long)gridDim.x * blockDim.x) {
        const uint4 w = __ldcg(reinterpret_cast<const uint4*>(S) + v);
        const unsigned key[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (4 * v + j < a.n && (key[j] >> hi) == prefix) atomicAdd(&h[(key[j] >> lo) & mask], 1u);
    }
    __syncthreads();
    lk_flush_hist(h, a.hist + ((size_t)level * a.nq_pass + qi) * LK_BINS, LK_BINS);
}

// ---------------------------------------------------------------------------------------------
// 3. window cut and compaction; the best excluded key (for the margin)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) lk_compact_kernel(LargeKArgs a) {
    const int qi = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    lk_wait();
    LargeKQuery* st = a.st + qi;
    const unsigned cut = __ldcg(&st->cut);
    const unsigned* S = a.S + (size_t)qi * a.npad;
    unsigned* C = a.C + (size_t)qi * a.npad;
    unsigned best = 0u;
    for (long long i0 = ((long long)blockIdx.x * nwarps + warp) * 32; i0 < a.n; i0 += (long long)gridDim.x * nwarps * 32) {
        const long long i = i0 + lane;
        const bool in = i < a.n;
        const unsigned key = in ? __ldcg(S + i) : 0u;
        const bool take = in && key >= cut;
        if (in && !take) best = max(best, key);
        const unsigned m = __ballot_sync(0xffffffffu, take);
        if (m) {
            unsigned pos = 0u;
            if (lane == 0) pos = atomicAdd(&st->ncand, (unsigned)__popc(m));
            pos = __shfl_sync(0xffffffffu, pos, 0);
            if (take) C[pos + __popc(m & ((1u << lane) - 1u))] = (unsigned)i;
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, off));
    if (lane == 0 && best) atomicMax(&st->best_excl, best);
}

// ---------------------------------------------------------------------------------------------
// 4. canonical re-score of C, spread over the grid
// ---------------------------------------------------------------------------------------------
template <bool FAST>
__global__ void __launch_bounds__(256) lk_rescore_kernel(LargeKArgs a) {
    extern __shared__ __align__(16) double qs[];  // [d]
    constexpr int R = 4;
    const int qi = blockIdx.y, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    lk_wait();
    for (int i = threadIdx.x; i < a.d; i += blockDim.x) qs[i] = (double)a.xq[(size_t)qi * a.d + i];
    __syncthreads();
    const long long nc = __ldcg(&a.st[qi].ncand);
    const unsigned* C = a.C + (size_t)qi * a.npad;
    u64* Rk = a.R + (size_t)qi * a.npad;
    for (long long c = ((long long)blockIdx.x * nwarps + warp) * R; c < nc; c += (long long)gridDim.x * nwarps * R) {
        const float* xr[R];
#pragma unroll
        for (int r = 0; r < R; r++) xr[r] = c + r < nc ? a.xb + (size_t)__ldcg(C + c + r) * a.d : nullptr;
        double sv[R];
        canon32_dot_multi<R, FAST>(xr, qs, a.d, lane, sv);
        double mine = sv[0];
#pragma unroll
        for (int r = 1; r < R; r++) mine = lane == r ? sv[r] : mine;
        if (lane < R && c + lane < nc) Rk[c + lane] = isnan(mine) ? 0ull : score_rank_key(mine);  // NaN never enters
    }
}

// ---------------------------------------------------------------------------------------------
// 5. rank and emit: one CTA of 1024 threads per query
// ---------------------------------------------------------------------------------------------
typedef unsigned __int128 u128;
// (canonical desc, row asc) as one unsigned order
__device__ __forceinline__ u128 lk_composite(u64 key, unsigned row) { return ((u128)key << 32) | (u128)(0xFFFFFFFFu - row); }

__global__ void __launch_bounds__(1024) lk_rank_kernel(LargeKArgs a) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    u64* skey = reinterpret_cast<u64*>(smem_raw);                    // [LK_SORT]
    unsigned* srow = reinterpret_cast<unsigned*>(skey + LK_SORT);    // [LK_SORT]
    unsigned* h = srow;                                              // [LK_BINS] digit histogram of the general path
    __shared__ unsigned s_warp[32], s_count, s_above;
    __shared__ int s_digit;
    const int qi = blockIdx.x, t = threadIdx.x, nt = blockDim.x;
    lk_wait();
    const LargeKQuery* st = a.st + qi;
    const long long nc = __ldcg(&st->ncand);
    const unsigned* C = a.C + (size_t)qi * a.npad;
    const u64* Rk = a.R + (size_t)qi * a.npad;
    if (t == 0) s_count = 0u;
    __syncthreads();
    unsigned nv = 0u;
    for (long long j = t; j < nc; j += nt) nv += __ldcg(Rk + j) != 0ull ? 1u : 0u;
    if (nv) atomicAdd(&s_count, nv);
    __syncthreads();
    const unsigned nvalid = s_count;
    __syncthreads();
    // general path (more candidates than one sort holds, so k < nvalid): the k-th best (score, row) pair T by a radix select
    // over the 96-bit composite, 11 bits at a time; the pairs >= T are then exactly the k best
    u128 T = 0;
    if (nvalid > LK_SORT) {
        u128 prefix = 0;
        unsigned krem = (unsigned)a.k;
        for (int consumed = 0; consumed < 96;) {
            const int bits = 96 - consumed < 11 ? 96 - consumed : 11, shift = 96 - consumed - bits;
            for (int b = t; b < LK_BINS; b += nt) h[b] = 0u;
            if (t == 0) s_digit = -1;
            __syncthreads();
            for (long long j = t; j < nc; j += nt) {
                const u64 key = __ldcg(Rk + j);
                if (!key) continue;
                const u128 c = lk_composite(key, __ldcg(C + j));
                if ((c >> (shift + bits)) == prefix) atomicAdd(&h[(unsigned)(c >> shift) & ((1u << bits) - 1u)], 1u);
            }
            __syncthreads();
            lk_find_digit(h, krem, s_warp, &s_digit, &s_above);
            prefix = (prefix << bits) | (u128)(unsigned)s_digit;
            krem -= s_above;
            consumed += bits;
            __syncthreads();
        }
        T = prefix;
    }
    if (t == 0) s_count = 0u;
    __syncthreads();
    for (long long j = t; j < nc; j += nt) {
        const u64 key = __ldcg(Rk + j);
        if (!key) continue;
        const unsigned row = __ldcg(C + j);
        if (lk_composite(key, row) < T) continue;
        const unsigned pos = atomicAdd(&s_count, 1u);
        skey[pos] = key;
        srow[pos] = row;
    }
    __syncthreads();
    const int m = (int)s_count;  // <= LK_SORT: every valid candidate, or exactly k
    int P = 2;
    while (P < m) P <<= 1;
    for (int i = m + t; i < P; i += nt) {
        skey[i] = 0ull;
        srow[i] = 0xFFFFFFFFu;
    }
    for (int size = 2; size <= P; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int e = t; e < (P >> 1); e += nt) {
                const int i = bitonic_low(e, stride), j = i + stride;
                const u64 ki = skey[i], kj = skey[j];
                const unsigned ri = srow[i], rj = srow[j];
                const bool j_better = kj > ki || (kj == ki && rj < ri);
                if (((i & size) == 0) == j_better) {  // descending runs: the better one first
                    skey[i] = kj;
                    skey[j] = ki;
                    srow[i] = rj;
                    srow[j] = ri;
                }
            }
        }
    }
    __syncthreads();
    const int nout = m < a.k ? m : a.k;
    for (int r = t; r < a.k; r += nt) {
        const size_t o = (size_t)qi * a.k + r;
        if (r < nout) {
            const double s = rank_key_score(skey[r]);
            const long long id = (long long)srow[r] + a.id_base;
            if (a.D) {
                a.D[o] = (float)s;
                a.I[o] = id;
            } else {
                a.P_scores[o] = s;
                a.P_ids[o] = id;
            }
        } else if (a.D) {
            a.D[o] = -FLT_MAX;
            a.I[o] = -1;
        } else {
            a.P_scores[o] = -DBL_MAX;
            a.P_ids[o] = -1;
        }
    }
    if (t == 0) {
        // margin: canonical score of rank k minus (best excluded scan score + E); FLT_MAX when no row was excluded
        const unsigned bx = __ldcg(&st->best_excl);
        if (a.margins)
            a.margins[qi] = (nout == a.k && bx != 0u)
                                ? (float)(rank_key_score(skey[a.k - 1]) - (double)ordered_to_score(bx)) - __ldcg(&st->E)
                                : FLT_MAX;
        atomicMax(a.stats, (unsigned)nc);
    }
}

// ---------------------------------------------------------------------------------------------
// host: one pass
// ---------------------------------------------------------------------------------------------
size_t large_k_state_bytes(int qpp) { return (size_t)3 * qpp * LK_BINS * sizeof(unsigned) + (size_t)qpp * sizeof(LargeKQuery); }

template <int NQ, int NV>
static cudaError_t launch_score_nv(const LargeKArgs& a, cudaStream_t st) {
    return launch_pdl(lk_score_kernel<NQ, NV>, dim3((unsigned)a.grid), dim3(256), 0, st, a);
}
template <int NV>
static cudaError_t launch_score_nq(const LargeKArgs& a, cudaStream_t st) {
    switch (a.nq_pass) {
        case 1: return launch_score_nv<1, NV>(a, st);
        case 2: return launch_score_nv<2, NV>(a, st);
        case 3: return launch_score_nv<3, NV>(a, st);
        case 4: return launch_score_nv<4, NV>(a, st);
        default: return cudaErrorInvalidValue;
    }
}

template <int NV>
static cudaError_t i8_kernel_setup(int sm_count, int* grid) {
    static std::atomic<int> occ_dev[16];  // per instantiation and device: CTAs per SM once the attribute is set (0: not yet)
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    int occ = occ_dev[dev & 15].load();
    if (occ == 0) {
        const size_t smem = (size_t)LK_I8_NQ * LK_BINS * sizeof(unsigned);
        e = cudaFuncSetAttribute(lk_score_i8_kernel<LK_I8_NQ, NV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
        if (e == cudaSuccess) e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, lk_score_i8_kernel<LK_I8_NQ, NV>, 256, smem);
        if (e != cudaSuccess) return e;
        if (occ < 1) return cudaErrorInvalidConfiguration;
        occ_dev[dev & 15].store(occ);
    }
    *grid = sm_count * occ;
    return cudaSuccess;
}
int i8_batch_grid(int nv, int sm_count) {
    int grid = 0;
    cudaError_t e;
    switch (nv) {
        case 1: e = i8_kernel_setup<1>(sm_count, &grid); break;
        case 2: e = i8_kernel_setup<2>(sm_count, &grid); break;
        case 3: e = i8_kernel_setup<3>(sm_count, &grid); break;
        case 4: e = i8_kernel_setup<4>(sm_count, &grid); break;
        default: e = cudaErrorInvalidValue;
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return grid;
}
static cudaError_t launch_score_i8(const LargeKArgs& a, cudaStream_t st) {
    const size_t smem = (size_t)LK_I8_NQ * LK_BINS * sizeof(unsigned);
    const dim3 grid((unsigned)a.grid), block(256);
    switch (a.nv) {
        case 1: return launch_pdl(lk_score_i8_kernel<LK_I8_NQ, 1>, grid, block, smem, st, a);
        case 2: return launch_pdl(lk_score_i8_kernel<LK_I8_NQ, 2>, grid, block, smem, st, a);
        case 3: return launch_pdl(lk_score_i8_kernel<LK_I8_NQ, 3>, grid, block, smem, st, a);
        case 4: return launch_pdl(lk_score_i8_kernel<LK_I8_NQ, 4>, grid, block, smem, st, a);
        default: return cudaErrorInvalidValue;
    }
}

cudaError_t launch_large_k_scan(const LargeKArgs& a, cudaStream_t st) {
    if (a.xi8) {  // up to LK_I8_NQ queries, a.grid from i8_batch_grid
        if (a.n <= 0 || a.nq_pass < 1 || a.nq_pass > LK_I8_NQ || a.grid < 1) return cudaErrorInvalidValue;
        const cudaError_t e = launch_score_i8(a, st);
        g_kernel_launches.fetch_add(1);
        if (e != cudaSuccess) return e;
        return cudaGetLastError();
    }
    if (a.n <= 0 || a.nq_pass < 1 || a.nq_pass > 4) return cudaErrorInvalidValue;
    cudaError_t e;
    switch (a.nv) {
        case 0: e = launch_pdl(lk_score_generic_kernel, dim3((unsigned)a.grid, (unsigned)a.nq_pass), dim3(256), 0, st, a); break;
        case 1: e = launch_score_nq<1>(a, st); break;
        case 2: e = launch_score_nq<2>(a, st); break;
        case 3: e = launch_score_nq<3>(a, st); break;
        case 4: e = launch_score_nq<4>(a, st); break;
        case 6: e = launch_score_nq<6>(a, st); break;
        case 8: e = launch_score_nq<8>(a, st); break;
        default: return cudaErrorInvalidValue;
    }
    g_kernel_launches.fetch_add(1);
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

cudaError_t launch_large_k_rest(const LargeKArgs& a, int sm_count, cudaStream_t st) {
    const unsigned nq = (unsigned)a.nq_pass;
    const long long per_q = (long long)sm_count * 2 / a.nq_pass;
    const long long want = (a.npad / 4 + 255) / 256;
    const unsigned gx = (unsigned)(want < per_q ? (want < 1 ? 1 : want) : (per_q < 1 ? 1 : per_q));
    const size_t qs_bytes = (size_t)a.d * sizeof(double);
    const size_t rank_bytes = (size_t)LK_SORT * (sizeof(u64) + sizeof(unsigned));
    static size_t optin_rescore[2][16] = {};
    static size_t optin_rank[16] = {};
    cudaError_t e = ensure_smem_optin(lk_rescore_kernel<true>, qs_bytes, optin_rescore[1]);
    if (e == cudaSuccess) e = ensure_smem_optin(lk_rescore_kernel<false>, qs_bytes, optin_rescore[0]);
    // (+ 1 KB: the kernel's static shared words count against the same limit, and 48 KB of dynamic memory alone is at it)
    if (e == cudaSuccess) e = ensure_smem_optin(lk_rank_kernel, rank_bytes + 1024, optin_rank);
    if (e != cudaSuccess) return e;
    auto step = [&](cudaError_t le) {
        g_kernel_launches.fetch_add(1);
        if (e == cudaSuccess) e = le;
    };
    step(launch_pdl(lk_select_kernel, dim3(nq), dim3(1024), 0, st, a, 0));
    for (int level = 1; level <= 2 && e == cudaSuccess; level++) {
        step(launch_pdl(lk_hist_kernel, dim3(gx, nq), dim3(256), 0, st, a, level));
        if (e == cudaSuccess) step(launch_pdl(lk_select_kernel, dim3(nq), dim3(1024), 0, st, a, level));
    }
    if (e == cudaSuccess) step(launch_pdl(lk_compact_kernel, dim3(gx, nq), dim3(256), 0, st, a));
    if (e == cudaSuccess) {
        const unsigned gr = (unsigned)(per_q * 2 < 1 ? 1 : per_q * 2);
        step(a.fast_widen ? launch_pdl(lk_rescore_kernel<true>, dim3(gr, nq), dim3(256), qs_bytes, st, a)
                          : launch_pdl(lk_rescore_kernel<false>, dim3(gr, nq), dim3(256), qs_bytes, st, a));
    }
    if (e == cudaSuccess) step(launch_pdl(lk_rank_kernel, dim3(nq), dim3(1024), rank_bytes, st, a));
    if (e != cudaSuccess) return e;
    return cudaGetLastError();
}

}  // namespace evs
