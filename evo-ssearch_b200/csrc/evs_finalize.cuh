// evs_finalize.cuh -- the per-query finalise step as a device function.
//
// Input: L candidate lists of one query (kp keys each, sorted descending, 0 = empty) as the scans write them.
// Work:  pick the kp best keys of the union, re-score them in the canonical fp64 order (CANON-32, DESIGN.md section 2),
//        rank by (score desc, id asc), emit the k best as final (D, I), as a shard partial, or straight into every
//        rank's exchange slot over NVLink; compute the safety margin and decide whether the result is certified.
// Callers: finalize_kernel (one CTA per query, evs_kernels.cu) and -- for single-query searches -- the LAST CTA of
//        the GEMV scan itself (evs_scan.cuh, ticket counter), which removes a launch from the latency path of
//        index.search(q.reshape(1,-1), k) (/root/reference/oldapp.py:2005, :2112).
#pragma once
#include <float.h>
#include <limits.h>

#include <type_traits>

#include "evs_common.cuh"
#include "evs_internal.h"

namespace evs {

__device__ __forceinline__ void st_release_sys_u64(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

// The canonical order on integers (DSETP is quarter-rate on B200, and short-circuit logic branches):
// map the score to an order-preserving u64 (-0.0 folded onto +0.0 so that equal doubles stay equal).
__device__ __forceinline__ u64 score_rank_key(double s) { return f64_to_ordered(s == 0.0 ? 0.0 : s); }
__device__ __forceinline__ int better_i(u64 oa, long long ia, u64 ob, long long ib) {
    return (int)(oa > ob) | ((int)(oa == ob) & (int)(ia < ib));
}

// ---- merge of sorted shard partials (one query; merge_partials_kernel, exchange_merge) ----
// Every part holds the shard's k best sorted by (score desc, id asc), padding (id < 0) at the end.  `at(part, j)` returns
// entry j of a part (key = score_rank_key(score); any value for padding), so one body serves the entries staged in shared
// memory, the [part][nq][k] partials in global memory and the flagged exchange entries.
struct PartEntry {
    double score;
    u64 key;
    long long id;
};
// Rank in the merged order of entry (part, r), whose rank key and id are (key, id): r plus, for every other part, the
// number of its entries that beat it -- a binary search in which padding never beats (it sits at the end).  Asked with
// key 0 and id LLONG_MAX, a padding entry ranks behind every real one.
template <class At>
__device__ __forceinline__ int merge_rank(const At& at, int nparts, int k, int part, int r, u64 key, long long id) {
    int rank = r;
    for (int pp = 0; pp < nparts; pp++) {
        if (pp == part) continue;
        int lo = 0, hi = k;  // first position in part pp that does not beat (part, r)
        while (lo < hi) {
            const int mid = (lo + hi) >> 1;
            const PartEntry o = at(pp, mid);
            if (o.id >= 0 && better_i(o.key, o.id, key, id)) lo = mid + 1;
            else hi = mid;
        }
        rank += lo;
    }
    return rank;
}
// The merge of one query by one CTA: every real entry is written to its rank in D[0..k) / I[0..k) (the query's row) and
// counted in *nvalid (a shared int, 0 before), then the slots [nvalid, k) are padded.  Called by all threads of the CTA.
template <class At>
__device__ __forceinline__ void merge_query(const At& at, int nparts, int k, float* __restrict__ D, long long* __restrict__ I,
                                            int* nvalid) {
    for (int e = threadIdx.x; e < nparts * k; e += blockDim.x) {
        const int part = e / k, r = e - part * k;
        const PartEntry t = at(part, r);
        if (t.id < 0) continue;
        atomicAdd(nvalid, 1);
        const int rank = merge_rank(at, nparts, k, part, r, t.key, t.id);
        if (rank < k) {
            D[rank] = (float)at(part, r).score;
            I[rank] = t.id;
        }
    }
    __syncthreads();
    for (int r = *nvalid + threadIdx.x; r < k; r += blockDim.x) {
        D[r] = -FLT_MAX;
        I[r] = -1;
    }
}
// The entries of `nparts` parts staged in shared memory: score[m] | id[m] | key[m], m = nparts * k (24 bytes an entry).
struct StagedParts {
    double* sc;
    long long* id;
    u64* key;
    int k;
    __device__ StagedParts(unsigned char* smem, int nparts, int k_) : k(k_) {
        const int m = nparts * k;
        sc = reinterpret_cast<double*>(smem);
        id = reinterpret_cast<long long*>(sc + m);
        key = reinterpret_cast<u64*>(id + m);
    }
    __device__ void put(int e, double s, long long i) const {
        sc[e] = s;
        id[e] = i;
        key[e] = score_rank_key(s);
    }
    __device__ PartEntry operator()(int part, int j) const {
        const int e = part * k + j;
        return {sc[e], key[e], id[e]};
    }
};
// exact fp32 -> fp64 widening with integer ops for normal numbers (F2F.F64.F32 issues at 1/8 rate)
__device__ __forceinline__ double widen_f32(float f) {
    const uint32_t u = __float_as_uint(f);
    const uint32_t e = (u >> 23) & 0xFFu;
    if (e == 0u || e == 255u) return (double)f;  // zero, subnormal, inf, nan: the slow exact path
    const uint32_t hi = (u & 0x80000000u) | ((e + 896u) << 20) | ((u & 0x007FFFFFu) >> 3);
    const uint32_t lo = u << 29;
    return __hiloint2double((int)hi, (int)lo);
}

__device__ __forceinline__ double canon32_dot_bf16(const __nv_bfloat16* __restrict__ x, const double* __restrict__ q,
                                                   int d, int lane) {
    double acc = 0.0;
    const unsigned short* xs = reinterpret_cast<const unsigned short*>(x);
    for (int i = lane; i < d; i += 32) acc = fma((double)__uint_as_float(((uint32_t)xs[i]) << 16), q[i], acc);
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) acc = acc + __shfl_xor_sync(0xffffffffu, acc, off);
    return acc;
}

// fp32 -> fp64, exact for zero and normal numbers, branch-free (5 + 2 integer instructions).  F2F.F64.F32 is very slow on
// B200: re-scoring 64 rows of 512 values through it took 32 us instead of 10 (scripts/scan_tail_probe.py); the general
// widen_f32 above pays ~19 instructions for its special-case branch.  Used when the index is known to hold no subnormal,
// infinite or NaN element (row_norm_max_kernel records that at add time).
__device__ __forceinline__ double widen_f32_normal(float f) {
    const uint32_t u = __float_as_uint(f);
    const uint32_t t = u & 0x7FFFFFFFu;
    uint32_t hi = (t >> 3) + 0x38000000u;
    hi = t ? hi : 0u;
    return __hiloint2double((int)(hi | (u & 0x80000000u)), (int)(u << 29));
}

// CANON-32 of R rows at once with the row loads batched (the same accumulation order per row; the rows' load latencies
// and fp64 chains overlap).  A null row pointer yields -DBL_MAX.
template <int R, bool FAST, int UW = 0>
__device__ __forceinline__ void canon32_dot_multi(const float* const (&x)[R], const double* __restrict__ qs, int d, int lane,
                                                  double (&res)[R]) {
    double acc[R];
#pragma unroll
    for (int r = 0; r < R; r++) acc[r] = 0.0;
    // values per row held at a time: R * U loads in flight per lane (UW: a kernel with registers to spare asks for more; the
    // order of a lane's additions does not depend on it)
    constexpr int U = UW > 0 ? UW : (R <= 2 ? 16 : 8);
    for (int base = 0; base < d; base += 32 * U) {
        float v[R][U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int i = base + lane + 32 * u;
#pragma unroll
            for (int r = 0; r < R; r++) v[r][u] = (x[r] && i < d) ? __ldg(x[r] + i) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int i = base + lane + 32 * u;
            if (i < d) {
                const double qv = qs[i];
#pragma unroll
                for (int r = 0; r < R; r++) acc[r] = fma(FAST ? widen_f32_normal(v[r][u]) : widen_f32(v[r][u]), qv, acc[r]);
            }
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
        for (int r = 0; r < R; r++) acc[r] = acc[r] + __shfl_xor_sync(0xffffffffu, acc[r], off);
    }
#pragma unroll
    for (int r = 0; r < R; r++) res[r] = x[r] ? acc[r] : -DBL_MAX;
}

// Canonical re-score of the candidates keys[0..n) (0 = empty slot): slot c gets its canonical score sc[c], row id[c] (-1 when
// empty) and rank key ok[c] (0 when empty).  A warp takes R candidates at a time with U values per row and lane in flight
// (canon32_dot_multi: the order of a lane's additions, hence every score's bits, depend on neither).  Called by every
// thread of the CTA; the slots are visible after the next barrier.
template <int R, int UW = 0>
__device__ __forceinline__ void canon_rescore(const FinalizeParams& p, const u64* keys, int n, double* sc, long long* id, u64* ok,
                                              const double* qs) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    const float* xb32 = reinterpret_cast<const float*>(p.xb);
    auto run = [&](auto ftag) {
        constexpr bool FAST = decltype(ftag)::value;
        for (int c = R * warp; c < n; c += R * nwarps) {
            u64 key[R];
            long long row[R];
            const float* xr[R];
            double sv[R];
#pragma unroll
            for (int r = 0; r < R; r++) {
                key[r] = (c + r < n) ? keys[c + r] : 0ull;
                row[r] = key[r] ? (long long)key_row(key[r]) : -1;
                xr[r] = (key[r] && !p.xb_is_bf16) ? xb32 + (size_t)row[r] * p.d : nullptr;
            }
            canon32_dot_multi<R, FAST, UW>(xr, qs, p.d, lane, sv);
            if (p.xb_is_bf16) {
                const __nv_bfloat16* xb16 = reinterpret_cast<const __nv_bfloat16*>(p.xb);
#pragma unroll
                for (int r = 0; r < R; r++) sv[r] = key[r] ? canon32_dot_bf16(xb16 + (size_t)row[r] * p.d, qs, p.d, lane) : -DBL_MAX;
            }
            if (lane == 0) {
#pragma unroll
                for (int r = 0; r < R; r++)
                    if (c + r < n) {
                        sc[c + r] = sv[r];
                        id[c + r] = row[r];
                        ok[c + r] = row[r] >= 0 ? score_rank_key(sv[r]) : 0ull;
                    }
            }
        }
    };
    if (p.special != nullptr && __ldg(p.special) == 0u) run(std::true_type{});  // CTA-uniform
    else run(std::false_type{});
}

// The L per-CTA lists are sorted, so the global top-kp is found without merging them all:
//   T0 = kp-th largest list HEAD is a lower bound of the kp-th best key (kp heads are >= it), only the
//   <= kp lists whose head is >= T0 can hold survivors, and only their prefix >= T0 does.  The
//   survivors (about kp + a few for unordered data, kp*kp at most) are sorted in shared memory.
// Latency shape (the single-query search runs this in ONE 256-thread CTA at the end of the scan kernel):
//   * one round of independent loads brings the first two keys (16 bytes) of EVERY list: the heads for T0 and, for
//     unordered data, almost all survivors (a list contributes 0.2 keys on average); only lists whose second key also
//     survives are read in full ("deep" lists, a warp each, all loads of a list in flight together);
//   * the rows of the survivors are prefetched into L2 while they are being ranked, so that the canonical re-score
//     (two candidates per warp at a time) waits on L2, not on HBM.
// shared memory (finalize_smem_bytes): FinalizeShared | surv[finalize_surv_slots(L, kp)] u64 | pre[2 L] u64 | deep[L] int
//   (padded to 8 bytes) | sc[kp] f64 | id[kp] i64 | ok[kp] u64 | qs[d] f64
// (survivor capacity scap = min(L, kp) * kp: with one list per query -- the tensor-core scans -- the kernel needs
// 7 KB instead of 38 KB of shared memory and eight 256-thread CTAs fit an SM)
__host__ __device__ inline int finalize_surv_cap(int L, int kp) { return (L < kp ? L : kp) * kp; }
__host__ __device__ inline int finalize_surv_slots(int L, int kp) {
    const int scap = finalize_surv_cap(L, kp);
    int pow2 = kp;
    while (pow2 < scap) pow2 <<= 1;  // the sort path pads the survivors to a power of two
    return pow2 > scap + kp ? pow2 : scap + kp;  // the counting path puts kp result slots behind the survivors
}
struct FinalizeShared {
    int nsurv, nvalid;
    unsigned maxerr;  // ordered-uint of the largest (canonical - scan) score difference among the candidates
    int ndeep;
    u64 T0;
    double qnorm2;    // |q|^2
    int fail;         // fused exchange merge: 1 = a rank never arrived, 2 = a rank reported failure
    int uncert;       // the result did not clear the scan's error bound (set by the thread that ranks k-th)
};
__host__ __device__ inline size_t finalize_deep_slots(int L) { return (size_t)((L + 1) / 2); }  // ints, in 8-byte units
__host__ __device__ inline size_t finalize_smem_bytes(int L, int kp, int d) {
    return sizeof(FinalizeShared) + ((size_t)finalize_surv_slots(L, kp) + 2 * (size_t)L + finalize_deep_slots(L) + 3 * (size_t)kp + (size_t)d) * 8;
}

// the part that does not depend on the scan's output: the query widened to fp64 (may run before griddepcontrol.wait)
__device__ __forceinline__ void finalize_prologue_at(const FinalizeParams& p, long long qi, FinalizeShared* sh, double* qs) {
    const int t = threadIdx.x, nt = blockDim.x;
    const float* q = p.xq + (size_t)qi * p.d;
    for (int i = t; i < p.d; i += nt) qs[i] = (double)q[i];
    if (t == 0) {
        sh->nsurv = 0;
        sh->nvalid = 0;
        sh->maxerr = 0u;
        sh->ndeep = 0;
        sh->T0 = 0ull;
        sh->qnorm2 = 0.0;
        sh->fail = 0;
        sh->uncert = 0;
    }
}
__device__ __forceinline__ void finalize_prologue(const FinalizeParams& p, long long qi, unsigned char* smem_raw) {
    FinalizeShared* sh = reinterpret_cast<FinalizeShared*>(smem_raw);
    double* qs = reinterpret_cast<double*>(smem_raw + sizeof(FinalizeShared) +
                                           ((size_t)finalize_surv_slots(p.L, p.kp) + 2 * (size_t)p.L + finalize_deep_slots(p.L) + 3 * (size_t)p.kp) * 8);
    finalize_prologue_at(p, qi, sh, qs);
}

// |q|^2 for the certification bound, by warp 0 (qs complete and visible: call after a barrier; visible after the next one)
__device__ __forceinline__ void finalize_qnorm2(const FinalizeParams& p, FinalizeShared* sh, const double* qs) {
    if (p.err_coef > 0.f && (threadIdx.x >> 5) == 0) {
        const int lane = threadIdx.x & 31;
        double s2 = 0.0;
        for (int i = lane; i < p.d; i += 32) s2 = fma(qs[i], qs[i], s2);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        if (lane == 0) sh->qnorm2 = s2;
    }
}

__device__ __forceinline__ void fin_stamp(const FinalizeParams& p, int slot) {
    if (p.dbg != nullptr && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        p.dbg[slot] = t;
    }
}
// a count beside the stamps (slots 11-13: the int8 window pass)
__device__ __forceinline__ void fin_note(const FinalizeParams& p, int slot, unsigned long long v) {
    if (p.dbg != nullptr && threadIdx.x == 0) p.dbg[slot] = v;
}

// ---- exchange entries (evs_internal.h: Exchange): payload and flag in the same 16-byte stores ----
__device__ __forceinline__ uint32_t exchange_flag(unsigned long long seq) { return (uint32_t)(seq & 0x7FFFFFFFull); }
__device__ __forceinline__ void st_volatile_v4(void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(p), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ld_volatile_v4(const void* p) {
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "l"(p) : "memory");
    return v;
}
// store one (score, id) entry of this shard's partial into slot `x.rank` of EVERY rank's buffer over NVLink (peer stores)
__device__ __forceinline__ void exchange_store_entry(const Exchange& x, size_t e, double score, long long id, uint32_t flag) {
    const unsigned long long sb = (unsigned long long)__double_as_longlong(score), ib = (unsigned long long)id;
    for (int g = 0; g < x.world; g++) {
        unsigned char* ent = x.peer[g] + ((size_t)x.parity * x.world + x.rank) * x.slot_bytes + e * kExchangeEntryBytes;
        st_volatile_v4(ent, (uint32_t)sb, flag, (uint32_t)(sb >> 32), flag);
        st_volatile_v4(ent + 16, (uint32_t)ib, flag, (uint32_t)(ib >> 32), flag);
    }
}

// entry (part, r) of query qi in the LOCAL gather buffer, and its payload
__device__ __forceinline__ const unsigned char* exchange_entry(const Exchange& x, long long qi, int k, int part, int r) {
    return x.peer[x.rank] + ((size_t)x.parity * x.world + part) * x.slot_bytes + ((size_t)qi * k + r) * kExchangeEntryBytes;
}
__device__ __forceinline__ PartEntry exchange_decode(uint4 a, uint4 b) {
    const double s = __longlong_as_double((long long)(((unsigned long long)a.z << 32) | a.x));
    return {s, score_rank_key(s), (long long)(((unsigned long long)b.z << 32) | b.x)};
}
// Poll entry (part, r) of query qi until it carries the flag of search x.seq and return its payload in *v.  False when the
// merge must not happen: that rank reported failure (poisoned flag; *fail raised to 2), it never arrived (~10 s watchdog;
// *fail raised to 1), or another thread of the CTA already gave up.  `fail` is a shared int of the CTA, 0 before.
__device__ __forceinline__ bool exchange_wait_entry(const Exchange& x, long long qi, int k, int part, int r, int* fail, PartEntry* v) {
    const unsigned char* ent = exchange_entry(x, qi, k, part, r);
    const uint32_t want = exchange_flag(x.seq);
    const long long t0 = clock64();
    for (;;) {
        const uint4 a = ld_volatile_v4(ent), b = ld_volatile_v4(ent + 16);
        if (a.y == want && a.w == want && b.y == want && b.w == want) {
            *v = exchange_decode(a, b);
            return true;
        }
        if (a.y == (want | kExchangePoison) || b.y == (want | kExchangePoison)) {
            atomicMax(fail, 2);
            return false;
        }
        if (*reinterpret_cast<volatile int*>(fail)) return false;
        if (clock64() - t0 > 20000000000ll) {
            atomicMax(fail, 1);
            return false;
        }
        __nanosleep(20);
    }
}
// The result of a merge that did not get every rank's partial: padding in the query's row D[0..k) / I[0..k), and the
// failure code in *x.status (host-mapped).  Never a merge of what sits in the slots: it may be an older search's partial.
__device__ __forceinline__ void exchange_fail_result(const Exchange& x, int k, int fail, float* __restrict__ D, long long* __restrict__ I) {
    for (int r = threadIdx.x; r < k; r += blockDim.x) {
        D[r] = -FLT_MAX;
        I[r] = -1;
    }
    if (threadIdx.x == 0 && x.status) {
        *reinterpret_cast<volatile int*>(x.status) = fail;
        __threadfence_system();
    }
}

// Merge after the peer-store exchange: wait for the world*k entries of query `qi` in the local gather buffer, then rank them
// into (D, I) with merge_query.  STAGED: the entries are copied to smem_raw (world*k*24 bytes) as they arrive, which
// k <= EVS_MAX_K always fits; otherwise they are ranked where they lie.  Called by all threads of the CTA; `fail` / `nvalid`
// are shared ints set to 0 before.
template <bool STAGED>
__device__ __forceinline__ void exchange_merge(const Exchange& x, long long qi, int k, float* __restrict__ D, long long* __restrict__ I,
                                               unsigned char* smem_raw, int* fail, int* nvalid) {
    const int m = x.world * k;
    const StagedParts staged(smem_raw, x.world, k);
    for (int e = threadIdx.x; e < m; e += blockDim.x) {
        PartEntry v;
        if (exchange_wait_entry(x, qi, k, e / k, e % k, fail, &v) && STAGED) staged.put(e, v.score, v.id);
    }
    __syncthreads();
    D += (size_t)qi * k;
    I += (size_t)qi * k;
    if (*fail) {  // CTA-uniform
        exchange_fail_result(x, k, *fail, D, I);
        return;
    }
    const auto in_place = [&](int part, int j) {
        const unsigned char* ent = exchange_entry(x, qi, k, part, j);
        return exchange_decode(ld_volatile_v4(ent), ld_volatile_v4(ent + 16));
    };
    if (STAGED) merge_query(staged, x.world, k, D, I, nvalid);
    else merge_query(in_place, x.world, k, D, I, nvalid);
}

// Second half of the finalise, shared by every candidate source (per-CTA lists: finalize_query; the survivor pool of the
// single-query scan: evs_scan.cuh).  A[0..kp) = the kp best scan keys in descending order (0 = empty); every row outside A
// has a smaller scan key.  Canonical re-score, ranking, output (final / shard partial / peer stores + fused merge), margin
// and certification.  Called by every thread of the CTA; `scratch` holds at least max(world * k * 24 + 8, 0) bytes that
// no longer hold anything needed (the exchange merge ranks the gathered partials there).
// shadow_E > 0 (the pool kernel over bf16 rows, evs_scan.cuh): A holds EVERY row whose scan key is >= cut (1: every row),
// unsorted, and every other row's scan score is below key_score(cut); the result is exact by construction and the margin is
// the canonical score of rank k minus (that scan score + E).  scored: sc / id / ok already hold the canonical re-score of
// A[0..kp_use) (canon_rescore), which is not repeated.
template <int MAXR = 4, int UW = 0>  // candidates a warp re-scores at a time at most (kernels held to 64 registers pass 2)
__device__ __forceinline__ void finalize_rank_emit(const FinalizeParams& p, long long qi, const u64* A, FinalizeShared* sh, double* sc,
                                                   long long* id, u64* ok, const double* qs, unsigned char* scratch, int kp_use = 0,
                                                   float shadow_E = 0.f, u64 cut = 0ull, bool scored = false) {
    const int t = threadIdx.x, nt = blockDim.x;
    const int nwarps = nt >> 5;
    const int kp = kp_use > 0 ? kp_use : p.kp;  // kp_use: only the best kp_use (<= p.kp) entries of A are candidates
    // 4. canonical re-score of the kp candidates: a warp takes two candidates at a time, or four when the CTA has fewer than
    //    kp / 2 warps (the 256-thread CTA of the single-query scan: two rounds instead of four)
    if (!scored) {
        if (MAXR < 4 || 2 * nwarps >= kp) canon_rescore<2, UW>(p, A, kp, sc, id, ok, qs);
        else canon_rescore<MAXR < 4 ? 2 : 4, UW>(p, A, kp, sc, id, ok, qs);
    }
    __syncthreads();
    fin_stamp(p, 3);  // re-scored
    // how far the scan under-estimated its own candidates at most (tf32 truncates towards zero: a bias of ~1e-3 relative;
    // bf16 and fp32 scans scatter around zero)
    const bool want_margin = p.margins != nullptr || p.guard_count != nullptr || p.pred_slot != nullptr;
    for (int c = t; c < kp; c += nt)
        if (id[c] >= 0 && want_margin) atomicMax(&sh->maxerr, score_to_ordered((float)(sc[c] - widen_f32(key_score(A[c])))));
    __syncthreads();

    // 5. rank by counting under (score desc, id asc); ids are unique so ranks are a permutation
    for (int c = t; c < kp; c += nt) {
        if (id[c] < 0) continue;
        atomicAdd(&sh->nvalid, 1);
        const double st = sc[c];
        const long long it = id[c];
        const u64 ot = ok[c];
        int rank = 0;
        // empty slots have id -1 and key 0: a real candidate never loses to them -> mask by id >= 0 arithmetically
        for (int j = 0; j < kp; j++) rank += better_i(ok[j], id[j], ot, it) & (int)(id[j] >= 0);
        if (rank < p.k) {
            if (p.D) {
                p.D[(size_t)qi * p.k + rank] = (float)st;
                p.I[(size_t)qi * p.k + rank] = it + p.id_base;
            } else if (p.x.world > 0) {  // the same entry to every rank's slot for this shard
                exchange_store_entry(p.x, (size_t)(p.x.q_off + qi) * p.k + rank, st, it + p.id_base, exchange_flag(p.x.seq));
            } else {
                p.P_scores[(size_t)qi * p.k + rank] = st;
                p.P_ids[(size_t)qi * p.k + rank] = it + p.id_base;
            }
            if (rank == p.k - 1 && want_margin && shadow_E > 0.f) {
                if (p.margins) p.margins[qi] = cut > 1ull ? (float)(st - widen_f32(key_score(cut))) - shadow_E : INFINITY;
            } else if (rank == p.k - 1 && want_margin) {
                // All kp slots taken -> every row outside the list has a scan score <= the worst retained one, so its
                // true score is at most that plus the scan's error.  margin = canonical score of rank k minus (worst
                // retained scan score + the largest under-estimate observed on the retained candidates); the result is
                // CERTIFIED exact when it clears the error bound of the scan that produced the lists (below).
                const float worst = key_score(A[kp - 1]);
                const float under = fmaxf(ordered_to_score(sh->maxerr), 0.f);
                const float gap = (A[kp - 1] != 0ull) ? (float)(st - widen_f32(worst)) : INFINITY;
                const float margin = gap - under;
                if (p.margins) p.margins[qi] = margin;
                if (p.err_coef > 0.f) {
                    const float mx = p.max_norm ? *p.max_norm : 1.f;
                    const float B = sqrtf((float)sh->qnorm2) * 1.000001f * mx;  // >= sum |x_i q_i| of any row (Cauchy-Schwarz); fp32 sqrt, inflated
                    // Symmetric scan error (fp32 GEMV, 3xTF32): |scan - true| <= err_coef * B.
                    // Truncating scan (single tf32: both operands lose their low 13 mantissa bits, towards zero): every product
                    // shrinks by a factor in (1 - 2^-9, 1], so a row is UNDER-estimated by at most 2^-9 * (sum of its positive
                    // products) <= 2^-10 * (B + true score): a row the scan dropped (scan score <= w) has a true score
                    // <= w + err_trunc * (B + |w|) + accumulation error.  A bound, not a statistic.
                    const bool certified = p.err_trunc > 0.f ? gap > p.err_trunc * (B + fabsf(worst)) + p.err_coef * B  // false for NaN
                                                             : margin > p.err_coef * B;
                    if (!certified) sh->uncert = 1;  // acted on by thread 0 below (after the barrier)
                }
            }
        }
    }
    __syncthreads();
    fin_stamp(p, 7);  // ranked
    // 6. padding (-FLT_MAX,-1) / (-DBL_MAX,-1) for the slots no candidate ranked into
    const int nvalid = sh->nvalid;
    for (int r = nvalid + t; r < p.k; r += nt) {
        if (p.D) {
            p.D[(size_t)qi * p.k + r] = -FLT_MAX;
            p.I[(size_t)qi * p.k + r] = -1;
        } else if (p.x.world > 0) {
            exchange_store_entry(p.x, (size_t)(p.x.q_off + qi) * p.k + r, -DBL_MAX, -1, exchange_flag(p.x.seq));
        } else {
            p.P_scores[(size_t)qi * p.k + r] = -DBL_MAX;
            p.P_ids[(size_t)qi * p.k + r] = -1;
        }
    }
    if (t == 0 && p.margins && nvalid < p.k) p.margins[qi] = INFINITY;  // every row was a candidate
    if (t == 0) {
        // the guard: a result that did not clear its scan's error bound, or whose candidate buffers overflowed in the
        // threshold scan, is queued for the exact re-run (first phase), flagged for the host (guard_cap = 0), or counted
        const bool over = p.overflow != nullptr && p.overflow[qi] != 0;
        if (sh->uncert || over) {
            if (p.guard_count) {
                const int slot = atomicAdd(p.guard_count, 1);
                if (slot < p.guard_cap) {
                    p.guard_slot[qi] = slot;
                    p.guard_q[slot] = (int)qi;
                } else {
                    p.guard_slot[qi] = -2;  // flagged only: the host re-runs it (guard_cap = 0), or the queue is full
                    if (p.guard_cap > 0 && p.uncertified) atomicAdd(p.uncertified, 1ull);
                }
            } else if (p.uncertified) {  // second phase (or no re-run available): best effort, counted
                atomicAdd(p.uncertified, 1ull);
            }
        }
    }
    fin_stamp(p, 4);  // ranked, results written
    if (p.x.world > 0 && p.D == nullptr) {
        // nothing to publish: every entry carries its own flag.  (The fenced protocol -- slot stores, one system fence, a
        // done-counter and a flag per rank -- cost 32 us per search at 8 ranks.)
        if (t == 0) sh->nvalid = 0;
        if (p.x.merge_D != nullptr) {
            // single-query search fused into the scan kernel: the same CTA waits for the peers' partials and merges
            __syncthreads();
            exchange_merge<true>(p.x, p.x.q_off + qi, p.k, p.x.merge_D, p.x.merge_I, scratch, &sh->fail, &sh->nvalid);
        }
    }
}



// Finalise query `qi` (index into xq / the outputs) from the lists at `lists` ([L][kp]).  Called by every thread of the
// CTA (a multiple of 32 threads, at least 64) after finalize_prologue and a point where the lists are visible.
__device__ __forceinline__ void finalize_query(const FinalizeParams& p, long long qi, const u64* __restrict__ lists,
                                               unsigned char* smem_raw) {
    const int t = threadIdx.x, nt = blockDim.x;
    const int warp = t >> 5, lane = t & 31, nwarps = nt >> 5;
    const int kp = p.kp, L = p.L;
    const int scap = finalize_surv_cap(L, kp);
    FinalizeShared* sh = reinterpret_cast<FinalizeShared*>(smem_raw);
    u64* surv = reinterpret_cast<u64*>(smem_raw + sizeof(FinalizeShared));  // [finalize_surv_slots(L, kp)]
    u64* pre = surv + finalize_surv_slots(L, kp);           // [L][2]: the first two keys of every list
    int* deep = reinterpret_cast<int*>(pre + 2 * (size_t)L);  // [L]: lists that must be read in full
    double* sc = reinterpret_cast<double*>(pre + 2 * (size_t)L + finalize_deep_slots(L));  // [kp]
    long long* id = reinterpret_cast<long long*>(sc + kp);  // [kp]
    u64* ok = reinterpret_cast<u64*>(id + kp);              // [kp] integer rank keys of the scores
    double* qs = reinterpret_cast<double*>(ok + kp);        // [d] the query widened once

    // 0. the first two keys of every list, all loads independent.  Lists were written by other SMs (possibly during this
    //    very kernel): read them past L1.
    for (int l = t; l < L; l += nt) {
        const ulonglong2 v = __ldcg(reinterpret_cast<const ulonglong2*>(lists + (size_t)l * kp));
        pre[2 * l] = v.x;
        pre[2 * l + 1] = v.y;
    }
    if (qi == 0 && t == 0 && p.guard_count_next) *p.guard_count_next = 0;  // ready for the next guarded search of this handle
    __syncthreads();
    fin_stamp(p, 0);  // head blocks loaded
    if (p.err_coef > 0.f && warp == 0) {  // |q|^2 for the certification bound (qs is complete: barrier above)
        double s2 = 0.0;
        for (int i = lane; i < p.d; i += 32) s2 = fma(qs[i], qs[i], s2);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        if (lane == 0) sh->qnorm2 = s2;
    }
    // 1. T0 = kp-th largest head (non-empty keys are unique, so exactly one head has rank kp-1).
    //    `nper` adjacent lanes share one head and split the comparison range.
    //    Only every `hs`-th head is ranked (about 2.3*kp of them): still a valid bound (kp keys are >= it),
    //    a quarter of the comparisons, a few more survivors.  If the survivors then overflow their
    //    buffer the bound is recomputed from every head (then at most kp lists qualify: <= kp*kp keys).
    int hs = 1;
    while ((L / (hs * 2)) * 10 >= kp * 23) hs <<= 1;
    for (int attempt = 0; attempt < 2; attempt++) {
        if (attempt == 1) {
            if (sh->nsurv <= scap || hs == 1) break;  // uniform: read after the barrier below
            __syncthreads();
            if (t == 0) {
                sh->nsurv = 0;
                sh->ndeep = 0;
                sh->T0 = 0ull;
            }
            hs = 1;
            __syncthreads();
        }
        const int Ls = (L + hs - 1) / hs;  // sampled heads: lists 0, hs, 2hs, ...
        if (Ls >= kp) {
            int nper = 1;
            while (nper < 32 && nper * 2 * Ls <= nt) nper <<= 1;
            const int part = t & (nper - 1);
            for (int l0 = 0; l0 < Ls; l0 += nt / nper) {
                const int l = l0 + t / nper;
                const u64 h = l < Ls ? pre[2 * (l * hs)] : 0ull;
                int r = 0;
                if (h != 0ull)
                    for (int j = part; j < Ls; j += nper) r += pre[2 * (j * hs)] > h ? 1 : 0;
                for (int off = 1; off < nper; off <<= 1) r += __shfl_xor_sync(0xffffffffu, r, off);
                if (h != 0ull && part == 0 && r == kp - 1) sh->T0 = h;
            }
        }
        __syncthreads();
        const u64 T0 = sh->T0;  // 0: fewer than kp non-empty lists -> every key survives (at most kp*kp)
        // 2a. survivors among the first two keys of every list (a thread per list); a list whose second key survives too
        //     goes to the deep queue
        for (int l = t; l < L; l += nt) {
            const u64 k0 = pre[2 * l], k1 = pre[2 * l + 1];
            if (k0 == 0ull || k0 < T0) continue;
            const int both = (k1 != 0ull && k1 >= T0) ? 1 : 0;
            const int pos = atomicAdd(&sh->nsurv, 1 + both);
            if (pos < scap) surv[pos] = k0;
            if (both) {
                if (pos + 1 < scap) surv[pos + 1] = k1;
                deep[atomicAdd(&sh->ndeep, 1)] = l;
            }
        }
        __syncthreads();
        // 2b. deep lists: one warp per list, keys 2 .. kp-1, prefix >= T0
        const int ndeep = sh->ndeep;
        for (int di = warp; di < ndeep; di += nwarps) {
            const u64* src = lists + (size_t)deep[di] * kp;
            u64 keys[4];  // kp <= 128: all loads of the list issued before the first use
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int i = 32 * u + lane;
                keys[u] = (i >= 2 && i < kp) ? __ldcg(src + i) : 0ull;
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const bool keep = keys[u] != 0ull && keys[u] >= T0;
                const unsigned m = __ballot_sync(0xffffffffu, keep);
                if (m == 0u) break;
                int pos = 0;
                if (lane == 0) pos = atomicAdd(&sh->nsurv, __popc(m));
                pos = __shfl_sync(0xffffffffu, pos, 0);
                const int dst = pos + __popc(m & ((1u << lane) - 1u));
                if (keep && dst < scap) surv[dst] = keys[u];
            }
        }
        __syncthreads();
    }  // attempt
    fin_stamp(p, 1);  // T0 + survivors
    // 3. the kp best survivors in descending order -> A[0..kp)
    const int nsurv = sh->nsurv;
    // the re-score below reads the survivors' rows: start them on their way from HBM to L2 now (fp32 master rows)
    if (!p.xb_is_bf16 && nsurv <= 4 * kp) {
        const int lines = (p.d * 4 + 127) / 128;
        for (int i = t; i < nsurv * lines; i += nt) {
            const u64 key = surv[i / lines];
            if (key != 0ull) {
                const char* row = reinterpret_cast<const char*>(p.xb) + (size_t)key_row(key) * p.d * 4 + (size_t)(i % lines) * 128;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(row));
            }
        }
    }
    const u64* A;
    if (nsurv <= nt) {
        // usual case (a few more than kp survivors): rank by counting, one barrier instead of a sort
        u64* top = surv + nsurv;  // kp slots behind the survivors
        for (int i = t; i < kp; i += nt) top[i] = 0ull;
        __syncthreads();
        if (t < nsurv) {
            const u64 key = surv[t];
            int r = 0;
            for (int j = 0; j < nsurv; j++) r += surv[j] > key ? 1 : 0;
            if (r < kp) top[r] = key;
        }
        __syncthreads();
        A = top;
    } else {
        int pow2 = kp;
        while (pow2 < nsurv) pow2 <<= 1;
        for (int i = nsurv + t; i < pow2; i += nt) surv[i] = 0ull;
        for (int size = 2; size <= pow2; size <<= 1) {
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                __syncthreads();
                for (int e = t; e < (pow2 >> 1); e += nt) {
                    const int i = bitonic_low(e, stride);
                    cmpx_desc(surv, i, i + stride, (i & size) == 0);
                }
            }
        }
        __syncthreads();
        A = surv;  // A[0..kp) = the kp best scan keys
    }

    fin_stamp(p, 2);  // the kp best survivors ranked
    finalize_rank_emit(p, qi, A, sh, sc, id, ok, qs, reinterpret_cast<unsigned char*>(surv));
}

}  // namespace evs
