// evs_scan.cuh -- streaming score + fused per-warp top-k' selection for 1..4 queries per pass.
//
// Replaces the inner loop of faiss exhaustive_inner_product_seq + HeapBlockResultHandler that
// index.search() runs at /root/reference/oldapp.py:2005 and :2112 (SURVEY.md section 8 a5).
//
// HBM-bound: every database row is read exactly once per pass; the score matrix is never written.
// A warp owns a row: the 32 lanes split d in 16-byte vectors, multiply against query values held
// in registers, and butterfly-reduce.  Each warp keeps its own candidate buffer in shared memory
// (no atomics, no block barriers in the steady state): a key enters if it beats the warp's running
// threshold tau; when the buffer (2*KP keys) fills, the warp bitonic-sorts it, keeps KP and raises
// tau.  At the end the CTA tree-merges its warps' lists and writes one sorted KP-list per query.
//
// Two variants share all of that and differ only in how rows reach the lanes:
//   scan_direct : ld.global.nc.L1::no_allocate.v4 straight into registers, 4 rows in flight / warp
//   scan_ring   : a producer lane streams row tiles into a shared-memory ring with the bulk async
//                 copy engine (cp.async.bulk + mbarrier complete_tx, SASS UBLKCP); consumer warps
//                 read conflict-free 16-byte vectors from the ring.
#pragma once
#include "evs_common.cuh"
#include "evs_finalize.cuh"

namespace evs {

struct ScanParams {
    const void* xb;    // database rows, row-major [n][d], fp32, bf16 or int8 codes
    const float* xs;   // int8 codes: the scale of each row [n] (row = scale * codes)
    long long n;       // rows in this shard
    int d;             // dimension
    const float* xq;   // queries fp32 [*, d] on the device
    int q0;            // first query handled by this launch
    u64* lists;        // out: [query][gridDim.x][kp] keys sorted descending, 0 = empty
    int lists_stride_q;  // = gridDim.x * kp
    int kp;            // candidates kept per list (64 or 128)
    int tile_rows;     // ring variant: rows per stage
    int stages;        // ring variant: ring depth
    // direct variant only:
    unsigned* ticket;  // non-null (single-query launches): the LAST CTA to retire finalises the query in this launch
    unsigned* next_chunk;  // non-null: rows are dealt dynamically, `chunk_groups` row groups per grab (evens out the tail)
    int chunk_groups;
    const int* qmap;   // guard re-run: the launch walks the queries qmap[0 .. *nactive), NQ at a time, and writes the
    const int* nactive;  //   lists of queue slot s at lists[s * lists_stride_q ...]; null = queries q0 .. q0+NQ-1
    int qcap;          // capacity of qmap
    unsigned long long* cta_clock;  // diagnostics (option "scan_clock"): [gridDim.x][2] globaltimer at CTA start / end of its scan loop
};

template <typename T> struct Elem;
template <> struct Elem<float> { static constexpr int VEC = 4; };           // fp32: 4 per 16 B
template <> struct Elem<__nv_bfloat16> { static constexpr int VEC = 8; };  // bf16: 8 per 16 B

// ---------------------------------------------------------------------------------------------
// Query registers: lane l holds, for vector j, the VEC query values that pair with the row
// elements at [VEC*(l + 32 j), VEC*(l + 32 j) + VEC).
// ---------------------------------------------------------------------------------------------
template <typename T, int NQ, int NV>
struct QueryRegs {
    static constexpr int VEC = Elem<T>::VEC;
    float v[NQ][NV][VEC];
    __device__ __forceinline__ void load(const float* __restrict__ xq, int q0, int d, int lane) {
        int qidx[NQ];
#pragma unroll
        for (int qi = 0; qi < NQ; qi++) qidx[qi] = q0 + qi;
        load_idx(xq, qidx, d, lane);
    }
    __device__ __forceinline__ void load_idx(const float* __restrict__ xq, const int (&qidx)[NQ], int d, int lane) {
#pragma unroll
        for (int qi = 0; qi < NQ; qi++)
#pragma unroll
            for (int j = 0; j < NV; j++) {
                const float4* src = reinterpret_cast<const float4*>(xq + (size_t)qidx[qi] * d + VEC * (lane + 32 * j));
#pragma unroll
                for (int h = 0; h < VEC / 4; h++) {
                    float4 t = src[h];
                    v[qi][j][4 * h + 0] = t.x;
                    v[qi][j][4 * h + 1] = t.y;
                    v[qi][j][4 * h + 2] = t.z;
                    v[qi][j][4 * h + 3] = t.w;
                }
            }
    }
};

// unpack one 16-byte vector of row elements to fp32
__device__ __forceinline__ void unpack(const float4& raw, float (&x)[4]) {
    x[0] = raw.x; x[1] = raw.y; x[2] = raw.z; x[3] = raw.w;
}
__device__ __forceinline__ void unpack(const uint4& raw, float (&x)[8]) {
    x[0] = __uint_as_float(raw.x << 16); x[1] = __uint_as_float(raw.x & 0xFFFF0000u);
    x[2] = __uint_as_float(raw.y << 16); x[3] = __uint_as_float(raw.y & 0xFFFF0000u);
    x[4] = __uint_as_float(raw.z << 16); x[5] = __uint_as_float(raw.z & 0xFFFF0000u);
    x[6] = __uint_as_float(raw.w << 16); x[7] = __uint_as_float(raw.w & 0xFFFF0000u);
}
template <typename T> struct RawVec;
template <> struct RawVec<float> { typedef float4 type; };
template <> struct RawVec<__nv_bfloat16> { typedef uint4 type; };

// ---------------------------------------------------------------------------------------------
// int8 scan copy (scan_pool_kernel only): row x^ = s_r c_r with int8 codes c_r, the query q^ = s_q c_q with 16-bit codes
// |c_q| <= I8_QMAX split as c_q = 256 h + l into signed bytes, so that the dot product of the codes is two IDP.4A chains,
// I = 256 sum(h c) + sum(l c), exact in int32, and the scan score is s~ = fl(fl(I) * fl(s_q s_r)).
// NV = d / 256 counts 8 bytes of a row per lane.  Lane l reads NV / 2 16-byte vectors, at bytes [16 (l + 32 j), +16),
// and for odd NV (d = 256, 768) one 8-byte vector at [512 (NV / 2) + 8 l, +8): at d = 512 one LDG.128 reads a whole row.
// Word w (4 codes) of a lane's row data pairs with word w of its packed query bytes.
// ---------------------------------------------------------------------------------------------
template <> struct Elem<int8_t> { static constexpr int VEC = 8; };
constexpr int I8_QMAX = 127 * 256 + 127;  // largest |c_q| whose high byte stays within [-127, 127]

template <int NV>
struct I8Lane {
    static constexpr int V16 = NV / 2, WORDS = 2 * NV;
    // rows per group: 128 bytes per lane, so that two groups in registers (one scored, one in flight) stay near 64
    // registers; a power of two for the halving reduction (i8_warp_sum)
    static constexpr int ROWS = NV == 1 ? 16 : (NV == 2 ? 8 : 4);
    static constexpr int RSH = ROWS == 16 ? 1 : (ROWS == 8 ? 2 : 3);  // 32 / ROWS = 1 << RSH lanes end with each row's sum
    // the column of byte 0 of word w
    __device__ __forceinline__ static int col(int w, int lane) {
        return w < 4 * V16 ? 16 * (lane + 32 * (w >> 2)) + 4 * (w & 3) : 512 * V16 + 8 * lane + 4 * (w - 4 * V16);
    }
    __device__ __forceinline__ static void load(const int8_t* __restrict__ row, int lane, unsigned (&w)[WORDS]) {
#pragma unroll
        for (int j = 0; j < V16; j++) {
            const uint4 v = ldg_stream_u4(reinterpret_cast<const uint4*>(row) + lane + 32 * j);
            w[4 * j + 0] = v.x; w[4 * j + 1] = v.y; w[4 * j + 2] = v.z; w[4 * j + 3] = v.w;
        }
        if constexpr (NV & 1) {
            const uint2 v = ldg_stream_u2(reinterpret_cast<const uint2*>(row + 512 * V16) + lane);
            w[4 * V16] = v.x; w[4 * V16 + 1] = v.y;
        }
    }
};

// Sums M per-lane values (M a power of two <= 32) over the warp with a halving exchange: at xor step `off` a lane keeps
// the half of its values that the lane bit `off` selects and sends the other half; once one value is left the steps are a
// plain butterfly.  M = 8: 4 + 2 + 1 + 1 + 1 shuffles.  Lane l ends with the sum of value l >> (5 - log2 M) in v[0].
// Integer sums: exact in any order.
template <int M>
__device__ __forceinline__ void i8_warp_sum(int (&v)[M], int lane) {
#pragma unroll
    for (int s = 0; s < 5; s++) {
        const int off = 16 >> s, m = M >> s;  // values left
        if (m > 1) {
            const bool up = lane & off;
#pragma unroll
            for (int i = 0; i < m / 2; i++) {
                const int send = up ? v[i] : v[i + m / 2];
                const int keep = up ? v[i + m / 2] : v[i];
                v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
            }
        } else {
            v[0] += __shfl_xor_sync(0xffffffffu, v[0], off);
        }
    }
}

// the query code of one element: every CTA and the bound below derive the same codes from the same fp32 values
__device__ __forceinline__ int i8_query_code(float v, float sq) {
    if (!(sq > 0.f)) return 0;  // zero (or underflowing) query: q^ = 0, the bound then holds |q| max|x| in full
    const float c = rintf(__fdiv_rn(v, sq));
    return (int)fminf(fmaxf(c, (float)-I8_QMAX), (float)I8_QMAX);
}
// s_q = max|q_i| / I8_QMAX (fp32); warp-uniform
__device__ __forceinline__ float i8_query_scale(const float* __restrict__ q, int d, int lane) {
    float m = 0.f;
    for (int i = lane; i < d; i += 32) m = fmaxf(m, fabsf(q[i]));
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, off));
    return __fdiv_rn(m, (float)I8_QMAX);
}
template <int NQ, int NV>
struct QueryRegs<int8_t, NQ, NV> {
    static_assert(NQ == 1, "the int8 copy is scanned for single queries only");
    int h[2 * NV], l[2 * NV];  // packed signed bytes of the query codes that pair with word w of the lane's row data
    float sq;
    __device__ __forceinline__ void load(const float* __restrict__ xq, int q0, int d, int lane) {
        const float* q = xq + (size_t)q0 * d;
        sq = i8_query_scale(q, d, lane);
#pragma unroll
        for (int w = 0; w < 2 * NV; w++) {
            unsigned hw = 0u, lw = 0u;
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const int c = i8_query_code(q[I8Lane<NV>::col(w, lane) + b], sq);
                const int lo = ((c + 128) & 255) - 128;
                const int hi = (c - lo) >> 8;
                hw |= ((unsigned)hi & 255u) << (8 * b);
                lw |= ((unsigned)lo & 255u) << (8 * b);
            }
            h[w] = (int)hw;
            l[w] = (int)lw;
        }
    }
};

// Scan score of one row against NQ queries.  Fixed order: four partial sums per lane (vector
// component mod 4) over j, combined as (p0+p1)+(p2+p3), then the xor butterfly 16,8,4,2,1.
template <typename T, int NQ, int NV>
__device__ __forceinline__ void row_scores(const typename RawVec<T>::type (&raw)[NV], const QueryRegs<T, NQ, NV>& q,
                                           float (&out)[NQ]) {
    constexpr int VEC = Elem<T>::VEC;
    float p[NQ][4];
#pragma unroll
    for (int qi = 0; qi < NQ; qi++) p[qi][0] = p[qi][1] = p[qi][2] = p[qi][3] = 0.f;
#pragma unroll
    for (int j = 0; j < NV; j++) {
        float x[VEC];
        unpack(raw[j], x);
#pragma unroll
        for (int qi = 0; qi < NQ; qi++)
#pragma unroll
            for (int e = 0; e < VEC; e++) p[qi][e & 3] = fmaf(x[e], q.v[qi][j][e], p[qi][e & 3]);
    }
#pragma unroll
    for (int qi = 0; qi < NQ; qi++) {
        float s = (p[qi][0] + p[qi][1]) + (p[qi][2] + p[qi][3]);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        out[qi] = s;
    }
}

// ---------------------------------------------------------------------------------------------
// Per-warp candidate selection state (registers: count + threshold; shared memory: the buffer).
// ---------------------------------------------------------------------------------------------
template <int NQ>
struct WarpSelect {
    u64* buf;   // shared memory, [NQ][capw] for this warp
    int capw;   // 2 * kp
    int kp;
    int cnt[NQ];
    u64 tau[NQ];

    __device__ __forceinline__ void init(u64* warp_buf, int kp_) {
        buf = warp_buf;
        kp = kp_;
        capw = 2 * kp_;
#pragma unroll
        for (int qi = 0; qi < NQ; qi++) {
            cnt[qi] = 0;
            tau[qi] = 0ull;
        }
    }
    // sort the buffer of query qi, keep the best kp, raise the threshold
    __device__ __forceinline__ void compact(int qi, int lane) {
        u64* b = buf + qi * capw;
        __syncwarp();
        for (int i = cnt[qi] + lane; i < capw; i += 32) b[i] = 0ull;
        warp_bitonic_sort_desc(b, capw, lane);
        u64 t = b[kp - 1];
        tau[qi] = umax64(tau[qi], t);
        cnt[qi] = cnt[qi] < kp ? cnt[qi] : kp;
    }
    // warp-uniform: every lane passes the same score
    __device__ __forceinline__ void offer(int qi, float score, uint32_t row, int lane) {
        u64 key = make_key(score, row);
        if (key > tau[qi]) {
            if (lane == 0) buf[qi * capw + cnt[qi]] = key;
            cnt[qi]++;
            if (cnt[qi] == capw) compact(qi, lane);
        }
    }
    __device__ __forceinline__ void finish(int lane) {
#pragma unroll
        for (int qi = 0; qi < NQ; qi++) compact(qi, lane);
    }
};

// CTA epilogue shared by both variants: tree-merge the consumer warps' sorted lists, write one list
// per query.  `nwarps_sel` warps own buffers sel_base + warp * NQ * capw.  Called by ALL threads.
template <int NQ>
__device__ __forceinline__ void cta_merge_and_store(u64* sel_base, int nwarps_sel, int kp, const ScanParams& p, int slot0 = -1,
                                                    int nvalid = NQ) {
    if (slot0 < 0) slot0 = p.q0;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int capw = 2 * kp;
    for (int step = 1; step < nwarps_sel; step <<= 1) {
        __syncthreads();
        if (warp < nwarps_sel && (warp % (2 * step)) == 0 && warp + step < nwarps_sel) {
#pragma unroll
            for (int qi = 0; qi < NQ; qi++)
                warp_merge_top(sel_base + (size_t)(warp * NQ + qi) * capw,
                               sel_base + (size_t)((warp + step) * NQ + qi) * capw, kp, lane);
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nvalid * kp; i += blockDim.x) {
        int qi = i / kp, r = i % kp;
        p.lists[(size_t)(slot0 + qi) * p.lists_stride_q + (size_t)blockIdx.x * kp + r] = sel_base[(size_t)qi * capw + r];
    }
}

// ---------------------------------------------------------------------------------------------
// Variant 1: direct loads.  grid = ctas, block = 32 * warps.  Warps walk groups of RPG rows.
// dynamic smem: max(warps * NQ * 2*kp * 8, finalize_smem_bytes when the finalise is fused) bytes.
//
// Launched with programmatic stream serialisation: the CTAs may become resident while the preceding kernel of the
// stream drains and wait (griddepcontrol.wait) until it has completed before they read anything.
//   * rows are dealt statically (group g to warp g mod W) or -- next_chunk != null -- dynamically: a warp's first chunk
//     is static, every further one comes from a global counter, fetched one chunk ahead so that the atomic's latency
//     hides behind the loads.  A static deal leaves the SMs that the memory system serves more slowly still streaming
//     while the others idle; at 1.25M rows per GPU (the metric at N = 8) that tail is several percent of the scan.
//   * ticket != null (single-query searches): the last CTA to retire finalises the query right here (merge of the
//     per-CTA lists, canonical fp64 re-score, ranking, output / peer stores): no second launch on the latency path.
//   * nactive != null: guard re-run of the queries queued by the first finalise (evs_finalize.cuh), NQ at a time.
// ---------------------------------------------------------------------------------------------
template <typename T, int NQ, int NV>
struct ScanOcc {  // CTAs per SM the register allocation is held to (the measured optimum: 2 for fp32 and int8 rows, 4 for bf16 rows;
                  // int8 rows hold two groups in registers)
    static constexpr int value = NQ == 1 ? ((sizeof(T) == 2 && NV <= 2) ? 4 : 2) : 1;
};

__device__ __forceinline__ unsigned long long globaltimer_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}

template <typename T, int NQ, int NV>
__global__ void __launch_bounds__(256, ScanOcc<T, NQ, NV>::value) scan_direct_kernel(ScanParams p, FinalizeParams f) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int s_last;
    typedef typename RawVec<T>::type raw_t;
    // rows in flight per warp, sized so that query registers + raw vectors stay near 100 registers
    constexpr int QREGS = NQ * NV * Elem<T>::VEC;
    constexpr int RPG_RAW = (100 - QREGS) / (NV * 4);
    constexpr int RPG = RPG_RAW < 1 ? 1 : (RPG_RAW > 4 ? 4 : RPG_RAW);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    u64* sel_base = reinterpret_cast<u64*>(smem_raw);

    // The queries (and, for a guard re-run, the queue) may be the output of the preceding kernel of the stream, which may
    // itself have triggered this launch early: nothing is read before it has completed.
    asm volatile("griddepcontrol.wait;" ::: "memory");
    // only now may the next kernel of the stream (finalise / merge / the next search's scan) become resident: its own
    // prologue may read the queries too, and they are complete from here on
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    unsigned long long t_start = 0, t_fin = 0, t_merged = 0;
    if (p.cta_clock && threadIdx.x == 0) t_start = globaltimer_ns();

    int nact = NQ;
    if (p.nactive) {
        nact = *p.nactive;
        if (nact > p.qcap) nact = p.qcap;
        if (nact <= 0) return;  // nothing queued (the usual case): grid-uniform
    }
    const long long total_warps = (long long)gridDim.x * nwarps;
    const long long gw = (long long)blockIdx.x * nwarps + warp;
    const long long ngroups = (p.n + RPG - 1) / RPG;
    const size_t row_vecs = (size_t)p.d / Elem<T>::VEC;  // 16-byte vectors per row
    const raw_t* base = reinterpret_cast<const raw_t*>(p.xb);

    for (int g0 = 0; g0 < nact; g0 += NQ) {
        int qidx[NQ];
#pragma unroll
        for (int qi = 0; qi < NQ; qi++) {
            int sl = g0 + qi < nact ? g0 + qi : nact - 1;  // a short last group repeats its last query (lists not stored)
            qidx[qi] = p.nactive ? p.qmap[sl] : p.q0 + sl;
        }
        QueryRegs<T, NQ, NV> q;
        q.load_idx(p.xq, qidx, p.d, lane);
        WarpSelect<NQ> sel;
        sel.init(sel_base + (size_t)warp * NQ * 2 * p.kp, p.kp);

        auto do_group = [&](long long g) {
            const long long r0 = g * RPG;
            raw_t raw[RPG][NV];
#pragma unroll
            for (int r = 0; r < RPG; r++) {
                long long row = r0 + r < p.n ? r0 + r : p.n - 1;  // clamp: tail rows are re-read, not offered
                const raw_t* src = base + (size_t)row * row_vecs + lane;
#pragma unroll
                for (int j = 0; j < NV; j++) {
                    if constexpr (sizeof(T) == 4) raw[r][j] = ldg_stream_f4(src + 32 * j);
                    else raw[r][j] = ldg_stream_u4(src + 32 * j);
                }
            }
#pragma unroll
            for (int r = 0; r < RPG; r++) {
                float s[NQ];
                row_scores<T, NQ, NV>(raw[r], q, s);
                if (r0 + r < p.n) {
#pragma unroll
                    for (int qi = 0; qi < NQ; qi++) sel.offer(qi, s[qi], (uint32_t)(r0 + r), lane);
                }
            }
        };

        if (p.next_chunk != nullptr && p.nactive == nullptr) {
            const long long C = p.chunk_groups;
            const long long nchunks = (ngroups + C - 1) / C;
            long long chunk = gw;
            while (chunk < nchunks) {
                long long next = 0;
                if (lane == 0) next = total_warps + (long long)atomicAdd(p.next_chunk, 1u);  // consumed after this chunk
                const long long gend = (chunk + 1) * C < ngroups ? (chunk + 1) * C : ngroups;
                for (long long g = chunk * C; g < gend; g++) do_group(g);
                chunk = __shfl_sync(0xffffffffu, next, 0);
            }
        } else {
            for (long long g = gw; g < ngroups; g += total_warps) do_group(g);
        }
        if (p.cta_clock && threadIdx.x == 0 && g0 == 0) {
            p.cta_clock[2 * blockIdx.x] = t_start;
            p.cta_clock[2 * blockIdx.x + 1] = globaltimer_ns();
        }
        sel.finish(lane);
        __syncwarp();
        if (p.cta_clock && threadIdx.x == 0) t_fin = globaltimer_ns();
        const int left = nact - g0;
        cta_merge_and_store<NQ>(sel_base, nwarps, p.kp, p, p.nactive ? g0 : p.q0, left < NQ ? left : NQ);
        __syncthreads();  // the selection buffers are reused by the next group / by the finalise below
        if (p.cta_clock && threadIdx.x == 0) t_merged = globaltimer_ns();
    }

    if constexpr (NQ == 1) {
        if (p.ticket != nullptr) {
            __threadfence();  // this thread's list stores are visible device-wide before the CTA takes its ticket
            __syncthreads();
            if (threadIdx.x == 0) s_last = atomicAdd(p.ticket, 1u) == gridDim.x - 1 ? 1 : 0;
            __syncthreads();
            if (s_last) {  // CTA-uniform: every other CTA's list is complete
                if (threadIdx.x == 0) {
                    *p.ticket = 0u;  // ready for the next search (its CTAs take tickets only after this kernel has completed)
                    if (p.next_chunk) *p.next_chunk = 0u;
                }
                __threadfence();
                if (p.cta_clock && threadIdx.x == 0) {
                    unsigned long long* x = p.cta_clock + 2 * gridDim.x;
                    x[0] = globaltimer_ns();  // this (the last) CTA holds its ticket
                    x[2] = t_fin;             // ... had sorted its warps' buffers
                    x[3] = t_merged;          // ... had merged them and stored its list
                    x[4] = p.cta_clock[2 * blockIdx.x + 1];  // ... had left its scan loop (warp 0)
                }
                finalize_prologue(f, p.q0, smem_raw);
                __syncthreads();
                finalize_query(f, p.q0, f.lists + (size_t)p.q0 * f.L * f.kp, smem_raw);
                if (p.cta_clock && threadIdx.x == 0) p.cta_clock[2 * gridDim.x + 1] = globaltimer_ns();
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Variant 1p: the single-query search in ONE launch with a GLOBAL running threshold ("pool" selection).
//
// What index.search(q.reshape(1,-1), k) (/root/reference/oldapp.py:2005, :2112) issues, and the metric's step.  The streaming
// loop is scan_direct's; what differs is everything after the last byte, which at 1.25M rows per GPU (the metric over 8
// GPUs) was 10 % of the kernel: every warp bitonic-sorted its 128-key buffer, the CTA tree-merged eight lists and stored
// one, and the last CTA ranked 296 list heads before it could pick the survivors (scripts/scan_tail_probe.py: 7 + 9 + 27 us).
//   * 64 slot maxima G[s] live in global memory (L2): a warp publishes the best keys of a compaction with
//     atomicMax(G[row mod 64], key).  tau_g = min_s G[s] is a lower bound of the 64th best key of the whole shard (the 64
//     maxima belong to 64 different rows), so a warp may raise its own threshold to it: after the first compactions
//     hardly anything is admitted any more, anywhere.
//   * At the end a warp does NOT sort: it re-reads tau_g, appends the few buffered keys >= tau_g (0.2 per warp on
//     unordered data) to one survivor pool S and publishes them to G.  The last CTA (ticket) filters S by the final
//     tau_g -- some hundreds of keys -- ranks them by counting and continues with the canonical re-score
//     (finalize_rank_emit).  No lists, no merge tree, no head ranking.
// Exactness does not depend on the data: a key is dropped only below a threshold that 64 other rows are known to beat, the
// pool holds every warp's whole buffer in the worst case (capacity = warps x 128), and the last CTA streams a pool of any
// size through a 2048-key bitonic top-k' (ascending-score data: tests/test_gpu_parity.py).
// The slot maxima sit 128 bytes apart: atomics on one L2 line serialise, and all warps publish their first compaction at
// about the same time (with the 64 slots packed into four lines that storm stalled the scan for ~30 us: 385 instead of
// 357 us at 1.25M rows); a key is published only if it beats the slot value the warp has just read.
// pool layout (u64 words): G[s] at 16 s, s < 64 | [1024] survivor count (low word) | [1040] ticket (low word) | [1056, 1056 + cap) S
// ---------------------------------------------------------------------------------------------
constexpr int POOL_SLOTS = 64;          // slot maxima; must be >= the largest kp served (64): one row per slot
constexpr int POOL_GSTRIDE = 16;        // u64 words between slot maxima (one 128-byte line each)
constexpr int POOL_COUNT = POOL_SLOTS * POOL_GSTRIDE;   // word of the survivor counter
constexpr int POOL_TICKET = POOL_COUNT + 16;            // ... of the ticket counter
constexpr int POOL_HDR = POOL_TICKET + 16;              // u64 words before S
constexpr int POOL_SURV = 2048;         // survivors the last CTA holds in shared memory at a time
constexpr int POOL_KPMAX = 256;         // re-score slots of the fp32 / bf16 scans' finalise area; an int8 window of more candidates
                                        // is counted as wide (evs_index_shadow_stats)
constexpr int POOL_CMAX = 1024;         // candidates of the int8 copy's window the last CTA re-scores in one pass
// re-score slots (sc / id / ok) of the pool kernel's finalise area
__host__ __device__ inline int pool_rescore_slots(const FinalizeParams& f) { return f.shadow_emax != nullptr ? POOL_CMAX : POOL_KPMAX; }
__host__ __device__ inline size_t pool_finalize_smem_bytes(int kp, int d, int world_k) {
    size_t surv = (size_t)(POOL_SURV + kp) * 8;
    const size_t merge = (size_t)world_k * 24 + 8;  // the fused exchange merge ranks world * k partials in the same place
    if (merge > surv) surv = (merge + 7) & ~(size_t)7;
    return sizeof(FinalizeShared) + surv + (3 * (size_t)kp + (size_t)d) * 8 + 16;
}

// byte offset of the fp32 query copy of scan_small_kernel<.., QP = true> (behind the finalise area), 16-byte aligned
__host__ __device__ inline size_t small_query_smem_offset(int kp, int d, int world_k) {
    return (pool_finalize_smem_bytes(kp, d, world_k) + 15) & ~(size_t)15;
}

// ---------------------------------------------------------------------------------------------
// Exact single-query search from the int8 copy (T = int8_t, f.shadow_emax != null; DESIGN.md section 2).  Row x, its copy
// x^ = s_r c_r, e_max >= max_r |x - x^| (fp64, rounded up at add time); query q, q^ = s_q c_q; N >= max_r |x|.  The codes'
// dot product I is exact, so with P = fl(s_q s_r) and s~ = fl(fl(I) P) -- three roundings of relative 2^-24 each, plus an
// absolute 2^-150 per product should one underflow, times |fl(I)| <= 2^31 for the first --
//   |q.x - q^.x^| <= |q - q^| |x| + |q^| |x - x^| <= |q - q^| N + |q^| e_max
//   |q^.x^ - s~|  <= ((1 + 2^-24)^3 - 1) |q^| |x^| + 2^-118 <= 2^-22 |q^| (N + e_max) + 2^-118
// E = the sum of both, with |q - q^| and |q^| summed in fp64 (inflated by 2^-20 for their roundings), N = the fp32 norm
// estimate max_norm inflated by 2^-7 (a d-term fp32 sum of squares is within d 2^-24 of the truth), rounded up.
//   rule 1: a key is dropped only below key_floor(score(t) - 2E), t the score of a key 64 rows are known to reach (a warp's
//           own 64th best, tau_g): the dropped row's true score is < t - E <= that of each of those 64 rows;
//   rule 2: the last CTA re-scores every survivor with s~ >= s~_(k) - 2E exactly (C): any row outside C has a true score
//           < s~_(k) - E, below each of the k best-by-scan rows, so the top k of C is the exact answer.
// With shadow_emax == null the lowered threshold IS the threshold (twoE = 0): the fp32 / bf16 scans as before.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float shadow_bound_i8(const FinalizeParams& f, double dq2, double qh2) {
    const double dq = sqrt(dq2) * (1.0 + 0x1p-20), qh = sqrt(qh2) * (1.0 + 0x1p-20);  // |q - q^|, |q^|
    const double nx = (double)__ldg(f.max_norm) * (1.0 + 0x1p-7);
    const double em = (double)__ldg(f.shadow_emax);
    const double e = (dq * nx + qh * em + 0x1p-22 * qh * (nx + em)) * (1.0 + 0x1p-20) + 0x1p-117;
    return __double2float_ru(e);  // inf when it does not fit: every key is kept below
}
// the smallest key of score score(t) - 2E (rounded down); 1 (every key) without a finite bound
__device__ __forceinline__ u64 key_lowered(u64 t, float twoE) {
    if (twoE == 0.f || t == 0ull) return t;
    if (!(twoE <= FLT_MAX)) return 1ull;
    const uint32_t o = score_to_ordered(__fsub_rd(key_score(t), twoE));
    return o == 0u ? 1ull : ((u64)o << 32);
}

// The int8 copy's window C (rule 2) is re-scored by warps of four rows with all 16 values per lane and row in flight (64
// loads per lane; the row's lines were sent to L2 when it joined C).
__device__ __forceinline__ void pool_rescore(const FinalizeParams& f, const u64* keys, int n, double* sc, long long* id, u64* ok,
                                             const double* qs) {
    canon_rescore<4, 16>(f, keys, n, sc, id, ok, qs);
}
__device__ __forceinline__ void prefetch_row_l2(const FinalizeParams& f, u64 key) {
    const char* row = reinterpret_cast<const char*>(f.xb) + (size_t)key_row(key) * f.d * 4;
    const int lines = (f.d * 4 + 127) / 128;
    for (int i = 0; i < lines; i++) asm volatile("prefetch.global.L2 [%0];" ::"l"(row + (size_t)i * 128));
}

// C has more than POOL_CMAX keys (near-tie bursts): walk the pool in blocks of 128 keys and, whenever the next block may not
// fit, re-score what was gathered and keep its exact top k (as scan keys: a row re-scores to the same canonical score) in
// front of the buffer.  The next block's keys are in flight while a block is filtered, and a member's fp32 row is sent to L2
// as soon as it joins.  Returns the number of candidates left in cand[] (<= POOL_CMAX) for the final re-score and ranking.
// Called by all threads.
__device__ __forceinline__ int pool_wide_rounds(const FinalizeParams& f, const u64* S, unsigned m, u64 cut, u64* cand, u64* keep,
                                             double* sc, long long* id, u64* ok, const double* qs, int* s_n) {
    const int t = threadIdx.x, nt = blockDim.x;
    int fill = 0;  // CTA-uniform
    u64 key = (t < 128 && t < m) ? __ldcg(S + t) : 0ull;
    for (unsigned b0 = 0; b0 < m; b0 += 128) {
        const u64 nkey = (t < 128 && b0 + 128 + t < m) ? __ldcg(S + b0 + 128 + t) : 0ull;
        const bool mem = key != 0ull && key >= cut;
        if (mem) prefetch_row_l2(f, key);
        const int nb = __syncthreads_count(mem);
        if (fill + nb > POOL_CMAX) {
            pool_rescore(f, cand, fill, sc, id, ok, qs);
            __syncthreads();
            for (int c = t; c < fill; c += nt) {
                int rank = 0;
                for (int j = 0; j < fill; j++) rank += better_i(ok[j], id[j], ok[c], id[c]);
                if (rank < f.k) keep[rank] = cand[c];
            }
            __syncthreads();
            fill = fill < f.k ? fill : f.k;
            for (int c = t; c < fill; c += nt) cand[c] = keep[c];
        }
        if (t == 0) *s_n = fill;
        __syncthreads();
        if (mem) cand[atomicAdd(s_n, 1)] = key;
        fill += nb;
        key = nkey;
        __syncthreads();
    }
    return fill;
}

__device__ __forceinline__ u64 warp_min_u64(u64 v) {
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
        const u64 o = __shfl_xor_sync(0xffffffffu, v, off);
        v = o < v ? o : v;
    }
    return v;
}
// tau_g: the smallest slot maximum (0 while a slot is still empty).  Read past L1: other SMs raise the slots.
// Lane l leaves with G[l] in ga and G[l + 32] in gb.
__device__ __forceinline__ u64 pool_tau(const u64* G, int lane, u64& ga, u64& gb) {
    ga = __ldcg(G + (size_t)lane * POOL_GSTRIDE);
    gb = __ldcg(G + (size_t)(lane + 32) * POOL_GSTRIDE);
    return warp_min_u64(ga < gb ? ga : gb);
}
// every lane passes its key (or 0): published where it beats the slot value read by pool_tau.  Warp-synchronous.
__device__ __forceinline__ void pool_publish(u64* G, u64 key, u64 ga, u64 gb) {
    const int slot = (int)((~(uint32_t)key) & (POOL_SLOTS - 1));
    const u64 va = __shfl_sync(0xffffffffu, ga, slot & 31), vb = __shfl_sync(0xffffffffu, gb, slot & 31);
    const u64 cur = slot < 32 ? va : vb;
    if (key != 0ull && key > cur) atomicMax(reinterpret_cast<unsigned long long*>(G + (size_t)slot * POOL_GSTRIDE), (unsigned long long)key);
}

template <typename T, int NV>
__global__ void __launch_bounds__(256, ScanOcc<T, 1, NV>::value) scan_pool_kernel(ScanParams p, FinalizeParams f, u64* pool) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int s_last, s_ns, s_wcnt[9];
    __shared__ unsigned s_base;
    __shared__ u64 s_tau, s_wtau[8];  // s_wtau: each warp's running threshold (read only when it compacts: registers stay for the loop)
    __shared__ float s_twoE;
    constexpr bool I8 = sizeof(T) == 1;
    constexpr int QREGS = NV * Elem<T>::VEC;
    constexpr int RPG_RAW = (100 - QREGS) / (NV * 4);
    constexpr int RPG = I8 ? I8Lane<NV>::ROWS : (RPG_RAW < 1 ? 1 : (RPG_RAW > 4 ? 4 : RPG_RAW));
    constexpr int KP = 64, CAPW = 128;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    u64* G = pool;
    unsigned* count = reinterpret_cast<unsigned*>(pool + POOL_COUNT);
    unsigned* ticket = reinterpret_cast<unsigned*>(pool + POOL_TICKET);
    u64* S = pool + POOL_HDR;
    u64* buf = reinterpret_cast<u64*>(smem_raw) + (size_t)warp * CAPW;

    asm volatile("griddepcontrol.wait;" ::: "memory");               // the query may be the preceding kernel's output
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next search's prologue may overlap our tail
    unsigned long long t_start = 0, t_loop = 0, t_app = 0;
    if (p.cta_clock && threadIdx.x == 0) t_start = globaltimer_ns();

    const long long total_warps = (long long)gridDim.x * nwarps;
    const long long gw = (long long)blockIdx.x * nwarps + warp;
    const long long ngroups = (p.n + RPG - 1) / RPG;
    QueryRegs<T, 1, NV> q;
    q.load(p.xq, p.q0, p.d, lane);
    int cnt = 0;
    bool early = false;
    if (lane == 0) s_wtau[warp] = 0ull;
    // the last CTA's re-score wants the query in fp64: every CTA widens it now, off the critical path (the area lies behind
    // the warps' buffers and is not touched in between)
    double* qs;
    {
        size_t surv_bytes = (size_t)(POOL_SURV + KP) * 8;
        const size_t merge = (size_t)f.x.world * f.k * 24 + 8;
        if (merge > surv_bytes) surv_bytes = (merge + 7) & ~(size_t)7;
        qs = reinterpret_cast<double*>(smem_raw + sizeof(FinalizeShared) + surv_bytes + 3 * (size_t)pool_rescore_slots(f) * 8);
        const float* qf = p.xq + (size_t)p.q0 * p.d;
        for (int i = threadIdx.x; i < p.d; i += blockDim.x) qs[i] = (double)qf[i];
    }
    // int8 rows under the bound: thresholds are lowered by 2E (rules 1 and 2 above); every warp derives the same E from the
    // same query codes (each warp stores the same bits to s_twoE; nothing reads it before the barrier ahead of the last
    // CTA's work)
    bool bounded = false;  // CTA-uniform
    if constexpr (I8) {
        if (f.shadow_emax != nullptr) {
            bounded = true;
            __syncthreads();  // qs complete
            double dq2 = 0.0, qh2 = 0.0;
            for (int i = lane; i < p.d; i += 32) {
                const double qh = (double)q.sq * (double)i8_query_code((float)qs[i], q.sq);  // exact: 24 x 16 bits
                dq2 = fma(qs[i] - qh, qs[i] - qh, dq2);
                qh2 = fma(qh, qh, qh2);
            }
#pragma unroll
            for (int off = 16; off >= 1; off >>= 1) {
                dq2 += __shfl_xor_sync(0xffffffffu, dq2, off);
                qh2 += __shfl_xor_sync(0xffffffffu, qh2, off);
            }
            if (lane == 0) s_twoE = 2.f * shadow_bound_i8(f, dq2, qh2);
        }
    }
    if (!bounded && threadIdx.x == 0) s_twoE = 0.f;
    u64 tcut = 0ull;  // = key_lowered(own threshold, 2E): what a key must beat to enter the buffer

    // buffer full: sort, keep the best 64, publish the best 8 where they raise their slot (a warp sees ~n / warps rows: whatever it holds of the shard's
    // best few hundred is among its own best 8), raise the threshold to max(own 64th best, tau_g)
    auto compact = [&]() {
        __syncwarp();
        for (int i = cnt + lane; i < CAPW; i += 32) buf[i] = 0ull;
        warp_bitonic_sort_desc(buf, CAPW, lane);
        u64 ga, gb;
        const u64 tg = pool_tau(G, lane, ga, gb);
        pool_publish(G, lane < 8 ? buf[lane] : 0ull, ga, gb);
        const u64 tau = umax64(s_wtau[warp], umax64(buf[KP - 1], tg));
        __syncwarp();
        if (lane == 0) s_wtau[warp] = tau;
        tcut = key_lowered(tau, f.shadow_emax ? s_twoE : 0.f);
        cnt = 0;
#pragma unroll
        for (int h = 0; h < CAPW / 32; h++) {  // sorted: the keys >= tcut are a prefix (of at most KP when tcut = tau)
            const u64 kh = buf[lane + 32 * h];
            cnt += __popc(__ballot_sync(0xffffffffu, kh != 0ull && kh >= tcut));
        }
        if (cnt > CAPW - 32) {
            // lowered threshold, near-tie burst: the best KP stay, the rest of the window goes to the pool (which has room for
            // one key per row: a key is in the pool or in a buffer, never both)
            unsigned b = 0;
            if (lane == 0) b = atomicAdd(count, (unsigned)(cnt - KP));
            b = __shfl_sync(0xffffffffu, b, 0);
            for (int i = KP + lane; i < cnt; i += 32) S[b + i - KP] = buf[i];
            cnt = KP;
            __syncwarp();
        }
    };

    // the best of the first 16 keys goes to its slot right away: on shards where a warp sees fewer than 128 rows (100k-row
    // indexes) nobody ever compacts, and without this the slot maxima would stay empty and the pool would receive every key
    // of the shard
    auto publish_first16 = [&]() {
        early = true;
        __syncwarp();
        u64 mx = lane < 16 ? buf[lane] : 0ull;
#pragma unroll
        for (int off = 8; off >= 1; off >>= 1) mx = umax64(mx, __shfl_xor_sync(0xffffffffu, mx, off));
        if (lane == 0) atomicMax(reinterpret_cast<unsigned long long*>(G + (size_t)((~(uint32_t)mx) & (POOL_SLOTS - 1)) * POOL_GSTRIDE), (unsigned long long)mx);
    };
    // Rows are dealt statically (group g to warp g mod W: the whole machine walks one window of the database, DRAM-friendly,
    // no counter traffic) for the first part of the shard and dynamically -- `chunk_groups` groups per grab from a global
    // counter, the next grab always in flight -- for the last `dyn_groups` groups: the SMs that the memory system served
    // more slowly would otherwise still be streaming while the others idle (scripts/scan_tail_probe.py: the last CTA left
    // its loop 10-14 us after the median one with a purely static deal at 1.25M rows).
    // (small shards -- fewer than 32 groups per warp -- stay static: the first grab is on every warp's critical path there)
    const long long dyn_groups = (p.next_chunk && ngroups >= 32 * total_warps) ? (ngroups / 8 > 64 * total_warps ? 64 * total_warps : ngroups / 8) : 0;
    const long long static_end = ngroups - dyn_groups;
    long long next = -1;
    if (dyn_groups > 0 && lane == 0) next = (long long)atomicAdd(p.next_chunk, 1u);  // the first grab: needed only after the static part
    if constexpr (I8) {
        // int8 rows: a group of R rows is scored as a whole -- IDP.4A partial sums of every row, one halving reduction
        // (i8_warp_sum), one admission ballot -- while the next group's loads are in flight in a second register buffer.
        // Lanes rl * 2^RSH .. end with row rl's sum; the first of them offers its key.
        typedef I8Lane<NV> L;
        constexpr int R = L::ROWS, RSH = L::RSH;
        const int8_t* codes = reinterpret_cast<const int8_t*>(p.xb);
        const int rl = lane >> RSH;
        const bool rep = (lane & ((1 << RSH) - 1)) == 0;
        struct Group {
            unsigned w[R][L::WORDS];
            float sr;  // the scale of row rl
        };
        auto load = [&](Group& b, long long g) {
            const long long r0 = g * R;
            b.sr = __ldg(p.xs + (r0 + rl < p.n ? r0 + rl : p.n - 1));
#pragma unroll
            for (int r = 0; r < R; r++) {
                const long long row = r0 + r < p.n ? r0 + r : p.n - 1;  // clamp: tail rows are re-read, not offered
                L::load(codes + (size_t)row * p.d, lane, b.w[r]);
            }
        };
        auto score = [&](const Group& b, long long g) {
            // |I| <= d * I8_QMAX * 127 < 2^31 for d <= 512 (NV <= 2): the lane sums are combined in int32; wider rows reduce
            // both chains (each < 2^31, interleaved) and combine them in fp64, exactly
            constexpr int M = NV <= 2 ? R : 2 * R;
            int v[M];
#pragma unroll
            for (int r = 0; r < R; r++) {
                int ih = 0, il = 0;
#pragma unroll
                for (int w = 0; w < L::WORDS; w++) {
                    ih = __dp4a((int)b.w[r][w], q.h[w], ih);
                    il = __dp4a((int)b.w[r][w], q.l[w], il);
                }
                if constexpr (NV <= 2) v[r] = ih * 256 + il;
                else {
                    v[2 * r] = ih;
                    v[2 * r + 1] = il;
                }
            }
            i8_warp_sum<M>(v, lane);
            float fi;
            if constexpr (NV <= 2) fi = __int2float_rn(v[0]);
            else {  // lanes with bit RSH - 1 clear hold the row's h sum, the others its l sum
                const int o = __shfl_xor_sync(0xffffffffu, v[0], 1 << (RSH - 1));
                const bool lo = lane & (1 << (RSH - 1));
                fi = __double2float_rn(fma((double)(lo ? o : v[0]), 256.0, (double)(lo ? v[0] : o)));
            }
            const float s = __fmul_rn(fi, __fmul_rn(q.sq, b.sr));
            const long long row = g * R + rl;
            const u64 key = make_key(s, (uint32_t)row);
            bool pass = rep && row < p.n && key > tcut;
            unsigned m = __ballot_sync(0xffffffffu, pass);
            if (m == 0u) return;
            if (cnt + __popc(m) > CAPW) {  // after a compact cnt <= CAPW - 32: the group fits
                compact();
                pass = rep && row < p.n && key > tcut;
                m = __ballot_sync(0xffffffffu, pass);
            }
            if (pass) buf[cnt + __popc(m & ((1u << lane) - 1u))] = key;
            cnt += __popc(m);
            if (cnt >= 16 && !early) publish_first16();
        };
        // the group after g in this warp's deal (-1: none); a grab consumes the one in flight and issues the next
        const long long C = p.chunk_groups;
        const long long nchunks = dyn_groups > 0 ? (dyn_groups + C - 1) / C : 0;
        long long cend = 0;  // end of the grabbed chunk being walked
        auto grab = [&]() -> long long {
            const long long chunk = dyn_groups > 0 ? __shfl_sync(0xffffffffu, next, 0) : nchunks;
            if (chunk >= nchunks) return -1;
            if (lane == 0) next = (long long)atomicAdd(p.next_chunk, 1u);
            const long long g0 = static_end + chunk * C;
            cend = g0 + C < ngroups ? g0 + C : ngroups;
            return g0;
        };
        auto advance = [&](long long g) -> long long {
            if (g < static_end) return g + total_warps < static_end ? g + total_warps : grab();
            return g + 1 < cend ? g + 1 : grab();
        };
        Group A, B;
        long long g = gw < static_end ? gw : grab();
        if (g >= 0) load(A, g);
        while (g >= 0) {
            const long long g1 = advance(g);
            if (g1 >= 0) load(B, g1);
            score(A, g);
            if (g1 < 0) break;
            g = advance(g1);
            if (g >= 0) load(A, g);
            score(B, g1);
        }
    } else {
        typedef typename RawVec<T>::type raw_t;
        const size_t row_vecs = (size_t)p.d / Elem<T>::VEC;
        const raw_t* base = reinterpret_cast<const raw_t*>(p.xb);
        auto do_group = [&](long long g) {
            const long long r0 = g * RPG;
            raw_t raw[RPG][NV];
#pragma unroll
            for (int r = 0; r < RPG; r++) {
                long long row = r0 + r < p.n ? r0 + r : p.n - 1;  // clamp: tail rows are re-read, not offered
                const raw_t* src = base + (size_t)row * row_vecs + lane;
#pragma unroll
                for (int j = 0; j < NV; j++) {
                    if constexpr (sizeof(T) == 4) raw[r][j] = ldg_stream_f4(src + 32 * j);
                    else raw[r][j] = ldg_stream_u4(src + 32 * j);
                }
            }
#pragma unroll
            for (int r = 0; r < RPG; r++) {
                float s[1];
                row_scores<T, 1, NV>(raw[r], q, s);
                if (r0 + r < p.n) {
                    const u64 key = make_key(s[0], (uint32_t)(r0 + r));  // warp-uniform
                    if (key > tcut) {
                        if (lane == 0) buf[cnt] = key;
                        if (++cnt == CAPW) compact();
                        else if (cnt == 16 && !early) publish_first16();
                    }
                }
            }
        };
        for (long long g = gw; g < static_end; g += total_warps) do_group(g);
        if (dyn_groups > 0) {
            const long long C = p.chunk_groups;
            const long long nchunks = (dyn_groups + C - 1) / C;
            long long chunk = __shfl_sync(0xffffffffu, next, 0);
            while (chunk < nchunks) {
                if (lane == 0) next = (long long)atomicAdd(p.next_chunk, 1u);  // consumed after this chunk
                const long long g0 = static_end + chunk * C;
                const long long gend = g0 + C < ngroups ? g0 + C : ngroups;
                for (long long g = g0; g < gend; g++) do_group(g);
                chunk = __shfl_sync(0xffffffffu, next, 0);
            }
        }
    }
    if (p.cta_clock && threadIdx.x == 0) t_loop = globaltimer_ns();

    // end of this warp's rows: no sort.  Survivors = buffered keys >= the current tau_g: compacted to the front of the warp's
    // buffer and published to the slot maxima; the CTA then reserves room in the pool with ONE atomic for all of its warps
    // (with one atomic per warp a 10k-row index -- every warp ends at once, every key survives -- spent ~25 us queueing
    // on the counter) and copies them out.
    {
        __syncwarp();
        u64 ga, gb;
        const u64 tg = pool_tau(G, lane, ga, gb);
        tcut = key_lowered(umax64(s_wtau[warp], tg), f.shadow_emax ? s_twoE : 0.f);
        int kept = 0;
        for (int i0 = 0; i0 < cnt; i0 += 32) {  // warp-uniform
            const u64 key = (i0 + lane < cnt) ? buf[i0 + lane] : 0ull;
            const bool keep = key != 0ull && key >= tcut;
            const unsigned m = __ballot_sync(0xffffffffu, keep);
            __syncwarp();
            if (keep) buf[kept + __popc(m & ((1u << lane) - 1u))] = key;  // kept <= i0: never ahead of the reads
            pool_publish(G, keep ? key : 0ull, ga, gb);
            kept += __popc(m);
            __syncwarp();
        }
        if (lane == 0) s_wcnt[warp] = kept;
    }
    if (p.cta_clock && threadIdx.x == 0) {
        t_app = globaltimer_ns();
        p.cta_clock[2 * blockIdx.x] = t_start;
        p.cta_clock[2 * blockIdx.x + 1] = t_loop;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int total = 0;
        for (int w = 0; w < nwarps; w++) {
            const int c = s_wcnt[w];
            s_wcnt[w] = total;  // exclusive prefix
            total += c;
        }
        s_wcnt[nwarps] = total;
        s_base = total ? atomicAdd(count, (unsigned)total) : 0u;
    }
    __syncthreads();
    {
        const int off = s_wcnt[warp], end = warp + 1 < nwarps ? s_wcnt[warp + 1] : s_wcnt[nwarps];
        for (int i = lane; i < end - off; i += 32) S[s_base + off + i] = buf[i];
    }

    __threadfence();  // this thread's pool stores / slot updates are visible device-wide before the CTA takes its ticket
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
    __syncthreads();
    if (!s_last) return;  // CTA-uniform

    // ---------------- the last CTA: every other CTA's survivors are in S ----------------
    __threadfence();
    const int t = threadIdx.x, nt = blockDim.x;
    FinalizeShared* sh = reinterpret_cast<FinalizeShared*>(smem_raw);
    u64* surv = reinterpret_cast<u64*>(smem_raw + sizeof(FinalizeShared));  // [POOL_SURV + KP] (or the merge scratch, if larger)
    size_t surv_bytes = (size_t)(POOL_SURV + KP) * 8;
    {
        const size_t merge = (size_t)f.x.world * f.k * 24 + 8;
        if (merge > surv_bytes) surv_bytes = (merge + 7) & ~(size_t)7;
    }
    double* sc = reinterpret_cast<double*>(smem_raw + sizeof(FinalizeShared) + surv_bytes);
    long long* id = reinterpret_cast<long long*>(sc + pool_rescore_slots(f));
    u64* ok = reinterpret_cast<u64*>(id + pool_rescore_slots(f));  // qs (filled at kernel start) follows
    if (p.cta_clock && t == 0) {
        unsigned long long* x = p.cta_clock + 2 * gridDim.x;
        x[0] = globaltimer_ns();  // this (the last) CTA holds its ticket
        x[2] = t_app;             // ... its warp 0 had appended its survivors
        x[3] = t_app;
        x[4] = t_loop;            // ... had left its scan loop
    }
    // one round of loads: the survivor count, the slot maxima and -- speculatively -- the first keys of the pool
    const unsigned m = __ldcg(count);
    u64 spec[POOL_SURV / 2 / 256];
#pragma unroll
    for (int u = 0; u < POOL_SURV / 2 / 256; u++) spec[u] = __ldcg(S + t + 256 * u);  // blockDim.x = 256; stale beyond m: masked below
    if (warp == 0) {
        u64 ga, gb;
        const u64 tg = pool_tau(G, lane, ga, gb);
        if (lane == 0) s_tau = tg;
    }
    if (t == 0) {
        s_ns = 0;
        sh->nsurv = 0;
        sh->nvalid = 0;
        sh->maxerr = 0u;
        sh->ndeep = 0;
        sh->T0 = 0ull;
        sh->qnorm2 = 0.0;
        sh->fail = 0;
        sh->uncert = 0;
    }
    __syncthreads();
    if (f.err_coef > 0.f && warp == 0) {  // |q|^2 for the certification bound
        double s2 = 0.0;
        for (int i = lane; i < f.d; i += 32) s2 = fma(qs[i], qs[i], s2);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        if (lane == 0) sh->qnorm2 = s2;
    }
    // stream the pool through the shared-memory buffer: keys >= thr are kept; when more than half of the buffer is taken
    // it is sorted, cut to the best KP and thr rises to the KP-th best (at most POOL_SURV / 2 new keys per round: no overflow)
    u64 thr = s_tau;
    if (m > POOL_SURV / 2) {
        // A large pool (a small index: no warp ever filled its buffer, so the slot maxima are empty; or adversarial order):
        // first a threshold from the pool's first 1024 keys -- KP-th largest of 2 KP strided chunk maxima: at least KP keys
        // are >= it -- so that the rounds below keep about KP * m / 1024 keys instead of sorting everything.
        u64* cmax = reinterpret_cast<u64*>(sc);  // 2 KP words: sc | id are free until the re-score
        u64 mine = 0ull;
#pragma unroll
        for (int u = 0; u < POOL_SURV / 2 / 256; u++) mine = umax64(mine, spec[u]);  // thread t: keys t, t + 256, ... = chunk t mod 128
        mine = umax64(mine, __shfl_xor_sync(0xffffffffu, mine, 0));  // (keeps the warp converged)
        if (t >= 2 * KP) cmax[t - 2 * KP] = mine;
        __syncthreads();
        if (t < 2 * KP) cmax[t] = umax64(cmax[t], mine);
        __syncthreads();
        if (t < 2 * KP) {
            const u64 v = cmax[t];
            int r = 0;
            for (int j = 0; j < 2 * KP; j++) r += cmax[j] > v ? 1 : 0;
            if (r == KP - 1 && v > s_tau) s_tau = v;  // keys are unique: exactly one chunk maximum has this rank
        }
        __syncthreads();
        thr = s_tau;
    }
    for (unsigned b0 = 0; b0 < m; b0 += POOL_SURV / 2) {
        const unsigned bend = b0 + POOL_SURV / 2 < m ? b0 + POOL_SURV / 2 : m;
        u64 nxt[POOL_SURV / 2 / 256];  // the next round's keys are on their way while this round is filtered
#pragma unroll
        for (int u = 0; u < POOL_SURV / 2 / 256; u++) {
            const unsigned i = bend + t + 256 * u;
            nxt[u] = i < m ? __ldcg(S + i) : 0ull;
        }
#pragma unroll
        for (int u = 0; u < POOL_SURV / 2 / 256; u++) {
            if (b0 + t + 256 * u < bend && spec[u] != 0ull && spec[u] >= thr) surv[atomicAdd(&s_ns, 1)] = spec[u];
            spec[u] = nxt[u];
        }
        __syncthreads();
        const int ns_round = s_ns;
        __syncthreads();  // ... read by every thread before the next round's appends change it (the branch must be CTA-uniform)
        if (ns_round > POOL_SURV / 2 && bend < m) {
            const int ns = ns_round;
            for (int i = ns + t; i < POOL_SURV; i += nt) surv[i] = 0ull;
            for (int size = 2; size <= POOL_SURV; size <<= 1)
                for (int stride = size >> 1; stride > 0; stride >>= 1) {
                    __syncthreads();
                    for (int e = t; e < (POOL_SURV >> 1); e += nt) {
                        const int i = bitonic_low(e, stride);
                        cmpx_desc(surv, i, i + stride, (i & size) == 0);
                    }
                }
            __syncthreads();
            if (surv[KP - 1] > thr) thr = surv[KP - 1];
            if (t == 0) s_ns = KP;
            __syncthreads();
        }
    }
    const int ns = s_ns;
    __syncthreads();  // s_ns is reused as a counter below
    fin_stamp(f, 0);  // pool read
    // reset the pool for the next search of this handle (its CTAs touch it only after this kernel has completed)
    if (t < POOL_SLOTS) G[(size_t)t * POOL_GSTRIDE] = 0ull;
    if (t == 0) {
        *count = 0u;
        *ticket = 0u;
        if (p.next_chunk) *p.next_chunk = 0u;
    }
    fin_stamp(f, 1);
    const u64* A;
    if (ns <= POOL_SURV / 2) {
        const u64* src = surv;
        int nsrc = ns;
        if (ns > 3 * KP) {
            // a few hundred survivors of which KP are wanted: cut them into 2 KP strided chunks, T = KP-th largest chunk maximum
            // (at least KP keys are >= T, typically ~1.5 KP), keep the keys >= T in the upper half of the buffer
            u64* cmax = reinterpret_cast<u64*>(sc);  // 2 KP words: sc | id are free until the re-score
            if (t < 2 * KP) {
                u64 mx = 0ull;
                for (int i = t; i < ns; i += 2 * KP) mx = umax64(mx, surv[i]);
                cmax[t] = mx;
            }
            if (t == 0) s_ns = 0;
            __syncthreads();
            if (t < 2 * KP) {
                const u64 mine = cmax[t];
                int r = 0;
                for (int j = 0; j < 2 * KP; j++) r += cmax[j] > mine ? 1 : 0;
                if (r == KP - 1) s_tau = mine;  // keys are unique and every chunk is non-empty: exactly one chunk has this rank
            }
            __syncthreads();
            const u64 T = s_tau;
            u64* dst = surv + POOL_SURV / 2;
            for (int i = t; i < ns; i += nt) {
                const u64 key = surv[i];
                if (key >= T) dst[atomicAdd(&s_ns, 1)] = key;
            }
            __syncthreads();
            src = dst;
            nsrc = s_ns;
        }
        // the re-score reads the candidates' rows: start them on their way from HBM to L2 now (fp32 master rows).  (Prefetching
        // every pool survivor earlier -- ~300 rows -- delayed the 64 rows that matter: re-score 6.8 -> 9.2 us.)
        if (!f.xb_is_bf16 && nsrc <= 4 * KP) {
            const int lines = (f.d * 4 + 127) / 128;
            for (int i = t; i < nsrc * lines; i += nt) {
                const char* row = reinterpret_cast<const char*>(f.xb) + (size_t)key_row(src[i / lines]) * f.d * 4 + (size_t)(i % lines) * 128;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(row));
            }
        }
        // rank by counting (keys are unique)
        u64* top = surv + POOL_SURV;  // KP slots behind the buffer
        for (int i = t; i < KP; i += nt) top[i] = 0ull;
        __syncthreads();
        for (int i = t; i < nsrc; i += nt) {
            const u64 key = src[i];
            int r = 0;
            for (int j = 0; j < nsrc; j++) r += src[j] > key ? 1 : 0;
            if (r < KP) top[r] = key;
        }
        __syncthreads();
        A = top;
    } else {
        for (int i = ns + t; i < POOL_SURV; i += nt) surv[i] = 0ull;
        for (int size = 2; size <= POOL_SURV; size <<= 1)
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                __syncthreads();
                for (int e = t; e < (POOL_SURV >> 1); e += nt) {
                    const int i = bitonic_low(e, stride);
                    cmpx_desc(surv, i, i + stride, (i & size) == 0);
                }
            }
        __syncthreads();
        A = surv;
    }
    fin_stamp(f, 2);  // the KP best ranked
    const float twoE = s_twoE;
    if (!I8 || f.shadow_emax == nullptr) {  // (only the int8 copy is searched under the bound)
        finalize_rank_emit<(ScanOcc<T, 1, NV>::value >= 4 ? 2 : 4)>(f, p.q0, A, sh, sc, id, ok, qs, reinterpret_cast<unsigned char*>(surv));
    } else {
        // rule 2: C = every pool key >= key_lowered(s~_(k)), read again from the pool (the survivors above were cut at the
        // plain KP-th best).  Every key C needs is in the pool: rule 1 never dropped one.  A member's fp32 row is sent to
        // L2 by the thread that finds it, so that all of C's rows are on their way before the re-score starts.  (A window of
        // more than POOL_CMAX keys is gathered again by pool_wide_rounds, which walks the pool in the same order: the rows
        // prefetched here are those its first round re-scores.)
        const u64 kth = A[f.k - 1];
        __syncthreads();  // A lives in surv: read before C is gathered there
        const u64 cut = kth ? key_lowered(kth, twoE) : 1ull;  // fewer than k keys: all of them
        u64* cand = surv;
        if (t == 0) s_ns = 0;
        __syncthreads();
        constexpr int GU = 8;  // pool keys per thread in flight
        for (unsigned b0 = 0; b0 < m; b0 += GU * nt) {
            u64 kg[GU];
#pragma unroll
            for (int u = 0; u < GU; u++) {
                const unsigned i = b0 + t + u * nt;
                kg[u] = i < m ? __ldcg(S + i) : 0ull;
            }
#pragma unroll
            for (int u = 0; u < GU; u++) {
                if (kg[u] != 0ull && kg[u] >= cut) {
                    const int pos = atomicAdd(&s_ns, 1);
                    if (pos < POOL_CMAX) {
                        cand[pos] = kg[u];
                        prefetch_row_l2(f, kg[u]);
                    }
                }
            }
        }
        __syncthreads();
        fin_stamp(f, 5);  // C gathered
        int nc = s_ns;
        if (t == 0 && f.wide) {
            f.wide[1] = (unsigned)nc;
            if (nc > POOL_KPMAX) atomicAdd(f.wide, 1u);
        }
        if (nc > POOL_CMAX) nc = pool_wide_rounds(f, S, m, cut, cand, surv + POOL_CMAX, sc, id, ok, qs, &s_ns);
        for (int i = nc + t; i < KP; i += nt) cand[i] = 0ull;  // at least KP slots, empty ones as padding
        __syncthreads();
        // every member of C re-scored exactly once, then ranked from these scores
        const int nk = nc > KP ? nc : KP;
        pool_rescore(f, cand, nk, sc, id, ok, qs);
        __syncthreads();
        fin_stamp(f, 6);  // C re-scored
        // Only members with a canonical score >= b = fl_down(s~_(k) - E (1 + 2^-10)) are ranked.  The k best-by-scan rows are
        // in C with exact scores >= s~_(k) - E.  A canonical score is within (d / 32 + 5) 2^-53 |x| |q| of the exact one (fp64
        // sums of exact products), and E >= 2^-22 (|q - q^| + |q^|) N >= 2^-22 |q| N, so that is below 2^-25 E at d <= 1024
        // (the argument needs 2^-10 E): at least k members reach b, and every member below b ranks below all of them.
        // Ranking by counting is quadratic in the members ranked.
        int nr = nk;
        if (kth != 0ull && twoE <= FLT_MAX) {
            const double b = (double)__fsub_rd(key_score(kth), __fmul_ru(twoE, 0.5f * (1.f + 0x1p-10f)));
            constexpr int PT = POOL_CMAX / 256;  // slots per thread (blockDim.x = 256)
            u64 ck[PT], co[PT];
            double cs[PT];
            long long ci[PT];
            bool keep[PT];
#pragma unroll
            for (int u = 0; u < PT; u++) {
                const int c = t + u * nt;
                keep[u] = c < nk && id[c] >= 0 && sc[c] >= b;
                if (keep[u]) {
                    ck[u] = cand[c];
                    cs[u] = sc[c];
                    ci[u] = id[c];
                    co[u] = ok[c];
                }
            }
            if (t == 0) s_ns = 0;
            __syncthreads();
#pragma unroll
            for (int u = 0; u < PT; u++)
                if (keep[u]) {  // ranks by counting do not depend on the order
                    const int pos = atomicAdd(&s_ns, 1);
                    cand[pos] = ck[u];
                    sc[pos] = cs[u];
                    id[pos] = ci[u];
                    ok[pos] = co[u];
                }
            __syncthreads();
            nr = s_ns > KP ? s_ns : KP;
            for (int i = s_ns + t; i < nr; i += nt) {  // empty padding up to KP slots
                cand[i] = 0ull;
                id[i] = -1;
                ok[i] = 0ull;
            }
            __syncthreads();
        }
        finalize_rank_emit<(ScanOcc<T, 1, NV>::value >= 4 ? 2 : 4)>(f, p.q0, cand, sh, sc, id, ok, qs, reinterpret_cast<unsigned char*>(surv),
                                                                     nr, twoE * 0.5f, cut, true);
    }
    if (p.cta_clock && t == 0) p.cta_clock[2 * gridDim.x + 1] = globaltimer_ns();
}

// ns survivors in surv[0 .. ns), ns <= POOL_SURV: returns the KP best in descending order (0 = empty) -- in the KP slots behind
// the buffer (counting rank; more than 3 KP survivors are first cut by 2 KP strided chunk maxima) or, for more than
// POOL_SURV / 2 survivors, at the front of the sorted buffer.  Starts the candidates' rows on their way to L2.  Called by all
// 256 threads; cmax = 2 KP scratch words; *s_ns / *s_tau = shared scratch.
__device__ __forceinline__ const u64* pool_rank_survivors(const FinalizeParams& f, u64* surv, int ns, int* s_ns, u64* s_tau, u64* cmax) {
    constexpr int KP = 64;
    const int t = threadIdx.x, nt = blockDim.x;
    if (ns <= POOL_SURV / 2) {
        const u64* src = surv;
        int nsrc = ns;
        if (ns > 3 * KP) {
            if (t < 2 * KP) {
                u64 mx = 0ull;
                for (int i = t; i < ns; i += 2 * KP) mx = umax64(mx, surv[i]);
                cmax[t] = mx;
            }
            if (t == 0) *s_ns = 0;
            __syncthreads();
            if (t < 2 * KP) {
                const u64 mine = cmax[t];
                int r = 0;
                for (int j = 0; j < 2 * KP; j++) r += cmax[j] > mine ? 1 : 0;
                if (r == KP - 1) *s_tau = mine;  // keys are unique and every chunk is non-empty: exactly one chunk has this rank
            }
            __syncthreads();
            const u64 T = *s_tau;
            u64* dst = surv + POOL_SURV / 2;
            for (int i = t; i < ns; i += nt) {
                const u64 key = surv[i];
                if (key >= T) dst[atomicAdd(s_ns, 1)] = key;
            }
            __syncthreads();
            src = dst;
            nsrc = *s_ns;
        }
        if (!f.xb_is_bf16 && nsrc <= 4 * KP) {
            const int lines = (f.d * 4 + 127) / 128;
            for (int i = t; i < nsrc * lines; i += nt) {
                const char* row = reinterpret_cast<const char*>(f.xb) + (size_t)key_row(src[i / lines]) * f.d * 4 + (size_t)(i % lines) * 128;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(row));
            }
        }
        u64* top = surv + POOL_SURV;  // KP slots behind the buffer
        for (int i = t; i < KP; i += nt) top[i] = 0ull;
        __syncthreads();
        for (int i = t; i < nsrc; i += nt) {
            const u64 key = src[i];
            int r = 0;
            for (int j = 0; j < nsrc; j++) r += src[j] > key ? 1 : 0;
            if (r < KP) top[r] = key;
        }
        __syncthreads();
        return top;
    }
    for (int i = ns + t; i < POOL_SURV; i += nt) surv[i] = 0ull;
    for (int size = 2; size <= POOL_SURV; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            __syncthreads();
            for (int e = t; e < (POOL_SURV >> 1); e += nt) {
                const int i = bitonic_low(e, stride);
                cmpx_desc(surv, i, i + stride, (i & size) == 0);
            }
        }
    __syncthreads();
    return surv;
}

// ---------------------------------------------------------------------------------------------
// Variant 1s: the single-query search of a SMALL shard in one launch (n <= SMALL_MAX_ROWS: the 10k-row indexes the
// application really holds -- BASELINE config 1, /root/reference/oldapp.py:2005 with MAX_RESULTS <= 48).
//
// Such a shard is L2-resident and the scan loop is over after ~3 us; what the search costs is the chain of dependent
// memory round trips behind it.  With the pool selection above no warp of a small shard ever fills a buffer, so the slot
// maxima stay empty, EVERY key goes to the pool (a counter reservation per CTA) and the last CTA streams them all in
// rounds of 1024 (scripts/scan_tail_probe.py at 10k rows: 2.4 + 2.2 us from the end of the loop to the ticket, 6.9 us for
// the pool read).  Here instead
//   * a warp stores the key of row r straight to S[r] (fire and forget, inside the loop) and raises the maximum of its
//     CHUNK (warp index mod 128) with one reduction at the end: no buffer, no tau_g read, no reservation;
//   * the chunks partition the rows, so T = the 64th largest of the 128 chunk maxima has at least 64 keys >= it: it is a
//     lower bound of the 64th best key, and on unordered data ~90 keys pass it;
//   * the last CTA has its first 40 keys per thread (10 240 rows) in flight before it knows T and appends the keys >= T
//     from the registers to the survivor buffer.  More than 2048 of them (ordered / tied data) -> the general rounds with
//     sort-and-cut, from global memory.
// The tail (ranking, canonical re-score, certification, output, fused exchange merge) is the pool kernel's.
// pool layout: chunk maxima M[c] at word 8 c, c < 128 (the pool kernel's 64 slots are the even ones; both kernels leave the
// header zeroed) | [1040] ticket | [1056, 1056 + n) S
// ---------------------------------------------------------------------------------------------
constexpr int SMALL_CHUNKS = 2 * 64;    // chunk maxima (2 KP)
constexpr int SMALL_MSTRIDE = 8;        // u64 words between them (64 bytes)
constexpr int SMALL_PF = 40;            // keys per thread of the last CTA in flight at once (256 threads: 10 240 rows)
static_assert(SMALL_CHUNKS * SMALL_MSTRIDE <= POOL_COUNT, "chunk maxima overlap the pool counters");

// QP: the query travels in the kernel's parameter block (host searches, evs_index_search: no pinned staging copy, no
// host-to-device copy ahead of the launch -- the 2-3 KB ride along with the launch itself) and the last CTA raises a
// host-mapped flag behind the results, which the host polls instead of waiting for the stream to drain.
struct SmallQuery { float v[EVS_SMALL_QUERY_MAX_D]; };
struct NoQuery { int unused; };
template <bool QP> struct SmallQueryArg { typedef NoQuery type; };
template <> struct SmallQueryArg<true> { typedef SmallQuery type; };

template <typename T, int NV, bool QP>
__global__ void __launch_bounds__(256, 2) scan_small_kernel(ScanParams p, FinalizeParams f, u64* pool, int fast_cap,
                                                            const __grid_constant__ typename SmallQueryArg<QP>::type qb) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    __shared__ int s_last, s_ns;
    __shared__ u64 s_tau;
    typedef typename RawVec<T>::type raw_t;
    constexpr int QREGS = NV * Elem<T>::VEC;
    constexpr int RPG_RAW = (100 - QREGS) / (NV * 4);
    constexpr int RPG = RPG_RAW < 1 ? 1 : (RPG_RAW > 4 ? 4 : RPG_RAW);
    constexpr int KP = 64;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    u64* M = pool;
    unsigned* ticket = reinterpret_cast<unsigned*>(pool + POOL_TICKET);
    u64* S = pool + POOL_HDR;

    asm volatile("griddepcontrol.wait;" ::: "memory");               // the query may be the preceding kernel's output
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next search's prologue may overlap our tail
    unsigned long long t_start = 0, t_loop = 0;
    if (p.cta_clock && threadIdx.x == 0) t_start = globaltimer_ns();

    const long long total_warps = (long long)gridDim.x * nwarps;
    const long long gw = (long long)blockIdx.x * nwarps + warp;
    const long long ngroups = (p.n + RPG - 1) / RPG;
    const size_t row_vecs = (size_t)p.d / Elem<T>::VEC;
    const raw_t* base = reinterpret_cast<const raw_t*>(p.xb);
    QueryRegs<T, 1, NV> q;
    // shared memory as in the pool kernel: FinalizeShared | surv | sc | id | ok | qs (the query in fp64, widened by every CTA now)
    // QP: | the fp32 query (16-byte aligned), copied out of the parameter block
    size_t surv_bytes = (size_t)(POOL_SURV + KP) * 8;
    {
        const size_t merge = (size_t)f.x.world * f.k * 24 + 8;
        if (merge > surv_bytes) surv_bytes = (merge + 7) & ~(size_t)7;
    }
    double* qs = reinterpret_cast<double*>(smem_raw + sizeof(FinalizeShared) + surv_bytes + 3 * (size_t)KP * 8);
    if constexpr (QP) {
        float* qsm = reinterpret_cast<float*>(smem_raw + small_query_smem_offset(KP, p.d, f.x.world * f.k));
        for (int i = threadIdx.x; i < p.d; i += blockDim.x) {
            const float v = qb.v[i];
            qsm[i] = v;
            qs[i] = (double)v;
        }
        __syncthreads();
        q.load(qsm, 0, p.d, lane);
    } else {
        q.load(p.xq, p.q0, p.d, lane);
        const float* qf = p.xq + (size_t)p.q0 * p.d;
        for (int i = threadIdx.x; i < p.d; i += blockDim.x) qs[i] = (double)qf[i];
    }

    u64 wmax = 0ull;  // warp-uniform
    for (long long g = gw; g < ngroups; g += total_warps) {
        const long long r0 = g * RPG;
        raw_t raw[RPG][NV];
#pragma unroll
        for (int r = 0; r < RPG; r++) {
            long long row = r0 + r < p.n ? r0 + r : p.n - 1;  // clamp: tail rows are re-read, not stored
            const raw_t* src = base + (size_t)row * row_vecs + lane;
#pragma unroll
            for (int j = 0; j < NV; j++) {
                if constexpr (sizeof(T) == 4) raw[r][j] = ldg_stream_f4(src + 32 * j);
                else raw[r][j] = ldg_stream_u4(src + 32 * j);
            }
        }
#pragma unroll
        for (int r = 0; r < RPG; r++) {
            float s[1];
            row_scores<T, 1, NV>(raw[r], q, s);
            if (r0 + r < p.n) {
                const u64 key = make_key(s[0], (uint32_t)(r0 + r));  // warp-uniform; 0 for a NaN score: never a candidate
                if (lane == r) S[r0 + r] = key;
                wmax = umax64(wmax, key);
            }
        }
    }
    if (lane == 0 && wmax != 0ull)
        atomicMax(reinterpret_cast<unsigned long long*>(M + (size_t)(gw & (SMALL_CHUNKS - 1)) * SMALL_MSTRIDE), (unsigned long long)wmax);
    if (p.cta_clock && threadIdx.x == 0) {
        t_loop = globaltimer_ns();
        p.cta_clock[2 * blockIdx.x] = t_start;
        p.cta_clock[2 * blockIdx.x + 1] = t_loop;
    }

    __threadfence();  // this thread's key stores / chunk maximum are visible device-wide before the CTA takes its ticket
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == gridDim.x - 1 ? 1 : 0;
    __syncthreads();
    if (!s_last) return;  // CTA-uniform

    // ---------------- the last CTA: every row's key is in S, every chunk's maximum in M ----------------
    __threadfence();
    const int t = threadIdx.x, nt = blockDim.x;
    const int m = (int)p.n;
    FinalizeShared* sh = reinterpret_cast<FinalizeShared*>(smem_raw);
    u64* surv = reinterpret_cast<u64*>(smem_raw + sizeof(FinalizeShared));  // [POOL_SURV + KP] (or the merge scratch, if larger)
    double* sc = reinterpret_cast<double*>(smem_raw + sizeof(FinalizeShared) + surv_bytes);
    long long* id = reinterpret_cast<long long*>(sc + KP);
    u64* ok = reinterpret_cast<u64*>(id + KP);  // qs follows
    if (p.cta_clock && t == 0) {
        unsigned long long* x = p.cta_clock + 2 * gridDim.x;
        x[0] = globaltimer_ns();  // this (the last) CTA holds its ticket
        x[2] = t_loop;
        x[3] = t_loop;
        x[4] = t_loop;
    }
    // one round of loads: the first SMALL_PF keys of every thread and the chunk maxima
    u64 kreg[SMALL_PF];
#pragma unroll
    for (int u = 0; u < SMALL_PF; u++) {
        const int i = t + 256 * u;  // blockDim.x = 256
        kreg[u] = i < m ? __ldcg(S + i) : 0ull;
    }
    u64* cmax = reinterpret_cast<u64*>(sc);  // 2 KP words: sc | id are free until the re-score
    if (t < SMALL_CHUNKS) cmax[t] = __ldcg(M + (size_t)t * SMALL_MSTRIDE);
    if (t == 0) {
        s_ns = 0;
        s_tau = 0ull;
        sh->nsurv = 0;
        sh->nvalid = 0;
        sh->maxerr = 0u;
        sh->ndeep = 0;
        sh->T0 = 0ull;
        sh->qnorm2 = 0.0;
        sh->fail = 0;
        sh->uncert = 0;
    }
    __syncthreads();
    if (f.err_coef > 0.f && warp == nwarps - 1) {  // |q|^2 for the certification bound (a warp that ranks no chunk maximum)
        double s2 = 0.0;
        for (int i = lane; i < f.d; i += 32) s2 = fma(qs[i], qs[i], s2);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s2 += __shfl_xor_sync(0xffffffffu, s2, off);
        if (lane == 0) sh->qnorm2 = s2;
    }
    // T = the KP-th largest chunk maximum (non-empty maxima are unique: exactly one has KP - 1 larger ones; fewer than KP
    // non-empty chunks -> T stays 0 and every key is kept)
    if (t < SMALL_CHUNKS) {
        const u64 v = cmax[t];
        int r = 0;
        for (int j = 0; j < SMALL_CHUNKS; j++) r += cmax[j] > v ? 1 : 0;
        if (v != 0ull && r == KP - 1) s_tau = v;
    }
    __syncthreads();
    const u64 thr = s_tau;
    // reset the pool header for the next search of this handle (its CTAs touch it only after this kernel has completed)
    if (t < SMALL_CHUNKS) M[(size_t)t * SMALL_MSTRIDE] = 0ull;
    if (t == 0) *ticket = 0u;
    fin_stamp(f, 0);  // chunk maxima ranked
    // fast path: the keys >= T go from the registers straight into the survivor buffer, batch by batch with no barrier in
    // between; an append past `fast_cap` is dropped and sends the CTA to the general path afterwards
    for (int b0 = 0; b0 < m; b0 += SMALL_PF * 256) {  // CTA-uniform
        if (b0 > 0) {
#pragma unroll
            for (int u = 0; u < SMALL_PF; u++) {
                const int i = b0 + t + 256 * u;
                kreg[u] = i < m ? __ldcg(S + i) : 0ull;
            }
        }
#pragma unroll
        for (int u = 0; u < SMALL_PF; u++)
            if (kreg[u] != 0ull && kreg[u] >= thr) {
                const int pos = atomicAdd(&s_ns, 1);
                if (pos < fast_cap) surv[pos] = kreg[u];
            }
    }
    __syncthreads();
    const bool slow = s_ns > fast_cap;  // CTA-uniform: more keys above T than the fast path takes (ordered rows, exact ties)
    __syncthreads();                    // ... read by every thread before the general path resets the counter
    if (slow) {
        // ordered or tied data: the keys once more from global memory in rounds of POOL_SURV / 2; when more than half of the
        // buffer is taken it is sorted, cut to the best KP and the threshold rises to the KP-th best (no overflow)
        if (t == 0) s_ns = 0;
        __syncthreads();
        u64 th2 = thr;
        for (int b0 = 0; b0 < m; b0 += POOL_SURV / 2) {
#pragma unroll
            for (int u = 0; u < POOL_SURV / 2 / 256; u++) {
                const int i = b0 + t + 256 * u;
                const u64 key = i < m ? __ldcg(S + i) : 0ull;
                if (key != 0ull && key >= th2) surv[atomicAdd(&s_ns, 1)] = key;
            }
            __syncthreads();
            const int ns0 = s_ns;
            __syncthreads();  // ... read by every thread before the next round adds to it
            if (ns0 > POOL_SURV / 2 && b0 + POOL_SURV / 2 < m) {  // CTA-uniform
                for (int i = ns0 + t; i < POOL_SURV; i += nt) surv[i] = 0ull;
                for (int size = 2; size <= POOL_SURV; size <<= 1)
                    for (int stride = size >> 1; stride > 0; stride >>= 1) {
                        __syncthreads();
                        for (int e = t; e < (POOL_SURV >> 1); e += nt) {
                            const int i = bitonic_low(e, stride);
                            cmpx_desc(surv, i, i + stride, (i & size) == 0);
                        }
                    }
                __syncthreads();
                if (surv[KP - 1] > th2) th2 = surv[KP - 1];
                __syncthreads();
                if (t == 0) s_ns = KP;
                __syncthreads();
            }
        }
    }
    const int ns = s_ns;
    __syncthreads();  // s_ns is reused as a counter below
    fin_stamp(f, 1);  // survivors in shared memory
    const u64* A = pool_rank_survivors(f, surv, ns, &s_ns, &s_tau, reinterpret_cast<u64*>(sc));
    fin_stamp(f, 2);  // the KP best ranked
    // k <= 16 (the application's default page of results): the canonical re-score takes the best 32 candidates -- one round of
    // four rows per warp instead of two; every row outside them has a scan key below A[31], which is what the certification
    // of finalize_rank_emit compares against
    finalize_rank_emit<4, 16>(f, p.q0, A, sh, sc, id, ok, qs, reinterpret_cast<unsigned char*>(surv), f.k <= KP / 4 ? KP / 2 : KP);
    if constexpr (QP) {
        // the results (host-mapped memory) are complete: tell the host, which polls this word
        if (f.done_flag != nullptr) {
            __syncthreads();
            if (t == 0) {
                __threadfence_system();
                *reinterpret_cast<volatile unsigned*>(f.done_flag) = f.done_seq;
            }
        }
    }
    if (p.cta_clock && t == 0) p.cta_clock[2 * gridDim.x + 1] = globaltimer_ns();
}

// ---------------------------------------------------------------------------------------------
// Variant 2: bulk-async ring.  block = 32 * (consumer warps + 1) <= 288; the LAST warp is the producer.
// dynamic smem layout (bytes):
//   [0, stages*stage_bytes)                       ring, stage_bytes = tile_rows * d * sizeof(T) (mult. of 128)
//   [.., + 2*stages*8)                            full[stages], empty[stages] mbarriers
//   [.., + cw*NQ*2*kp*8)                          per-warp candidate buffers
// Tiles are dealt to CTAs round-robin: tile t = blockIdx.x + i * gridDim.x.
// ---------------------------------------------------------------------------------------------
template <typename T, int NQ, int NV>
__global__ void __launch_bounds__(288) scan_ring_kernel(ScanParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    typedef typename RawVec<T>::type raw_t;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int cw = (blockDim.x >> 5) - 1;  // consumer warps
    const int S = p.stages, TR = p.tile_rows;
    const size_t row_bytes = (size_t)p.d * sizeof(T);
    const size_t stage_bytes = (size_t)TR * row_bytes;
    unsigned char* ring = smem_raw;
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)S * stage_bytes);
    uint64_t* empty = full + S;
    u64* sel_base = reinterpret_cast<u64*>(empty + S);

    if (threadIdx.x == 0) {
        for (int s = 0; s < S; s++) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], cw);
        }
        mbar_fence_init();
    }
    __syncthreads();

    const long long ntiles = (p.n + TR - 1) / TR;

    if (warp == cw) {
        // ---------------- producer: one lane feeds the ring ----------------
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            const unsigned char* src = reinterpret_cast<const unsigned char*>(p.xb);
            for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
                mbar_wait(&empty[stage], phase ^ 1u);
                long long rows = p.n - t * TR;
                if (rows > TR) rows = TR;
                uint32_t bytes = (uint32_t)(rows * row_bytes);
                mbar_arrive_expect_tx(&full[stage], bytes);
                // one bulk copy per <= 32 KiB piece (rows are contiguous in HBM)
                const unsigned char* g = src + (size_t)t * stage_bytes;
                unsigned char* s = ring + (size_t)stage * stage_bytes;
                uint32_t off = 0;
                while (off < bytes) {
                    uint32_t piece = bytes - off < 32768u ? bytes - off : 32768u;
                    bulk_g2s(s + off, g + off, piece, &full[stage]);
                    off += piece;
                }
                if (++stage == S) {
                    stage = 0;
                    phase ^= 1u;
                }
            }
        }
        __syncwarp();
    } else {
        // ---------------- consumers ----------------
        QueryRegs<T, NQ, NV> q;
        q.load(p.xq, p.q0, p.d, lane);
        WarpSelect<NQ> sel;
        sel.init(sel_base + (size_t)warp * NQ * 2 * p.kp, p.kp);
        int stage = 0;
        uint32_t phase = 0;
        const size_t row_vecs = row_bytes / 16;
        for (long long t = blockIdx.x; t < ntiles; t += gridDim.x) {
            mbar_wait(&full[stage], phase);
            const raw_t* tile = reinterpret_cast<const raw_t*>(ring + (size_t)stage * stage_bytes);
            long long rows = p.n - t * TR;
            if (rows > TR) rows = TR;
            const long long row_base = t * TR;
#pragma unroll 2
            for (int r = warp; r < (int)rows; r += cw) {
                raw_t raw[NV];
                const raw_t* src = tile + (size_t)r * row_vecs + lane;
#pragma unroll
                for (int j = 0; j < NV; j++) raw[j] = src[32 * j];
                float s[NQ];
                row_scores<T, NQ, NV>(raw, q, s);
#pragma unroll
                for (int qi = 0; qi < NQ; qi++) sel.offer(qi, s[qi], (uint32_t)(row_base + r), lane);
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(&empty[stage]);
            if (++stage == S) {
                stage = 0;
                phase ^= 1u;
            }
        }
        sel.finish(lane);
    }
    cta_merge_and_store<NQ>(sel_base, cw, p.kp, p);
}

// ---------------------------------------------------------------------------------------------
// Generic-d fallback (d not a multiple of the vector width * 32): scalar coalesced loads, queries
// read from global through L1.  Correct for any d >= 1; not a roofline kernel.
// ---------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ float load_elem(const T* p);
template <>
__device__ __forceinline__ float load_elem<float>(const float* p) { return __ldg(p); }
template <>
__device__ __forceinline__ float load_elem<__nv_bfloat16>(const __nv_bfloat16* p) {
    return __uint_as_float(((uint32_t) * reinterpret_cast<const unsigned short*>(p)) << 16);
}

template <typename T>
__global__ void __launch_bounds__(256) scan_generic_kernel(ScanParams p) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nwarps = blockDim.x >> 5;
    u64* sel_base = reinterpret_cast<u64*>(smem_raw);
    WarpSelect<1> sel;
    sel.init(sel_base + (size_t)warp * 2 * p.kp, p.kp);
    const float* q = p.xq + (size_t)p.q0 * p.d;
    const T* xb = reinterpret_cast<const T*>(p.xb);
    const long long total_warps = (long long)gridDim.x * nwarps;
    for (long long row = (long long)blockIdx.x * nwarps + warp; row < p.n; row += total_warps) {
        const T* x = xb + (size_t)row * p.d;
        float s = 0.f;
        for (int i = lane; i < p.d; i += 32) s = fmaf(load_elem<T>(x + i), __ldg(q + i), s);
#pragma unroll
        for (int off = 16; off >= 1; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
        sel.offer(0, s, (uint32_t)row, lane);
    }
    sel.finish(lane);
    cta_merge_and_store<1>(sel_base, nwarps, p.kp, p);
}

}  // namespace evs
