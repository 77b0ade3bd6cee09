// evs_internal.h -- host-side declarations shared by evs_kernels.cu, evs_tc*.cu and evs_api.cu.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <atomic>

#include "../../include/evs.h"

#define EVS_SMALL_QUERY_MAX_D 768  // a query of up to this many dimensions fits the 4 KB kernel parameter block beside the rest

namespace evs {

extern std::atomic<long long> g_kernel_launches;

struct ScanTuning {
    int scan_variant = 0;  // 0 auto, 1 direct loads, 2 bulk-async ring
    int tile_rows = 0;     // ring: rows per stage (0 = ~32 KiB)
    int stages = 0;        // ring: depth (0 = 4)
    int ctas_per_sm = 0;   // direct: CTAs per SM (0 = 2 fp32 and int8 / 4 bf16)
    int tc_min_nq = 2;     // query batches of at least this many use the tensor-core scan (0 = never); measured
                           // (scripts/small_nq_sweep.py): from 2 queries on it beats the CUDA-core GEMV for fp32 and bf16 rows
    int tc_pair_min_nq = 129;  // ... and of at least this many the CTA-pair kernel (evs_tc2.cu); 0 = never
    int fuse_finalize = 1;     // single-query GEMV searches: the scan's last CTA finalises (no second launch)
    int scan_dynamic = 1;      // ... rows are dealt statically for the first 7/8 of the shard and dynamically (`scan_chunk_groups` row
                               // groups per grab) for the tail: neutral on one GPU (scripts/scan_tail_probe.py), but it halves the
                               // spread of the CTAs' end times, and a sharded search waits for the slowest of G ranks (+1.3 % at 8)
    int scan_chunk_groups = 4;
    int pool_select = 1;       // ... and (k <= 48) candidates meet in one survivor pool under a global running threshold instead of
                               // per-CTA sorted lists (evs_scan.cuh: scan_pool_kernel): no per-warp final sort, no CTA merge tree,
                               // no head ranking in the last CTA
    int scan_clock = 0;        // diagnostics: record per-CTA start / end-of-scan-loop times of fused single-query scans
    int x3 = 0;                // fp32 rows, batches up to x3_max_nq queries: 3xTF32 split scan (fp32-class scan error, so the
                               // guard practically never re-runs) instead of the single-tf32 scan + guard.  Off by default:
                               // measured at 1M x 512, 16 queries: 0.417 ms against 0.343 ms (the split doubles the MMAs per
                               // staged byte and MMAs this small cost ~100 cycles each: 5.3 TB/s instead of 6.4); worth it for
                               // data whose near-duplicates would make the tf32 guard re-run most queries
    int x3_max_nq = 16;
    int guard = 1;             // certify fp32-storage batch results on the device and re-run uncertified queries exactly
    int small_max_rows = 32768;  // single-query searches of shards up to this many rows take scan_small_kernel (evs_scan.cuh: keys
                                 // stored by row, threshold from 128 chunk maxima; 10k x 512: 27 -> ~20 us); 0 = never
    int small_fast_cap = 2048;   // ... whose last CTA takes the register fast path up to this many keys above the threshold (tests
                                 // lower it to drive the general path)
    int scan_shadow = 1;         // fp32 indexes keep an int8 scan copy (built at add); single-query searches with k <= 48 of shards
                                 // of at least shadow_min_rows rows scan it -- a quarter of the bytes -- and stay exact (scan_pool_kernel)
    int shadow_min_rows = 262144;  // below it the fp32 rows are scanned: the int8 copy's search costs ~64 us however small the
                                   // shard (the last CTA re-scores a window of ~200 rows in rounds); 131 072 x 512: 64 against
                                   // 57 us; 262 144: 80 against 97 us (profiles/int8_min_rows_sweep.jsonl)
    int max_k = EVS_MAX_K;         // largest k a search accepts, in [EVS_MAX_K, EVS_MAX_K_LARGE]; k > EVS_MAX_K takes the
                                   // large-k path (evs_large_k.cu)
};

struct ScanPlan {
    int variant;  // 0 generic-d, 1 direct, 2 ring
    int nv;       // 16-byte vectors per lane per row (0 for generic)
    int grid, threads;
    size_t smem_bytes;
    int tile_rows, stages;
};

// Peer-store exchange of shard partials (row sharding): every rank owns a symmetric buffer
//   [2 parities][world shards][slot_bytes]  gather slots, one 32-byte ENTRY per (query, rank-in-partial):
//       { score bits 31..0, flag, score bits 63..32, flag, id bits 31..0, flag, id bits 63..32, flag }   (eight u32)
// and sees all ranks' buffers through peer-mapped pointers.  The flag travels WITH the data (the protocol NCCL calls LL):
// an entry is written with two 16-byte stores whose 8-byte halves (4 bytes of payload + the flag) are each atomic, and a
// reader polls an entry until all four flags carry the sequence number of the search it is merging.  No fence, no separate
// arrival flag: one NVLink traversal instead of three (data, fence round trip, flag) -- at 8 ranks the fenced protocol
// spent 32 us between "partial stored" and "merged" on every rank (scripts/exchange_probe.py).
// flag = low 31 bits of the search sequence number (never 0: buffers start zeroed, sequence numbers at 1); bit 31 set = that
// rank FAILED this search.  Two parities: a fast rank may start search s+1 while a slow one still merges s.
constexpr unsigned kExchangePoison = 1u << 31;
constexpr int kExchangeEntryBytes = 32;
struct Exchange {
    unsigned char* peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    int rank = 0, world = 0, parity = 0;
    unsigned long long seq = 0;
    size_t slot_bytes = 0;
    long long nq_total = 0;    // queries of the whole search (a search may be finalised in several launches)
    long long q_off = 0;       // first query of this launch
    int k = 0;                 // results per query of this search (entry index = query * k + rank)
    int* status = nullptr;     // host-mapped: 1 = a merge gave up waiting for a rank (~10 s), 2 = a rank reported failure
    float* merge_D = nullptr;  // non-null (single-query searches finalised inside the scan kernel): the same CTA also waits
    long long* merge_I = nullptr;  //   for the peers' partials and merges them into (D, I): one launch per search at N > 1 too
};

// everything the finalise step needs (evs_finalize.cuh: finalize_query).  Plain data, filled by evs_api.cu.
struct FinalizeParams {
    const unsigned long long* lists = nullptr;  // [nq][L][kp]  (guard phase 2: [slot][L][kp], slot = pred_slot[query])
    int L = 0;
    int kp = 0;
    const void* xb = nullptr;  // rows used for the canonical re-score (the fp32 master copy)
    int xb_is_bf16 = 0;
    const float* xq = nullptr;  // [nq][d]
    int d = 0;
    int k = 0;
    long long id_base = 0;
    // mode 0: final results
    float* D = nullptr;         // [nq][k]
    long long* I = nullptr;     // [nq][k]
    // mode 1: shard partial
    double* P_scores = nullptr;  // [nq][k]
    long long* P_ids = nullptr;  // [nq][k]
    float* margins = nullptr;    // [nq] (may be null)
    // mode 2: shard partial written straight into every rank's gather buffer over NVLink (peer stores); x.world > 0
    Exchange x;
    // certification: the result of a query is certified when  margin > err_coef * |q| * max|x|  (see finalize_query)
    float err_coef = 0.f;             // error bound of the scan that produced the lists, relative to |q|*|x|; 0 = do not certify
    float err_trunc = 0.f;            // > 0: the scan TRUNCATES its operands (single tf32): the result is certified when
                                      //   (score of rank k) - (worst retained scan score w) > err_trunc * (|q| max|x| + |w|) + err_coef * |q| max|x|
    const float* max_norm = nullptr;  // device: largest row norm of the index (null -> 1)
    const unsigned* special = nullptr;  // device: non-zero when the index holds subnormal / inf / NaN elements (null -> assume so)
    // guard, first phase: uncertified queries are queued for the exact re-run
    int* guard_count = nullptr;       // device counter (null -> no guard)
    int* guard_count_next = nullptr;  // the counter the NEXT guarded search will use: zeroed here (no memset node in the chain)
    int* guard_slot = nullptr;        // [nq]: slot of the query in the re-run queue, -1 = certified, -2 = uncertified but not queued
    int* guard_q = nullptr;           // [guard_cap]: query of each slot
    int guard_cap = 0;                // 0: flag only (the host re-runs)
    const int* overflow = nullptr;    // [nq] (optional): non-zero = a candidate buffer of the threshold scan overflowed for this
                                      // query: its result is not to be trusted whatever the margin says -> queued like an
                                      // uncertified one
    // guard, second phase: only the queries with pred_slot[q] >= 0 are finalised again, from the re-run's lists
    const int* pred_slot = nullptr;
    unsigned long long* uncertified = nullptr;  // device counter: results that stayed uncertified
    unsigned long long* reruns = nullptr;       // device counter: queries finalised again from the exact re-run
    unsigned long long* dbg = nullptr;          // diagnostics (option "scan_clock"): %globaltimer stamps of the finalise's phases
    unsigned* done_flag = nullptr;              // host-mapped word (scan_small_kernel with the query in its parameters): set to
    unsigned done_seq = 0;                      //   done_seq behind the results, polled by evs_index_search
    // pool kernel scanning the int8 copy of the fp32 master rows (scan_pool_kernel): the scan error is bounded by
    // E = |q - q^| max|x| + |q^| emax + rounding (evs_scan.cuh: shadow_bound_i8) and the thresholds are lowered by 2E, which
    // makes the result exact
    const float* shadow_emax = nullptr;         // device: largest |x - s c|_2 of a row of the int8 copy (null: the scan is not
                                                //   bounded this way)
    unsigned* wide = nullptr;                   // device counter: searches whose window held more than 256 candidates;
                                                //   wide[1] = the number of candidates the last search re-scored
};

// element type of the rows a scan reads
enum { SCAN_F32 = 0, SCAN_BF16 = 1, SCAN_I8 = 2 /* the int8 copy: codes in xb, one fp32 scale per row in xs */ };

struct ScanArgs {
    const void* xb = nullptr;
    const float* xs = nullptr;
    int is_bf16 = 0;
    int is_i8 = 0;
    long long n = 0;
    int d = 0;
    const float* xq = nullptr;
    int q0 = 0;
    int nq_pass = 1;  // 1..4 queries handled by this launch
    void* lists = nullptr;  // u64 [nq_chunk][grid][kp]
    int kp = 64;
    // direct variant only (all optional):
    const FinalizeParams* fuse = nullptr;  // single-query launch: the last CTA finalises the query (needs `ticket` or `pool`)
    unsigned* ticket = nullptr;
    const float* q_inline = nullptr;       // host pointer (small-shard kernel only): the query travels in the kernel parameters
    int small_fast_cap = 0;                // > 0 (with `pool`): the small-shard kernel (scan_small_kernel), fast path up to this many keys
    unsigned long long* pool = nullptr;    // kp = 64: pool selection (slot maxima, counters, survivor pool of pool_words(grid) words)
    unsigned* next_chunk = nullptr;        // dynamic row dealing (with `ticket` only: the last CTA resets the counter)
    int chunk_groups = 0;
    const int* qmap = nullptr;             // guard re-run: queries qmap[0 .. *nactive), nq_pass at a time
    const int* nactive = nullptr;
    int qcap = 0;
    unsigned long long* cta_clock = nullptr;
};

// host-encoded TMA descriptors are cached per (base pointer, rows, d, element type, box rows)
struct TmapCache {
    struct Entry {
        const void* base = nullptr;
        long long rows = 0;
        int d = 0, f32 = 0, box = 0;
        CUtensorMap map;
    };
    Entry e[16];
    int next = 0;
};

// tensor-core scan (evs_tc.cu)
struct TcPlan {
    int npad, nblocks, nqp, nk, stages, grid, pre_grid, groups, gpow2, cap, cap_total, kp;
    int inline_pre;  // the threshold pre-pass runs inside the scan launch (one sample tile per CTA, two grid barriers)
    int heap;  // 1: MODE_HEAP (small batch, lists [nq][grid][64] come straight out of the scan, L = grid for finalize); 2: ... seeded by a pre-pass
    int x3;    // 3xTF32: fp32 rows split hi + lo on the fly, queries split once; scan error ~1e-6 instead of ~1e-3
    size_t smem;
    long long ntiles, pre_tiles, pre_stride;
    size_t off_gmax, off_tau0, off_counts, off_overflow, off_spill_cnt, off_cand, off_spill, off_qbf16, off_end;
};
struct TcArgs {
    const void* xb;   // database rows (fp32 or bf16)
    int is_bf16;
    long long n;
    int d;
    const float* xq;  // the queries of this launch set, fp32 [nq][d]
    int nq;
    void* lists;      // out: u64 [nq][kp]
    int* overflow_out;  // out (optional): int [nq]
    TmapCache* tmaps = nullptr;
    unsigned* bar = nullptr;  // three zero-initialised device words for the in-launch pre-pass's grid barrier (null: separate launches)
    const FinalizeParams* fin = nullptr;  // threshold scans: the gather kernel finalises the query itself (no list, no second
                                          // launch); fin->overflow != null -> it is pointed at the scan's own overflow flags
};
// CTA-pair tensor-core scan for large batches (evs_tc2.cu)
struct Tc2Plan {
    int npad, half, nqb, nqp, nk, stages, grid, pre_grid, groups, gpow2, cap, cap_total, kp;
    int slice_tiles, pre_slice_tiles;
    size_t smem;
    long long ntiles, nslices, pre_tiles, pre_stride, pre_nslices;
    size_t off_gmax, off_tau0, off_counts, off_overflow, off_spill_cnt, off_cand, off_spill, off_qbf16, off_end;
};
extern int g_tc2_slice_tiles;
int tc2_max_half(int d, int is_bf16);
cudaError_t tc2_plan(long long n, int d, int is_bf16, int nq, int kp, int sm_count, Tc2Plan* pl);
size_t tc2_workspace_bytes(const Tc2Plan& pl);
cudaError_t tc2_scan(const TcArgs& a, const Tc2Plan& pl, unsigned char* ws, cudaStream_t st);
cudaError_t tc2_dump_scores(const TcArgs& a, const Tc2Plan& pl, unsigned char* ws, float* out, cudaStream_t st);
constexpr int TC_SPILL_CAP = 1024;  // per-query spill list behind the (CTA, query) candidate buffers
extern int g_tc_max_stages;
extern int g_tc_sample_rows;
extern int g_tc_heap_max_nq;
extern int g_tc_heap_pure_max_nq;
extern int g_tc_inline_pre;
int tc_sample_rows(int nq);
int tc_max_queries(int d, int is_bf16);
int tc_x3_max_queries(int d);  // queries one 3xTF32 pass serves (0 = dimension not supported)
cudaError_t tc_plan(long long n, int d, int is_bf16, int nq, int kp, int sm_count, int x3, TcPlan* pl);
size_t tc_workspace_bytes(const TcPlan& pl);
cudaError_t tc_scan_block(const TcArgs& a, const TcPlan& pl, unsigned char* ws, cudaStream_t st);
cudaError_t tc_dump_scores(const TcArgs& a, const TcPlan& pl, unsigned char* ws, float* out, cudaStream_t st);

// Launch with programmatic stream serialisation: the kernel may become resident while the preceding kernel of the stream is
// still draining (once its CTAs have called griddepcontrol.launch_dependents); the kernel itself must execute
// griddepcontrol.wait before it reads anything a predecessor wrote.  Hides launch latency and prologues on the
// multi-kernel search paths.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

cudaError_t plan_scan(long long n, int d, int elem /* SCAN_* */, int kp, int nq_pass, int sm_count, const ScanTuning& tune,
                      ScanPlan* plan);
int max_queries_per_pass(int d, int is_bf16);
cudaError_t launch_scan(const ScanArgs& a, ScanPlan* plan, cudaStream_t st);
size_t scan_pool_key_slots(size_t pool_words);  // key slots behind the header of a pool of that many words
size_t scan_pool_words(const ScanPlan& plan);  // u64 words of the pool a fused single-query launch of this plan needs (zeroed once)
size_t scan_pool_window_words();  // u64 words of the int8 window pass's list W, behind the pool's room for one key per row
cudaError_t launch_finalize(const FinalizeParams& p, long long nq, cudaStream_t st);
size_t finalize_smem_bytes_host(int L, int kp, int d);
cudaError_t launch_publish_partials(const Exchange& x, long long nq, int k, const double* scores, const long long* ids,
                                    cudaStream_t st);
cudaError_t launch_publish_poison(const Exchange& x, cudaStream_t st);
cudaError_t launch_merge_exchange(const Exchange& x, long long nq, int k, float* D, long long* I, cudaStream_t st);
cudaError_t launch_merge_partials(int nparts, long long nq, int k, const double* scores, const long long* ids,
                                  long long part_stride, float* D,
                                  long long* I, cudaStream_t st);
cudaError_t launch_l2_normalize(void* x, long long n, int d, int dtype, int sm_count, cudaStream_t st);
cudaError_t launch_f32_to_bf16(const float* src, void* dst, long long count, int sm_count, cudaStream_t st);
cudaError_t launch_to_f32(const void* src, int dtype, float* dst, long long count, int sm_count, cudaStream_t st);
cudaError_t launch_gather_rows(const float* src, const long long* ids_dev, float* dst, long long n, int d, int sm_count,
                               cudaStream_t st);
cudaError_t launch_synth_fill(float* out, long long n, int d, unsigned long long seed, long long row_base, int sm_count,
                              cudaStream_t st);
// max_norm[0] = max(max_norm[0], largest |row|) over rows [0, n): float bits compared as unsigned (norms are >= 0);
// NaN rows are ignored.  *special |= 1 when a row holds a subnormal, infinite or NaN element.  dst16 != null: the same pass
// writes the rows rounded to bf16 there.  dst8 != null: it writes the int8 copy (codes to dst8, one scale per row to
// scale8) and raises *emax (float bits) to the largest |x - s c|_2 of a row.
cudaError_t launch_row_norm_max(const float* rows, long long n, int d, float* max_norm, unsigned* special, int sm_count, cudaStream_t st,
                                void* dst16 = nullptr, signed char* dst8 = nullptr, float* scale8 = nullptr, float* emax = nullptr);
// small device fills used on the search path instead of memset nodes
cudaError_t launch_fill_i32(int* p, long long count, int value, cudaStream_t st);

// ---- large-k search (EVS_MAX_K < k <= EVS_MAX_K_LARGE; evs_large_k.cu, DESIGN.md section 2) ----
constexpr int LK_BINS = 2048;  // radix digits of 11 bits
struct LargeKQuery {           // per query of a pass, device; written by the threshold select at level 0
    unsigned prefix;           // digits of the k-th largest scan key found so far
    unsigned krem;             // rank of that key among the keys that share the prefix
    unsigned cut;              // candidates: scan key >= cut (0: every row)
    unsigned ncand;            // |C|
    unsigned best_excl;        // largest scan key below the cut (0: none)
    unsigned done;             // the cut is known (every row is a candidate): the later digit passes have nothing to do
    float E;                   // bound of |scan score - exact score| of every row for this query
    unsigned pad;
};
struct LargeKArgs {
    const float* xb = nullptr;  // the fp32 rows
    long long n = 0;
    long long npad = 0;         // row stride of the per-query workspace arrays (n rounded up to 32)
    int d = 0;
    int nv = 0;                 // 16-byte vectors per lane per row (0: generic-d kernel)
    int grid = 0;               // score scan: CTAs of 256 threads
    const float* xq = nullptr;  // the queries of this pass [nq_pass][d]
    int nq_pass = 0;
    int k = 0;
    int fast_widen = 0;         // the index holds no subnormal / inf / NaN element
    int all_rows = 0;           // ... it does: every row is a candidate
    float err_coef = 0.f;       // scan error relative to |q| max|x| (gemv_err_coef)
    const float* max_norm = nullptr;
    const signed char* xi8 = nullptr;  // non-null: the score scan reads the int8 copy (codes [n][d], scales xs8 [n]) and E is
    const float* xs8 = nullptr;        //   its bound (i8_scan_bound, e_max at *emax); nv = d / 256; the re-score reads xb
    const float* emax = nullptr;
    unsigned* S = nullptr;      // [nq_pass][npad] order-preserving scan keys
    unsigned* C = nullptr;      // [nq_pass][npad] candidate rows
    unsigned long long* R = nullptr;  // [nq_pass][npad] canonical rank keys of the candidates (0: NaN)
    unsigned* hist = nullptr;   // [3][nq_pass][LK_BINS] digit histograms (zeroed before the pass)
    LargeKQuery* st = nullptr;  // [nq_pass]
    unsigned* stats = nullptr;  // largest |C| of this search
    long long id_base = 0;
    float* D = nullptr;         // final results of the pass's first query, row stride k (or null)
    long long* I = nullptr;
    double* P_scores = nullptr;  // shard partial (when D is null)
    long long* P_ids = nullptr;
    float* margins = nullptr;   // [nq_pass]
};
size_t large_k_state_bytes(int qpp);  // hist + st of a pass (zeroed before it)
// queries per pass of the int8 score scan (lk_score_i8_kernel): 8 ran at half the read rate, limited by IDP.4A
// (scripts/i8_batch_probe.py, profiles/i8_batch_probe_pass8.jsonl)
constexpr int LK_I8_NQ = 4;
int i8_batch_grid(int nv, int sm_count);  // its CTAs, nv = d / 256: as many as are resident at once (0: none)
cudaError_t launch_large_k_scan(const LargeKArgs& a, cudaStream_t st);
cudaError_t launch_large_k_rest(const LargeKArgs& a, int sm_count, cudaStream_t st);

}  // namespace evs
