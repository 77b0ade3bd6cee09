/*
 * evs.h -- C ABI of libevs.so, the B200 (sm_100a) flat inner-product top-k engine that replaces the
 * faiss-cpu calls on evo-ssearch's similarity-search hot path.
 *
 * The reference has no FFI layer of its own: its hot path is five calls into the third-party faiss
 * Python module (SURVEY.md section 8b).  Each entry point below names the reference call site it
 * stands in for (file:line into the reference tree) and the de-facto faiss C++ signature underneath.
 *
 * Conventions
 *   - every function returns 0 on success, a negative EVS_E* code otherwise; it never aborts or
 *     exits.  evs_last_error() returns a thread-local message for the last failure on this thread.
 *   - plain pointers and sizes only.  "host" pointers are ordinary process memory owned by the
 *     caller; "dev" pointers are CUDA device pointers on the index's device (e.g. torch tensors'
 *     data_ptr()); `stream` is a cudaStream_t passed as void*, used as CUDA itself would use it
 *     (NULL = the legacy default stream, which is what torch's default stream is).
 *   - the index handle owns all device memory it allocates; the caller owns every buffer it passes.
 *     add() copies, so the caller may free its array immediately (oldapp.py:86-88 does).
 *   - search on one handle may be entered from several threads (the Flask dev server is threaded,
 *     oldapp.py:2258); calls on the same handle are serialised internally.  Single-query
 *     evs_index_search calls (k <= EVS_MAX_K) that arrive while another one runs are queued and served
 *     together, up to 16 at a time, as ONE search of the largest k, each receiving its own prefix
 *     (group commit: no timer, and a caller that finds the handle idle runs alone at once).  Groups
 *     form on shards with an int8 copy of at least option shadow_min_rows rows, where one search of
 *     m queries costs less than m lone ones; there every answer is the answer of the same call made
 *     alone (fp32 storage; bf16 storage in groups of up to 4 with k <= 48, which read the int8 copy
 *     either way), so results never depend on concurrency.  Elsewhere queued callers are searched
 *     one by one.  See evs_index_coalesce_stats.
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails with
 *     EVS_ENODEV.
 *
 * Result contract (faiss IndexFlat::search with METRIC_INNER_PRODUCT, k-entry heap handler):
 *   D[nq*k] float32 scores in descending order, I[nq*k] int64 row ids, unfilled slots
 *   (-FLT_MAX, -1).  Ranking is by the inner product of the fp32 inputs accumulated in fp64 in the
 *   fixed CANON-32 order (DESIGN.md), ties by ascending id -- independent of tile shape, batch
 *   size, storage precision of the scan and GPU count.
 */
#ifndef EVS_H_
#define EVS_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(EVS_BUILDING) && defined(__GNUC__)
#define EVS_API __attribute__((visibility("default")))
#else
#define EVS_API
#endif

#define EVS_VERSION 200 /* 0.2.0 */

/* error codes */
#define EVS_OK 0
#define EVS_EINVAL (-1)   /* bad argument (faiss: assert / FAISS_THROW_IF_NOT)         */
#define EVS_ENODEV (-2)   /* no usable CUDA device                                      */
#define EVS_ECUDA (-3)    /* a CUDA runtime call or kernel failed                       */
#define EVS_ENOMEM (-4)   /* host or device allocation failed                           */
#define EVS_EIO (-5)      /* file could not be opened / read / written                  */
#define EVS_EFORMAT (-6)  /* not a flat index.faiss file, or corrupt                    */
#define EVS_ELIMIT (-7)   /* outside the limits of this build (k > option max_k, ...)   */
#define EVS_ETIMEOUT (-8) /* a collective (row-sharded) search lost a rank: it never arrived, or reported failure */

/* element types of device buffers */
#define EVS_F32 0
#define EVS_F16 1
#define EVS_BF16 2

/* storage / scan modes of an index */
#define EVS_STORE_F32 0        /* fp32 rows; fp32 scan                                             */
#define EVS_STORE_BF16_F32 1   /* fp32 master + derived bf16 copy; bf16 scan, fp32 canonical rerank */

#define EVS_MAX_K 112          /* app limit is 48 (config.py:29); candidates kept per list: 64 or 128 */
#define EVS_MAX_K_LARGE 2048   /* ceiling of the option "max_k": searches with EVS_MAX_K < k <= max_k take the large-k path */

typedef struct evs_index evs_index; /* opaque */

/* ---- library ------------------------------------------------------------------------------- */
EVS_API int evs_version(void);
EVS_API const char* evs_last_error(void);
/* number of visible CUDA devices (0 and EVS_OK when there is none) */
EVS_API int evs_device_count(int* count);

/* ---- index lifecycle ------------------------------------------------------------------------
 * evs_index_create   <- faiss.IndexFlatIP(d)                         oldapp.py:87
 *                       (faiss::IndexFlatIP::IndexFlatIP(idx_t d)); ntotal = 0, is_trained = 1.
 *                       `device` = CUDA ordinal, `storage` = EVS_STORE_*.
 * evs_index_free     <- Python GC of the faiss index object.
 */
EVS_API int evs_index_create(int d, int device, int storage, evs_index** out);
EVS_API int evs_index_free(evs_index* idx);
EVS_API int evs_index_d(const evs_index* idx, int* d);
EVS_API int evs_index_ntotal(const evs_index* idx, int64_t* ntotal);
EVS_API int evs_index_device(const evs_index* idx, int* device);
EVS_API int evs_index_storage(const evs_index* idx, int* storage);
/* global id of local row 0 (row sharding: this handle owns rows [base, base+ntotal)) */
EVS_API int evs_index_set_id_base(evs_index* idx, int64_t base);
EVS_API int evs_index_id_base(const evs_index* idx, int64_t* base);
/* switch the scan precision in place: EVS_STORE_BF16_F32 derives the bf16 scan copy of an fp32-storage index (large query
 * batches otherwise scan in tf32 straight from the fp32 rows), EVS_STORE_F32 drops it (keeps it as the scan copy of the
 * fp32 index while the option "scan_shadow" is on).  Waits for searches in flight. */
EVS_API int evs_index_set_storage(evs_index* idx, int storage);
/* largest row norm of the index (maintained by add; it scales the certification bound of the searches) */
EVS_API int evs_index_max_row_norm(evs_index* idx, float* max_norm);

/* ---- add ------------------------------------------------------------------------------------
 * evs_index_add         <- index.add(embeddings_array)              oldapp.py:88
 *                          (void faiss::IndexFlatCodes::add(idx_t n, const float* x)); host fp32,
 *                          C-contiguous n x d; ids continue from ntotal.
 * evs_index_add_dev     same from a device buffer of dtype EVS_F32/F16/BF16 (keeps CLIP output on
 *                          the GPU instead of the .cpu().numpy() bounce at oldapp.py:36/44/52).
 * evs_index_reserve     optional capacity hint (rows) to avoid regrowth copies.
 * evs_index_add_synth   appends n synthetic rows generated on the device: counter-based function of
 *                          (seed, id_base + local row, column), optionally L2-normalised
 *                          (bench/tests only; 100M rows cannot come from the host).
 */
EVS_API int evs_index_reserve(evs_index* idx, int64_t nrows);
EVS_API int evs_index_add(evs_index* idx, int64_t n, const float* x_host);
EVS_API int evs_index_add_dev(evs_index* idx, int64_t n, const void* x_dev, int dtype, void* stream);
EVS_API int evs_index_add_synth(evs_index* idx, int64_t n, uint64_t seed, int normalize);
/* append rows `rows_host[0..n)` of `src` (same d, same device) to `dst`, device to device: the incremental
 * re-index of SURVEY.md section 8(f) rank 4 keeps the embeddings of unchanged files without a host round trip */
EVS_API int evs_index_add_rows_from(evs_index* dst, const evs_index* src, int64_t n, const int64_t* rows_host);
/* copy rows [row0, row0+n) back to host fp32 (faiss reconstruct_n; used by write and tests) */
EVS_API int evs_index_get_rows(const evs_index* idx, int64_t row0, int64_t n, float* out_host);

/* ---- search ---------------------------------------------------------------------------------
 * evs_index_search      <- index.search(q.reshape(1,-1), k)         oldapp.py:2005, :2112
 *                          (void faiss::IndexFlat::search(idx_t n, const float* x, idx_t k,
 *                           float* distances, idx_t* labels, ...) const).  Host pointers.
 *                          k <= 0 -> EVS_EINVAL (FAISS_THROW_IF_NOT(k > 0)); nq == 0 is a no-op.
 * evs_index_search_dev  same with device pointers for queries and results, enqueued on `stream`.
 *                          Batches of up to 256 queries never synchronise with the host: overflowed candidate buffers
 *                          (adversarial data only) and uncertified results are repaired by predicated launches on the
 *                          device.  Larger batches synchronise `stream` once, after the results are enqueued, to read those
 *                          flags, and the host re-runs the flagged queries with the fp32 GEMV scan.
 *                          A single query is ONE kernel launch: the scan's last CTA finalises (shards of up to 32 768
 *                          rows -- the application's index sizes -- take a latency-shaped variant of that launch; from
 *                          evs_index_search the query then travels in the kernel's parameter block and the host polls a
 *                          mapped completion word instead of draining the stream).
 *
 * Exactness of fp32-storage indexes (every entry point: host, device, partial, exchange):
 *   1 query        fp32 CUDA-core GEMV scan (or the int8 copy, exact by construction: option "scan_shadow");
 *   2..4 queries   over shards with an int8 copy, above small_max_rows and of at least shadow_min_rows rows, d a multiple
 *                  of 256 up to 1024: one pass over the int8 copy, every row's scan key kept, every row
 *                  within 2E of the k-th re-scored exactly (E the copy's proven bound): exact by construction, for bf16
 *                  storage too, and last_margins = canonical k-th score - (best excluded scan score + E);
 *   2..32 queries  otherwise: single-tf32 tensor-core scan with the top-k' kept on chip (option "x3": batches of up to 16
 *                  queries take the 3xTF32 split scan instead -- fp32-class scan error, ~1e-6 on unit vectors);
 *   more           single-tf32 tensor-core scan, candidates k' = 64/128 selected through sampled thresholds.
 *   Every result is then ranked by the canonical fp64 re-score of its candidates, and the finalise step CERTIFIES it: the
 *   k-th canonical score must clear the worst retained scan score by more than the error bound of the scan that selected
 *   the candidates, scaled by |q| * max|x| (see evs_index_last_margins).  For the GEMV and 3xTF32 scans that bound is an
 *   error model of the arithmetic; for single tf32 it is the rigorous truncation bound of DESIGN.md section 2 (both
 *   operands lose their low 13 mantissa bits towards zero); option "tf32_guard_eps_e6" replaces it by a statistical one
 *   for experiments.  Uncertified queries are re-run with the fp32 GEMV scan and k' = 128 (on the device up to 256
 *   queries per batch, by the host beyond).  bf16 storage is the recall mode (north_star: recall@k >= 0.999): not
 *   certified.
 * evs_index_search_partial_dev
 *                       row-sharded search, stage 1: this shard's k best as (fp64 canonical score,
 *                          int64 global id) pairs, sorted best first, padded with
 *                          (-DBL_MAX, -1): out_scores[nq*k], out_ids[nq*k] device buffers.  The
 *                          caller all-gathers these across ranks (NCCL) and calls evs_merge_partials_dev.
 * evs_merge_partials_dev
 *                       stage 2: merge `nparts` partial lists laid out [part][nq][k] into the
 *                          final D float32[nq*k], I int64[nq*k] on `device`.  `part_stride` is the
 *                          distance between consecutive parts in 8-byte elements, for both arrays
 *                          (0 = dense, nq*k), so one all-gathered buffer can hold scores and ids.
 */
EVS_API int evs_index_search(evs_index* idx, int64_t nq, const float* q_host, int64_t k, float* D_host, int64_t* I_host);
EVS_API int evs_index_search_dev(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, float* D_dev, int64_t* I_dev,
                         void* stream);
EVS_API int evs_index_search_partial_dev(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, double* out_scores_dev,
                                 int64_t* out_ids_dev, void* stream);
EVS_API int evs_merge_partials_dev(int device, int nparts, int64_t nq, int64_t k, const double* scores_dev,
                           const int64_t* ids_dev, int64_t part_stride, float* D_dev, int64_t* I_dev, void* stream);
/* ---- peer-store exchange (row sharding without a host-launched collective) ---------------------
 * Replaces the all-gather + merge of SURVEY.md section 8(e) -- (fp64 score, id)[nq][k] per rank -- by
 * stores over NVLink: every rank owns one symmetric buffer of `world` slots (two generations) that all
 * ranks map (CUDA IPC).  evs_index_search_exchange_dev scans the local shard, and its finalise kernel
 * writes the shard's k best into slot `rank` of EVERY rank's buffer as 32-byte entries that carry the
 * search's sequence number beside the payload (two 16-byte stores per entry; no fence, no separate
 * flag); the merge on each rank polls the world*k entries of a query until all carry this search's
 * number and ranks them into the final (D, I).  No NCCL call, no host
 * synchronisation; all ranks must call it in the same order with the same nq and k.
 *   evs_exchange_create   allocate the local buffer for at most max_nq queries x max_k results.
 *   evs_exchange_handle   64-byte IPC handle of the local buffer (all-gather these out of band).
 *   evs_exchange_connect  map the peers' buffers from `world` handles laid out by rank.
 *   evs_exchange_status   *timed_out = 1 if some merge waited ~10 s for a rank that never arrived, 2 if a rank reported that
 *                         it failed a search.  In both cases that search's results are padding (-FLT_MAX, -1), never a
 *                         merge of stale slots, and the search call that sees it returns EVS_ETIMEOUT (the host entry
 *                         point for its own search; the asynchronous device entry point on the next call) and clears it.
 * world == 1 needs no connect.  One process per GPU (two ranks of one exchange must not share a GPU).
 */
#define EVS_IPC_HANDLE_BYTES 64
typedef struct evs_exchange evs_exchange; /* opaque */
EVS_API int evs_exchange_create(int device, int rank, int world, int64_t max_nq, int64_t max_k, evs_exchange** out);
EVS_API int evs_exchange_handle(evs_exchange* ex, void* handle_out, int64_t handle_bytes);
EVS_API int evs_exchange_connect(evs_exchange* ex, const void* handles, int64_t handles_bytes);
EVS_API int evs_exchange_status(evs_exchange* ex, int* timed_out, int64_t* searches);
EVS_API int evs_exchange_free(evs_exchange* ex);
EVS_API int evs_index_search_exchange_dev(evs_index* idx, evs_exchange* ex, int64_t nq, const float* q_dev, int64_t k,
                                  float* D_dev, int64_t* I_dev, void* stream);
/* the same with host pointers (the sharded counterpart of evs_index_search: pinned staging, one H2D, one D2H, one sync) */
EVS_API int evs_index_search_exchange(evs_index* idx, evs_exchange* ex, int64_t nq, const float* q_host, int64_t k,
                              float* D_host, int64_t* I_host);
/* per-query safety margin of the last search on this handle: canonical score of the k-th result minus
 * (scan score of the worst retained candidate + the largest amount by which the scan under-estimated any
 * retained candidate); +inf when every row was a candidate.  Rows that were not retained scored below that
 * candidate, so a margin larger than the scan's error bound certifies the result exact. */
EVS_API int evs_index_last_margins(evs_index* idx, int64_t nq, float* margins_host);
/* counters of this handle: queries finalised again from the device-side exact re-run, and results that stayed
 * uncertified (more than k' - k rows within the scan error of rank k: ties at fp32 resolution) */
EVS_API int evs_index_guard_stats(evs_index* idx, int64_t* reruns, int64_t* uncertified);
/* the int8 scan copy: single-query searches whose window held more than 256 candidates (rows re-scored exactly; at 10M rows
 * most searches), the largest |x - s c|_2 of a row (-1 when the index has no copy), and the number of candidates (the window
 * C) the last search of the copy re-scored exactly */
EVS_API int evs_index_shadow_stats(evs_index* idx, int64_t* wide_searches, float* emax, int64_t* last_candidates);
/* large-k searches (k > EVS_MAX_K) on this handle, and the number of candidates the last one re-scored exactly (the largest
 * over its queries): rows whose fp32 scan score lies within twice the scan's error bound of the k-th best scan score */
EVS_API int evs_index_large_k_stats(evs_index* idx, int64_t* searches, int64_t* last_candidates);
/* coalescing of concurrent single-query evs_index_search calls on this handle: groups of two or more callers served as one
 * search, and the queries they held (a caller that ran alone moves neither); and the passes of the int8 batch search
 * (2..4 queries, any entry point; its largest window |C| is the last_candidates of evs_index_shadow_stats) */
EVS_API int evs_index_coalesce_stats(evs_index* idx, int64_t* groups, int64_t* grouped_queries, int64_t* i8_batch_passes);

/* ---- persistence: <folder>/.clip_index/index.faiss -------------------------------------------
 * evs_index_write       <- faiss.write_index(index, path)           oldapp.py:98
 * evs_index_read        <- faiss.read_index(path)                   oldapp.py:117
 *                          45-byte IndexFlat header + fp32 row-major payload (DESIGN.md);
 *                          accepts fourcc IxFI / IxF2 / IxFl like faiss's reader, keeps the
 *                          inner-product metric only (EVS_EFORMAT for L2 files).
 */
EVS_API int evs_index_write(const evs_index* idx, const char* path);
EVS_API int evs_index_read(const char* path, int device, int storage, evs_index** out);
/* evs_index_read_rows   the shard loader of a row-sharded index (SURVEY.md section 8(f) rank 1): reads ONLY rows
 *                          [row_lo, row_hi) of the payload -- bytes [45 + 4 d row_lo, 45 + 4 d row_hi) -- through the
 *                          same double-buffered pinned path; the new handle's id_base is row_lo.  row_hi < 0 = to the
 *                          end.  *ntotal_file (optional) = rows in the file.
 * evs_index_file_info   header only: d and ntotal of an index.faiss (to lay out the shards before reading). */
EVS_API int evs_index_read_rows(const char* path, int device, int storage, int64_t row_lo, int64_t row_hi, evs_index** out,
                        int64_t* ntotal_file);
EVS_API int evs_index_file_info(const char* path, int* d, int64_t* ntotal);

/* ---- stand-alone kernels ---------------------------------------------------------------------
 * evs_l2_normalize_dev  <- x /= x.norm(dim=-1, keepdim=True)        oldapp.py:35, :43, :51
 *                          in place on an n x d device buffer of dtype EVS_F32/F16/BF16; no epsilon
 *                          (a zero row becomes NaN, as in the reference).
 * evs_l2_normalize      same for a host fp32 buffer (staged through the device).
 * evs_f32_to_bf16_dev   the one-time fp32 -> bf16 database layout kernel (round to nearest even).
 */
EVS_API int evs_l2_normalize_dev(int device, void* x_dev, int64_t n, int d, int dtype, void* stream);
EVS_API int evs_l2_normalize(int device, float* x_host, int64_t n, int d);
EVS_API int evs_f32_to_bf16_dev(int device, const float* src_dev, void* dst_dev, int64_t count, void* stream);

/* ---- tuning / introspection (bench and tests) -------------------------------------------------
 * evs_set_option: "scan_variant" (0 = auto, 1 = direct-load kernel, 2 = bulk-async ring kernel),
 *                 "tile_rows", "stages", "ctas_per_sm", "profile_scans", "tc_min_nq" (query batches of at
 *                 least this many use the tensor-core scan; 0 = never), "tc_pair_min_nq" (... and of at
 *                 least this many the CTA-pair kernel; 0 = never), "tc_stages", "tc2_slice_tiles", "tc_sample_rows", "tc_heap_max_nq" (batches up to
 *                 this size keep a running top-k' per CTA in shared memory: no gather, no overflow case, no host sync),
 *                 "tc_heap_pure_max_nq" (... and up to this size also without the threshold pre-pass).
 *                 fp32 rows, batches: scanned in single tf32 and certified on the device against the rigorous truncation
 *                 bound of that scan (DESIGN.md section 2); "guard" (default 1): uncertified queries are re-run exactly in
 *                 the same call (0: only certified and counted); "x3" (default 0) / "x3_max_nq" (default 16): batches up to
 *                 that many queries use the 3xTF32 split scan instead (fp32-class scan scores, ~20 % slower);
 *                 "tf32_guard_eps_e6" (default 0 = the rigorous bound): a statistical bound instead, in millionths relative
 *                 to |q| max|x| (experiments); "exact_reruns" counts the queries the HOST re-ran (batches beyond 256
 *                 queries; evs_index_guard_stats counts the device's re-runs and the results that stayed uncertified).
 *                 "fuse_finalize" (default 1): single-query searches are ONE launch (the scan's last CTA finalises);
 *                 "pool_select" (default 1): ... with the candidates in one survivor pool under a global running threshold
 *                 (k <= 48) instead of per-CTA sorted lists; "scan_dynamic" (0 static, 1 = default: dynamic tail in the pool
 *                 kernel, 2: also fully dynamic dealing in the list-based scan) / "scan_chunk_groups" (row groups per grab);
 *                 "scan_clock": record per-CTA scan times and the last CTA's phase stamps (evs_index_scan_clocks);
 *                 "tc_inline_pre" (default 1): batches on the one-CTA tensor-core kernel over shards of up to ~2.4M rows take
 *                 their thresholds from one sampled tile per CTA inside the scan launch (two grid barriers) instead of a
 *                 pre-pass launch and a threshold launch;
 *                 "small_max_rows" (default 32768; 0 = never): single-query searches (k <= 48) of shards up to this many rows take
 *                 the small-shard kernel (keys stored by row, threshold from 128 chunk maxima: 10k x 512 in 16 us instead of 27);
 *                 "small_fast_cap" (default 2048, tests lower it): its register fast path up to this many keys above the threshold;
 *                 "scan_shadow" (default 1): an fp32 index added to while it is on keeps an int8 copy of its rows (one byte
 *                 per element and one fp32 scale per row: +25 % device memory; added to while it is off, it drops the copy;
 *                 bf16-storage indexes always keep it).  Single-query searches (k <= 48, d a multiple of 256 up to 1024) of
 *                 shards above small_max_rows and of at least "shadow_min_rows" rows (default 262144) scan that copy -- a
 *                 quarter of the fp32 bytes -- under a proven bound on its rounding, so their results are those of the fp32
 *                 scan (DESIGN.md section 2).  Indexes with subnormal, infinite or NaN elements scan their own rows;
 *                 "io_threads" (default 0 = auto: one per hardware thread, at most 16): threads that pread each 64 MiB chunk of
 *                 index.faiss into the pinned staging buffers (evs_index_read[_rows]; 6.5 GB/s with 1, 35 GB/s with 16);
 *                 "exchange_fail_next" (tests): the next exchange-mode search of this process fails after taking its
 *                 sequence number, so that the peers' failure reporting can be exercised.
 *                 evs_get_option also reads "tc_fallbacks": queries the HOST re-ran through the GEMV scan because a
 *                 tensor-core candidate buffer overflowed (batches beyond 256 queries; smaller batches repair on the device
 *                 and count in evs_index_guard_stats; should stay 0 on ordinary data).
 *                 "max_k" (default EVS_MAX_K = 112, range [112, EVS_MAX_K_LARGE = 2048]): the largest k a search, a merge and
 *                 an exchange accept; searches with k > 112 scan the fp32 rows once per pass of up to 4 queries, keep every
 *                 row's scan key, select the k-th and re-score exactly every row within twice the scan's error bound of it
 *                 (exact by construction, DESIGN.md section 2); k <= 112 routes as before whatever the value.
 *                 Unknown names -> EVS_EINVAL.
 * evs_kernel_launches: number of kernels this library has launched in this process.
 * evs_index_time_scan: runs the scan stage alone `iters` times on the index's stream for queries
 *                 already on the device and returns the mean kernel time in ms measured with CUDA
 *                 events on that stream (roofline measurement; results are discarded).
 */
EVS_API int evs_set_option(const char* name, int64_t value);
EVS_API int evs_get_option(const char* name, int64_t* value);
EVS_API int64_t evs_kernel_launches(void);
EVS_API int evs_index_time_scan(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, int iters, float* mean_ms);
/* With option "profile_scans" = 1 every search records a CUDA event pair around its scan launches on
 * the stream it runs on.  This call waits for them, returns how many searches were recorded since the
 * last call and the sum of their scan durations in ms, and resets the record. */
EVS_API int evs_index_scan_profile(evs_index* idx, int64_t* count, double* total_ms);
/* With option "scan_clock" = 1 every fused single-query scan records, per CTA, the %globaltimer at its start and at the
 * end of its scan loop: out_host = uint64 [nctas][2] of the last such search (ns); a call with out_host = NULL only returns
 * the count.  With cap_ctas >= nctas + 8 the rows behind the CTAs receive 8 uint64 stamps of the last CTA and the first 8
 * phase stamps of its finalise; with cap_ctas >= nctas + 12 all 16 finalise slots (slots 8-13: the int8 window pass,
 * evs_scan.cuh).  Diagnostics for the tail of the streaming scan. */
EVS_API int evs_index_scan_clocks(evs_index* idx, uint64_t* out_host, int64_t cap_ctas, int64_t* nctas);
/* Diagnostics for the tensor-core scans (tcgen05): raw scan scores of every row against nq queries,
 * out_dev = float32 [ntotal][pitch]; the pitch (queries padded per block) is returned in *npad, and a call
 * with out_dev = NULL only returns it.  nq <= evs_index_tc_max_queries() uses the one-CTA kernel; batches of
 * at least option "tc_pair_min_nq" queries (<= 4096) the CTA-pair kernel (cta_group::2).  bf16 storage scores
 * bf16 rows x bf16-rounded queries, fp32 storage scores in tf32; both accumulate in fp32. */
EVS_API int evs_index_tc_max_queries(const evs_index* idx, int* max_queries);
/* queries one 3xTF32 pass serves (0: bf16 storage, option "x3" off, or a dimension whose split query block does not fit) */
EVS_API int evs_index_tc_x3_max_queries(const evs_index* idx, int* max_queries);
EVS_API int evs_index_tc_scores_dev(evs_index* idx, int64_t nq, const float* q_dev, float* out_dev, int* npad, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* EVS_H_ */
