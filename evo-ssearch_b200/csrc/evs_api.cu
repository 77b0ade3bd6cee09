// evs_api.cu -- the C ABI of libevs.so (include/evs.h): index handles, add / search / persistence.
// No CPU fallback anywhere: without a CUDA device every compute entry point returns EVS_ENODEV.
#include <errno.h>
#include <float.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <atomic>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <utility>
#include <vector>

#include "evs_internal.h"

using namespace evs;

// ---------------------------------------------------------------------------------------------
// errors
// ---------------------------------------------------------------------------------------------
static thread_local char t_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(t_err, sizeof(t_err), fmt, ap);
    va_end(ap);
    return code;
}
#define CU(call)                                                                                          \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess) {                                                                         \
            int c__ = (e__ == cudaErrorMemoryAllocation) ? EVS_ENOMEM                                     \
                      : (e__ == cudaErrorNoDevice || e__ == cudaErrorInsufficientDriver) ? EVS_ENODEV     \
                                                                                         : EVS_ECUDA;    \
            return fail(c__, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
        }                                                                                                 \
    } while (0)

static ScanTuning g_tune;
static std::mutex g_tune_mu;
static int g_profile_scans = 0;                    // record CUDA events around every search's scan launches
static std::atomic<long long> g_tc_fallbacks{0};   // queries re-run through the GEMV scan after a tensor-core buffer overflow
static std::atomic<long long> g_exact_reruns{0};   // queries the HOST re-ran with the fp32 GEMV scan because the finalise could not
                                                   // certify them (the device-side re-runs are counted per handle: evs_index_guard_stats)
static std::atomic<int> g_io_threads{0};           // option "io_threads": reader / writer threads per index.faiss chunk (0 = auto)
static std::atomic<int> g_exchange_fail_next{0};   // option "exchange_fail_next" (tests): the next exchange-mode search of this process
                                                   // fails after it has taken its sequence number, as an allocation failure would
static int g_tf32_guard_eps_e6 = 0;                // option "tf32_guard_eps_e6": 0 (default) = the single-tf32 scans are certified against
                                                   // their RIGOROUS truncation bound (tf32_trunc_coef); > 0 = a statistical bound instead
                                                   // (x 1e-6, relative to |q| max|x|; round 1 used 150) -- experiments only

// ---------------------------------------------------------------------------------------------
// the handle
// ---------------------------------------------------------------------------------------------
static const int kQueryChunk = 256;     // GEMV path: queries finalised per launch (bounds the list workspace)
static const int kTcQueryChunk = 4096;  // tensor-core path: queries per launch set

// per-handle device words (idx->words): counters the kernels share across searches
enum { W_TICKET = 0, W_NEXT_CHUNK = 1, W_GUARD_COUNT0 = 2, W_GUARD_COUNT1 = 3, W_UNCERT = 4 /* u64 */, W_RERUNS = 6 /* u64 */,
       W_MAX_NORM = 8 /* float */, W_SPECIAL = 9, W_BAR = 10 /* 3 words: grid barrier of the in-launch pre-pass */,
       W_EMAX = 13 /* float: largest |x - s c|_2 of a row of the int8 copy */, W_WIDE = 14 /* single-query searches of the int8
       copy whose window held more than 256 candidates */, W_LASTC = 15 /* candidates the last of them re-scored */, W_WORDS = 16 };

struct CoalesceWaiter;  // a single-query caller of evs_index_search waiting for its group (see there)

struct evs_index {
    int d = 0, device = 0, storage = EVS_STORE_F32;
    int64_t ntotal = 0, capacity = 0, id_base = 0;
    float* xb32 = nullptr;            // fp32 rows (the master copy; what index.faiss holds)
    void* xb16 = nullptr;             // derived bf16 rows (EVS_STORE_BF16_F32 only)
    signed char* xi8 = nullptr;       // the int8 scan copy of the single-query searches (bf16 storage, or an fp32 index while the
    float* xs8 = nullptr;             //   option "scan_shadow" is on): codes [capacity][d] and one scale per row [capacity];
                                      //   when present it always holds every row, and W_EMAX bounds its rounding
    unsigned special_host = 0;        // host copies of W_MAX_NORM, W_SPECIAL and W_EMAX, read back by every add
    float max_norm_host = 0.f, emax_host = 0.f;
    int sm_count = 0;
    cudaStream_t stream = nullptr;    // the handle's own stream
    cudaEvent_t ws_free = nullptr;    // recorded after each search: the workspace may be reused after it
    mutable std::mutex mu;            // serialises add/search/write/get_rows on this handle (Flask threads)
    // workspace (device)
    float* q_dev = nullptr;  size_t q_cap = 0;         // staged queries [chunk][d]
    void* lists = nullptr;   size_t lists_cap = 0;     // candidate lists
    float* D_dev = nullptr;  int64_t* I_dev = nullptr; size_t out_cap = 0;  // [chunk][k]
    float* margins_dev = nullptr; size_t margins_cap = 0;   // [nq of last search]
    unsigned char* tc_ws = nullptr; size_t tc_ws_cap = 0;   // tensor-core scan workspace
    int* tc_overflow = nullptr; size_t tc_overflow_cap = 0; // [nq] overflow flags of the tensor-core scan
    int* tc_overflow_pin = nullptr; size_t tc_overflow_pin_cap = 0;
    int64_t last_nq = 0;
    unsigned* words = nullptr;        // W_WORDS device words shared by the kernels across searches (ticket, chunk counter, guard
                                      // counters, uncertified / re-run counters, the largest row norm)
    int* guard_slot = nullptr; size_t guard_slot_cap = 0;   // [max(nq, 32)] slot per query, then [max(nq, 32)] the re-run queue
    unsigned long long* guard_lists = nullptr; size_t guard_lists_cap = 0;  // lists of the device-side exact re-run
    unsigned long long guard_seq = 0;                       // guarded searches so far (parity of the counter in use)
    unsigned long long* pool = nullptr; size_t pool_cap = 0;  // single-query pool selection (slot maxima, counters, survivors); zeroed
                                                              // at allocation, left zeroed by every search's last CTA
    unsigned long long* cta_clock = nullptr; size_t cta_clock_cap = 0; int cta_clock_n = 0;  // option "scan_clock"
    cudaStream_t last_stream = nullptr; bool have_last_stream = false;  // the stream the workspace was last used on
    TmapCache tmaps;
    bool bar_used = false;            // the search being enqueued contains a launch with a grid barrier (in-launch pre-pass)
    // optional per-search timing of the scan stage (option "profile_scans")
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> prof_events;
    size_t prof_used = 0;
    // pinned host staging
    float* q_pin = nullptr;  size_t q_pin_cap = 0;
    float* D_pin = nullptr;  int64_t* I_pin = nullptr; size_t out_pin_cap = 0;
    int64_t* I_pin_dev = nullptr;     // device address of the (mapped) pinned result buffer: the one-launch single-query search
                                      // writes (D, I) straight into host memory -- no device-to-host copy on the latency path
    float* m_pin = nullptr;  size_t m_pin_cap = 0;     // margins of the last host search (tf32 guard)
    unsigned* done_pin = nullptr;     // host-mapped word the small-shard kernel raises behind its results (polled by evs_index_search)
    unsigned* done_pin_dev = nullptr;
    unsigned done_seq = 0;
    // large-k searches (evs_large_k.cu): per query of a pass S, C [npad] u32 and R [npad] u64, then the pass state and one
    // stats word; allocated by the first such search
    unsigned char* lk_ws = nullptr; size_t lk_ws_cap = 0;
    int64_t lk_searches = 0;
    int64_t i8_batch_passes = 0;      // passes of the int8 batch route (plan_path), any entry point
    // concurrent single-query callers of evs_index_search (group commit; see there)
    std::mutex cq_mu;
    std::condition_variable cq_cv;
    std::deque<CoalesceWaiter*> cq;  // queued callers, first = next leader
    bool cq_busy = false;             // a single-query host search runs (alone or as the leader of a group)
    int64_t co_groups = 0, co_queries = 0;  // groups of two or more callers and the queries they held (under mu)
    unsigned* lk_stats = nullptr;     // into lk_ws: largest |C| of the last large-k search
};

static int use_device(int device) {
    CU(cudaSetDevice(device));
    return EVS_OK;
}

template <typename T>
static int ensure_dev(T** ptr, size_t* cap, size_t need_elems) {
    if (*cap >= need_elems && *ptr) return EVS_OK;
    if (*ptr) CU(cudaFree(*ptr));
    *ptr = nullptr;
    *cap = 0;
    CU(cudaMalloc(reinterpret_cast<void**>(ptr), need_elems * sizeof(T)));
    *cap = need_elems;
    return EVS_OK;
}

static int pick_kp(int64_t k) { return k <= 48 ? 64 : 128; }

namespace evs {
int max_queries_per_pass(int d, int is_bf16) {
    // keep the query registers of the vectorised kernels at <= 64 per lane
    int per_lane = d / 32;  // query values held per lane per query
    if (per_lane <= 0) return 1;
    int m = 64 / per_lane;
    if (m > 4) m = 4;
    if (m < 1) m = 1;
    (void)is_bf16;
    return m;
}
}  // namespace evs

// ---------------------------------------------------------------------------------------------
// library
// ---------------------------------------------------------------------------------------------
extern "C" int evs_version(void) { return EVS_VERSION; }
extern "C" const char* evs_last_error(void) { return t_err; }

extern "C" int evs_device_count(int* count) {
    if (!count) return fail(EVS_EINVAL, "count is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        cudaGetLastError();
        n = 0;
    }
    *count = n;
    return EVS_OK;
}

extern "C" int64_t evs_kernel_launches(void) { return (int64_t)g_kernel_launches.load(); }

extern "C" int evs_set_option(const char* name, int64_t value) {
    if (!name) return fail(EVS_EINVAL, "name is NULL");
    std::lock_guard<std::mutex> lk(g_tune_mu);
    if (!strcmp(name, "scan_variant")) {
        if (value < 0 || value > 2) return fail(EVS_EINVAL, "scan_variant must be 0, 1 or 2");
        g_tune.scan_variant = (int)value;
    } else if (!strcmp(name, "tile_rows")) {
        if (value < 0 || value > 1024) return fail(EVS_EINVAL, "tile_rows out of range");
        g_tune.tile_rows = (int)value;
    } else if (!strcmp(name, "stages")) {
        if (value < 0 || value > 16) return fail(EVS_EINVAL, "stages out of range");
        g_tune.stages = (int)value;
    } else if (!strcmp(name, "ctas_per_sm")) {
        if (value < 0 || value > 8) return fail(EVS_EINVAL, "ctas_per_sm out of range");
        g_tune.ctas_per_sm = (int)value;
    } else if (!strcmp(name, "tc_min_nq")) {
        if (value < 0) return fail(EVS_EINVAL, "tc_min_nq must be >= 0");
        g_tune.tc_min_nq = (int)value;
    } else if (!strcmp(name, "tc_pair_min_nq")) {
        if (value < 0) return fail(EVS_EINVAL, "tc_pair_min_nq must be >= 0");
        g_tune.tc_pair_min_nq = (int)value;
    } else if (!strcmp(name, "tc2_slice_tiles")) {
        if (value < 0 || value > 4096) return fail(EVS_EINVAL, "tc2_slice_tiles must be in [0, 4096]");
        g_tc2_slice_tiles = (int)value;
    } else if (!strcmp(name, "tc_heap_max_nq")) {
        if (value < 0 || value > 32) return fail(EVS_EINVAL, "tc_heap_max_nq must be in [0, 32]");
        g_tc_heap_max_nq = (int)value;
    } else if (!strcmp(name, "tc_heap_pure_max_nq")) {
        if (value < 0 || value > 128) return fail(EVS_EINVAL, "tc_heap_pure_max_nq must be in [0, 128]");
        g_tc_heap_pure_max_nq = (int)value;
    } else if (!strcmp(name, "tf32_guard_eps_e6")) {
        if (value < 0 || value > 100000) return fail(EVS_EINVAL, "tf32_guard_eps_e6 must be in [0, 100000]");
        g_tf32_guard_eps_e6 = (int)value;
    } else if (!strcmp(name, "tc_inline_pre")) {
        g_tc_inline_pre = value ? 1 : 0;
    } else if (!strcmp(name, "tc_sample_rows")) {
        if (value != 0 && (value < 1024 || value > (1 << 24))) return fail(EVS_EINVAL, "tc_sample_rows must be 0 (auto) or in [1024, 2^24]");
        g_tc_sample_rows = (int)value;
    } else if (!strcmp(name, "tc_stages")) {
        if (value < 2 || value > 14) return fail(EVS_EINVAL, "tc_stages must be in [2, 14]");
        g_tc_max_stages = (int)value;
    } else if (!strcmp(name, "profile_scans")) {
        g_profile_scans = value ? 1 : 0;
    } else if (!strcmp(name, "fuse_finalize")) {
        g_tune.fuse_finalize = value ? 1 : 0;
    } else if (!strcmp(name, "scan_dynamic")) {
        if (value < 0 || value > 2) return fail(EVS_EINVAL, "scan_dynamic must be 0, 1 or 2");
        g_tune.scan_dynamic = (int)value;  // 1: dynamic tail in the pool kernel; 2: also fully dynamic dealing in the list-based fused scan
    } else if (!strcmp(name, "scan_chunk_groups")) {
        if (value < 1 || value > 64) return fail(EVS_EINVAL, "scan_chunk_groups must be in [1, 64]");
        g_tune.scan_chunk_groups = (int)value;
    } else if (!strcmp(name, "exchange_fail_next")) {
        g_exchange_fail_next.store(value ? 1 : 0);
    } else if (!strcmp(name, "pool_select")) {
        g_tune.pool_select = value ? 1 : 0;
    } else if (!strcmp(name, "scan_clock")) {
        g_tune.scan_clock = value ? 1 : 0;
    } else if (!strcmp(name, "x3")) {
        g_tune.x3 = value ? 1 : 0;
    } else if (!strcmp(name, "x3_max_nq")) {
        if (value < 0 || value > 32) return fail(EVS_EINVAL, "x3_max_nq must be in [0, 32]");
        g_tune.x3_max_nq = (int)value;
    } else if (!strcmp(name, "guard")) {
        g_tune.guard = value ? 1 : 0;
    } else if (!strcmp(name, "small_max_rows")) {
        if (value < 0 || value > (1 << 20)) return fail(EVS_EINVAL, "small_max_rows must be in [0, 2^20]");
        g_tune.small_max_rows = (int)value;
    } else if (!strcmp(name, "small_fast_cap")) {
        if (value < 1 || value > 2048) return fail(EVS_EINVAL, "small_fast_cap must be in [1, 2048]");
        g_tune.small_fast_cap = (int)value;
    } else if (!strcmp(name, "scan_shadow")) {
        g_tune.scan_shadow = value ? 1 : 0;
    } else if (!strcmp(name, "shadow_min_rows")) {
        if (value < 0 || value > INT32_MAX) return fail(EVS_EINVAL, "shadow_min_rows must be in [0, 2^31 - 1]");
        g_tune.shadow_min_rows = (int)value;
    } else if (!strcmp(name, "io_threads")) {
        if (value < 0 || value > 64) return fail(EVS_EINVAL, "io_threads must be in [0, 64]");
        g_io_threads.store((int)value);
    } else if (!strcmp(name, "max_k")) {
        if (value < EVS_MAX_K || value > EVS_MAX_K_LARGE) return fail(EVS_EINVAL, "max_k must be in [%d, %d]", EVS_MAX_K, EVS_MAX_K_LARGE);
        g_tune.max_k = (int)value;
    } else {
        return fail(EVS_EINVAL, "unknown option '%s'", name);
    }
    return EVS_OK;
}

extern "C" int evs_get_option(const char* name, int64_t* value) {
    if (!name || !value) return fail(EVS_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(g_tune_mu);
    if (!strcmp(name, "scan_variant")) *value = g_tune.scan_variant;
    else if (!strcmp(name, "tile_rows")) *value = g_tune.tile_rows;
    else if (!strcmp(name, "stages")) *value = g_tune.stages;
    else if (!strcmp(name, "ctas_per_sm")) *value = g_tune.ctas_per_sm;
    else if (!strcmp(name, "tc_min_nq")) *value = g_tune.tc_min_nq;
    else if (!strcmp(name, "tc_pair_min_nq")) *value = g_tune.tc_pair_min_nq;
    else if (!strcmp(name, "tc2_slice_tiles")) *value = g_tc2_slice_tiles;
    else if (!strcmp(name, "tc_heap_max_nq")) *value = g_tc_heap_max_nq;
    else if (!strcmp(name, "tc_heap_pure_max_nq")) *value = g_tc_heap_pure_max_nq;
    else if (!strcmp(name, "tc_inline_pre")) *value = g_tc_inline_pre;
    else if (!strcmp(name, "tc_sample_rows")) *value = g_tc_sample_rows;
    else if (!strcmp(name, "tc_stages")) *value = g_tc_max_stages;
    else if (!strcmp(name, "profile_scans")) *value = g_profile_scans;
    else if (!strcmp(name, "tc_fallbacks")) *value = g_tc_fallbacks.load();  // read-only counter
    else if (!strcmp(name, "exact_reruns")) *value = g_exact_reruns.load();  // read-only counter
    else if (!strcmp(name, "tf32_guard_eps_e6")) *value = g_tf32_guard_eps_e6;
    else if (!strcmp(name, "fuse_finalize")) *value = g_tune.fuse_finalize;
    else if (!strcmp(name, "scan_dynamic")) *value = g_tune.scan_dynamic;
    else if (!strcmp(name, "scan_chunk_groups")) *value = g_tune.scan_chunk_groups;
    else if (!strcmp(name, "exchange_fail_next")) *value = g_exchange_fail_next.load();
    else if (!strcmp(name, "pool_select")) *value = g_tune.pool_select;
    else if (!strcmp(name, "scan_clock")) *value = g_tune.scan_clock;
    else if (!strcmp(name, "x3")) *value = g_tune.x3;
    else if (!strcmp(name, "x3_max_nq")) *value = g_tune.x3_max_nq;
    else if (!strcmp(name, "guard")) *value = g_tune.guard;
    else if (!strcmp(name, "io_threads")) *value = g_io_threads.load();
    else if (!strcmp(name, "small_max_rows")) *value = g_tune.small_max_rows;
    else if (!strcmp(name, "small_fast_cap")) *value = g_tune.small_fast_cap;
    else if (!strcmp(name, "scan_shadow")) *value = g_tune.scan_shadow;
    else if (!strcmp(name, "shadow_min_rows")) *value = g_tune.shadow_min_rows;
    else if (!strcmp(name, "max_k")) *value = g_tune.max_k;
    else return fail(EVS_EINVAL, "unknown option '%s'", name);
    return EVS_OK;
}

// ---------------------------------------------------------------------------------------------
// lifecycle
// ---------------------------------------------------------------------------------------------
extern "C" int evs_index_create(int d, int device, int storage, evs_index** out) {
    if (!out) return fail(EVS_EINVAL, "out is NULL");
    *out = nullptr;
    if (d <= 0) return fail(EVS_EINVAL, "d must be > 0 (got %d)", d);
    if (storage != EVS_STORE_F32 && storage != EVS_STORE_BF16_F32) return fail(EVS_EINVAL, "unknown storage %d", storage);
    int ndev = 0;
    evs_device_count(&ndev);
    if (ndev <= 0) return fail(EVS_ENODEV, "no CUDA device: libevs has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(EVS_EINVAL, "device %d out of range (have %d)", device, ndev);
    int rc = use_device(device);
    if (rc) return rc;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(EVS_ENODEV, "device %d is sm_%d%d; libevs is built for sm_100a only", device, prop.major, prop.minor);
    evs_index* idx = new (std::nothrow) evs_index();
    if (!idx) return fail(EVS_ENOMEM, "out of host memory");
    idx->d = d;
    idx->device = device;
    idx->storage = storage;
    idx->sm_count = prop.multiProcessorCount;
    cudaError_t e = cudaStreamCreateWithFlags(&idx->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&idx->ws_free, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&idx->words), W_WORDS * sizeof(unsigned));
    if (e == cudaSuccess) e = cudaMemset(idx->words, 0, W_WORDS * sizeof(unsigned));
    if (e != cudaSuccess) {
        cudaFree(idx->words);
        if (idx->ws_free) cudaEventDestroy(idx->ws_free);
        if (idx->stream) cudaStreamDestroy(idx->stream);
        delete idx;
        return fail(EVS_ECUDA, "stream/event/workspace creation failed: %s", cudaGetErrorString(e));
    }
    *out = idx;
    return EVS_OK;
}

extern "C" int evs_index_free(evs_index* idx) {
    if (!idx) return EVS_OK;
    cudaSetDevice(idx->device);
    cudaDeviceSynchronize();  // searches may still be in flight on the caller's streams
    cudaFree(idx->xb32);
    cudaFree(idx->xb16);
    cudaFree(idx->xi8);
    cudaFree(idx->xs8);
    cudaFree(idx->q_dev);
    cudaFree(idx->lists);
    cudaFree(idx->I_dev);  // D_dev points into the same allocation
    cudaFree(idx->margins_dev);
    cudaFree(idx->tc_ws);
    cudaFree(idx->tc_overflow);
    cudaFree(idx->words);
    cudaFree(idx->guard_slot);
    cudaFree(idx->guard_lists);
    cudaFree(idx->cta_clock);
    cudaFree(idx->pool);
    cudaFree(idx->lk_ws);
    cudaFreeHost(idx->tc_overflow_pin);
    cudaFreeHost(idx->q_pin);
    cudaFreeHost(idx->I_pin);  // D_pin points into the same allocation
    cudaFreeHost(idx->m_pin);
    cudaFreeHost(idx->done_pin);
    for (auto& pe : idx->prof_events) {
        cudaEventDestroy(pe.first);
        cudaEventDestroy(pe.second);
    }
    if (idx->ws_free) cudaEventDestroy(idx->ws_free);
    if (idx->stream) cudaStreamDestroy(idx->stream);
    delete idx;
    return EVS_OK;
}

#define GETTER(name, type, expr)                                            \
    extern "C" int name(const evs_index* idx, type* out) {                  \
        if (!idx || !out) return fail(EVS_EINVAL, #name ": NULL argument"); \
        *out = (expr);                                                      \
        return EVS_OK;                                                      \
    }
GETTER(evs_index_d, int, idx->d)
GETTER(evs_index_ntotal, int64_t, idx->ntotal)
GETTER(evs_index_device, int, idx->device)
GETTER(evs_index_storage, int, idx->storage)
GETTER(evs_index_id_base, int64_t, idx->id_base)

extern "C" int evs_index_set_id_base(evs_index* idx, int64_t base) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    if (base < 0) return fail(EVS_EINVAL, "id base must be >= 0");
    idx->id_base = base;
    return EVS_OK;
}

static bool shadow_wanted() {
    std::lock_guard<std::mutex> lk(g_tune_mu);
    return g_tune.scan_shadow != 0;
}
// whether an add keeps the int8 scan copy: always for bf16 storage, for fp32 storage while the option "scan_shadow" is on
static bool copy_wanted(const evs_index* idx) { return idx->storage == EVS_STORE_BF16_F32 || shadow_wanted(); }

static void drop_i8_copy(evs_index* idx) {
    cudaFree(idx->xi8);
    cudaFree(idx->xs8);
    idx->xi8 = nullptr;
    idx->xs8 = nullptr;
}
static int alloc_i8_copy(evs_index* idx) {
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&idx->xi8), (size_t)idx->capacity * idx->d);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&idx->xs8), (size_t)idx->capacity * sizeof(float));
    if (e != cudaSuccess) {
        drop_i8_copy(idx);
        return fail(EVS_ENOMEM, "cudaMalloc of the int8 copy failed: %s", cudaGetErrorString(e));
    }
    return EVS_OK;
}

// grow the row storage to hold at least `rows` rows (device-to-device copy of what is there)

static int grow_locked(evs_index* idx, int64_t rows) {
    if (rows <= idx->capacity) return EVS_OK;
    if (rows >= (int64_t)0xFFFFFFFFll) return fail(EVS_ELIMIT, "a shard holds at most 2^32-2 rows");
    const size_t d = (size_t)idx->d;
    float* n32 = nullptr;
    void* n16 = nullptr;
    signed char* n8 = nullptr;
    float* ns8 = nullptr;
    CU(cudaMalloc(reinterpret_cast<void**>(&n32), (size_t)rows * d * sizeof(float)));
    // the derived copies grow with the rows; an index that has no int8 copy yet but holds rows gets it built by its next add
    cudaError_t e = cudaSuccess;
    if (idx->storage == EVS_STORE_BF16_F32) e = cudaMalloc(&n16, (size_t)rows * d * 2);
    if (e == cudaSuccess && (idx->xi8 != nullptr || (idx->ntotal == 0 && copy_wanted(idx)))) {
        e = cudaMalloc(reinterpret_cast<void**>(&n8), (size_t)rows * d);
        if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&ns8), (size_t)rows * sizeof(float));
    }
    if (e != cudaSuccess) {
        cudaFree(n32);
        cudaFree(n16);
        cudaFree(n8);
        cudaFree(ns8);
        return fail(EVS_ENOMEM, "cudaMalloc of the derived row copies failed: %s", cudaGetErrorString(e));
    }
    if (idx->ntotal > 0) {
        e = cudaMemcpyAsync(n32, idx->xb32, (size_t)idx->ntotal * d * sizeof(float), cudaMemcpyDeviceToDevice, idx->stream);
        if (e == cudaSuccess && n16 && idx->xb16)
            e = cudaMemcpyAsync(n16, idx->xb16, (size_t)idx->ntotal * d * 2, cudaMemcpyDeviceToDevice, idx->stream);
        if (e == cudaSuccess && n8 && idx->xi8) {
            e = cudaMemcpyAsync(n8, idx->xi8, (size_t)idx->ntotal * d, cudaMemcpyDeviceToDevice, idx->stream);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(ns8, idx->xs8, (size_t)idx->ntotal * sizeof(float), cudaMemcpyDeviceToDevice, idx->stream);
        }
        const cudaError_t es = cudaStreamSynchronize(idx->stream);  // also on the error path: nothing may still read the old rows
        if (e == cudaSuccess) e = es;
        if (e != cudaSuccess) {
            cudaFree(n32);
            cudaFree(n16);
            cudaFree(n8);
            cudaFree(ns8);
            return fail(EVS_ECUDA, "copying the rows into the grown storage failed: %s", cudaGetErrorString(e));
        }
    }
    cudaFree(idx->xb32);
    cudaFree(idx->xb16);
    cudaFree(idx->xi8);
    cudaFree(idx->xs8);
    idx->xb32 = n32;
    idx->xb16 = n16;
    idx->xi8 = n8;
    idx->xs8 = ns8;
    idx->capacity = rows;
    return EVS_OK;
}

static int grow_for_add_locked(evs_index* idx, int64_t n) {
    int64_t need = idx->ntotal + n;
    if (need <= idx->capacity) return EVS_OK;
    int64_t cap = idx->capacity + idx->capacity / 2;  // 1.5x amortised growth
    if (cap < need) cap = need;
    return grow_locked(idx, cap);
}

// the rows [r0, r0 + n): largest row norm and special elements (the certification bound of the searches, finalize_query)
// and -- when the index keeps them -- the bf16 rows and the int8 copy with its rounding bound, in one pass; then the host
// copies of the flags
static int derive_rows_locked(evs_index* idx, int64_t r0, int64_t n) {
    const size_t d = (size_t)idx->d;
    void* dst16 = idx->xb16 ? reinterpret_cast<unsigned char*>(idx->xb16) + (size_t)r0 * d * 2 : nullptr;
    signed char* dst8 = idx->xi8 ? idx->xi8 + (size_t)r0 * d : nullptr;
    float* scale8 = idx->xs8 ? idx->xs8 + r0 : nullptr;
    CU(launch_row_norm_max(idx->xb32 + (size_t)r0 * d, (long long)n, idx->d, reinterpret_cast<float*>(idx->words + W_MAX_NORM),
                           idx->words + W_SPECIAL, idx->sm_count, idx->stream, dst16, dst8, scale8,
                           reinterpret_cast<float*>(idx->words + W_EMAX)));
    CU(cudaStreamSynchronize(idx->stream));
    unsigned w[W_EMAX - W_MAX_NORM + 1];
    CU(cudaMemcpy(w, idx->words + W_MAX_NORM, sizeof(w), cudaMemcpyDeviceToHost));
    memcpy(&idx->max_norm_host, &w[0], sizeof(float));
    idx->special_host = w[W_SPECIAL - W_MAX_NORM];
    memcpy(&idx->emax_host, &w[W_EMAX - W_MAX_NORM], sizeof(float));
    return EVS_OK;
}

// after new fp32 rows [ntotal, ntotal+n) are in place (enqueued on idx->stream): derive the copies, publish.  An fp32 index
// keeps its int8 scan copy while the option "scan_shadow" is on at add time (built over every row if it has none yet) and
// drops it otherwise.
static int finish_add_locked(evs_index* idx, int64_t n) {
    const bool want8 = copy_wanted(idx);
    int64_t r0 = idx->ntotal;
    if (!want8 && idx->xi8) {
        CU(cudaStreamSynchronize(idx->stream));
        drop_i8_copy(idx);
    } else if (want8 && !idx->xi8) {
        const int rc = alloc_i8_copy(idx);
        if (rc) return rc;
        r0 = 0;
    }
    int rc = derive_rows_locked(idx, r0, idx->ntotal + n - r0);
    if (rc) return rc;
    idx->ntotal += n;
    return EVS_OK;
}

extern "C" int evs_index_reserve(evs_index* idx, int64_t nrows) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    if (nrows < 0) return fail(EVS_EINVAL, "nrows must be >= 0");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    return grow_locked(idx, nrows);
}

extern "C" int evs_index_add(evs_index* idx, int64_t n, const float* x_host) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    if (n < 0) return fail(EVS_EINVAL, "n must be >= 0");
    if (n == 0) return EVS_OK;
    if (!x_host) return fail(EVS_EINVAL, "x is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    if ((rc = grow_for_add_locked(idx, n))) return rc;
    const size_t d = (size_t)idx->d;
    CU(cudaMemcpyAsync(idx->xb32 + (size_t)idx->ntotal * d, x_host, (size_t)n * d * sizeof(float), cudaMemcpyHostToDevice,
                       idx->stream));
    return finish_add_locked(idx, n);
}

extern "C" int evs_index_add_dev(evs_index* idx, int64_t n, const void* x_dev, int dtype, void* stream) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    if (n < 0) return fail(EVS_EINVAL, "n must be >= 0");
    if (n == 0) return EVS_OK;
    if (!x_dev) return fail(EVS_EINVAL, "x is NULL");
    if (dtype != EVS_F32 && dtype != EVS_F16 && dtype != EVS_BF16) return fail(EVS_EINVAL, "bad dtype %d", dtype);
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    if ((rc = grow_for_add_locked(idx, n))) return rc;
    // the producer of x_dev ran on `stream`: order our stream after it
    if ((cudaStream_t)stream != idx->stream) {
        cudaEvent_t ev;
        CU(cudaEventCreateWithFlags(&ev, cudaEventDisableTiming));
        CU(cudaEventRecord(ev, (cudaStream_t)stream));
        CU(cudaStreamWaitEvent(idx->stream, ev, 0));
        CU(cudaEventDestroy(ev));
    }
    const size_t d = (size_t)idx->d;
    float* dst = idx->xb32 + (size_t)idx->ntotal * d;
    if (dtype == EVS_F32)
        CU(cudaMemcpyAsync(dst, x_dev, (size_t)n * d * sizeof(float), cudaMemcpyDeviceToDevice, idx->stream));
    else
        CU(launch_to_f32(x_dev, dtype, dst, (long long)n * idx->d, idx->sm_count, idx->stream));
    return finish_add_locked(idx, n);
}

extern "C" int evs_index_add_synth(evs_index* idx, int64_t n, uint64_t seed, int normalize) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    if (n < 0) return fail(EVS_EINVAL, "n must be >= 0");
    if (n == 0) return EVS_OK;
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    if ((rc = grow_for_add_locked(idx, n))) return rc;
    float* dst = idx->xb32 + (size_t)idx->ntotal * idx->d;
    CU(launch_synth_fill(dst, n, idx->d, seed, idx->id_base + idx->ntotal, idx->sm_count, idx->stream));
    if (normalize) CU(launch_l2_normalize(dst, n, idx->d, EVS_F32, idx->sm_count, idx->stream));
    return finish_add_locked(idx, n);
}

extern "C" int evs_index_add_rows_from(evs_index* dst, const evs_index* src, int64_t n, const int64_t* rows_host) {
    if (!dst || !src) return fail(EVS_EINVAL, "NULL index");
    if (dst == src) return fail(EVS_EINVAL, "source and destination must be different indexes");
    if (n < 0) return fail(EVS_EINVAL, "n must be >= 0");
    if (n == 0) return EVS_OK;
    if (!rows_host) return fail(EVS_EINVAL, "rows is NULL");
    if (dst->d != src->d) return fail(EVS_EINVAL, "dimension mismatch: %d vs %d", dst->d, src->d);
    if (dst->device != src->device) return fail(EVS_EINVAL, "indexes live on different devices (%d, %d)", dst->device, src->device);
    for (int64_t i = 0; i < n; i++)
        if (rows_host[i] < 0 || rows_host[i] >= src->ntotal)
            return fail(EVS_EINVAL, "row %lld out of range [0, %lld)", (long long)rows_host[i], (long long)src->ntotal);
    // both handles: the source must not be grown (its row storage reallocated) while its rows are read
    std::unique_lock<std::mutex> lk(dst->mu, std::defer_lock);
    std::unique_lock<std::mutex> lks(const_cast<evs_index*>(src)->mu, std::defer_lock);
    std::lock(lk, lks);
    for (int64_t i = 0; i < n; i++)  // re-checked under the lock
        if (rows_host[i] >= src->ntotal) return fail(EVS_EINVAL, "row %lld out of range", (long long)rows_host[i]);
    int rc = use_device(dst->device);
    if (rc) return rc;
    if ((rc = grow_for_add_locked(dst, n))) return rc;
    long long* ids_dev = nullptr;
    CU(cudaMalloc(reinterpret_cast<void**>(&ids_dev), (size_t)n * sizeof(long long)));
    cudaError_t e = cudaMemcpyAsync(ids_dev, rows_host, (size_t)n * sizeof(long long), cudaMemcpyHostToDevice, dst->stream);
    if (e == cudaSuccess)
        e = launch_gather_rows(src->xb32, ids_dev, dst->xb32 + (size_t)dst->ntotal * dst->d, n, dst->d, dst->sm_count, dst->stream);
    if (e == cudaSuccess) rc = finish_add_locked(dst, n);  // synchronises the stream
    else cudaStreamSynchronize(dst->stream);
    cudaFree(ids_dev);
    if (e != cudaSuccess) return fail(EVS_ECUDA, "row gather failed: %s", cudaGetErrorString(e));
    return rc;
}

extern "C" int evs_index_get_rows(const evs_index* idx, int64_t row0, int64_t n, float* out_host) {
    if (!idx || (!out_host && n > 0)) return fail(EVS_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);  // a concurrent add() that regrows frees xb32
    if (row0 < 0 || n < 0 || row0 + n > idx->ntotal) return fail(EVS_EINVAL, "rows [%lld,%lld) out of range", (long long)row0, (long long)(row0 + n));
    if (n == 0) return EVS_OK;
    int rc = use_device(idx->device);
    if (rc) return rc;
    CU(cudaMemcpy(out_host, idx->xb32 + (size_t)row0 * idx->d, (size_t)n * idx->d * sizeof(float), cudaMemcpyDeviceToHost));
    return EVS_OK;
}

// ---------------------------------------------------------------------------------------------
// search
// ---------------------------------------------------------------------------------------------
struct SearchOut {
    float* D = nullptr;        // final mode
    int64_t* I = nullptr;
    double* P_scores = nullptr;  // partial mode
    int64_t* P_ids = nullptr;
    const Exchange* x = nullptr;  // exchange mode: the finalise kernel stores the partial into every rank's slot
    // host single-query search of a small shard (evs_index_search; the caller checked small_shard_applies): the query travels in
    // the kernel's parameter block and the kernel raises *done_flag = done_seq behind the results
    const float* q_host = nullptr;
    unsigned* done_flag = nullptr;
    unsigned done_seq = 0;
};

// Which scan serves a batch.  Decided ONCE per search from one snapshot of the tuning options and passed down, so that the
// exchange entry points and the search itself can never disagree (they used to read the options twice).
enum { PATH_GEMV = 0, PATH_TC_HEAP = 1, PATH_TC_SYNC = 2, PATH_LARGE_K = 3 /* k > EVS_MAX_K: evs_large_k.cu */ };
struct PathInfo {
    int kind = PATH_GEMV;
    int kp = 64;
    bool x3 = false;     // PATH_TC_HEAP over fp32 rows: 3xTF32 split scan, `blk` queries per launch set
    bool guard = false;  // results are certified on the device and uncertified queries re-run exactly (fp32 storage, batches)
    int blk = 0;         // PATH_TC_HEAP: queries per launch set
    float err_coef = 0.f;  // scan error bound relative to |q| * max|x| (0 = not certified: bf16 storage)
    float err_trunc = 0.f; // single tf32: the truncation part of the bound, relative to (|q| max|x| + |worst retained score|)
    bool fused = false;  // PATH_GEMV, one query: the scan's last CTA finalises (and, in exchange mode, merges): ONE launch
    bool shadow = false; // ... with the pool kernel over the int8 copy under the bound W_EMAX (exact: evs_scan.cuh)
    bool i8 = false;     // PATH_LARGE_K over the int8 copy: batches of 2..kI8BatchMaxNQ queries, k <= EVS_MAX_K
};

// scan error models, relative to |q| * |x| (DESIGN.md section 2).  fp32 GEMV: 4 partial chains of d/128 FMAs per lane, 3 + 5
// additions to combine: (d/128 + 9) roundings of 2^-24, stated generously.  3xTF32: three dropped terms of 2^-20 each plus
// one fp32 accumulation per MMA (3 per 8 elements of K), each taken as a full 2^-23 truncation of the running sum.
static float gemv_err_coef(int d) { return (float)((d / 32 + 8) * ldexp(1.0, -24)); }
// single tf32 (kind::tf32 on raw fp32 operands: the low 13 mantissa bits of BOTH operands are ignored, i.e. truncation
// towards zero -- tests/test_gpu_tensorcore.py::test_tf32_scan_truncates_its_operands pins that): each product is scaled
// by (1 - a)(1 - b), a, b in [0, 2^-10), so a row is under-estimated by at most (2^-9) * (sum of its positive products)
// <= 2^-10 * (|q||x| + score).  Solving  s <= w + 2^-10 (B + s) + acc  for s gives the coefficient below (the 1/(1 - 2^-10)
// factor folded in).  The products themselves are exact in fp32 (11 x 11 significant bits); what is left is the fp32
// accumulation: one rounding of the running sum per MMA (d/8 of them) and one per product, taken as full 2^-23 truncations.
static float tf32_trunc_coef() { return (float)(ldexp(1.0, -10) * (1.0 + ldexp(1.0, -9))); }
static float tf32_acc_coef(int d) { return (float)((d / 8.0 + 16.0) * ldexp(1.0, -22)); }
static float x3_err_coef(int d) { return (float)(3.0 * ldexp(1.0, -20) + (3.0 * d / 8.0 + 8.0) * ldexp(1.0, -23)); }

static bool takes_tc_path(const evs_index* idx, int64_t nq, const ScanTuning& tune) {
    // TMA row coordinates are int32: shards beyond 2^31 rows (4 TB of bf16 at d = 512: not on this hardware) keep the GEMV scan
    return tune.tc_min_nq > 0 && nq >= tune.tc_min_nq && idx->ntotal >= 65536 && idx->ntotal < ((int64_t)1 << 31) - 1024 &&
           tc_max_queries(idx->d, idx->storage == EVS_STORE_BF16_F32) > 0;
}

// A fused single-query search scans the int8 copy with the pool kernel under its bound (exact for any data) when the copy
// exists (it always holds every row), the index has no subnormal / inf / NaN element, a finite largest norm and a finite
// bound, d is a multiple of 256 up to 1024, and the shard is above the small-shard cut (those are L2-resident and
// latency-bound: scan_small_kernel over the fp32 rows) and holds at least shadow_min_rows rows.
// bf16-storage indexes take the same path; an fp32 index only while the option "scan_shadow" is on.
static bool shadow_applies(const evs_index* idx, int64_t nq, int kp, const ScanTuning& tune) {
    if (nq != 1 || !tune.fuse_finalize || !tune.pool_select || kp != 64 || idx->xi8 == nullptr) return false;
    if (idx->storage != EVS_STORE_BF16_F32 && !tune.scan_shadow) return false;
    if (idx->special_host != 0 || !(idx->emax_host <= FLT_MAX) || !(idx->max_norm_host <= FLT_MAX) ||
        idx->ntotal <= tune.small_max_rows || idx->ntotal < tune.shadow_min_rows)
        return false;
    ScanPlan plan;
    return plan_scan(idx->ntotal, idx->d, SCAN_I8, kp, 1, idx->sm_count, tune, &plan) == cudaSuccess && plan.variant == 1 &&
           plan.threads == 256;
}

// Batches of 2..kI8BatchMaxNQ queries (k <= EVS_MAX_K) scan the int8 copy once per pass of LK_I8_NQ queries, keep
// every row's scan key and re-score exactly every row within 2E of the k-th (evs_large_k.cu: the large-k selection with the
// int8 bound), under the conditions of shadow_applies other than nq == 1.  Exact by construction for fp32 and bf16 storage.
// One pass of up to LK_I8_NQ = 4 queries costs less than the tf32 scan of the fp32 rows (k = 48, x 512: 1.27-1.78 ms against
// 2.91 at 10M rows, 0.20-0.22 against 0.41 at 1.25M, 0.091-0.094 against 0.14 at 300k; profiles/i8_batch_probe.jsonl); two
// passes (5-8 queries) cost as much or more (2.90-3.28 ms at 10M; profiles/i8_batch_probe_pass4.jsonl), so larger batches
// keep the tensor-core scan (scripts/i8_batch_probe.py; one B200, 1000 W).
static const int kI8BatchMaxNQ = LK_I8_NQ;
static bool i8_batch_applies(const evs_index* idx, int64_t nq, int64_t k, const ScanTuning& tune) {
    if (nq < 2 || nq > kI8BatchMaxNQ || k > EVS_MAX_K || idx->xi8 == nullptr) return false;
    if (idx->storage != EVS_STORE_BF16_F32 && !tune.scan_shadow) return false;
    return idx->special_host == 0 && idx->emax_host <= FLT_MAX && idx->max_norm_host <= FLT_MAX && idx->d % 256 == 0 &&
           idx->d <= 1024 && idx->ntotal > tune.small_max_rows && idx->ntotal >= tune.shadow_min_rows &&
           idx->ntotal < ((int64_t)1 << 32) - 32 && i8_batch_grid(idx->d / 256, idx->sm_count) > 0;
}

static PathInfo plan_path(const evs_index* idx, int64_t nq, int64_t k, const ScanTuning& tune, bool allow_tc) {
    PathInfo pi;
    if (k > EVS_MAX_K) {  // whatever nq, storage or tensor-core routing say: the fp32 rows, exact by construction
        pi.kind = PATH_LARGE_K;
        return pi;
    }
    if (i8_batch_applies(idx, nq, k, tune)) {
        pi.kind = PATH_LARGE_K;
        pi.i8 = true;
        return pi;
    }
    const bool bf16 = idx->storage == EVS_STORE_BF16_F32;
    pi.kp = pick_kp(k);
    pi.err_coef = bf16 ? 0.f : gemv_err_coef(idx->d);
    if (!allow_tc || !takes_tc_path(idx, nq, tune)) {
        if (nq == 1 && tune.fuse_finalize && idx->ntotal > 0) {
            pi.shadow = shadow_applies(idx, nq, pi.kp, tune);
            if (pi.shadow) pi.err_coef = 0.f;  // exact by construction: nothing to certify
            ScanPlan plan;
            pi.fused = plan_scan(idx->ntotal, idx->d, pi.shadow ? SCAN_I8 : bf16, pi.kp, 1, idx->sm_count, tune, &plan) == cudaSuccess &&
                       plan.variant == 1;
        }
        return pi;
    }
    // the device-side guard re-runs with the vectorised fp32 GEMV scan: dimensions it does not cover are certified and
    // counted (evs_index_guard_stats) but not re-run
    ScanPlan gplan;
    ScanTuning gt = tune;
    gt.scan_variant = 1;
    const bool gemv_ok = plan_scan(idx->ntotal, idx->d, 0, 128, 1, idx->sm_count, gt, &gplan) == cudaSuccess && gplan.variant == 1;
    pi.guard = !bf16 && tune.guard != 0 && gemv_ok;
    // small fp32 batches: 3xTF32 on-chip-heap blocks (fp32-class scan error, no host synchronisation)
    const int x3max = (!bf16 && tune.x3 && pi.kp == 64) ? tc_x3_max_queries(idx->d) : 0;
    if (x3max > 0 && nq <= tune.x3_max_nq && nq <= g_tc_heap_max_nq) {
        pi.kind = PATH_TC_HEAP;
        pi.x3 = true;
        pi.blk = x3max;
        pi.err_coef = x3_err_coef(idx->d);
        return pi;
    }
    if (!bf16) {
        if (g_tf32_guard_eps_e6 > 0) {
            pi.err_coef = (float)g_tf32_guard_eps_e6 * 1e-6f;  // statistical override (option), not a proof
        } else {
            pi.err_coef = tf32_acc_coef(idx->d);
            pi.err_trunc = tf32_trunc_coef();
        }
    } else {
        pi.err_coef = 0.f;
        pi.guard = false;
    }
    pi.kind = PATH_TC_SYNC;
    if (nq <= kTcQueryChunk) {
        const bool pair = tune.tc_pair_min_nq > 0 && (nq >= tune.tc_pair_min_nq || nq > tc_max_queries(idx->d, bf16)) &&
                          tc2_max_half(idx->d, bf16) > 0 && idx->sm_count >= 2;
        TcPlan pl;
        if (!pair && tc_plan(idx->ntotal, idx->d, bf16, (int)nq, pi.kp, idx->sm_count, 0, &pl) == cudaSuccess && pl.heap) {
            pi.kind = PATH_TC_HEAP;
            pi.blk = (int)nq;
        }
    }
    return pi;
}

// Scan launches that synchronise their own grid (the in-launch threshold pre-pass) need every CTA resident: two of them from
// different streams (two handles searched concurrently) could each hold part of the SMs and wait forever.  They are therefore
// ordered one after the other per device: every such search records an event behind its last launch, and a search on
// another stream than the previous one first waits for that event.  (The event, not the previous stream, is what is kept:
// a stream may have been destroyed by its owner in the meantime.)
static std::mutex g_bar_mu;
static cudaStream_t g_bar_stream[16];
static bool g_bar_has[16];
static cudaEvent_t g_bar_event[16];
static int barrier_scan_order(int device, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_bar_mu);
    const int dv = device & 15;
    if (g_bar_has[dv] && g_bar_stream[dv] != st) CU(cudaStreamWaitEvent(st, g_bar_event[dv], 0));
    return EVS_OK;
}
static int barrier_scan_done(int device, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(g_bar_mu);
    const int dv = device & 15;
    if (!g_bar_event[dv]) CU(cudaEventCreateWithFlags(&g_bar_event[dv], cudaEventDisableTiming));
    CU(cudaEventRecord(g_bar_event[dv], st));
    g_bar_stream[dv] = st;
    g_bar_has[dv] = true;
    return EVS_OK;
}

static const int kGuardCap = 32;  // queries one device-side guard re-run can take (the on-chip-heap batches are <= 32 queries)
static const int kRepairCap = 256;  // threshold-scan batches up to this size repair overflowed / uncertified queries on the device
                                    // too (no host synchronisation); larger batches read the flags on the host

template <typename T>
static int ensure_pinned(T** ptr, size_t* cap, size_t need_elems);

// The workspace of a handle is used by one search at a time.  Searches enqueued on the SAME stream are ordered by the stream
// (no event between them: an event record would also break the programmatic overlap of consecutive searches); a search on
// another stream first waits for everything enqueued on the previous one.
static int ws_acquire(evs_index* idx, cudaStream_t st) {
    if (idx->have_last_stream && idx->last_stream != st) {
        cudaError_t e = cudaEventRecord(idx->ws_free, idx->last_stream);
        if (e == cudaSuccess) e = cudaStreamWaitEvent(st, idx->ws_free, 0);
        if (e != cudaSuccess) {  // the previous stream is gone: be safe
            cudaGetLastError();
            CU(cudaDeviceSynchronize());
        }
    }
    idx->last_stream = st;
    idx->have_last_stream = true;
    return EVS_OK;
}

static FinalizeParams make_finalize(evs_index* idx, const void* lists, int L, int kp, const float* xq, int64_t k, const SearchOut& out,
                                    int64_t c0, int64_t nq_total, float err_coef, float err_trunc = 0.f) {
    FinalizeParams f;
    f.lists = reinterpret_cast<const unsigned long long*>(lists);
    f.L = L;
    f.kp = kp;
    f.xb = idx->xb32;
    f.xb_is_bf16 = 0;
    f.xq = xq;
    f.d = idx->d;
    f.k = (int)k;
    f.id_base = idx->id_base;
    f.D = out.D ? out.D + (size_t)c0 * k : nullptr;
    f.I = out.I ? reinterpret_cast<long long*>(out.I + (size_t)c0 * k) : nullptr;
    f.P_scores = out.P_scores ? out.P_scores + (size_t)c0 * k : nullptr;
    f.P_ids = out.P_ids ? reinterpret_cast<long long*>(out.P_ids + (size_t)c0 * k) : nullptr;
    f.margins = idx->margins_dev + c0;
    if (out.x) {
        f.x = *out.x;
        f.x.nq_total = nq_total;
        f.x.q_off = c0;
    }
    f.err_coef = err_coef;
    f.err_trunc = err_trunc;
    f.max_norm = reinterpret_cast<const float*>(idx->words + W_MAX_NORM);
    f.special = idx->words + W_SPECIAL;
    f.uncertified = reinterpret_cast<unsigned long long*>(idx->words + W_UNCERT);
    return f;
}

struct ProfileScope {  // optional CUDA event pair around the scan launches of one search (option "profile_scans")
    std::pair<cudaEvent_t, cudaEvent_t>* pe = nullptr;
    int begin(evs_index* idx, int profile, cudaStream_t st) {
        if (!profile || idx->prof_used >= 65536) return EVS_OK;
        if (idx->prof_used == idx->prof_events.size()) {
            cudaEvent_t a = nullptr, b = nullptr;
            CU(cudaEventCreate(&a));
            CU(cudaEventCreate(&b));
            idx->prof_events.emplace_back(a, b);
        }
        pe = &idx->prof_events[idx->prof_used++];
        CU(cudaEventRecord(pe->first, st));
        return EVS_OK;
    }
    int end(cudaStream_t st) {
        if (pe) CU(cudaEventRecord(pe->second, st));
        return EVS_OK;
    }
};

// one query over a shard of up to small_max_rows rows (k <= 48, fused pool selection): scan_small_kernel (evs_scan.cuh)
static bool small_shard_applies(const evs_index* idx, const ScanTuning& tune, int kp, const ScanPlan& plan) {
    return tune.pool_select && kp == 64 && tune.small_max_rows > 0 && idx->ntotal > 0 && idx->ntotal <= tune.small_max_rows &&
           plan.variant == 1 && plan.threads == 256 && (size_t)idx->ntotal <= scan_pool_key_slots(scan_pool_words(plan));
}

static int search_enqueue_locked(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, const SearchOut& out, cudaStream_t st,
                                 const ScanTuning& tune, const PathInfo& pi, bool scan_only = false, int kp_override = 0);

static TcArgs make_tc_args(evs_index* idx, const float* xq, int64_t nq, void* lists, int* overflow_out) {
    const bool bf16 = idx->storage == EVS_STORE_BF16_F32;
    TcArgs a;
    a.xb = bf16 ? idx->xb16 : (const void*)idx->xb32;
    a.is_bf16 = bf16;
    a.n = idx->ntotal;
    a.d = idx->d;
    a.xq = xq;
    a.nq = (int)nq;
    a.lists = lists;
    a.overflow_out = overflow_out;
    a.tmaps = &idx->tmaps;
    a.bar = idx->words + W_BAR;
    return a;
}

// Small batches served from on-chip heaps (MODE_HEAP): one launch set per block of pi.blk queries (the whole batch, or the
// 3xTF32 block size for fp32 rows), ONE finalise over the per-CTA lists of all queries, and -- fp32 storage -- the
// device-side guard: the finalise certifies each result against the scan's error bound, uncertified queries are queued,
// an fp32 GEMV re-run (k' = 128) walks the queue inside one launch that returns at once when the queue is empty, and a
// predicated second finalise overwrites their results.  No host synchronisation anywhere.
static int search_tc_heap_locked(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, const SearchOut& out, cudaStream_t st,
                                 const ScanTuning& tune, const PathInfo& pi, bool scan_only, int profile) {
    const int kp = 64;
    const bool bf16 = idx->storage == EVS_STORE_BF16_F32;
    const int blk = pi.blk;
    TcPlan pl0;
    CU(tc_plan(idx->ntotal, idx->d, bf16, (int)(nq < blk ? nq : blk), kp, idx->sm_count, pi.x3, &pl0));
    if (!pl0.heap) return fail(EVS_ECUDA, "internal: the on-chip-heap path was planned for a batch it cannot serve");
    const int grid = pl0.grid;
    int rc = ensure_dev(&idx->tc_ws, &idx->tc_ws_cap, tc_workspace_bytes(pl0));
    if (rc) return rc;
    if ((rc = ensure_dev(reinterpret_cast<unsigned long long**>(&idx->lists), &idx->lists_cap, (size_t)nq * grid * kp))) return rc;
    if ((rc = ensure_dev(&idx->margins_dev, &idx->margins_cap, (size_t)nq))) return rc;
    idx->last_nq = nq;
    const bool guard = pi.guard && !scan_only && out.x == nullptr && nq <= kGuardCap;
    ScanPlan gp;
    ScanTuning gt = tune;
    gt.scan_variant = 1;
    const int gq = max_queries_per_pass(idx->d, 0);
    if (guard) {
        CU(plan_scan(idx->ntotal, idx->d, 0, 128, gq, idx->sm_count, gt, &gp));
        if (gp.variant != 1) return fail(EVS_ECUDA, "internal: no vectorised GEMV scan for the guard at d = %d", idx->d);
        if ((rc = ensure_dev(&idx->guard_slot, &idx->guard_slot_cap, (size_t)(nq > kGuardCap ? nq : kGuardCap) * 2))) return rc;
        if ((rc = ensure_dev(&idx->guard_lists, &idx->guard_lists_cap, (size_t)kGuardCap * gp.grid * 128))) return rc;
    }
    if (pl0.inline_pre) {
        if ((rc = barrier_scan_order(idx->device, st))) return rc;
        idx->bar_used = true;
    }
    ProfileScope prof;
    if ((rc = prof.begin(idx, profile, st))) return rc;
    for (int64_t b0 = 0; b0 < nq; b0 += blk) {
        const int64_t cn = (nq - b0) < blk ? (nq - b0) : blk;
        TcPlan plb;
        CU(tc_plan(idx->ntotal, idx->d, bf16, (int)cn, kp, idx->sm_count, pi.x3, &plb));
        if (!plb.heap || plb.grid != grid || tc_workspace_bytes(plb) > idx->tc_ws_cap)
            return fail(EVS_ECUDA, "internal: inconsistent plans for the blocks of one on-chip-heap batch");
        TcArgs a = make_tc_args(idx, q_dev + (size_t)b0 * idx->d, cn,
                                reinterpret_cast<unsigned long long*>(idx->lists) + (size_t)b0 * grid * kp, nullptr);
        CU(tc_scan_block(a, plb, idx->tc_ws, st));
    }
    if ((rc = prof.end(st))) return rc;
    if (scan_only) return EVS_OK;
    FinalizeParams f = make_finalize(idx, idx->lists, grid, kp, q_dev, k, out, 0, nq, pi.err_coef, pi.err_trunc);
    int* gslot = idx->guard_slot;
    int* gqueue = idx->guard_slot ? idx->guard_slot + (nq > kGuardCap ? nq : kGuardCap) : nullptr;
    int* gcount = nullptr;
    if (guard) {
        const int par = (int)(++idx->guard_seq & 1ull);
        gcount = reinterpret_cast<int*>(idx->words) + W_GUARD_COUNT0 + par;
        f.guard_count = gcount;
        f.guard_count_next = reinterpret_cast<int*>(idx->words) + W_GUARD_COUNT0 + (par ^ 1);
        f.guard_slot = gslot;
        f.guard_q = gqueue;
        f.guard_cap = kGuardCap;
    }
    CU(launch_finalize(f, nq, st));
    if (!guard) return EVS_OK;
    ScanArgs ga;
    ga.xb = idx->xb32;
    ga.is_bf16 = 0;
    ga.n = idx->ntotal;
    ga.d = idx->d;
    ga.xq = q_dev;
    ga.q0 = 0;
    ga.nq_pass = gq;
    ga.lists = idx->guard_lists;
    ga.kp = 128;
    ga.qmap = gqueue;
    ga.nactive = gcount;
    ga.qcap = kGuardCap;
    CU(launch_scan(ga, &gp, st));
    FinalizeParams f2 = make_finalize(idx, idx->guard_lists, gp.grid, 128, q_dev, k, out, 0, nq, gemv_err_coef(idx->d));
    f2.pred_slot = gslot;
    f2.guard_cap = kGuardCap;
    f2.reruns = reinterpret_cast<unsigned long long*>(idx->words + W_RERUNS);
    CU(launch_finalize(f2, nq, st));
    return EVS_OK;
}

// Tensor-core path for larger batches: one database pass per block of up to tc_max_queries queries (one-CTA kernel) or the
// CTA-pair kernel.  These scans select by thresholds into bounded candidate buffers; a query whose buffers overflowed
// (adversarial data) -- and, for fp32 storage, a query the finalise could not certify against the scan's error bound -- is
// re-run through the fp32 GEMV scan with k' = 128.  Both flags come back in ONE host synchronisation.
static int search_tc_sync_locked(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, const SearchOut& out, cudaStream_t st,
                                 const ScanTuning& tune, const PathInfo& pi, bool scan_only, int profile) {
    const int kp = pi.kp;
    const bool bf16 = idx->storage == EVS_STORE_BF16_F32;
    const int pair_min_nq = tune.tc_pair_min_nq;
    if (out.x) return fail(EVS_ECUDA, "internal: exchange-mode search took a path that needs the host");
    // batches of pair_min_nq or more queries go through the CTA-pair kernel (N up to 256 per MMA, L2-shared slices)
    const bool can_pair = pair_min_nq > 0 && tc2_max_half(idx->d, bf16) > 0 && idx->sm_count >= 2;
    // ... and so do batches that would need more than one pass of the one-CTA kernel (fp32 rows: 64 queries per pass)
    const int one_cta_max = tc_max_queries(idx->d, bf16);
    auto use_pair = [&](int64_t cn) { return can_pair && (cn >= pair_min_nq || cn > one_cta_max); };
    const int64_t first = nq < kTcQueryChunk ? nq : kTcQueryChunk;
    size_t ws_need = 0;
    if (use_pair(first)) {
        Tc2Plan p2;
        CU(tc2_plan(idx->ntotal, idx->d, bf16, (int)first, kp, idx->sm_count, &p2));
        ws_need = tc2_workspace_bytes(p2);
    }
    const int64_t last = nq % kTcQueryChunk;  // a shorter final chunk may take the other kernel
    size_t lists_need = (size_t)first * kp;
    if (!use_pair(first) || (last && !use_pair(last))) {
        TcPlan pl;
        const int64_t cn1 = use_pair(first) ? last : first;
        CU(tc_plan(idx->ntotal, idx->d, bf16, (int)cn1, kp, idx->sm_count, 0, &pl));
        if (tc_workspace_bytes(pl) > ws_need) ws_need = tc_workspace_bytes(pl);
        if (pl.heap && (size_t)cn1 * pl.grid * kp > lists_need) lists_need = (size_t)cn1 * pl.grid * kp;  // one list per CTA
    }
    int rc = ensure_dev(&idx->tc_ws, &idx->tc_ws_cap, ws_need);
    if (rc) return rc;
    if ((rc = ensure_dev(&idx->tc_overflow, &idx->tc_overflow_cap, (size_t)nq))) return rc;
    if ((rc = ensure_dev(reinterpret_cast<unsigned long long**>(&idx->lists), &idx->lists_cap, lists_need))) return rc;
    if ((rc = ensure_dev(&idx->margins_dev, &idx->margins_cap, (size_t)nq))) return rc;
    const bool guard = pi.guard && !scan_only;
    // Batches of up to kRepairCap queries repair themselves on the device: the finalise queues every query whose candidate
    // buffers overflowed (adversarial data) or -- fp32 storage -- whose result did not clear the scan's error bound, an fp32
    // GEMV re-run (k' = 128) walks the queue in one launch that returns at once when the queue is empty, and a predicated
    // second finalise overwrites those results.  The search never touches the host: the device API stays asynchronous.
    ScanPlan gp;
    ScanTuning gt = tune;
    gt.scan_variant = 1;
    const int gq = max_queries_per_pass(idx->d, 0);
    const bool dev_repair = !scan_only && nq <= kRepairCap &&
                            plan_scan(idx->ntotal, idx->d, 0, 128, gq, idx->sm_count, gt, &gp) == cudaSuccess && gp.variant == 1;
    if ((guard || dev_repair) && (rc = ensure_dev(&idx->guard_slot, &idx->guard_slot_cap, (size_t)(nq > kGuardCap ? nq : kGuardCap) * 2))) return rc;
    if (dev_repair && (rc = ensure_dev(&idx->guard_lists, &idx->guard_lists_cap, (size_t)nq * gp.grid * 128))) return rc;
    int* gcount = nullptr;
    int* gcount_next = nullptr;
    if (guard || dev_repair) {
        const int par = (int)(++idx->guard_seq & 1ull);
        gcount = reinterpret_cast<int*>(idx->words) + W_GUARD_COUNT0 + par;
        gcount_next = reinterpret_cast<int*>(idx->words) + W_GUARD_COUNT0 + (par ^ 1);
    }
    idx->last_nq = nq;
    for (int64_t c0 = 0; c0 < nq; c0 += kTcQueryChunk) {
        const int64_t cn = (nq - c0) < kTcQueryChunk ? (nq - c0) : kTcQueryChunk;
        ProfileScope prof;
        if ((rc = prof.begin(idx, profile, st))) return rc;
        int lists_per_query = 1;
        // the finalise parameters first: the threshold scans end in a gather kernel that finalises the query itself
        FinalizeParams f = make_finalize(idx, idx->lists, 1, kp, q_dev + (size_t)c0 * idx->d, k, out, c0, nq, pi.err_coef, pi.err_trunc);
        int* gqueue = idx->guard_slot ? idx->guard_slot + (nq > kGuardCap ? nq : kGuardCap) : nullptr;
        if (dev_repair) {  // one chunk (nq <= kRepairCap): queue on the device, re-run below
            f.guard_count = gcount;
            f.guard_count_next = gcount_next;
            f.guard_slot = idx->guard_slot;
            f.guard_q = gqueue;
            f.guard_cap = (int)nq;
            f.overflow = idx->tc_overflow;  // the fused gather reads the scan's own flags instead
        } else if (guard) {  // certification only: the flags are read by the host below, nothing is re-run on the device
            f.guard_count = gcount;
            f.guard_count_next = gcount_next;
            f.guard_slot = idx->guard_slot + c0;
            f.guard_q = gqueue;
            f.guard_cap = 0;  // slots are not used: every uncertified query gets guard_slot = -2
        }
        bool fused_finalize = false;
        {
            TcArgs a = make_tc_args(idx, q_dev + (size_t)c0 * idx->d, cn, idx->lists, idx->tc_overflow + c0);
            if (use_pair(cn)) {
                Tc2Plan plb;
                CU(tc2_plan(idx->ntotal, idx->d, bf16, (int)cn, kp, idx->sm_count, &plb));
                if (tc2_workspace_bytes(plb) > idx->tc_ws_cap) return fail(EVS_ECUDA, "internal: tensor-core workspace too small");
                if (!scan_only) {
                    a.fin = &f;
                    fused_finalize = true;
                }
                CU(tc2_scan(a, plb, idx->tc_ws, st));
            } else {
                TcPlan plb;  // same workspace bound: cn <= the chunk the workspace was sized for
                CU(tc_plan(idx->ntotal, idx->d, bf16, (int)cn, kp, idx->sm_count, 0, &plb));
                if (tc_workspace_bytes(plb) > idx->tc_ws_cap) return fail(EVS_ECUDA, "internal: tensor-core workspace too small");
                if (plb.inline_pre) {
                    if ((rc = barrier_scan_order(idx->device, st))) return rc;
                    idx->bar_used = true;
                }
                if (plb.heap) {
                    lists_per_query = plb.grid;
                    f.L = plb.grid;
                    if ((size_t)cn * plb.grid * kp > idx->lists_cap) return fail(EVS_ECUDA, "internal: list workspace too small");
                } else if (!scan_only) {
                    a.fin = &f;
                    fused_finalize = true;
                }
                CU(tc_scan_block(a, plb, idx->tc_ws, st));
            }
        }
        if ((rc = prof.end(st))) return rc;
        if (scan_only) continue;
        (void)lists_per_query;
        if (!fused_finalize) {
            CU(launch_finalize(f, cn, st));
        }
        if (dev_repair) {
            ScanArgs ga;
            ga.xb = idx->xb32;
            ga.is_bf16 = 0;
            ga.n = idx->ntotal;
            ga.d = idx->d;
            ga.xq = q_dev;
            ga.q0 = 0;
            ga.nq_pass = gq;
            ga.lists = idx->guard_lists;
            ga.kp = 128;
            ga.qmap = gqueue;
            ga.nactive = gcount;
            ga.qcap = (int)nq;
            CU(launch_scan(ga, &gp, st));
            FinalizeParams f2 = make_finalize(idx, idx->guard_lists, gp.grid, 128, q_dev, k, out, 0, nq, gemv_err_coef(idx->d));
            f2.pred_slot = idx->guard_slot;
            f2.guard_cap = (int)nq;
            f2.reruns = reinterpret_cast<unsigned long long*>(idx->words + W_RERUNS);
            CU(launch_finalize(f2, nq, st));
            return EVS_OK;
        }
    }
    if (scan_only) return EVS_OK;
    // exactness guards: re-run overflowed and uncertified queries with the fp32 GEMV scan
    const size_t words = guard ? 2 * (size_t)nq : (size_t)nq;
    if ((rc = ensure_pinned(&idx->tc_overflow_pin, &idx->tc_overflow_pin_cap, words))) return rc;
    CU(cudaMemcpyAsync(idx->tc_overflow_pin, idx->tc_overflow, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (guard)
        CU(cudaMemcpyAsync(idx->tc_overflow_pin + nq, idx->guard_slot, (size_t)nq * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    ScanTuning t1 = tune;
    PathInfo p1 = plan_path(idx, 1, k, t1, false);
    for (int64_t q = 0; q < nq; q++) {
        const bool over = idx->tc_overflow_pin[q] != 0;
        const bool uncert = guard && idx->tc_overflow_pin[nq + q] != -1;
        if (!over && !uncert) continue;
        if (over) g_tc_fallbacks.fetch_add(1);
        else g_exact_reruns.fetch_add(1);
        SearchOut o1;
        o1.D = out.D ? out.D + (size_t)q * k : nullptr;
        o1.I = out.I ? out.I + (size_t)q * k : nullptr;
        o1.P_scores = out.P_scores ? out.P_scores + (size_t)q * k : nullptr;
        o1.P_ids = out.P_ids ? out.P_ids + (size_t)q * k : nullptr;
        float* keep = idx->margins_dev;
        idx->margins_dev = keep + q;  // the re-run writes this query's margin in place
        rc = search_enqueue_locked(idx, 1, q_dev + (size_t)q * idx->d, k, o1, st, t1, p1, false, k <= 112 ? 128 : 0);
        idx->margins_dev = keep;
        idx->last_nq = nq;
        if (rc) return rc;
    }
    return EVS_OK;
}

// k > EVS_MAX_K (evs_large_k.cu): passes of max_queries_per_pass(d) queries over the fp32 rows, each a score scan that keeps
// every row's scan key, a radix select of the k-th key, the window cut at 2E below it, a grid-wide canonical re-score of the
// window and the ranking.  Exact by construction (DESIGN.md section 2): nothing is certified afterwards or re-run.
// With i8 (plan_path: batches of 2..kI8BatchMaxNQ queries) the score scan reads the int8 copy and E is its bound.
static int search_large_k_locked(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, const SearchOut& out, cudaStream_t st,
                                 const ScanTuning& tune, bool scan_only, int profile, bool i8) {
    if (out.x) return fail(EVS_ECUDA, "internal: a large-k search writes its partial to staging, not to the exchange slots");
    const int qpp = i8 ? LK_I8_NQ : max_queries_per_pass(idx->d, 0);
    ScanTuning gt = tune;
    gt.scan_variant = 1;  // the direct-load grid (the ring variant keeps lists, not keys)
    ScanPlan plan;
    if (i8) {
        plan.variant = 1;
        plan.nv = idx->d / 256;
        plan.grid = i8_batch_grid(plan.nv, idx->sm_count);
        if (plan.grid < 1) return fail(EVS_ECUDA, "int8 batch scan: no resident CTA");
    } else {
        CU(plan_scan(idx->ntotal, idx->d, SCAN_F32, 64, qpp, idx->sm_count, gt, &plan));
    }
    const size_t npad = ((size_t)idx->ntotal + 31) & ~(size_t)31;
    const size_t arrays = (size_t)qpp * npad * 16;  // S, C (u32) and R (u64)
    const size_t state = large_k_state_bytes(qpp);
    int rc = ensure_dev(&idx->lk_ws, &idx->lk_ws_cap, arrays + state + 16);
    if (rc) return rc;
    unsigned char* ws = idx->lk_ws;
    idx->lk_stats = reinterpret_cast<unsigned*>(ws + arrays + state);
    // the int8 batches report their largest |C| where the single-query searches of the copy do (W_LASTC)
    unsigned* stats = i8 ? idx->words + W_LASTC : idx->lk_stats;
    if (!scan_only) {
        if ((rc = ensure_dev(&idx->margins_dev, &idx->margins_cap, (size_t)nq))) return rc;
        idx->last_nq = nq;
        if (!i8) idx->lk_searches++;
        CU(cudaMemsetAsync(stats, 0, sizeof(unsigned), st));
    }
    LargeKArgs a;
    a.xb = idx->xb32;
    a.n = idx->ntotal;
    a.npad = (long long)npad;
    a.d = idx->d;
    a.nv = plan.variant == 1 ? plan.nv : 0;
    a.grid = plan.grid;
    a.k = (int)k;
    a.fast_widen = idx->special_host == 0u;
    a.all_rows = idx->special_host != 0u;  // subnormal / inf / NaN elements: the fp32 scan has no bound, every row is a candidate
    a.err_coef = gemv_err_coef(idx->d);
    a.max_norm = reinterpret_cast<const float*>(idx->words + W_MAX_NORM);
    a.S = reinterpret_cast<unsigned*>(ws);
    a.C = a.S + (size_t)qpp * npad;
    a.R = reinterpret_cast<unsigned long long*>(a.C + (size_t)qpp * npad);
    a.hist = reinterpret_cast<unsigned*>(ws + arrays);
    a.st = reinterpret_cast<LargeKQuery*>(a.hist + (size_t)3 * qpp * LK_BINS);
    a.stats = stats;
    a.id_base = idx->id_base;
    if (i8) {
        a.xi8 = idx->xi8;
        a.xs8 = idx->xs8;
        a.emax = reinterpret_cast<const float*>(idx->words + W_EMAX);
    }
    for (int64_t p0 = 0; p0 < nq; p0 += qpp) {
        a.nq_pass = (int)((nq - p0) < qpp ? (nq - p0) : qpp);
        a.xq = q_dev + (size_t)p0 * idx->d;
        a.D = out.D ? out.D + (size_t)p0 * k : nullptr;
        a.I = out.I ? reinterpret_cast<long long*>(out.I + (size_t)p0 * k) : nullptr;
        a.P_scores = out.P_scores ? out.P_scores + (size_t)p0 * k : nullptr;
        a.P_ids = out.P_ids ? reinterpret_cast<long long*>(out.P_ids + (size_t)p0 * k) : nullptr;
        a.margins = scan_only ? nullptr : idx->margins_dev + p0;
        CU(cudaMemsetAsync(a.hist, 0, state, st));
        ProfileScope prof;
        if ((rc = prof.begin(idx, profile, st))) return rc;
        CU(launch_large_k_scan(a, st));
        if ((rc = prof.end(st))) return rc;
        if (!scan_only) CU(launch_large_k_rest(a, idx->sm_count, st));
        if (i8) idx->i8_batch_passes++;
    }
    return EVS_OK;
}

static int search_enqueue_locked(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, const SearchOut& out, cudaStream_t st,
                                 const ScanTuning& tune, const PathInfo& pi, bool scan_only, int kp_override) {
    int profile;
    {
        std::lock_guard<std::mutex> lk(g_tune_mu);
        profile = g_profile_scans && !scan_only;
    }
    if (pi.kind == PATH_LARGE_K) return search_large_k_locked(idx, nq, q_dev, k, out, st, tune, scan_only, profile, pi.i8);
    if (pi.kind == PATH_TC_HEAP || pi.kind == PATH_TC_SYNC) {
        idx->bar_used = false;
        int rc = pi.kind == PATH_TC_HEAP ? search_tc_heap_locked(idx, nq, q_dev, k, out, st, tune, pi, scan_only, profile)
                                         : search_tc_sync_locked(idx, nq, q_dev, k, out, st, tune, pi, scan_only, profile);
        if (idx->bar_used) {  // also on failure: whatever was launched is ordered before the next such search
            const int rc2 = barrier_scan_done(idx->device, st);
            if (!rc) rc = rc2;
        }
        return rc;
    }
    const int kp = kp_override ? kp_override : pi.kp;
    const bool bf16 = idx->storage == EVS_STORE_BF16_F32;
    const bool shadow = pi.shadow && kp_override == 0;
    const bool scan_bf16 = bf16 && !shadow && kp_override == 0;  // an exact re-run always scans the fp32 rows
    const void* scan_rows = shadow ? (const void*)idx->xi8 : scan_bf16 ? idx->xb16 : (const void*)idx->xb32;
    const int qpp = shadow ? 1 : max_queries_per_pass(idx->d, scan_bf16);
    ScanPlan plan;
    CU(plan_scan(idx->ntotal, idx->d, shadow ? SCAN_I8 : scan_bf16, kp, qpp, idx->sm_count, tune, &plan));
    const int64_t chunk_cap = nq < kQueryChunk ? nq : kQueryChunk;
    int rc = ensure_dev(reinterpret_cast<unsigned long long**>(&idx->lists), &idx->lists_cap, (size_t)chunk_cap * plan.grid * kp);
    if (rc) return rc;
    if (kp_override == 0) {
        if ((rc = ensure_dev(&idx->margins_dev, &idx->margins_cap, (size_t)nq))) return rc;
        idx->last_nq = nq;
    }
    // single-query searches (what the app issues, oldapp.py:2005): the scan's last CTA finalises -- one launch in all
    const bool fused = (kp_override ? (tune.fuse_finalize && nq == 1 && plan.variant == 1) : pi.fused) && !scan_only;
    if (out.x && out.x->merge_D && !fused) return fail(EVS_ECUDA, "internal: the exchange expected a fused single-query search");
    const float err_coef = (scan_bf16 || shadow) ? 0.f : gemv_err_coef(idx->d);
    if (shadow && !(fused && tune.pool_select && kp == 64))
        return fail(EVS_ECUDA, "internal: the int8 scan copy is searched by the fused pool kernel only");

    for (int64_t c0 = 0; c0 < nq; c0 += kQueryChunk) {
        const int64_t cn = (nq - c0) < kQueryChunk ? (nq - c0) : kQueryChunk;
        const float* qc = q_dev + (size_t)c0 * idx->d;
        ProfileScope prof;
        if ((rc = prof.begin(idx, profile, st))) return rc;
        FinalizeParams f = make_finalize(idx, idx->lists, plan.grid, kp, qc, k, out, c0, nq, err_coef);
        if (shadow) {
            f.shadow_emax = reinterpret_cast<const float*>(idx->words + W_EMAX);
            f.wide = idx->words + W_WIDE;  // W_LASTC follows
        }
        for (int64_t p0 = 0; p0 < cn; p0 += qpp) {
            ScanArgs a;
            a.xb = scan_rows;
            a.xs = shadow ? idx->xs8 : nullptr;
            a.is_bf16 = scan_bf16;
            a.is_i8 = shadow;
            a.n = idx->ntotal;
            a.d = idx->d;
            a.xq = qc;
            a.q0 = (int)p0;
            a.nq_pass = (int)((cn - p0) < qpp ? (cn - p0) : qpp);
            a.lists = idx->lists;
            a.kp = kp;
            if (fused) {
                a.fuse = &f;
                a.ticket = idx->words + W_TICKET;
                if (tune.pool_select && kp == 64) {
                    // under the lowered thresholds of the int8 scan a near-tie burst may send any number of keys to the pool:
                    // room for one per row (each row's key enters the pool at most once), then the window pass's list
                    const size_t need = scan_pool_words(plan) + (shadow ? (size_t)idx->ntotal + scan_pool_window_words() : 0);
                    if (idx->pool_cap < need) {  // (re)allocated zeroed; every search's last CTA leaves it zeroed
                        if (idx->pool) CU(cudaFree(idx->pool));
                        idx->pool = nullptr;
                        idx->pool_cap = 0;
                        CU(cudaMalloc(reinterpret_cast<void**>(&idx->pool), need * 8));
                        CU(cudaMemsetAsync(idx->pool, 0, need * 8, st));
                        idx->pool_cap = need;
                    }
                    a.pool = idx->pool;
                    // small shards (the application's 10k-row indexes): one key slot per row instead of the survivor pool
                    if (small_shard_applies(idx, tune, kp, plan)) {
                        a.small_fast_cap = tune.small_fast_cap > 0 ? tune.small_fast_cap : 1;
                        if (out.q_host != nullptr) {
                            a.q_inline = out.q_host;
                            f.done_flag = out.done_flag;
                            f.done_seq = out.done_seq;
                        }
                    }
                }
                if (out.q_host != nullptr && a.q_inline == nullptr)
                    return fail(EVS_ECUDA, "internal: the host search expected the small-shard kernel");
                if (tune.scan_dynamic > 1 || (tune.scan_dynamic == 1 && a.pool != nullptr)) {
                    a.next_chunk = idx->words + W_NEXT_CHUNK;
                    a.chunk_groups = tune.scan_chunk_groups > 0 ? tune.scan_chunk_groups : 2;
                }
                if (tune.scan_clock) {
                    if ((rc = ensure_dev(&idx->cta_clock, &idx->cta_clock_cap, (size_t)plan.grid * 2 + 24))) return rc;
                    idx->cta_clock_n = plan.grid;
                    a.cta_clock = idx->cta_clock;
                    f.dbg = idx->cta_clock + (size_t)plan.grid * 2 + 8;
                }
            }
            // the plan's shared-memory size was computed for qpp queries per pass: large enough for fewer
            CU(launch_scan(a, &plan, st));
        }
        if ((rc = prof.end(st))) return rc;
        if (scan_only || fused) continue;
        CU(launch_finalize(f, cn, st));
    }
    return EVS_OK;
}

// ---- fill kernels for the empty-index case (faiss returns all padding) ----
__global__ void fill_final_kernel(float* D, long long* I, long long count) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
        D[i] = -FLT_MAX;
        I[i] = -1;
    }
}
__global__ void fill_partial_kernel(double* S, long long* I, long long count) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (long long)gridDim.x * blockDim.x) {
        S[i] = -DBL_MAX;
        I[i] = -1;
    }
}

static ScanTuning tune_snapshot() {
    std::lock_guard<std::mutex> lk(g_tune_mu);
    return g_tune;
}

// k is tested against the option "max_k" of the snapshot that then routes the search
static int check_search_args(const evs_index* idx, int64_t nq, const void* q, int64_t k, const void* o1, const void* o2,
                             const ScanTuning& tune) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    if (nq < 0) return fail(EVS_EINVAL, "nq must be >= 0");
    if (k <= 0) return fail(EVS_EINVAL, "k must be > 0 (got %lld)", (long long)k);  // FAISS_THROW_IF_NOT(k > 0)
    if (k > tune.max_k) return fail(EVS_ELIMIT, "k = %lld exceeds the option max_k = %d (EVS_MAX_K = %d, EVS_MAX_K_LARGE = %d)",
                                    (long long)k, tune.max_k, EVS_MAX_K, EVS_MAX_K_LARGE);
    if (nq > 0 && (!q || !o1 || !o2)) return fail(EVS_EINVAL, "NULL query or output buffer");
    return EVS_OK;
}

// order stream `st` after the previous user of the handle's workspace and enqueue the search
static int search_dev_common(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, const SearchOut& out, cudaStream_t st,
                             const ScanTuning& tune, const PathInfo& pi) {
    int rc = ws_acquire(idx, st);
    if (rc) return rc;
    if (idx->ntotal == 0) {
        long long count = (long long)nq * k;
        int grid = (int)((count + 255) / 256 < 1024 ? (count + 255) / 256 : 1024);
        if (out.D) fill_final_kernel<<<grid, 256, 0, st>>>(out.D, reinterpret_cast<long long*>(out.I), count);
        else fill_partial_kernel<<<grid, 256, 0, st>>>(out.P_scores, reinterpret_cast<long long*>(out.P_ids), count);
        g_kernel_launches.fetch_add(1);
        CU(cudaGetLastError());
        idx->last_nq = 0;
        return EVS_OK;
    }
    return search_enqueue_locked(idx, nq, q_dev, k, out, st, tune, pi);
}

extern "C" int evs_index_search_dev(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, float* D_dev, int64_t* I_dev,
                                    void* stream) {
    const ScanTuning tune = tune_snapshot();
    int rc = check_search_args(idx, nq, q_dev, k, D_dev, I_dev, tune);
    if (rc || nq == 0) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    if ((rc = use_device(idx->device))) return rc;
    SearchOut out;
    out.D = D_dev;
    out.I = I_dev;
    return search_dev_common(idx, nq, q_dev, k, out, (cudaStream_t)stream, tune, plan_path(idx, nq, k, tune, true));
}

extern "C" int evs_index_search_partial_dev(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, double* out_scores_dev,
                                            int64_t* out_ids_dev, void* stream) {
    const ScanTuning tune = tune_snapshot();
    int rc = check_search_args(idx, nq, q_dev, k, out_scores_dev, out_ids_dev, tune);
    if (rc || nq == 0) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    if ((rc = use_device(idx->device))) return rc;
    SearchOut out;
    out.P_scores = out_scores_dev;
    out.P_ids = out_ids_dev;
    return search_dev_common(idx, nq, q_dev, k, out, (cudaStream_t)stream, tune, plan_path(idx, nq, k, tune, true));
}

extern "C" int evs_merge_partials_dev(int device, int nparts, int64_t nq, int64_t k, const double* scores_dev,
                                      const int64_t* ids_dev, int64_t part_stride, float* D_dev, int64_t* I_dev, void* stream) {
    if (nparts <= 0 || nq < 0 || k <= 0) return fail(EVS_EINVAL, "bad nparts/nq/k");
    if (nq == 0) return EVS_OK;
    if (!scores_dev || !ids_dev || !D_dev || !I_dev) return fail(EVS_EINVAL, "NULL buffer");
    if (k <= EVS_MAX_K) {  // the entries of a query are staged in shared memory
        if ((size_t)nparts * k * 24 > 200 * 1024) return fail(EVS_ELIMIT, "nparts*k too large for one merge");
    } else {  // large k: up to 8 parts, ranked in global memory
        const ScanTuning tune = tune_snapshot();
        if (k > tune.max_k) return fail(EVS_ELIMIT, "k = %lld exceeds the option max_k = %d", (long long)k, tune.max_k);
        if (nparts > 8) return fail(EVS_ELIMIT, "a merge for k > %d takes at most 8 parts (got %d)", EVS_MAX_K, nparts);
    }
    int rc = use_device(device);
    if (rc) return rc;
    if (part_stride == 0) part_stride = nq * k;
    if (part_stride < nq * k) return fail(EVS_EINVAL, "part_stride smaller than nq*k");
    CU(launch_merge_partials(nparts, nq, (int)k, scores_dev, reinterpret_cast<const long long*>(ids_dev), part_stride, D_dev,
                             reinterpret_cast<long long*>(I_dev), (cudaStream_t)stream));
    return EVS_OK;
}

template <typename T>
static int ensure_pinned(T** ptr, size_t* cap, size_t need_elems) {
    if (*cap >= need_elems && *ptr) return EVS_OK;
    if (*ptr) CU(cudaFreeHost(*ptr));
    *ptr = nullptr;
    *cap = 0;
    CU(cudaMallocHost(reinterpret_cast<void**>(ptr), need_elems * sizeof(T)));
    *cap = need_elems;
    return EVS_OK;
}

// host staging shared by evs_index_search and evs_index_search_exchange: queries go caller memory -> pinned -> device in
// one async copy; (I, D) live in ONE device buffer ([I int64 nq*k][D float32 nq*k]) so that they come back in one copy.
static int host_stage_locked(evs_index* idx, int64_t nq, int64_t k) {
    const size_t d = (size_t)idx->d;
    int rc = ensure_pinned(&idx->q_pin, &idx->q_pin_cap, (size_t)nq * d);
    if (rc) return rc;
    if ((rc = ensure_dev(&idx->q_dev, &idx->q_cap, (size_t)nq * d))) return rc;
    const size_t out_need = (size_t)nq * k;
    if (idx->out_cap < out_need) {
        if (idx->I_dev) cudaFree(idx->I_dev);
        idx->I_dev = nullptr;
        idx->D_dev = nullptr;
        idx->out_cap = 0;
        CU(cudaMalloc(reinterpret_cast<void**>(&idx->I_dev), out_need * (sizeof(int64_t) + sizeof(float))));
        idx->D_dev = reinterpret_cast<float*>(idx->I_dev + out_need);
        idx->out_cap = out_need;
    } else {
        idx->D_dev = reinterpret_cast<float*>(idx->I_dev + out_need);  // packed for this nq*k
    }
    if (idx->out_pin_cap < out_need) {
        if (idx->I_pin) cudaFreeHost(idx->I_pin);
        idx->I_pin = nullptr;
        idx->D_pin = nullptr;
        idx->out_pin_cap = 0;
        CU(cudaHostAlloc(reinterpret_cast<void**>(&idx->I_pin), out_need * (sizeof(int64_t) + sizeof(float)), cudaHostAllocMapped));
        idx->I_pin_dev = nullptr;
        if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&idx->I_pin_dev), idx->I_pin, 0) != cudaSuccess) {
            cudaGetLastError();
            idx->I_pin_dev = nullptr;  // no mapped access: the copy path is used
        }
        idx->out_pin_cap = out_need;
    }
    idx->D_pin = reinterpret_cast<float*>(idx->I_pin + out_need);
    return EVS_OK;
}

static int host_fetch_locked(evs_index* idx, int64_t nq, int64_t k, float* D_host, int64_t* I_host, cudaStream_t st) {
    const size_t out_need = (size_t)nq * k;
    CU(cudaMemcpyAsync(idx->I_pin, idx->I_dev, out_need * (sizeof(int64_t) + sizeof(float)), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    memcpy(D_host, idx->D_pin, out_need * sizeof(float));
    memcpy(I_host, idx->I_pin, out_need * sizeof(int64_t));
    return EVS_OK;
}

static int search_host_locked(evs_index* idx, int64_t nq, const float* q_host, int64_t k, float* D_host, int64_t* I_host,
                              const ScanTuning& tune) {
    int rc = use_device(idx->device);
    if (rc) return rc;
    if ((rc = host_stage_locked(idx, nq, k))) return rc;
    cudaStream_t st = idx->stream;
    if ((rc = ws_acquire(idx, st))) return rc;
    SearchOut out;
    out.D = idx->D_dev;
    out.I = idx->I_dev;
    const PathInfo pi = plan_path(idx, nq, k, tune, true);
    // one query, one launch: the kernel's last CTA writes the k results (k * 12 bytes) straight into the mapped pinned
    // buffer; the host only waits for the stream (what the application issues, oldapp.py:2005: ~6 us less per search)
    const bool direct = nq == 1 && pi.kind == PATH_GEMV && pi.fused && idx->I_pin_dev != nullptr && idx->ntotal > 0;
    if (direct) {
        out.I = idx->I_pin_dev;
        out.D = reinterpret_cast<float*>(idx->I_pin_dev + (size_t)nq * k);
    }
    // ... over a small shard (the application's index sizes): the query rides in the kernel's parameter block -- no staging
    // copy, no host-to-device copy ahead of the launch -- and the kernel raises a host-mapped word behind the results, which is
    // polled here instead of waiting for the stream to drain
    bool inline_q = false;
    if (direct && idx->d <= EVS_SMALL_QUERY_MAX_D) {
        const bool bf16 = idx->storage == EVS_STORE_BF16_F32;
        ScanPlan plan;
        if (plan_scan(idx->ntotal, idx->d, bf16, pi.kp, max_queries_per_pass(idx->d, bf16), idx->sm_count, tune, &plan) == cudaSuccess &&
            small_shard_applies(idx, tune, pi.kp, plan)) {
            if (idx->done_pin == nullptr) {
                void* hp = nullptr;
                if (cudaHostAlloc(&hp, 64, cudaHostAllocMapped) == cudaSuccess) {
                    memset(hp, 0, 64);
                    if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&idx->done_pin_dev), hp, 0) == cudaSuccess) {
                        idx->done_pin = reinterpret_cast<unsigned*>(hp);
                    } else {
                        cudaGetLastError();
                        cudaFreeHost(hp);
                    }
                } else {
                    cudaGetLastError();
                }
            }
            inline_q = idx->done_pin != nullptr;
        }
    }
    if (inline_q) {
        if (++idx->done_seq == 0u) idx->done_seq = 1u;
        out.q_host = q_host;
        out.done_flag = idx->done_pin_dev;
        out.done_seq = idx->done_seq;
    } else {
        memcpy(idx->q_pin, q_host, (size_t)nq * idx->d * sizeof(float));
        CU(cudaMemcpyAsync(idx->q_dev, idx->q_pin, (size_t)nq * idx->d * sizeof(float), cudaMemcpyHostToDevice, st));
    }
    rc = search_dev_common(idx, nq, idx->q_dev, k, out, st, tune, pi);
    if (!rc && inline_q) {
        // the flag arrives behind the results (system-scope fence in the kernel); a failed launch or kernel never raises it, so
        // the stream is queried from time to time
        const volatile unsigned* flag = idx->done_pin;
        const unsigned want = idx->done_seq;
        unsigned spins = 0;
        while (*flag != want) {
            if ((++spins & 1023u) == 0u) {
                const cudaError_t qe = cudaStreamQuery(st);
                if (qe == cudaSuccess) break;  // the stream has drained: the results are there (flag or not)
                if (qe != cudaErrorNotReady) return fail(EVS_ECUDA, "search failed: %s", cudaGetErrorString(qe));
            }
#if defined(__x86_64__) || defined(__i386__)
            __builtin_ia32_pause();
#endif
        }
        std::atomic_thread_fence(std::memory_order_acquire);
        memcpy(D_host, idx->D_pin, (size_t)nq * k * sizeof(float));
        memcpy(I_host, idx->I_pin, (size_t)nq * k * sizeof(int64_t));
    } else if (!rc && direct) {
        CU(cudaStreamSynchronize(st));
        memcpy(D_host, idx->D_pin, (size_t)nq * k * sizeof(float));
        memcpy(I_host, idx->I_pin, (size_t)nq * k * sizeof(int64_t));
    } else if (!rc) {
        rc = host_fetch_locked(idx, nq, k, D_host, I_host, st);
    }
    if (rc) cudaStreamSynchronize(st);  // the pinned query buffer may still be in flight: it is reused by the next call
    return rc;
}

// ---- coalescing of concurrent single-query callers (group commit) ----
// A single-query caller (k <= EVS_MAX_K) that finds no such search running on the handle runs alone, exactly as above.  One
// that arrives while one runs queues itself; when the running search returns, the first queued caller leads the next group:
// it takes up to kCoalesceCap queued callers and, where group_runs_as_one, searches them as ONE search of nq = m queries
// and k = the largest k, handing each its prefix (the top k under (canonical desc, id asc) is a prefix of the top k_max);
// otherwise it searches them one by one.  The others wait for their results; leadership then passes to the next queued
// caller, so no thread serves other callers' requests for long.
struct CoalesceWaiter {
    const float* q;
    int64_t k;
    float* D;
    int64_t* I;
    int rc = 0;
    bool done = false, lead = false;
    char err[512] = "";
};

// A group runs as one search only on shards where the int8 batch route applies (an int8 copy, at least shadow_min_rows
// rows): groups of up to kI8BatchMaxNQ take that route, larger fp32 groups the tensor-core scan (2.9 ms for 16 queries at
// 10M x 512 against 0.75 ms per lone search; scripts/i8_batch_probe.py).  On smaller shards it does not pay: at 10 000 rows
// (the small-shard kernel, ~30 us end to end) groups of 2-4 through the batch GEMV search ran at 0.78x the lone rate
// (scripts/coalesce_probe.py, profiles/coalesce_probe_every_size.jsonl), so those callers are searched one by one.
// The answer is the lone answer for fp32 storage (every path is exact); for bf16 storage only where both read the int8
// copy (groups of up to kI8BatchMaxNQ, k <= 48) -- its other paths are the uncertified recall mode.
static const int kCoalesceCap = 16;
static bool group_runs_as_one(const evs_index* idx, int64_t m, int64_t kmax, const ScanTuning& tune) {
    if (!i8_batch_applies(idx, 2, kmax, tune)) return false;
    if (idx->storage != EVS_STORE_BF16_F32) return true;
    return m <= kI8BatchMaxNQ && kmax <= 48 && shadow_applies(idx, 1, pick_kp(kmax), tune);
}

// idx->mu is held.  The group's queries go through the pinned staging buffer, its results come back in one copy.
static int search_group_locked(evs_index* idx, CoalesceWaiter* const* g, int m, const ScanTuning& tune) {
    int64_t kmax = 0;
    for (int j = 0; j < m; j++) kmax = g[j]->k > kmax ? g[j]->k : kmax;
    int rc = use_device(idx->device);
    if (rc) return rc;
    if ((rc = host_stage_locked(idx, m, kmax))) return rc;
    cudaStream_t st = idx->stream;
    if ((rc = ws_acquire(idx, st))) return rc;
    const size_t d = (size_t)idx->d;
    for (int j = 0; j < m; j++) memcpy(idx->q_pin + j * d, g[j]->q, d * sizeof(float));
    CU(cudaMemcpyAsync(idx->q_dev, idx->q_pin, (size_t)m * d * sizeof(float), cudaMemcpyHostToDevice, st));
    SearchOut out;
    out.D = idx->D_dev;
    out.I = idx->I_dev;
    rc = search_dev_common(idx, m, idx->q_dev, kmax, out, st, tune, plan_path(idx, m, kmax, tune, true));
    if (!rc) {
        const size_t n = (size_t)m * kmax;
        const cudaError_t e = cudaMemcpyAsync(idx->I_pin, idx->I_dev, n * (sizeof(int64_t) + sizeof(float)), cudaMemcpyDeviceToHost, st);
        if (e != cudaSuccess) rc = fail(EVS_ECUDA, "%s", cudaGetErrorString(e));
    }
    if (!rc) {
        const cudaError_t e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) rc = fail(EVS_ECUDA, "search failed: %s", cudaGetErrorString(e));
    }
    if (rc) {
        cudaStreamSynchronize(st);  // the pinned query buffer may still be in flight
        return rc;
    }
    for (int j = 0; j < m; j++) {
        memcpy(g[j]->D, idx->D_pin + (size_t)j * kmax, (size_t)g[j]->k * sizeof(float));
        memcpy(g[j]->I, idx->I_pin + (size_t)j * kmax, (size_t)g[j]->k * sizeof(int64_t));
    }
    idx->co_groups++;
    idx->co_queries += m;
    return EVS_OK;
}

// the leader `self`, already off the queue: takes up to kCoalesceCap - 1 more callers, searches them, wakes them
static int lead_group(evs_index* idx, CoalesceWaiter* self, const ScanTuning& tune) {
    CoalesceWaiter* g[kCoalesceCap];
    int m = 0;
    g[m++] = self;
    {
        std::lock_guard<std::mutex> lq(idx->cq_mu);
        while (m < kCoalesceCap && !idx->cq.empty()) {
            g[m++] = idx->cq.front();
            idx->cq.pop_front();
        }
    }
    {
        std::lock_guard<std::mutex> lk(idx->mu);
        // bf16 storage: sub-groups of at most kI8BatchMaxNQ (the int8 route); fp32: the whole group
        const int step = idx->storage == EVS_STORE_BF16_F32 ? kI8BatchMaxNQ : m;
        for (int j0 = 0; j0 < m; j0 += step) {
            const int n = m - j0 < step ? m - j0 : step;
            int64_t kmax = 0;
            for (int j = j0; j < j0 + n; j++) kmax = g[j]->k > kmax ? g[j]->k : kmax;
            if (n >= 2 && group_runs_as_one(idx, n, kmax, tune)) {
                const int rc = search_group_locked(idx, g + j0, n, tune);
                for (int j = j0; j < j0 + n; j++) {
                    g[j]->rc = rc;
                    if (rc) snprintf(g[j]->err, sizeof(g[j]->err), "%s", t_err);
                }
            } else {
                for (int j = j0; j < j0 + n; j++) {
                    g[j]->rc = search_host_locked(idx, 1, g[j]->q, g[j]->k, g[j]->D, g[j]->I, tune);
                    if (g[j]->rc) snprintf(g[j]->err, sizeof(g[j]->err), "%s", t_err);
                }
            }
        }
    }
    {
        std::lock_guard<std::mutex> lq(idx->cq_mu);
        for (int j = 1; j < m; j++) g[j]->done = true;
    }
    idx->cq_cv.notify_all();
    return self->rc ? fail(self->rc, "%s", self->err) : EVS_OK;
}

extern "C" int evs_index_search(evs_index* idx, int64_t nq, const float* q_host, int64_t k, float* D_host, int64_t* I_host) {
    const ScanTuning tune = tune_snapshot();
    int rc = check_search_args(idx, nq, q_host, k, D_host, I_host, tune);
    if (rc || nq == 0) return rc;
    if (nq != 1 || k > EVS_MAX_K) {
        std::lock_guard<std::mutex> lk(idx->mu);
        return search_host_locked(idx, nq, q_host, k, D_host, I_host, tune);
    }
    CoalesceWaiter w;
    w.q = q_host;
    w.k = k;
    w.D = D_host;
    w.I = I_host;
    {
        std::unique_lock<std::mutex> lq(idx->cq_mu);
        if (idx->cq_busy) {
            idx->cq.push_back(&w);
            idx->cq_cv.wait(lq, [&] { return w.done || w.lead; });
            if (w.done) return w.rc ? fail(w.rc, "%s", w.err) : EVS_OK;
        } else {
            idx->cq_busy = true;
        }
    }
    if (w.lead) {
        rc = lead_group(idx, &w, tune);
    } else {
        std::lock_guard<std::mutex> lk(idx->mu);
        rc = search_host_locked(idx, nq, q_host, k, D_host, I_host, tune);
    }
    {  // hand the handle to the next queued caller, or leave it idle
        std::lock_guard<std::mutex> lq(idx->cq_mu);
        if (idx->cq.empty()) {
            idx->cq_busy = false;
        } else {
            idx->cq.front()->lead = true;
            idx->cq.pop_front();
        }
    }
    idx->cq_cv.notify_all();
    return rc;
}

// ---------------------------------------------------------------------------------------------
// peer-store exchange of shard partials (row sharding, one process per GPU)
// ---------------------------------------------------------------------------------------------
struct evs_exchange {
    int device = 0, rank = 0, world = 0;
    int64_t max_nq = 0, max_k = 0;
    size_t slot_bytes = 0, total_bytes = 0;
    unsigned char* local = nullptr;     // [2][world][slot_bytes] slots of flagged 32-byte entries
    unsigned char* peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
    bool opened[8] = {false, false, false, false, false, false, false, false};
    bool connected = false;
    unsigned long long seq = 0;
    double* stage_scores = nullptr;     // local partial staging for the paths that cannot write the slots themselves
    int64_t* stage_ids = nullptr;
    volatile int* status_host = nullptr;  // host-mapped word the merge kernel writes on failure (1 timeout, 2 peer failed)
    int* status_dev = nullptr;
    std::mutex mu;
};

extern "C" int evs_exchange_create(int device, int rank, int world, int64_t max_nq, int64_t max_k, evs_exchange** out) {
    if (!out) return fail(EVS_EINVAL, "out is NULL");
    *out = nullptr;
    if (world < 1 || world > 8) return fail(EVS_ELIMIT, "world must be in [1, 8] (one NVSwitch box), got %d", world);
    if (rank < 0 || rank >= world) return fail(EVS_EINVAL, "rank %d out of range for world %d", rank, world);
    if (max_nq <= 0 || max_k <= 0 || max_k > tune_snapshot().max_k) return fail(EVS_EINVAL, "bad max_nq/max_k");
    int ndev = 0;
    evs_device_count(&ndev);
    if (ndev <= 0) return fail(EVS_ENODEV, "no CUDA device: libevs has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(EVS_EINVAL, "device %d out of range (have %d)", device, ndev);
    int rc = use_device(device);
    if (rc) return rc;
    evs_exchange* ex = new (std::nothrow) evs_exchange();
    if (!ex) return fail(EVS_ENOMEM, "out of host memory");
    ex->device = device;
    ex->rank = rank;
    ex->world = world;
    ex->max_nq = max_nq;
    ex->max_k = max_k;
    ex->slot_bytes = ((size_t)max_nq * max_k * kExchangeEntryBytes + 255) & ~(size_t)255;
    ex->total_bytes = 2 * (size_t)world * ex->slot_bytes;
    cudaError_t e = cudaMalloc(reinterpret_cast<void**>(&ex->local), ex->total_bytes);
    if (e == cudaSuccess) e = cudaMemset(ex->local, 0, ex->total_bytes);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&ex->stage_scores), (size_t)max_nq * max_k * 8);
    if (e == cudaSuccess) e = cudaMalloc(reinterpret_cast<void**>(&ex->stage_ids), (size_t)max_nq * max_k * 8);
    void* sh = nullptr;
    if (e == cudaSuccess) e = cudaHostAlloc(&sh, 64, cudaHostAllocMapped);
    if (e == cudaSuccess) {
        memset(sh, 0, 64);
        ex->status_host = reinterpret_cast<volatile int*>(sh);
        e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&ex->status_dev), sh, 0);
    }
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    if (e != cudaSuccess) {
        cudaFree(ex->local);
        cudaFree(ex->stage_scores);
        cudaFree(ex->stage_ids);
        if (sh) cudaFreeHost(sh);
        delete ex;
        return fail(e == cudaErrorMemoryAllocation ? EVS_ENOMEM : EVS_ECUDA, "exchange allocation failed: %s", cudaGetErrorString(e));
    }
    ex->peer[rank] = ex->local;
    ex->connected = (world == 1);
    *out = ex;
    return EVS_OK;
}

extern "C" int evs_exchange_handle(evs_exchange* ex, void* handle_out, int64_t handle_bytes) {
    if (!ex || !handle_out) return fail(EVS_EINVAL, "NULL argument");
    if (handle_bytes != EVS_IPC_HANDLE_BYTES) return fail(EVS_EINVAL, "handle buffer must be %d bytes", EVS_IPC_HANDLE_BYTES);
    static_assert(sizeof(cudaIpcMemHandle_t) == EVS_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t is 64 bytes");
    int rc = use_device(ex->device);
    if (rc) return rc;
    cudaIpcMemHandle_t h;
    CU(cudaIpcGetMemHandle(&h, ex->local));
    memcpy(handle_out, &h, sizeof(h));
    return EVS_OK;
}

extern "C" int evs_exchange_connect(evs_exchange* ex, const void* handles, int64_t handles_bytes) {
    if (!ex || !handles) return fail(EVS_EINVAL, "NULL argument");
    if (handles_bytes != (int64_t)ex->world * EVS_IPC_HANDLE_BYTES)
        return fail(EVS_EINVAL, "expected %d handles of %d bytes", ex->world, EVS_IPC_HANDLE_BYTES);
    std::lock_guard<std::mutex> lk(ex->mu);
    int rc = use_device(ex->device);
    if (rc) return rc;
    for (int g = 0; g < ex->world; g++) {
        if (g == ex->rank || ex->opened[g]) continue;
        cudaIpcMemHandle_t h;
        memcpy(&h, reinterpret_cast<const unsigned char*>(handles) + (size_t)g * EVS_IPC_HANDLE_BYTES, sizeof(h));
        void* p = nullptr;
        CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));  // maps the peer's buffer over NVLink
        ex->peer[g] = reinterpret_cast<unsigned char*>(p);
        ex->opened[g] = true;
    }
    ex->connected = true;
    return EVS_OK;
}

// *timed_out = the failure word (0 ok, 1 = a merge gave up waiting for a rank, 2 = a rank reported that it failed a search);
// reading it does not clear it -- the next search call on this exchange reports and clears it
extern "C" int evs_exchange_status(evs_exchange* ex, int* timed_out, int64_t* searches) {
    if (!ex) return fail(EVS_EINVAL, "ex is NULL");
    std::lock_guard<std::mutex> lk(ex->mu);
    if (timed_out) *timed_out = *ex->status_host;
    if (searches) *searches = (int64_t)ex->seq;
    return EVS_OK;
}

extern "C" int evs_exchange_free(evs_exchange* ex) {
    if (!ex) return EVS_OK;
    cudaSetDevice(ex->device);
    cudaDeviceSynchronize();
    for (int g = 0; g < ex->world; g++)
        if (ex->opened[g]) cudaIpcCloseMemHandle(ex->peer[g]);
    cudaFree(ex->local);
    cudaFree(ex->stage_scores);
    cudaFree(ex->stage_ids);
    if (ex->status_host) cudaFreeHost(const_cast<int*>(ex->status_host));
    delete ex;
    return EVS_OK;
}

// a failure an earlier search of this exchange ran into (seen by its merge kernel) is reported once, by the next call
static int exchange_take_failure(evs_exchange* ex) {
    const int s = *ex->status_host;
    if (s == 0) return EVS_OK;
    *ex->status_host = 0;
    return fail(EVS_ETIMEOUT, s == 2 ? "a peer rank failed a collective search: its results were padding, not a merge without that shard"
                                     : "a collective search waited ~10 s for a rank that never arrived: its results were padding");
}

// enqueue scan -> finalise (-> publish) -> merge for one exchange-mode search; idx->mu and ex->mu are held
static int search_exchange_enqueue_locked(evs_index* idx, evs_exchange* ex, int64_t nq, const float* q_dev, int64_t k, float* D_dev,
                                          int64_t* I_dev, cudaStream_t st, const ScanTuning& tune) {
    Exchange x;
    for (int g = 0; g < ex->world; g++) x.peer[g] = ex->peer[g];
    x.rank = ex->rank;
    x.world = ex->world;
    x.seq = ex->seq + 1;             // every rank calls in the same order: the sequence numbers agree
    x.parity = (int)(x.seq & 1ull);  // two generations of slots: a fast rank may start search s+1 while a slow one merges s
    x.slot_bytes = ex->slot_bytes;
    x.nq_total = nq;
    x.k = (int)k;
    x.status = ex->status_dev;
    const PathInfo pi = plan_path(idx, nq, k, tune, true);  // ONE snapshot decides the path here and inside the search
    // empty shard / scans that need the host (overflow repair) / device-guarded batches (their second finalise may still
    // overwrite results): the partial goes to local staging and a publish kernel stores it into the peers' slots;
    // otherwise the finalise kernel stores this shard's k best straight into every rank's slot
    const bool staged = idx->ntotal == 0 || pi.kind == PATH_TC_SYNC || (pi.kind == PATH_TC_HEAP && pi.guard) || pi.kind == PATH_LARGE_K;
    const bool one_launch = !staged && pi.kind == PATH_GEMV && pi.fused;  // scan + finalise + peer stores + wait + merge
    SearchOut out;
    if (staged) {
        out.P_scores = ex->stage_scores;
        out.P_ids = ex->stage_ids;
    } else {
        if (one_launch) {
            x.merge_D = D_dev;
            x.merge_I = reinterpret_cast<long long*>(I_dev);
        }
        out.x = &x;
    }
    int rc = g_exchange_fail_next.exchange(0) ? fail(EVS_ECUDA, "injected failure (option exchange_fail_next)")
                                              : search_dev_common(idx, nq, q_dev, k, out, st, tune, pi);
    cudaError_t e = cudaSuccess;
    if (!rc && staged) e = launch_publish_partials(x, nq, (int)k, ex->stage_scores, reinterpret_cast<const long long*>(ex->stage_ids), st);
    if (!rc && e == cudaSuccess && !one_launch) e = launch_merge_exchange(x, nq, (int)k, D_dev, reinterpret_cast<long long*>(I_dev), st);
    if (!rc && e != cudaSuccess) rc = fail(EVS_ECUDA, "exchange launch failed: %s", cudaGetErrorString(e));
    ex->seq = x.seq;  // stay in step with the peers whatever happened
    if (rc) {
        // this rank cannot deliver its partial: tell the peers (poisoned flag) instead of leaving them to wait ~10 s, or to
        // merge without this shard
        char keep[sizeof(t_err)];
        memcpy(keep, t_err, sizeof(keep));
        launch_publish_poison(x, st);
        cudaGetLastError();
        memcpy(t_err, keep, sizeof(keep));
    }
    return rc;
}

static int check_exchange_args(const evs_index* idx, const evs_exchange* ex, int64_t nq, int64_t k) {
    if (!ex) return fail(EVS_EINVAL, "ex is NULL");
    if (!ex->connected) return fail(EVS_EINVAL, "exchange is not connected (evs_exchange_connect)");
    if (ex->device != idx->device) return fail(EVS_EINVAL, "exchange lives on device %d, index on %d", ex->device, idx->device);
    if (nq > ex->max_nq || k > ex->max_k)
        return fail(EVS_ELIMIT, "nq=%lld k=%lld exceed the exchange's capacity (%lld, %lld)", (long long)nq, (long long)k,
                    (long long)ex->max_nq, (long long)ex->max_k);
    return EVS_OK;
}

extern "C" int evs_index_search_exchange_dev(evs_index* idx, evs_exchange* ex, int64_t nq, const float* q_dev, int64_t k,
                                             float* D_dev, int64_t* I_dev, void* stream) {
    const ScanTuning tune = tune_snapshot();
    int rc = check_search_args(idx, nq, q_dev, k, D_dev, I_dev, tune);
    if (rc || nq == 0) return rc;
    if ((rc = check_exchange_args(idx, ex, nq, k))) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    std::lock_guard<std::mutex> lkx(ex->mu);
    if ((rc = use_device(idx->device))) return rc;
    // asynchronous entry point: a failure seen by an EARLIER search's merge kernel is reported here (once), before this
    // search is enqueued -- every rank still enqueues its searches in step
    const int late = exchange_take_failure(ex);
    rc = search_exchange_enqueue_locked(idx, ex, nq, q_dev, k, D_dev, I_dev, (cudaStream_t)stream, tune);
    return rc ? rc : late;
}

extern "C" int evs_index_search_exchange(evs_index* idx, evs_exchange* ex, int64_t nq, const float* q_host, int64_t k, float* D_host,
                                         int64_t* I_host) {
    const ScanTuning tune = tune_snapshot();
    int rc = check_search_args(idx, nq, q_host, k, D_host, I_host, tune);
    if (rc || nq == 0) return rc;
    if ((rc = check_exchange_args(idx, ex, nq, k))) return rc;
    std::lock_guard<std::mutex> lk(idx->mu);
    std::lock_guard<std::mutex> lkx(ex->mu);
    if ((rc = use_device(idx->device))) return rc;
    if ((rc = host_stage_locked(idx, nq, k))) return rc;
    memcpy(idx->q_pin, q_host, (size_t)nq * idx->d * sizeof(float));
    cudaStream_t st = idx->stream;
    if ((rc = ws_acquire(idx, st))) return rc;
    CU(cudaMemcpyAsync(idx->q_dev, idx->q_pin, (size_t)nq * idx->d * sizeof(float), cudaMemcpyHostToDevice, st));
    // one query: the one-launch search (scan + finalise + peer stores + merge) writes the merged (D, I) straight into the
    // mapped pinned buffer (decided like search_exchange_enqueue_locked decides the path: same options snapshot rules)
    bool direct = false;
    {
        const PathInfo pi = plan_path(idx, nq, k, tune, true);
        direct = nq == 1 && idx->ntotal > 0 && pi.kind == PATH_GEMV && pi.fused && idx->I_pin_dev != nullptr;
    }
    float* Dd = direct ? reinterpret_cast<float*>(idx->I_pin_dev + (size_t)nq * k) : idx->D_dev;
    int64_t* Id = direct ? idx->I_pin_dev : idx->I_dev;
    rc = search_exchange_enqueue_locked(idx, ex, nq, idx->q_dev, k, Dd, Id, st, tune);
    if (!rc && direct) {
        cudaError_t se = cudaStreamSynchronize(st);
        if (se != cudaSuccess) rc = fail(EVS_ECUDA, "search failed: %s", cudaGetErrorString(se));
        else {
            memcpy(D_host, idx->D_pin, (size_t)nq * k * sizeof(float));
            memcpy(I_host, idx->I_pin, (size_t)nq * k * sizeof(int64_t));
        }
    } else if (!rc) {
        rc = host_fetch_locked(idx, nq, k, D_host, I_host, st);
    }
    if (rc) {
        cudaStreamSynchronize(st);
        return rc;
    }
    return exchange_take_failure(ex);  // synchronous entry point: this search's own failure, if any
}

extern "C" int evs_index_last_margins(evs_index* idx, int64_t nq, float* margins_host) {
    if (!idx || !margins_host) return fail(EVS_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    if (nq != idx->last_nq) return fail(EVS_EINVAL, "last search had %lld queries, not %lld", (long long)idx->last_nq, (long long)nq);
    if (nq == 0) return EVS_OK;
    int rc = use_device(idx->device);
    if (rc) return rc;
    if (idx->have_last_stream) CU(cudaStreamSynchronize(idx->last_stream));
    CU(cudaMemcpy(margins_host, idx->margins_dev, (size_t)nq * sizeof(float), cudaMemcpyDeviceToHost));
    return EVS_OK;
}

extern "C" int evs_index_time_scan(evs_index* idx, int64_t nq, const float* q_dev, int64_t k, int iters, float* mean_ms) {
    const ScanTuning tune = tune_snapshot();
    int rc = check_search_args(idx, nq, q_dev, k, mean_ms, mean_ms, tune);
    if (rc) return rc;
    if (nq == 0 || iters <= 0 || idx->ntotal == 0) return fail(EVS_EINVAL, "nothing to time");
    std::lock_guard<std::mutex> lk(idx->mu);
    if ((rc = use_device(idx->device))) return rc;
    cudaStream_t st = idx->stream;
    cudaEvent_t e0, e1;
    CU(cudaEventCreate(&e0));
    CU(cudaEventCreate(&e1));
    if ((rc = ws_acquire(idx, st))) return rc;
    SearchOut none;
    const PathInfo pi = plan_path(idx, nq, k, tune, true);
    // the int8 copy is scanned only by the fused search kernel: its scan is the whole search, results to the workspace
    if (pi.shadow && !(rc = host_stage_locked(idx, nq, k))) {
        none.D = idx->D_dev;
        none.I = idx->I_dev;
    }
    const bool scan_only = !pi.shadow;
    if (!rc) rc = search_enqueue_locked(idx, nq, q_dev, k, none, st, tune, pi, scan_only);  // warm-up
    if (!rc) {
        cudaEventRecord(e0, st);
        for (int i = 0; i < iters && !rc; i++) rc = search_enqueue_locked(idx, nq, q_dev, k, none, st, tune, pi, scan_only);
        cudaEventRecord(e1, st);
    }
    cudaError_t e = cudaStreamSynchronize(st);
    float ms = 0.f;
    if (!rc && e == cudaSuccess) cudaEventElapsedTime(&ms, e0, e1);
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(EVS_ECUDA, "scan failed: %s", cudaGetErrorString(e));
    *mean_ms = ms / iters;
    return EVS_OK;
}

extern "C" int evs_index_scan_profile(evs_index* idx, int64_t* count, double* total_ms) {
    if (!idx || !count || !total_ms) return fail(EVS_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    double sum = 0.0;
    for (size_t i = 0; i < idx->prof_used; i++) {
        CU(cudaEventSynchronize(idx->prof_events[i].second));
        float ms = 0.f;
        CU(cudaEventElapsedTime(&ms, idx->prof_events[i].first, idx->prof_events[i].second));
        sum += ms;
    }
    *count = (int64_t)idx->prof_used;
    *total_ms = sum;
    idx->prof_used = 0;
    return EVS_OK;
}

extern "C" int evs_index_guard_stats(evs_index* idx, int64_t* reruns, int64_t* uncertified) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    if (idx->have_last_stream) CU(cudaStreamSynchronize(idx->last_stream));
    unsigned long long w[2] = {0, 0};
    CU(cudaMemcpy(w, idx->words + W_UNCERT, sizeof(w), cudaMemcpyDeviceToHost));  // W_UNCERT, W_RERUNS are adjacent u64
    if (uncertified) *uncertified = (int64_t)w[0];
    if (reruns) *reruns = (int64_t)w[1];
    return EVS_OK;
}

extern "C" int evs_index_shadow_stats(evs_index* idx, int64_t* wide_searches, float* emax, int64_t* last_candidates) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    if (idx->have_last_stream) CU(cudaStreamSynchronize(idx->last_stream));
    unsigned w[2] = {0, 0};
    CU(cudaMemcpy(w, idx->words + W_WIDE, sizeof(w), cudaMemcpyDeviceToHost));  // W_WIDE, W_LASTC are adjacent
    if (wide_searches) *wide_searches = (int64_t)w[0];
    if (last_candidates) *last_candidates = (int64_t)w[1];
    if (emax) *emax = idx->xi8 ? idx->emax_host : -1.f;
    return EVS_OK;
}

extern "C" int evs_index_large_k_stats(evs_index* idx, int64_t* searches, int64_t* last_candidates) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    if (idx->have_last_stream) CU(cudaStreamSynchronize(idx->last_stream));
    unsigned c = 0;
    if (idx->lk_stats) CU(cudaMemcpy(&c, idx->lk_stats, sizeof(c), cudaMemcpyDeviceToHost));
    if (searches) *searches = idx->lk_searches;
    if (last_candidates) *last_candidates = (int64_t)c;
    return EVS_OK;
}

extern "C" int evs_index_coalesce_stats(evs_index* idx, int64_t* groups, int64_t* grouped_queries, int64_t* i8_batch_passes) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    std::lock_guard<std::mutex> lk(idx->mu);
    if (groups) *groups = idx->co_groups;
    if (grouped_queries) *grouped_queries = idx->co_queries;
    if (i8_batch_passes) *i8_batch_passes = idx->i8_batch_passes;
    return EVS_OK;
}

extern "C" int evs_index_max_row_norm(evs_index* idx, float* max_norm) {
    if (!idx || !max_norm) return fail(EVS_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    CU(cudaMemcpy(max_norm, idx->words + W_MAX_NORM, sizeof(float), cudaMemcpyDeviceToHost));
    return EVS_OK;
}

extern "C" int evs_index_scan_clocks(evs_index* idx, uint64_t* out_host, int64_t cap_ctas, int64_t* nctas) {
    if (!idx || !nctas) return fail(EVS_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    *nctas = idx->cta_clock_n;
    if (!out_host || idx->cta_clock_n == 0) return EVS_OK;
    if (cap_ctas < idx->cta_clock_n) return fail(EVS_EINVAL, "buffer holds %lld CTAs, need %d", (long long)cap_ctas, idx->cta_clock_n);
    if (idx->have_last_stream) CU(cudaStreamSynchronize(idx->last_stream));
    CU(cudaMemcpy(out_host, idx->cta_clock, (size_t)idx->cta_clock_n * 16, cudaMemcpyDeviceToHost));
    // then the last CTA's own stamps (8) and the phases of its finalise: 8 with room for n + 8 CTAs, 16 with room for n + 12
    if (cap_ctas >= idx->cta_clock_n + 8)
        CU(cudaMemcpy(out_host + 2 * (size_t)idx->cta_clock_n, idx->cta_clock + 2 * (size_t)idx->cta_clock_n,
                      cap_ctas >= idx->cta_clock_n + 12 ? 192 : 128, cudaMemcpyDeviceToHost));
    return EVS_OK;
}

extern "C" int evs_index_tc_max_queries(const evs_index* idx, int* max_queries) {
    if (!idx || !max_queries) return fail(EVS_EINVAL, "NULL argument");
    *max_queries = tc_max_queries(idx->d, idx->storage == EVS_STORE_BF16_F32);
    return EVS_OK;
}

extern "C" int evs_index_tc_x3_max_queries(const evs_index* idx, int* max_queries) {
    if (!idx || !max_queries) return fail(EVS_EINVAL, "NULL argument");
    const ScanTuning tune = tune_snapshot();
    *max_queries = (idx->storage == EVS_STORE_F32 && tune.x3) ? tc_x3_max_queries(idx->d) : 0;
    return EVS_OK;
}

extern "C" int evs_index_tc_scores_dev(evs_index* idx, int64_t nq, const float* q_dev, float* out_dev, int* npad, void* stream) {
    if (!idx || !q_dev || !npad) return fail(EVS_EINVAL, "NULL argument");
    const bool bf16 = idx->storage == EVS_STORE_BF16_F32;
    const int nb_max = tc_max_queries(idx->d, bf16);
    if (nb_max == 0) return fail(EVS_ELIMIT, "d = %d is not supported by the tensor-core scan", idx->d);
    const ScanTuning tune = tune_snapshot();
    const int pair_min = tune.tc_pair_min_nq;
    const bool pair = pair_min > 0 && (nq >= pair_min || nq > nb_max) && tc2_max_half(idx->d, bf16) > 0;
    // fp32 rows, small batches: the scores of the 3xTF32 split scan the searches use
    const int x3 = (!bf16 && !pair && tune.x3 && nq <= tc_x3_max_queries(idx->d)) ? 1 : 0;
    if (nq <= 0 || (!pair && nq > nb_max) || nq > 4096) return fail(EVS_EINVAL, "nq must be in [1, %d]", pair ? 4096 : nb_max);
    if (idx->ntotal == 0) return fail(EVS_EINVAL, "empty index");
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    TcArgs a = make_tc_args(idx, q_dev, nq, nullptr, nullptr);
    cudaStream_t st = (cudaStream_t)stream;
    if (pair) {
        Tc2Plan pl;
        CU(tc2_plan(idx->ntotal, idx->d, bf16, (int)nq, 64, idx->sm_count, &pl));
        *npad = pl.nqp;
        if (!out_dev) return EVS_OK;  // pitch query
        if ((rc = ensure_dev(&idx->tc_ws, &idx->tc_ws_cap, tc2_workspace_bytes(pl)))) return rc;
        if ((rc = ws_acquire(idx, st))) return rc;
        CU(tc2_dump_scores(a, pl, idx->tc_ws, out_dev, st));
        *npad = pl.nqp;
    } else {
        TcPlan pl;
        CU(tc_plan(idx->ntotal, idx->d, bf16, (int)nq, 64, idx->sm_count, x3, &pl));
        *npad = pl.npad;
        if (!out_dev) return EVS_OK;  // pitch query
        if ((rc = ensure_dev(&idx->tc_ws, &idx->tc_ws_cap, tc_workspace_bytes(pl)))) return rc;
        if ((rc = ws_acquire(idx, st))) return rc;
        CU(tc_dump_scores(a, pl, idx->tc_ws, out_dev, st));
    }
    return EVS_OK;
}

// ---------------------------------------------------------------------------------------------
// stand-alone kernels
// ---------------------------------------------------------------------------------------------
static int device_sm_count(int device, int* sms) {
    CU(cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, device));
    return EVS_OK;
}

extern "C" int evs_l2_normalize_dev(int device, void* x_dev, int64_t n, int d, int dtype, void* stream) {
    if (n < 0 || d <= 0) return fail(EVS_EINVAL, "bad n/d");
    if (dtype != EVS_F32 && dtype != EVS_F16 && dtype != EVS_BF16) return fail(EVS_EINVAL, "bad dtype %d", dtype);
    if (n == 0) return EVS_OK;
    if (!x_dev) return fail(EVS_EINVAL, "x is NULL");
    int ndev = 0;
    evs_device_count(&ndev);
    if (ndev <= 0) return fail(EVS_ENODEV, "no CUDA device: libevs has no CPU fallback");
    int rc = use_device(device), sms = 0;
    if (rc || (rc = device_sm_count(device, &sms))) return rc;
    if ((size_t)d * 4 * 8 > 200 * 1024) return fail(EVS_ELIMIT, "d = %d too large for the normalise kernel", d);
    CU(launch_l2_normalize(x_dev, n, d, dtype, sms, (cudaStream_t)stream));
    return EVS_OK;
}

extern "C" int evs_l2_normalize(int device, float* x_host, int64_t n, int d) {
    if (n < 0 || d <= 0) return fail(EVS_EINVAL, "bad n/d");
    if (n == 0) return EVS_OK;
    if (!x_host) return fail(EVS_EINVAL, "x is NULL");
    int ndev = 0;
    evs_device_count(&ndev);
    if (ndev <= 0) return fail(EVS_ENODEV, "no CUDA device: libevs has no CPU fallback");
    int rc = use_device(device);
    if (rc) return rc;
    float* dev = nullptr;
    size_t bytes = (size_t)n * d * sizeof(float);
    CU(cudaMalloc(reinterpret_cast<void**>(&dev), bytes));
    cudaError_t e = cudaMemcpy(dev, x_host, bytes, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = evs_l2_normalize_dev(device, dev, n, d, EVS_F32, nullptr);
        if (!rc) e = cudaMemcpy(x_host, dev, bytes, cudaMemcpyDeviceToHost);  // default-stream copy orders after the kernel
    }
    cudaFree(dev);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(EVS_ECUDA, "copy failed: %s", cudaGetErrorString(e));
    return EVS_OK;
}

extern "C" int evs_f32_to_bf16_dev(int device, const float* src_dev, void* dst_dev, int64_t count, void* stream) {
    if (count < 0) return fail(EVS_EINVAL, "bad count");
    if (count == 0) return EVS_OK;
    if (!src_dev || !dst_dev) return fail(EVS_EINVAL, "NULL buffer");
    int rc = use_device(device), sms = 0;
    if (rc || (rc = device_sm_count(device, &sms))) return rc;
    CU(launch_f32_to_bf16(src_dev, dst_dev, count, sms, (cudaStream_t)stream));
    return EVS_OK;
}

// ---------------------------------------------------------------------------------------------
// persistence: index.faiss (45-byte IndexFlat header + fp32 payload, little-endian)
// ---------------------------------------------------------------------------------------------
#pragma pack(push, 1)
struct FlatHeader {
    char fourcc[4];
    int32_t d;
    int64_t ntotal;
    int64_t dummy1, dummy2;
    uint8_t is_trained;
    int32_t metric_type;
    uint64_t count;  // number of float32 values
};
#pragma pack(pop)
static_assert(sizeof(FlatHeader) == 45, "index.faiss flat header is 45 bytes");

static const size_t kIoChunk = (size_t)64 << 20;

// One chunk of the file is read (or written) by several threads at once, each with its own pread / pwrite over a disjoint
// 4 KiB-aligned slice: a single thread copies out of the page cache at 2-3 GB/s, far below what the host-to-device copy
// behind it takes (PCIe 5 x16), and a cold file wants several requests in flight anyway.
static int io_threads_for(size_t nb) {
    int t = g_io_threads.load();
    if (t <= 0) {
        // measured on the pool's 16-thread B200 hosts, page cache -> pinned -> HBM: 6.5 GB/s with 1 thread, 23 with 4, 35 with 16
        unsigned hc = std::thread::hardware_concurrency();
        t = hc >= 16 ? 16 : hc >= 2 ? (int)hc : 1;
    }
    size_t most = nb / ((size_t)4 << 20);  // at least 4 MiB per thread
    if ((size_t)t > most) t = (int)most;
    return t < 1 ? 1 : t;
}

static bool rw_full(int fd, unsigned char* buf, size_t nb, off_t off, bool write) {
    while (nb) {
        ssize_t r = write ? pwrite(fd, buf, nb, off) : pread(fd, buf, nb, off);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) return false;  // error, or end of file inside the payload
        buf += r;
        off += r;
        nb -= (size_t)r;
    }
    return true;
}

static bool rw_parallel(int fd, void* buf, size_t nb, off_t off, bool write) {
    const int t = io_threads_for(nb);
    unsigned char* p = static_cast<unsigned char*>(buf);
    if (t == 1) return rw_full(fd, p, nb, off, write);
    size_t slice = ((nb + t - 1) / t + 4095) & ~(size_t)4095;
    std::atomic<int> bad{0};
    std::vector<std::thread> th;
    th.reserve(t - 1);
    auto job = [&](size_t lo) {
        size_t n = nb - lo < slice ? nb - lo : slice;
        if (!rw_full(fd, p + lo, n, off + (off_t)lo, write)) bad.store(1);
    };
    size_t lo = slice;
    try {
        for (; lo < nb; lo += slice) th.emplace_back(job, lo);
    } catch (...) {  // no more threads: this one takes the rest
        for (; lo < nb; lo += slice) job(lo);
    }
    job(0);
    for (auto& x : th) x.join();
    return bad.load() == 0;
}

// The two pinned staging chunks are kept for the life of the process (cudaMallocHost of 64 MiB costs tens of milliseconds,
// the application loads an index per request until the resident cache holds it); a second concurrent load or save
// allocates its own pair.
struct IoStage {
    void* pin[2] = {nullptr, nullptr};
    size_t bytes = 0;
    bool cached = false;
};
static std::mutex g_io_stage_mu;
static IoStage g_io_stage;

static int io_stage_acquire(size_t chunk, IoStage* st) {
    if (g_io_stage_mu.try_lock()) {
        if (g_io_stage.bytes < chunk) {
            cudaFreeHost(g_io_stage.pin[0]);
            cudaFreeHost(g_io_stage.pin[1]);
            g_io_stage.pin[0] = g_io_stage.pin[1] = nullptr;
            g_io_stage.bytes = 0;
            if (cudaMallocHost(&g_io_stage.pin[0], chunk) != cudaSuccess || cudaMallocHost(&g_io_stage.pin[1], chunk) != cudaSuccess) {
                cudaGetLastError();
                cudaFreeHost(g_io_stage.pin[0]);
                cudaFreeHost(g_io_stage.pin[1]);
                g_io_stage.pin[0] = g_io_stage.pin[1] = nullptr;
                g_io_stage_mu.unlock();
                return fail(EVS_ENOMEM, "cudaMallocHost of the staging chunks failed");
            }
            g_io_stage.bytes = chunk;
        }
        *st = g_io_stage;
        st->cached = true;
        return EVS_OK;
    }
    st->cached = false;
    st->bytes = chunk;
    if (cudaMallocHost(&st->pin[0], chunk) != cudaSuccess || cudaMallocHost(&st->pin[1], chunk) != cudaSuccess) {
        cudaGetLastError();
        cudaFreeHost(st->pin[0]);
        cudaFreeHost(st->pin[1]);
        st->pin[0] = st->pin[1] = nullptr;
        return fail(EVS_ENOMEM, "cudaMallocHost of the staging chunks failed");
    }
    return EVS_OK;
}

static void io_stage_release(IoStage* st) {
    if (st->cached) {
        g_io_stage_mu.unlock();
    } else {
        cudaFreeHost(st->pin[0]);
        cudaFreeHost(st->pin[1]);
    }
    st->pin[0] = st->pin[1] = nullptr;
}

extern "C" int evs_index_write(const evs_index* idx, const char* path) {
    if (!idx || !path) return fail(EVS_EINVAL, "NULL argument");
    std::lock_guard<std::mutex> lk(idx->mu);  // save_index may race a re-index on another Flask thread
    int rc = use_device(idx->device);
    if (rc) return rc;
    int fd = open(path, O_WRONLY | O_CREAT | O_TRUNC | O_CLOEXEC, 0666);
    if (fd < 0) return fail(EVS_EIO, "cannot open '%s' for writing: %s", path, strerror(errno));
    FlatHeader h;
    memcpy(h.fourcc, "IxFI", 4);
    h.d = idx->d;
    h.ntotal = idx->ntotal;
    h.dummy1 = h.dummy2 = (int64_t)1 << 20;
    h.is_trained = 1;
    h.metric_type = 0;
    h.count = (uint64_t)idx->ntotal * (uint64_t)idx->d;
    bool ok = rw_full(fd, reinterpret_cast<unsigned char*>(&h), sizeof(h), 0, true);
    const size_t total = (size_t)h.count * sizeof(float);
    if (ok && total) {
        const size_t chunk = total < kIoChunk ? total : kIoChunk;
        IoStage st;
        rc = io_stage_acquire(chunk, &st);
        if (rc) {
            close(fd);
            return rc;
        }
        // double-buffered: the device-to-host copy of chunk i+1 runs while the threads write chunk i
        cudaEvent_t ready[2] = {nullptr, nullptr};
        cudaEventCreateWithFlags(&ready[0], cudaEventDisableTiming);
        cudaEventCreateWithFlags(&ready[1], cudaEventDisableTiming);
        cudaError_t e = cudaSuccess;
        auto fetch = [&](size_t off, int b) {
            size_t nb = total - off < chunk ? total - off : chunk;
            cudaError_t r = cudaMemcpyAsync(st.pin[b], reinterpret_cast<const unsigned char*>(idx->xb32) + off, nb, cudaMemcpyDeviceToHost,
                                            idx->stream);
            if (r == cudaSuccess) r = cudaEventRecord(ready[b], idx->stream);
            return r;
        };
        e = fetch(0, 0);
        int b = 0;
        for (size_t off = 0; ok && e == cudaSuccess && off < total; off += chunk, b ^= 1) {
            size_t nb = total - off < chunk ? total - off : chunk;
            if (off + chunk < total) e = fetch(off + chunk, b ^ 1);
            if (e == cudaSuccess) e = cudaEventSynchronize(ready[b]);
            // one writer: concurrent pwrites to one file serialise on the inode lock (8 threads measured slower than 1)
            if (e == cudaSuccess) ok = rw_full(fd, static_cast<unsigned char*>(st.pin[b]), nb, (off_t)(sizeof(h) + off), true);
        }
        cudaStreamSynchronize(idx->stream);
        cudaEventDestroy(ready[0]);
        cudaEventDestroy(ready[1]);
        io_stage_release(&st);
        if (e != cudaSuccess) {
            close(fd);
            return fail(EVS_ECUDA, "device read failed: %s", cudaGetErrorString(e));
        }
    }
    if (close(fd) != 0) ok = false;
    if (!ok) return fail(EVS_EIO, "short write to '%s': %s", path, strerror(errno));
    return EVS_OK;
}

// Read rows [row_lo, row_hi) of the file's payload (row_hi < 0: to the end) into a new index whose id_base is row_lo:
// the loader of one shard of a row-sharded index -- every rank reads only its own byte range of index.faiss.
static int read_rows(const char* path, int device, int storage, int64_t row_lo, int64_t row_hi, evs_index** out, int64_t* ntotal_file) {
    if (!path || !out) return fail(EVS_EINVAL, "NULL argument");
    *out = nullptr;
    int fd = open(path, O_RDONLY | O_CLOEXEC);
    if (fd < 0) return fail(EVS_EIO, "cannot open '%s': %s", path, strerror(errno));
    FlatHeader h;
    if (!rw_full(fd, reinterpret_cast<unsigned char*>(&h), sizeof(h), 0, false)) {
        close(fd);
        return fail(EVS_EFORMAT, "'%s': truncated header", path);
    }
    const bool ip = !memcmp(h.fourcc, "IxFI", 4);
    if (!ip && memcmp(h.fourcc, "IxF2", 4) && memcmp(h.fourcc, "IxFl", 4)) {
        close(fd);
        return fail(EVS_EFORMAT, "'%s': not a flat index (fourcc %.4s)", path, h.fourcc);
    }
    if (h.metric_type != 0) {
        close(fd);
        return fail(EVS_EFORMAT, "'%s': metric %d is not inner product", path, h.metric_type);
    }
    if (h.d <= 0 || h.ntotal < 0 || h.count >= ((uint64_t)1 << 40) || h.count != (uint64_t)h.ntotal * (uint64_t)h.d) {
        close(fd);
        return fail(EVS_EFORMAT, "'%s': inconsistent header (d=%d ntotal=%lld count=%llu)", path, h.d, (long long)h.ntotal,
                    (unsigned long long)h.count);
    }
    struct stat sb;
    if (fstat(fd, &sb) == 0 && (uint64_t)sb.st_size < sizeof(h) + h.count * 4) {
        close(fd);
        return fail(EVS_EFORMAT, "'%s': truncated payload", path);
    }
    if (ntotal_file) *ntotal_file = h.ntotal;
    if (row_hi < 0 || row_hi > h.ntotal) row_hi = h.ntotal;
    if (row_lo < 0 || row_lo > row_hi) {
        close(fd);
        return fail(EVS_EINVAL, "rows [%lld, %lld) out of range for '%s' (%lld rows)", (long long)row_lo, (long long)row_hi, path,
                    (long long)h.ntotal);
    }
    const int64_t nrows = row_hi - row_lo;
    evs_index* idx = nullptr;
    int rc = evs_index_create(h.d, device, storage, &idx);
    if (rc) {
        close(fd);
        return rc;
    }
    idx->id_base = row_lo;
    const size_t total = (size_t)nrows * (size_t)h.d * sizeof(float);
    if (total) {
        const off_t base = (off_t)(sizeof(h) + (size_t)row_lo * (size_t)h.d * sizeof(float));
#ifdef POSIX_FADV_SEQUENTIAL
        posix_fadvise(fd, base, (off_t)total, POSIX_FADV_SEQUENTIAL);
#endif
        {
            std::lock_guard<std::mutex> lk(idx->mu);
            rc = grow_locked(idx, nrows);
        }
        const size_t chunk = total < kIoChunk ? total : kIoChunk;
        IoStage st;
        bool staged = false;
        if (!rc) {
            rc = io_stage_acquire(chunk, &st);
            staged = !rc;
        }
        // double-buffered: the threads fill one pinned chunk while the other is in flight to the device
        cudaEvent_t done[2] = {nullptr, nullptr};
        if (!rc) {
            cudaEventCreateWithFlags(&done[0], cudaEventDisableTiming);
            cudaEventCreateWithFlags(&done[1], cudaEventDisableTiming);
        }
        int b = 0;
        for (size_t off = 0; !rc && off < total; off += chunk, b ^= 1) {
            size_t nb = total - off < chunk ? total - off : chunk;
            cudaEventSynchronize(done[b]);
            if (!rw_parallel(fd, st.pin[b], nb, base + (off_t)off, false)) {
                rc = fail(EVS_EFORMAT, "'%s': short read", path);
                break;
            }
            cudaError_t e = cudaMemcpyAsync(reinterpret_cast<unsigned char*>(idx->xb32) + off, st.pin[b], nb, cudaMemcpyHostToDevice,
                                            idx->stream);
            if (e == cudaSuccess) e = cudaEventRecord(done[b], idx->stream);
            if (e != cudaSuccess) rc = fail(EVS_ECUDA, "upload failed: %s", cudaGetErrorString(e));
        }
        if (!rc) {
            std::lock_guard<std::mutex> lk(idx->mu);
            rc = finish_add_locked(idx, nrows);
        }
        // the staging chunks go back to the next load: nothing of this one may still be reading them
        if (staged) cudaStreamSynchronize(idx->stream);
        if (done[0]) cudaEventDestroy(done[0]);
        if (done[1]) cudaEventDestroy(done[1]);
        if (staged) io_stage_release(&st);
    }
    close(fd);
    if (rc) {
        evs_index_free(idx);
        return rc;
    }
    *out = idx;
    return EVS_OK;
}

extern "C" int evs_index_read(const char* path, int device, int storage, evs_index** out) {
    return read_rows(path, device, storage, 0, -1, out, nullptr);
}

extern "C" int evs_index_read_rows(const char* path, int device, int storage, int64_t row_lo, int64_t row_hi, evs_index** out,
                                   int64_t* ntotal_file) {
    return read_rows(path, device, storage, row_lo, row_hi, out, ntotal_file);
}

extern "C" int evs_index_file_info(const char* path, int* d, int64_t* ntotal) {
    if (!path) return fail(EVS_EINVAL, "path is NULL");
    FILE* f = fopen(path, "rb");
    if (!f) return fail(EVS_EIO, "cannot open '%s': %s", path, strerror(errno));
    FlatHeader h;
    const bool ok = fread(&h, sizeof(h), 1, f) == 1;
    fclose(f);
    if (!ok) return fail(EVS_EFORMAT, "'%s': truncated header", path);
    if (memcmp(h.fourcc, "IxFI", 4) && memcmp(h.fourcc, "IxF2", 4) && memcmp(h.fourcc, "IxFl", 4))
        return fail(EVS_EFORMAT, "'%s': not a flat index (fourcc %.4s)", path, h.fourcc);
    if (h.d <= 0 || h.ntotal < 0 || h.count != (uint64_t)h.ntotal * (uint64_t)h.d)
        return fail(EVS_EFORMAT, "'%s': inconsistent header", path);
    if (d) *d = h.d;
    if (ntotal) *ntotal = h.ntotal;
    return EVS_OK;
}

// Switch the scan precision of an index in place: EVS_STORE_BF16_F32 derives the bf16 scan copy (large batches over
// fp32-storage indexes otherwise scan in tf32 straight from the fp32 rows: twice the bytes through L2 for no gain in
// accuracy after the canonical re-score); EVS_STORE_F32 drops it.
extern "C" int evs_index_set_storage(evs_index* idx, int storage) {
    if (!idx) return fail(EVS_EINVAL, "idx is NULL");
    if (storage != EVS_STORE_F32 && storage != EVS_STORE_BF16_F32) return fail(EVS_EINVAL, "unknown storage %d", storage);
    std::lock_guard<std::mutex> lk(idx->mu);
    int rc = use_device(idx->device);
    if (rc) return rc;
    if (storage == idx->storage) return EVS_OK;
    CU(cudaDeviceSynchronize());  // no search may be in flight while the scan rows change
    if (storage == EVS_STORE_F32) {
        cudaFree(idx->xb16);
        idx->xb16 = nullptr;
        if (!shadow_wanted()) drop_i8_copy(idx);  // otherwise the int8 copy stays: it is the fp32 index's scan copy
        idx->storage = storage;
        return EVS_OK;
    }
    if (idx->capacity > 0) {  // the bf16 rows, and the int8 copy bf16 storage always keeps, in one pass over the rows
        CU(cudaMalloc(&idx->xb16, (size_t)idx->capacity * idx->d * 2));
        if (idx->xi8 == nullptr && (rc = alloc_i8_copy(idx))) {
            cudaFree(idx->xb16);
            idx->xb16 = nullptr;
            return rc;
        }
        if (idx->ntotal > 0) {
            const int rc2 = derive_rows_locked(idx, 0, idx->ntotal);
            if (rc2) {
                cudaFree(idx->xb16);
                idx->xb16 = nullptr;
                return rc2;
            }
        }
    }
    idx->storage = storage;
    return EVS_OK;
}
