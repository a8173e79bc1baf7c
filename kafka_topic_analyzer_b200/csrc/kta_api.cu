// kta_api.cu — host side of libkta_gpu.so: the C ABI of include/kta.h over the sm_100a kernels.
//
// Mirrors, for this one path, what the reference's host does around the handlers:
//   MessageMetrics::new / LogCompactionInMemoryMetrics::new      src/metric.rs:30-46, 267-271
//   one handle_message per polled record                         src/kafka.rs:107-109
//   getters + derived values read by the report                  src/metric.rs:104-203, src/main.rs:130-170
// There is deliberately no CPU implementation of the scan in this file: if CUDA is unusable every
// compute entry point fails with KTA_ERR_CUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

#include "kta_kernels.cuh"
#include "kta_logdecode.cuh"
#include "kta_synth.h"

using namespace kta;

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                                     \
    do {                                                                                             \
        cudaError_t e_ = (call);                                                                     \
        if (e_ != cudaSuccess)                                                                       \
            return fail(e_ == cudaErrorMemoryAllocation ? KTA_ERR_NOMEM : KTA_ERR_CUDA, "%s: %s (%s:%d)", #call, \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                                 \
    } while (0)

extern "C" const char *kta_last_error(void) { return g_err; }
extern "C" int kta_abi_version(void) { return KTA_ABI_VERSION; }
extern "C" int kta_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return -1;
    }
    return n;
}

// ------------------------------------------------------------------------------------------------
// handle
// ------------------------------------------------------------------------------------------------
static constexpr int NCHUNK = 3;
static constexpr int32_t ALIVE_DEFAULT_KIB = 256 * 1024;       // initial alive-key table: 256 MiB = 2^25 slots (KTA_ALIVE_TABLE_KIB overrides: tuning)
static constexpr int32_t ALIVE_MAX_KIB = 32 * 1024 * 1024;     // 32 GiB = one slot per possible 32-bit hash
static constexpr int64_t ALIVE_CACHE_MIN_RECORDS = 1 << 20;    // smaller batches go straight to the table
static constexpr int64_t DEFAULT_RING_RECORDS = 1 << 22;  // 4 Mi records per chunk

struct Chunk {
    // device staging (shared by kta_push and kta_push_batch_host)
    int32_t *d_partition = nullptr, *d_klen = nullptr, *d_vlen = nullptr;
    int64_t *d_ts = nullptr;
    uint64_t *d_seq = nullptr;
    uint8_t *d_keys = nullptr;
    uint64_t *d_tile_base = nullptr;
    cudaEvent_t free_ev = nullptr;  // recorded after the scan that reads this chunk
    uint32_t *h_status = nullptr;   // pinned [2]: snapshot of the alive-table status words taken right after that scan
    // pinned landing area for kta_push
    int32_t *h_partition = nullptr, *h_klen = nullptr, *h_vlen = nullptr;
    int64_t *h_ts = nullptr;
    uint8_t *h_keys = nullptr;
    uint64_t *h_tile_base = nullptr;
};

// a MODE_EXACT scan whose stamps have not been confirmed yet (the alive table may turn out too small: then it is
// grown and these are re-run stamps-only; their input buffers are still valid — caller buffers until kta_sync /
// kta_finalize by contract, ring chunks until they are reused)
struct PendingScan {
    ScanParams prm;
    int64_t key_readable, key_bytes;
    int chunk;   // ring chunk the columns live in, -1 = caller-owned / scratch device buffers
};

struct kta_handle {
    kta_config cfg{};
    int device = 0;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = true;
    bool need_hash = false;
    // device state
    unsigned long long *d_sums = nullptr;
    long long *d_minmax = nullptr;
    uint32_t *d_hll = nullptr;
    uint32_t *d_hll_floor = nullptr;
    unsigned long long *d_alive_table = nullptr;   // open-addressed last-writer table, 2 * alive_pairs slots
    uint32_t alive_pairs = 0;
    uint64_t alive_origin = 0;               // seq that a stamp's field value 1 stands for
    bool alive_rebased = false;              // a rebase dropped absolute sequence numbers (exports are refused then)
    uint32_t *d_alive_cache = nullptr;       // seen cache of the batch being scanned (32 MiB, cleared per launch)
    uint32_t *d_alive_status = nullptr;      // [0] stamps that found no slot, [1] records outside the seq window
    uint32_t *h_alive_status = nullptr;      // pinned copy
    uint64_t alive_window_errors = 0;        // sticky until reset: reported by kta_finalize
    uint64_t alive_grows = 0, alive_reruns = 0;
    uint64_t alive_now = 0, alive_occupied = 0;   // counted by the last alive_check
    std::vector<PendingScan> pending;
    unsigned long long *d_scalar = nullptr;  // [0] alive count, [1] export cursor, [2] occupied slots, [3] spare,
                                             // [4..] hll floor + slice minima (u32)
    uint32_t *d_hash_out = nullptr;          // test hook
    uint64_t *d_tb_scratch = nullptr;        // key_tile_base scratch for device batches
    int64_t tb_scratch_tiles = 0;
    // RecordBatch decoder scratch (kta_scan_log_segment_device / kta_push_log_segment_host)
    uint8_t *d_log_bytes = nullptr; int64_t log_bytes_cap = 0;       // raw segment staged from the host
    uint64_t *d_log_off = nullptr;                                    // batch offsets staged from the host
    LogBatchInfo *d_log_info = nullptr; uint64_t *d_log_cnt = nullptr; int64_t log_batch_cap = 0;
    int32_t *d_dec_part = nullptr, *d_dec_klen = nullptr, *d_dec_vlen = nullptr; int64_t *d_dec_ts = nullptr; int64_t dec_rec_cap = 0;
    uint8_t *d_dec_keys = nullptr; int64_t dec_key_cap = 0;
    uint64_t *d_dec_ksrc = nullptr;          // per decoded record: where its key bytes lie in the segment buffer
    uint8_t *d_unc = nullptr; int64_t unc_cap = 0;   // uncompressed images of LZ4 / Snappy batches
    uint64_t *d_unc_slot = nullptr; int64_t unc_slot_cap = 0;
    uint32_t *d_log_err = nullptr;
    size_t nsums = 0, nhll = 0;
    // landing ring
    Chunk chunks[NCHUNK];
    bool ring_dev_ready = false, ring_host_ready = false;
    int64_t ring_records = 0, ring_key_bytes = 0;
    int cur = 0;          // chunk being filled by kta_push
    // kta_push's hot state: raw cursors into that chunk's pinned landing area (one cache line, no indirection per call)
    struct PushCursor {
        int32_t *part = nullptr, *klen = nullptr, *vlen = nullptr;
        int64_t *ts = nullptr;
        uint8_t *keys = nullptr;
        uint64_t *tile_base = nullptr;
        int64_t n = 0, cap = 0;     // records in the chunk / its capacity (0 until the ring exists: first push takes the slow path)
        int64_t kb = 0, kcap = 0;   // key bytes in the chunk / capacity
        bool hash = false;          // key bytes travel only when they are hashed
    } pc;
    uint64_t next_seq = 0;   // seq of the first record not yet handed to a scan (records in the open chunk follow it)
    // host mirror (valid after finalize)
    bool finalized = false;
    std::vector<uint64_t> h_sums;
    long long h_minmax[4] = {0, 0, 0, 0};
    std::vector<uint32_t> h_hll;
    uint64_t h_alive = 0;
    // occupancy-derived grids
    int shard_world = 1, shard_rank = 0;     // partition-sharded scan: only partitions p % world == rank reach this handle
    int columns = 0;                         // counter columns the scan kernel carves = partitions this handle owns
    bool smem_counters = true;               // per-partition counters fit in shared memory
    size_t smem_optin = 0;
    // stats / timing
    uint64_t launches = 0, records = 0;
    bool timing = false;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> ev_pool;
    size_t ev_used = 0;
    double scan_ms = 0;
    uint64_t scan_launches_timed = 0;
};

static int set_device(const kta_handle *h) {
    CU(cudaSetDevice(h->device));
    return KTA_OK;
}

static size_t scan_smem_bytes(bool hash, bool smem, int P, int threads, int keybuf, bool exact) {
    return (smem ? smem_counter_bytes(P) : CTA_SCRATCH) + (size_t)(threads / 32) * warp_smem_bytes(hash, keybuf, exact);
}

// Launch shape for one scan: key-stage bytes from the batch's mean key length, then as many warps as fit.
static void scan_shape(const kta_handle *h, bool hash, bool exact, int64_t n, int64_t key_bytes, int &threads, int &keybuf, size_t &smem) {
    keybuf = KEYBUF_MIN;
    if (hash && n > 0) {
        const int64_t per_tile = (key_bytes * TILE + n - 1) / n;           // mean key bytes per 128-record tile
        int64_t want = per_tile + per_tile / 8 + 64 + KEYBUF_SLACK;       // 12.5 % headroom for ragged tiles (~2.4 sigma for 0..40 B keys)
        want = (want + 127) / 128 * 128;
        keybuf = (int)std::min<int64_t>(std::max<int64_t>(want, KEYBUF_MIN), KEYBUF_MAX);
        keybuf = (keybuf + 15) / 16 * 16;
    }
    const int P = h->columns;
    // Leave the SM some L1: the header loads stream through it, and with (almost) all 228 KB carved out as shared
    // memory the loads in flight are throttled (measured at P = 256).  KTA_SCAN_L1_RESERVE (bytes) is a tuning knob.
    static const size_t l1_reserve = [] { const char *e = getenv("KTA_SCAN_L1_RESERVE"); return e ? (size_t)atoll(e) : (size_t)0; }();
    const size_t budget = h->smem_optin > l1_reserve ? h->smem_optin - l1_reserve : h->smem_optin;
    for (threads = MAX_THREADS;; threads -= 128) {
        smem = scan_smem_bytes(hash, h->smem_counters, P, threads, keybuf, exact);
        if (smem <= budget || threads <= 256) break;
    }
    if (smem > h->smem_optin) {   // still too big with 8 warps: fall back to the smallest stage (long keys go through global)
        keybuf = KEYBUF_MIN;
        for (threads = MAX_THREADS;; threads -= 128) {
            smem = scan_smem_bytes(hash, h->smem_counters, P, threads, keybuf, exact);
            if (smem <= h->smem_optin || threads <= 128) break;
        }
    }
}

// one persistent CTA per SM; every variant may use the whole opt-in shared memory (the shape is chosen per launch).
// variant index: 0 counters, 1 HLL, 2 exact, 3 HLL+capture, 4 exact+capture, 5..7 = 0..2 for a partition-sharded handle
template <int MODE, bool SMEM, bool CAPTURE, bool SHARD>
static int prepare_variant(kta_handle *h) {
    CU(cudaFuncSetAttribute(scan_kernel<MODE, SMEM, CAPTURE, SHARD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_optin));
    return KTA_OK;
}

template <bool SMEM>
static int prepare_all(kta_handle *h) {
    int rc;
    if ((rc = prepare_variant<MODE_COUNTERS, SMEM, false, false>(h))) return rc;
    if ((rc = prepare_variant<MODE_HLL, SMEM, false, false>(h))) return rc;
    if ((rc = prepare_variant<MODE_EXACT, SMEM, false, false>(h))) return rc;
    if ((rc = prepare_variant<MODE_HLL, SMEM, true, false>(h))) return rc;
    if ((rc = prepare_variant<MODE_EXACT, SMEM, true, false>(h))) return rc;
    if ((rc = prepare_variant<MODE_COUNTERS, SMEM, false, true>(h))) return rc;
    if ((rc = prepare_variant<MODE_HLL, SMEM, false, true>(h))) return rc;
    if ((rc = prepare_variant<MODE_EXACT, SMEM, false, true>(h))) return rc;
    return KTA_OK;
}

template <bool SMEM>
static void launch_variant(int v, int grid, int threads, size_t sm, cudaStream_t st, const ScanParams &prm) {
    switch (v) {
        case 0: scan_kernel<MODE_COUNTERS, SMEM, false><<<grid, threads, sm, st>>>(prm); break;
        case 1: scan_kernel<MODE_HLL, SMEM, false><<<grid, threads, sm, st>>>(prm); break;
        case 2: scan_kernel<MODE_EXACT, SMEM, false><<<grid, threads, sm, st>>>(prm); break;
        case 3: scan_kernel<MODE_HLL, SMEM, true><<<grid, threads, sm, st>>>(prm); break;
        case 4: scan_kernel<MODE_EXACT, SMEM, true><<<grid, threads, sm, st>>>(prm); break;
        case 5: scan_kernel<MODE_COUNTERS, SMEM, false, true><<<grid, threads, sm, st>>>(prm); break;
        case 6: scan_kernel<MODE_HLL, SMEM, false, true><<<grid, threads, sm, st>>>(prm); break;
        default: scan_kernel<MODE_EXACT, SMEM, false, true><<<grid, threads, sm, st>>>(prm); break;
    }
}

static int state_reset_device(kta_handle *h) {
    state_init_kernel<<<64, 256, 0, h->stream>>>(h->d_sums, h->nsums, h->d_minmax, h->d_hll, h->nhll, h->d_hll_floor);
    h->launches++;
    CU(cudaGetLastError());
    if (h->d_alive_table) {
        // the table is a few hundred MB at most for the topics it is meant for: wiping it is a ~20 µs memset
        CU(cudaMemsetAsync(h->d_alive_table, 0xff, (size_t)h->alive_pairs * 16, h->stream));
        CU(cudaMemsetAsync(h->d_scalar, 0, 32, h->stream));
        CU(cudaMemsetAsync(h->d_alive_status, 0, 8, h->stream));
        h->alive_now = h->alive_occupied = 0;
        h->alive_origin = 0;
        h->alive_rebased = false;
        h->alive_window_errors = 0;
        h->pending.clear();
    }
    return KTA_OK;
}

static void free_chunk(Chunk &c) {
    cudaFreeHost(c.h_status);
    cudaFree(c.d_partition); cudaFree(c.d_klen); cudaFree(c.d_vlen); cudaFree(c.d_ts); cudaFree(c.d_seq);
    cudaFree(c.d_keys); cudaFree(c.d_tile_base);
    if (c.free_ev) cudaEventDestroy(c.free_ev);
    cudaFreeHost(c.h_partition); cudaFreeHost(c.h_klen); cudaFreeHost(c.h_vlen); cudaFreeHost(c.h_ts);
    cudaFreeHost(c.h_keys); cudaFreeHost(c.h_tile_base);
    c = Chunk{};
}

extern "C" int kta_destroy(kta_handle *h) {
    if (!h) return KTA_OK;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (auto &c : h->chunks) free_chunk(c);
    cudaFree(h->d_sums); cudaFree(h->d_minmax); cudaFree(h->d_hll); cudaFree(h->d_alive_table);
    cudaFree(h->d_alive_status); cudaFree(h->d_alive_cache); cudaFreeHost(h->h_alive_status); cudaFree(h->d_scalar); cudaFree(h->d_tb_scratch);
    cudaFree(h->d_log_bytes); cudaFree(h->d_log_off); cudaFree(h->d_log_info); cudaFree(h->d_log_cnt);
    cudaFree(h->d_dec_part); cudaFree(h->d_dec_klen); cudaFree(h->d_dec_vlen); cudaFree(h->d_dec_ts); cudaFree(h->d_dec_keys); cudaFree(h->d_dec_ksrc); cudaFree(h->d_unc); cudaFree(h->d_unc_slot);
    cudaFree(h->d_log_err);
    for (auto &e : h->ev_pool) { cudaEventDestroy(e.first); cudaEventDestroy(e.second); }
    if (h->stream && h->own_stream) cudaStreamDestroy(h->stream);
    cudaGetLastError();
    delete h;
    return KTA_OK;
}

static int create_impl(const kta_config *cfg, kta_handle *h) {
    h->cfg = *cfg;
    if (cfg->num_partitions < 1 || cfg->num_partitions > (1 << 20))
        return fail(KTA_ERR_INVALID, "num_partitions %d out of range [1, 2^20]", cfg->num_partitions);
    if (cfg->hll_precision != 0 && (cfg->hll_precision < 4 || cfg->hll_precision > 18))
        return fail(KTA_ERR_INVALID, "hll_precision %d not 0 or 4..18", cfg->hll_precision);
    int ndev = 0;
    CU(cudaGetDeviceCount(&ndev));
    if (ndev < 1) return fail(KTA_ERR_CUDA, "no CUDA device (this library has no CPU fallback)");
    if (cfg->device >= 0) h->device = cfg->device;
    else CU(cudaGetDevice(&h->device));
    if (h->device >= ndev) return fail(KTA_ERR_INVALID, "device %d >= device count %d", h->device, ndev);
    CU(cudaSetDevice(h->device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, h->device));
    if (prop.major < 10) return fail(KTA_ERR_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only",
                                     prop.name, prop.major, prop.minor);
    h->sm_count = prop.multiProcessorCount;
    CU(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    h->need_hash = cfg->count_alive_keys == 1 || cfg->hll_precision != 0;
    h->pc.hash = h->need_hash;   // kta_push reads it before its first (slow-path) call has bound the ring
    if (cfg->now_s == INT64_MIN) {
        const auto now = std::chrono::system_clock::now().time_since_epoch();
        const int64_t ns = std::chrono::duration_cast<std::chrono::nanoseconds>(now).count();
        h->cfg.now_s = ns / 1000000000ll;
        h->cfg.now_ns = (int32_t)(ns % 1000000000ll);
    }
    h->ring_records = cfg->ring_records > 0 ? cfg->ring_records : DEFAULT_RING_RECORDS;
    h->ring_records = (h->ring_records + TILE - 1) / TILE * TILE;
    h->ring_key_bytes = cfg->ring_key_bytes > 0 ? cfg->ring_key_bytes : h->ring_records * 24;

    const int P = cfg->num_partitions;
    h->nsums = sums_words(P);
    h->nhll = cfg->hll_precision ? ((size_t)1 << cfg->hll_precision) : 0;
    CU(cudaMalloc(&h->d_sums, h->nsums * 8));
    CU(cudaMalloc(&h->d_minmax, 4 * 8));
    CU(cudaMalloc(&h->d_scalar, 4 * 8 + (HLL_SLICES + 1) * 4 + 4));
    h->d_hll_floor = reinterpret_cast<uint32_t *>(h->d_scalar + 4);
    if (h->nhll) CU(cudaMalloc(&h->d_hll, h->nhll * 4));
    if (cfg->count_alive_keys == 1) {
        // open-addressed last-writer table keyed by the 32-bit hash, sized by the number of DISTINCT hashes and grown
        // on demand (alive_check): 256 MiB = 2^25 slots holds the 1e7 keys of BASELINE configs[2] at load 0.3 (measured:
        // at 0.6 every third first-seen key finds its home pair taken and probes on — 10 % of the kernel time; the
        // table does not fit L2 at either size)
        if (cfg->alive_table_kib < 0 || cfg->alive_table_kib > ALIVE_MAX_KIB)
            return fail(KTA_ERR_INVALID, "alive_table_kib %d out of range [0, %d]", cfg->alive_table_kib, ALIVE_MAX_KIB);
        static const int64_t env_kib = [] { const char *e = getenv("KTA_ALIVE_TABLE_KIB"); return e ? atoll(e) : 0ll; }();   // tuning knob
        const int64_t kib = cfg->alive_table_kib ? cfg->alive_table_kib : env_kib > 0 ? env_kib : ALIVE_DEFAULT_KIB;
        h->alive_pairs = (uint32_t)std::max<int64_t>(kib * 64, 16);   // 16 bytes per pair
        CU(cudaMalloc(&h->d_alive_table, (size_t)h->alive_pairs * 16));
        CU(cudaMalloc(&h->d_alive_status, 8));
        CU(cudaMalloc(&h->d_alive_cache, ((size_t)4 << ALIVE_CACHE_SET_BITS)));
        CU(cudaHostAlloc(&h->h_alive_status, 8, cudaHostAllocDefault));
    }
    h->smem_optin = prop.sharedMemPerBlockOptin;
    if (cfg->shard_world > 1) {
        if (cfg->shard_rank < 0 || cfg->shard_rank >= cfg->shard_world || cfg->shard_world > P)
            return fail(KTA_ERR_INVALID, "shard_rank %d / shard_world %d invalid for %d partitions", cfg->shard_rank, cfg->shard_world, P);
        h->shard_world = cfg->shard_world;
        h->shard_rank = cfg->shard_rank;
    }
    h->columns = (P - h->shard_rank + h->shard_world - 1) / h->shard_world;   // partitions p < P with p % world == rank
    // counters in shared memory as long as at least 8 warps still fit beside them
    h->smem_counters = smem_counter_bytes(h->columns) + 8 * warp_smem_bytes(true, KEYBUF_MIN, true) <= h->smem_optin;
    int rc;
    if ((rc = h->smem_counters ? prepare_all<true>(h) : prepare_all<false>(h))) return rc;
    if ((rc = state_reset_device(h))) return rc;
    CU(cudaStreamSynchronize(h->stream));
    return KTA_OK;
}

extern "C" int kta_create(const kta_config *cfg, kta_handle **out) {
    if (!cfg || !out) return fail(KTA_ERR_INVALID, "null argument");
    if (cfg->struct_size != (int32_t)sizeof(kta_config))
        return fail(KTA_ERR_INVALID, "kta_config.struct_size %d != %zu (ABI version %d)", cfg->struct_size, sizeof(kta_config), KTA_ABI_VERSION);
    kta_handle *h = new (std::nothrow) kta_handle();
    if (!h) return fail(KTA_ERR_NOMEM, "out of host memory");
    const int rc = create_impl(cfg, h);
    if (rc) {
        char keep[sizeof(g_err)];
        memcpy(keep, g_err, sizeof(keep));
        kta_destroy(h);
        memcpy(g_err, keep, sizeof(keep));
        *out = nullptr;
        return rc;
    }
    *out = h;
    return KTA_OK;
}

extern "C" void *kta_stream(kta_handle *h) { return h ? (void *)h->stream : nullptr; }

extern "C" int kta_set_stream(kta_handle *h, void *stream) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    int rc;
    if ((rc = set_device(h))) return rc;
    CU(cudaStreamSynchronize(h->stream));
    if (h->own_stream) CU(cudaStreamDestroy(h->stream));
    h->stream = (cudaStream_t)stream;
    h->own_stream = false;
    return KTA_OK;
}

// ------------------------------------------------------------------------------------------------
// scan launch
// ------------------------------------------------------------------------------------------------
// one launch of the fused scan; prm is complete apart from the state pointers filled in here
static int launch_scan_raw(kta_handle *h, ScanParams prm, int64_t key_readable, int64_t key_bytes, const uint64_t *seq_ends = nullptr) {
    const int P = h->cfg.num_partitions;
    const bool exact = h->cfg.count_alive_keys == 1;
    const bool capture = h->d_hash_out != nullptr && !prm.alive_only;
    // with -c the sketch is built from the resolved set at finalize, not in-stream.  A capture-only
    // handle (no -c, no HLL) runs the HLL-mode kernel against a null sketch of precision 0.
    const int mode = exact ? MODE_EXACT : (h->cfg.hll_precision || capture) ? MODE_HLL : MODE_COUNTERS;
    if (mode == MODE_HLL && !h->cfg.hll_precision)
        return fail(KTA_ERR_INVALID, "hash capture needs count_alive_keys or hll_precision");
    prm.shard_world = h->shard_world;
    prm.shard_rank = h->shard_rank;
    prm.Pc = h->columns;
    prm.shard_magic = h->shard_world > 1 ? (uint32_t)((((uint64_t)1 << 32) + (uint64_t)h->shard_world - 1) / (uint64_t)h->shard_world) : 0u;
    prm.ntiles = (prm.n + TILE - 1) / TILE;
    if (prm.ntiles >= (int64_t)1 << 30) return fail(KTA_ERR_INVALID, "batch of %lld records: split it (one scan takes < 2^37 records)", (long long)prm.n);
    prm.P = P;
    prm.hll_p = h->cfg.hll_precision;
    prm.sums = h->d_sums;
    prm.minmax = h->d_minmax;
    prm.hll = h->d_hll;
    prm.hll_floor = h->d_hll_floor;
    prm.alive_table = h->d_alive_table;
    prm.alive_pairs = h->alive_pairs;
    prm.alive_origin = h->alive_origin;
    prm.alive_count = h->d_scalar;
    prm.alive_status = h->d_alive_status;
    prm.alive_cache = nullptr;
    if (exact && prm.n >= ALIVE_CACHE_MIN_RECORDS) {
        // the seen cache pays for its clearing (32 MiB, ~10 µs) on batches of a million records and more.
        // Waves cut the batch's seq range [lo, hi] into <= 127 equal slices (any monotone function of seq will do).
        static const bool off = getenv("KTA_ALIVE_NO_CACHE") != nullptr;   // tuning / ablation knob
        uint64_t lo = prm.seq_base, hi = prm.seq_base + (uint64_t)prm.n - 1;
        bool ok = !off;
        if (ok && prm.seq) {
            // explicit sequence numbers: the range is read off the column's ends (records of a batch are in seq order; a
            // record outside the range just lands in the first or last wave)
            uint64_t ends[2];
            if (seq_ends) { ends[0] = seq_ends[0]; ends[1] = seq_ends[1]; }
            else {
                CU(cudaMemcpyAsync(&ends[0], prm.seq, 8, cudaMemcpyDeviceToHost, h->stream));
                CU(cudaMemcpyAsync(&ends[1], prm.seq + (prm.n - 1), 8, cudaMemcpyDeviceToHost, h->stream));
                CU(cudaStreamSynchronize(h->stream));
            }
            lo = std::min(ends[0], ends[1]);
            hi = std::max(ends[0], ends[1]);
            ok = lo >= h->alive_origin && hi - h->alive_origin < (uint64_t)ALIVE_FIELD_MAX;
        }
        if (ok) {
            CU(cudaMemsetAsync(h->d_alive_cache, 0, (size_t)4 << ALIVE_CACHE_SET_BITS, h->stream));
            prm.alive_cache = h->d_alive_cache;
            int sh = 0;
            while (((hi - lo) >> sh) + 1 > (uint64_t)ALIVE_CACHE_WAVES) sh++;
            prm.alive_wave_shift = sh;
            prm.alive_wave_base = (uint32_t)(lo - h->alive_origin + 1ull);   // the stamp field of seq lo
        }
    }
    prm.hash_out = capture ? h->d_hash_out : nullptr;
    if (mode != MODE_COUNTERS) {
        if (!prm.key_tile_base) return fail(KTA_ERR_INVALID, "internal: key_tile_base missing");
        if (!prm.key_bytes && key_readable > 0) return fail(KTA_ERR_INVALID, "key_bytes is NULL but keys are required");
        prm.stage_limit = (((uintptr_t)prm.key_bytes & 15u) == 0) ? ((uint64_t)key_readable & ~15ull) : 0;
    }
    if (capture && h->shard_world > 1) return fail(KTA_ERR_INVALID, "hash capture is not available on a partition-sharded handle");
    const int variant = h->shard_world > 1 ? 5 + mode : mode + (capture ? 2 : 0);
    int threads = 0, keybuf = 0;
    size_t sm = 0;
    scan_shape(h, mode != MODE_COUNTERS, mode == MODE_EXACT, prm.n, key_bytes, threads, keybuf, sm);
    if (sm > h->smem_optin) return fail(KTA_ERR_INVALID, "scan kernel does not fit: %zu B shared memory", sm);
    prm.keybuf = keybuf;
    const int grid = (int)std::min<int64_t>((prm.ntiles + threads / 32 - 1) / (threads / 32), h->sm_count);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (h->timing) {
        if (h->ev_used == h->ev_pool.size()) {
            cudaEvent_t a, b;
            CU(cudaEventCreate(&a));
            CU(cudaEventCreate(&b));
            h->ev_pool.emplace_back(a, b);
        }
        e0 = h->ev_pool[h->ev_used].first;
        e1 = h->ev_pool[h->ev_used].second;
        h->ev_used++;
        CU(cudaEventRecord(e0, h->stream));
    }
    if (h->smem_counters) launch_variant<true>(variant, grid, threads, sm, h->stream, prm);
    else launch_variant<false>(variant, grid, threads, sm, h->stream, prm);
    CU(cudaGetLastError());
    h->launches++;
    if (h->timing) CU(cudaEventRecord(e1, h->stream));
    return KTA_OK;
}

// ------------------------------------------------------------------------------------------------
// alive-key table upkeep: seq window (rebase), confirmation of pending stamps, growth (rehash + re-run)
// ------------------------------------------------------------------------------------------------
static int alive_grow(kta_handle *h, uint32_t new_pairs) {
    cudaStream_t s = h->stream;
    unsigned long long *nt = nullptr;
    CU(cudaMalloc(&nt, (size_t)new_pairs * 16));
    CU(cudaMemsetAsync(nt, 0xff, (size_t)new_pairs * 16, s));
    const size_t old_slots = (size_t)h->alive_pairs * 2;
    alive_rehash_kernel<<<h->sm_count * 8, THREADS, 0, s>>>(h->d_alive_table, old_slots, nt, new_pairs, h->d_alive_status);
    h->launches++;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(s));
    cudaFree(h->d_alive_table);
    h->d_alive_table = nt;
    h->alive_pairs = new_pairs;
    h->alive_grows++;
    return KTA_OK;
}

// Confirms every pending MODE_EXACT scan: waits for the stream, reads the status words, and while stamps were dropped
// for lack of room grows the table and re-runs the pending batches stamps-only (idempotent: atomicMax).  Afterwards
// nothing is pending.  Also grows ahead of need once the table is more than 70 % full.
static int alive_check(kta_handle *h) {
    if (!h->d_alive_table) return KTA_OK;
    cudaStream_t s = h->stream;
    for (int round = 0;; round++) {
        unsigned long long counts[3] = {0, 0, 0};   // alive, (export cursor), occupied
        CU(cudaMemsetAsync(h->d_scalar, 0, 24, s));
        alive_count_kernel<<<h->sm_count * 8, THREADS, 0, s>>>(h->d_alive_table, (size_t)h->alive_pairs * 2, h->d_scalar);
        h->launches++;
        CU(cudaGetLastError());
        CU(cudaMemcpyAsync(h->h_alive_status, h->d_alive_status, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(counts, h->d_scalar, 24, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        const unsigned long long occupied = counts[2];
        h->alive_now = counts[0];
        h->alive_occupied = occupied;
        const uint32_t dropped = h->h_alive_status[0];
        h->alive_window_errors += h->h_alive_status[1];
        if (dropped || h->h_alive_status[1]) CU(cudaMemsetAsync(h->d_alive_status, 0, 8, s));
        const uint64_t slots = (uint64_t)h->alive_pairs * 2;
        const bool crowded = occupied * 10 > slots * 6;
        if (!dropped && !crowded) break;
        if (h->alive_pairs >= (uint32_t)ALIVE_MAX_KIB * 64u) {
            if (dropped) return fail(KTA_ERR_NOMEM, "alive-key table is at its maximum (32 GiB) and still too full");
            break;
        }
        // at least double; enough for every known entry plus every dropped stamp at load <= 0.5
        uint64_t want = slots * 2;
        while (want < (occupied + dropped) * 2) want *= 2;
        want = std::min<uint64_t>(want, (uint64_t)ALIVE_MAX_KIB * 128ull);
        int rc;
        if ((rc = alive_grow(h, (uint32_t)(want / 2)))) return rc;
        if (!dropped) break;   // grown ahead of need: every pending stamp had landed
        if (round > 40) return fail(KTA_ERR_INVALID, "alive-key table growth did not converge");
        for (const PendingScan &ps : h->pending) {
            ScanParams prm = ps.prm;
            prm.alive_only = 1;
            if ((rc = launch_scan_raw(h, prm, ps.key_readable, ps.key_bytes))) return rc;
            h->alive_reruns++;
        }
    }
    h->pending.clear();
    return KTA_OK;
}

static int launch_scan(kta_handle *h, ScanParams prm, int64_t key_readable, int64_t key_bytes, int chunk = -1,
                       const uint64_t *seq_ends = nullptr /* host copy of seq[0], seq[n-1] when the column came from the host */) {
    if (prm.n <= 0) return KTA_OK;
    int rc;
    if (h->cfg.count_alive_keys == 1) {
        // the stamps of this batch must fit the table's 31-bit window [origin, origin + ALIVE_FIELD_MAX)
        if ((uint64_t)prm.n > (uint64_t)ALIVE_FIELD_MAX - 1)
            return fail(KTA_ERR_INVALID, "batch of %lld records with count_alive_keys: split it (< 2^31 per scan)", (long long)prm.n);
        if (prm.seq_base < h->alive_origin)
            return fail(KTA_ERR_INVALID, "seq_base %llu lies before the alive-key table's window origin %llu (batches must not "
                        "go back past a rebase)", (unsigned long long)prm.seq_base, (unsigned long long)h->alive_origin);
        // explicit seq columns are checked record by record in the kernel; the implicit range is checked here
        if (!prm.seq && prm.seq_base - h->alive_origin + (uint64_t)prm.n > (uint64_t)ALIVE_FIELD_MAX) {
            // rebase: everything already in the table is older than this batch; forget by how much
            if ((rc = alive_check(h))) return rc;
            alive_rebase_kernel<<<h->sm_count * 8, THREADS, 0, h->stream>>>(h->d_alive_table, (size_t)h->alive_pairs * 2);
            h->launches++;
            CU(cudaGetLastError());
            h->alive_origin = prm.seq_base;
            h->alive_rebased = true;
        }
        prm.alive_fbase = prm.seq_base - h->alive_origin + 1ull;
        prm.alive_only = 0;
    }
    if ((rc = launch_scan_raw(h, prm, key_readable, key_bytes, seq_ends))) return rc;
    if (h->cfg.count_alive_keys == 1) h->pending.push_back(PendingScan{prm, key_readable, key_bytes, chunk});
    h->records += (uint64_t)prm.n;
    h->finalized = false;
    return KTA_OK;
}

// a ring chunk is about to be overwritten: its scan must be confirmed first (the chunk's event has been waited for,
// so its status snapshot is valid)
static int alive_release_chunk(kta_handle *h, int ci) {
    if (!h->d_alive_table || h->pending.empty()) return KTA_OK;
    bool mine = false;
    for (const PendingScan &ps : h->pending) mine = mine || ps.chunk == ci;
    if (!mine) return KTA_OK;
    const Chunk &c = h->chunks[ci];
    if (c.h_status[0] | c.h_status[1]) return alive_check(h);   // something was dropped up to this scan: settle everything
    // nothing dropped up to and including this chunk's scan: it — and every older pending scan — is confirmed
    size_t keep = 0;
    bool seen = false;
    for (size_t i = h->pending.size(); i-- > 0;) {   // find the newest entry of this chunk; drop it and everything older
        if (h->pending[i].chunk == ci) { keep = i + 1; seen = true; break; }
    }
    if (seen) h->pending.erase(h->pending.begin(), h->pending.begin() + (long)keep);
    return KTA_OK;
}

static int collect_timing(kta_handle *h) {
    for (size_t i = 0; i < h->ev_used; i++) {
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, h->ev_pool[i].first, h->ev_pool[i].second));
        h->scan_ms += ms;
        h->scan_launches_timed++;
    }
    h->ev_used = 0;
    return KTA_OK;
}

static int derive_tile_base(kta_handle *h, const int32_t *d_klen, int64_t n, uint64_t *d_tile_base) {
    const int64_t ntiles = (n + TILE - 1) / TILE;
    const int grid = (int)std::min<int64_t>((ntiles + 7) / 8, (int64_t)h->sm_count * 8);
    tile_key_bytes_kernel<<<grid, 256, 0, h->stream>>>(d_klen, n, ntiles, d_tile_base);
    CU(cudaGetLastError());
    tile_base_scan_kernel<<<1, 1024, 0, h->stream>>>(d_tile_base, ntiles);
    CU(cudaGetLastError());
    h->launches += 2;
    return KTA_OK;
}

static int ring_flush(kta_handle *h);

// seq of a batch's record 0.  KTA_SEQ_AUTO continues the handle's running count (what kta_push and the log-segment
// entry points do).  With -c and no explicit seq column, last-writer-wins is decided by seq_base + i alone, so a batch
// that re-uses sequence numbers the handle has already handed out would silently let OLDER records win: refused.
static int resolve_seq_base(kta_handle *h, const kta_batch *b, uint64_t *out) {
    if (b->seq_base == KTA_SEQ_AUTO) {
        *out = h->next_seq;
        return KTA_OK;
    }
    if (h->cfg.count_alive_keys == 1 && !b->seq && b->seq_base < h->next_seq)
        return fail(KTA_ERR_INVALID, "seq_base %llu < %llu, the next sequence number of this handle: batches without a seq "
                    "column must be pushed in stream order (use KTA_SEQ_AUTO to continue the running count)",
                    (unsigned long long)b->seq_base, (unsigned long long)h->next_seq);
    *out = b->seq_base;
    return KTA_OK;
}

extern "C" int kta_scan_batch_device(kta_handle *h, const kta_batch *b) {
    if (!h || !b) return fail(KTA_ERR_INVALID, "null argument");
    if (b->n < 0) return fail(KTA_ERR_INVALID, "negative n");
    if (b->n == 0) return KTA_OK;
    if (!b->partition || !b->ts_ms || !b->key_len || !b->value_len)
        return fail(KTA_ERR_INVALID, "partition/ts_ms/key_len/value_len columns are required");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;   // records pushed earlier come first in seq order
    uint64_t seq_base = 0;
    if ((rc = resolve_seq_base(h, b, &seq_base))) return rc;
    ScanParams prm{};
    prm.n = b->n;
    prm.seq_base = seq_base;
    prm.partition = b->partition;
    prm.ts_ms = b->ts_ms;
    prm.key_len = b->key_len;
    prm.value_len = b->value_len;
    prm.key_bytes = b->key_bytes;
    prm.seq = b->seq;
    prm.key_tile_base = b->key_tile_base;
    if ((h->need_hash || h->d_hash_out) && !prm.key_tile_base) {
        const int64_t ntiles = (b->n + TILE - 1) / TILE;
        if (ntiles + 1 > h->tb_scratch_tiles) {
            // stream-ordered: earlier scans that still read the old scratch finish first
            CU(cudaStreamSynchronize(h->stream));
            cudaFree(h->d_tb_scratch);
            h->d_tb_scratch = nullptr;
            h->tb_scratch_tiles = 0;
            CU(cudaMalloc(&h->d_tb_scratch, (size_t)(ntiles + 1) * 8));
            h->tb_scratch_tiles = ntiles + 1;
        }
        if ((rc = derive_tile_base(h, b->key_len, b->n, h->d_tb_scratch))) return rc;
        prm.key_tile_base = h->d_tb_scratch;
    }
    if ((rc = launch_scan(h, prm, b->key_bytes_len, b->key_bytes_len))) return rc;
    h->next_seq = std::max<uint64_t>(h->next_seq, seq_base + (uint64_t)b->n);
    return KTA_OK;
}

// ------------------------------------------------------------------------------------------------
// Kafka RecordBatch v2 segments → SoA → scan (SURVEY.md §8 f2; kernels in kta_logdecode.cuh)
// ------------------------------------------------------------------------------------------------

template <typename T>
static int grow(T *&ptr, int64_t &cap, int64_t need, cudaStream_t s) {
    if (need <= cap) return KTA_OK;
    CU(cudaStreamSynchronize(s));   // queued work may still read the old buffer
    cudaFree(ptr);
    ptr = nullptr;
    cap = 0;
    const int64_t n = need + need / 4 + 64;
    CU(cudaMalloc(&ptr, (size_t)n * sizeof(T)));
    cap = n;
    return KTA_OK;
}

static int scan_log_batches(kta_handle *h, int32_t partition, const int32_t *dev_batch_partition, const uint8_t *dev_bytes,
                            int64_t len, int64_t readable /* bytes of dev_bytes that may be READ (>= len when the buffer has slack) */,
                            const uint64_t *dev_batch_off, int64_t nbatches, int64_t *records_out) {
    if (!h || len < 0 || nbatches < 0 || (nbatches && (!dev_bytes || !dev_batch_off))) return fail(KTA_ERR_INVALID, "bad argument");
    if (records_out) *records_out = 0;
    if (nbatches == 0) return KTA_OK;
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;   // keep seq order with records pushed earlier
    if (!h->pending.empty() && (rc = alive_check(h))) return rc;   // the decode scratch of an earlier call is about to be reused
    cudaStream_t s = h->stream;
    if (nbatches + 1 > h->log_batch_cap) {
        CU(cudaStreamSynchronize(s));
        cudaFree(h->d_log_info); cudaFree(h->d_log_cnt);
        h->d_log_info = nullptr; h->d_log_cnt = nullptr; h->log_batch_cap = 0;
        const int64_t n = nbatches + nbatches / 4 + 64;
        CU(cudaMalloc(&h->d_log_info, (size_t)n * sizeof(LogBatchInfo)));
        CU(cudaMalloc(&h->d_log_cnt, (size_t)n * 8));
        h->log_batch_cap = n;
    }
    if (!h->d_log_err) CU(cudaMalloc(&h->d_log_err, 8));   // [0] error flags, [1] longest batch
    CU(cudaMemsetAsync(h->d_log_err, 0, 8, s));
    const int grid = (int)std::min<int64_t>((nbatches + 127) / 128, (int64_t)h->sm_count * 16);
    log_header_kernel<<<grid, 128, 0, s>>>(dev_bytes, len, dev_batch_off, nbatches, partition, dev_batch_partition, h->d_log_info,
                                            h->d_log_cnt, h->d_log_err);
    tile_base_scan_kernel<<<1, 1024, 0, s>>>(h->d_log_cnt, nbatches);   // inclusive scan of [1..nbatches] in place
    CU(cudaGetLastError());
    h->launches += 2;
    uint64_t nrec = 0;
    uint32_t err[2] = {0, 0};
    CU(cudaMemcpyAsync(&nrec, h->d_log_cnt + nbatches, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(err, h->d_log_err, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if (err[0] & LOGB_COMPRESSED)
        return fail(KTA_ERR_INVALID, "unknown compression codec in a record batch of partition %d", partition);
    if (err[0] & LOGB_BAD) return fail(KTA_ERR_INVALID, "malformed record batch header in partition %d", partition);
    if (nrec == 0) return KTA_OK;
    if (err[0] & LOGB_CODECS) {
        // compressed batches: size pass, scratch allocation, decompression; afterwards they are ordinary batches that
        // happen to lie in the scratch buffer
        const uint32_t codecs = err[0] & LOGB_CODECS;   // the codecs present (err[0] is reused by the size pass)
        if ((rc = grow(h->d_unc_slot, h->unc_slot_cap, nbatches + 2, s))) return rc;
        CU(cudaMemsetAsync(h->d_log_err, 0, 4, s));
        log_unc_size_kernel<<<grid, 128, 0, s>>>(dev_bytes, h->d_log_info, nbatches, h->d_unc_slot, h->d_log_err);
        if (codecs & LOGB_ZSTD) {   // warp per batch
            log_zstd_size_kernel<<<(int)std::min<int64_t>((nbatches + 3) / 4, (int64_t)h->sm_count * 16), 128, 0, s>>>(
                dev_bytes, h->d_log_info, nbatches, h->d_unc_slot, h->d_log_err);
            h->launches++;
        }
        tile_base_scan_kernel<<<1, 1024, 0, s>>>(h->d_unc_slot, nbatches);
        CU(cudaGetLastError());
        h->launches += 2;
        uint64_t unc_total = 0;
        CU(cudaMemcpyAsync(&unc_total, h->d_unc_slot + nbatches, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(err, h->d_log_err, 4, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        if (err[0]) return fail(KTA_ERR_INVALID, "malformed compressed record batch in partition %d", partition);
        if ((rc = grow(h->d_unc, h->unc_cap, (int64_t)unc_total + 64, s))) return rc;
        const int dgrid = (int)std::min<int64_t>((nbatches + 3) / 4, (int64_t)h->sm_count * 16);
        if (codecs & ~LOGB_ZSTD) {
            log_decompress_kernel<false><<<dgrid, 128, 0, s>>>(dev_bytes, h->d_log_info, nbatches, h->d_unc_slot, h->d_unc, h->d_log_err);
            h->launches++;
        }
        if (codecs & LOGB_ZSTD) {
            log_decompress_kernel<true><<<dgrid, 128, 0, s>>>(dev_bytes, h->d_log_info, nbatches, h->d_unc_slot, h->d_unc, h->d_log_err);
            h->launches++;
        }
        CU(cudaGetLastError());
    }
    if ((int64_t)nrec >= ((int64_t)1 << 31) - 2) return fail(KTA_ERR_INVALID, "%llu records in one call: split the segments", (unsigned long long)nrec);
    const bool hash = h->need_hash || h->d_hash_out;
    if ((int64_t)nrec > h->dec_rec_cap) {
        CU(cudaStreamSynchronize(s));
        cudaFree(h->d_dec_part); cudaFree(h->d_dec_klen); cudaFree(h->d_dec_vlen); cudaFree(h->d_dec_ts); cudaFree(h->d_dec_ksrc);
        h->d_dec_part = h->d_dec_klen = h->d_dec_vlen = nullptr; h->d_dec_ts = nullptr; h->d_dec_ksrc = nullptr; h->dec_rec_cap = 0;
        const int64_t n = (int64_t)nrec + (int64_t)nrec / 4 + 1024;
        CU(cudaMalloc(&h->d_dec_part, (size_t)n * 4));
        CU(cudaMalloc(&h->d_dec_klen, (size_t)n * 4));
        CU(cudaMalloc(&h->d_dec_vlen, (size_t)n * 4));
        CU(cudaMalloc(&h->d_dec_ts, (size_t)n * 8));
        CU(cudaMalloc(&h->d_dec_ksrc, (size_t)n * 8));
        h->dec_rec_cap = n;
    }
    // one warp per batch; the batch is staged in shared memory when the longest one fits a stage of <= 48 KiB
    const uint32_t maxlen = err[1];
    const uint32_t stage = (uint32_t)(((size_t)maxlen + 16 + 1023) / 1024 * 1024);
    const bool staged = stage <= 48u * 1024u;
    const size_t dsm = (size_t)(LOG_DECODE_THREADS / 32) * (LOG_WARP_HEADER + (staged ? stage : 0u));
    static bool attr_set = false;
    if (!attr_set) {
        CU(cudaFuncSetAttribute(log_decode_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)h->smem_optin));
        attr_set = true;
    }
    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(16, h->smem_optin / std::max<size_t>(dsm, 1)));
    const int dgrid = (int)std::min<int64_t>((nbatches + 3) / 4, (int64_t)h->sm_count * per_sm);
    uint64_t *ksrc = hash ? h->d_dec_ksrc : nullptr;
    if (staged)
        log_decode_kernel<true><<<dgrid, LOG_DECODE_THREADS, dsm, s>>>(dev_bytes, (uint64_t)readable, h->d_log_info, nbatches, h->d_log_cnt, h->d_dec_part,
                                                                       nullptr, h->d_dec_ts, h->d_dec_klen, h->d_dec_vlen, ksrc, stage, h->d_log_err);
    else
        log_decode_kernel<false><<<dgrid, LOG_DECODE_THREADS, dsm, s>>>(dev_bytes, (uint64_t)readable, h->d_log_info, nbatches, h->d_log_cnt, h->d_dec_part,
                                                                        nullptr, h->d_dec_ts, h->d_dec_klen, h->d_dec_vlen, ksrc, 0u, h->d_log_err);
    CU(cudaGetLastError());
    h->launches++;
    kta_batch b{};
    b.n = (int64_t)nrec;
    b.seq_base = KTA_SEQ_AUTO;
    b.partition = h->d_dec_part;
    b.ts_ms = h->d_dec_ts;
    b.key_len = h->d_dec_klen;
    b.value_len = h->d_dec_vlen;
    if (hash) {
        // pack the keys in record order: tile bases from the key_len column, then one gather pass (no second walk of the log)
        const int64_t ntiles = ((int64_t)nrec + TILE - 1) / TILE;
        if (ntiles + 1 > h->tb_scratch_tiles) {
            CU(cudaStreamSynchronize(s));
            cudaFree(h->d_tb_scratch);
            h->d_tb_scratch = nullptr;
            h->tb_scratch_tiles = 0;
            CU(cudaMalloc(&h->d_tb_scratch, (size_t)(ntiles + 1) * 8));
            h->tb_scratch_tiles = ntiles + 1;
        }
        if ((rc = derive_tile_base(h, h->d_dec_klen, (int64_t)nrec, h->d_tb_scratch))) return rc;
        uint64_t nkey = 0;
        CU(cudaMemcpyAsync(&nkey, h->d_tb_scratch + ntiles, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaMemcpyAsync(err, h->d_log_err, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        if (err[0]) return fail(KTA_ERR_INVALID, "malformed record inside a batch of partition %d", partition);
        if ((rc = grow(h->d_dec_keys, h->dec_key_cap, (int64_t)nkey + 64, s))) return rc;
        log_gather_keys_kernel<<<(int)std::min<int64_t>((ntiles + 7) / 8, (int64_t)h->sm_count * 8), 256, 0, s>>>(
            dev_bytes, h->d_dec_ksrc, h->d_dec_klen, (int64_t)nrec, h->d_tb_scratch, h->d_dec_keys);
        CU(cudaGetLastError());
        h->launches++;
        b.key_bytes = h->d_dec_keys;
        b.key_bytes_len = (int64_t)nkey;
        b.key_tile_base = h->d_tb_scratch;
    } else {
        CU(cudaMemcpyAsync(err, h->d_log_err, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaStreamSynchronize(s));
        if (err[0]) return fail(KTA_ERR_INVALID, "malformed record inside a batch of partition %d", partition);
    }
    if ((rc = kta_scan_batch_device(h, &b))) return rc;
    if (records_out) *records_out = (int64_t)nrec;
    return KTA_OK;
}

extern "C" int kta_scan_log_segment_device(kta_handle *h, int32_t partition, const uint8_t *dev_bytes, int64_t len,
                                           const uint64_t *dev_batch_off, int64_t nbatches, int64_t *records_out) {
    return scan_log_batches(h, partition, nullptr, dev_bytes, len, len, dev_batch_off, nbatches, records_out);
}

extern "C" int kta_scan_log_batches_device(kta_handle *h, const uint8_t *dev_bytes, int64_t len, const uint64_t *dev_batch_off,
                                           const int32_t *dev_batch_partition, int64_t nbatches, int64_t *records_out) {
    if (nbatches && !dev_batch_partition) return fail(KTA_ERR_INVALID, "dev_batch_partition is NULL");
    return scan_log_batches(h, 0, dev_batch_partition, dev_bytes, len, len, dev_batch_off, nbatches, records_out);
}

extern "C" int kta_push_log_segments_host(kta_handle *h, int32_t nsegs, const int32_t *partitions, const uint8_t *const *bytes,
                                          const int64_t *lens, int64_t *records_out) {
    if (!h || nsegs < 0 || (nsegs && (!partitions || !bytes || !lens))) return fail(KTA_ERR_INVALID, "bad argument");
    if (records_out) *records_out = 0;
    // hop from batch header to batch header on the host (12 + batchLength bytes each); a truncated tail is ignored,
    // as a consumer would ignore a partially fetched batch.  All segments go to ONE staging buffer and are decoded
    // and scanned together (one decode, one scan, two host round trips in total).
    std::vector<uint64_t> offs;
    std::vector<int32_t> parts;
    std::vector<int64_t> used((size_t)nsegs, 0), base((size_t)nsegs, 0);
    int64_t total = 0;
    for (int32_t sgi = 0; sgi < nsegs; sgi++) {
        if (lens[sgi] < 0 || (lens[sgi] && !bytes[sgi])) return fail(KTA_ERR_INVALID, "bad segment %d", sgi);
        base[(size_t)sgi] = total;
        int64_t pos = 0;
        while (pos + LOG_HEADER_BYTES <= lens[sgi]) {
            const uint8_t *p = bytes[sgi] + pos;
            const int64_t bl = (int64_t)(int32_t)(((uint32_t)p[8] << 24) | ((uint32_t)p[9] << 16) | ((uint32_t)p[10] << 8) | p[11]);
            if (bl < LOG_HEADER_BYTES - 12 || pos + 12 + bl > lens[sgi]) break;
            offs.push_back((uint64_t)(total + pos));
            parts.push_back(partitions[sgi]);
            pos += 12 + bl;
        }
        used[(size_t)sgi] = pos;
        total += (pos + 15) & ~(int64_t)15;
    }
    if (offs.empty()) return KTA_OK;
    int rc;
    if ((rc = set_device(h))) return rc;
    cudaStream_t s = h->stream;
    if ((rc = grow(h->d_log_bytes, h->log_bytes_cap, total + 64, s))) return rc;
    CU(cudaStreamSynchronize(s));
    cudaFree(h->d_log_off);
    h->d_log_off = nullptr;
    CU(cudaMalloc(&h->d_log_off, offs.size() * 12));
    int32_t *d_parts = reinterpret_cast<int32_t *>(h->d_log_off + offs.size());
    for (int32_t sgi = 0; sgi < nsegs; sgi++)
        if (used[(size_t)sgi])
            CU(cudaMemcpyAsync(h->d_log_bytes + base[(size_t)sgi], bytes[sgi], (size_t)used[(size_t)sgi], cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(h->d_log_off, offs.data(), offs.size() * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(d_parts, parts.data(), parts.size() * 4, cudaMemcpyHostToDevice, s));
    // the staging buffer has 64 bytes of slack behind `total`: 16-byte-granular bulk copies may run into it
    if ((rc = scan_log_batches(h, 0, d_parts, h->d_log_bytes, total, total + 48, h->d_log_off, (int64_t)offs.size(), records_out))) return rc;
    CU(cudaStreamSynchronize(s));   // the caller may reuse its buffers, and the scratch may be reused by the next call
    return collect_timing(h);
}

extern "C" int kta_push_log_segment_host(kta_handle *h, int32_t partition, const uint8_t *bytes, int64_t len,
                                         int64_t *records_out) {
    return kta_push_log_segments_host(h, 1, &partition, &bytes, &len, records_out);
}

// ------------------------------------------------------------------------------------------------
// landing ring: host records → pinned chunk → cudaMemcpyAsync → HBM chunk → scan
// ------------------------------------------------------------------------------------------------
static int ring_dev_init(kta_handle *h) {
    if (h->ring_dev_ready) return KTA_OK;
    const int64_t R = h->ring_records, KB = h->ring_key_bytes;
    for (auto &c : h->chunks) {
        CU(cudaMalloc(&c.d_partition, R * 4));
        CU(cudaMalloc(&c.d_klen, R * 4));
        CU(cudaMalloc(&c.d_vlen, R * 4));
        CU(cudaMalloc(&c.d_ts, R * 8));
        CU(cudaMalloc(&c.d_seq, R * 8));
        CU(cudaMalloc(&c.d_keys, KB + 64));
        CU(cudaMalloc(&c.d_tile_base, (R / TILE + 2) * 8));
        CU(cudaEventCreateWithFlags(&c.free_ev, cudaEventDisableTiming));
        CU(cudaHostAlloc(&c.h_status, 8, cudaHostAllocDefault));
        c.h_status[0] = c.h_status[1] = 0;
    }
    h->ring_dev_ready = true;
    return KTA_OK;
}

static int ring_host_init(kta_handle *h) {
    if (h->ring_host_ready) return KTA_OK;
    int rc;
    if ((rc = ring_dev_init(h))) return rc;
    const int64_t R = h->ring_records, KB = h->ring_key_bytes;
    for (auto &c : h->chunks) {
        CU(cudaHostAlloc(&c.h_partition, R * 4, cudaHostAllocDefault));
        CU(cudaHostAlloc(&c.h_klen, R * 4, cudaHostAllocDefault));
        CU(cudaHostAlloc(&c.h_vlen, R * 4, cudaHostAllocDefault));
        CU(cudaHostAlloc(&c.h_ts, R * 8, cudaHostAllocDefault));
        CU(cudaHostAlloc(&c.h_keys, KB + 64, cudaHostAllocDefault));
        CU(cudaHostAlloc(&c.h_tile_base, (R / TILE + 2) * 8, cudaHostAllocDefault));
    }
    h->ring_host_ready = true;
    return KTA_OK;
}

static void push_cursor_bind(kta_handle *h) {
    Chunk &c = h->chunks[h->cur];
    auto &pc = h->pc;
    pc.part = c.h_partition; pc.klen = c.h_klen; pc.vlen = c.h_vlen; pc.ts = c.h_ts; pc.keys = c.h_keys; pc.tile_base = c.h_tile_base;
    pc.n = 0; pc.kb = 0;
    pc.cap = h->ring_host_ready ? h->ring_records : 0;
    pc.kcap = h->ring_key_bytes;
    pc.hash = h->need_hash || h->d_hash_out;
}

// stage one pinned chunk and scan it
static int ring_flush(kta_handle *h) {
    if (h->pc.n == 0) return KTA_OK;
    Chunk &c = h->chunks[h->cur];
    const int64_t n = h->pc.n, kb = h->pc.kb;
    const int64_t ntiles = (n + TILE - 1) / TILE;
    c.h_tile_base[ntiles] = (uint64_t)kb;
    cudaStream_t s = h->stream;
    CU(cudaMemcpyAsync(c.d_partition, c.h_partition, n * 4, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(c.d_ts, c.h_ts, n * 8, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(c.d_klen, c.h_klen, n * 4, cudaMemcpyHostToDevice, s));
    CU(cudaMemcpyAsync(c.d_vlen, c.h_vlen, n * 4, cudaMemcpyHostToDevice, s));
    if (h->need_hash || h->d_hash_out) {
        if (kb) CU(cudaMemcpyAsync(c.d_keys, c.h_keys, kb, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(c.d_tile_base, c.h_tile_base, (ntiles + 1) * 8, cudaMemcpyHostToDevice, s));
    }
    ScanParams prm{};
    prm.n = n;
    prm.seq_base = h->next_seq;
    prm.partition = c.d_partition;
    prm.ts_ms = c.d_ts;
    prm.key_len = c.d_klen;
    prm.value_len = c.d_vlen;
    prm.key_bytes = c.d_keys;
    prm.key_tile_base = c.d_tile_base;
    int rc;
    if ((rc = launch_scan(h, prm, (kb + 15) & ~(int64_t)15, kb, h->cur))) return rc;
    h->next_seq += (uint64_t)n;
    if (h->d_alive_table) CU(cudaMemcpyAsync(c.h_status, h->d_alive_status, 8, cudaMemcpyDeviceToHost, s));
    CU(cudaEventRecord(c.free_ev, s));
    h->cur = (h->cur + 1) % NCHUNK;
    push_cursor_bind(h);
    // the next chunk may still be in flight from NCHUNK flushes ago
    CU(cudaEventSynchronize(h->chunks[h->cur].free_ev));
    return alive_release_chunk(h, h->cur);
}

// kta_push off the fast path: first call (ring not yet allocated), chunk full, or an oversized key
static int __attribute__((noinline)) push_slow(kta_handle *h, int64_t kl) {
    int rc;
    if ((rc = set_device(h))) return rc;
    if (!h->ring_host_ready) {
        if ((rc = ring_host_init(h))) return rc;
        push_cursor_bind(h);
    }
    if (kl > h->ring_key_bytes) return fail(KTA_ERR_INVALID, "key of %lld bytes exceeds ring_key_bytes", (long long)kl);
    if (h->pc.n == h->pc.cap || h->pc.kb + kl > h->pc.kcap) return ring_flush(h);
    return KTA_OK;
}

extern "C" int kta_push(kta_handle *h, int32_t partition, int64_t offset, int64_t ts_ms, const uint8_t *key,
                        int32_t key_len, int32_t value_len) {
    (void)offset;  // never read by a metric (SURVEY.md D7); termination logic stays with the caller
    if (__builtin_expect(!h, 0)) return fail(KTA_ERR_INVALID, "null handle");
    auto &pc = h->pc;
    const int64_t kl = (pc.hash && key_len > 0) ? key_len : 0;  // key bytes only travel when they are hashed
    if (__builtin_expect(pc.n == pc.cap || pc.kb + kl > pc.kcap, 0)) {
        const int rc = push_slow(h, kl);
        if (rc) return rc;
    }
    const int64_t i = pc.n;
    if ((i & (TILE - 1)) == 0) pc.tile_base[i / TILE] = (uint64_t)pc.kb;
    pc.part[i] = partition;
    pc.ts[i] = ts_ms;
    pc.klen[i] = key_len < 0 ? -1 : key_len;
    pc.vlen[i] = value_len < 0 ? -1 : value_len;
    if (kl) {
        if (__builtin_expect(!key, 0)) return fail(KTA_ERR_INVALID, "key is NULL with key_len %d", key_len);
        uint8_t *dst = pc.keys + pc.kb;
        if (kl == 16) {            // ids, hashes, UUIDs: two register moves instead of a call
            uint64_t a, b;
            memcpy(&a, key, 8); memcpy(&b, key + 8, 8);
            memcpy(dst, &a, 8); memcpy(dst + 8, &b, 8);
        } else if (kl <= 8) {      // short keys: byte-exact, no call (the landing area has slack only at its end)
            for (int64_t j = 0; j < kl; j++) dst[j] = key[j];
        } else {
            memcpy(dst, key, (size_t)kl);
        }
        pc.kb += kl;
    }
    pc.n = i + 1;
    h->finalized = false;
    return KTA_OK;
}

extern "C" int kta_push_batch_host(kta_handle *h, const kta_batch *b) {
    if (!h || !b) return fail(KTA_ERR_INVALID, "null argument");
    if (b->n < 0) return fail(KTA_ERR_INVALID, "negative n");
    if (b->n == 0) return KTA_OK;
    if (!b->partition || !b->ts_ms || !b->key_len || !b->value_len)
        return fail(KTA_ERR_INVALID, "partition/ts_ms/key_len/value_len columns are required");
    const bool hash = h->need_hash || h->d_hash_out;
    if (hash && !b->key_bytes && b->key_bytes_len > 0) return fail(KTA_ERR_INVALID, "key_bytes is NULL");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;  // keep seq order with earlier kta_push records
    if ((rc = ring_dev_init(h))) return rc;
    uint64_t seq_base = 0;
    if ((rc = resolve_seq_base(h, b, &seq_base))) return rc;
    cudaStream_t s = h->stream;
    const bool use_seq = b->seq && h->cfg.count_alive_keys == 1;
    std::vector<uint64_t> tb_host;  // only when the caller gave no tile bases
    uint64_t koff = 0;              // absolute key byte offset of the next chunk's first key
    int64_t r0 = 0;
    while (r0 < b->n) {
        int64_t cn = std::min<int64_t>(h->ring_records, b->n - r0);
        const int ci = h->cur;
        Chunk &c = h->chunks[ci];
        uint64_t k0 = 0, k1 = 0;
        const uint64_t *tb_src = nullptr;
        if (hash) {
            // the chunk ends at a tile boundary chosen so that its keys fit the staging buffer; only a SINGLE tile
            // whose keys exceed ring_key_bytes cannot be staged
            const int64_t tiles_max = (cn + TILE - 1) / TILE;
            int64_t tiles = 0;
            if (b->key_tile_base) {
                const uint64_t *tb = b->key_tile_base + r0 / TILE;
                k0 = tb[0];
                // largest t with tb[t] - k0 <= ring_key_bytes (tile bases are non-decreasing)
                tiles = std::upper_bound(tb, tb + tiles_max + 1, k0 + (uint64_t)h->ring_key_bytes) - tb - 1;
                tiles = std::min<int64_t>(tiles, tiles_max);
                if (tiles >= 1) k1 = tb[tiles];
                tb_src = tb;
            } else {
                tb_host.resize((size_t)tiles_max + 1);
                uint64_t acc = koff;
                tb_host[0] = acc;
                for (; tiles < tiles_max; tiles++) {
                    const int64_t lo = r0 + tiles * TILE, hi = std::min<int64_t>(lo + TILE, r0 + cn);
                    uint64_t tile_bytes = 0;
                    for (int64_t i = lo; i < hi; i++) tile_bytes += b->key_len[i] > 0 ? (uint64_t)b->key_len[i] : 0;
                    if (acc + tile_bytes - koff > (uint64_t)h->ring_key_bytes) break;
                    acc += tile_bytes;
                    tb_host[(size_t)tiles + 1] = acc;
                }
                k0 = koff;
                k1 = acc;
                tb_src = tb_host.data();
            }
            if (tiles < 1)
                return fail(KTA_ERR_INVALID, "the keys of one %d-record tile (records %lld..) exceed ring_key_bytes %lld; "
                            "%lld earlier record(s) of this batch were scanned", TILE, (long long)r0, (long long)h->ring_key_bytes,
                            (long long)r0);
            cn = std::min<int64_t>(cn, tiles * TILE);
        }
        // chunk ci's buffers are about to be overwritten: wait for the scan that read them and confirm its stamps
        CU(cudaEventSynchronize(c.free_ev));
        if ((rc = alive_release_chunk(h, ci))) return rc;
        const int64_t ntiles = (cn + TILE - 1) / TILE;
        CU(cudaMemcpyAsync(c.d_partition, b->partition + r0, cn * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(c.d_ts, b->ts_ms + r0, cn * 8, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(c.d_klen, b->key_len + r0, cn * 4, cudaMemcpyHostToDevice, s));
        CU(cudaMemcpyAsync(c.d_vlen, b->value_len + r0, cn * 4, cudaMemcpyHostToDevice, s));
        if (use_seq) CU(cudaMemcpyAsync(c.d_seq, b->seq + r0, cn * 8, cudaMemcpyHostToDevice, s));
        ScanParams prm{};
        if (hash) {
            // keep absolute offsets: place the keys so that (virtual base + k0) is where they land and the
            // virtual base stays 16-byte aligned
            const uint64_t shift = k0 & 15ull;
            if (k1 > k0) CU(cudaMemcpyAsync(c.d_keys + shift, b->key_bytes + k0, k1 - k0, cudaMemcpyHostToDevice, s));
            CU(cudaMemcpyAsync(c.d_tile_base, tb_src, (ntiles + 1) * 8, cudaMemcpyHostToDevice, s));
            prm.key_bytes = c.d_keys + shift - k0;
            prm.key_tile_base = c.d_tile_base;
        }
        prm.n = cn;
        prm.seq_base = seq_base + (uint64_t)r0;
        prm.partition = c.d_partition;
        prm.ts_ms = c.d_ts;
        prm.key_len = c.d_klen;
        prm.value_len = c.d_vlen;
        prm.seq = use_seq ? c.d_seq : nullptr;
        const uint64_t seq_ends[2] = {use_seq ? b->seq[r0] : 0, use_seq ? b->seq[r0 + cn - 1] : 0};
        if ((rc = launch_scan(h, prm, (int64_t)((k1 + 15) & ~15ull), (int64_t)(k1 - k0), ci, use_seq ? seq_ends : nullptr))) return rc;
        if (h->d_alive_table) CU(cudaMemcpyAsync(c.h_status, h->d_alive_status, 8, cudaMemcpyDeviceToHost, s));
        CU(cudaEventRecord(c.free_ev, s));
        h->cur = (h->cur + 1) % NCHUNK;
        koff = k1;
        r0 += cn;
    }
    // the caller may reuse its buffers when we return: all host→device copies must have been consumed
    CU(cudaStreamSynchronize(s));
    int rc2;
    if ((rc2 = collect_timing(h))) return rc2;
    h->next_seq = std::max<uint64_t>(h->next_seq, seq_base + (uint64_t)b->n);
    return KTA_OK;
}

extern "C" int kta_sync(kta_handle *h) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;
    CU(cudaStreamSynchronize(h->stream));
    if ((rc = alive_check(h))) return rc;
    return collect_timing(h);
}

extern "C" int kta_reset(kta_handle *h) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    int rc;
    if ((rc = set_device(h))) return rc;
    h->pc.n = 0;
    h->pc.kb = 0;
    h->next_seq = 0;
    h->finalized = false;
    h->launches = 0;
    h->records = 0;
    return state_reset_device(h);
}

extern "C" int kta_finalize(kta_handle *h) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;
    cudaStream_t s = h->stream;
    if ((rc = alive_check(h))) return rc;   // every stamp has landed (grows the table and re-runs batches if it was too small)
    if (h->d_alive_table && h->nhll) {
        // EXTENSION: with -c the sketch describes the resolved alive set, so it is rebuilt from the table
        CU(cudaMemsetAsync(h->d_hll, 0, h->nhll * 4, s));
        alive_hll_kernel<<<h->sm_count * 8, THREADS, 0, s>>>(h->d_alive_table, (size_t)h->alive_pairs * 2, h->d_hll,
                                                             h->cfg.hll_precision);
        CU(cudaGetLastError());
        h->launches++;
    }
    h->h_sums.resize(h->nsums);
    h->h_hll.resize(h->nhll);
    CU(cudaMemcpyAsync(h->h_sums.data(), h->d_sums, h->nsums * 8, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(h->h_minmax, h->d_minmax, 32, cudaMemcpyDeviceToHost, s));
    if (h->nhll) CU(cudaMemcpyAsync(h->h_hll.data(), h->d_hll, h->nhll * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    if ((rc = collect_timing(h))) return rc;
    h->h_alive = h->alive_now;   // counted over the table by alive_check above (sum_all_alive, src/metric.rs:282-284)
    h->finalized = true;
    if (h->alive_window_errors)
        return fail(KTA_ERR_INVALID, "%llu record(s) carried a sequence number outside the alive-key table's window "
                    "[origin, origin + 2^31 - 2): with an explicit seq column the span between kta_reset calls is limited",
                    (unsigned long long)h->alive_window_errors);
    // Records with a partition outside [0, P) took part in nothing (no counter, no extremum, no alive key): the getters
    // are valid and describe the in-range records; the status tells the caller that some were left out.
    const uint64_t bad = h->h_sums[h->nsums - 1];
    if (bad)
        return fail(KTA_ERR_PARTITION, "%llu record(s) had a partition outside [0, %d) and were left out of every metric",
                    (unsigned long long)bad, h->cfg.num_partitions);
    return KTA_OK;
}

// ------------------------------------------------------------------------------------------------
// getters (host arithmetic on the finalized state)
// ------------------------------------------------------------------------------------------------
static int check_read(const kta_handle *h, int32_t p, bool per_partition) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    if (!h->finalized) return fail(KTA_ERR_NOT_FINALIZED, "call kta_finalize first");
    if (per_partition && (p < 0 || p >= h->cfg.num_partitions)) return -1;  // unseen partition: reads as 0
    return KTA_OK;
}

static uint64_t raw_counter(const kta_handle *h, int which, int32_t p) {
    const int P = h->cfg.num_partitions;
    const uint64_t *s = h->h_sums.data();
    uint64_t knn = 0, alive = 0;
    for (int b = 0; b < NB; b++) {
        knn += s[(size_t)p * NB + b];
        alive += s[(size_t)(P + p) * NB + b];
    }
    const uint64_t knull = s[(size_t)P * (2 * NB + 2) + p];
    const uint64_t total = knn + knull;
    switch (which) {
        case KTA_TOTAL: return total;
        case KTA_TOMBSTONES: return total - alive;
        case KTA_ALIVE: return alive;
        case KTA_KEY_NULL: return knull;
        case KTA_KEY_NON_NULL: return knn;
        case KTA_KEY_SIZE_SUM: return s[(size_t)P * (2 * NB) + p];
        case KTA_VALUE_SIZE_SUM: return s[(size_t)P * (2 * NB + 1) + p];
    }
    return 0;
}

extern "C" int kta_counter(const kta_handle *h, int which, int32_t partition, uint64_t *out) {
    if (!out || which < 0 || which > KTA_VALUE_SIZE_SUM) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, partition, true);
    if (rc > 0) return rc;
    *out = rc < 0 ? 0 : raw_counter(h, which, partition);  // src/metric.rs:198-203: None => 0
    return KTA_OK;
}

extern "C" int kta_avg(const kta_handle *h, int which, int32_t partition, uint64_t *out) {
    if (!out || which < 0 || which > KTA_MESSAGE_SIZE_AVG) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, partition, true);
    if (rc > 0) return rc;
    if (rc < 0) { *out = 0; return KTA_OK; }
    const uint64_t ks = raw_counter(h, KTA_KEY_SIZE_SUM, partition), vs = raw_counter(h, KTA_VALUE_SIZE_SUM, partition);
    const uint64_t alive = raw_counter(h, KTA_ALIVE, partition);
    // src/metric.rs:132-157: every average divides by alive(p), guarded only by `sum > 0`
    const uint64_t sum = which == KTA_KEY_SIZE_AVG ? ks : which == KTA_VALUE_SIZE_AVG ? vs : ks + vs;
    if (sum > 0) {
        if (alive == 0)
            return fail(KTA_ERR_DIV_BY_ZERO, "partition %d: sum %llu > 0 with alive == 0 (the reference panics here)",
                        partition, (unsigned long long)sum);
        *out = sum / alive;
    } else {
        *out = 0;
    }
    return KTA_OK;
}

extern "C" int kta_dirty_ratio(const kta_handle *h, int32_t partition, float *out) {
    if (!out) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, partition, true);
    if (rc > 0) return rc;
    *out = 0.0f;
    if (rc < 0) return KTA_OK;
    const uint64_t total = raw_counter(h, KTA_TOTAL, partition), tomb = raw_counter(h, KTA_TOMBSTONES, partition);
    if (total > 0 && tomb > 0) {  // src/metric.rs:159-167, f32 throughout, same operation order
        const volatile float t = (float)tomb;
        const volatile float d = (float)total / 100.0f;
        *out = t / d;
    }
    return KTA_OK;
}

extern "C" int kta_global(const kta_handle *h, int which, uint64_t *out) {
    if (!out) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, 0, false);
    if (rc) return rc;
    const int P = h->cfg.num_partitions;
    const unsigned long long *mm = reinterpret_cast<const unsigned long long *>(h->h_minmax);
    switch (which) {
        case KTA_SMALLEST_MESSAGE: *out = mm[2] == ~0ull ? 0 : mm[2]; return KTA_OK;  // metric.rs:177-183
        case KTA_LARGEST_MESSAGE: *out = mm[3]; return KTA_OK;
        case KTA_OVERALL_SIZE: {
            uint64_t s = 0;
            for (int p = 0; p < P; p++) s += raw_counter(h, KTA_KEY_SIZE_SUM, p) + raw_counter(h, KTA_VALUE_SIZE_SUM, p);
            *out = s;  // metric.rs:224,238
            return KTA_OK;
        }
        case KTA_OVERALL_COUNT: {
            uint64_t s = 0;
            for (int p = 0; p < P; p++) s += raw_counter(h, KTA_TOTAL, p);
            *out = s;  // metric.rs:215
            return KTA_OK;
        }
    }
    return fail(KTA_ERR_INVALID, "bad global id %d", which);
}

extern "C" int kta_timestamps(const kta_handle *h, int64_t *earliest_s, int32_t *earliest_ns, int64_t *latest_s) {
    const int rc = check_read(h, 0, false);
    if (rc) return rc;
    // src/metric.rs:39-40,65-72,209-211: seconds = ms / 1000 truncating; earliest starts at Utc::now(),
    // latest at the epoch.  Truncating division is monotone, so min/max commute with it.
    // The device tracks the extrema of the RAW ts_ms column; "not available" (-1) maps to 0 (metric.rs:209).
    // That map only moves -1 to 0, so: raw min == -1 ⇒ every other value is >= 0 ⇒ mapped min is 0, otherwise
    // the mapped min is the raw min; raw max == -1 ⇒ every other value is < -1 ⇒ mapped max is 0, otherwise
    // the mapped max is the raw max.
    int64_t es = h->cfg.now_s, ls = 0;
    int32_t ens = h->cfg.now_ns;
    if (h->h_minmax[0] != INT64_MAX) {
        const int64_t raw_mn = h->h_minmax[0] == -1 ? 0 : h->h_minmax[0];
        const int64_t raw_mx = h->h_minmax[1] == -1 ? 0 : h->h_minmax[1];
        const int64_t mn = raw_mn / 1000, mx = raw_mx / 1000;
        if (es > mn || (es == mn && ens > 0)) { es = mn; ens = 0; }
        if (ls < mx) ls = mx;
    }
    if (earliest_s) *earliest_s = es;
    if (earliest_ns) *earliest_ns = ens;
    if (latest_s) *latest_s = ls;
    return KTA_OK;
}

extern "C" int kta_alive_keys(const kta_handle *h, uint64_t *out) {
    if (!out) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, 0, false);
    if (rc) return rc;
    if (h->cfg.count_alive_keys != 1) return fail(KTA_ERR_NOT_ENABLED, "count_alive_keys was not enabled");
    *out = h->h_alive;
    return KTA_OK;
}

extern "C" int kta_bad_partition_records(const kta_handle *h, uint64_t *out) {
    if (!out) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, 0, false);
    if (rc) return rc;
    *out = h->h_sums[h->nsums - 1];
    return KTA_OK;
}

extern "C" int kta_hist(const kta_handle *h, int which, int32_t partition, uint64_t out[KTA_HIST_BUCKETS]) {
    if (!out || which < 0 || which > 1) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, partition, true);
    if (rc > 0) return rc;
    const int P = h->cfg.num_partitions;
    for (int b = 0; b < NB; b++)
        out[b] = rc < 0 ? 0 : h->h_sums[(size_t)((which ? P : 0) + partition) * NB + b];
    return KTA_OK;
}

// Ertl 2017, "New cardinality estimation algorithms for HyperLogLog sketches": improved raw estimator
static double hll_sigma(double x) {
    if (x == 1.0) return INFINITY;
    double y = 1.0, z = x, zo;
    do { x *= x; zo = z; z += x * y; y += y; } while (zo != z);
    return z;
}
static double hll_tau(double x) {
    if (x == 0.0 || x == 1.0) return 0.0;
    double y = 1.0, z = 1.0 - x, zo;
    do { x = std::sqrt(x); zo = z; y *= 0.5; z -= (1.0 - x) * (1.0 - x) * y; } while (zo != z);
    return z / 3.0;
}

extern "C" int kta_alive_keys_hll(const kta_handle *h, double *out) {
    if (!out) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, 0, false);
    if (rc) return rc;
    if (!h->nhll) return fail(KTA_ERR_NOT_ENABLED, "hll_precision was 0");
    const int p = h->cfg.hll_precision, q = 32 - p;
    const double m = (double)h->nhll;
    std::vector<double> C((size_t)q + 2, 0.0);
    for (uint32_t r : h->h_hll) C[std::min<uint32_t>(r, (uint32_t)q + 1)] += 1.0;
    double z = m * hll_tau(1.0 - C[(size_t)q + 1] / m);
    for (int k = q; k >= 1; k--) z = 0.5 * (z + C[(size_t)k]);
    z += m * hll_sigma(C[0] / m);
    *out = 0.72134752044448170368 * m * m / z;
    return KTA_OK;
}

extern "C" int kta_hll_registers(const kta_handle *h, uint8_t *out, size_t cap) {
    if (!out) return fail(KTA_ERR_INVALID, "bad argument");
    const int rc = check_read(h, 0, false);
    if (rc) return rc;
    if (!h->nhll) return fail(KTA_ERR_NOT_ENABLED, "hll_precision was 0");
    if (cap < h->nhll) return fail(KTA_ERR_INVALID, "buffer too small: %zu < %zu", cap, h->nhll);
    for (size_t i = 0; i < h->nhll; i++) out[i] = (uint8_t)h->h_hll[i];
    return KTA_OK;
}

extern "C" int kta_fnv32_host(kta_handle *h, int64_t n, const int32_t *key_len, const uint8_t *key_bytes,
                              int64_t key_bytes_len, uint32_t *out) {
    if (!h || n < 0 || (n && (!key_len || !out))) return fail(KTA_ERR_INVALID, "bad argument");
    if (n == 0) return KTA_OK;
    int rc;
    if ((rc = set_device(h))) return rc;
    std::vector<uint64_t> off((size_t)n);
    uint64_t acc = 0;
    for (int64_t i = 0; i < n; i++) {
        off[(size_t)i] = acc;
        acc += key_len[i] > 0 ? (uint64_t)key_len[i] : 0;
    }
    if ((int64_t)acc > key_bytes_len) return fail(KTA_ERR_INVALID, "key_bytes_len %lld < sum of key_len %llu",
                                                  (long long)key_bytes_len, (unsigned long long)acc);
    int32_t *d_len = nullptr;
    uint64_t *d_off = nullptr;
    uint8_t *d_keys = nullptr;
    uint32_t *d_out = nullptr;
    cudaStream_t s = h->stream;
    cudaError_t e = cudaSuccess;
    do {
        if ((e = cudaMalloc(&d_len, n * 4))) break;
        if ((e = cudaMalloc(&d_off, n * 8))) break;
        if ((e = cudaMalloc(&d_keys, acc + 16))) break;
        if ((e = cudaMalloc(&d_out, n * 4))) break;
        if ((e = cudaMemcpyAsync(d_len, key_len, n * 4, cudaMemcpyHostToDevice, s))) break;
        if ((e = cudaMemcpyAsync(d_off, off.data(), n * 8, cudaMemcpyHostToDevice, s))) break;
        if (acc && (e = cudaMemcpyAsync(d_keys, key_bytes, acc, cudaMemcpyHostToDevice, s))) break;
        fnv32_kernel<<<(int)std::min<int64_t>((n + 255) / 256, 1024), 256, 0, s>>>(n, d_len, d_off, d_keys, d_out);
        h->launches++;
        if ((e = cudaGetLastError())) break;
        if ((e = cudaMemcpyAsync(out, d_out, n * 4, cudaMemcpyDeviceToHost, s))) break;
        e = cudaStreamSynchronize(s);
    } while (0);
    cudaFree(d_len); cudaFree(d_off); cudaFree(d_keys); cudaFree(d_out);
    if (e != cudaSuccess) return fail(KTA_ERR_CUDA, "kta_fnv32_host: %s", cudaGetErrorString(e));
    return KTA_OK;
}

// test hook: capture the per-record hash computed inside the fused scan (device buffer of n u32, or NULL)
extern "C" int kta_set_hash_capture(kta_handle *h, uint32_t *dev_out) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;   // records already landed were taken with the old setting
    h->d_hash_out = dev_out;
    h->pc.hash = h->need_hash || h->d_hash_out;
    return KTA_OK;
}

// ------------------------------------------------------------------------------------------------
// multi-GPU merge
// ------------------------------------------------------------------------------------------------
extern "C" int64_t kta_merge_words(const kta_handle *h, int32_t world) {
    if (!h || world < 1) return -1;
    return (int64_t)(h->nsums + (size_t)world * 4 + (size_t)world * (h->nhll / 8));
}

extern "C" int kta_merge_export_device(kta_handle *h, int32_t rank, int32_t world, uint64_t *dev_buf) {
    if (!h || !dev_buf || world < 1 || rank < 0 || rank >= world) return fail(KTA_ERR_INVALID, "bad argument");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;
    if (!h->pending.empty() && (rc = alive_check(h))) return rc;
    merge_export_kernel<<<h->sm_count, 256, 0, h->stream>>>(h->d_sums, h->nsums, h->d_minmax, h->d_hll, h->nhll, rank,
                                                           world, reinterpret_cast<unsigned long long *>(dev_buf));
    h->launches++;
    CU(cudaGetLastError());
    // With its own stream the handle must finish before the caller's collective may read the buffer.  On an
    // adopted stream (kta_set_stream) the caller's collective is ordered behind this kernel by the stream itself.
    if (h->own_stream) {
        CU(cudaStreamSynchronize(h->stream));
        return collect_timing(h);
    }
    return KTA_OK;
}

extern "C" int kta_merge_import_device(kta_handle *h, int32_t world, const uint64_t *dev_buf) {
    if (!h || !dev_buf || world < 1) return fail(KTA_ERR_INVALID, "bad argument");
    int rc;
    if ((rc = set_device(h))) return rc;
    merge_import_kernel<<<h->sm_count, 256, 0, h->stream>>>(h->d_sums, h->nsums, h->d_minmax, h->d_hll, h->nhll,
                                                           h->d_hll_floor, world,
                                                           reinterpret_cast<const unsigned long long *>(dev_buf));
    h->launches++;
    CU(cudaGetLastError());
    h->finalized = false;
    if (h->own_stream) CU(cudaStreamSynchronize(h->stream));
    return KTA_OK;
}

static int alive_export(kta_handle *h, int mode, uint32_t *dh, uint64_t *ds, int64_t cap, int64_t *count) {
    if (!h || !count) return fail(KTA_ERR_INVALID, "bad argument");
    if (!h->d_alive_table) return fail(KTA_ERR_NOT_ENABLED, "count_alive_keys was not enabled");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;
    if ((rc = alive_check(h))) return rc;
    if (h->alive_rebased)
        return fail(KTA_ERR_INVALID, "the alive-key table was rebased (more than 2^31 sequence numbers since kta_reset): its "
                    "entries no longer carry absolute sequence numbers and cannot be merged across GPUs");
    CU(cudaMemsetAsync(h->d_scalar + 1, 0, 8, h->stream));
    alive_export_kernel<<<h->sm_count * 8, THREADS, 0, h->stream>>>(
        h->d_alive_table, (size_t)h->alive_pairs * 2, h->alive_origin, mode, h->d_scalar + 1, dh,
        reinterpret_cast<unsigned long long *>(ds), (unsigned long long)cap);
    h->launches++;
    CU(cudaGetLastError());
    unsigned long long c = 0;
    CU(cudaMemcpyAsync(&c, h->d_scalar + 1, 8, cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    *count = (int64_t)c;
    if (mode == 1 && (int64_t)c > cap) return fail(KTA_ERR_INVALID, "export buffer too small: %llu > %lld", c, (long long)cap);
    return KTA_OK;
}

extern "C" int kta_alive_export_count(kta_handle *h, int64_t *count) { return alive_export(h, 0, nullptr, nullptr, 0, count); }

extern "C" int kta_alive_export_device(kta_handle *h, uint32_t *dev_hash, uint64_t *dev_stamp, int64_t cap, int64_t *count) {
    if (!dev_hash || !dev_stamp) return fail(KTA_ERR_INVALID, "bad argument");
    return alive_export(h, 1, dev_hash, dev_stamp, cap, count);
}

extern "C" int kta_alive_import_device(kta_handle *h, const uint32_t *dev_hash, const uint64_t *dev_stamp, int64_t count) {
    if (!h || count < 0 || (count && (!dev_hash || !dev_stamp))) return fail(KTA_ERR_INVALID, "bad argument");
    if (!h->d_alive_table) return fail(KTA_ERR_NOT_ENABLED, "count_alive_keys was not enabled");
    if (count == 0) return KTA_OK;
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = alive_check(h))) return rc;   // nothing pending: a re-run below only concerns the imported stamps
    const int grid = (int)std::min<int64_t>((count + THREADS - 1) / THREADS, (int64_t)h->sm_count * 8);
    for (int round = 0;; round++) {
        const AliveTable t{h->d_alive_table, h->alive_pairs, h->d_alive_status, 0};
        alive_import_kernel<<<grid, THREADS, 0, h->stream>>>(t, h->alive_origin, dev_hash,
                                                             reinterpret_cast<const unsigned long long *>(dev_stamp), count);
        h->launches++;
        CU(cudaGetLastError());
        // the imported list is the caller's and still valid: if the table was too small, alive_check grew it (nothing
        // is pending, so it re-ran nothing) and the import is simply applied again — stamping is idempotent
        CU(cudaMemcpyAsync(h->h_alive_status, h->d_alive_status, 8, cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        const bool dropped = h->h_alive_status[0] != 0;
        if ((rc = alive_check(h))) return rc;
        if (!dropped) break;
        if (round > 40) return fail(KTA_ERR_INVALID, "alive-key table growth did not converge");
    }
    h->finalized = false;
    return KTA_OK;
}

// ------------------------------------------------------------------------------------------------
// introspection
// ------------------------------------------------------------------------------------------------
extern "C" int kta_stats(const kta_handle *h, uint64_t *kernel_launches, uint64_t *records_scanned) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    if (kernel_launches) *kernel_launches = h->launches;
    if (records_scanned) *records_scanned = h->records;
    return KTA_OK;
}

extern "C" int kta_alive_table_stats(kta_handle *h, uint64_t *slots, uint64_t *occupied, uint64_t *grows, uint64_t *reruns) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    if (!h->d_alive_table) return fail(KTA_ERR_NOT_ENABLED, "count_alive_keys was not enabled");
    int rc;
    if ((rc = set_device(h))) return rc;
    if ((rc = ring_flush(h))) return rc;
    if ((rc = alive_check(h))) return rc;   // settles pending stamps and counts the table
    if (slots) *slots = (uint64_t)h->alive_pairs * 2;
    if (occupied) *occupied = h->alive_occupied;
    if (grows) *grows = h->alive_grows;
    if (reruns) *reruns = h->alive_reruns;
    return KTA_OK;
}

extern "C" int kta_set_timing(kta_handle *h, int enabled) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    h->timing = enabled != 0;
    h->scan_ms = 0;
    h->scan_launches_timed = 0;
    return KTA_OK;
}

extern "C" int kta_scan_time_ms(kta_handle *h, double *total_ms, uint64_t *launches) {
    if (!h) return fail(KTA_ERR_INVALID, "null handle");
    int rc;
    if ((rc = set_device(h))) return rc;
    CU(cudaStreamSynchronize(h->stream));
    if ((rc = collect_timing(h))) return rc;
    if (total_ms) *total_ms = h->scan_ms;
    if (launches) *launches = h->scan_launches_timed;
    return KTA_OK;
}
