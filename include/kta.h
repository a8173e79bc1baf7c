/*
 * kta.h — C ABI of libkta_gpu.so: the B200-native (sm_100a) replacement for the per-message
 * metric-aggregation path of xenji/kafka-topic-analyzer.
 *
 * Boundary being replaced (reference, Rust):
 *   trait MetricHandler { fn handle_message(&mut self, m: &BorrowedMessage) }    src/kafka.rs:18-20
 *   TopicAnalyzer::add_metric_handler                                            src/kafka.rs:56-58
 *   call site, once per handler per polled message                               src/kafka.rs:107-109
 *   impl MetricHandler for MessageMetrics                                        src/metric.rs:206-253
 *   impl MetricHandler for LogCompactionInMemoryMetrics                          src/metric.rs:288-305
 *   read-back: getters src/metric.rs:104-195, sum_all_alive :282-284, used at    src/main.rs:130-170
 *
 * One kta_handle is BOTH handlers (MessageMetrics always; LogCompactionInMemoryMetrics when
 * cfg.count_alive_keys == 1, mirroring `-c`, src/main.rs:77-80).
 *
 * Rules of the boundary
 *   - plain C types only; no exceptions or unwinding cross it; every entry point returns a status
 *     (KTA_OK == 0) and kta_last_error() gives the text for the last failure on the calling thread.
 *   - single-producer: all calls on one handle come from one host thread, as in the reference
 *     (handlers are `&mut`, src/kafka.rs:15).  Different handles are independent.
 *   - the library copies what it needs before a push returns; caller buffers are never retained
 *     (BorrowedMessage is only borrowed for the call, src/kafka.rs:107-109).
 *   - there is NO CPU fallback: without a usable CUDA device kta_create fails with KTA_ERR_CUDA.
 *
 * Record encoding (rdkafka 0.25.0 accessor semantics, call sites src/metric.rs:208-209,218,233):
 *   key_len   == -1  key() is None            key_len   == 0  Some(&[])  (hashes to 0x811c9dc5)
 *   value_len == -1  payload() is None (tombstone)             value_len == 0  Some(&[])  (alive)
 *   ts_ms     == -1  timestamp().to_millis() is None → treated as 0 (src/metric.rs:209)
 *   partition must lie in [0, cfg.num_partitions)
 *   value BYTES never cross the boundary: the reference only reads v.len() (src/metric.rs:235).
 */
#ifndef KTA_H
#define KTA_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KTA_ABI_VERSION 2
#define KTA_KEY_TILE 128      /* records per key tile (granularity of kta_batch.key_tile_base) */
#define KTA_HIST_BUCKETS 32   /* bucket(len) = len == 0 ? 0 : 1 + floor(log2(len)) */

enum {
    KTA_OK = 0,
    KTA_ERR_INVALID = 1,       /* bad argument / bad state */
    KTA_ERR_CUDA = 2,          /* CUDA runtime failure (including: no device) */
    KTA_ERR_NOMEM = 3,
    KTA_ERR_PARTITION = 4,     /* a record's partition was outside [0, num_partitions) */
    KTA_ERR_DIV_BY_ZERO = 5,   /* the reference would panic here: avg with sum > 0 && alive == 0
                                  (src/metric.rs:132-157) */
    KTA_ERR_NOT_ENABLED = 6,   /* getter for a feature that was not enabled at create */
    KTA_ERR_NOT_FINALIZED = 7
};

typedef struct kta_handle kta_handle;

typedef struct kta_config {
    int32_t struct_size;       /* = sizeof(kta_config) */
    int32_t device;            /* CUDA device ordinal, -1 = current device */
    int32_t num_partitions;    /* P; partition ids are 0..P-1 (metadata, src/kafka.rs:60-72) */
    int32_t count_alive_keys;  /* 1 = exact alive-key table, i.e. `-c` given once (src/main.rs:77-80) */
    int32_t hll_precision;     /* EXTENSION: 0 = off, else 4..18 HyperLogLog index bits */
    int32_t alive_table_kib;   /* initial size of the alive-key table in KiB (8 bytes per distinct key hash, kept at
                                  load <= 0.7 and grown on demand); 0 = default (131072 = 128 MiB: 1e7 keys) */
    int64_t ring_records;      /* records per landing-ring chunk for kta_push / host batches; 0 = default */
    int64_t ring_key_bytes;    /* key bytes per landing-ring chunk; 0 = default */
    int64_t now_s;             /* construction wall clock for earliest_message (Utc::now(), */
    int32_t now_ns;            /*   src/metric.rs:39); now_s == INT64_MIN → library reads the clock */
    int32_t reserved1;
    int32_t shard_world;       /* partition-sharded job (one handle per GPU, gpu = partition mod G, SURVEY.md §8 e): this */
    int32_t shard_rank;        /*   handle scans only partitions p with p % shard_world == shard_rank; records of other
                                    partitions are left out like out-of-range ones.  0 or 1 = not sharded.  The handle
                                    still holds (and, after kta_merge_import_device, reports) all num_partitions. */
} kta_config;

/* kta_batch.seq_base value that means "continue this handle's running count" (what kta_push does: the consumer's
 * `seq += 1`, src/kafka.rs:99) */
#define KTA_SEQ_AUTO UINT64_MAX

/* SoA record batch.  Pointers are all host or all device (see the two scan entry points). */
typedef struct kta_batch {
    int64_t n;                     /* records */
    uint64_t seq_base;             /* seq of record 0; record i has seq_base + i (src/kafka.rs:99), or KTA_SEQ_AUTO.
                                      With count_alive_keys the LAST record of a key decides (src/metric.rs:295,298) and
                                      "last" is by seq: a batch without a seq column whose seq_base lies below the
                                      handle's running count is refused (it would let older records win silently). */
    const int32_t *partition;      /* [n] */
    const int64_t *offset;         /* [n] carried for the caller; never read by a metric (may be NULL) */
    const int64_t *ts_ms;          /* [n] */
    const int32_t *key_len;        /* [n] */
    const int32_t *value_len;      /* [n] */
    const uint8_t *key_bytes;      /* keys packed back to back in record order (null/empty keys take
                                      0 bytes); may be NULL when neither -c nor HLL is enabled */
    int64_t key_bytes_len;         /* = sum(max(key_len, 0)) */
    const uint64_t *key_tile_base; /* optional [ceil(n/KTA_KEY_TILE)+1]: byte offset into key_bytes
                                      of the first key of each tile (+ total at the end).  NULL →
                                      the library derives it with one extra pass over key_len. */
    const uint64_t *seq;           /* optional [n] explicit sequence numbers (partition-sharded
                                      scans, where the global order is not base+i); NULL → seq_base+i.
                                      The alive-key table keeps 31 bits of seq: explicit sequence numbers must stay
                                      below 2^31 - 2 between kta_reset calls (kta_finalize reports violations);
                                      implicit ones are unlimited (the table is rebased as the stream advances). */
} kta_batch;

enum kta_counter_id { /* per-partition counters, src/metric.rs:13-19 / getters :104-130 */
    KTA_TOTAL = 0,
    KTA_TOMBSTONES = 1,
    KTA_ALIVE = 2,
    KTA_KEY_NULL = 3,
    KTA_KEY_NON_NULL = 4,
    KTA_KEY_SIZE_SUM = 5,
    KTA_VALUE_SIZE_SUM = 6
};
enum kta_avg_id { KTA_KEY_SIZE_AVG = 0, KTA_VALUE_SIZE_AVG = 1, KTA_MESSAGE_SIZE_AVG = 2 };
enum kta_global_id { /* src/metric.rs:22-25 / getters :177-195 */
    KTA_SMALLEST_MESSAGE = 0,
    KTA_LARGEST_MESSAGE = 1,
    KTA_OVERALL_SIZE = 2,
    KTA_OVERALL_COUNT = 3
};

const char *kta_last_error(void);
int kta_abi_version(void);
/* number of CUDA devices visible, or -1 if the runtime cannot initialise (no throw, no abort) */
int kta_device_count(void);

/* MessageMetrics::new + (cfg.count_alive_keys) LogCompactionInMemoryMetrics::new
 * src/metric.rs:30-46, 267-271; registration src/main.rs:108-115 */
int kta_create(const kta_config *cfg, kta_handle **out);
int kta_destroy(kta_handle *h);
/* back to the just-constructed state (keeps device allocations) */
int kta_reset(kta_handle *h);

/* MetricHandler::handle_message for one record (src/kafka.rs:107-109).  Lands the record in a
 * pinned ring chunk; full chunks are staged to HBM with cudaMemcpyAsync and scanned asynchronously.
 * `offset` is accepted for interface parity and ignored.  `key` may be NULL iff key_len <= 0. */
int kta_push(kta_handle *h, int32_t partition, int64_t offset, int64_t ts_ms, const uint8_t *key,
             int32_t key_len, int32_t value_len);

/* The same for a whole SoA batch in HOST memory (pinned or pageable): chunked host→device copies
 * overlapped with the scan kernels.  Returns once the caller's buffers may be reused. */
int kta_push_batch_host(kta_handle *h, const kta_batch *b);

/* The same for an SoA batch already resident in DEVICE memory (asynchronous on the handle's
 * stream; the buffers must stay valid until kta_sync / kta_finalize). */
int kta_scan_batch_device(kta_handle *h, const kta_batch *b);

/* drain the ring and wait for all queued scans */
int kta_sync(kta_handle *h);
/* kta_sync + resolve the alive-key table + bring the metric state to the host.  Getters below are
 * valid after this.  More records may be pushed afterwards; finalize again to refresh. */
int kta_finalize(kta_handle *h);

/* getters — src/metric.rs:104-130 */
int kta_counter(const kta_handle *h, int which, int32_t partition, uint64_t *out);
/* src/metric.rs:132-157; KTA_ERR_DIV_BY_ZERO where the reference panics */
int kta_avg(const kta_handle *h, int which, int32_t partition, uint64_t *out);
/* src/metric.rs:159-167 (f32 arithmetic, same operation order) */
int kta_dirty_ratio(const kta_handle *h, int32_t partition, float *out);
/* src/metric.rs:177-195 */
int kta_global(const kta_handle *h, int which, uint64_t *out);
/* earliest_message / latest_message, src/metric.rs:169-175, as UTC seconds (+ ns of the
 * construction clock when no record was earlier than it) */
int kta_timestamps(const kta_handle *h, int64_t *earliest_s, int32_t *earliest_ns, int64_t *latest_s);
/* LogCompactionInMemoryMetrics::sum_all_alive, src/metric.rs:282-284 (exact) */
int kta_alive_keys(const kta_handle *h, uint64_t *out);
/* records whose partition was outside [0, num_partitions): they are left out of EVERY metric (kta_finalize returns
 * KTA_ERR_PARTITION to say so; the getters stay valid and describe the in-range records) */
int kta_bad_partition_records(const kta_handle *h, uint64_t *out);

/* ---- EXTENSIONS: not in the reference (SURVEY.md D2, D3) ---- */
/* per-partition log2 size histogram: which = 0 key sizes, 1 value sizes */
int kta_hist(const kta_handle *h, int which, int32_t partition, uint64_t out[KTA_HIST_BUCKETS]);
/* HyperLogLog estimate of distinct alive key hashes.  With count_alive_keys the sketch is built
 * from the resolved alive set; otherwise it is the in-stream sketch of every (key, value) insert,
 * which equals the alive count only on tombstone-free topics. */
int kta_alive_keys_hll(const kta_handle *h, double *out);
/* raw registers (one byte each, 1 << hll_precision of them) */
int kta_hll_registers(const kta_handle *h, uint8_t *out, size_t cap);
/* the hash itself, computed on the device for n packed keys given in HOST memory (test hook for
 * src/fnv32.rs:92-101 known-answer vectors).  key_len[i] < 0 yields 0. */
int kta_fnv32_host(kta_handle *h, int64_t n, const int32_t *key_len, const uint8_t *key_bytes,
                   int64_t key_bytes_len, uint32_t *out);

/* ---- multi-GPU merge (one process per GPU; the collective itself is the caller's: NCCL via
 * torch.distributed, or ncclAllReduce directly) ----
 * The mergeable state is exported as ONE array of u64 laid out so that a single SUM all-reduce
 * merges everything: sums as they are; min/max scalars and HLL registers in per-rank slots
 * (zero elsewhere) that the import folds with min/max.  words = kta_merge_words(h, world). */
int64_t kta_merge_words(const kta_handle *h, int32_t world);
int kta_merge_export_device(kta_handle *h, int32_t rank, int32_t world, uint64_t *dev_buf);
int kta_merge_import_device(kta_handle *h, int32_t world, const uint64_t *dev_buf);
/* exact alive-key exchange: compact (hash, stamp) entries of the local table, to be all-gathered
 * and re-applied on every rank (last-writer-wins by global seq is associative/commutative). */
int kta_alive_export_count(kta_handle *h, int64_t *count);
int kta_alive_export_device(kta_handle *h, uint32_t *dev_hash, uint64_t *dev_stamp, int64_t cap,
                            int64_t *count);
int kta_alive_import_device(kta_handle *h, const uint32_t *dev_hash, const uint64_t *dev_stamp,
                            int64_t count);

/* ---- Kafka log segments (SURVEY.md §8 f2): the step before the handlers ----
 * A segment is the concatenation of RecordBatch v2 (magic 2) batches of ONE partition — what a broker stores in
 * <topic>-<partition>/NNN.log and returns in a fetch response.  The library decodes it on the GPU into the SoA
 * columns above (what librdkafka's parser + BorrowedMessage accessors do per message, src/kafka.rs:93,
 * src/metric.rs:208-209,218,233) and scans it.  Control batches are skipped, LogAppendTime batches use
 * maxTimestamp, a record's timestamp is baseTimestamp + timestampDelta (only a result of -1 is "not available"),
 * CRCs are not verified (librdkafka default check.crcs=false).  gzip, LZ4 (frame format), Snappy (raw or
 * xerial-framed) and zstd batches are decompressed on the GPU (zstd: no dictionaries; the content checksum is not
 * verified); batches naming an unassigned codec (5-7) are rejected (KTA_ERR_INVALID).
 * Differences from a librdkafka consumer: records of aborted transactions ARE delivered (read_committed filtering
 * needs the transaction index, which is not read), legacy magic 0/1 message sets are reported as malformed. */
/* raw bytes already in device memory; batch_off[nbatches] = byte offset of every batch header (device memory) */
int kta_scan_log_segment_device(kta_handle *h, int32_t partition, const uint8_t *dev_bytes, int64_t len,
                                const uint64_t *dev_batch_off, int64_t nbatches, int64_t *records_out);
/* the same for batches of SEVERAL partitions lying in one device buffer (e.g. a whole fetch response, or many segments
 * staged back to back): dev_batch_partition[nbatches] names each batch's partition.  One decode and one scan. */
int kta_scan_log_batches_device(kta_handle *h, const uint8_t *dev_bytes, int64_t len, const uint64_t *dev_batch_off,
                                const int32_t *dev_batch_partition, int64_t nbatches, int64_t *records_out);
/* raw bytes in host memory (e.g. an mmap of a .log file); returns when `bytes` may be reused */
int kta_push_log_segment_host(kta_handle *h, int32_t partition, const uint8_t *bytes, int64_t len, int64_t *records_out);
/* several segments (any partitions) in one go: one staging copy per segment, ONE decode and ONE scan for all of them */
int kta_push_log_segments_host(kta_handle *h, int32_t nsegs, const int32_t *partitions, const uint8_t *const *bytes,
                               const int64_t *lens, int64_t *records_out);

/* ---- introspection for benchmarks ---- */
/* kernels launched by this handle since create/reset, and device time of the scan kernels (ms,
 * CUDA events on the handle's stream; only collected when enabled) */
int kta_stats(const kta_handle *h, uint64_t *kernel_launches, uint64_t *records_scanned);
int kta_set_timing(kta_handle *h, int enabled);
int kta_scan_time_ms(kta_handle *h, double *total_ms, uint64_t *launches);
/* alive-key table: slots allocated, slots occupied (= distinct key hashes seen), how often it was grown and how many
 * batches had to be re-stamped because it was too small when they were scanned (any pointer may be NULL) */
int kta_alive_table_stats(kta_handle *h, uint64_t *slots, uint64_t *occupied, uint64_t *grows, uint64_t *reruns);
/* raw cudaStream_t of the handle (so a torch caller can order against it) */
void *kta_stream(kta_handle *h);
/* adopt a caller-owned cudaStream_t (e.g. torch's current stream) for all further work of this handle */
int kta_set_stream(kta_handle *h, void *stream);

/* ---- synthetic in-memory topic (configs[0..4] of BASELINE.json; SURVEY.md §8 d) ----
 * Counter-based: every field of record i is a pure function of (seed, i); the same code runs on
 * host and device.  Partition p of record i: runs of run_len records, runs dealt round-robin with a
 * per-cycle pseudo-random rotation, so per-partition offsets are closed-form and a rank that owns
 * partitions {p : p % world == rank} can enumerate exactly its records. */
/* key_mode flags.  Both are integer-only so that host and device generate identical topics.
 * KEYS_LOGUNIFORM: key ids are drawn log-uniformly (a staircase approximation of Zipf s = 1: id k of a partition
 *   is about as likely as 1/(k+1)) instead of uniformly — a few hot keys, a long tail of cold ones.
 * VALUES_GEOMETRIC: the uniform value length is multiplied by 2^g, P(g = k) = 2^-(k+1), g <= 6 — a geometric tail. */
#define KTA_SYNTH_KEYS_LOGUNIFORM 0x100
#define KTA_SYNTH_VALUES_GEOMETRIC 0x200

typedef struct kta_synth_spec {
    uint64_t seed;               /* default 0x4B544131 ("KTA1") */
    int64_t n_total;             /* records in the whole topic; multiple of num_partitions*run_len */
    int32_t num_partitions;
    int32_t run_len;             /* >= 1 */
    uint64_t distinct_keys;      /* D; rounded down to a multiple of num_partitions, >= P */
    int32_t key_mode;            /* low byte: 0 = 16-byte binary (id, id*phi64) LE; 1 = ASCII "key-<id>";
                                    2 = variable-length binary, 0..40 bytes.  Optional flags (stress cases):
                                    KTA_SYNTH_KEYS_LOGUNIFORM, KTA_SYNTH_VALUES_GEOMETRIC */
    int32_t value_mean;          /* value_len uniform in [mean/2, 3*mean/2] */
    int32_t null_key_per_10k;
    int32_t tombstone_per_10k;
    int32_t ts_missing_per_10k;
    int32_t empty_value_per_10k;
} kta_synth_spec;

/* number of records of the topic owned by `rank` of `world` (partitions p % world == rank) */
int64_t kta_synth_shard_records(const kta_synth_spec *s, int32_t rank, int32_t world);
/* Fill host SoA columns for local records [start, start+count) of the shard.  Any output pointer
 * may be NULL.  key_bytes_cap bounds key_bytes; *key_bytes_len receives the bytes written. */
int kta_synth_fill_host(const kta_synth_spec *s, int32_t rank, int32_t world, int64_t start,
                        int64_t count, int32_t *partition, int64_t *offset, int64_t *ts_ms,
                        int32_t *key_len, int32_t *value_len, uint64_t *seq, uint8_t *key_bytes,
                        int64_t key_bytes_cap, int64_t *key_bytes_len);
/* Same on the device (pointers are device memory; key_tile_base must hold
 * ceil(count/KTA_KEY_TILE)+1 words).  Synchronous. */
int kta_synth_fill_device(const kta_synth_spec *s, int32_t device, int32_t rank, int32_t world,
                          int64_t start, int64_t count, int32_t *partition, int64_t *offset,
                          int64_t *ts_ms, int32_t *key_len, int32_t *value_len, uint64_t *seq,
                          uint8_t *key_bytes, int64_t key_bytes_cap, uint64_t *key_tile_base,
                          int64_t *key_bytes_len);

/* The same topic as a broker stores it: records [start, start+count) (offset order) of one partition as an
 * uncompressed RecordBatch v2 log segment, `batch_records` records per batch (feeds kta_push_log_segment_host). */
int kta_synth_encode_segment_host(const kta_synth_spec *s, int32_t partition, int64_t start, int64_t count,
                                  int32_t batch_records, uint8_t *out, int64_t cap, int64_t *len);

#ifdef __cplusplus
}
#endif
#endif
