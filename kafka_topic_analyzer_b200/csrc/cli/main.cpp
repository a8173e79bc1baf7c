// kafka-topic-analyzer (B200 build) — the reference's CLI surface (src/main.rs:32-67) over libkta_gpu.so.
//
//   -t/--topic TOPIC  -b/--bootstrap-server HOSTS  [--librdkafka k=v,...]  [-c/--count-alive-keys]
//   --synthetic n=...,partitions=...,value_mean=...,run_len=...,distinct_keys=...,key_mode=...,seed=...,
//               tombstone_per_10k=...,null_key_per_10k=...,zipf_keys=1,geometric_values=1
//                                                                (the in-memory topic of BASELINE.json configs)
//   --log-dir DIR              read Kafka log segments from DIR/<topic>-<partition>/*.log (a broker's data directory)
//                              and decode them on the GPU (RecordBatch v2, magic 2; uncompressed, gzip, LZ4, Snappy or
//                              zstd batches).  Differences from a librdkafka
//                              consumer: records of ABORTED transactions are counted (a consumer with the default
//                              isolation.level=read_committed filters them; the .txnindex files are not read here),
//                              and legacy magic 0/1 message sets are reported as malformed.
//   --feed push|batch|device   how records reach the handlers: kta_push per record (the reference's call shape),
//                              kta_push_batch_host, or generated and scanned in HBM
//
// There is no librdkafka and no broker in this build (SURVEY.md D9): without --synthetic the program explains
// that and exits, like the reference does when it cannot fetch metadata.  Everything numeric comes from the
// GPU library; this file only feeds records and prints.
#include <cuda_runtime_api.h>

#include <dirent.h>
#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <fstream>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "../../../include/kta.h"
#include "kta_report.hpp"

static void die(const char *what) {
    fprintf(stderr, "error: %s: %s\n", what, kta_last_error());
    exit(1);
}
#define KTA(call) do { if ((call) != KTA_OK) die(#call); } while (0)

// kta_finalize reports records whose partition lies outside the topic's metadata with KTA_ERR_PARTITION; the state is
// valid (those records were left out of every metric), so the report is still printed — with a warning, like the
// reference's warn!() for a failed poll (src/kafka.rs:95-97).
static void finalize_or_warn(kta_handle *h) {
    const int rc = kta_finalize(h);
    if (rc == KTA_ERR_PARTITION) fprintf(stderr, "warning: %s\n", kta_last_error());
    else if (rc != KTA_OK) die("kta_finalize");
}


// ---- --log-dir: a broker's data directory instead of a live cluster ------------------------------------------------
static bool read_file(const std::string &path, std::vector<uint8_t> &out) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    if (!f) return false;
    const std::streamsize n = f.tellg();
    f.seekg(0);
    out.resize((size_t)n);
    return n == 0 || (bool)f.read(reinterpret_cast<char *>(out.data()), n);
}

static int print_report(kta_handle *h, const std::string &topic, const std::vector<int> &partitions, const std::vector<int64_t> &start_offsets,
                        const std::vector<int64_t> &end_offsets, bool alive, int hll, uint64_t duration_secs);

static int analyze_log_dir(const std::string &topic, const std::string &dir, bool alive, int hll,
                           std::chrono::steady_clock::time_point start_time) {
    // get_topic_offsets (src/kafka.rs:60-72) from the files: partitions = <topic>-<n> directories, low watermark =
    // first batch's baseOffset, high watermark = last batch's baseOffset + lastOffsetDelta + 1
    std::map<int, std::vector<std::string>> segs;
    DIR *d = opendir(dir.c_str());
    if (!d) { fprintf(stderr, "Error fetching metadata: cannot open %s\n", dir.c_str()); return 101; }
    while (dirent *e = readdir(d)) {
        const std::string name = e->d_name;
        if (name.size() <= topic.size() + 1 || name.compare(0, topic.size() + 1, topic + "-") != 0) continue;
        const std::string num = name.substr(topic.size() + 1);
        if (num.empty() || num.find_first_not_of("0123456789") != std::string::npos) continue;
        const int p = atoi(num.c_str());
        DIR *pd = opendir((dir + "/" + name).c_str());
        if (!pd) continue;
        std::vector<std::string> files;
        while (dirent *fe = readdir(pd)) {
            const std::string fn = fe->d_name;
            if (fn.size() > 4 && fn.substr(fn.size() - 4) == ".log") files.push_back(dir + "/" + name + "/" + fn);
        }
        closedir(pd);
        std::sort(files.begin(), files.end());
        segs[p] = files;
    }
    closedir(d);
    if (segs.empty()) { fprintf(stderr, "Topic not found!\n"); return 101; }  // src/kafka.rs:62
    const int P = segs.rbegin()->first + 1;
    std::vector<int64_t> start_offsets(P, 0), end_offsets(P, 0);
    kta_config cfg{};
    cfg.struct_size = sizeof cfg;
    cfg.device = -1;
    cfg.num_partitions = P;
    cfg.count_alive_keys = alive ? 1 : 0;
    cfg.hll_precision = hll;
    cfg.now_s = INT64_MIN;
    kta_handle *h = nullptr;
    KTA(kta_create(&cfg, &h));
    printf("Subscribing to %s\n", topic.c_str());
    printf("Starting message consumption...\n");
    auto be64 = [](const uint8_t *p) { uint64_t v = 0; for (int i = 0; i < 8; i++) v = (v << 8) | p[i]; return (int64_t)v; };
    auto be32 = [](const uint8_t *p) { return (int32_t)(((uint32_t)p[0] << 24) | ((uint32_t)p[1] << 16) | ((uint32_t)p[2] << 8) | p[3]); };
    // segments are handed over in groups of up to 512 MiB: one staging copy each, one GPU decode + scan per group
    std::vector<std::vector<uint8_t>> bufs;
    std::vector<int32_t> parts;
    int64_t total = 0, pending = 0;
    auto flush = [&]() {
        if (bufs.empty()) return;
        std::vector<const uint8_t *> ptrs;
        std::vector<int64_t> lens;
        for (auto &b : bufs) { ptrs.push_back(b.data()); lens.push_back((int64_t)b.size()); }
        int64_t nrec = 0;
        KTA(kta_push_log_segments_host(h, (int32_t)bufs.size(), parts.data(), ptrs.data(), lens.data(), &nrec));
        total += nrec;
        bufs.clear(); parts.clear(); pending = 0;
    };
    for (auto &kv : segs) {
        bool first = true;
        for (const auto &path : kv.second) {
            std::vector<uint8_t> buf;
            if (!read_file(path, buf)) { fprintf(stderr, "cannot read %s\n", path.c_str()); return 1; }
            for (int64_t pos = 0; pos + 61 <= (int64_t)buf.size();) {
                const int64_t bl = be32(buf.data() + pos + 8);
                if (bl < 49 || pos + 12 + bl > (int64_t)buf.size()) break;
                if (first) { start_offsets[kv.first] = be64(buf.data() + pos); first = false; }
                end_offsets[kv.first] = be64(buf.data() + pos) + be32(buf.data() + pos + 23) + 1;
                pos += 12 + bl;
            }
            pending += (int64_t)buf.size();
            parts.push_back(kv.first);
            bufs.push_back(std::move(buf));
            if (pending >= ((int64_t)512 << 20)) flush();
        }
    }
    flush();
    if (std::all_of(end_offsets.begin(), end_offsets.end(), [](int64_t v) { return v == 0; })) {
        fprintf(stderr, "Given topic has no content, no analysis possible. Exiting.\n");  // main.rs:98-101
        return 254;
    }
    finalize_or_warn(h);
    const uint64_t secs = (uint64_t)std::chrono::duration_cast<std::chrono::seconds>(std::chrono::steady_clock::now() - start_time).count();
    // the report has one row per partition of the topic's metadata (main.rs:103-106): the <topic>-<n> directories found
    std::vector<int> present;
    for (auto &kv : segs) present.push_back(kv.first);
    const int rc = print_report(h, topic, present, start_offsets, end_offsets, alive, hll, secs);
    kta_destroy(h);
    return rc;
}

int main(int argc, char **argv) {
    std::string topic, bootstrap, librdkafka, synthetic, log_dir, feed = "batch";
    int count_alive_occurrences = 0, hll = 0;
    for (int i = 1; i < argc; i++) {
        const std::string a = argv[i];
        auto val = [&]() -> std::string { if (i + 1 >= argc) { fprintf(stderr, "error: %s needs a value\n", a.c_str()); exit(2); } return argv[++i]; };
        if (a == "-t" || a == "--topic") topic = val();
        else if (a == "-b" || a == "--bootstrap-server") bootstrap = val();
        else if (a == "--librdkafka") librdkafka = val();
        else if (a == "-c" || a == "--count-alive-keys") count_alive_occurrences++;
        else if (a == "-cc") count_alive_occurrences += 2;
        else if (a == "--synthetic") synthetic = val();
        else if (a == "--log-dir") log_dir = val();
        else if (a == "--feed") feed = val();
        else if (a == "--hll") hll = atoi(val().c_str());
        else if (a == "-V" || a == "--version") { puts("Kafka Topic Analyzer 0.4.1"); return 0; }  // main.rs:35
        else if (a == "-h" || a == "--help") {
            puts("Kafka Topic Analyzer 0.4.1\n\nUSAGE:\n    kafka-topic-analyzer [FLAGS] [OPTIONS] --bootstrap-server <BOOTSTRAP_SERVER> --topic <TOPIC>\n\n"
                 "FLAGS:\n    -c, --count-alive-keys    Counts the effective number of alive keys in a log compacted topic\n\n"
                 "OPTIONS:\n    -b, --bootstrap-server <BOOTSTRAP_SERVER>    Bootstrap server(s) to work with, comma separated\n"
                 "        --librdkafka <LIBRDKAFKA>                Options to pass into the underlying librdkafka\n"
                 "    -t, --topic <TOPIC>                          The topic to analyze\n"
                 "        --synthetic <k=v,...>                    in-memory synthetic topic (this build has no Kafka client)\n"
                 "        --feed <push|batch|device>               how records are handed to the metric handlers");
            return 0;
        } else { fprintf(stderr, "error: Found argument '%s' which wasn't expected\n", a.c_str()); return 2; }
    }
    if (topic.empty() || bootstrap.empty()) {
        fprintf(stderr, "error: The following required arguments were not provided:\n    --bootstrap-server <BOOTSTRAP_SERVER>\n    --topic <TOPIC>\n");
        return 2;
    }
    if (synthetic.empty() && log_dir.empty()) {
        fprintf(stderr, "Error fetching metadata: this build has no librdkafka client (no broker access); pass --log-dir DIR or --synthetic n=...,partitions=...\n");
        return 101;  // the reference panics here (src/kafka.rs:61)
    }
    const auto start_time = std::chrono::steady_clock::now();  // main.rs:69
    if (!log_dir.empty()) return analyze_log_dir(topic, log_dir, count_alive_occurrences == 1, hll, start_time);

    std::map<std::string, std::string> kv;
    for (size_t p = 0; p < synthetic.size();) {
        size_t e = synthetic.find(',', p);
        if (e == std::string::npos) e = synthetic.size();
        const std::string item = synthetic.substr(p, e - p);
        const size_t q = item.find('=');
        if (q != std::string::npos) kv[item.substr(0, q)] = item.substr(q + 1);
        p = e + 1;
    }
    auto geti = [&](const char *k, long long d) { return kv.count(k) ? atoll(kv[k].c_str()) : d; };
    kta_synth_spec spec{};
    spec.seed = (uint64_t)geti("seed", 0x4B544131);
    spec.num_partitions = (int32_t)geti("partitions", 4);
    spec.run_len = (int32_t)geti("run_len", 1);
    spec.n_total = geti("n", 100000);
    spec.n_total -= spec.n_total % ((int64_t)spec.num_partitions * spec.run_len);
    spec.distinct_keys = (uint64_t)geti("distinct_keys", spec.n_total / 10 > spec.num_partitions ? spec.n_total / 10 : spec.num_partitions);
    spec.key_mode = (int32_t)geti("key_mode", 0) | (geti("zipf_keys", 0) ? KTA_SYNTH_KEYS_LOGUNIFORM : 0) |
                    (geti("geometric_values", 0) ? KTA_SYNTH_VALUES_GEOMETRIC : 0);
    spec.value_mean = (int32_t)geti("value_mean", 256);
    spec.null_key_per_10k = (int32_t)geti("null_key_per_10k", 100);
    spec.tombstone_per_10k = (int32_t)geti("tombstone_per_10k", 500);
    spec.ts_missing_per_10k = (int32_t)geti("ts_missing_per_10k", 0);
    spec.empty_value_per_10k = (int32_t)geti("empty_value_per_10k", 0);
    const int P = spec.num_partitions;
    const int64_t n = spec.n_total;

    // get_topic_offsets (src/kafka.rs:60-72): synthetic watermarks
    std::vector<int64_t> start_offsets(P, 0), end_offsets(P, n / P);
    if (n == 0) { fprintf(stderr, "Given topic has no content, no analysis possible. Exiting.\n"); return 254; }  // main.rs:98-101

    kta_config cfg{};
    cfg.struct_size = sizeof cfg;
    cfg.device = -1;
    cfg.num_partitions = P;
    cfg.count_alive_keys = count_alive_occurrences == 1 ? 1 : 0;  // occurrences_of == 1, main.rs:77-80
    cfg.hll_precision = hll;
    cfg.now_s = INT64_MIN;
    kta_handle *h = nullptr;
    KTA(kta_create(&cfg, &h));

    printf("Subscribing to %s\n", topic.c_str());          // src/kafka.rs:88
    printf("Starting message consumption...\n");            // src/kafka.rs:91
    const int64_t CH = 1 << 20;
    double feed_s = 0;   // time spent inside the library's entry points only (not in the synthetic generator)
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    if (feed == "device") {
        const int64_t ntiles = (n + KTA_KEY_TILE - 1) / KTA_KEY_TILE;
        int32_t *dp, *dk, *dv; int64_t *dt; uint8_t *dkb; uint64_t *dtb;
        const int64_t cap = n * 40 + 64;
        if (cudaMalloc((void **)&dp, n * 4) || cudaMalloc((void **)&dk, n * 4) || cudaMalloc((void **)&dv, n * 4) || cudaMalloc((void **)&dt, n * 8) ||
            cudaMalloc((void **)&dkb, cap) || cudaMalloc((void **)&dtb, (ntiles + 1) * 8)) { fprintf(stderr, "cudaMalloc failed\n"); return 1; }
        int64_t kbl = 0;
        if (kta_synth_fill_device(&spec, -1, 0, 1, 0, n, dp, nullptr, dt, dk, dv, nullptr, dkb, cap, dtb, &kbl)) { fprintf(stderr, "synthetic fill failed\n"); return 1; }
        kta_batch b{};
        b.n = n; b.partition = dp; b.ts_ms = dt; b.key_len = dk; b.value_len = dv; b.key_bytes = dkb; b.key_bytes_len = kbl; b.key_tile_base = dtb;
        const double t0 = now();
        KTA(kta_scan_batch_device(h, &b));
        KTA(kta_sync(h));
        feed_s += now() - t0;
    } else {
        if (feed == "push") {
            // the pinned landing ring (3 chunks, ~0.5 GB) is allocated by the first push: do that outside the timed feed —
            // a real run amortises it over the whole topic, a 2e7-record measurement would be dominated by it
            KTA(kta_push(h, 0, 0, 0, nullptr, -1, 0));
            KTA(kta_sync(h));
            KTA(kta_reset(h));
        }
        std::vector<int32_t> part(CH), kl(CH), vl(CH);
        std::vector<int64_t> off(CH), ts(CH);
        std::vector<uint8_t> kb((size_t)CH * 40 + 16);
        for (int64_t s0 = 0; s0 < n; s0 += CH) {
            const int64_t c = std::min(CH, n - s0);
            int64_t kbl = 0;
            if (kta_synth_fill_host(&spec, 0, 1, s0, c, part.data(), off.data(), ts.data(), kl.data(), vl.data(), nullptr,
                                    kb.data(), (int64_t)kb.size(), &kbl)) { fprintf(stderr, "synthetic fill failed\n"); return 1; }
            const double t0 = now();
            if (feed == "push") {
                // the reference's shape: one handle_message per polled message (src/kafka.rs:107-109)
                int64_t ko = 0;
                for (int64_t i = 0; i < c; i++) {
                    KTA(kta_push(h, part[i], off[i], ts[i], kl[i] > 0 ? kb.data() + ko : (kl[i] == 0 ? kb.data() : nullptr), kl[i], vl[i]));
                    if (kl[i] > 0) ko += kl[i];
                }
            } else {
                kta_batch b{};
                b.n = c; b.seq_base = (uint64_t)s0; b.partition = part.data(); b.offset = off.data(); b.ts_ms = ts.data();
                b.key_len = kl.data(); b.value_len = vl.data(); b.key_bytes = kb.data(); b.key_bytes_len = kbl;
                KTA(kta_push_batch_host(h, &b));
            }
            feed_s += now() - t0;
        }
    }
    {
        const double t0 = now();
        finalize_or_warn(h);
        feed_s += now() - t0;
    }
    fprintf(stderr, "[kta] feed=%s: %lld records through the handlers in %.4f s = %.3e msg/s (generator excluded)\n", feed.c_str(),
            (long long)n, feed_s, feed_s > 0 ? (double)n / feed_s : 0.0);
    const uint64_t duration_secs = (uint64_t)std::chrono::duration_cast<std::chrono::seconds>(std::chrono::steady_clock::now() - start_time).count();

    std::vector<int> all_partitions(P);
    for (int p = 0; p < P; p++) all_partitions[p] = p;
    const int rc = print_report(h, topic, all_partitions, start_offsets, end_offsets, cfg.count_alive_keys == 1, hll, duration_secs);
    kta_destroy(h);
    return rc;
}

static int print_report(kta_handle *h, const std::string &topic, const std::vector<int> &partitions, const std::vector<int64_t> &start_offsets,
                        const std::vector<int64_t> &end_offsets, bool alive, int hll, uint64_t duration_secs) {
    kta_report::Summary s{};
    s.topic = topic;
    s.duration_secs = duration_secs;
    KTA(kta_global(h, KTA_OVERALL_COUNT, &s.overall_count));
    KTA(kta_timestamps(h, &s.earliest_s, &s.earliest_ns, &s.latest_s));
    KTA(kta_global(h, KTA_LARGEST_MESSAGE, &s.largest_message));
    KTA(kta_global(h, KTA_SMALLEST_MESSAGE, &s.smallest_message));
    KTA(kta_global(h, KTA_OVERALL_SIZE, &s.overall_size));
    s.has_alive_keys = alive;
    if (s.has_alive_keys) KTA(kta_alive_keys(h, &s.alive_keys));
    std::vector<kta_report::PartitionRow> rows;
    for (int p : partitions) {  // partitions of the metadata, sorted ascending, main.rs:103-106
        kta_report::PartitionRow r{};
        r.partition = p; r.start_offset = start_offsets[p]; r.end_offset = end_offsets[p];
        KTA(kta_counter(h, KTA_TOTAL, p, &r.total)); KTA(kta_counter(h, KTA_ALIVE, p, &r.alive));
        KTA(kta_counter(h, KTA_TOMBSTONES, p, &r.tombstones)); KTA(kta_dirty_ratio(h, p, &r.dirty_ratio));
        KTA(kta_counter(h, KTA_KEY_NULL, p, &r.key_null)); KTA(kta_counter(h, KTA_KEY_NON_NULL, p, &r.key_non_null));
        KTA(kta_counter(h, KTA_KEY_SIZE_SUM, p, &r.key_size_sum)); KTA(kta_counter(h, KTA_VALUE_SIZE_SUM, p, &r.value_size_sum));
        // the reference panics ("attempt to divide by zero") when sum > 0 && alive == 0 (metric.rs:132-157)
        int rc = kta_avg(h, KTA_KEY_SIZE_AVG, p, &r.key_size_avg);
        if (rc == KTA_OK) rc = kta_avg(h, KTA_VALUE_SIZE_AVG, p, &r.value_size_avg);
        if (rc == KTA_OK) rc = kta_avg(h, KTA_MESSAGE_SIZE_AVG, p, &r.message_size_avg);
        if (rc == KTA_ERR_DIV_BY_ZERO) { fprintf(stderr, "thread 'main' panicked at 'attempt to divide by zero', src/metric.rs\n"); return 101; }
        if (rc != KTA_OK) die("kta_avg");
        rows.push_back(r);
    }
    fputs(kta_report::render(s, rows).c_str(), stdout);
    if (hll) { double e = 0; KTA(kta_alive_keys_hll(h, &e)); printf("| extension: HyperLogLog(p=%d) alive-key estimate: %.0f\n", hll, e); }
    return 0;
}
