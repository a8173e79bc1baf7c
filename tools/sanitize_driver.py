"""Small end-to-end runs of every scan-kernel mode for compute-sanitizer (tools/sanitize.sh): counters, in-stream HLL,
exact alive keys (table starting far too small, so growth + stamps-only re-runs happen too), ragged keys, a tail tile,
the host ring path and the log-segment decoder.  Each run is checked against the oracle so a 'clean' sanitizer log is the
log of a run that also computed the right answer."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import kafka_topic_analyzer_b200 as kta
from kafka_topic_analyzer_b200 import synth
from parity import assert_parity, oracle_for

NOW = (4102444800, 1)
which = sys.argv[1:] or ["counters", "hll", "exact", "ragged", "ring", "log", "logz"]


def compress_segment(seg, b0=0):
    """every batch of an uncompressed segment re-written with its records section compressed: gzip, LZ4, Snappy, zstd in turn
    (zstd with and without a content size in the frame header)"""
    import zlib
    import pyarrow as pa
    raw, out, pos, b = seg.tobytes(), bytearray(), 0, b0
    while pos + 61 <= len(raw):
        bl = int.from_bytes(raw[pos + 8:pos + 12], "big", signed=True)
        hdr, body = bytearray(raw[pos:pos + 61]), raw[pos + 61:pos + 12 + bl]
        codec = ("gzip", "lz4", "snappy", "zstd", "zstd-nofcs")[b % 5]
        if codec == "gzip":
            c = zlib.compressobj(6, zlib.DEFLATED, 31)
            body = c.compress(body) + c.flush()
        elif codec.startswith("zstd"):
            body = pa.Codec("zstd", compression_level=3).compress(body, asbytes=True)
            if codec == "zstd-nofcs":
                import zstd_codec
                body = zstd_codec.without_fcs(body)
            codec = "zstd"
        else:
            body = pa.compress(body, codec=codec, asbytes=True)
        hdr[8:12] = (49 + len(body)).to_bytes(4, "big")
        hdr[22] |= {"gzip": 1, "snappy": 2, "lz4": 3, "zstd": 4}[codec]
        out += hdr + body
        pos += 12 + bl
        b += 1
    return np.frombuffer(bytes(out), dtype=np.uint8)

P = 8
n = P * 4096 + 0
for name in which:
    key_mode = 2 if name in ("ragged", "ring") else 0
    spec = synth.make_spec(n, P, key_mode=key_mode, distinct_keys=3000, tombstone_per_10k=2500, ts_missing_per_10k=20,
                           run_len=64 if name == "counters" else 1)
    if name in ("log", "logz"):
        host = synth.fill_host(spec)
        o = oracle_for(host, count_alive_keys=True, now=NOW)
        with kta.KtaEngine(P, count_alive_keys=True, hll_precision=10, device=0, now=NOW, alive_table_kib=1) as e:
            per = n // P
            segs = [(p, synth.encode_segment(spec, p, 0, per, batch_records=100)) for p in range(P)]
            if name == "logz":   # gzip / LZ4 / Snappy / zstd batches: the decompressors run first
                segs = [(p, compress_segment(s, p)) for p, s in segs]
            e.push_log_segments(segs)
            e.finalize()
            got = (e.message_metrics.overall_count(), e.alive_keys())
            assert e.alive_keys() == o.scalar("sum_all_alive")
        print(name, "ok", got)
        assert got[0] == n
        continue
    topic = synth.DeviceTopic(spec, device=0, count=n - 37)     # a ragged tail tile
    host = topic.to_host()
    exact = name in ("exact", "ragged", "ring")
    with kta.KtaEngine(P, count_alive_keys=exact, hll_precision=0 if name == "counters" else 10, device=0, now=NOW,
                       ring_records=4096, alive_table_kib=1 if exact else 0) as e:
        if name == "ring":
            e.push_batch_host(host.partition, host.ts_ms, host.key_len, host.value_len, host.key_bytes, None)
        else:
            e.scan_batch_device(topic.partition, topic.ts_ms, topic.key_len, topic.value_len, key_bytes=topic.key_bytes,
                                key_bytes_len=topic.key_bytes_len, key_tile_base=topic.key_tile_base)
        e.finalize()
        o = oracle_for(host, count_alive_keys=exact, track_stream=not exact, now=NOW)
        regs = None if name == "counters" else (o.hll_alive_regs(10) if exact else o.hll_stream_regs(10))
        assert_parity(e, o, P, check_alive=exact, hll_regs=regs)
        print(name, "ok", e.stats(), e.alive_table_stats() if exact else "")
