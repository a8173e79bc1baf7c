"""Throughput of the GPU RecordBatch v2 decoder (SURVEY.md §8 f2) on the synthetic topic stored broker-style.
Segments are encoded on the host (C++), staged to HBM once, then decoded + scanned from device memory."""
import ctypes as C, os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import kafka_topic_analyzer_b200 as kta
from kafka_topic_analyzer_b200 import synth
from kafka_topic_analyzer_b200._native import lib, check

P, N, VM = 16, 8_000_000, int(sys.argv[1]) if len(sys.argv) > 1 else 256
BR = int(sys.argv[2]) if len(sys.argv) > 2 else 56   # ~16 KB batches (the producer default batch.size) at 256 B values
CODEC = sys.argv[3] if len(sys.argv) > 3 else None   # gzip | lz4 | snappy | zstd: every batch's records section compressed (zlib / pyarrow) on the host
if CODEC:
    N = 2_000_000


def compress_segment(seg: np.ndarray, codec: str) -> np.ndarray:
    """re-writes every batch of an uncompressed segment with its records section compressed"""
    import pyarrow as pa
    raw, out, pos = seg.tobytes(), bytearray(), 0
    while pos + 61 <= len(raw):
        bl = int.from_bytes(raw[pos + 8:pos + 12], "big", signed=True)
        hdr = bytearray(raw[pos:pos + 61])
        if codec == "gzip":
            import zlib
            c = zlib.compressobj(6, zlib.DEFLATED, 31)
            body = c.compress(raw[pos + 61:pos + 12 + bl]) + c.flush()
        elif codec == "zstd":   # level 3, librdkafka's default
            body = pa.Codec("zstd", compression_level=3).compress(raw[pos + 61:pos + 12 + bl], asbytes=True)
        else:
            body = pa.compress(raw[pos + 61:pos + 12 + bl], codec=codec, asbytes=True)
        hdr[8:12] = (49 + len(body)).to_bytes(4, "big")
        hdr[22] |= {"gzip": 1, "snappy": 2, "lz4": 3, "zstd": 4}[codec]
        out += hdr + body
        pos += 12 + bl
    return np.frombuffer(bytes(out), dtype=np.uint8)

spec = synth.make_spec(N, P, value_mean=VM, distinct_keys=1_000_000)
chunks, offs, parts = [], [], []
t0 = time.time()
total = 0
for p in range(P):
    s = synth.encode_segment(spec, p, batch_records=BR)
    unc = int(s.size)
    if CODEC:
        s = compress_segment(s, CODEC)
    pos = 0
    while pos + 61 <= s.size:      # batch offsets by hopping headers on the host
        offs.append(total + pos)
        parts.append(p)
        pos += 12 + int.from_bytes(s[pos + 8:pos + 12].tobytes(), "big", signed=True)
    chunks.append(s)
    total += (s.size + 15) // 16 * 16
raw = sum(int(s.size) for s in chunks)
buf = torch.zeros(total + 64, dtype=torch.uint8, device="cuda")
at = 0
for s in chunks:
    buf[at:at + s.size] = torch.from_numpy(s).cuda()
    at += (s.size + 15) // 16 * 16
d_off = torch.tensor(offs, dtype=torch.int64).cuda()
d_part = torch.tensor(parts, dtype=torch.int32).cuda()
print("encoded %d records, %.2f GB raw log%s, %d batches of ~%d KB in %.1f s" % (N, raw / 1e9, " (%s-compressed)" % CODEC if CODEC else "", len(offs), raw // len(offs) // 1024, time.time() - t0), flush=True)
for mode, kw in (("counters", {}), ("fused HLL", dict(hll_precision=14)), ("-c exact", dict(count_alive_keys=True))):
    e = kta.KtaEngine(P, **kw)
    best = 1e9
    for it in range(5):
        e.reset(); e.sync()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        tot = e.scan_log_batches_device(buf, total, d_off, d_part, len(offs))   # all 16 partitions: ONE decode + ONE scan
        e.finalize()
        best = min(best, time.perf_counter() - t0)
    assert tot == N and e.message_metrics.overall_count() == N
    print("%-10s decode+scan %.3f ms  %.2e msg/s  %.0f GB/s of raw log (value mean %d B)" % (mode, best * 1e3, N / best, raw / best / 1e9, VM), flush=True)
    e.close()
