"""zstd record batches (attributes codec 4) — what producers with compression.type=zstd write and librdkafka built with
libzstd decompresses inside poll (src/kafka.rs:93) — decompressed on the GPU (csrc/kta_zstd.cuh) and scanned, against the
CPU oracle fed the same records message by message."""
import os
import subprocess

import numpy as np
import pytest

from kafka_topic_analyzer_b200 import KtaEngine, KtaError, synth
from parity import assert_parity
from test_logdecode import NOW, _oracle_over, _partition_lists
import kafka_codec as kc
import zstd_codec as zc


def _topic(P, n_per, seed, value_mean=120):
    spec = synth.make_spec(P * n_per, P, key_mode=1, distinct_keys=900, tombstone_per_10k=2000, null_key_per_10k=300,
                           empty_value_per_10k=100, value_mean=value_mean)
    return spec, _partition_lists(synth.fill_host(spec))


@pytest.mark.gpu
@pytest.mark.parametrize("codec", ["zstd", "zstd-nofcs", "mixed"])
def test_zstd_segments_decode_and_scan(codec):
    """with a content size in the frame header (one-shot compressors), without one (streaming compressors: the size pass
    decodes the sequences), and a mix of zstd, gzip, LZ4, Snappy and uncompressed batches in one segment; then all partitions
    in one call"""
    rng = np.random.default_rng(31)
    P = 5
    spec, per = _topic(P, 4000, 31)
    o = _oracle_over(per, count_alive_keys=True)
    comp = ["zstd", "zstd-nofcs", "gzip", "lz4", "snappy", "snappy-xerial", None] if codec == "mixed" else codec
    with KtaEngine(P, count_alive_keys=True, hll_precision=10, now=NOW) as e:
        total = raw = comp_bytes = 0
        for p in sorted(per):
            seg = zc.encode_partition(per[p], rng, max_batch=200, compression=comp)
            raw += len(kc.encode_partition(per[p], np.random.default_rng(1), max_batch=200))
            comp_bytes += len(seg)
            total += e.push_log_segment(p, seg)
        e.finalize()
        assert total == spec.n_total and comp_bytes < raw            # it really was compressed
        assert_parity(e, o, P, check_alive=True, hll_regs=o.hll_alive_regs(10))
        e.reset()
        rng = np.random.default_rng(32)
        assert e.push_log_segments([(p, zc.encode_partition(per[p], rng, max_batch=64, compression=comp)) for p in sorted(per)]) == spec.n_total
        e.finalize()
        assert_parity(e, o, P, check_alive=True, hll_regs=o.hll_alive_regs(10))


@pytest.mark.gpu
def test_zstd_batches_in_one_device_buffer():
    """kta_scan_log_batches_device over zstd batches of every partition packed back to back in one device buffer"""
    import torch
    rng = np.random.default_rng(41)
    P = 4
    spec, per = _topic(P, 3000, 41)
    o = _oracle_over(per, count_alive_keys=True)
    chunks, offs, parts, total = [], [], [], 0
    for p in sorted(per):
        s = np.frombuffer(zc.encode_partition(per[p], rng, max_batch=100, compression=["zstd", "zstd-nofcs"]), np.uint8)
        pos = 0
        while pos + 61 <= s.size:
            offs.append(total + pos)
            parts.append(p)
            pos += 12 + int.from_bytes(s[pos + 8:pos + 12].tobytes(), "big", signed=True)
        chunks.append(s)
        total += s.size
    buf = torch.from_numpy(np.concatenate(chunks)).cuda()
    d_off = torch.tensor(offs, dtype=torch.int64).cuda()
    d_part = torch.tensor(parts, dtype=torch.int32).cuda()
    with KtaEngine(P, count_alive_keys=True, hll_precision=10, now=NOW) as e:
        assert e.scan_log_batches_device(buf, total, d_off, d_part, len(offs)) == spec.n_total
        e.finalize()
        assert_parity(e, o, P, check_alive=True, hll_regs=o.hll_alive_regs(10))


@pytest.mark.gpu
@pytest.mark.parametrize("nofcs", [False, True])
def test_zstd_batches_of_several_blocks(nofcs):
    """batches of ~350 KB of records at level 19: several 128 KiB blocks per frame, matches across blocks, repeat tables"""
    P = 2
    spec, per = _topic(P, 6000, 51, value_mean=200)
    o = _oracle_over(per, count_alive_keys=True)
    with KtaEngine(P, count_alive_keys=True, hll_precision=10, now=NOW) as e:
        for p in sorted(per):
            seg = bytearray()
            recs = per[p]
            for i in range(0, len(recs), 2000):
                chunk = recs[i:i + 2000]
                base_ts = chunk[0][0] if chunk[0][0] != -1 else 0
                plain = kc.encode_batch(i, base_ts, [(j, r[0] - base_ts, r[1], r[2]) for j, r in enumerate(chunk)])
                assert len(plain) > 2 * 131072                   # three blocks or more
                seg += zc.recompress_batch(plain, "zstd-nofcs" if nofcs else "zstd", level=19)
            assert e.push_log_segment(p, bytes(seg)) == len(recs)
        e.finalize()
        assert_parity(e, o, P, check_alive=True, hll_regs=o.hll_alive_regs(10))


@pytest.mark.gpu
def test_damaged_zstd_batches_are_rejected():
    recs = [(i, i, b"key-%d" % (i % 5), 30) for i in range(50)]
    good = zc.encode_batch(0, 1000, recs, compression="zstd")
    plain = kc.encode_batch(0, 1000, recs)
    with KtaEngine(1, now=NOW) as e:
        assert e.push_log_segment(0, good) == 50
        bad_cases = []
        b = bytearray(good)
        b[61] ^= 0x15                                         # the magic
        bad_cases.append(b)
        b = bytearray(good)
        b[65] |= 0x01                                         # a dictionary id flag
        bad_cases.append(b)
        fcs_at = 66                                           # single segment, 2-byte Frame_Content_Size
        assert good[65] >> 6 == 1 and good[65] >> 5 & 1
        for d in (1, -1):                                     # a forged content size, one byte off either way
            b = bytearray(good)
            b[fcs_at:fcs_at + 2] = (int.from_bytes(good[fcs_at:fcs_at + 2], "little") + d).to_bytes(2, "little")
            bad_cases.append(b)
        cut = bytearray(good[:-7])                            # a shorter section under an adjusted batchLength
        cut[8:12] = (len(cut) - 12).to_bytes(4, "big")
        bad_cases.append(cut)
        b = bytearray(good)
        b[68] |= 0x06                                         # the reserved block type
        bad_cases.append(b)
        b = bytearray(zc.recompress_batch(plain, "zstd"))
        b[57:61] = (len(plain) // 7 + 1).to_bytes(4, "big")   # more records than the uncompressed size can hold
        bad_cases.append(b)
        b = bytearray(plain)
        b[22] |= 5                                            # an unassigned codec
        bad_cases.append(b)
        for b in bad_cases:
            with pytest.raises(KtaError):
                e.push_log_segment(0, bytes(b))
        assert e.push_log_segment(0, good) == 50              # the engine goes on with good batches
        assert e.push_log_segment(0, zc.recompress_batch(plain, "zstd-nofcs")) == 50


@pytest.mark.gpu
def test_cli_log_dir_over_zstd_segments(tmp_path):
    """the C++ CLI's --log-dir over a broker-style directory of zstd segments (with and without content sizes) prints the
    oracle's table"""
    from test_report import CLI_DIR, _build
    _build()
    rng = np.random.default_rng(61)
    P = 3
    spec = synth.make_spec(P * 2000, P, key_mode=1, distinct_keys=300, tombstone_per_10k=3000, value_mean=30)
    per = _partition_lists(synth.fill_host(spec))
    for p, recs in per.items():
        d = tmp_path / ("orders-%d" % p)
        d.mkdir()
        (d / "00000000000000000000.log").write_bytes(zc.encode_partition(recs, rng, compression=["zstd", "zstd-nofcs"]))
    r = subprocess.run([os.path.join(CLI_DIR, "kafka-topic-analyzer"), "-t", "orders", "-b", "unused:9092", "-c", "--log-dir",
                        str(tmp_path)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    o = _oracle_over(per, count_alive_keys=True)
    lines = r.stdout.splitlines()
    assert "Alive keys: %d" % o.scalar("sum_all_alive") in lines
    assert "Topic Size: %d bytes" % o.scalar("overall_size") in lines
    rows = [l for l in lines if l.startswith("| ") and l[2].isdigit()]
    assert len(rows) == P
    for l in rows:
        c = [x.strip() for x in l.strip("|").split("|")]
        p = int(c[0])
        assert (int(c[1]), int(c[2])) == (0, len(per[p]))
        assert [int(c[3]), int(c[4]), int(c[5])] == [o.counter("total", p), o.counter("alive", p), o.counter("tombstones", p)]
        assert [int(c[10]), int(c[11])] == [o.counter("key_size_sum", p), o.counter("value_size_sum", p)]


def test_zstd_sections_roundtrip_on_the_host():
    """the test encoder's zstd sections are what they claim: pyarrow decompresses them, the FCS-less rewrite keeps the blocks"""
    import pyarrow as pa
    recs = b"".join(kc.encode_record(i, i, b"key-%d" % (i % 7), 40 + i % 5) for i in range(300))
    z = zc.compress_records(recs, "zstd")
    assert z[:4] == b"\x28\xb5\x2f\xfd" and len(z) < len(recs)
    assert pa.decompress(z, decompressed_size=len(recs), codec="zstd", asbytes=True) == recs
    n = zc.compress_records(recs, "zstd-nofcs")
    assert n[4] >> 6 == 0 and not n[4] >> 5 & 1 and n[6:] == z[7:]
    b = zc.encode_batch(5, 1000, [(0, 0, b"k", 3)], compression="zstd")
    assert b[22] & 7 == 4 and int.from_bytes(b[8:12], "big") == len(b) - 12
