"""zstd records sections for the RecordBatch v2 encoder of kafka_codec.py — TEST INFRASTRUCTURE for the GPU decoder
(kta_zstd.cuh).  The compressor is pyarrow's (libzstd's one-shot API): independent of the decompressor under test.
Batches are encoded uncompressed by kafka_codec and their records section re-written here."""
import kafka_codec as kc

ZSTD_CODECS = ("zstd", "zstd-nofcs")


def without_fcs(frame: bytes, fcs_bytes: int = 0) -> bytes:
    """A one-frame zstd stream with its header rewritten (RFC 8878 3.1.1.1), blocks kept: fcs_bytes=0 drops the
    Frame_Content_Size and states a Window_Descriptor at least the content size; fcs_bytes=8 states the size in an 8-byte
    field instead (single segment)."""
    assert frame[:4] == b"\x28\xb5\x2f\xfd"
    fhd = frame[4]
    single, fcs_flag = (fhd >> 5) & 1, fhd >> 6
    assert fhd & 3 == 0                                  # no dictionary id
    at = 5
    wd = None
    if not single:
        wd = frame[at]
        at += 1
    size_len = {0: single, 1: 2, 2: 4, 3: 8}[fcs_flag]
    fcs = int.from_bytes(frame[at:at + size_len], "little") + (256 if size_len == 2 else 0)
    blocks = frame[at + size_len:]
    if fcs_bytes == 8:
        return frame[:4] + bytes([0xE0 | (fhd & 0x04)]) + fcs.to_bytes(8, "little") + blocks
    if wd is None:                                       # smallest power-of-two window >= the content (>= 1 KiB)
        e = max(0, (max(fcs, 1) - 1).bit_length() - 10)
        wd = e << 3
    return frame[:4] + bytes([fhd & 0x04, wd]) + blocks


def compress_records(recs: bytes, codec: str, level: int = 3) -> bytes:
    """'zstd': what a one-shot compressor writes (a single-segment frame with its content size); 'zstd-nofcs': what
    streaming compressors write (no content size).  Other codecs: kafka_codec's."""
    if codec not in ZSTD_CODECS:
        return kc.compress_records(recs, codec)
    import pyarrow as pa
    frame = pa.Codec("zstd", compression_level=level).compress(recs, asbytes=True)
    return without_fcs(frame) if codec == "zstd-nofcs" else frame


def recompress_batch(batch: bytes, codec, level: int = 3) -> bytes:
    """an uncompressed batch re-written with its records section compressed by `codec` (None: unchanged)"""
    if codec is None:
        return batch
    body = compress_records(batch[61:], codec, level)
    hdr = bytearray(batch[:61])
    hdr[8:12] = (49 + len(body)).to_bytes(4, "big")      # batchLength
    hdr[22] |= 4 if codec in ZSTD_CODECS else kc.CODEC_BITS[codec]
    return bytes(hdr) + body


def encode_batch(base_offset, base_ts, records, attributes=0, max_ts=None, compression=None, level: int = 3):
    """kafka_codec.encode_batch, with the zstd codecs too"""
    return recompress_batch(kc.encode_batch(base_offset, base_ts, records, attributes=attributes, max_ts=max_ts), compression, level)


def split_batches(seg: bytes):
    pos = 0
    while pos + 61 <= len(seg):
        end = pos + 12 + int.from_bytes(seg[pos + 8:pos + 12], "big", signed=True)
        yield seg[pos:end]
        pos = end


def encode_partition(partition_records, rng, max_batch=40, compression=None):
    """kafka_codec.encode_partition, with the zstd codecs too; a list of codecs: every batch picks its own"""
    seg = kc.encode_partition(partition_records, rng, max_batch=max_batch)
    out = bytearray()
    for batch in split_batches(seg):
        codec = compression
        if isinstance(compression, (list, tuple)):
            codec = compression[int(rng.integers(0, len(compression)))]
        out += recompress_batch(batch, codec)
    return bytes(out)
