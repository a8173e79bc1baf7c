// kta_logdecode.cuh — Kafka RecordBatch v2 (magic 2) → SoA columns, on the GPU (SURVEY.md §8 f2).
//
// This is the step BEFORE the metric path: in the reference it happens inside librdkafka's fetch parser, which
// hands one BorrowedMessage per record to the handlers (src/kafka.rs:93,107-109).  Here a whole log segment
// (the concatenated record batches of one partition, exactly what a broker stores in <topic>-<p>/*.log and
// sends in a fetch response) is decoded where it lies in HBM:
//   batch header (61 bytes, big-endian): baseOffset i64 | batchLength i32 | partitionLeaderEpoch i32 | magic i8 |
//     crc u32 | attributes i16 | lastOffsetDelta i32 | baseTimestamp i64 | maxTimestamp i64 | producerId i64 |
//     producerEpoch i16 | baseSequence i32 | recordsCount i32
//   record: length varint | attributes i8 | timestampDelta varlong | offsetDelta varint | keyLength varint | key |
//     valueLength varint | value | headersCount varint | headers…          (varints are zig-zag, LSB group first)
// Semantics kept from the consumer: control batches (attributes bit 5) are not delivered to the application;
// LogAppendTime batches (attributes bit 3) stamp every record with maxTimestamp; a record's timestamp is baseTimestamp +
// timestampDelta as the consumer computes it, and only a RESULT of -1 means "not available"; key/value length -1 means
// null.  CRCs are not verified (librdkafka's default check.crcs=false).
// Compression (attributes bits 0-2, librdkafka decompresses inside poll, src/kafka.rs:93): gzip (kta_inflate.cuh), LZ4 (frame
// format), Snappy (raw or xerial-framed) and zstd (kta_zstd.cuh) batches are decompressed on the GPU into a scratch buffer and
// then decoded like the others; codes 5-7 are rejected.
// Not handled: records of aborted transactions are delivered (a read_committed consumer would filter them through the
// .txnindex / abort markers), legacy magic 0/1 message sets are flagged as malformed.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "kta_inflate.cuh"

namespace kta {

constexpr int LOG_HEADER_BYTES = 61;
// LOGB_COMPRESSED: an unknown codec (attributes codes 5-7).  LOGB_LZ4 / LOGB_SNAPPY / LOGB_GZIP / LOGB_ZSTD: the records section
// must be decompressed first (log_unc_size_kernel, log_zstd_size_kernel + log_decompress_kernel turn such a batch into LOGB_OK).
enum LogBatchFlags { LOGB_OK = 0, LOGB_SKIP_CONTROL = 1, LOGB_BAD = 2, LOGB_COMPRESSED = 4, LOGB_LZ4 = 8, LOGB_SNAPPY = 16, LOGB_GZIP = 32,
                     LOGB_ZSTD = 64 };
constexpr uint32_t LOGB_CODECS = LOGB_LZ4 | LOGB_SNAPPY | LOGB_GZIP | LOGB_ZSTD;   // batches log_decompress_kernel turns into LOGB_OK

__device__ __forceinline__ uint64_t be_u64(const uint8_t *p) {
    uint64_t v = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) v = (v << 8) | __ldg(p + i);
    return v;
}
__device__ __forceinline__ uint32_t be_u32(const uint8_t *p) {
    return ((uint32_t)__ldg(p) << 24) | ((uint32_t)__ldg(p + 1) << 16) | ((uint32_t)__ldg(p + 2) << 8) | __ldg(p + 3);
}
__device__ __forceinline__ uint32_t be_u16(const uint8_t *p) { return ((uint32_t)__ldg(p) << 8) | __ldg(p + 1); }

__device__ __forceinline__ int64_t unzigzag(uint64_t u) { return (int64_t)(u >> 1) ^ -(int64_t)(u & 1); }

struct LogBatchInfo {      // one per record batch, filled by log_header_kernel
    uint64_t off;          // byte offset of the batch in the segment buffer
    uint32_t len;          // 12 + batchLength
    uint32_t flags;        // LogBatchFlags
    int32_t partition;
    int32_t records;       // records delivered to the handlers (0 for skipped batches)
    int64_t base_offset, base_ts, max_ts;
    uint32_t log_append_time;
    uint32_t pad;
};

// thread per batch: validate + read the header
__global__ void log_header_kernel(const uint8_t *bytes, int64_t nbytes, const uint64_t *batch_off, int64_t nbatches,
                                  int32_t partition, const int32_t *batch_partition /* per batch, or NULL = `partition` */,
                                  LogBatchInfo *info, uint64_t *rec_count /*[nbatches+1], [b+1]*/, uint32_t *error_flags) {
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nbatches; b += (int64_t)gridDim.x * blockDim.x) {
        LogBatchInfo bi{};
        bi.off = batch_off[b];
        bi.partition = batch_partition ? batch_partition[b] : partition;
        bi.flags = LOGB_BAD;
        if (bi.off + LOG_HEADER_BYTES <= (uint64_t)nbytes) {
            const uint8_t *p = bytes + bi.off;
            const int32_t batch_len = (int32_t)be_u32(p + 8);
            const int magic = (int8_t)__ldg(p + 16);
            const uint32_t attrs = be_u16(p + 21);
            const int32_t count = (int32_t)be_u32(p + 57);
            // recordsCount sizes the output columns, so it must be plausible before anything is allocated for it: the
            // smallest record is 7 bytes (length, attributes, two deltas, key length, value length, header count)
            const uint32_t codec = attrs & 0x7u;
            // (for a compressed batch the 7-bytes-per-record bound is checked against the uncompressed size later)
            if (magic == 2 && batch_len >= LOG_HEADER_BYTES - 12 && bi.off + 12 + (uint64_t)batch_len <= (uint64_t)nbytes && count >= 0 &&
                (codec != 0 || (uint64_t)count * 7u + (uint64_t)(LOG_HEADER_BYTES - 12) <= (uint64_t)batch_len)) {
                bi.len = 12u + (uint32_t)batch_len;
                bi.base_offset = (int64_t)be_u64(p);
                bi.base_ts = (int64_t)be_u64(p + 27);
                bi.max_ts = (int64_t)be_u64(p + 35);
                bi.log_append_time = (attrs >> 3) & 1u;
                if (attrs & 0x20u) bi.flags = LOGB_SKIP_CONTROL;
                else if (codec <= 4) {
                    bi.flags = codec == 0 ? LOGB_OK : codec == 1 ? LOGB_GZIP : codec == 2 ? LOGB_SNAPPY : codec == 3 ? LOGB_LZ4 : LOGB_ZSTD;
                    bi.records = count;
                } else bi.flags = LOGB_COMPRESSED;   // unassigned codes
            }
        }
        if (bi.flags & (LOGB_BAD | LOGB_COMPRESSED | LOGB_CODECS)) atomicOr(error_flags, bi.flags);
        else if (bi.flags == LOGB_OK) atomicMax(error_flags + 1, bi.len);   // [1]: the longest batch (sizes the decode stage)
        info[b] = bi;
        rec_count[b + 1] = (uint64_t)bi.records;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) rec_count[0] = 0;
}

// unsigned LEB128 at p (bounded by end); returns bytes consumed, 0 on malformed input.  Generic byte loads: the batch may
// sit in shared memory or in global memory.
__host__ __device__ __forceinline__ int uvarint_g(const uint8_t *p, const uint8_t *end, uint64_t &out) {
    uint64_t v = 0;
    int shift = 0, n = 0;
    while (p + n < end && n < 10) {
        const uint8_t b = p[n];
        n++;
        v |= (uint64_t)(b & 0x7f) << shift;
        if (!(b & 0x80)) {
            out = v;
            return n;
        }
        shift += 7;
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Decompression of the records section (everything behind the 61-byte header) of LZ4 and Snappy batches.
//   LZ4: the frame format (magic 0x184D2204 | FLG | BD | [content size] | [dict id] | HC | blocks… | EndMark | [checksum]);
//        a block is a u32 LE size (top bit = stored uncompressed) + data [+ block checksum]; block data = sequences of
//        token | literal length… | literals | offset u16 | match length… ; matches may reach back into earlier blocks.
//   Snappy: raw (uvarint uncompressed length, then elements: literal / copy with 1-, 2-, 4-byte offset) or the xerial
//        framing Java clients write ("\x82SNAPPY\0", two version words, then chunks of u32 BE length + raw snappy).
// A "walk" goes through the elements once; with out == nullptr it only adds up the output size.  One lane parses, all 32
// lanes of the warp copy (a match that overlaps itself repeats with period `offset`, so every byte's source is known up
// front: out[op + i] = out[op - offset + i % offset]).
// ------------------------------------------------------------------------------------------------
struct LzWalk {
    uint64_t out_len;   // bytes produced
    bool ok;
};

// (the walks are __host__ __device__ like kta_inflate.cuh: tests/test_lzwalk_host.py runs them on the host, where the
// "warp" is one lane; the product calls them on the device only)
template <bool COPY>
__host__ __device__ __forceinline__ void lz_emit_literals(uint8_t *out, uint64_t op, const uint8_t *in, uint32_t n, int lane) {
    if (COPY) for (uint32_t i = lane; i < n; i += KTA_INF_LANES) out[op + i] = in[i];
}
template <bool COPY>
__host__ __device__ __forceinline__ void lz_emit_match(uint8_t *out, uint64_t op, uint32_t offset, uint32_t n, int lane) {
    if (COPY) {
        KTA_INF_SYNC();   // the bytes the match refers to have been written
        for (uint32_t i = lane; i < n; i += KTA_INF_LANES) out[op + i] = out[op - offset + (i % offset)];
        KTA_INF_SYNC();
    }
}

// LZ4 frame at in[0, n).  COPY: the whole warp calls this (lane-uniform control flow: every lane parses the same bytes).
template <bool COPY>
__host__ __device__ LzWalk lz4_frame_walk(const uint8_t *in, uint32_t n, uint8_t *out, uint64_t out_cap, int lane) {
    LzWalk w{0, false};
    if (n < 7 || in[0] != 0x04 || in[1] != 0x22 || in[2] != 0x4D || in[3] != 0x18) return w;
    const uint32_t flg = in[4];
    if ((flg >> 6) != 1) return w;
    uint32_t ip = 6 + ((flg & 0x08) ? 8u : 0u) + ((flg & 0x01) ? 4u : 0u) + 1u;   // FLG, BD, [content size], [dict id], HC
    const bool block_checksum = (flg & 0x10) != 0;
    for (;;) {
        if (ip + 4 > n) return w;
        const uint32_t bs = (uint32_t)in[ip] | ((uint32_t)in[ip + 1] << 8) | ((uint32_t)in[ip + 2] << 16) | ((uint32_t)in[ip + 3] << 24);
        ip += 4;
        if (bs == 0) break;                                  // EndMark
        const uint32_t blen = bs & 0x7fffffffu;
        if (blen > n - ip) return w;
        if (bs & 0x80000000u) {                              // stored block
            if (COPY && w.out_len + blen > out_cap) return w;
            lz_emit_literals<COPY>(out, w.out_len, in + ip, blen, lane);
            w.out_len += blen;
        } else {
            uint32_t p = ip;
            const uint32_t bend = ip + blen;
            while (p < bend) {
                const uint32_t token = in[p++];
                uint32_t lit = token >> 4;
                if (lit == 15) {
                    uint32_t b;
                    do { if (p >= bend) return w; b = in[p++]; lit += b; } while (b == 255);
                }
                if (lit > bend - p) return w;
                if (COPY && w.out_len + lit > out_cap) return w;
                lz_emit_literals<COPY>(out, w.out_len, in + p, lit, lane);
                w.out_len += lit;
                p += lit;
                if (p >= bend) break;                        // the last sequence of a block has no match
                if (p + 2 > bend) return w;
                const uint32_t offset = (uint32_t)in[p] | ((uint32_t)in[p + 1] << 8);
                p += 2;
                uint32_t ml = (token & 15u) + 4u;
                if ((token & 15u) == 15u) {
                    uint32_t b;
                    do { if (p >= bend) return w; b = in[p++]; ml += b; } while (b == 255);
                }
                if (offset == 0 || offset > w.out_len) return w;
                if (COPY && w.out_len + ml > out_cap) return w;
                lz_emit_match<COPY>(out, w.out_len, offset, ml, lane);
                w.out_len += ml;
            }
        }
        ip += blen + (block_checksum ? 4u : 0u);
    }
    w.ok = true;
    return w;
}

// one raw Snappy block at in[0, n)
template <bool COPY>
__host__ __device__ bool snappy_raw_walk(const uint8_t *in, uint32_t n, uint8_t *out, uint64_t out_cap, uint64_t &op, int lane) {
    uint64_t want;
    const int hn = uvarint_g(in, in + n, want);
    if (hn <= 0) return false;
    const uint64_t start = op;
    uint32_t p = (uint32_t)hn;
    while (p < n) {
        const uint32_t tag = in[p++];
        if ((tag & 3u) == 0) {                               // literal
            uint32_t len = (tag >> 2) + 1u;
            if (len > 60) {
                const uint32_t nb = len - 60;                // 1..4 length bytes follow
                if (p + nb > n) return false;
                len = 0;
                for (uint32_t i = 0; i < nb; i++) len |= (uint32_t)in[p + i] << (8 * i);
                len += 1u;
                p += nb;
            }
            if (len > n - p) return false;
            if (COPY && op + len > out_cap) return false;
            lz_emit_literals<COPY>(out, op, in + p, len, lane);
            op += len;
            p += len;
        } else {
            uint32_t len, offset;
            if ((tag & 3u) == 1) {
                if (p + 1 > n) return false;
                len = ((tag >> 2) & 7u) + 4u;
                offset = ((tag >> 5) << 8) | in[p];
                p += 1;
            } else if ((tag & 3u) == 2) {
                if (p + 2 > n) return false;
                len = (tag >> 2) + 1u;
                offset = (uint32_t)in[p] | ((uint32_t)in[p + 1] << 8);
                p += 2;
            } else {
                if (p + 4 > n) return false;
                len = (tag >> 2) + 1u;
                offset = (uint32_t)in[p] | ((uint32_t)in[p + 1] << 8) | ((uint32_t)in[p + 2] << 16) | ((uint32_t)in[p + 3] << 24);
                p += 4;
            }
            if (offset == 0 || offset > op - start) return false;
            if (COPY && op + len > out_cap) return false;
            lz_emit_match<COPY>(out, op, offset, len, lane);
            op += len;
        }
    }
    return op - start == want;
}

template <bool COPY>
__host__ __device__ LzWalk snappy_walk(const uint8_t *in, uint32_t n, uint8_t *out, uint64_t out_cap, int lane) {
    LzWalk w{0, false};
    const bool xerial = n >= 16 && in[0] == 0x82 && in[1] == 'S' && in[2] == 'N' && in[3] == 'A' && in[4] == 'P' && in[5] == 'P' &&
                        in[6] == 'Y' && in[7] == 0;
    if (!xerial) {
        w.ok = snappy_raw_walk<COPY>(in, n, out, out_cap, w.out_len, lane);
        return w;
    }
    uint32_t p = 16;                                         // magic (8) + version (4) + compatible version (4)
    while (p < n) {
        if (p + 4 > n) return w;
        const uint32_t cl = ((uint32_t)in[p] << 24) | ((uint32_t)in[p + 1] << 16) | ((uint32_t)in[p + 2] << 8) | in[p + 3];
        p += 4;
        if (cl > n - p) return w;
        if (!snappy_raw_walk<COPY>(in + p, cl, out, out_cap, w.out_len, lane)) return w;
        p += cl;
    }
    w.ok = true;
    return w;
}

}  // namespace kta
#include "kta_zstd.cuh"   // zstd_walk: built on LzWalk and the copy helpers above
namespace kta {

// gzip: one member (what producers write: the records section is one gzip stream).  The size pass trusts ISIZE; the copy
// pass is bounded by it and must produce exactly that many bytes.  The CRC32 of the trailer is not verified (like the batch
// CRC: check.crcs=false).
struct InfWarpOut {
    uint8_t *out;
    uint64_t op, cap;
    int lane;
    __device__ bool lit(uint8_t b) {
        if (op >= cap) return false;
        if (lane == 0) out[op] = b;
        op++;
        return true;
    }
    __device__ bool match(uint32_t dist, uint32_t len) {
        if (dist > op || op + len > cap) return false;
        lz_emit_match<true>(out, op, dist, len, lane);   // syncs the warp first: lane 0's literals are visible
        op += len;
        return true;
    }
    __device__ bool stored(const uint8_t *src, uint32_t len) {
        if (op + len > cap) return false;
        lz_emit_literals<true>(out, op, src, len, lane);
        op += len;
        return true;
    }
};
__device__ inline LzWalk gzip_walk(const uint8_t *in, uint32_t n, uint8_t *out, uint64_t out_cap, InfWork &work, int lane) {
    LzWalk w{0, false};
    const uint32_t hl = gzip_header_len(in, n);
    if (!hl) return w;
    InfBits s{in + hl, n - hl - 8u, 0u, 0ull, 0, false};
    InfWarpOut o{out, 0, out_cap, lane};
    const bool ok = inf_stream(s, o, work, lane);
    w.out_len = o.op;
    w.ok = ok && o.op == (uint64_t)gzip_isize(in, n);
    return w;
}

// thread per batch: the uncompressed size of a compressed batch's records section → slot[b + 1] = bytes its uncompressed
// image (header + records, rounded up to 16) needs in the scratch buffer (0 for batches that are not compressed; zstd
// batches are sized by log_zstd_size_kernel afterwards)
__global__ void log_unc_size_kernel(const uint8_t *bytes, const LogBatchInfo *info, int64_t nbatches, uint64_t *slot, uint32_t *error_flags) {
    for (int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; b < nbatches; b += (int64_t)gridDim.x * blockDim.x) {
        const LogBatchInfo bi = info[b];
        uint64_t need = 0;
        if (bi.flags & (LOGB_CODECS & ~LOGB_ZSTD)) {
            const uint8_t *in = bytes + bi.off + LOG_HEADER_BYTES;
            const uint32_t n = bi.len - LOG_HEADER_BYTES;
            LzWalk w{0, false};
            if (bi.flags == LOGB_GZIP) {
                // ISIZE is taken on trust here (the copy pass must then produce exactly that much), but not beyond what
                // DEFLATE can expand to (1032 : 1): a forged trailer must not size the scratch buffer
                if (gzip_header_len(in, n) && (uint64_t)gzip_isize(in, n) <= (uint64_t)n * 1032u + 64u) w = LzWalk{gzip_isize(in, n), true};
            } else w = bi.flags == LOGB_LZ4 ? lz4_frame_walk<false>(in, n, nullptr, 0, 0) : snappy_walk<false>(in, n, nullptr, 0, 0);
            // recordsCount sizes the output columns: it must be plausible for the uncompressed size (7 bytes per record at least)
            if (!w.ok || w.out_len > 0x7fffff00ull || (uint64_t)bi.records * 7u > w.out_len) atomicOr(error_flags, (uint32_t)LOGB_BAD);
            else need = ((uint64_t)LOG_HEADER_BYTES + w.out_len + 15u) & ~15ull;
        }
        slot[b + 1] = need;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) slot[0] = 0;
}

// warp per zstd batch (the sequence tables live in shared memory), after log_unc_size_kernel: slot[b + 1] as there.  A frame
// that states its content size is taken at that size within what its blocks can hold (the copy pass must then produce
// exactly that much); a frame without one is walked: literal section sizes plus decoded match lengths, no copies.
__global__ void __launch_bounds__(128) log_zstd_size_kernel(const uint8_t *bytes, const LogBatchInfo *info, int64_t nbatches, uint64_t *slot,
                                                            uint32_t *error_flags) {
    __shared__ ZstdWork zstd_work[4];
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, gs = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = gw; b < nbatches; b += gs) {
        const LogBatchInfo bi = info[b];
        if (bi.flags != LOGB_ZSTD) continue;
        const LzWalk w = zstd_walk<false>(bytes + bi.off + LOG_HEADER_BYTES, bi.len - LOG_HEADER_BYTES, nullptr, 0, zstd_work[threadIdx.x >> 5],
                                          lane, true);
        if (lane == 0) {
            uint64_t need = 0;
            if (!w.ok || w.out_len > 0x7fffff00ull || (uint64_t)bi.records * 7u > w.out_len) atomicOr(error_flags, (uint32_t)LOGB_BAD);
            else need = ((uint64_t)LOG_HEADER_BYTES + w.out_len + 15u) & ~15ull;
            slot[b + 1] = need;
        }
    }
}

// warp per compressed batch: header copy (compression bits cleared, batchLength = uncompressed) + decompressed records into
// scratch + slot[b]; the batch's info then points there (offsets are relative to `bytes`: the scratch buffer is simply
// another place in the same address space) and it is an ordinary LOGB_OK batch for the decoder.
// ZSTD: the zstd batches, with their larger tables (ZstdWork) in shared memory; otherwise the LZ4 / Snappy / gzip batches, so
// that those keep the registers and shared memory of a kernel without zstd (twice the blocks per SM, measured 1.5x the rate).
template <bool ZSTD>
__global__ void __launch_bounds__(128) log_decompress_kernel(const uint8_t *bytes, LogBatchInfo *info, int64_t nbatches, const uint64_t *slot,
                                                             uint8_t *scratch, uint32_t *error_flags) {
    using Work = typename std::conditional<ZSTD, ZstdWork, InfWork>::type;
    __shared__ Work work[4];   // Huffman / FSE tables of the warp's gzip or zstd batch
    const int lane = threadIdx.x & 31;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, gs = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = gw; b < nbatches; b += gs) {
        const LogBatchInfo bi = info[b];
        if (ZSTD ? bi.flags != LOGB_ZSTD : !(bi.flags & (LOGB_CODECS & ~LOGB_ZSTD))) continue;
        const uint64_t need = slot[b + 1] - slot[b];
        uint8_t *dst = scratch + slot[b];
        if (need < (uint64_t)LOG_HEADER_BYTES) {             // the size pass rejected it
            if (lane == 0) info[b].flags = LOGB_BAD;
            continue;
        }
        const uint8_t *src = bytes + bi.off;
        const uint64_t cap = need - LOG_HEADER_BYTES;
        const uint8_t *in = src + LOG_HEADER_BYTES;
        const uint32_t n = bi.len - LOG_HEADER_BYTES;
        uint8_t *out = dst + LOG_HEADER_BYTES;
        LzWalk w;
        if constexpr (ZSTD) {
            // the records section must come out at exactly the size pass's length (the slot is that, rounded up to 16)
            w = zstd_walk<true>(in, n, out, cap, work[threadIdx.x >> 5], lane);
            w.ok = w.ok && ((LOG_HEADER_BYTES + w.out_len + 15u) & ~15ull) == need;
        } else {
            w = bi.flags == LOGB_LZ4    ? lz4_frame_walk<true>(in, n, out, cap, lane)
              : bi.flags == LOGB_GZIP ? gzip_walk(in, n, out, cap, work[threadIdx.x >> 5], lane)
                                      : snappy_walk<true>(in, n, out, cap, lane);
        }
        for (int i = lane; i < LOG_HEADER_BYTES; i += 32) dst[i] = src[i];
        __syncwarp();
        if (lane == 0) {
            const uint32_t ulen = LOG_HEADER_BYTES + (uint32_t)w.out_len, bl = ulen - 12u;
            dst[8] = (uint8_t)(bl >> 24); dst[9] = (uint8_t)(bl >> 16); dst[10] = (uint8_t)(bl >> 8); dst[11] = (uint8_t)bl;   // batchLength
            dst[22] &= 0xf8;                                  // attributes: no compression
            if (!w.ok) atomicOr(error_flags, (uint32_t)LOGB_BAD);
            info[b].off = (uint64_t)(dst - bytes);            // relative to `bytes` (may wrap: one address space)
            info[b].len = ulen;
            info[b].flags = w.ok ? LOGB_OK : LOGB_BAD;
        }
    }
}

// One WARP per batch.  Records are length-prefixed, so finding where record i starts is a serial chain: lane 0 hops through
// 32 record-length varints at a time and publishes the 32 start positions; then the 32 lanes parse their records in
// parallel and write the columns coalesced.
// STAGED: the whole batch (what a producer's batch.size bounds: 16 KiB by default) is first brought global→shared by ONE
// bulk async copy per batch per warp (cp.async.bulk → UBLKCP, mbarrier completion), so every hop of the chain is a
// 29-cycle shared-memory read instead of a dependent global access to a new line (measured: the chain of global hops was
// the decoder's bottleneck).  Batches that do not fit the stage, or whose 16-byte-aligned copy would run past the readable
// bytes, are read in place.
// Output: the header columns and, per record, the position of its key bytes in the segment buffer (key_src, only when the
// keys will be hashed) — the keys themselves are packed afterwards by log_gather_keys_kernel, without a second walk.
constexpr int LOG_DECODE_THREADS = 128;
constexpr int LOG_WARP_HEADER = 192;   // per warp: mbarrier (8 B) + 33 record starts (132 B), padded

template <bool STAGED>
__global__ void __launch_bounds__(LOG_DECODE_THREADS) log_decode_kernel(
    const uint8_t *bytes, uint64_t readable /* bytes that may be read from `bytes` */, const LogBatchInfo *info, int64_t nbatches,
    const uint64_t *rec_base, int32_t *partition, int64_t *offset, int64_t *ts_ms, int32_t *key_len, int32_t *value_len,
    uint64_t *key_src, uint32_t stage_bytes /* per warp, multiple of 16 */, uint32_t *error_flags) {
    extern __shared__ __align__(128) unsigned char log_smem[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const unsigned full = 0xffffffffu;
    unsigned char *wsm = log_smem + (size_t)wib * (LOG_WARP_HEADER + (STAGED ? stage_bytes : 0u));
    uint32_t *s_start = reinterpret_cast<uint32_t *>(wsm + 16);
    unsigned char *stage = wsm + LOG_WARP_HEADER;
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(wsm);
    uint32_t phase = 0;
    if (STAGED && lane == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, gs = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t b = gw; b < nbatches; b += gs) {
        const LogBatchInfo bi = info[b];
        if (bi.flags == LOGB_OK && bi.records > 0) {
            const uint8_t *base = bytes + bi.off;
            if (STAGED) {
                const uint32_t lead = (uint32_t)(bi.off & 15u), span = (lead + bi.len + 15u) & ~15u;
                if (span <= stage_bytes && (bi.off - lead) + span <= readable) {
                    if (lane == 0) {
                        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(span) : "memory");
                        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                                     ::"r"((uint32_t)__cvta_generic_to_shared(stage)), "l"(bytes + (bi.off - lead)), "r"(span), "r"(bar)
                                     : "memory");
                    }
                    asm volatile(
                        "{\n\t.reg .pred p;\n\t"
                        "LOGW_%=:\n\t"
                        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
                        "@p bra LOGD_%=;\n\t"
                        "bra LOGW_%=;\n\t"
                        "LOGD_%=:\n\t}" ::"r"(bar), "r"(phase) : "memory");
                    phase ^= 1u;
                    base = stage + lead;
                }
            }
            const uint8_t *end = base + bi.len;
            uint32_t pos = LOG_HEADER_BYTES;          // offset of the next record inside the batch
            const uint64_t r0 = rec_base[b];
            bool ok = true;
            for (int32_t i0 = 0; i0 < bi.records && ok; i0 += 32) {
                const int cnt = min(32, bi.records - i0);
                if (lane == 0) {
                    for (int j = 0; j < cnt; j++) {
                        s_start[j] = pos;
                        uint64_t u;
                        const int n = uvarint_g(base + pos, end, u);
                        const int64_t rec_len = unzigzag(u);
                        if (n <= 0 || rec_len < 0 || (uint64_t)pos + n + rec_len > bi.len) { ok = false; break; }
                        pos += (uint32_t)n + (uint32_t)rec_len;
                    }
                    s_start[32] = ok ? pos : 0xffffffffu;
                }
                __syncwarp();
                pos = s_start[32];
                ok = pos != 0xffffffffu;
                if (!ok) break;
                int64_t klen = -1, vlen = -1, ts_delta = 0, off_delta = 0;
                uint32_t key_at = 0;
                bool lane_ok = true;
                if (lane < cnt) {
                    const uint8_t *q = base + s_start[lane];
                    const uint8_t *rec_end = lane + 1 < cnt ? base + s_start[lane + 1] : base + pos;
                    uint64_t u;
                    int n = uvarint_g(q, rec_end, u); q += n;            // record length (validated by lane 0)
                    q += 1;                                               // record attributes (unused)
                    n = uvarint_g(q, rec_end, u); lane_ok = lane_ok && n > 0; q += n;
                    ts_delta = unzigzag(u);
                    n = uvarint_g(q, rec_end, u); lane_ok = lane_ok && n > 0; q += n;
                    off_delta = unzigzag(u);
                    n = uvarint_g(q, rec_end, u); lane_ok = lane_ok && n > 0; q += n;
                    klen = unzigzag(u);
                    lane_ok = lane_ok && klen >= -1 && klen <= 0x7fffffff && (klen <= 0 || q + klen <= rec_end);
                    key_at = (uint32_t)(q - base);
                    if (lane_ok && klen > 0) q += klen;
                    n = lane_ok ? uvarint_g(q, rec_end, u) : 0; lane_ok = lane_ok && n > 0; q += n;
                    vlen = unzigzag(u);
                    lane_ok = lane_ok && vlen >= -1 && vlen <= 0x7fffffff && (vlen <= 0 || q + vlen <= rec_end);
                }
                __syncwarp();   // every lane has read its start before lane 0 overwrites them
                ok = __all_sync(full, lane_ok);
                if (!ok) break;
                if (lane < cnt) {
                    const uint64_t r = r0 + (uint64_t)i0 + lane;
                    partition[r] = bi.partition;
                    if (offset) offset[r] = bi.base_offset + off_delta;
                    ts_ms[r] = bi.log_append_time ? bi.max_ts : bi.base_ts + ts_delta;
                    key_len[r] = (int32_t)klen;
                    value_len[r] = (int32_t)vlen;
                    if (key_src) key_src[r] = bi.off + key_at;
                }
            }
            if (!ok && lane == 0) atomicOr(error_flags, (uint32_t)LOGB_BAD);
            __syncwarp();   // the stage is free for the next batch's copy
        }
    }
}

// Packs the key bytes in record order (what the scan kernel hashes): one warp per 128-record tile, a lane owns four
// consecutive records; byte offsets from the tile base (key_tile_base, derived from key_len beforehand) plus an in-tile scan.
__global__ void __launch_bounds__(256) log_gather_keys_kernel(const uint8_t *bytes, const uint64_t *key_src, const int32_t *key_len,
                                                              int64_t n, const uint64_t *tile_base, uint8_t *key_out) {
    const int lane = threadIdx.x & 31;
    const int64_t ntiles = (n + 127) / 128;
    const int64_t gw = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, gs = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t tile = gw; tile < ntiles; tile += gs) {
        int32_t len[4];
        uint64_t src[4];
        uint32_t mine = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            const int64_t r = tile * 128 + (int64_t)lane * 4 + k;
            len[k] = r < n ? key_len[r] : -1;
            src[k] = len[k] > 0 ? key_src[r] : 0;
            mine += len[k] > 0 ? (uint32_t)len[k] : 0u;
        }
        uint32_t inc = mine;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += t;
        }
        uint8_t *o = key_out + tile_base[tile] + (inc - mine);
#pragma unroll
        for (int k = 0; k < 4; k++) {
            if (len[k] > 0) {
                const uint8_t *sp = bytes + src[k];
                int j = 0;
                if ((reinterpret_cast<uintptr_t>(o) & 3u) == 0) {
                    // word-aligned destination (always, for keys whose lengths are multiples of 4: ids, hashes, UUIDs): whole
                    // words, from aligned source words put together with a funnel shift
                    const uintptr_t a = reinterpret_cast<uintptr_t>(sp);
                    const uint32_t *wp = reinterpret_cast<const uint32_t *>(a & ~(uintptr_t)3);
                    const uint32_t sh = (uint32_t)(a & 3u) * 8u;
                    const int nw = len[k] >> 2;
                    uint32_t *ow = reinterpret_cast<uint32_t *>(o);
                    if (sh == 0) {
                        for (int w = 0; w < nw; w++) ow[w] = __ldg(wp + w);
                        j = nw * 4;
                    } else {
                        // the aligned word behind the last full one may reach past the key (and past the buffer): the last
                        // word is left to the byte loop
                        uint32_t lo = __ldg(wp);
                        for (int w = 0; w + 1 < nw; w++) {
                            const uint32_t hi = __ldg(wp + w + 1);
                            ow[w] = __funnelshift_r(lo, hi, sh);
                            lo = hi;
                        }
                        j = nw > 0 ? (nw - 1) * 4 : 0;
                    }
                }
                for (; j < len[k]; j++) o[j] = __ldg(sp + j);
                o += len[k];
            }
        }
    }
}

}  // namespace kta
