// kta_zstd.cuh — Zstandard frames (RFC 8878): the records section of a Kafka record batch whose attributes name codec 4
// (zstd), which librdkafka decompresses inside poll before the handlers see a message (src/kafka.rs:93).  Used by
// log_zstd_size_kernel and log_decompress_kernel (kta_logdecode.cuh), one warp per batch.
//
// Shape (as kta_inflate.cuh): every lane of the warp walks the same bytes and bit streams (lane-uniform control flow,
// shared-memory tables read as broadcasts); lane 0 writes the FSE / Huffman tables, all lanes fill the Huffman lookup table;
// the four streams of a 4-stream literals section are decoded by lanes 0-3, one each; all 32 lanes copy literal runs and
// matches (lz_emit_literals / lz_emit_match).  Sequences are decoded on the lane-uniform path.
// Accepted: zstd frames (any FCS field size, single segment or Window_Descriptor, content checksum skipped unverified like
// the batch CRC: check.crcs=false), skippable frames, several frames one after the other (outputs concatenated; a match
// never reaches before the start of its own frame).  Rejected: dictionaries, reserved bits / block types / modes.
// Huffman-coded literals of a block are decoded into the TAIL of the batch's output slot, [cap - size, cap): the output
// never catches up with a literal it has not read yet (every literal is part of the remaining output), so no scratch beyond
// the exact output image is needed; a write that would pass the next unread literal is a damaged block.
// __host__ __device__ so that tests/test_zstd_host.py runs the same statements on the host (one "lane") against pyarrow's
// compressor under the address sanitizer; the product calls it on the device only.
#pragma once
#include <stdint.h>

#ifdef __CUDA_ARCH__
#define KTA_ZSTD_ALL(p) __all_sync(0xffffffffu, (p))
#else
#define KTA_ZSTD_ALL(p) (p)
#endif

namespace kta {

constexpr uint32_t ZSTD_BLOCK_MAX = 128u * 1024u;
constexpr int ZSTD_HUF_LOG_MAX = 11;

// decoding counts per mode, for the host test (which modes an input exercised); nullptr on the device
enum ZstdMode {
    ZM_FRAME, ZM_SKIPPABLE, ZM_SINGLE_SEGMENT, ZM_WINDOW_DESC, ZM_CHECKSUM, ZM_FCS_NONE, ZM_FCS_1, ZM_FCS_2, ZM_FCS_4, ZM_FCS_8,
    ZM_BLOCK_RAW, ZM_BLOCK_RLE, ZM_BLOCK_COMPRESSED,
    ZM_LIT_RAW, ZM_LIT_RLE, ZM_LIT_COMPRESSED, ZM_LIT_TREELESS,
    ZM_LIT_HDR1, ZM_LIT_HDR2, ZM_LIT_HDR3,                          // Raw / RLE size formats: 1-, 2-, 3-byte headers
    ZM_HUF_SF0, ZM_HUF_SF1, ZM_HUF_SF2, ZM_HUF_SF3,                 // Compressed / Treeless size formats
    ZM_STREAMS1, ZM_STREAMS4, ZM_HUF_DIRECT, ZM_HUF_FSE,
    ZM_NSEQ0, ZM_NSEQ1, ZM_NSEQ2, ZM_NSEQ3,                         // Number_of_Sequences: 0, 1-, 2-, 3-byte encodings
    ZM_LL_PREDEF, ZM_LL_RLE, ZM_LL_FSE, ZM_LL_REPEAT,
    ZM_OF_PREDEF, ZM_OF_RLE, ZM_OF_FSE, ZM_OF_REPEAT,
    ZM_ML_PREDEF, ZM_ML_RLE, ZM_ML_FSE, ZM_ML_REPEAT,
    ZM_REP1, ZM_REP2, ZM_REP3, ZM_REP1_MINUS1, ZM_REP_LL0,          // repeat offsets used (resolved), any with Literals_Length 0
    ZM_COUNT
};

// per warp, in shared memory on the device.  FSE entries: symbol | nbBits << 8 | baseline of the next state << 16;
// Huffman entries: symbol | nbBits << 8, indexed by the next huf_log bits of the stream.
struct ZstdWork {
    uint32_t ll[1 << 9], ml[1 << 9], of[1 << 8];   // sequence tables (kept across blocks for Repeat mode)
    uint16_t huf[1 << ZSTD_HUF_LOG_MAX];            // literal table (kept across blocks for Treeless literals)
    uint32_t wt[1 << 6];                            // FSE table of the Huffman weights
    int16_t norm[256];                              // normalized counts of the table being built
    uint16_t next[256];                             // FSE: next state per symbol; Huffman: first table slot per symbol
    uint8_t weight[256];
};

// what lives across the blocks of one frame (lane-uniform, in registers)
struct ZstdFrame {
    uint64_t rep[3];
    int ll_log, of_log, ml_log;   // -1: no table yet (Repeat mode is an error)
    int huf_log;                  // 0: no Huffman table yet (Treeless literals are an error)
};

__host__ __device__ inline void zm_count(uint32_t *modes, int m) {
    if (modes) modes[m]++;
}

__host__ __device__ inline int zstd_highbit(uint32_t v) {   // v > 0
    int h = 0;
    while (v >>= 1) h++;
    return h;
}

__host__ __device__ inline uint64_t zstd_le(const uint8_t *p, int n) {
    uint64_t v = 0;
    for (int i = n - 1; i >= 0; i--) v = (v << 8) | p[i];
    return v;
}

// Backward bit stream (RFC 8878 4.1): read from the end towards the start, the last byte's highest set bit is padding.
// pos = bits not yet read; bits before the start of the stream read as zeros (pos goes negative: overflow).
struct ZstdBits {
    const uint8_t *p;
    int64_t pos;
};
__host__ __device__ inline bool zb_init(ZstdBits &b, const uint8_t *p, uint32_t n) {
    if (n == 0 || p[n - 1] == 0) return false;
    b.p = p;
    b.pos = 8 * (int64_t)(n - 1) + zstd_highbit(p[n - 1]);
    return true;
}
__host__ __device__ inline uint32_t zb_peek(const ZstdBits &b, int k) {   // k <= 31
    if (k == 0 || b.pos <= 0) return 0;
    const int64_t lo = b.pos - k;
    const int64_t first = lo >= 0 ? lo >> 3 : -((-lo + 7) >> 3), last = (b.pos - 1) >> 3;
    uint64_t v = 0;
    for (int64_t i = last; i >= first; i--) v = (v << 8) | (i >= 0 ? b.p[i] : 0u);
    return (uint32_t)(v >> (lo - first * 8)) & ((1u << k) - 1u);
}
__host__ __device__ inline uint32_t zb_read(ZstdBits &b, int k) {
    const uint32_t v = zb_peek(b, k);
    b.pos -= k;
    return v;
}

// Predefined distributions (RFC 8878 3.1.1.3.2.2), as characters '0' + count + 1 (string literals live in device memory
// without a table declaration per compilation pass)
__host__ __device__ inline const char *zstd_default_norm(int kind) {
    return kind == 0 ? "543333333333322233333333343222220000"                                          // LL, log 6
         : kind == 1 ? "22222233322222222222222200000"                                                 // OF, log 5
                     : "25433333322222222222222222222222222222222222220000000";                        // ML, log 6
}

// Literals_Length / Match_Length codes → baseline and extra bits (RFC 8878 3.1.1.3.2.1.1), in closed form
__host__ __device__ inline int zstd_ll_bits(int c) {
    return c < 16 ? 0 : c < 20 ? 1 : c < 22 ? 2 : c < 24 ? 3 : c == 24 ? 4 : c - 19;
}
__host__ __device__ inline uint32_t zstd_ll_base(int c) {
    return c < 16 ? (uint32_t)c : c < 20 ? 16u + 2u * (c - 16) : c < 22 ? 24u + 4u * (c - 20) : c < 24 ? 32u + 8u * (c - 22) : c == 24 ? 48u : 1u << (c - 19);
}
__host__ __device__ inline int zstd_ml_bits(int c) {
    return c < 32 ? 0 : c < 36 ? 1 : c < 38 ? 2 : c < 40 ? 3 : c < 42 ? 4 : c == 42 ? 5 : c - 36;
}
__host__ __device__ inline uint32_t zstd_ml_base(int c) {
    return c < 32 ? (uint32_t)c + 3u : c < 36 ? 35u + 2u * (c - 32) : c < 38 ? 43u + 4u * (c - 36) : c < 40 ? 51u + 8u * (c - 38)
         : c < 42 ? 67u + 16u * (c - 40) : c == 42 ? 99u : (1u << (c - 36)) + 3u;
}

// FSE table description (RFC 8878 4.1.1), a forward little-endian bit stream.  Every lane reads it; lane 0 stores the
// counts.  Returns the bytes used (0: malformed), the accuracy log and the number of symbols described.
__host__ __device__ inline uint32_t zstd_read_ncount(const uint8_t *p, uint32_t n, int max_log, int max_sym, int16_t *norm, int &log,
                                                     int &nsym, int lane) {
    const uint64_t nbits = 8ull * n;
    uint64_t bit = 0;
    auto peek = [&](int k) -> uint32_t {   // k <= 16; bits past the end read as zeros (the caller checks the position)
        uint32_t v = 0;
        for (int i = 0; i < k; i++) {
            const uint64_t q = bit + i;
            if (q < nbits) v |= (uint32_t)((p[q >> 3] >> (q & 7)) & 1u) << i;
        }
        return v;
    };
    if (n == 0) return 0;
    log = (int)peek(4) + 5;
    bit = 4;
    if (log > max_log) return 0;
    int remaining = (1 << log) + 1, threshold = 1 << log, nb = log + 1, sym = 0;
    bool prev0 = false;
    while (remaining > 1 && sym <= max_sym) {
        if (prev0) {
            int n0 = sym;
            for (;;) {
                const uint32_t r = peek(2);
                bit += 2;
                if (bit > nbits) return 0;
                n0 += (int)r;
                if (r != 3) break;
            }
            if (n0 > max_sym) return 0;
            for (; sym < n0; sym++)
                if (lane == 0) norm[sym] = 0;
        }
        const int max = (2 * threshold - 1) - remaining;
        const uint32_t v = peek(nb);
        int count;
        if ((int)(v & (uint32_t)(threshold - 1)) < max) {
            count = (int)(v & (uint32_t)(threshold - 1));
            bit += nb - 1;
        } else {
            count = (int)(v & (uint32_t)(2 * threshold - 1));
            if (count >= threshold) count -= max;
            bit += nb;
        }
        if (bit > nbits) return 0;
        count--;                                   // -1: "less than 1", one cell at the top of the table
        remaining -= count < 0 ? -count : count;
        if (lane == 0) norm[sym] = (int16_t)count;
        sym++;
        prev0 = count == 0;
        while (remaining < threshold) {
            nb--;
            threshold >>= 1;
        }
    }
    if (remaining != 1) return 0;
    nsym = sym;
    return (uint32_t)((bit + 7) >> 3);
}

// FSE decoding table from normalized counts that add up to 1 << log (RFC 8878 4.1.1: cells of "less than 1" symbols at
// the top, the others spread with step 5/8 size + 3).  Lane 0 builds it.
__host__ __device__ inline void zstd_fse_build(uint32_t *dt, const int16_t *norm, int nsym, int log, uint16_t *next, int lane) {
    if (lane == 0) {
        const uint32_t size = 1u << log, mask = size - 1, step = (size >> 1) + (size >> 3) + 3;
        uint32_t high = size - 1;
        for (int s = 0; s < nsym; s++) {
            if (norm[s] == -1) {
                dt[high--] = (uint32_t)s;
                next[s] = 1;
            } else next[s] = (uint16_t)norm[s];
        }
        uint32_t pos = 0;   // the counts add up to the table size, so the spread ends where it began
        for (int s = 0; s < nsym; s++)
            for (int i = 0; i < norm[s]; i++) {
                dt[pos] = (uint32_t)s;
                do pos = (pos + step) & mask; while (pos > high);
            }
        for (uint32_t u = 0; u < size; u++) {
            const uint32_t s = dt[u] & 0xffu, ns = next[s]++;
            const uint32_t nb = (uint32_t)log - (uint32_t)zstd_highbit(ns);
            dt[u] = s | nb << 8 | ((ns << nb) - size) << 16;
        }
    }
    KTA_INF_SYNC();
}

// one of the three sequence tables per its Symbol_Compression_Mode; returns false on malformed input, `used` = bytes
// of table description read
__host__ __device__ inline bool zstd_seq_table(int mode, int kind /* 0 LL, 1 OF, 2 ML */, const uint8_t *p, uint32_t n, uint32_t &used,
                                               uint32_t *dt, int &log, ZstdWork &w, int lane, uint32_t *modes) {
    const int max_sym = kind == 0 ? 35 : kind == 1 ? 31 : 52, max_log = kind == 1 ? 8 : 9;
    zm_count(modes, (kind == 0 ? ZM_LL_PREDEF : kind == 1 ? ZM_OF_PREDEF : ZM_ML_PREDEF) + mode);
    used = 0;
    if (mode == 3) return log >= 0;                  // Repeat: the previous block's table of this frame
    KTA_INF_SYNC();                                  // every lane is done with the previous table
    if (mode == 0) {
        const char *d = zstd_default_norm(kind);
        int nsym = 0;
        while (d[nsym]) nsym++;
        if (lane == 0)
            for (int s = 0; s < nsym; s++) w.norm[s] = (int16_t)(d[s] - '0' - 1);
        log = kind == 1 ? 5 : 6;
        zstd_fse_build(dt, w.norm, nsym, log, w.next, lane);
    } else if (mode == 1) {
        if (n < 1 || p[0] > max_sym) return false;
        if (lane == 0) dt[0] = p[0];                 // one state, no bits
        log = 0;
        used = 1;
        KTA_INF_SYNC();
    } else {
        int nsym;
        used = zstd_read_ncount(p, n, max_log, max_sym, w.norm, log, nsym, lane);
        if (!used) return false;
        zstd_fse_build(dt, w.norm, nsym, log, w.next, lane);
    }
    return true;
}

// Huffman tree description (RFC 8878 4.2.1) → w.huf; returns the bytes used, 0 if malformed
__host__ __device__ inline uint32_t zstd_huf_table(const uint8_t *p, uint32_t n, ZstdWork &w, int &huf_log, int lane, uint32_t *modes) {
    if (n < 1) return 0;
    const uint32_t hb = p[0];
    uint32_t used;
    int nw = 0;
    KTA_INF_SYNC();                                  // every lane is done with the previous table
    if (hb >= 128) {                                 // direct: 4-bit weights, two per byte, high nibble first
        zm_count(modes, ZM_HUF_DIRECT);
        nw = (int)hb - 127;
        used = 1 + ((uint32_t)nw + 1) / 2;
        if (used > n) return 0;
        if (lane == 0)
            for (int i = 0; i < nw; i++) w.weight[i] = (uint8_t)(i & 1 ? p[1 + i / 2] & 15 : p[1 + i / 2] >> 4);
    } else {                                         // FSE-compressed weights, two interleaved states
        zm_count(modes, ZM_HUF_FSE);
        used = 1 + hb;
        if (used > n || hb == 0) return 0;
        int log, nsym;
        const uint32_t h = zstd_read_ncount(p + 1, hb, 6, ZSTD_HUF_LOG_MAX + 1, w.norm, log, nsym, lane);
        if (!h || h >= hb) return 0;
        zstd_fse_build(w.wt, w.norm, nsym, log, w.next, lane);
        ZstdBits b;
        if (!zb_init(b, p + 1 + h, hb - h)) return 0;
        uint32_t st[2];
        st[0] = zb_read(b, log);
        st[1] = zb_read(b, log);
        for (int k = 0;; k ^= 1) {                   // the state that decodes the next weight
            if (nw > 255 - 2) return 0;
            const uint32_t e = w.wt[st[k]];
            if (lane == 0) w.weight[nw] = (uint8_t)e;
            nw++;
            st[k] = (e >> 16) + zb_read(b, (int)((e >> 8) & 0xffu));
            if (b.pos < 0) {                         // out of bits: the other state's symbol is the last weight
                if (lane == 0) w.weight[nw] = (uint8_t)w.wt[st[k ^ 1]];
                nw++;
                break;
            }
        }
    }
    KTA_INF_SYNC();
    // the last symbol's weight completes the sum of 2^(weight - 1) to a power of two
    uint32_t total = 0, rank[ZSTD_HUF_LOG_MAX + 2];
    for (int r = 0; r <= ZSTD_HUF_LOG_MAX + 1; r++) rank[r] = 0;
    for (int i = 0; i < nw; i++) {
        const uint32_t wi = w.weight[i];
        if (wi > (uint32_t)ZSTD_HUF_LOG_MAX) return 0;
        rank[wi]++;
        total += (1u << wi) >> 1;
    }
    if (total == 0) return 0;
    const int log = zstd_highbit(total) + 1;
    if (log > ZSTD_HUF_LOG_MAX) return 0;
    const uint32_t rest = (1u << log) - total;
    if (rest != 1u << zstd_highbit(rest)) return 0;
    const int last = zstd_highbit(rest) + 1;
    rank[last]++;
    if (rank[1] < 2 || (rank[1] & 1)) return 0;
    const int nsym = nw + 1;
    if (lane == 0) {
        w.weight[nw] = (uint8_t)last;
        // weight 1 (the longest codes) first, symbols in order within a weight; a symbol of weight v fills 2^(v-1) slots
        uint32_t start[ZSTD_HUF_LOG_MAX + 2], cur = 0;
        for (int v = 1; v <= log; v++) {
            start[v] = cur;
            cur += rank[v] << (v - 1);
        }
        for (int s = 0; s < nsym; s++) {
            const int v = w.weight[s];
            if (v) {
                w.next[s] = (uint16_t)start[v];
                start[v] += 1u << (v - 1);
            }
        }
    }
    KTA_INF_SYNC();
    for (int s = lane; s < nsym; s += KTA_INF_LANES) {
        const int v = w.weight[s];
        if (v) {
            const uint16_t e = (uint16_t)(s | (log + 1 - v) << 8);
            for (uint32_t i = 0; i < (1u << (v - 1)); i++) w.huf[w.next[s] + i] = e;
        }
    }
    KTA_INF_SYNC();
    huf_log = log;
    return used;
}

// one Huffman stream: exactly `cnt` symbols that use up exactly the stream's bits
__host__ __device__ inline bool zstd_huf_stream(const uint8_t *p, uint32_t n, uint8_t *dst, uint32_t cnt, const uint16_t *huf, int log) {
    ZstdBits b;
    if (!zb_init(b, p, n)) return false;
    for (uint32_t k = 0; k < cnt; k++) {
        const uint32_t e = huf[zb_peek(b, log)];
        dst[k] = (uint8_t)e;
        b.pos -= e >> 8;
    }
    return b.pos == 0;
}

// literals of a sequence: Raw (in place in the input), RLE (one byte, repeated by a match of offset 1), or Huffman-decoded
// at the tail of the output slot (`lp` = the next unread one): copied forward in pieces that do not overlap their source
// (the output may be just behind the literals it reads), or not at all when it has caught up with them
enum { ZLIT_RAW, ZLIT_RLE, ZLIT_TAIL };
template <bool COPY>
__host__ __device__ inline void zstd_emit_literals(uint8_t *out, uint64_t op, int kind, const uint8_t *raw, uint64_t lp, uint32_t cnt, int lane) {
    if (!COPY || cnt == 0) return;
    if (kind == ZLIT_RAW) {
        lz_emit_literals<true>(out, op, raw, cnt, lane);
    } else if (kind == ZLIT_RLE) {
        if (lane == 0) out[op] = raw[0];
        lz_emit_match<true>(out, op + 1, 1, cnt - 1, lane);   // syncs first: lane 0's byte is visible
    } else if (lp != op) {
        const uint64_t gap = lp - op;
        for (uint32_t done = 0; done < cnt;) {
            const uint32_t c = (uint32_t)(gap < (uint64_t)(cnt - done) ? gap : (uint64_t)(cnt - done));
            lz_emit_literals<true>(out, op + done, out + lp + done, c, lane);
            KTA_INF_SYNC();   // read before the next piece overwrites it
            done += c;
        }
    }
}

// Compressed block (RFC 8878 3.1.1.3): literals section, sequences section, execution.  `op` advances by the block's output.
template <bool COPY>
__host__ __device__ inline bool zstd_block(const uint8_t *in, uint32_t n, uint8_t *out, uint64_t cap, uint64_t &op, uint64_t frame_start,
                                           uint64_t block_max, ZstdFrame &f, ZstdWork &w, int lane, uint32_t *modes) {
    const uint64_t block_start = op;
    if (n < 1) return false;
    // ---- literals section header
    const uint32_t b0 = in[0], ltype = b0 & 3u, sf = (b0 >> 2) & 3u;
    uint32_t lsize, csize = 0, hdr;
    int nstreams = 1;
    if (ltype <= 1) {
        hdr = sf == 1 ? 2 : sf == 3 ? 3 : 1;
        if (n < hdr) return false;
        lsize = hdr == 1 ? b0 >> 3 : hdr == 2 ? (b0 >> 4) | ((uint32_t)in[1] << 4) : (b0 >> 4) | ((uint32_t)in[1] << 4) | ((uint32_t)in[2] << 12);
        zm_count(modes, ltype == 0 ? ZM_LIT_RAW : ZM_LIT_RLE);
        zm_count(modes, ZM_LIT_HDR1 + (int)hdr - 1);
    } else {
        nstreams = sf == 0 ? 1 : 4;
        hdr = sf <= 1 ? 3 : sf == 2 ? 4 : 5;
        if (n < hdr) return false;
        const int bits = sf <= 1 ? 10 : sf == 2 ? 14 : 18;
        const uint64_t h = zstd_le(in, (int)hdr);
        lsize = (uint32_t)(h >> 4) & ((1u << bits) - 1u);
        csize = (uint32_t)(h >> (4 + bits)) & ((1u << bits) - 1u);
        zm_count(modes, ltype == 2 ? ZM_LIT_COMPRESSED : ZM_LIT_TREELESS);
        zm_count(modes, ZM_HUF_SF0 + (int)sf);
        zm_count(modes, nstreams == 1 ? ZM_STREAMS1 : ZM_STREAMS4);
    }
    if (lsize > block_max) return false;
    int lkind;
    const uint8_t *lsrc = nullptr;
    uint32_t pos;
    if (ltype == 0) {
        if (lsize > n - hdr) return false;
        lkind = ZLIT_RAW;
        lsrc = in + hdr;
        pos = hdr + lsize;
    } else if (ltype == 1) {
        if (n - hdr < 1) return false;
        lkind = ZLIT_RLE;
        lsrc = in + hdr;
        pos = hdr + 1;
    } else {
        if (csize > n - hdr) return false;
        lkind = ZLIT_TAIL;
        pos = hdr + csize;
        if (nstreams == 4 && lsize < 6) return false;
        const uint8_t *p = in + hdr;
        uint32_t m = csize;
        if (ltype == 2) {
            const uint32_t t = zstd_huf_table(p, m, w, f.huf_log, lane, modes);
            if (!t) return false;
            p += t;
            m -= t;
        } else if (!f.huf_log) return false;         // Treeless literals need an earlier table of this frame
        if (COPY) {
            if (op + lsize > cap) return false;      // the literals would overwrite output already written
            uint8_t *dst = out + (cap - lsize);
            bool ok = true;
            if (nstreams == 1) {
                if (lane == 0) ok = zstd_huf_stream(p, m, dst, lsize, w.huf, f.huf_log);
            } else {
                if (m < 6) return false;
                const uint32_t s1 = (uint32_t)zstd_le(p, 2), s2 = (uint32_t)zstd_le(p + 2, 2), s3 = (uint32_t)zstd_le(p + 4, 2);
                if ((uint64_t)s1 + s2 + s3 > m - 6) return false;
                const uint32_t seg = (lsize + 3) / 4;
                if (3 * seg > lsize) return false;
                for (int k = lane; k < 4; k += KTA_INF_LANES) {   // lanes 0-3: one stream each, into disjoint ranges
                    const uint32_t at = 6 + (k > 0 ? s1 : 0) + (k > 1 ? s2 : 0) + (k > 2 ? s3 : 0);
                    const uint32_t len = k == 0 ? s1 : k == 1 ? s2 : k == 2 ? s3 : m - 6 - s1 - s2 - s3;
                    ok = ok && zstd_huf_stream(p + at, len, dst + (uint32_t)k * seg, k < 3 ? seg : lsize - 3 * seg, w.huf, f.huf_log);
                }
            }
            ok = KTA_ZSTD_ALL(ok);
            if (!ok) return false;
            KTA_INF_SYNC();                          // the decoded literals are visible to every lane
        }
    }
    // ---- sequences section header
    if (pos >= n) return false;
    uint32_t nseq = in[pos++];
    if (nseq == 0) zm_count(modes, ZM_NSEQ0);
    else if (nseq < 128) zm_count(modes, ZM_NSEQ1);
    else if (nseq < 255) {
        if (pos >= n) return false;
        nseq = ((nseq - 128) << 8) + in[pos++];
        zm_count(modes, ZM_NSEQ2);
    } else {
        if (n - pos < 2) return false;
        nseq = (uint32_t)in[pos] + ((uint32_t)in[pos + 1] << 8) + 0x7F00u;
        pos += 2;
        zm_count(modes, ZM_NSEQ3);
    }
    uint64_t lp = cap - lsize;                       // ZLIT_TAIL: the next unread literal
    uint32_t lit_left = lsize;
    if (nseq > 0) {
        if (pos >= n) return false;
        const uint32_t cm = in[pos++];
        if (cm & 3u) return false;                   // reserved bits
        uint32_t used;
        if (!zstd_seq_table((int)(cm >> 6), 0, in + pos, n - pos, used, w.ll, f.ll_log, w, lane, modes)) return false;
        pos += used;
        if (!zstd_seq_table((int)((cm >> 4) & 3u), 1, in + pos, n - pos, used, w.of, f.of_log, w, lane, modes)) return false;
        pos += used;
        if (!zstd_seq_table((int)((cm >> 2) & 3u), 2, in + pos, n - pos, used, w.ml, f.ml_log, w, lane, modes)) return false;
        pos += used;
        KTA_INF_SYNC();
        ZstdBits b;
        if (!zb_init(b, in + pos, n - pos)) return false;
        uint32_t sll = zb_read(b, f.ll_log), sof = zb_read(b, f.of_log), sml = zb_read(b, f.ml_log);
        for (uint32_t i = 0; i < nseq; i++) {
            const uint32_t ell = w.ll[sll], eof = w.of[sof], eml = w.ml[sml];
            const int ofc = (int)(eof & 0xffu), mlc = (int)(eml & 0xffu), llc = (int)(ell & 0xffu);
            // extra bits: offset, match length, literals length
            const uint64_t ofv = (1ull << ofc) + zb_read(b, ofc);
            const uint32_t ml = zstd_ml_base(mlc) + zb_read(b, zstd_ml_bits(mlc));
            const uint32_t ll = zstd_ll_base(llc) + zb_read(b, zstd_ll_bits(llc));
            uint64_t off;
            if (ofv > 3) {
                off = ofv - 3;
                f.rep[2] = f.rep[1];
                f.rep[1] = f.rep[0];
                f.rep[0] = off;
            } else {
                // repeat offsets; with Literals_Length 0 they shift by one and the third means rep1 - 1
                const int r = (int)ofv - 1 + (ll == 0 ? 1 : 0);
                zm_count(modes, ZM_REP1 + r);
                if (ll == 0) zm_count(modes, ZM_REP_LL0);
                if (r == 0) off = f.rep[0];
                else {
                    off = r == 3 ? f.rep[0] - 1 : f.rep[r];
                    if (r != 1) f.rep[2] = f.rep[1];
                    f.rep[1] = f.rep[0];
                    f.rep[0] = off;
                }
            }
            if (i + 1 < nseq) {                      // state updates: LL, ML, OF
                sll = (ell >> 16) + zb_read(b, (int)((ell >> 8) & 0xffu));
                sml = (eml >> 16) + zb_read(b, (int)((eml >> 8) & 0xffu));
                sof = (eof >> 16) + zb_read(b, (int)((eof >> 8) & 0xffu));
            }
            if (b.pos < 0 || ll > lit_left) return false;
            if (COPY && lkind != ZLIT_TAIL && op + ll > cap) return false;
            zstd_emit_literals<COPY>(out, op, lkind, lkind == ZLIT_RAW ? lsrc + (lsize - lit_left) : lsrc, lp, ll, lane);
            op += ll;
            lp += ll;
            lit_left -= ll;
            if (off == 0 || off > op - frame_start) return false;
            if (COPY && op + ml > (lkind == ZLIT_TAIL ? lp : cap)) return false;
            lz_emit_match<COPY>(out, op, (uint32_t)off, ml, lane);
            op += ml;
        }
        if (b.pos != 0) return false;                // the bit stream is used up exactly
    } else if (pos != n) return false;
    // ---- the literals after the last sequence
    if (COPY && lkind != ZLIT_TAIL && op + lit_left > cap) return false;
    zstd_emit_literals<COPY>(out, op, lkind, lkind == ZLIT_RAW ? lsrc + (lsize - lit_left) : lsrc, lp, lit_left, lane);
    op += lit_left;
    KTA_INF_SYNC();                                  // the next block may overwrite the tail
    return op - block_start <= block_max;
}

// The frames at in[0, n) (RFC 8878 3.1).  COPY: output into out[0, out_cap), the whole warp calls this.  Without COPY only
// the size is computed (no literal decoding, no copies); with trust_fcs a frame that states its Frame_Content_Size is taken
// at that size, bounded by what its blocks can hold (a forged size must not size the output), and its blocks are not decoded.
template <bool COPY>
__host__ __device__ LzWalk zstd_walk(const uint8_t *in, uint32_t n, uint8_t *out, uint64_t out_cap, ZstdWork &w, int lane,
                                     bool trust_fcs = false, uint32_t *modes = nullptr) {
    LzWalk r{0, false};
    uint32_t ip = 0;
    uint64_t op = 0;
    bool frames = false;
    while (ip < n) {
        if (n - ip < 4) return r;
        const uint32_t magic = (uint32_t)zstd_le(in + ip, 4);
        if ((magic & 0xFFFFFFF0u) == 0x184D2A50u) {  // skippable frame
            if (n - ip < 8) return r;
            const uint32_t fsz = (uint32_t)zstd_le(in + ip + 4, 4);
            if (fsz > n - ip - 8) return r;
            ip += 8 + fsz;
            zm_count(modes, ZM_SKIPPABLE);
            continue;
        }
        if (magic != 0xFD2FB528u || n - ip < 5) return r;
        ip += 4;
        const uint32_t fhd = in[ip++];
        const uint32_t fcs_flag = fhd >> 6, single = (fhd >> 5) & 1u, checksum = (fhd >> 2) & 1u, did_flag = fhd & 3u;
        if (fhd & 0x08u) return r;                   // reserved bit
        uint64_t window = 0;
        if (!single) {
            if (ip >= n) return r;
            const uint32_t wd = in[ip++];
            const uint64_t base = 1ull << (10 + (wd >> 3));
            window = base + (base >> 3) * (wd & 7u);
            zm_count(modes, ZM_WINDOW_DESC);
        } else zm_count(modes, ZM_SINGLE_SEGMENT);
        const uint32_t did_size = did_flag == 3 ? 4 : did_flag;
        if (n - ip < did_size || zstd_le(in + ip, (int)did_size) != 0) return r;   // dictionaries are not supported
        ip += did_size;
        const uint32_t fcs_size = fcs_flag == 0 ? single : fcs_flag == 1 ? 2 : fcs_flag == 2 ? 4 : 8;
        if (n - ip < fcs_size) return r;
        const bool has_fcs = fcs_size > 0;
        const uint64_t fcs = zstd_le(in + ip, (int)fcs_size) + (fcs_size == 2 ? 256u : 0u);
        ip += fcs_size;
        zm_count(modes, fcs_size == 0 ? ZM_FCS_NONE : fcs_size == 1 ? ZM_FCS_1 : fcs_size == 2 ? ZM_FCS_2 : fcs_size == 4 ? ZM_FCS_4 : ZM_FCS_8);
        if (checksum) zm_count(modes, ZM_CHECKSUM);
        zm_count(modes, ZM_FRAME);
        if (single) window = fcs;
        const uint64_t block_max = window < ZSTD_BLOCK_MAX ? window : ZSTD_BLOCK_MAX;
        const uint64_t frame_start = op;
        ZstdFrame f{{1, 4, 8}, -1, -1, -1, 0};
        uint64_t bound = 0;                          // trust_fcs: what the blocks can hold
        const bool skim = !COPY && trust_fcs && has_fcs;
        for (;;) {
            if (n - ip < 3) return r;
            const uint32_t bh = (uint32_t)zstd_le(in + ip, 3);
            ip += 3;
            const uint32_t last = bh & 1u, type = (bh >> 1) & 3u, bsize = bh >> 3;
            if (type == 3 || bsize > block_max) return r;
            const uint32_t csize = type == 1 ? 1u : bsize;
            if (csize > n - ip) return r;
            zm_count(modes, ZM_BLOCK_RAW + (int)type);
            if (skim) bound += type == 2 ? block_max : bsize;
            else if (type == 0) {
                if (COPY && op + bsize > out_cap) return r;
                lz_emit_literals<COPY>(out, op, in + ip, bsize, lane);
                op += bsize;
            } else if (type == 1) {
                if (COPY && op + bsize > out_cap) return r;
                zstd_emit_literals<COPY>(out, op, ZLIT_RLE, in + ip, 0, bsize, lane);
                op += bsize;
            } else if (!zstd_block<COPY>(in + ip, bsize, out, out_cap, op, frame_start, block_max, f, w, lane, modes)) return r;
            ip += csize;
            if (last) break;
        }
        if (skim) {
            if (fcs > bound) return r;
            op += fcs;
        } else if (has_fcs && op - frame_start != fcs) return r;
        if (checksum) {                              // XXH64 content checksum: not verified (check.crcs=false)
            if (n - ip < 4) return r;
            ip += 4;
        }
        frames = true;
    }
    KTA_INF_SYNC();
    r.out_len = op;
    r.ok = frames;
    return r;
}

}  // namespace kta
