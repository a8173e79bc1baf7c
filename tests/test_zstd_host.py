"""The zstd frame walk of the RecordBatch decoder (csrc/kta_zstd.cuh) on the host, compiled by nvcc with the address
sanitizer: the same statements the GPU runs per warp, against pyarrow's zstd compressor at levels that cover the fast,
lazy, btopt and btultra strategies, frames without a content size, skippable and concatenated frames, hand-made frames
for the rejections, and random damage — a damaged section must be rejected or decode to SOMETHING of the announced size,
never read or write outside its buffers (the harness allocates them at their exact sizes)."""
import ctypes
import ctypes.util
import os
import shutil
import struct
import subprocess

import numpy as np
import pytest

import kafka_codec as kc
import zstd_codec as zc

HERE = os.path.dirname(os.path.abspath(__file__))
NVCC = os.environ.get("NVCC") or "/usr/local/cuda/bin/nvcc"
LEVELS = (-5, 1, 3, 9, 19, 22)
# kta::ZstdMode, in order
MODES = ("FRAME SKIPPABLE SINGLE_SEGMENT WINDOW_DESC CHECKSUM FCS_NONE FCS_1 FCS_2 FCS_4 FCS_8 BLOCK_RAW BLOCK_RLE "
         "BLOCK_COMPRESSED LIT_RAW LIT_RLE LIT_COMPRESSED LIT_TREELESS LIT_HDR1 LIT_HDR2 LIT_HDR3 HUF_SF0 HUF_SF1 HUF_SF2 "
         "HUF_SF3 STREAMS1 STREAMS4 HUF_DIRECT HUF_FSE NSEQ0 NSEQ1 NSEQ2 NSEQ3 LL_PREDEF LL_RLE LL_FSE LL_REPEAT OF_PREDEF "
         "OF_RLE OF_FSE OF_REPEAT ML_PREDEF ML_RLE ML_FSE ML_REPEAT REP1 REP2 REP3 REP1_MINUS1 REP_LL0").split()
SKIPPABLE = struct.pack("<II", 0x184D2A53, 5) + b"skip!"


def zstd(data, level=3):
    import pyarrow as pa
    return pa.Codec("zstd", compression_level=level).compress(data, asbytes=True)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    nvcc = NVCC if os.path.exists(NVCC) else shutil.which("nvcc")
    if not nvcc:
        pytest.skip("nvcc not available")
    exe = str(tmp_path_factory.mktemp("zstd") / "zstd_harness")
    src = os.path.join(HERE, "native", "zstd_harness.cu")
    r = subprocess.run([nvcc, "-O1", "-g", "-std=c++17", "-Xcompiler", "-fsanitize=address,-fno-omit-frame-pointer", "-o", exe, src],
                       capture_output=True, text=True)
    if r.returncode != 0:        # no sanitizer runtime in this toolchain: the plain build still checks the results
        subprocess.run([nvcc, "-O1", "-std=c++17", "-o", exe, src], check=True, capture_output=True)
    return exe


def run_cases(exe, cases):
    """per case: (ok, size-pass length, full-walk length, bytes, {mode: count}); lengths are None when that pass rejected"""
    blob = b"".join(struct.pack("<I", len(d)) + d for d in cases)
    env = dict(os.environ, ASAN_OPTIONS="detect_leaks=0:protect_shadow_gap=0")
    r = subprocess.run([exe], input=blob, capture_output=True, env=env)
    assert r.returncode == 0, r.stderr.decode("utf-8", "replace")[-2000:]
    out, res, at = r.stdout, [], 0
    for _ in cases:
        ok, size_len, walk_len, n = out[at], *struct.unpack_from("<III", out, at + 1)
        data = out[at + 13:at + 13 + n]
        at += 13 + n
        counts = struct.unpack_from("<%dI" % len(MODES), out, at)
        at += 4 * len(MODES)
        none = lambda v: None if v == 0xFFFFFFFF else v
        res.append((bool(ok), none(size_len), none(walk_len), data, dict(zip(MODES, counts))))
    assert at == len(out)
    return res


def payloads():
    rng = np.random.default_rng(5)
    recs = b"".join(kc.encode_record(i, i, b"key-%d" % (i % 50), 30 + i % 9) for i in range(400))
    big = b"".join(kc.encode_record(i, i, bytes(rng.integers(0, 256, 16, dtype=np.uint8)), 200) for i in range(3000))  # > 128 KiB
    text = b"".join(b"%d: the quick brown fox %s over the lazy dog %d times\n" % (i, [b"jumps", b"leaps", b"hops"][i % 3], i * 7 % 13)
                    for i in range(6000))
    return {"empty": b"", "one": b"\x01", "records": recs, "big": big, "zeros": bytes(300_000),
            "random": rng.integers(0, 256, 20_000, dtype=np.uint8).tobytes(), "text": text}


def mode_payloads():
    """inputs that make the compressor use the rarer block / literal / sequence encodings"""
    rng = np.random.default_rng(8)
    letters = rng.choice(np.frombuffer(b"etaoinshrdlucmfw", np.uint8), 300_000).tobytes()      # Huffman only, no matches
    few = rng.choice(np.frombuffer(b"ab", np.uint8), 3000).tobytes()                            # small literal sections
    words = [bytes(rng.integers(97, 123, 4, dtype=np.uint8)) for _ in range(64)]
    wordy = b"".join(words[i] for i in rng.integers(0, 64, 100_000))                            # Treeless, repeat tables
    nib = rng.choice(np.arange(16, dtype=np.uint8), 50_000,                                     # direct Huffman weights
                     p=np.array([8, 1, 3, 1, 5, 1, 1, 2, 1, 1, 4, 1, 1, 1, 2, 7.]) / 40).tobytes()
    tri_words = [bytes(rng.integers(0, 256, 3, dtype=np.uint8)) for _ in range(512)]
    tri = b"".join(tri_words[i] for i in rng.integers(0, 512, 200_000))                         # > 32512 sequences a block
    base = rng.integers(0, 256, 131072, dtype=np.uint8).tobytes()
    parts = [base]
    for _ in range(4000):                                                                       # literals all 'q': RLE literals
        s = int(rng.integers(0, 131000))
        parts.append(b"q" + base[s:s + int(rng.integers(16, 40))])
    stutter = b"".join(b"x" * int(rng.integers(1, 6)) + b"y" * int(rng.integers(1, 6)) + bytes([int(rng.integers(97, 100))])
                       for _ in range(20000))                                                   # repeat offset rep1 - 1 (levels 19, 22)
    return {"letters": letters, "few": few, "wordy": wordy, "nib": nib, "tri": tri, "qlits": b"".join(parts), "stutter": stutter}


def frame_header(fhd, fcs=b"", wd=None):
    return b"\x28\xb5\x2f\xfd" + bytes([fhd]) + (bytes([wd]) if wd is not None else b"") + fcs


def crafted_block(offset_code, offset_extra, nbits):
    """one compressed block: Raw literals "ab", one sequence (LL 2, ML 3, offset from the given code) with all three
    tables in RLE mode, so the bit stream holds only the offset's extra bits and the padding sentinel"""
    body = bytes([0x10]) + b"ab" + bytes([0x01, 0x54, 0x02, offset_code, 0x00, (1 << nbits) | offset_extra])
    return struct.pack("<I", (len(body) << 3) | (2 << 1) | 1)[:3] + body


def good_crafted():    # "ab" + match (offset 2, length 3) = "ababa"; no content size, a 1 KiB window
    return frame_header(0x00, wd=0) + crafted_block(2, 1, 2)


def libzstd():
    name = ctypes.util.find_library("zstd")
    try:
        return ctypes.CDLL(name or "libzstd.so.1")
    except OSError:
        return None


def test_walk_matches_pyarrow_at_every_level(harness):
    cases, want = [], []
    for level in LEVELS:
        for name, data in payloads().items():
            cases.append(zstd(data, level))
            want.append(data)
    for (ok, size_len, walk_len, out, _), w in zip(run_cases(harness, cases), want):
        assert ok and out == w and size_len == walk_len == len(w)


def test_frames_without_content_size_and_header_variants(harness):
    """FCS absent (the size pass then decodes the sequences), an 8-byte FCS field, a content checksum, skippable frames and
    several frames in one section (outputs concatenated, as ZSTD_decompress does)"""
    p = payloads()
    cases, want = [], []
    for level in (1, 19):
        for name in ("one", "records", "big", "zeros", "random", "text"):
            f = zstd(p[name], level)
            cases += [zc.without_fcs(f), zc.without_fcs(f, fcs_bytes=8)]
            want += [p[name], p[name]]
    a, b = zstd(p["records"], 9), zc.without_fcs(zstd(p["text"], 3))
    cases += [a + SKIPPABLE + b, SKIPPABLE + a, a + a + b]
    want += [p["records"] + p["text"], p["records"], p["records"] * 2 + p["text"]]
    # checksum flag set by hand (the 4 bytes after the last block are skipped, not verified)
    f = zstd(p["records"], 3)
    cases.append(f[:4] + bytes([f[4] | 0x04]) + f[5:] + b"\xde\xad\xbe\xef")
    want.append(p["records"])
    res = run_cases(harness, cases)
    for (ok, size_len, walk_len, out, _), w in zip(res, want):
        assert ok and out == w and size_len == walk_len == len(w)
    seen = {m for *_, counts in res for m, c in counts.items() if c}
    assert {"FCS_NONE", "FCS_8", "WINDOW_DESC", "SKIPPABLE", "CHECKSUM"} <= seen


def test_every_decoding_mode_occurs(harness):
    """the inputs above (and the mode payloads) go through every block, literal and sequence encoding the decoder has"""
    cases = [zstd(d, level) for level in LEVELS for d in list(payloads().values()) + list(mode_payloads().values())]
    cases += [zc.without_fcs(zstd(payloads()["text"])), zc.without_fcs(zstd(b"x" * 100), 8),
              SKIPPABLE + zstd(b"abc") + b"\x00" * 0, good_crafted()]
    cases.append(cases[-1][:4] + bytes([cases[-1][4] | 4]) + cases[-1][5:] + b"\x00" * 4)
    res = run_cases(harness, cases)
    assert all(ok and size_len == walk_len for ok, size_len, walk_len, _, _ in res)
    total = {m: sum(r[4][m] for r in res) for m in MODES}
    assert [m for m, c in total.items() if c == 0] == []


def test_rejections(harness):
    f = zstd(payloads()["records"], 3)
    fhd = f[4]
    assert fhd >> 5 & 1 and fhd >> 6 == 1                # single segment, 2-byte FCS (content size - 256)
    fcs = int.from_bytes(f[5:7], "little")
    with_did = f[:4] + bytes([fhd | 1, 7]) + f[5:]       # Dictionary_ID 7
    hdr_end = 7
    bh = int.from_bytes(f[hdr_end:hdr_end + 3], "little")
    reserved = f[:hdr_end] + ((bh | 6).to_bytes(3, "little")) + f[hdr_end + 3:]   # block type 3
    plus = f[:5] + (fcs + 1).to_bytes(2, "little") + f[7:]
    minus = f[:5] + (fcs - 1).to_bytes(2, "little") + f[7:]
    before_start = zstd(b"0123456789") + frame_header(0x00, wd=0) + crafted_block(3, 0, 3)   # offset 5, 2 bytes into its frame
    cases = [with_did, reserved, plus, minus, before_start, f[:-1], f[:len(f) // 2], f[:6], f + b"\x28\xb5",
             frame_header(0x08, wd=0) + crafted_block(2, 1, 2),          # reserved header bit
             frame_header(0x00, wd=0) + crafted_block(3, 0, 3),          # offset before the (only) frame's start
             frame_header(0x20, b"\x05") + crafted_block(2, 1, 2),       # a 9-byte block in a 5-byte window
             b"", SKIPPABLE]                                             # no zstd frame at all
    res = run_cases(harness, cases)
    assert [ok for ok, *_ in res] == [False] * len(cases)
    # the crafted frame itself is fine
    (ok, size_len, walk_len, out, _), = run_cases(harness, [good_crafted()])
    assert ok and out == b"ababa" and size_len == walk_len == 5


def test_libzstd_agrees_when_available(harness):
    """extra cases from the system's libzstd, when one can be loaded: streaming-style frames without a content size and
    with a checksum; and libzstd decodes the header-rewritten and hand-made frames the tests above rely on"""
    lib = libzstd()
    if lib is None:
        pytest.skip("libzstd not loadable")
    lib.ZSTD_createCCtx.restype = ctypes.c_void_p
    lib.ZSTD_compress2.restype = ctypes.c_size_t
    lib.ZSTD_compress2.argtypes = [ctypes.c_void_p, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]
    lib.ZSTD_CCtx_setParameter.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]
    lib.ZSTD_freeCCtx.argtypes = [ctypes.c_void_p]
    lib.ZSTD_isError.argtypes = [ctypes.c_size_t]
    lib.ZSTD_decompress.restype = ctypes.c_size_t
    lib.ZSTD_decompress.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_char_p, ctypes.c_size_t]

    def compress(data, level):
        cctx = lib.ZSTD_createCCtx()
        for param, value in ((100, level), (200, 0), (201, 1)):   # level, contentSizeFlag=0, checksumFlag=1
            lib.ZSTD_CCtx_setParameter(cctx, param, value)
        buf = ctypes.create_string_buffer(len(data) + len(data) // 100 + 1024)
        n = lib.ZSTD_compress2(cctx, buf, len(buf), data, len(data))
        lib.ZSTD_freeCCtx(cctx)
        assert not lib.ZSTD_isError(n)
        return buf.raw[:n]

    def decompress(frame, size):
        buf = ctypes.create_string_buffer(max(size, 1))
        n = lib.ZSTD_decompress(buf, len(buf), frame, len(frame))
        return None if lib.ZSTD_isError(n) else buf.raw[:n]

    p = payloads()
    cases, want = [], []
    for level in (1, 9, 19):
        for name in ("records", "big", "text", "random"):
            cases.append(compress(p[name], level))
            want.append(p[name])
    res = run_cases(harness, cases)
    for (ok, size_len, walk_len, out, counts), w in zip(res, want):
        assert ok and out == w and size_len == walk_len == len(w) and counts["FCS_NONE"] and counts["CHECKSUM"]
    rewritten = zc.without_fcs(zstd(p["text"], 19))
    assert decompress(rewritten, len(p["text"])) == p["text"]
    assert decompress(zstd(p["one"]) + SKIPPABLE + rewritten, len(p["text"]) + 1) == p["one"] + p["text"]
    assert decompress(good_crafted(), 5) == b"ababa"


def test_damaged_sections_never_leave_their_buffers(harness):
    """Bit flips, truncations and spliced garbage: the harness runs under the address sanitizer with exact-size buffers, so
    any read past the input or write past the size pass's length ends the process with a report."""
    rng = np.random.default_rng(9)
    p = payloads()
    goods = [zstd(p["records"], 1), zstd(p["records"], 19), zc.without_fcs(zstd(p["text"][:40_000], 9)),
             zstd(p["big"][:150_000], 3), zstd(mode_payloads()["nib"][:5000], 3)]
    cases = []
    for good in goods:
        for _ in range(220):
            b = bytearray(good)
            kind = int(rng.integers(0, 4))
            if kind == 0:
                for _ in range(int(rng.integers(1, 3))):
                    b[int(rng.integers(0, len(b)))] ^= 1 << int(rng.integers(0, 8))
            elif kind == 1:
                b = b[: int(rng.integers(0, len(b)))]
            elif kind == 2:
                at = int(rng.integers(0, len(b)))
                b[at:at + 4] = bytes(rng.integers(0, 256, 4, dtype=np.uint8))
            else:
                b += bytes(rng.integers(0, 256, int(rng.integers(1, 9)), dtype=np.uint8))
            cases.append(bytes(b))
    res = run_cases(harness, cases)                 # returncode 0 = no sanitizer report, no crash
    assert len(res) == len(cases)
    rejected = 0
    for ok, size_len, _, out, _ in res:
        if ok:
            assert len(out) == size_len
        rejected += not ok
    assert rejected > len(cases) // 2
