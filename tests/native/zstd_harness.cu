// TEST INFRASTRUCTURE: the zstd frame walk of the RecordBatch decoder (csrc/kta_zstd.cuh: the __host__ __device__
// statements log_zstd_size_kernel and log_decompress_kernel run on the GPU) on the host, one "lane".
// stdin: cases of u32 length + bytes.  stdout per case: u8 ok, u32 size-pass length (Frame_Content_Size trusted within its
// bound, as the size kernel does), u32 length of the size-only walk that decodes every frame, u32 length, bytes, then
// ZM_COUNT u32 counts of the decoding modes the copy pass went through.  The output buffer is allocated at exactly the
// size pass's length, so that an overrun of the copy pass is a heap overflow an address-sanitizer build reports.
#include <cstdio>
#include <cstdint>
#include <cstdlib>
#include <cstring>

#include "../../kafka_topic_analyzer_b200/csrc/kta_logdecode.cuh"

int main() {
    uint32_t n;
    kta::ZstdWork *w = (kta::ZstdWork *)malloc(sizeof(kta::ZstdWork));
    while (fread(&n, 4, 1, stdin) == 1) {
        // exact-size heap copies: reads past the input are heap overflows too
        uint8_t *in = (uint8_t *)malloc(n ? n : 1);
        if (n && fread(in, 1, n, stdin) != n) return 2;
        uint32_t modes[kta::ZM_COUNT] = {};
        const kta::LzWalk size = kta::zstd_walk<false>(in, n, nullptr, 0, *w, 0, true);
        const kta::LzWalk walk = kta::zstd_walk<false>(in, n, nullptr, 0, *w, 0, false);
        kta::LzWalk copy{0, false};
        uint8_t *out = (uint8_t *)malloc(size.ok && size.out_len ? size.out_len : 1);
        if (size.ok && size.out_len <= (64u << 20)) copy = kta::zstd_walk<true>(in, n, out, size.out_len, *w, 0, false, modes);
        const uint8_t okb = size.ok && copy.ok && copy.out_len == size.out_len ? 1 : 0;
        const uint32_t sl = size.ok ? (uint32_t)size.out_len : 0xffffffffu, wl = walk.ok ? (uint32_t)walk.out_len : 0xffffffffu;
        const uint32_t len = okb ? (uint32_t)copy.out_len : 0;
        fwrite(&okb, 1, 1, stdout);
        fwrite(&sl, 4, 1, stdout);
        fwrite(&wl, 4, 1, stdout);
        fwrite(&len, 4, 1, stdout);
        if (len) fwrite(out, 1, len, stdout);
        fwrite(modes, 4, kta::ZM_COUNT, stdout);
        free(out);
        free(in);
    }
    free(w);
    return 0;
}
