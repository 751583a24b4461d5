// Sanitizer run of the product's JPEG encoding arithmetic (csrc/jpeg_enc_core.cuh) built for the host (tests/test_jpeg_encode_host.py):
// random sizes, qualities and frames (noise, flat, checkerboards) through the encoder into a buffer of exactly the worst-case size,
// then through the product's own parser and decoder (csrc/jpeg_core.cuh + jpeg_host.h), which must accept every file.
#include <stdio.h>
#include <stdlib.h>
#include <vector>

#include "../triton-racer-sim_b200/csrc/jpeg_core.cuh"
#include "../triton-racer-sim_b200/csrc/jpeg_host.h"
#include "host_jpeg_encode_check.cpp"

int main(int argc, char** argv)
{
    const int runs = argc > 1 ? atoi(argv[1]) : 300;
    uint64_t s = 12345;
    auto rnd = [&]() { s = s * 6364136223846793005ull + 1442695040888963407ull; return (uint32_t)(s >> 33); };
    size_t total = 0;
    for (int i = 0; i < runs; ++i) {
        const int h = 1 + rnd() % (i % 4 ? 70 : 260), w = 1 + rnd() % (i % 4 ? 90 : 330), q = 1 + rnd() % 100, kind = rnd() % 4;
        std::vector<uint8_t> img((size_t)h * w * 3);
        for (size_t k = 0; k < img.size(); ++k) {
            const size_t px = k / 3, y = px / w, x = px % w;
            img[k] = kind == 0 ? (uint8_t)rnd() : kind == 1 ? (uint8_t)(i * 37) : kind == 2 ? (uint8_t)(((x + y) & 1) * 255) : (uint8_t)(x * 7 + y * 3 + k % 3 * 50);
        }
        std::vector<uint8_t> out((size_t)jpe_max_bytes_host(h, w));
        const unsigned long long n = jpe_encode_host(img.data(), h, w, q, out.data(), out.size());
        if (n == 0) { printf("encode failed %dx%d q%d\n", h, w, q); return 1; }
        JpegTables T;
        JpegScan S;
        if (jpg_parse(out.data(), (size_t)n, &T, &S) || S.h != h || S.w != w || S.hs != 2 || S.vs != 2) {
            printf("parse failed %dx%d q%d\n", h, w, q);
            return 1;
        }
        // entropy-decode every block: the scan must hold exactly the blocks of the frame
        JpegBits b{out.data() + S.data_off, out.data() + S.data_off + S.data_len, 0, 0};
        const int mw = (w + 15) / 16, mh = (h + 15) / 16;
        int dc[3] = {0, 0, 0}, err = 0;
        int16_t coef[64];
        for (int m = 0; m < mw * mh && !err; ++m)
            for (int k = 0; k < 6; ++k) jpg_decode_block(b, k < 4 ? T.dc[0] : T.dc[1], k < 4 ? T.ac[0] : T.ac[1], dc[k < 4 ? 0 : k - 3], coef, err);
        if (err) { printf("decode failed %dx%d q%d\n", h, w, q); return 1; }
        total += (size_t)n;
    }
    printf("runs %d bytes %zu\n", runs, total);
    return 0;
}
