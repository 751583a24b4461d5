// Host build of the product's JPEG encoding arithmetic (csrc/jpeg_enc_core.cuh is pure host/device functions) for the CPU-side
// parity test against Pillow (tests/test_jpeg_encode_host.py).  Test infrastructure: mirrors the MCU loop of k_jpeg_encode one
// record at a time, with the sequential bit emitter in place of the kernel's scan-placed bits and separate stuffing pass.
#include <stdlib.h>
#include <string.h>

#include "../triton-racer-sim_b200/csrc/jpeg_enc_core.cuh"
using namespace trs;

// worst-case file size of an h x w record: headers, every block at its bit bound with every byte stuffed, padding, EOI
extern "C" unsigned long long jpe_max_bytes_host(int h, int w)
{
    const JpeGeom g = jpe_geom(h, w);
    return JPE_HEADER_BYTES + 2ull * ((unsigned long long)g.mw * g.mh * 6 * JPE_MAX_BLOCK_BITS / 8) + 2 + 2;
}

// rgb: h x w x 3; returns the file size, or 0 if `cap` is too small or the arguments are out of range
extern "C" unsigned long long jpe_encode_host(const uint8_t* rgb, int h, int w, int quality, uint8_t* out, unsigned long long cap)
{
    if (h < 1 || w < 1 || h > 65535 || w > 65535 || quality < 1 || quality > 100 || cap < jpe_max_bytes_host(h, w)) return 0;
    JpeEncTables T;
    jpe_make_tables(quality, T);
    const int hl = jpe_build_header(h, w, quality, out);
    JpeByteWriter bw{out + hl};
    const JpeGeom g = jpe_geom(h, w);
    uint8_t ty[256], tcb[256], tcr[256];
    int last[3] = {0, 0, 0};
    for (int my = 0; my < g.mh; ++my)
        for (int mx = 0; mx < g.mw; ++mx) {
            for (int r = 0; r < 16; ++r)
                for (int c = 0; c < 16; ++c) {
                    const int y = my * 16 + r < h ? my * 16 + r : h - 1, x = mx * 16 + c < w ? mx * 16 + c : w - 1;
                    const uint8_t* p = rgb + ((size_t)y * w + x) * 3;
                    int Y, Cb, Cr;
                    jpe_rgb_to_ycc(p[0], p[1], p[2], Y, Cb, Cr);
                    ty[r * 16 + c] = (uint8_t)Y; tcb[r * 16 + c] = (uint8_t)Cb; tcr[r * 16 + c] = (uint8_t)Cr;
                }
            for (int sub = 0; sub < 6; ++sub) {
                const int comp = sub < 4 ? 0 : sub - 3, t = comp ? 1 : 0;
                int zz[64];
                if (jpe_dummy(g, my, mx, sub)) {
                    for (int k = 0; k < 64; ++k) zz[k] = 0;
                    zz[0] = last[0];                                      // DC of the block before it, AC 0
                } else {
                    int d[64];
                    jpe_block_samples(ty, tcb, tcr, 16, g, my, sub, d);
                    jpe_block_coefficients(d, T.div[t], T.recip[t], zz);
                }
                jpe_encode_block(zz, zz[0] - last[comp], T.dc[t], T.ac[t], bw);
                last[comp] = zz[0];
            }
        }
    bw.flush();
    uint8_t* e = out + hl + bw.n;
    e[0] = 0xff; e[1] = 0xd9;
    return (unsigned long long)(hl + bw.n + 2);
}

// block bit counts of the count sink against the emitted bits, and the reciprocal quantisation against a division, exhaustively:
// every divisor 8q (q = 1..255) and every numerator below 2^16.  Returns 0 when all agree.
extern "C" int jpe_self_check_host(void)
{
    for (uint32_t q = 1; q <= 255; ++q) {
        const uint32_t d = 8 * q, r = (uint32_t)((1ull << 32) / d + 1);
        for (uint32_t x = 0; x < (1u << 16); ++x)
            if ((uint32_t)(((uint64_t)x * r) >> 32) != x / d) return 1;
    }
    return 0;
}
