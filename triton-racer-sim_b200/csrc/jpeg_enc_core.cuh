// jpeg_enc_core.cuh — baseline JPEG encoding arithmetic for tub records, written once for host and device.
//
// Replaces `Image.fromarray(img).save(path)` in the reference's recorder (TritonRacerSim/components/datastorage.py:78) and
// `cv2.imwrite` in utils/post_process.py: Pillow / OpenCV -> libjpeg(-turbo) with its default compression settings (baseline
// sequential, 8 bit, YCbCr 4:2:0, one interleaved scan, standard Huffman tables, no restart intervals).  Every stage restates the
// published libjpeg algorithm that default path runs, bit for bit:
//   quantisation tables       jcparam.c jpeg_set_quality / jpeg_add_quant_table (Annex K tables, libjpeg quality scaling)
//   colour conversion         jccolor.c rgb_ycc_convert (16-bit fixed point)
//   edge padding, 4:2:0       jcprepct.c (row / column replication), jcsample.c h2v2_downsample (bias 1, 2, 1, 2, ...)
//   forward DCT               jfdctint.c jpeg_fdct_islow (CONST_BITS 13, PASS1_BITS 2; output scaled by 8)
//   quantisation              jcdctmgr.c (divisor 8q, rounding half away from zero)
//   entropy coding            jchuff.c encode_one_block (Annex K.3 tables, ZRL, EOB), byte stuffing, 1-bit padding
//   headers                   jcmarker.c (SOI, APP0 JFIF 1.01, DQT, SOF0, DHT, SOS)
// The functions are pure (memory in, memory out, no threads), so the same source is compiled by nvcc into the kernels
// (jpeg_enc_kernels.cuh) and by g++ into a host-side check against Pillow (tests/test_jpeg_encode_host.py).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define TRS_JEHD __host__ __device__ __forceinline__
#else
#define TRS_JEHD inline
#endif

namespace trs {

// bytes of the headers trs_jpe_build_header writes (they depend on nothing but h, w and the quality): SOI 2, APP0 18, 2 x DQT 69,
// SOF0 19, DHT 33 + 183 + 33 + 183, SOS 14
enum { JPE_HEADER_BYTES = 623, JPE_MAX_BLOCK_BITS = 1664 };

// zigzag position k -> natural index (jutils.c jpeg_natural_order); a function so host and device code share one definition
TRS_JEHD int jpe_natural(int k)
{
    constexpr uint8_t t[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                               41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                               30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};
    return t[k];
}

// ---- tables (Annex K) -------------------------------------------------------------------------------------------------------
struct JpeStdTables {
    uint8_t luma_q[64], chroma_q[64];                      // K.1 / K.2, natural order
    uint8_t dc_bits[2][16], dc_vals[2][12];                // K.3: [0] luma, [1] chroma
    uint8_t ac_bits[2][16], ac_vals[2][162];
};

inline const JpeStdTables& jpe_std_tables()
{
    static const JpeStdTables T = {
        {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,  14, 13, 16, 24, 40,  57,  69,  56,
         14, 17, 22, 29, 51,  87,  80,  62,  18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
         49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99},
        {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99, 24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
         99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99},
        {{0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0}, {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0}},
        {{0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}, {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11}},
        {{0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d}, {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77}},
        {{0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81,
          0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18,
          0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48,
          0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75,
          0x76, 0x77, 0x78, 0x79, 0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99,
          0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
          0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5,
          0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa},
         {0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08,
          0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25,
          0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47,
          0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74,
          0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97,
          0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
          0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4,
          0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa}},
    };
    return T;
}

// Everything the block coder needs for one quality, in the form the kernels keep in shared memory.
//   div / recip: quantisation divisor 8q (natural order) and floor(2^32 / div) + 1, so that x / div == (x * recip) >> 32 exactly
//                for every x < 2^16 (the numerators here stay below 2^15 + 2^10; the CPU test checks the identity exhaustively)
//   dc / ac:     Huffman code of every symbol, (length << 16) | code (jchuff.c jpeg_make_c_derived_tbl); length 0 = no code
struct JpeEncTables {
    uint32_t div[2][64];
    uint32_t recip[2][64];
    uint32_t dc[2][16];
    uint32_t ac[2][256];
};

// jcparam.c jpeg_quality_scaling + jpeg_add_quant_table (force_baseline): one quantisation step, 1..255
inline int jpe_quant_step(int base, int quality)
{
    const int s = quality < 50 ? 5000 / quality : 200 - 2 * quality;
    long v = ((long)base * s + 50) / 100;
    return v < 1 ? 1 : (v > 255 ? 255 : (int)v);
}

inline void jpe_make_codes(const uint8_t* bits, const uint8_t* vals, uint32_t* out, int n_out)
{
    for (int i = 0; i < n_out; ++i) out[i] = 0;
    uint32_t code = 0;
    int k = 0;
    for (int l = 1; l <= 16; ++l) {
        for (int i = 0; i < bits[l - 1]; ++i, ++k, ++code) out[vals[k]] = ((uint32_t)l << 16) | code;
        code <<= 1;
    }
}

inline void jpe_make_tables(int quality, JpeEncTables& T)
{
    const JpeStdTables& S = jpe_std_tables();
    for (int c = 0; c < 2; ++c) {
        for (int i = 0; i < 64; ++i) {
            const uint32_t d = 8u * (uint32_t)jpe_quant_step(c ? S.chroma_q[i] : S.luma_q[i], quality);
            T.div[c][i] = d;
            T.recip[c][i] = (uint32_t)((1ull << 32) / d + 1);
        }
        jpe_make_codes(S.dc_bits[c], S.dc_vals[c], T.dc[c], 16);
        jpe_make_codes(S.ac_bits[c], S.ac_vals[c], T.ac[c], 256);
    }
}

// ---- headers (jcmarker.c write_file_header / write_frame_header / write_scan_header) --------------------------------------
// writes JPE_HEADER_BYTES bytes to `out`, returns that count
inline int jpe_build_header(int h, int w, int quality, uint8_t* out)
{
    const JpeStdTables& S = jpe_std_tables();
    int n = 0;
    auto b = [&](int v) { out[n++] = (uint8_t)v; };
    auto b2 = [&](int v) { b(v >> 8); b(v & 0xff); };
    b2(0xffd8);                                                                      // SOI
    b2(0xffe0); b2(16);                                                              // APP0 JFIF 1.01, no units, density 1x1, no thumbnail
    b('J'); b('F'); b('I'); b('F'); b(0); b(1); b(1); b(0); b2(1); b2(1); b(0); b(0);
    for (int c = 0; c < 2; ++c) {                                                    // DQT, 8-bit precision, zigzag order
        b2(0xffdb); b2(67); b(c);
        for (int k = 0; k < 64; ++k) b(jpe_quant_step(c ? S.chroma_q[jpe_natural(k)] : S.luma_q[jpe_natural(k)], quality));
    }
    b2(0xffc0); b2(17); b(8); b2(h); b2(w); b(3);                                     // SOF0: Y 2x2 table 0, Cb / Cr 1x1 table 1
    b(1); b(0x22); b(0); b(2); b(0x11); b(1); b(3); b(0x11); b(1);
    for (int t = 0; t < 4; ++t) {                                                    // DHT: DC0, AC0, DC1, AC1
        const int c = t >> 1, ac = t & 1;
        const uint8_t* bits = ac ? S.ac_bits[c] : S.dc_bits[c];
        const uint8_t* vals = ac ? S.ac_vals[c] : S.dc_vals[c];
        int nv = 0;
        for (int l = 0; l < 16; ++l) nv += bits[l];
        b2(0xffc4); b2(2 + 1 + 16 + nv); b((ac << 4) | c);
        for (int l = 0; l < 16; ++l) b(bits[l]);
        for (int i = 0; i < nv; ++i) b(vals[i]);
    }
    b2(0xffda); b2(12); b(3); b(1); b(0x00); b(2); b(0x11); b(3); b(0x11); b(0); b(63); b(0);     // SOS
    return n;
}

// ---- samples -----------------------------------------------------------------------------------------------------------------
// jccolor.c rgb_ycc_convert: FIX(x) = (int)(x * 65536 + 0.5); Cb / Cr carry CBCR_OFFSET and ONE_HALF - 1
TRS_JEHD void jpe_rgb_to_ycc(int r, int g, int b, int& y, int& cb, int& cr)
{
    y = (19595 * r + 38470 * g + 7471 * b + 32768) >> 16;
    cb = (-11059 * r - 21709 * g + 32768 * b + (128 << 16) + 32767) >> 16;
    cr = (32768 * r - 27439 * g - 5329 * b + (128 << 16) + 32767) >> 16;
}

// jcsample.c h2v2_downsample: four samples of a 2x2 group, chroma column cx of the output row (bias 1 for even, 2 for odd columns)
TRS_JEHD int jpe_h2v2(int a, int b, int c, int d, int cx) { return (a + b + c + d + 1 + (cx & 1)) >> 2; }

// ---- jfdctint.c jpeg_fdct_islow: in place over 64 centred samples (natural order); outputs scaled up by 8 ---------------------
TRS_JEHD void jpe_fdct_islow(int (&d)[64])
{
    const int CB = 13, P1 = 2;
    const int F_0_298631336 = 2446, F_0_390180644 = 3196, F_0_541196100 = 4433, F_0_765366865 = 6270, F_0_899976223 = 7373,
              F_1_175875602 = 9633, F_1_501321110 = 12299, F_1_847759065 = 15137, F_1_961570560 = 16069, F_2_053119869 = 16819,
              F_2_562915447 = 20995, F_3_072711026 = 25172;
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
        const int step = pass ? 8 : 1, stride = pass ? 1 : 8;          // pass 1 over rows, pass 2 over columns
        const int sh = pass ? CB + P1 : CB - P1;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            int* p = d + i * stride;
            const int tmp0 = p[0] + p[7 * step], tmp7 = p[0] - p[7 * step];
            const int tmp1 = p[step] + p[6 * step], tmp6 = p[step] - p[6 * step];
            const int tmp2 = p[2 * step] + p[5 * step], tmp5 = p[2 * step] - p[5 * step];
            const int tmp3 = p[3 * step] + p[4 * step], tmp4 = p[3 * step] - p[4 * step];
            const int tmp10 = tmp0 + tmp3, tmp13 = tmp0 - tmp3, tmp11 = tmp1 + tmp2, tmp12 = tmp1 - tmp2;
            if (pass == 0) {
                p[0] = (tmp10 + tmp11) * (1 << P1);
                p[4 * step] = (tmp10 - tmp11) * (1 << P1);
            } else {
                p[0] = (tmp10 + tmp11 + (1 << (P1 - 1))) >> P1;
                p[4 * step] = (tmp10 - tmp11 + (1 << (P1 - 1))) >> P1;
            }
            const int rnd = 1 << (sh - 1);
            int z1 = (tmp12 + tmp13) * F_0_541196100;
            p[2 * step] = (z1 + tmp13 * F_0_765366865 + rnd) >> sh;
            p[6 * step] = (z1 - tmp12 * F_1_847759065 + rnd) >> sh;
            z1 = tmp4 + tmp7;
            int z2 = tmp5 + tmp6, z3 = tmp4 + tmp6, z4 = tmp5 + tmp7;
            const int z5 = (z3 + z4) * F_1_175875602;
            const int t4 = tmp4 * F_0_298631336, t5 = tmp5 * F_2_053119869, t6 = tmp6 * F_3_072711026, t7 = tmp7 * F_1_501321110;
            z1 *= -F_0_899976223; z2 *= -F_2_562915447; z3 *= -F_1_961570560; z4 *= -F_0_390180644;
            z3 += z5; z4 += z5;
            p[7 * step] = (t4 + z1 + z3 + rnd) >> sh;
            p[5 * step] = (t5 + z2 + z4 + rnd) >> sh;
            p[3 * step] = (t6 + z2 + z3 + rnd) >> sh;
            p[step] = (t7 + z1 + z4 + rnd) >> sh;
        }
    }
}

// jcdctmgr.c quantisation: sign(c) * ((|c| + d/2) / d), the division as a multiplication by the reciprocal
TRS_JEHD int jpe_quantise(int c, uint32_t div, uint32_t recip)
{
    const uint32_t a = (uint32_t)(c < 0 ? -c : c) + (div >> 1);
    const int q = (int)(((uint64_t)a * recip) >> 32);
    return c < 0 ? -q : q;
}

// bits needed for |v| (jchuff.c: nbits of the magnitude category)
TRS_JEHD int jpe_nbits(int v)
{
    uint32_t a = (uint32_t)(v < 0 ? -v : v);
    int n = 0;
    while (a) { ++n; a >>= 1; }
    return n;
}

// ---- jchuff.c encode_one_block over a sink with put(bits, count) ------------------------------------------------------------
// zz: quantised coefficients in zigzag order (zz[0] unused: the DC difference to the component's predictor is `diff`).
// The same template gives the bit count (JpeCountSink) and the bits themselves, so the two can never disagree.
template <class Sink>
TRS_JEHD void jpe_encode_block(const int (&zz)[64], int diff, const uint32_t* dc, const uint32_t* ac, Sink& s)
{
    int nb = jpe_nbits(diff);
    s.put(dc[nb] & 0xffffu, (int)(dc[nb] >> 16));
    if (nb) s.put((uint32_t)(diff < 0 ? diff - 1 : diff) & ((1u << nb) - 1u), nb);
    int run = 0;
#pragma unroll
    for (int k = 1; k < 64; ++k) {
        const int v = zz[k];
        if (v == 0) { ++run; continue; }
        while (run > 15) { s.put(ac[0xf0] & 0xffffu, (int)(ac[0xf0] >> 16)); run -= 16; }
        nb = jpe_nbits(v);
        const uint32_t e = ac[(run << 4) | nb];
        s.put(e & 0xffffu, (int)(e >> 16));
        s.put((uint32_t)(v < 0 ? v - 1 : v) & ((1u << nb) - 1u), nb);
        run = 0;
    }
    if (run) s.put(ac[0] & 0xffffu, (int)(ac[0] >> 16));
}

struct JpeCountSink {
    uint32_t bits = 0;
    TRS_JEHD void put(uint32_t, int n) { bits += (uint32_t)n; }
};

// The sequential bit emitter of jchuff.c (emit_bits + flush_bits): MSB first, a 0x00 after every 0xFF byte, the last byte padded
// with 1-bits.  Host form (the kernels place a block's bits at its scanned offset and stuff in a separate pass; same bytes).
struct JpeByteWriter {
    uint8_t* out;
    uint64_t n = 0;
    uint64_t acc = 0;
    int nacc = 0;
    void put(uint32_t v, int len)
    {
        acc = (acc << len) | (v & ((1u << len) - 1u));
        nacc += len;
        while (nacc >= 8) {
            const uint8_t b = (uint8_t)(acc >> (nacc - 8));
            nacc -= 8;
            out[n++] = b;
            if (b == 0xff) out[n++] = 0;
        }
        acc &= (1ull << nacc) - 1;
    }
    void flush() { if (nacc) put(0x7f, 8 - nacc); }
};

// image geometry of the 4:2:0 encoding
struct JpeGeom {
    int h, w;
    int mw, mh;        // MCUs (16 x 16 pixels) per row / column; also the chroma block counts
    int ybw, ybh;      // luma blocks inside the component's extent (ceil(w/8), ceil(h/8)); blocks beyond are dummy blocks
    int ch;            // chroma rows before block padding, ceil(h/2)
};

TRS_JEHD JpeGeom jpe_geom(int h, int w)
{
    JpeGeom g;
    g.h = h; g.w = w;
    g.mw = (w + 15) / 16; g.mh = (h + 15) / 16;
    g.ybw = (w + 7) / 8; g.ybh = (h + 7) / 8;
    g.ch = (h + 1) / 2;
    return g;
}

// Samples of block `sub` (0..3 luma in raster order, 4 Cb, 5 Cr) of MCU (my, mx), centred, natural order, from the MCU's 16 x 16
// Y / Cb / Cr tile at full resolution (pixel (r, c) of the tile = image pixel (min(16 my + r, h - 1), min(16 mx + c, w - 1)):
// jcprepct.c's replication).  Chroma rows beyond ceil(h/2) repeat the last real chroma row (the 2x2 groups of rows 2 ch - 2, 2 ch - 1);
// chroma columns need no such rule (the tile is already replicated out to 16 mw columns).
TRS_JEHD void jpe_block_samples(const uint8_t* ty, const uint8_t* tcb, const uint8_t* tcr, int tile_stride, const JpeGeom& g, int my,
                                int sub, int (&d)[64])
{
    if (sub < 4) {
        const int r0 = (sub >> 1) * 8, c0 = (sub & 1) * 8;
#pragma unroll
        for (int r = 0; r < 8; ++r)
#pragma unroll
            for (int c = 0; c < 8; ++c) d[r * 8 + c] = (int)ty[(r0 + r) * tile_stride + c0 + c] - 128;
        return;
    }
    const uint8_t* t = sub == 4 ? tcb : tcr;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
        const int cy = my * 8 + r < g.ch ? r : g.ch - 1 - my * 8;        // replicate the last real chroma row
        const uint8_t* p = t + 2 * cy * tile_stride;
#pragma unroll
        for (int c = 0; c < 8; ++c)
            d[r * 8 + c] = jpe_h2v2(p[2 * c], p[2 * c + 1], p[tile_stride + 2 * c], p[tile_stride + 2 * c + 1], c) - 128;
    }
}

// samples -> quantised zigzag coefficients (zz[0] = quantised DC)
TRS_JEHD void jpe_block_coefficients(int (&d)[64], const uint32_t* div, const uint32_t* recip, int (&zz)[64])
{
    jpe_fdct_islow(d);
#pragma unroll
    for (int k = 0; k < 64; ++k) {
        const int i = jpe_natural(k);
        zz[k] = jpe_quantise(d[i], div[i], recip[i]);
    }
}

// is luma block `sub` of MCU (my, mx) outside the component's block extent (jccoefct.c compress_data: a dummy block with AC 0 and
// the DC of the block before it in MCU order)?
TRS_JEHD bool jpe_dummy(const JpeGeom& g, int my, int mx, int sub)
{
    return sub < 4 && (2 * mx + (sub & 1) >= g.ybw || 2 * my + (sub >> 1) >= g.ybh);
}

}  // namespace trs
