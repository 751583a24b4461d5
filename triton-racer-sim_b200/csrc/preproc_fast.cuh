// preproc_fast.cuh — frame-resident fast paths of the fused observation kernel (sm_100a).
//
// Same contract as k_preprocess (preproc_kernel.cuh) for frames that (a) fit shared memory whole, (b) have a
// width that is a multiple of 32 and (c) are 16-byte aligned.  Two kernels share the phase code below:
//
//  k_preprocess_fast one frame per CTA, two CTAs per SM, phases separated by __syncthreads.
//  k_preprocess_sw   the same plus store warps that take the output phase off the compute warps' critical path
//                    (every output channel a bit plane, edge filter on).
//  (A front/back warp-specialised kernel with double-buffered frames lived here until round 1 and measured slower:
//   see profiles/r01_phase_costs.md.)
//
// Common design points (DESIGN.md §kernels):
//  * a thread owns a 4-pixel-wide column strip and walks down its segment of rows with a rolling 3-row window in
//    registers; two adjacent lanes make one byte (8 pixels) of a bit plane with a single shuffle
//  * the Sobel arithmetic runs two pixels per instruction on the FMA pipe: a u8 value zero-extended to 16 bits is a
//    valid fp16 subnormal (n * 2^-24) and every intermediate stays below 2048, so HADD2/HFMA2 on the raw bit patterns
//    are exact integer add/sub/scale with free |x| and -x operand modifiers (results are sign-magnitude); HSET2 on
//    the same patterns gives the packed compares of the range tests and of the non-maximum suppression
//  * HSV: max/min/delta and the hue numerator are computed packed (VIMNMX3.U16x2, IADD3); the two fixed-point
//    multiplies per pixel stay scalar (IMAD) — bit-exact with OpenCV's integer path
//  * colour masks, NMS candidates and strong pixels live as bit planes; hysteresis is a word-parallel flood fill
//  * outputs are written once: u8 bytes expanded from plane nibbles by multiply-spread, f32 as bit * 0x3f800000
//    (masks are exactly 0.0 / 1.0 after /255)
//  * every shared-memory access in the hot loops goes through explicit ld.shared / st.shared on 32-bit window
//    addresses derived from ONE laundered base register: letting the compiler re-derive the window base costs a
//    S2R SR_CgaCtaId (long-scoreboard latency) inside every loop it decides to rematerialise it in
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "pixel_math.cuh"
#include "preproc_kernel.cuh"

namespace trs {

enum { FAST_MAX_THREADS = 320, WS_MAX_THREADS = 640, WS_MAX_WARPS = 20 };

struct FastGeom {
    int ws;                          // 1: warp-specialised layout (double buffers)
    int nsg;                         // strip groups per row (w / 32)
    int front_warps, back_warps;     // ws: warps per role; resident kernel: front == back == all warps
    int seg_rows_front, seg_rows_back;
    int threads;
    int mag_stride;                  // u16 elements per magnitude row (w + 4; pixel x at index x + 4, the zero to the right of a row is
                                     // element 0 of the next row)
    int mask_sets;                   // 2: the colour-mask planes are double-buffered by frame parity (store-warp kernel)
    int plane_bytes;                 // one bit plane incl. a zero row above and below, 16-byte multiple
    int off_pix[2], off_mag[2], off_mask, off_cand, off_edge, off_edge2, off_sdiv, off_hue, off_lut, off_bar, off_red, total;
    int band_h, n_bands;             // banded kernel: image rows per band (band_h == h: the whole frame is resident)
    int seg_rows_nms;                // banded kernel: rows per segment of the NMS walk (the strip walk also covers one row above and below)
    int tail_bytes;                  // store-warp layout: the last tail_bytes of the frame arrive by a second, later bulk copy (their
                                     // space holds the candidate plane during NMS + hysteresis); 0 = one copy
};

__host__ __device__ inline FastGeom fast_geometry(int h, int w, int n_ranges, int ws, int front_warps, int back_warps, int mask_sets = 1, int band_h = 0)
{
    FastGeom g;
    g.ws = ws;
    g.nsg = w / 32;
    g.front_warps = front_warps;
    g.back_warps = back_warps;
    const int fsegs = 4 * (front_warps / g.nsg), bsegs = 4 * (back_warps / g.nsg);
    if (band_h <= 0 || band_h >= h) { band_h = h; g.n_bands = 1; } else { g.n_bands = (h + band_h - 1) / band_h; }
    g.band_h = band_h;
    const int mag_rows = g.n_bands == 1 ? h : band_h + 2;              // magnitude rows a band's strip walk produces
    const int pix_rows = g.n_bands == 1 ? h : band_h + 4;              // pixel rows it reads
    g.seg_rows_front = (mag_rows + fsegs - 1) / fsegs;
    g.seg_rows_back = (h + bsegs - 1) / bsegs;
    g.seg_rows_nms = (band_h + fsegs - 1) / fsegs;
    g.threads = 32 * (ws ? front_warps + back_warps : front_warps);
    g.mag_stride = w + 4;
    g.mask_sets = mask_sets;
    g.plane_bytes = (((h + 2) * g.nsg * 4) + 15) & ~15;
    const int pix = ((pix_rows * w * 3 + 15) & ~15) + 16;
    const int mag = ((((mag_rows + 2) * g.mag_stride + 4) * 2) + 15) & ~15;
    int o = 16;                                                        // the strip walk reads the word LEFT of every row start unconditionally
    for (int b = 0; b < (ws ? 2 : 1); ++b) { g.off_pix[b] = o; o += pix; }
    for (int b = 0; b < (ws ? 2 : 1); ++b) { g.off_mag[b] = o; o += mag; }
    if (!ws) { g.off_pix[1] = g.off_pix[0]; g.off_mag[1] = g.off_mag[0]; }
    g.off_mask = o; o += g.plane_bytes * n_ranges * mask_sets;
    g.tail_bytes = 0;
    g.off_edge2 = -1;
    if (mask_sets == 2 && g.n_bands == 1 && ((h * w * 3) % 16) == 0 && h * w * 3 > 2 * g.plane_bytes) {
        g.tail_bytes = g.plane_bytes;                                  // a 16-byte multiple
        g.off_cand = g.off_pix[0] + h * w * 3 - g.plane_bytes;
        g.off_edge2 = o; o += g.plane_bytes;
    } else {
        g.off_cand = o; o += g.plane_bytes;
    }
    g.off_edge = o; o += g.plane_bytes;
    g.off_sdiv = o; o += 1024;                                     // int32[256]
    g.off_hue = o;  o += 1024;                                     // int32[256]
    g.off_lut = o;  o += 256;
    g.off_bar = o;  o += 64;                                       // 8 mbarriers
    g.off_red = o;  o += 32 + 128;                                 // 3 x u64 ROI sums, 16 x u64 statistics
    g.total = o;
    return g;
}

// packed-compare form of one colour range: fp16-subnormal bit patterns duplicated in both halves
struct FastRange {
    uint32_t lo[3], hi[3];
    uint32_t flags;                  // bit 2c: the lower bound of channel c can fail; bit 2c+1: the upper bound can fail
};

struct FastParams {
    PreKParams k;
    FastGeom g;
    FastRange fr[3];
    uint32_t low2, high2;            // edge thresholds as packed patterns
    int need_hue;                    // some range has a hue bound that can fail
    int use_store_warp;              // launch k_preprocess_sw (two extra warps per CTA own the output phase)
};

// ---- small PTX helpers --------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
// a * b + c kept as a multiply-add (FMA pipe) where the compiler would pick a shift-add on the busier ALU pipe
__device__ __forceinline__ uint32_t mad_u32(uint32_t a, uint32_t b, uint32_t c)
{
    uint32_t d;
    asm("mad.lo.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) { return __byte_perm(a, b, sel); }
// PTX prmt in its default mode: a selector nibble with bit 3 set replicates the sign bit of the selected byte over the output byte
__device__ __forceinline__ uint32_t prmt_sx(uint32_t a, uint32_t b, uint32_t sel)
{
    uint32_t d;
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(sel));
    return d;
}

// shared-memory accessors on 32-bit window addresses
__device__ __forceinline__ uint32_t lds8(uint32_t a) { uint32_t v; asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds16(uint32_t a) { uint32_t v; asm volatile("ld.shared.u16 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint32_t lds32(uint32_t a) { uint32_t v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint2 lds64(uint32_t a) { uint2 v; asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ uint4 lds128(uint32_t a)
{
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
    return v;
}
// four pixels' bytes through a 256-entry table in shared memory
__device__ __forceinline__ uint32_t lut4s(uint32_t a_lut, uint32_t v)
{
    return lds8(a_lut + (v & 0xff)) | (lds8(a_lut + ((v >> 8) & 0xff)) << 8) | (lds8(a_lut + ((v >> 16) & 0xff)) << 16) | (lds8(a_lut + (v >> 24)) << 24);
}
// ... of bytes 1..3 / bytes 0..2 only (the neighbour pixel of a strip); the fourth byte comes back as zero
__device__ __forceinline__ uint32_t lut3s_hi(uint32_t a_lut, uint32_t v)
{
    return (lds8(a_lut + ((v >> 8) & 0xff)) << 8) | (lds8(a_lut + ((v >> 16) & 0xff)) << 16) | (lds8(a_lut + (v >> 24)) << 24);
}
__device__ __forceinline__ uint32_t lut3s_lo(uint32_t a_lut, uint32_t v)
{
    return lds8(a_lut + (v & 0xff)) | (lds8(a_lut + ((v >> 8) & 0xff)) << 8) | (lds8(a_lut + ((v >> 16) & 0xff)) << 16);
}
__device__ __forceinline__ void sts8(uint32_t a, uint32_t v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts16(uint32_t a, uint32_t v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts64(uint32_t a, uint2 v) { asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(a), "r"(v.x), "r"(v.y) : "memory"); }
// predicated stores: a lane that does not store costs nothing (an `if` around a store becomes BSSY / BRA / BSYNC around it)
__device__ __forceinline__ void sts8_if(bool on, uint32_t a, uint32_t v)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %2, 0;\n@p st.shared.u8 [%0], %1;\n}\n" ::"r"(a), "r"(v), "r"((uint32_t)on) : "memory");
}
__device__ __forceinline__ void sts64_if(bool on, uint32_t a, uint2 v)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %3, 0;\n@p st.shared.v2.u32 [%0], {%1,%2};\n}\n" ::"r"(a), "r"(v.x), "r"(v.y), "r"((uint32_t)on) : "memory");
}

// predicated global stores (the output loops keep every lane in the loop and switch the stores of the idle lanes off)
__device__ __forceinline__ void stg128_if(bool on, void* p, uint32_t a, uint32_t b, uint32_t c, uint32_t d)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %5, 0;\n@p st.global.v4.u32 [%0], {%1,%2,%3,%4};\n}\n" ::"l"(__cvta_generic_to_global(p)), "r"(a), "r"(b),
                 "r"(c), "r"(d), "r"((uint32_t)on) : "memory");
}
__device__ __forceinline__ void stg64_if(bool on, void* p, uint32_t a, uint32_t b)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %3, 0;\n@p st.global.v2.u32 [%0], {%1,%2};\n}\n" ::"l"(__cvta_generic_to_global(p)), "r"(a), "r"(b), "r"((uint32_t)on) : "memory");
}
__device__ __forceinline__ void stg32_if(bool on, void* p, uint32_t a)
{
    asm volatile("{\n.reg .pred p;\nsetp.ne.u32 p, %2, 0;\n@p st.global.u32 [%0], %1;\n}\n" ::"l"(__cvta_generic_to_global(p)), "r"(a), "r"((uint32_t)on) : "memory");
}

// Frame dimensions as the phase functions see them.  The store-warp kernel is also instantiated with the reference's camera size
// (120 x 160, core/config.py:8-9) as compile-time constants: every row stride, plane pitch and loop bound of the walks becomes an
// immediate instead of a constant-bank load plus address arithmetic per row step.
struct Dims {
    int h, w, mag_stride, plane_bytes;
};
template <int H, int W>
__device__ __forceinline__ Dims make_dims(const FastParams& P)
{
    Dims d;
    if (H > 0 && W > 0) { d.h = H; d.w = W; d.mag_stride = W + 4; d.plane_bytes = (((H + 2) * (W / 32) * 4) + 15) & ~15; }
    else { d.h = P.k.h; d.w = P.k.w; d.mag_stride = P.g.mag_stride; d.plane_bytes = P.g.plane_bytes; }
    return d;
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// (the probe carries a suspend-time hint, which the compiler turns into a NANOSLEEP.SYNCS on the retry path; a hand-written probe + branch loop
// and explicit nanosleep back-offs of 32 / 128 ns all measured the same frames/s at both resolutions: the retries fill idle issue slots)
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    uint32_t done;
    do {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n" : "=r"(done) : "r"(bar), "r"(parity), "r"(0x989680u) : "memory");
    } while (!done);
}
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }
__device__ __forceinline__ int bar_or(int id, int nthreads, int pred)
{
    int r;
    asm volatile(
        "{\n"
        ".reg .pred p, q;\n"
        "setp.ne.s32 q, %3, 0;\n"
        "bar.red.or.pred p, %1, %2, q;\n"
        "selp.s32 %0, 1, 0, p;\n"
        "}\n" : "=r"(r) : "r"(id), "r"(nthreads), "r"(pred) : "memory");
    return r;
}

// one elected thread: arm the barrier with the byte count, then one bulk copy per 16 KB piece
__device__ __forceinline__ void issue_frame_load(uint32_t dst, const uint8_t* src, uint32_t frame_bytes, uint32_t bar)
{
    fence_proxy_async();
    mbar_expect_tx(bar, frame_bytes);
    for (uint32_t o = 0; o < frame_bytes; o += 16384u) tma_load_1d(dst + o, src + o, min(16384u, frame_bytes - o), bar);
}
// bytes [lo, hi) of a frame (16-byte multiples)
__device__ __forceinline__ void issue_frame_piece(uint32_t dst, const uint8_t* src, uint32_t lo, uint32_t hi, uint32_t bar)
{
    issue_frame_load(dst + lo, src + lo, hi - lo, bar);
}

// fp16x2 views of 32-bit registers (bit patterns are integers n < 2048 == fp16 subnormals n * 2^-24)
__device__ __forceinline__ __half2 h2(uint32_t x) { return *reinterpret_cast<__half2*>(&x); }
__device__ __forceinline__ uint32_t u32(__half2 x) { return *reinterpret_cast<uint32_t*>(&x); }
__device__ __forceinline__ uint32_t hsub(uint32_t a, uint32_t b) { return u32(__hsub2(h2(a), h2(b))); }
__device__ __forceinline__ uint32_t hadd(uint32_t a, uint32_t b) { return u32(__hadd2(h2(a), h2(b))); }
__device__ __forceinline__ uint32_t hx2p(uint32_t a, uint32_t b) { return u32(__hfma2(h2(a), __float2half2_rn(2.0f), h2(b))); }   // 2a + b
__device__ __forceinline__ uint32_t habsadd(uint32_t a, uint32_t b) { return u32(__hadd2(__habs2(h2(a)), __habs2(h2(b)))); }     // |a| + |b|
__device__ __forceinline__ uint32_t hmaxu(uint32_t a, uint32_t b) { return u32(__hmax2(h2(a), h2(b))); }
__device__ __forceinline__ uint32_t hgt_mask(uint32_t a, uint32_t b) { return __hgt2_mask(h2(a), h2(b)); }
__device__ __forceinline__ uint32_t hge_mask(uint32_t a, uint32_t b) { return __hge2_mask(h2(a), h2(b)); }
__device__ __forceinline__ uint32_t hle_mask(uint32_t a, uint32_t b) { return __hle2_mask(h2(a), h2(b)); }
__device__ __forceinline__ uint32_t heq_mask(uint32_t a, uint32_t b) { return __heq2_mask(h2(a), h2(b)); }
__device__ __forceinline__ uint32_t bsel(uint32_t m, uint32_t a, uint32_t b) { return (a & m) | (b & ~m); }                      // one LOP3
// (a0, a1) * b + (c0, c1) as ONE packed fp32 instruction (fma.rn.f32x2, SASS FFMA2: |x| / -x operand modifiers fold as for FFMA); each lane is a
// correctly rounded fma, bit-identical with __fmaf_rn.  Returns the two results' bit patterns.
__device__ __forceinline__ uint2 ffma2_bits(float a0, float a1, float b, float c0, float c1)
{
    uint2 d;
    asm("{\n.reg .b64 a, b, c, d;\nmov.b64 a, {%2, %3};\nmov.b64 b, {%4, %4};\nmov.b64 c, {%5, %6};\nfma.rn.f32x2 d, a, b, c;\nmov.b64 {%0, %1}, d;\n}\n"
        : "=r"(d.x), "=r"(d.y) : "f"(a0), "f"(a1), "f"(b), "f"(c0), "f"(c1));
    return d;
}

// direction class (pixel_math.cuh canny_dir) from sign bits: horizontal <=> ay*2^15 - ax*13573 < 0,
// vertical <=> ax*79109 - ay*2^15 < 0, else diagonal 2 + (sign(dx) != sign(dy))
__device__ __forceinline__ uint32_t dir_bits(uint32_t ax, uint32_t ay, uint32_t sdiff)
{
    const int t22 = (int)(ax * 13573u);
    const int nu = (int)(ay * 32768u) - t22;
    const int wv = t22 + (int)(ax * 65536u) - (int)(ay * 32768u);
    const uint32_t H = (uint32_t)(nu >> 31), V = (uint32_t)(wv >> 31);
    return ~H & ((V & 1u) | (~V & (2u | sdiff)));
}

// four 0xffff/0 half masks (pixels 0,2 in `a`; pixels 1,3 in `b`) -> nibble, bit q = pixel q
__device__ __forceinline__ uint32_t nibble_of(uint32_t a, uint32_t b)
{
    const uint32_t x = (a & 0x00040001u) | (b & 0x00080002u);
    return (x | (x >> 16)) & 0xfu;
}

// Two nibbles from eight 0xff/0x00 bytes in one multiply: a = bytes of pixels 0..3 for plane A, b = the same for plane B.
// Bits 0, 9, 18, 27 of a and 4, 13, 22, 31 of b survive the masks; times 0x01010101 every surviving bit lands once in the top
// byte (no two partial products share a position, so no carries): top byte = nibble A | nibble B << 4.
__device__ __forceinline__ uint32_t nibble_pair_top(uint32_t a, uint32_t b)
{
    const uint32_t t = b & 0x80402010u;
    return ((a & 0x08040201u) | t) * 0x01010101u;
}
// even lane: bytes for plane A and plane B from its own top byte and the odd neighbour's (low nibble = own 4 pixels)
__device__ __forceinline__ void merge_nibble_pairs(uint32_t top_own, uint32_t top_other, uint32_t& byteA, uint32_t& byteB)
{
    const uint32_t own = top_own >> 24, oth = top_other >> 24;
    byteA = bsel(0x0fu, own, oth << 4);
    byteB = bsel(0x0fu, own >> 4, oth);
}

// Flood the seed bits along the runs of ones of `c` (seeds must be a subset of c), both directions, O(1).
__device__ __forceinline__ uint32_t flood_run(uint32_t seeds, uint32_t c)
{
    const uint32_t up = (c & ~(c + seeds)) | seeds;          // carry ripples up through each run
    const uint32_t cr = __brev(c), sr = __brev(seeds);
    const uint32_t dn = __brev((cr & ~(cr + sr)) | sr);
    return up | dn;
}

// which strip / rows a lane owns in a strip walk: an 8-lane group is 8 adjacent strips (32 pixels) of one segment
struct StripMap {
    int strip, r0, r1;
    bool ok, store_lane;
};

// rows [row_lo, row_hi) split into segments of seg_rows; lanes whose segment starts past the end idle on row_lo (ok = false)
__device__ __forceinline__ StripMap strip_map(int group_warp, int lane, int nsg, int seg_rows, int row_hi, int row_lo = 0)
{
    StripMap m;
    m.strip = 8 * (group_warp % nsg) + (lane & 7);
    const int seg = 4 * (group_warp / nsg) + (lane >> 3);
    m.r0 = row_lo + seg * seg_rows;
    m.ok = m.r0 < row_hi;
    if (!m.ok) m.r0 = row_lo;
    m.r1 = m.ok ? min(row_hi, m.r0 + seg_rows) : m.r0;
    m.store_lane = m.ok && !(lane & 1);          // even lanes store the byte shared with the odd neighbour
    return m;
}

// shared-memory addresses (32-bit window) of every buffer, derived once from the laundered base
struct SmemMap {
    uint32_t pix[2], mag[2], mask, cand, edge, edge2, sdiv, hue, lut, bar, red;      // mask / cand / edge: address of image row 0
};

__device__ __forceinline__ SmemMap smem_map(uint32_t sb, const FastGeom& G)
{
    SmemMap s;
    s.pix[0] = sb + G.off_pix[0]; s.pix[1] = sb + G.off_pix[1];
    s.mag[0] = sb + G.off_mag[0]; s.mag[1] = sb + G.off_mag[1];
    s.mask = sb + G.off_mask + G.nsg * 4;
    s.cand = sb + G.off_cand + G.nsg * 4;
    s.edge = sb + G.off_edge + G.nsg * 4;
    s.edge2 = G.off_edge2 >= 0 ? sb + G.off_edge2 + G.nsg * 4 : s.edge;
    s.sdiv = sb + G.off_sdiv; s.hue = sb + G.off_hue; s.lut = sb + G.off_lut; s.bar = sb + G.off_bar; s.red = sb + G.off_red;
    return s;
}

// interleaved RGB words of 4 pixels -> planar zero-extended pairs: A = pixels (0,2), B = pixels (1,3), per channel
__device__ __forceinline__ void unpack_planar(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t (&A)[3], uint32_t (&B)[3])
{
    const uint32_t E0 = w0 & 0x00ff00ffu, O0 = prmt(w0, 0, 0x4341);      // E = (b0,b2), O = (b1,b3)
    const uint32_t E1 = w1 & 0x00ff00ffu, O1 = prmt(w1, 0, 0x4341);
    const uint32_t E2 = w2 & 0x00ff00ffu, O2 = prmt(w2, 0, 0x4341);
    A[0] = prmt(E0, E1, 0x7610); A[1] = prmt(O0, O1, 0x7610); A[2] = prmt(E0, E2, 0x5432);
    B[0] = prmt(O0, O2, 0x5432); B[1] = prmt(E1, E2, 0x7610); B[2] = prmt(O1, O2, 0x7610);
}

// =========================================================================================================
// colour-range tests of 4 pixels given as planar pairs; okm[r][half] = 0xffff/0 half masks.
// FLAGSk >= 0 bakes the "which bounds can fail" word of range k into the code (only the live compares are emitted);
// -1 reads it from the parameters.  The hue (two table reads, two multiplies per pixel) is computed only if some
// pixel of the warp survived the saturation / value tests of a range that has a live hue bound.
// =========================================================================================================
template <int F>
__device__ __forceinline__ uint32_t live_flags(const FastRange& R) { return F >= 0 ? (uint32_t)F : R.flags; }

// Saturation bounds without computing the saturation: s = (d * sdiv[v] + 2048) >> 12 is monotone in d, so "s <= K" is
// "d <= T_K[v]" with T_K[v] = min(v, (4096 K + 2047) / sdiv[v]) and "s >= K" is "d > T_{K-1}[v]".  When the live-bound words are
// compile-time constants with at most two saturation bounds, the 256-entry table (in the place of sdiv) holds the two thresholds of a
// value v as 16-bit halves: one table read per pixel, two packed compares per pixel pair, no multiply / shift / repack.
// Bounds take table halves in range order, the lower bound of a range before its upper bound.
// A range with a saturation bound in the table also has its value bounds folded into its thresholds (sat_threshold_entry_folded: a value outside
// them gets a threshold no delta passes), so its value compares are not emitted; a range without one keeps them.
template <int NR, int F0, int F1>
struct SatThresholds {
    static constexpr int n = (F0 >= 0 && F1 >= 0 && NR == 2) ? ((F0 >> 2) & 1) + ((F0 >> 3) & 1) + ((F1 >> 2) & 1) + ((F1 >> 3) & 1) : 99;
    static constexpr bool use = n >= 1 && n <= 2;
    __host__ __device__ static constexpr bool folds(int r) { return use && (((r == 0 ? F0 : F1) & 12) != 0); }
};

// Hue bounds without computing the hue: h = (h0 * hdiv[d] + 2048) >> 12 is monotone in the numerator h0, and the wrapped values (h0 < 0:
// h + 180 >= 150) can never pass an upper bound <= 149, so "lo <= h <= hi" is "A_lo[d] <= h0 <= A_hi[d]".  Used when the live-bound words
// are compile-time constants, exactly one of two ranges bounds the hue on both sides and the other does not look at it (the reference's
// defaults, core/config.py:23); the host only picks such a variant when that upper bound is <= 59 (see hsv_masks_of).  The table (in the place of hdiv) holds
// the two thresholds of a delta d, biased by 2048 like the packed numerators, as 16-bit halves.
template <int NR, int F0, int F1>
struct HueThresholds {
    static constexpr bool use = F0 >= 0 && F1 >= 0 && NR == 2 && (((F0 & 3) == 3 && (F1 & 3) == 0) || ((F0 & 3) == 0 && (F1 & 3) == 3));
    static constexpr int range = (F0 >= 0 && (F0 & 3) == 3) ? 0 : 1;
};

template <int NR, int F0, int F1>
__device__ __forceinline__ void hsv_masks_of(const FastParams& P, const uint32_t (&A)[3], const uint32_t (&B)[3], uint32_t a_sdiv, uint32_t a_hue,
                                             uint32_t (&okm)[NR > 0 ? NR : 1][2])
{
    // fl[r]: which compares are emitted for range r.  A range whose live-bound word is only known at run time gets ALL of them, unconditionally:
    // a bound that cannot fail was stored by the host as a pattern that never fails (a lower bound <= 0 compares as 0 or -1, an upper bound
    // >= 255 as itself, capped at 2047), and six packed compares in a row cost less than six predicated ones.  Whether the saturation and the
    // hue are computed at all stays a run-time decision (hl[r] / P.need_sat: a range without such a bound passes on a saturation or hue of 0).
    constexpr bool RT0 = F0 < 0, RT1 = F1 < 0;
    uint32_t fl[NR > 0 ? NR : 1], hl[NR > 0 ? NR : 1];
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const bool rt = r == 0 ? RT0 : (r == 1 ? RT1 : true);
        const uint32_t live = r == 0 ? live_flags<F0>(P.fr[0]) : (r == 1 ? live_flags<F1>(P.fr[1]) : P.fr[r].flags);
        fl[r] = rt ? 63u : live;
        hl[r] = live & 3u;
    }
    uint32_t any_s = 0, any_h = 0;
#pragma unroll
    for (int r = 0; r < NR; ++r) {
        const bool rt = r == 0 ? RT0 : (r == 1 ? RT1 : true);
        any_s |= rt ? (P.fr[r].flags & 12u) : (fl[r] & 12u);
        any_h |= hl[r];
    }
    uint32_t v2[2], d2[2];
    uint32_t alive = 0;
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        const uint32_t* X = half ? B : A;
        v2[half] = __vimax3_u16x2(X[0], X[1], X[2]);
        d2[half] = v2[half] - __vimin3_u16x2(X[0], X[1], X[2]);
        uint32_t s2 = 0, T2[2] = {0, 0};
        constexpr bool TT = SatThresholds<NR, F0, F1>::use;
        if (TT) {
            const uint32_t tl = lds32(mad_u32(v2[half] & 0xffffu, 4u, a_sdiv)), th = lds32(mad_u32(v2[half] >> 16, 4u, a_sdiv));
            T2[0] = prmt(tl, th, 0x5410); T2[1] = prmt(tl, th, 0x7632);
        } else if (any_s) {
            const uint32_t vlo = v2[half] & 0xffffu, vhi = v2[half] >> 16, dlo = d2[half] & 0xffffu, dhi = d2[half] >> 16;
            const uint32_t slo = (uint32_t)(((int)dlo * (int)lds32(a_sdiv + 4 * vlo) + 2048) >> 12);
            const uint32_t shi = (uint32_t)(((int)dhi * (int)lds32(a_sdiv + 4 * vhi) + 2048) >> 12);
            s2 = slo | (shi << 16);
        }
        int slot = 0;
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            const FastRange& R = P.fr[r];
            uint32_t ok = 0xffffffffu;
            if (TT) {
                if (fl[r] & 4u) ok &= hgt_mask(d2[half], T2[slot++ & 1]);
                if (fl[r] & 8u) ok &= hle_mask(d2[half], T2[slot++ & 1]);
            } else {
                if (fl[r] & 4u) ok &= hge_mask(s2, R.lo[1]);
                if (fl[r] & 8u) ok &= hle_mask(s2, R.hi[1]);
            }
            if (!SatThresholds<NR, F0, F1>::folds(r)) {
                if (fl[r] & 16u) ok &= hge_mask(v2[half], R.lo[2]);
                if (fl[r] & 32u) ok &= hle_mask(v2[half], R.hi[2]);
            }
            okm[r][half] = ok;
            if (hl[r]) alive |= ok;
        }
    }
    if (any_h && __any_sync(0xffffffffu, alive != 0u)) {
#pragma unroll
        for (int half = 0; half < 2; ++half) {
            const uint32_t* X = half ? B : A;
            // hue numerator + 2048 (always positive): g-b | b-r+2d | r-g+4d, chosen by v==r, then v==g
            const uint32_t gb = X[1] + 0x08000800u - X[2];
            const uint32_t br = X[2] + 0x08000800u - X[0] + d2[half] + d2[half];
            const uint32_t eqr = heq_mask(v2[half], X[0]);
            if (HueThresholds<NR, F0, F1>::use) {
                // (the host picks this variant only for an upper hue bound below 60: a pixel whose strongest channel is blue alone has a hue of
                // 120 .. 179; pushed through the green formula its numerator lies in [2d, 3d], a hue of 60 .. 90, which fails the bound just
                // the same, so the third numerator and the second equality test are never needed)
                const uint32_t h02 = bsel(eqr, gb, br);
                constexpr int HR = HueThresholds<NR, F0, F1>::range;
                const uint32_t tl = lds32(mad_u32(d2[half] & 0xffffu, 4u, a_hue)), th = lds32(mad_u32(d2[half] >> 16, 4u, a_hue));
                okm[HR][half] &= hge_mask(h02, prmt(tl, th, 0x5410)) & hle_mask(h02, prmt(tl, th, 0x7632));
                continue;
            }
            const uint32_t rg = X[0] + 0x08000800u - X[1] + (d2[half] << 2);
            const uint32_t eqg = heq_mask(v2[half], X[1]);
            const uint32_t h02 = bsel(eqr, gb, bsel(eqg, br, rg));
            // ((h0 + 2048) hd + (2048 - 2048 hd)) >> 12 == (h0 hd + 2048) >> 12
            const int tl = (int)lds32(a_hue + 4 * (d2[half] & 0xffffu)), th = (int)lds32(a_hue + 4 * (d2[half] >> 16));
            int hlo = ((int)(h02 & 0xffffu) * tl + (2048 - 2048 * tl)) >> 12;
            int hhi = ((int)(h02 >> 16) * th + (2048 - 2048 * th)) >> 12;
            hlo += (hlo >> 31) & 180;
            hhi += (hhi >> 31) & 180;
            const uint32_t hh2 = (uint32_t)hlo | ((uint32_t)hhi << 16);
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const FastRange& R = P.fr[r];
                uint32_t ok = okm[r][half];
                if (fl[r] & 1u) ok &= hge_mask(hh2, R.lo[0]);
                if (fl[r] & 2u) ok &= hle_mask(hh2, R.hi[0]);
                okm[r][half] = ok;
            }
        }
    } else if (any_h) {
        // no pixel of the warp can pass a range with a live hue bound: those ranges are all-zero here
#pragma unroll
        for (int r = 0; r < NR; ++r)
            if (hl[r]) { okm[r][0] = 0; okm[r][1] = 0; }
    }
}

// =========================================================================================================
// P1: strip walk — Sobel / magnitude / direction -> magnitude plane, colour masks -> bit planes
// =========================================================================================================
// tail_bar != 0: the last rows of the frame arrive under a second mbarrier; every thread waits for it at the top of trip `tail_k`
// (a multiple of 3, before any segment loads such a row)
// BANDED: a_pix / a_mag are VIRTUAL bases (the address image row 0 / magnitude row -1 would have), the segment rows of M lie in the
// band's magnitude rows, and colour-mask rows are stored only inside [mask_lo, mask_hi).
// SEG > 0 (a multiple of 3): seg_rows is this compile-time constant AND the segments tile the frame exactly (every lane owns SEG rows,
// r1 == r0 + SEG): the first and the last trip are peeled, so the steady-state row step carries no step-number tests, no row-range
// predicates and a constant row advance (the two replicated-border cases fall on peeled steps).
// LUT: the brightness / contrast table at S.lut is applied to every pixel word as it is loaded (the pixel rows stay raw: kernels whose warps
// cannot agree on a moment to rewrite the rows in place).
template <int NR, bool EDGE, int F0, int F1, bool BANDED = false, int SEG = 0, bool LUT = false>
__device__ __forceinline__ void p1_strip_walk(const FastParams& P, const Dims& Dm, uint32_t a_pix, uint32_t a_mag, uint32_t a_mask, const SmemMap& S,
                                              const StripMap& M, int seg_rows, uint32_t tail_bar = 0, uint32_t tail_parity = 0, int tail_k = 0,
                                              int mask_lo = 0, int mask_hi = 1 << 30)
{
    const int h = Dm.h, w = Dm.w;
    const int row_bytes = w * 3, prb = w >> 3, MS2 = Dm.mag_stride * 2, nstrips = w >> 2;
    const int r0 = M.r0, r1 = M.r1;
    // per-thread constants of the strip walk.  The words left and right of the strip are loaded from the same offsets by every lane
    // and the two edge strips patch them (replicated border: pixel -1 = pixel 0, pixel w = pixel w - 1), so the byte selectors of the
    // neighbour pairs are compile-time constants (per-lane selectors cost ~14 instructions per row step to rematerialise)
    const bool left_edge = M.strip == 0, right_edge = M.strip == nstrips - 1;
    const int nsteps = seg_rows + 2;
    const uint32_t strip_base = a_pix + 12 * M.strip;
    const uint32_t mask_base = a_mask + (M.strip >> 1);
    const uint32_t mag_base = a_mag + 2 * (4 + 4 * M.strip);

    uint32_t D[3][6], Hs[3][6];      // rolling rows: horizontal difference and horizontal smoothing, packed pairs
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 6; ++j) { D[i][j] = 0; Hs[i][j] = 0; }

    // running state of the walk: the image row being loaded and the three row addresses that follow it
    int y_row = r0 - 1;                                                   // may be -1 (frame top) and run past h - 1 (frame bottom): clamped
    uint32_t rp = strip_base + max(y_row, 0) * row_bytes;                 // pixel row y_row (clamped: replicated border)
    uint32_t mp = mask_base + y_row * prb;                                // mask plane byte of row y_row
    uint32_t gp = mag_base + (r0 + 1) * MS2;                              // magnitude row of the next output row (row y lives at row index y + 1)

    // do_mask / do_sobel: std::integral_constant<int, 1> on, <0> off, <-1> decided from the step number k at run time;
    // adv: bytes to the next pixel row (< 0: the run-time replicated-border rule)
    auto row_step = [&](auto mask_tag, auto sobel_tag, int adv, int k, uint32_t (&Dn)[6], uint32_t (&Hn)[6], const uint32_t (&D0)[6],
                        const uint32_t (&D1)[6], const uint32_t (&H0)[6]) {
        constexpr int MK = decltype(mask_tag)::value, SB = decltype(sobel_tag)::value;
        constexpr bool EXACT = SEG > 0;
        // load image row r0 - 1 + k into slot n; emit output row y = r0 + k - 2
        uint32_t w0 = lds32(rp), w1 = lds32(rp + 4), w2 = lds32(rp + 8);
        if (LUT) { w0 = lut4s(S.lut, w0); w1 = lut4s(S.lut, w1); w2 = lut4s(S.lut, w2); }
        uint32_t A[3], B[3];
        unpack_planar(w0, w1, w2, A, B);
        if (EDGE) {
            uint32_t wl = lds32(rp - 4), wr = lds32(rp + 12);       // bytes 1..3 of wl = pixel -1, bytes 0..2 of wr = pixel 4
            if (LUT) { wl = lut3s_hi(S.lut, wl); wr = lut3s_lo(S.lut, wr); }
            if (left_edge) wl = w0 << 8;                            // (the 16 spare bytes in front of the frame keep rp - 4 inside the window)
            if (right_edge) wr = w2 >> 8;
            // neighbours: Lh = pixels (-1,1), Rh = pixels (2,4)
            uint32_t Lh[3], Rh[3];
            Lh[0] = prmt(wl, B[0], 0x5451); Lh[1] = prmt(wl, B[1], 0x5452); Lh[2] = prmt(wl, B[2], 0x5453);
            Rh[0] = prmt(A[0], wr, 0x1412); Rh[1] = prmt(A[1], wr, 0x1512); Rh[2] = prmt(A[2], wr, 0x1612);
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                Dn[c] = hsub(B[c], Lh[c]);                      // pixels (0,2): p[x+1] - p[x-1]
                Dn[3 + c] = hsub(Rh[c], A[c]);                  // pixels (1,3)
                Hn[c] = hadd(hx2p(A[c], Lh[c]), B[c]);          // p[x-1] + 2 p[x] + p[x+1]
                Hn[3 + c] = hadd(hx2p(B[c], A[c]), Rh[c]);
            }
        }
        // ---- colour masks for the loaded row ---------------------------------------------------------
        if (NR > 0 && (MK < 0 ? (k >= 1 && k <= seg_rows) : MK == 1)) {      // warp-uniform: the halo rows above and below belong to other segments
            const bool row_in = M.store_lane && (EXACT || y_row < r1) && (!BANDED || (y_row >= mask_lo && y_row < mask_hi));      // the loaded row belongs to this segment (and band)
            uint32_t okm[NR > 0 ? NR : 1][2];                    // per range: half masks for pixels (0,2) and (1,3)
            hsv_masks_of<NR, F0, F1>(P, A, B, S.sdiv, S.hue, okm);
            if (NR == 2) {
                // pixels 0..3 of a range sit in (okm[r][0].lo, okm[r][1].lo, okm[r][0].hi, okm[r][1].hi)
                const uint32_t top = nibble_pair_top(prmt(okm[0][0], okm[0][1], 0x6240), prmt(okm[NR - 1][0], okm[NR - 1][1], 0x6240));
                const uint32_t other = __shfl_down_sync(0xffffffffu, top, 1);
                uint32_t b0, b1;
                merge_nibble_pairs(top, other, b0, b1);
                sts8_if(row_in, mp, b0);
                sts8_if(row_in, mp + Dm.plane_bytes, b1);
            } else {
                uint32_t v = 0;
#pragma unroll
                for (int r = 0; r < NR; ++r) v |= nibble_of(okm[r][0], okm[r][1]) << (8 * r);
                const uint32_t other = __shfl_down_sync(0xffffffffu, v, 1);
                v |= other << 4;
#pragma unroll
                for (int r = 0; r < NR; ++r) sts8_if(row_in, mp + r * Dm.plane_bytes, v >> (8 * r));
            }
        }
        // ---- Sobel combine for output row y = r0 + k - 2 ----------------------------------------------
        if (EDGE && (SB < 0 ? k >= 2 : SB == 1)) {
            const int y = r0 + k - 2;
            uint32_t mg[2], dxs[2], dys[2];
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                uint32_t m[3], dx[3], dy[3];
#pragma unroll
                for (int c = 0; c < 3; ++c) {
                    const int j = 3 * half + c;
                    dx[c] = hadd(hx2p(D1[j], D0[j]), Dn[j]);            // D[y-1] + 2 D[y] + D[y+1]
                    dy[c] = hsub(Hn[j], H0[j]);                          // H[y+1] - H[y-1]
                    m[c] = habsadd(dx[c], dy[c]);
                }
                const uint32_t g1 = hgt_mask(m[1], m[0]);                // strictly greater: the lowest channel wins ties
                uint32_t mm = hmaxu(m[0], m[1]);
                uint32_t bx = bsel(g1, dx[1], dx[0]), by = bsel(g1, dy[1], dy[0]);
                const uint32_t g2 = hgt_mask(m[2], mm);
                mm = hmaxu(mm, m[2]);
                bx = bsel(g2, dx[2], bx); by = bsel(g2, dy[2], by);
                mg[half] = mm; dxs[half] = bx; dys[half] = by;
            }
            // direction class of each pixel pair, branch-free, mostly on the FMA pipe (pixel_math.cuh canny_dir):
            //   horizontal <=> |dy| - |dx| 13573/2^15 < 0,  vertical <=> |dx| 79109/2^15 - |dy| < 0,  else diagonal 2 + (sign dx != sign dy)
            // the halves are widened to fp32 (exact: n * 2^-24) and each test is ONE fused multiply-add whose sign is exact
            // (the rounding of an fma never changes the sign of a non-zero exact result and an exact zero stays +0); the two pixels of a pair
            // share one packed FFMA2 per test
            uint32_t code[2];
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const __half2 hx = h2(dxs[half]), hy = h2(dys[half]);
                const float ax_lo = fabsf(__low2float(hx)), ax_hi = fabsf(__high2float(hx));
                const float ay_lo = fabsf(__low2float(hy)), ay_hi = fabsf(__high2float(hy));
                const float T22 = 13573.0f / 32768.0f, T67 = 79109.0f / 32768.0f;      // both exact in fp32 (14- and 17-bit numerators)
                const uint2 nu = ffma2_bits(ax_lo, ax_hi, -T22, ay_lo, ay_hi);
                const uint2 wv = ffma2_bits(ax_lo, ax_hi, T67, -ay_lo, -ay_hi);
                const uint32_t H2 = prmt_sx(nu.x, nu.y, 0xffbb), V2 = prmt_sx(wv.x, wv.y, 0xffbb);       // sign of each result spread over its half
                const uint32_t SD = prmt_sx(dxs[half] ^ dys[half], 0, 0xbb99);
                const uint32_t diag = (SD & 0x00010001u) | 0x00020002u;
                code[half] = ~H2 & bsel(V2, 0x00010001u, diag);
            }
            uint2 v;      // pixel order: (A.lo, B.lo) = pixels (0, 1), (A.hi, B.hi) = pixels (2, 3)
            v.x = prmt(mg[0], mg[1], 0x5410) | (prmt(code[0], code[1], 0x5410) << 11);
            v.y = prmt(mg[0], mg[1], 0x7632) | (prmt(code[0], code[1], 0x7632) << 11);
            if (EXACT) sts64(gp, v); else sts64_if(M.ok && y < r1, gp, v);
            gp += MS2;
        }
        // advance to the next image row: the pixel address stays put while the row index is outside [1, h - 1] (replicated borders)
        if (adv >= 0) {
            rp += adv;
        } else {
            ++y_row;
            if ((unsigned)(y_row - 1) < (unsigned)(h - 1)) rp += row_bytes;
        }
        mp += prb;
    };
    using On = std::integral_constant<int, 1>;
    using Off = std::integral_constant<int, 0>;
    using Rt = std::integral_constant<int, -1>;
    // rolling window by register renaming: slots (k % 3)
    if constexpr (SEG > 0) {
        static_assert(SEG % 3 == 0, "the peeled walk keeps the slot rotation of whole trips");
        // step k loads image row r0 - 1 + k (clamped) and, from k = 2 on, emits magnitude row r0 + k - 2; masks belong to steps 1 .. SEG.
        // The row address stands still once at the top of the frame (after step 0 of the first segment) and once at the bottom
        // (after step SEG of the last one).
        if (tail_bar && tail_k < 3) mbar_wait(tail_bar, tail_parity);
        row_step(Off{}, Off{}, r0 == 0 ? 0 : row_bytes, 0, D[0], Hs[0], D[1], D[2], Hs[1]);
        row_step(On{}, Off{}, row_bytes, 1, D[1], Hs[1], D[2], D[0], Hs[2]);
        row_step(On{}, On{}, row_bytes, 2, D[2], Hs[2], D[0], D[1], Hs[0]);
#pragma unroll 1
        for (int k = 3; k < SEG; k += 3) {
            if (tail_bar && k == tail_k) mbar_wait(tail_bar, tail_parity);
            row_step(On{}, On{}, row_bytes, k, D[0], Hs[0], D[1], D[2], Hs[1]);
            row_step(On{}, On{}, row_bytes, k + 1, D[1], Hs[1], D[2], D[0], Hs[2]);
            row_step(On{}, On{}, row_bytes, k + 2, D[2], Hs[2], D[0], D[1], Hs[0]);
        }
        if (tail_bar && tail_k >= SEG) mbar_wait(tail_bar, tail_parity);
        row_step(On{}, On{}, r1 == h ? 0 : row_bytes, SEG, D[0], Hs[0], D[1], D[2], Hs[1]);
        row_step(Off{}, On{}, 0, SEG + 1, D[1], Hs[1], D[2], D[0], Hs[2]);
    } else {
#pragma unroll 1
        for (int k = 0; k < nsteps; k += 3) {
            if (tail_bar && k == tail_k) mbar_wait(tail_bar, tail_parity);
            row_step(Rt{}, Rt{}, -1, k, D[0], Hs[0], D[1], D[2], Hs[1]);             // new = slot0, y-1 = slot1, y = slot2
            if (k + 1 < nsteps) row_step(Rt{}, Rt{}, -1, k + 1, D[1], Hs[1], D[2], D[0], Hs[2]);
            if (k + 2 < nsteps) row_step(Rt{}, Rt{}, -1, k + 2, D[2], Hs[2], D[0], D[1], Hs[0]);
        }
    }
}

// statistics live in shared memory (u64 slots after the three ROI sums): counters kept in registers across the frame loop cost the
// strip walk ~18 registers it does not have
__device__ __forceinline__ void stat_add(const SmemMap& S, int slot, uint32_t v)
{
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0 && v) {
        unsigned long long x = v;
        asm volatile("red.shared.add.u64 [%0], %1;" ::"r"(S.red + 32 + 8 * slot), "l"(x) : "memory");
    }
}

__device__ __forceinline__ void stat_add_one(const SmemMap& S, int slot, unsigned long long x = 1)     // one thread only
{
    asm volatile("red.shared.add.u64 [%0], %1;" ::"r"(S.red + 32 + 8 * slot), "l"(x) : "memory");
}

__device__ __forceinline__ void stats_zero(const SmemMap& S, int t0)
{
    if (t0 < 16) { sts32(S.red + 32 + 8 * t0, 0); sts32(S.red + 36 + 8 * t0, 0); }
}

// slots: 0 frames, 1..4 colour ranges, 5 edge, 6 strong, 7 cand, 8 sweeps, 9 ROI sum (TRS_STAT_*); call after every thread's last stat_add
__device__ __forceinline__ void stats_flush(const PreKParams& p, const SmemMap& S, int t0)
{
    if (t0 < 10) {
        const uint2 v = lds64(S.red + 32 + 8 * t0);
        const unsigned long long x = ((unsigned long long)v.y << 32) | v.x;
        if (x) atomicAdd(&p.stats[t0], x);
    }
}

// =========================================================================================================
// P2: non-maximum suppression, strip walk over the magnitude plane, two pixels per compare
// =========================================================================================================
// SEG > 0 (a multiple of 3): seg_rows is this constant and every lane owns exactly SEG rows (see p1_strip_walk): no row-range predicates,
// no clamp on the row fetched ahead (the fetch past the last row lands in the planes behind the magnitude buffer and is never used).
// COUNT = false: the caller counts the strong pixels itself (count_strong_band before the hysteresis touches the plane), which keeps the
// population count out of every row step.
template <int SEG = 0, bool COUNT = true>
__device__ __forceinline__ void p2_nms(const FastParams& P, const Dims& Dm, uint32_t a_mag, uint32_t a_cand, uint32_t a_edge, const SmemMap& S,
                                       const StripMap& M, int seg_rows)
{
    constexpr bool EXACT = SEG > 0;
    uint32_t n_strong = 0;
    const int h = Dm.h, prb = Dm.w >> 3, MS2 = Dm.mag_stride * 2;
    const uint32_t mbase = a_mag + 2 * (4 + 4 * M.strip);
    const uint32_t cbase = a_cand + (M.strip >> 1), ebase = a_edge + (M.strip >> 1);
    // one row as packed pairs of magnitudes: P01=(m0,m1) P23=(m2,m3) L01=(m-1,m0) M12=(m1,m2) R23=(m3,m4); raw keeps the codes
    struct Row { uint32_t p01, p23, l01, m12, r23, raw01, raw23; };
    struct Raw { uint2 c; uint32_t ml, mr; };                       // a row as loaded: the loads run one step ahead of their use
    auto fetch_at = [&](uint32_t rp) {
        Raw q;
        q.c = lds64(rp); q.ml = lds16(rp - 2); q.mr = lds16(rp + 8);
        return q;
    };
    auto fetch_row = [&](int y) { return fetch_at(mbase + (y + 1) * MS2); };
    auto unpack_row = [&](const Raw& q) {
        Row r;
        r.raw01 = q.c.x; r.raw23 = q.c.y;
        r.p01 = q.c.x & 0x07ff07ffu; r.p23 = q.c.y & 0x07ff07ffu;
        r.l01 = prmt(q.ml & 0x7ffu, r.p01, 0x5410);
        r.m12 = prmt(r.p01, r.p23, 0x5432);
        r.r23 = prmt(r.p23, q.mr & 0x7ffu, 0x5432);
        return r;
    };
    auto load_row = [&](int y) { return unpack_row(fetch_row(y)); };
    const int ya = M.r0;
    Raw ahead;
    uint32_t cp = cbase + ya * prb, ep = ebase + ya * prb;          // plane bytes of the row being decided
    uint32_t ap = mbase + (ya + 3) * MS2;                           // EXACT: running address of the row fetched ahead (row ya + 2 + k at step k)
    // rolling three-row window by register renaming (three steps per trip): step k decides row ya + k from rows (up, ce) and loads dn
    auto nms_step = [&](int k, const Row& up, const Row& ce, Row& dn) {
        const int y = ya + k;
        const bool row_in = EXACT || y < M.r1;
        dn = unpack_row(ahead);
        if (EXACT) { ahead = fetch_at(ap); ap += MS2; } else { ahead = fetch_row(min(y + 2, h)); }
        uint32_t cm[2], sm[2];
#pragma unroll
        for (int pr = 0; pr < 2; ++pr) {
            const uint32_t C = pr ? ce.p23 : ce.p01;
            const uint32_t raw = pr ? ce.raw23 : ce.raw01;
            const uint32_t L = pr ? ce.m12 : ce.l01, Rr = pr ? ce.r23 : ce.m12;
            const uint32_t U = pr ? up.p23 : up.p01, Dw = pr ? dn.p23 : dn.p01;
            const uint32_t UL = pr ? up.m12 : up.l01, DR = pr ? dn.r23 : dn.m12;
            const uint32_t UR = pr ? up.r23 : up.m12, DL = pr ? dn.m12 : dn.l01;
            // direction class bits as half masks: shift the bit to the half's sign position, replicate the sign over the half
            const uint32_t b0 = prmt_sx(raw << 4, 0, 0xbb99), b1 = prmt_sx(raw << 3, 0, 0xbb99);
            // the two neighbours along the gradient: a must be strictly below m; b may tie except on the diagonals
            const uint32_t na = bsel(b1, bsel(b0, UR, UL), bsel(b0, U, L));
            const uint32_t nb = bsel(b1, bsel(b0, DL, DR), bsel(b0, Dw, Rr)) + (b1 & 0x00010001u);     // m > b  <=>  m >= b + 1
            cm[pr] = hgt_mask(C, na) & hge_mask(C, nb) & hgt_mask(C, P.low2);
            sm[pr] = cm[pr] & hgt_mask(C, P.high2);
        }
        // pixels (0,1) sit in the halves of cm[0], (2,3) in cm[1]: one byte per pixel, then both nibbles by one multiply
        const uint32_t top = nibble_pair_top(prmt(cm[0], cm[1], 0x6420), prmt(sm[0], sm[1], 0x6420));
        const uint32_t other = __shfl_down_sync(0xffffffffu, top, 1);
        uint32_t bc, bs;
        merge_nibble_pairs(top, other, bc, bs);
        sts8_if(M.store_lane && row_in, cp, bc);
        sts8_if(M.store_lane && row_in, ep, bs);
        if (COUNT && P.k.stats && M.store_lane && row_in) n_strong += __popc(bs & 0xffu);
        cp += prb; ep += prb;
    };
    Row ra = load_row(ya - 1), rb = load_row(ya), rc;
    ahead = fetch_row(min(ya + 1, h));
    if (EXACT) {
        static_assert(SEG % 3 == 0, "whole trips only");
#pragma unroll 1
        for (int k = 0; k < SEG; k += 3) {
            nms_step(k, ra, rb, rc);
            nms_step(k + 1, rb, rc, ra);
            nms_step(k + 2, rc, ra, rb);
        }
    } else {
#pragma unroll 1
        for (int k = 0; k < seg_rows; k += 3) {
            nms_step(k, ra, rb, rc);
            if (k + 1 < seg_rows) nms_step(k + 1, rb, rc, ra);
            if (k + 2 < seg_rows) nms_step(k + 2, rc, ra, rb);
        }
    }
    if (COUNT && P.k.stats) stat_add(S, 6, n_strong);
}

// =========================================================================================================
// P3: hysteresis — grow the strong set through candidates, one plane word per thread per sweep, until stable.
// a_cand / a_edge address row 0; the rows just above and below hold zeros.  Returns the number of sweeps.
// =========================================================================================================
// Two-level schedule: a warp owns a band of rows and relaxes it to a local fixed point with warp-level synchronisation only
// (no CTA barrier, no waiting for other warps); one CTA-wide OR per round then tells whether any band changed, i.e. whether
// growth may still cross a band boundary.  The fixed point is unique, so the schedule does not affect the result.
// grow the edge bits of plane word t (column wi) from its 3x3 word neighbourhood through its candidates; returns whether it changed
__device__ __forceinline__ int p3_update_word(uint32_t a_cand, uint32_t a_edge, int t, int wi, int ww)
{
    const int rowb = ww * 4;
    const uint32_t c = lds32(a_cand + 4 * t);
    const uint32_t ea = a_edge + 4 * t;
    const uint32_t e = lds32(ea);
    if (c == e) return 0;
    const uint32_t mid = e | lds32(ea - rowb) | lds32(ea + rowb);
    uint32_t lft = 0, rgt = 0;
    if (wi > 0) lft = lds32(ea - 4) | lds32(ea - rowb - 4) | lds32(ea + rowb - 4);
    if (wi + 1 < ww) rgt = lds32(ea + 4) | lds32(ea - rowb + 4) | lds32(ea + rowb + 4);
    const uint32_t spread = mid | (mid << 1) | (mid >> 1) | (lft >> 31) | (rgt << 31);
    const uint32_t ne = flood_run((spread & c) | e, c);
    if (ne == e) return 0;
    sts32(ea, ne);
    return 1;
}

// statistics: the strong pixels of a warp's band of rows, counted from the edge plane BEFORE anything is grown into it (a warp's relaxation
// writes its own rows only, so the count taken right before it is exact)
__device__ __forceinline__ void count_strong_band(const SmemMap& S, uint32_t a_edge, int h, int ww, int lane, int gw, int nw)
{
    const int rows_per = (h + nw - 1) / nw;
    const int y0 = min(h, gw * rows_per), y1 = min(h, y0 + rows_per);
    uint32_t n = 0;
    for (int i = y0 * ww + lane; i < y1 * ww; i += 32) n += __popc(lds32(a_edge + 4 * i));
    stat_add(S, 6, n);
}

// one warp relaxes its band of rows to a local fixed point; returns whether anything changed
__device__ __forceinline__ int p3_relax_band(uint32_t a_cand, uint32_t a_edge, int h, int ww, int lane, int gw, int nw)
{
    const int rows_per = (h + nw - 1) / nw;
    const int y0 = min(h, gw * rows_per), y1 = min(h, y0 + rows_per);
    const int nwords = (y1 - y0) * ww, base = y0 * ww;
    const int wi0 = lane % ww, dwi = 32 % ww;             // word column of this lane's first word, and its step (no division per sweep)
    int band_changed = 0;
    while (true) {
        int changed = 0;
        int wi = wi0;
        for (int i = lane; i < nwords; i += 32, wi = wi + dwi >= ww ? wi + dwi - ww : wi + dwi) changed |= p3_update_word(a_cand, a_edge, base + i, wi, ww);
        __syncwarp();
        if (!__any_sync(0xffffffffu, changed)) break;
        band_changed = 1;
    }
    return band_changed;
}

// After every band of `rows_per` rows has been relaxed on its own (p3_relax_band by nb warps), the only words that can still be short
// of the global fixed point are those in the rows on either side of a band boundary: one pass over them.  Returns whether any changed
// (then the growth has to be carried on with full rounds).
__device__ __forceinline__ int p3_check_band_boundaries(uint32_t a_cand, uint32_t a_edge, int h, int ww, int rows_per, int t0, int tstride)
{
    const int nb = (h + rows_per - 1) / rows_per - 1;     // boundaries
    int changed = 0;
    for (int i = t0; i < nb * 2 * ww; i += tstride) {
        const int b = i / (2 * ww), rem = i - b * 2 * ww, rr = rem / ww, wi = rem - rr * ww;
        const int y = (b + 1) * rows_per - 1 + rr;
        if (y < h) changed |= p3_update_word(a_cand, a_edge, y * ww + wi, wi, ww);
    }
    return changed;
}

template <class OrReduce>
__device__ __forceinline__ int p3_hysteresis(uint32_t a_cand, uint32_t a_edge, int h, int ww, int t0, int tstride, OrReduce group_or)
{
    const int lane = t0 & 31, gw = t0 >> 5, nw = tstride >> 5;
    int rounds = 0, any;
    do {
        any = group_or(p3_relax_band(a_cand, a_edge, h, ww, lane, gw, nw));
        ++rounds;
    } while (any);
    return rounds;
}

// =========================================================================================================
// P4: merge + normalise, written once.  pa[c] = shared address of the bit plane (row 0) feeding output channel c,
// or 0 if that channel keeps the adjusted pixel.
// =========================================================================================================
// gpix != nullptr: the adjusted pixels are not resident any more (banded kernel): the frame is read again from global memory (an L2 hit: it was
// streamed in a moment ago) and goes through the brightness / contrast table at a_lut if use_lut.
__device__ __forceinline__ void p4_output(const FastParams& P, const Dims& Dm, const uint32_t (&pa)[3], uint32_t a_pix, uint8_t* __restrict__ gout,
                                          float* __restrict__ gf32, int t0, int tstride, const uint8_t* __restrict__ gpix = nullptr, uint32_t a_lut = 0,
                                          bool use_lut = false)
{
    const int npb = Dm.h * (Dm.w >> 3);                // groups of 8 pixels = plane bytes
    if (!P.k.need_pixels) {
        // All three channels are bit planes.  Six lanes share one plane byte (8 pixels = 24 output items = six 4-item chunks):
        // lane (g, s) emits chunk s of group g, i.e. one 16-byte f32 store and one 4-byte u8 store, so that consecutive lanes
        // write consecutive addresses (30 lanes = 480 contiguous f32 bytes per instruction; strided per-thread stores made the
        // LSU issue 2-3x the ideal sector count and left the output phase store-bound).
        // Chunk s covers items 4s..4s+3 of (pixel, channel) order: with r = s % 3 and X, Y, Z = planes r, r+1, r+2 (mod 3) it is
        // (X[p0], Y[p1], Z[p2], X[p0 + 1]); the pixel shifts (p0, p1, p2) are (0,0,0), (1,1,2), (2,3,3), plus 4 for s >= 3.
        // A warp owns a contiguous run of warp-iterations, so every address of an unrolled trip is base + immediate, and the
        // bit -> value expansion is one AND (ALU pipe) and multiplies by lane constants (FMA pipe): (x & 1<<sh) * (K >> sh);
        // the u8 word is assembled as 0x80-per-byte and widened to 0xff by one sign-replicating byte permute.
        const int lane = t0 & 31, gw = t0 >> 5, nw = tstride >> 5;
        if (!gf32) {
            // u8 image only (BASELINE.json configs[2], the mask workload): a lane expands one group of 8 pixels = one byte of each plane
            // into its 24 output bytes.  A nibble times 0x10204080 puts pixel q's bit on the sign bit of byte q (no two partial products
            // meet inside a nibble), one sign-replicating permute widens the four sign bits to 0xff / 0x00 bytes, and two permutes per
            // output word interleave the three channels: 39 instructions per 24 bytes instead of 10 per 4.
            if (!gout) return;
            const int per = (npb + nw - 1) / nw;
            const int g0 = min(npb, gw * per), g1 = min(npb, g0 + per);
            auto spread = [](uint32_t b, uint32_t& lo, uint32_t& hi) {
                lo = prmt_sx((b & 0x0fu) * 0x10204080u, 0, 0xba98);
                hi = prmt_sx((b & 0xf0u) * 0x01020408u, 0, 0xba98);
            };
            uint32_t ax = pa[0] + g0 + lane, ay = pa[1] + g0 + lane, az = pa[2] + g0 + lane;
            uint2* dst = reinterpret_cast<uint2*>(gout + (size_t)(g0 + lane) * 24);
#pragma unroll 1
            for (int g = g0; g < g1; g += 32) {
                const bool on = g + lane < g1;
                uint32_t X[2], Y[2], Z[2];
                spread(lds8(ax), X[0], X[1]);
                spread(lds8(ay), Y[0], Y[1]);
                spread(lds8(az), Z[0], Z[1]);
#pragma unroll
                for (int q = 0; q < 2; ++q) {               // pixels 4q .. 4q + 3: (x0 y0 z0 x1) (y1 z1 x2 y2) (z2 x3 y3 z3)
                    const uint32_t w0 = prmt(prmt(X[q], Y[q], 0x1040), Z[q], 0x3410);
                    const uint32_t w1 = prmt(prmt(X[q], Y[q], 0x6205), Z[q], 0x3250);
                    const uint32_t w2 = prmt(prmt(X[q], Y[q], 0x0730), Z[q], 0x7216);
                    if (q == 0) { stg64_if(on, dst, w0, w1); X[0] = w2; } else { stg64_if(on, dst + 1, X[0], w0); stg64_if(on, dst + 2, w1, w2); }
                }
                ax += 32; ay += 32; az += 32; dst += 96;
            }
            return;
        }
        const int gl = lane / 6, sc = lane - 6 * gl, r = sc % 3, hi4 = 4 * (sc / 3);
        const uint32_t paX = r == 0 ? pa[0] : (r == 1 ? pa[1] : pa[2]);
        const uint32_t paY = r == 0 ? pa[1] : (r == 1 ? pa[2] : pa[0]);
        const uint32_t paZ = r == 0 ? pa[2] : (r == 1 ? pa[0] : pa[1]);
        const int shX = r + hi4, shY = (r == 2 ? 3 : r) + hi4, shZ = (r == 0 ? 0 : r + 1) + hi4;
        const uint32_t one = 0x3f800000u;
        const uint32_t mX0 = 1u << shX, mX1 = 2u << shX, mY = 1u << shY, mZ = 1u << shZ;
        const uint32_t fX0 = one >> shX, fX1 = one >> (shX + 1), fY = one >> shY, fZ = one >> shZ;
        const uint32_t qX0 = 128u >> shX, qY = (128u >> shY) << 8, qZ = (128u >> shZ) << 16, qX1 = (128u >> (shX + 1)) << 24;
        // lanes 30 and 31 run the same instructions with their stores predicated off: the loop stays warp-uniform (inside a divergent
        // region the compiler re-derives the global-memory descriptor of every store: two R2UR per STG)
        const bool act = lane < 30;
        {
            const int nfull = npb / 5;                       // warp-iterations whose five groups all exist
            const int nwi = (npb + 4) / 5;
            const int per = (nwi + nw - 1) / nw;
            const int w0 = min(nwi, gw * per), w1 = min(nwi, w0 + per), wf = min(nfull, w1);
            auto emit = [&](auto has_f32, auto has_u8) {
                uint32_t ax = paX + 5 * w0 + gl, ay = paY + 5 * w0 + gl, az = paZ + 5 * w0 + gl;
                uint4* fp = reinterpret_cast<uint4*>(gf32) + 30 * w0 + lane;
                uint32_t* up = reinterpret_cast<uint32_t*>(gout) + 30 * w0 + lane;
                auto one_iter = [&](int k, bool on) {
                    const uint32_t xs = lds8(ax + 5 * k), ys = lds8(ay + 5 * k), zs = lds8(az + 5 * k);
                    const uint32_t b0 = xs & mX0, b1 = ys & mY, b2 = zs & mZ, b3 = xs & mX1;
                    if (decltype(has_f32)::value) {
                        const uint32_t f0 = b0 * fX0, f1 = b1 * fY, f2 = b2 * fZ, f3 = b3 * fX1;
                        stg128_if(on, fp + 30 * k, f0, f1, f2, f3);
                        // byte 2 of 1.0f is 0x80: its sign bit replicated over a byte is the u8 value
                        // (three ALU-pipe permutes measured 1.3 % faster end to end than four FMA-pipe multiplies + one permute)
                        if (decltype(has_u8)::value) stg32_if(on, up + 30 * k, prmt(prmt_sx(f0, f1, 0x00ea), prmt_sx(f2, f3, 0x00ea), 0x5410));
                    } else if (decltype(has_u8)::value) {
                        stg32_if(on, up + 30 * k, prmt_sx(b0 * qX0 + b1 * qY + b2 * qZ + b3 * qX1, 0, 0xba98));
                    }
                };
                int wi = w0;
#pragma unroll 1
                for (; wi + 4 <= wf; wi += 4) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) one_iter(k, act);
                    ax += 20; ay += 20; az += 20; fp += 120; up += 120;
                }
#pragma unroll 1
                for (; wi < w1; ++wi) {
                    one_iter(0, act && 5 * wi + gl < npb);
                    ax += 5; ay += 5; az += 5; fp += 30; up += 30;
                }
            };
            if (gf32 && gout) emit(std::true_type{}, std::true_type{});
            else if (gf32) emit(std::true_type{}, std::false_type{});
            else if (gout) emit(std::false_type{}, std::true_type{});
        }
    } else {
        // some channel keeps the adjusted pixel: bytes from the resident frame, floats by correctly rounded x/255
        const float rcp = 1.0f / 255.0f;
        for (int g = t0; g < 2 * npb; g += tstride) {          // groups of 4 pixels
            uint32_t wv[3];
            if (gpix) {
                const uint32_t* src = reinterpret_cast<const uint32_t*>(gpix) + 3 * (size_t)g;
                wv[0] = __ldg(src); wv[1] = __ldg(src + 1); wv[2] = __ldg(src + 2);
                if (use_lut) { wv[0] = lut4s(a_lut, wv[0]); wv[1] = lut4s(a_lut, wv[1]); wv[2] = lut4s(a_lut, wv[2]); }
            } else {
                const uint32_t src = a_pix + 12 * g;
                wv[0] = lds32(src); wv[1] = lds32(src + 4); wv[2] = lds32(src + 8);
            }
            uint8_t b[12];
#pragma unroll
            for (int k = 0; k < 12; ++k) b[k] = (uint8_t)(wv[k >> 2] >> ((k & 3) * 8));
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                if (pa[c]) {
                    const uint32_t bits = lds8(pa[c] + (g >> 1)) >> ((g & 1) * 4);
#pragma unroll
                    for (int q = 0; q < 4; ++q) b[q * 3 + c] = ((bits >> q) & 1u) ? 255 : 0;
                }
            }
            if (gout) {
                uint32_t* dst = reinterpret_cast<uint32_t*>(gout + (size_t)g * 12);
#pragma unroll
                for (int k = 0; k < 3; ++k)
                    dst[k] = (uint32_t)b[4 * k] | ((uint32_t)b[4 * k + 1] << 8) | ((uint32_t)b[4 * k + 2] << 16) | ((uint32_t)b[4 * k + 3] << 24);
            }
            if (gf32) {
                float fv[12];
#pragma unroll
                for (int k = 0; k < 12; ++k) {
                    // x/255 correctly rounded without a division: q0 = x*rcp, one fused residual correction (exhaustively checked for 0..255)
                    const float x = (float)b[k];
                    const float q0 = __fmul_rn(x, rcp);
                    fv[k] = __fmaf_rn(__fmaf_rn(-q0, 255.0f, x), rcp, q0);
                }
                float4* dst = reinterpret_cast<float4*>(gf32 + (size_t)g * 12);
                dst[0] = make_float4(fv[0], fv[1], fv[2], fv[3]);
                dst[1] = make_float4(fv[4], fv[5], fv[6], fv[7]);
                dst[2] = make_float4(fv[8], fv[9], fv[10], fv[11]);
            }
        }
    }
}

// ---- shared prologue pieces ---------------------------------------------------------------------------------
template <int NR, int F0, int F1>
__device__ __forceinline__ void init_tables(const PreKParams& p, const SmemMap& S, int t0, int tstride)
{
    for (int i = t0; i < 256; i += tstride) {
        const int sd = hsv_sdiv_entry(i);
        if (SatThresholds<NR, F0, F1>::use) {
            // the live saturation bounds in table order (see SatThresholds); K = the largest admissible saturation of "s <= K"; the range's
            // value bounds folded in
            uint32_t entry = 0;
            int slot = 0;
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const int fl = r == 0 ? F0 : F1;
#pragma unroll
                for (int side = 0; side < 2; ++side) {
                    if (!(fl & (4 << side))) continue;
                    const long long K = side == 0 ? (long long)p.ranges[r].lo[1] - 1 : (long long)p.ranges[r].hi[1];
                    entry |= sat_threshold_entry_folded(K, side == 1, i, sd, p.ranges[r].lo[2], p.ranges[r].hi[2]) << (16 * (slot & 1));
                    ++slot;
                }
            }
            sts32(S.sdiv + 4 * i, entry);
        } else {
            sts32(S.sdiv + 4 * i, (uint32_t)sd);
        }
        const int hd = hsv_hdiv_entry(i);
        if (HueThresholds<NR, F0, F1>::use) {
            sts32(S.hue + 4 * i, hue_threshold_entry(p.ranges[HueThresholds<NR, F0, F1>::range].lo[0], p.ranges[HueThresholds<NR, F0, F1>::range].hi[0], hd));
        } else {
            sts32(S.hue + 4 * i, (uint32_t)hd);
        }
        sts8(S.lut + i, p.lut[i]);
    }
}

__device__ __forceinline__ void zero_mag_borders(uint32_t a_mag, int h, int w, int MS, int t0, int tstride)
{
    for (int i = t0; i < MS; i += tstride) { sts16(a_mag + 2 * i, 0); sts16(a_mag + 2 * ((h + 1) * MS + i), 0); }
    // left neighbour of pixel 0 = element 3 of the row; right neighbour of pixel w - 1 = element 4 + w = element 0 of the next row
    for (int i = t0; i < h + 3; i += tstride) { sts16(a_mag + 2 * (i * MS), 0); if (i < h + 2) sts16(a_mag + 2 * (i * MS + 3), 0); }
}

__device__ __forceinline__ void zero_plane_pads(const SmemMap& S, int plane_words, int ww, int t0, int tstride)
{
    for (int i = t0; i < ww; i += tstride) {
        sts32(S.edge - 4 * ww + 4 * i, 0); sts32(S.edge + 4 * (plane_words + i), 0);       // (the pads of the candidate plane are never read)
        sts32(S.edge2 - 4 * ww + 4 * i, 0); sts32(S.edge2 + 4 * (plane_words + i), 0);
    }
}

// brightness / contrast on the resident frame (only when the table is not the identity); `sync` is the barrier of the
// thread group that owns the frame at this point; s_red = generic pointer to three u64 accumulators
template <class Sync>
__device__ __forceinline__ void adjust_in_place(const PreKParams& p, uint32_t a_pix, const SmemMap& S, unsigned long long* s_red, int t0,
                                                int tstride, int lane, Sync sync)
{
    const int h = p.h, w = p.w, row_bytes = w * 3;
    if (p.dynamic) {
        const int y0 = min(40, h), y1 = min(119, h);
        // four pixels = three words (R G B R | G B R G | B R G B) per trip, byte sums by dot products with 0/1 selectors; a thread's share stays
        // far below 2^32 (every caller has a width that is a multiple of 4, so the region is whole groups)
        uint32_t c0 = 0, c1 = 0, c2 = 0;
        const int npix = (y1 - y0) * w;
        const uint32_t roi = a_pix + y0 * row_bytes;
        for (int i = t0; i < (npix >> 2); i += tstride) {
            const uint32_t w0 = lds32(roi + 12 * i), w1 = lds32(roi + 12 * i + 4), w2 = lds32(roi + 12 * i + 8);
            c0 = __dp4a(w2, 0x00000100u, __dp4a(w1, 0x00010000u, __dp4a(w0, 0x01000001u, c0)));
            c1 = __dp4a(w2, 0x00010000u, __dp4a(w1, 0x01000001u, __dp4a(w0, 0x00000100u, c1)));
            c2 = __dp4a(w2, 0x01000001u, __dp4a(w1, 0x00000100u, __dp4a(w0, 0x00010000u, c2)));
        }
        for (int o = 16; o; o >>= 1) {
            c0 += __shfl_xor_sync(0xffffffffu, c0, o);
            c1 += __shfl_xor_sync(0xffffffffu, c1, o);
            c2 += __shfl_xor_sync(0xffffffffu, c2, o);
        }
        if (t0 < 3) s_red[t0] = 0;
        sync();
        if (lane == 0) { atomicAdd(&s_red[0], (unsigned long long)c0); atomicAdd(&s_red[1], (unsigned long long)c1); atomicAdd(&s_red[2], (unsigned long long)c2); }
        sync();
        const float fdelta = (float)brightness_delta(s_red[0], s_red[1], s_red[2], (double)npix, p.baseline);
        if (t0 == 0 && p.stats) s_red[4 + 9] += s_red[0] + s_red[1] + s_red[2];
        for (int i = t0; i < 256; i += tstride) sts8(S.lut + i, adjust_entry(i, true, fdelta, p.foff, p.fratio));
        sync();
    }
    if (p.dynamic || !p.lut_identity) {
        const int nquads = (h * row_bytes) >> 4;                  // (the frame is a whole number of 16-byte pieces and starts on one)
        for (int i = t0; i < nquads; i += tstride) {
            uint4 v = lds128(a_pix + 16 * i);
            v.x = lut4s(S.lut, v.x); v.y = lut4s(S.lut, v.y); v.z = lut4s(S.lut, v.z); v.w = lut4s(S.lut, v.w);
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(a_pix + 16 * i), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
        }
        sync();
    }
}

__device__ __forceinline__ void plane_sources(const PreKParams& p, uint32_t a_edge, uint32_t a_mask, int plane_bytes, uint32_t (&pa)[3])
{
#pragma unroll
    for (int c = 0; c < 3; ++c)
        pa[c] = p.src[c] == SRC_EDGE ? a_edge : (p.src[c] >= SRC_MASK0 ? a_mask + (p.src[c] - SRC_MASK0) * plane_bytes : 0u);
}

// population counts of the finished planes (statistics)
template <int NR, bool EDGE>
__device__ __forceinline__ void count_planes(const PreKParams& p, const SmemMap& S, uint32_t a_cand, uint32_t a_edge, uint32_t a_mask, int plane_bytes, int plane_words,
                                             int t0, int tstride)
{
    uint32_t n_edge = 0, n_cand = 0, n_mask[NR > 0 ? NR : 1] = {0};
    for (int i = t0; i < plane_words; i += tstride) {
        if (EDGE) { n_edge += __popc(lds32(a_edge + 4 * i)); n_cand += __popc(lds32(a_cand + 4 * i)); }
#pragma unroll
        for (int k = 0; k < NR; ++k) n_mask[k] += __popc(lds32(a_mask + k * plane_bytes + 4 * i));
    }
    if (EDGE) { stat_add(S, 5, n_edge); stat_add(S, 7, n_cand); }
#pragma unroll
    for (int k = 0; k < NR; ++k) stat_add(S, 1 + p.range_stat[k], n_mask[k]);
    if (t0 == 0) stat_add_one(S, 0);
}

// =========================================================================================================
// Resident kernel: one frame per CTA, two CTAs per SM
// =========================================================================================================
template <int NR, bool EDGE, int F0, int F1, bool LIST = false>
__global__ void __launch_bounds__(FAST_MAX_THREADS, 2) k_preprocess_fast(const __grid_constant__ FastParams P, const FrameList fl = {})
{
    extern __shared__ __align__(16) uint8_t smem[];
    const PreKParams& p = P.k;
    int n_list = 0;
    const int* list = nullptr;
    if constexpr (LIST) {                              // (preproc_kernel.cuh k_preprocess)
        plist_open(fl, list, n_list);
        if ((int)blockIdx.x >= n_list) return;
    }
    const FastGeom& G = P.g;
    uint32_t sb = smem_u32(smem);
    asm volatile("" : "+r"(sb));                       // launder: the window base lives in this register, never re-derived
    const SmemMap S = smem_map(sb, G);
    unsigned long long* s_red = reinterpret_cast<unsigned long long*>(smem + G.off_red);
    const int h = p.h, w = p.w, ww = G.nsg;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t frame_bytes = (uint32_t)h * w * 3;
    const int plane_words = h * ww;
    const StripMap M = strip_map(warp, lane, ww, G.seg_rows_front, h);
    const Dims Dm = make_dims<0, 0>(P);

    init_tables<NR, F0, F1>(p, S, tid, nthr);
    stats_zero(S, tid);
    if (EDGE) {
        zero_mag_borders(S.mag[0], h, w, G.mag_stride, tid, nthr);
        zero_plane_pads(S, plane_words, ww, tid, nthr);
    }
    if (tid == 0) { mbar_init(S.bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();
    if (tid == 0 && (int)blockIdx.x < (LIST ? n_list : p.n)) issue_frame_load(S.pix[0], p.in + (size_t)plist_frame<LIST>(list, blockIdx.x) * frame_bytes, frame_bytes, S.bar);
    uint32_t phase = 0;
    uint32_t pa[3];
    plane_sources(p, S.edge, S.mask, G.plane_bytes, pa);

    // cycle accounting of thread 0 (statistics runs only): TRS_STAT_T_* slots 10..15 = frame wait, strip walk, NMS, hysteresis, output, total
    // (compiled in only with -DTRS_PHASE_TIMERS: the counters cost registers the strip walk does not have to spare)
    long long tm[6] = {0, 0, 0, 0, 0, 0};
#ifdef TRS_PHASE_TIMERS
    const bool timing = p.stats != nullptr && tid == 0;
#else
    const bool timing = false;
#endif
    for (int j = blockIdx.x; j < (LIST ? n_list : p.n); j += gridDim.x) {
        const int f = plist_frame<LIST>(list, j);
        const long long tk0 = timing ? clock64() : 0;
        mbar_wait(S.bar, phase);
        phase ^= 1u;
        const long long tk1 = timing ? clock64() : 0;
        adjust_in_place(p, S.pix[0], S, s_red, tid, nthr, lane, [] { __syncthreads(); });
        p1_strip_walk<NR, EDGE, F0, F1>(P, Dm, S.pix[0], S.mag[0], S.mask, S, M, G.seg_rows_front);
        __syncthreads();
        const long long tk2 = timing ? clock64() : 0;
        if (!p.need_pixels && tid == 0 && j + (int)gridDim.x < (LIST ? n_list : p.n))         // pixels are dead: prefetch the next frame
            issue_frame_load(S.pix[0], p.in + (size_t)plist_frame<LIST>(list, j + gridDim.x) * frame_bytes, frame_bytes, S.bar);
        long long tk3 = tk2, tk4 = tk2;
        if (EDGE) {
            p2_nms(P, Dm, S.mag[0], S.cand, S.edge, S, M, G.seg_rows_front);
            __syncthreads();
            tk3 = timing ? clock64() : 0;
            const int sw = p3_hysteresis(S.cand, S.edge, h, ww, tid, nthr, [](int c) { return __syncthreads_or(c); });
            if (tid == 0 && p.stats) stat_add_one(S, 8, (unsigned long long)sw);
            tk4 = timing ? clock64() : 0;
        }
        p4_output(P, Dm, pa, S.pix[0], p.out_u8 ? p.out_u8 + (size_t)f * frame_bytes : nullptr, p.out_f32 ? p.out_f32 + (size_t)f * frame_bytes : nullptr,
                  tid, nthr);
        if (p.stats) count_planes<NR, EDGE>(p, S, S.cand, S.edge, S.mask, G.plane_bytes, plane_words, tid, nthr);
        __syncthreads();
        if (timing) {
            const long long tk5 = clock64();
            tm[0] += tk1 - tk0; tm[1] += tk2 - tk1; tm[2] += tk3 - tk2; tm[3] += tk4 - tk3; tm[4] += tk5 - tk4; tm[5] += tk5 - tk0;
        }
        if (p.need_pixels && tid == 0 && j + (int)gridDim.x < (LIST ? n_list : p.n))
            issue_frame_load(S.pix[0], p.in + (size_t)plist_frame<LIST>(list, j + gridDim.x) * frame_bytes, frame_bytes, S.bar);
    }
    if (timing) {
#pragma unroll
        for (int k = 0; k < 6; ++k) atomicAdd(&p.stats[10 + k], (unsigned long long)tm[k]);
    }
    if (p.stats) stats_flush(p, S, tid);          // (the frame loop ends with a CTA-wide barrier)
}

// Dynamic brightness for a frame that is NOT resident in shared memory: exact channel sums over rows 40..118 (img_preprocessing.py:88) straight
// from global memory (row bytes and frame bytes multiples of 4), then delta = (baseline - sum of channel means) / 3 as float32.  Every thread
// of the CTA calls it; contains CTA-wide barriers; s_red = three u64 accumulators (+ the statistics slots behind them).
__device__ __forceinline__ float dynamic_delta_global(const PreKParams& p, const uint8_t* __restrict__ gfr, unsigned long long* s_red, int tid, int nthr, int lane)
{
    const int h = p.h, w = p.w, row_words = (w * 3) >> 2;
    const int y0 = min(40, h), y1 = min(119, h);
    const uint32_t* roi = reinterpret_cast<const uint32_t*>(gfr + (size_t)y0 * w * 3);
    const int nw = (y1 - y0) * row_words;
    uint32_t c0 = 0, c1 = 0, c2 = 0;                             // word i of the region starts with channel i % 3 (4 i % 3 == i % 3)
    for (int i = tid; i < nw; i += nthr) {
        const uint32_t v = __ldg(roi + i);
        const int ph = i % 3;
        const uint32_t a = __dp4a(v, 0x01000001u, 0u), b = __dp4a(v, 0x00000100u, 0u), c = __dp4a(v, 0x00010000u, 0u);      // bytes (0, 3) | 1 | 2
        if (ph == 0) { c0 += a; c1 += b; c2 += c; } else if (ph == 1) { c1 += a; c2 += b; c0 += c; } else { c2 += a; c0 += b; c1 += c; }
    }
    for (int o = 16; o; o >>= 1) {
        c0 += __shfl_xor_sync(0xffffffffu, c0, o);
        c1 += __shfl_xor_sync(0xffffffffu, c1, o);
        c2 += __shfl_xor_sync(0xffffffffu, c2, o);
    }
    if (tid < 3) s_red[tid] = 0;
    __syncthreads();
    if (lane == 0) { atomicAdd(&s_red[0], (unsigned long long)c0); atomicAdd(&s_red[1], (unsigned long long)c1); atomicAdd(&s_red[2], (unsigned long long)c2); }
    __syncthreads();
    const float fdelta = (float)brightness_delta(s_red[0], s_red[1], s_red[2], (double)((y1 - y0) * w), p.baseline);
    if (tid == 0 && p.stats) s_red[4 + 9] += s_red[0] + s_red[1] + s_red[2];
    __syncthreads();                                             // (the accumulators are zeroed again by the next frame's call)
    return fdelta;
}

// =========================================================================================================
// Banded kernel: frames too large to be resident (240x320: 230 KB) go through the same phases band by band.  Per band of
// band_h rows: one bulk copy of the band's pixel rows plus a two-row halo, the strip walk over the band's magnitude rows
// (one extra row above and below, recomputed instead of kept), NMS for the band's rows into the FULL-FRAME candidate /
// edge planes (colour masks likewise); the next band's copy is issued as soon as the strip walk is done.  After the last
// band: hysteresis and output over the whole frame from the bit planes.  A brightness / contrast table is applied to each band's rows as
// they land (the dynamic one is built first from the frame's rows 40..118 in global memory); an output channel that keeps the adjusted pixel
// reads the frame again in the output phase (from L2: 296 frames in flight are 68 MB).
// =========================================================================================================
template <int NR, bool EDGE, int F0, int F1, bool LIST = false>
__global__ void __launch_bounds__(FAST_MAX_THREADS, 2) k_preprocess_banded(const __grid_constant__ FastParams P, const FrameList fl = {})
{
    extern __shared__ __align__(16) uint8_t smem[];
    const PreKParams& p = P.k;
    int n_list = 0;
    const int* list = nullptr;
    if constexpr (LIST) {
        plist_open(fl, list, n_list);
        if ((int)blockIdx.x >= n_list) return;
    }
    const FastGeom& G = P.g;
    uint32_t sb = smem_u32(smem);
    asm volatile("" : "+r"(sb));
    const SmemMap S = smem_map(sb, G);
    const int h = p.h, w = p.w, ww = G.nsg;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t row_bytes = (uint32_t)w * 3, frame_bytes = (uint32_t)h * row_bytes;
    const int plane_words = h * ww;
    const int BH = G.band_h, NB = G.n_bands, MS = G.mag_stride;
    const Dims Dm = make_dims<0, 0>(P);

    init_tables<NR, F0, F1>(p, S, tid, nthr);
    stats_zero(S, tid);
    if (EDGE) {
        zero_mag_borders(S.mag[0], BH + 2, w, MS, tid, nthr);
        zero_plane_pads(S, plane_words, ww, tid, nthr);
    }
    if (tid == 0) { mbar_init(S.bar, 1); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();
    // pixel rows of band b: [max(b BH - 2, 0), min((b + 1) BH + 2, h))
    auto issue_band = [&](size_t f, int b) {
        const int p0 = max(b * BH - 2, 0), p1 = min(min((b + 1) * BH, h) + 2, h);
        issue_frame_load(S.pix[0], p.in + f * frame_bytes + (size_t)p0 * row_bytes, (uint32_t)(p1 - p0) * row_bytes, S.bar);
    };
    if (tid == 0 && (int)blockIdx.x < (LIST ? n_list : p.n)) issue_band(plist_frame<LIST>(list, blockIdx.x), 0);

    uint32_t phase = 0;
    uint32_t pa[3];
    plane_sources(p, S.edge, S.mask, G.plane_bytes, pa);
    unsigned long long* s_red = reinterpret_cast<unsigned long long*>(smem + G.off_red);
    const bool use_lut = p.dynamic || !p.lut_identity;
    for (int j = blockIdx.x; j < (LIST ? n_list : p.n); j += gridDim.x) {
        const int f = plist_frame<LIST>(list, j);
        if (p.dynamic) {
            // the brightness statistic covers rows 40..118 (img_preprocessing.py:88), which no single band holds: exact channel sums from the
            // frame in global memory while the first band's copy is in flight (the bands read those rows again, from L2), then this frame's table
            const float fdelta = dynamic_delta_global(p, p.in + (size_t)f * frame_bytes, s_red, tid, nthr, lane);
            for (int i = tid; i < 256; i += nthr) sts8(S.lut + i, adjust_entry(i, true, fdelta, p.foff, p.fratio));
            __syncthreads();
        }
        for (int b = 0; b < NB; ++b) {
            const int by0 = b * BH, by1 = min(by0 + BH, h);
            const int m0 = EDGE ? max(by0 - 1, 0) : by0, m1 = EDGE ? min(by1 + 1, h) : by1;      // magnitude rows of this band
            const int p0 = max(by0 - 2, 0);
            const uint32_t a_pix = S.pix[0] - (uint32_t)p0 * row_bytes;                            // virtual address of image row 0
            const uint32_t a_mag = S.mag[0] - (uint32_t)(m0 * MS * 2);                            // virtual address of magnitude row -1
            mbar_wait(S.bar, phase);
            phase ^= 1u;
            if (use_lut) {                                          // brightness / contrast on the band's pixel rows as they land (halo rows twice)
                const int nquads = (min(by1 + 2, h) - p0) * (int)(row_bytes >> 4);      // (a row is a whole number of 16-byte pieces: w % 32 == 0)
                for (int i = tid; i < nquads; i += nthr) {
                    uint4 v = lds128(S.pix[0] + 16 * i);
                    v.x = lut4s(S.lut, v.x); v.y = lut4s(S.lut, v.y); v.z = lut4s(S.lut, v.z); v.w = lut4s(S.lut, v.w);
                    asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(S.pix[0] + 16 * i), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
                }
                __syncthreads();
            }
            if (EDGE && m1 == h) {                                  // the zero row below the frame: earlier bands left data there
                for (int i = tid; i < MS; i += nthr) sts16(a_mag + 2 * ((h + 1) * MS + i), 0);
            }
            const StripMap M1 = strip_map(warp, lane, ww, G.seg_rows_front, m1, m0);
            p1_strip_walk<NR, EDGE, F0, F1, true>(P, Dm, a_pix, a_mag, S.mask, S, M1, G.seg_rows_front, 0u, 0u, 0, by0, by1);
            __syncthreads();
            if (tid == 0) {                                         // pixels are dead: fetch the next band (of this or the next frame)
                if (b + 1 < NB) issue_band(f, b + 1);
                else if (j + (int)gridDim.x < (LIST ? n_list : p.n))
                    issue_band(LIST ? (size_t)plist_frame<LIST>(list, j + gridDim.x) : (size_t)f + gridDim.x, 0);
            }
            if (EDGE) {
                const StripMap M2 = strip_map(warp, lane, ww, G.seg_rows_nms, by1, by0);
                p2_nms(P, Dm, a_mag, S.cand, S.edge, S, M2, G.seg_rows_nms);
                __syncthreads();
            }
        }
        if (EDGE) {
            const int sw = p3_hysteresis(S.cand, S.edge, h, ww, tid, nthr, [](int c) { return __syncthreads_or(c); });
            if (tid == 0 && p.stats) stat_add_one(S, 8, (unsigned long long)sw);
        }
        p4_output(P, Dm, pa, 0u, p.out_u8 ? p.out_u8 + (size_t)f * frame_bytes : nullptr, p.out_f32 ? p.out_f32 + (size_t)f * frame_bytes : nullptr, tid, nthr,
                  p.in + (size_t)f * frame_bytes, S.lut, use_lut);
        if (p.stats) count_planes<NR, EDGE>(p, S, S.cand, S.edge, S.mask, G.plane_bytes, plane_words, tid, nthr);
        __syncthreads();
    }
    if (p.stats) stats_flush(p, S, tid);
}

// =========================================================================================================
// Store-warp kernel: the resident kernel plus TWO extra warps per CTA that own the output phase.
//
// Why: the SM -> L2 write port sustains ~29 B/clk (tools/ubench_store.cu: any store flavour, any number of SMs), so the
// 288,000 output bytes of a frame occupy it for ~10 k cycles.  With the output phase run by all warps the CTA sits in
// it for 13.6 k of its 56 k cycles per frame with almost nothing to issue.  Here the ten compute warps hand the finished
// planes of frame j to the store warps and start frame j + 1 at once.  What makes that legal:
//   * the colour-mask planes (written by the strip walk, P1) and the edge plane (written by the NMS, P2, grown by the
//     hysteresis, P3) are double-buffered by frame parity, so the store warps have a whole frame time;
//   * the shared memory for the second edge plane comes from the candidate plane, which only lives from P2 to P3 and sits
//     on the last 2.4 KB of the frame buffer: those bytes of the next frame arrive by a second, later bulk copy.
// Hand-over: named barrier 2 = "planes of frame j are final" (compute warps arrive, store warps sync);
//            "done with frame j's planes" is one mbarrier per plane set (frame parity): the store warps arrive after the output of frame j,
//            the compute warps wait for that phase before P1 of frame j + 2.  (A named barrier cannot carry this direction: the store warps
//            may finish frame j + 1 before the compute warps have asked about frame j - with a brightness / contrast table the compute warps
//            first wait for the tail copy the store warps issue and then rewrite the frame - and a second round of arrivals on a named
//            barrier whose first round is still open completes it early and strands the late compute warps.)
//            Frames come on demand (draw_frames): the store warps draw frame j + 3 while they work on frame j and publish it in the frame
//            ring before that same bar_free arrival, which is where the compute warps learn it (they need frame j + 1 after P1 of frame j).
// Compute-only phases use named barrier 1.
// =========================================================================================================
enum { SW_COMPUTE_THREADS = 320, SW_THREADS = 384, SW_MAXREG = 80 };      // register allocation rounds a CTA up to a multiple of 4 warps

__device__ __forceinline__ void bar_arrive(int id, int nthreads) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// Frames on demand (k_preprocess_sw, k_preprocess_bsw).  What a frame costs depends on its content, so a fixed stride (CTA b takes b, b + G,
// b + 2G, ...) leaves the launch waiting for the CTAs that drew the slow frames: a batch of interleaved sources with a period that divides G
// puts every CTA on one kind of frame.  Instead a CTA's first frame is blockIdx.x and each further one is gridDim.x + a ticket from the
// launch's counter.  One thread per CTA draws the tickets, one after the other, so a CTA's frames increase and the first one >= n ends its
// loop: every frame is processed exactly once whatever the timing, and outputs are addressed by frame, so results do not depend on the order.
// The tickets are drawn ahead and published in a ring of FRAME_RING frame indices in shared memory (slot j % FRAME_RING: the CTA's frame j),
// handed over by barriers the roles already share (DESIGN.md §4.9): no warp waits for the atomic's round trip.
enum { FRAME_RING = 4 };
__device__ __forceinline__ uint32_t draw_frames(const PreKParams& p, uint32_t k = 1) { return gridDim.x + atomicAdd(p.frame_ctr, k); }
__device__ __forceinline__ uint32_t ring_frame(uint32_t a_ring, int j) { return lds32(a_ring + 4 * (uint32_t)(j % FRAME_RING)); }

// H, W > 0: the frame size is a compile-time constant (the host launches such a variant only for exactly that size, with the geometry
// sw_static_geometry_ok() accepts); H = W = 0: any size that fits.
template <int H, int W>
__host__ __device__ constexpr int sw_seg_rows() { return (H + 4 * ((SW_COMPUTE_THREADS / 32) / (W / 32)) - 1) / (4 * ((SW_COMPUTE_THREADS / 32) / (W / 32))); }
template <int H, int W>
inline bool sw_static_geometry_ok(const FastGeom& g, int h, int w)
{
    return h == H && w == W && g.nsg == W / 32 && g.front_warps == SW_COMPUTE_THREADS / 32 && g.seg_rows_front == sw_seg_rows<H, W>() && g.mag_stride == W + 4 &&
           g.plane_bytes == ((((H + 2) * (W / 32) * 4) + 15) & ~15) && g.tail_bytes == g.plane_bytes && g.n_bands == 1 &&
           sw_seg_rows<H, W>() % 3 == 0 && 4 * ((SW_COMPUTE_THREADS / 32) / (W / 32)) * sw_seg_rows<H, W>() == H;      // the segments tile the rows exactly
}

template <int NR, int F0, int F1, int H = 0, int W = 0, bool LIST = false>
__global__ void __maxnreg__(SW_MAXREG) k_preprocess_sw(const __grid_constant__ FastParams P, const FrameList fl = {})
{
    extern __shared__ __align__(16) uint8_t smem[];
    const PreKParams& p = P.k;
    int n_list = 0;
    const int* list = nullptr;
    if constexpr (LIST) {                                          // (the frame ring holds positions in the list, the loads map them to frames)
        plist_open(fl, list, n_list);
        if ((int)blockIdx.x >= n_list) return;
    }
    const FastGeom& G = P.g;
    uint32_t sb = smem_u32(smem);
    asm volatile("" : "+r"(sb));
    const SmemMap S = smem_map(sb, G);
    unsigned long long* s_red = reinterpret_cast<unsigned long long*>(smem + G.off_red);
    constexpr bool STATIC = H > 0 && W > 0;
    const Dims Dm = make_dims<H, W>(P);
    const int h = Dm.h, w = Dm.w, ww = STATIC ? W / 32 : G.nsg;
    const int seg_rows = STATIC ? sw_seg_rows<(STATIC ? H : 32), (STATIC ? W : 32)>() : G.seg_rows_front;
    const int tail_bytes = STATIC ? Dm.plane_bytes : G.tail_bytes;
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31;
    const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);       // (tells the compiler that the role branch below is warp-uniform)
    const uint32_t frame_bytes = (uint32_t)h * w * 3;
    const int plane_words = h * ww;
    const int NC = SW_COMPUTE_THREADS;
    const uint32_t n = (uint32_t)(LIST ? n_list : p.n);
    const uint32_t mask_set_bytes = (uint32_t)(NR * Dm.plane_bytes);
    const uint32_t main_bytes = frame_bytes - (uint32_t)tail_bytes;
    const uint32_t bar_main = S.bar, bar_tail = S.bar + 8, bar_free = S.bar + 16;      // bar_free + 8 q: plane set q has been written out
    const uint32_t a_ring = S.bar + 32;                                                  // frame ring (the barrier block's free half)

    uint32_t ticket = 0;
    if (tid == NC) ticket = draw_frames(p, 2);                    // frames 1 and 2, in flight during the set-up
    init_tables<NR, F0, F1>(p, S, tid, nthr);
    stats_zero(S, tid);
    zero_mag_borders(S.mag[0], h, w, Dm.mag_stride, tid, nthr);
    zero_plane_pads(S, plane_words, ww, tid, nthr);
    if (tid == 0) {
        mbar_init(bar_main, 1); mbar_init(bar_tail, 1);
        mbar_init(bar_free, (SW_THREADS - SW_COMPUTE_THREADS) / 32); mbar_init(bar_free + 8, (SW_THREADS - SW_COMPUTE_THREADS) / 32);      // one arrival per store warp
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (tid == NC) { sts32(a_ring, blockIdx.x); sts32(a_ring + 4, ticket); sts32(a_ring + 8, ticket + 1); }
    __syncthreads();

    if (warp < (NC >> 5)) {
        // ------------------------------------------------ compute warps -----------------------------------------------
        const StripMap M = strip_map(warp, lane, ww, seg_rows, h);
        const bool use_lut = p.dynamic || !p.lut_identity;
        // first strip-walk trip (a multiple of 3) in which some segment loads a row of the tail piece
        const int nsegs = 4 * ((NC >> 5) / ww);
        const int tail_row = (int)(main_bytes / (uint32_t)(w * 3));
        int tail_k = tail_row - (nsegs - 1) * seg_rows + 1;
        tail_k = tail_k < 0 ? 0 : (tail_k / 3) * 3;
        if (tid == 0 && blockIdx.x < n) {
            const uint8_t* src = p.in + (size_t)plist_frame<LIST>(list, blockIdx.x) * frame_bytes;
            issue_frame_piece(S.pix[0], src, 0, main_bytes, bar_main);
            if (tail_bytes) issue_frame_piece(S.pix[0], src, main_bytes, frame_bytes, bar_tail);
        }
        uint32_t phase = 0;
#ifdef TRS_PHASE_TIMERS
        long long tm[6] = {0, 0, 0, 0, 0, 0};      // thread 0: frame wait, strip walk, wait for the store warps, NMS, hysteresis, total
        const bool timing = p.stats != nullptr && tid == 0;
#define TRS_TICK(v) const long long v = timing ? clock64() : 0
#else
#define TRS_TICK(v)
#endif
        // the CTA's frame k (k >= 3) is published before the store warps' arrival on bar_free for frame k - 3, which every compute thread
        // waits for before P1 of frame k - 1; it is read after that P1 (thread 0) and at the top of iteration k.  Frames 0..2: set-up barrier.
        for (int j = 0; ring_frame(a_ring, j) < n; ++j) {
            const uint32_t a_mask = S.mask + (j & 1) * mask_set_bytes;
            const uint32_t a_edge = (j & 1) ? S.edge2 : S.edge;
            TRS_TICK(tk0);
            mbar_wait(bar_main, phase);
            if (tail_bytes && use_lut) mbar_wait(bar_tail, phase);       // the table pass touches every pixel
            TRS_TICK(tk1);
            adjust_in_place(p, S.pix[0], S, s_red, tid, NC, lane, [NC] { bar_sync(1, NC); });
            TRS_TICK(tk2);
            if (j >= 2) mbar_wait(bar_free + 8 * (j & 1), (uint32_t)((j >> 1) - 1) & 1u);      // the store warps are done with frame j-2: this plane set is free
            TRS_TICK(tk3);
            p1_strip_walk<NR, true, F0, F1, false, (STATIC ? sw_seg_rows<(STATIC ? H : 32), (STATIC ? W : 32)>() : 0)>(
                P, Dm, S.pix[0], S.mag[0], a_mask, S, M, seg_rows, (tail_bytes && !use_lut) ? bar_tail : 0u, phase, tail_k);
            phase ^= 1u;
            bar_sync(1, NC);
            TRS_TICK(tk4);
            if (tid == 0) {                                              // pixels are dead: prefetch the next frame (all but its tail)
                const uint32_t fn = ring_frame(a_ring, j + 1);
                if (fn < n) issue_frame_piece(S.pix[0], p.in + (size_t)plist_frame<LIST>(list, fn) * frame_bytes, 0, main_bytes, bar_main);
            }
            p2_nms<(STATIC ? sw_seg_rows<(STATIC ? H : 32), (STATIC ? W : 32)>() : 0), false>(P, Dm, S.mag[0], S.cand, a_edge, S, M, seg_rows);
            bar_sync(1, NC);
            TRS_TICK(tk5);
            if (p.stats) count_strong_band(S, a_edge, h, ww, lane, warp, NC >> 5);
            // hysteresis, first level only: every warp relaxes its own band, no CTA-wide round trip; the store warps finish the job
            p3_relax_band(S.cand, a_edge, h, ww, lane, warp, NC >> 5);
#ifdef TRS_PHASE_TIMERS
            if (timing) {
                const long long tk6 = clock64();
                tm[0] += tk1 - tk0; tm[1] += tk4 - tk3; tm[2] += tk3 - tk2; tm[3] += tk5 - tk4; tm[4] += tk6 - tk5; tm[5] += tk6 - tk0;
            }
#endif
            bar_arrive(2, SW_THREADS);                                   // planes of frame j are final: the store warps take them from here
            // (no barrier here: the next strip walk writes the other plane set and the magnitude plane only)
        }
#ifdef TRS_PHASE_TIMERS
        if (timing)
            for (int k = 0; k < 6; ++k) atomicAdd(&p.stats[10 + k], (unsigned long long)tm[k]);
#endif
#undef TRS_TICK
    } else {
        // ------------------------------------------------ store warps -------------------------------------------------
        // slots j and j + 1 were written by thread NC at least two frames ago, before a barrier of both store warps
        for (int j = 0;; ++j) {
            const uint32_t fj = ring_frame(a_ring, j);
            if (fj >= n) break;
            const uint32_t f = plist_frame<LIST>(list, fj);
            if (tid == NC) ticket = draw_frames(p);                      // frame j + 3: published after this frame's output
            uint32_t pa[3];
            plane_sources(p, (j & 1) ? S.edge2 : S.edge, S.mask + (j & 1) * mask_set_bytes, Dm.plane_bytes, pa);
            bar_sync(2, SW_THREADS);
            {
                // growth across the compute warps' bands: rounds over the whole plane until nothing changes (usually one checking pass)
                const int NS = SW_THREADS - NC;
                const uint32_t a_edge = (j & 1) ? S.edge2 : S.edge, a_mask = S.mask + (j & 1) * mask_set_bytes;
                // the bands' interiors are at their fixed points: only rows next to a band boundary can still change
                int sw = 0;
                if (bar_or(4, NS, p3_check_band_boundaries(S.cand, a_edge, h, ww, (h + (NC >> 5) - 1) / (NC >> 5), tid - NC, NS)))
                    sw = p3_hysteresis(S.cand, a_edge, h, ww, tid - NC, NS, [NS](int c) { return bar_or(4, NS, c); });
                if (p.stats) {                                           // (the candidate plane is counted before the tail copy lands on it)
                    if (tid == NC) stat_add_one(S, 8, (unsigned long long)sw + 1);
                    count_planes<NR, true>(p, S, S.cand, a_edge, a_mask, Dm.plane_bytes, plane_words, tid - NC, NS);
                    bar_sync(4, NS);
                }
                if (tid == NC && tail_bytes) {                           // the candidate plane is dead: fetch the tail it was sitting in
                    const uint32_t fn = ring_frame(a_ring, j + 1);
                    if (fn < n) issue_frame_piece(S.pix[0], p.in + (size_t)plist_frame<LIST>(list, fn) * frame_bytes, main_bytes, frame_bytes, bar_tail);
                }
            }
            p4_output(P, Dm, pa, S.pix[0], p.out_u8 ? p.out_u8 + (size_t)f * frame_bytes : nullptr, p.out_f32 ? p.out_f32 + (size_t)f * frame_bytes : nullptr,
                      tid - NC, SW_THREADS - NC);
            __syncwarp();
            if (tid == NC) sts32(a_ring + 4 * (uint32_t)((j + 3) % FRAME_RING), ticket);      // (slot of frame j - 1: every reader is past it)
            if (lane == 0) mbar_arrive(bar_free + 8 * (j & 1));          // (use k of a plane set's barrier is its phase k: frame j + 2 waits for phase j >> 1)
        }
        if (p.stats) {                                                   // the store warps are the last to touch the counters
            bar_sync(4, SW_THREADS - NC);
            stats_flush(p, S, tid - NC);
        }
    }
}

// =========================================================================================================
// No colour filter, no edge filter (the reference's default configuration, core/config.py:22,25): __process is the brightness /
// contrast table alone (img_preprocessing.py:37-43), fused with the /255 tensor.  A pure stream: one CTA per frame at a time, the table
// of the frame in shared memory (static, or dynamic from the frame's rows 40..118), one 32-bit word in, one word + one 128-bit store out.
// Frame bytes and row bytes must be multiples of 4.
// =========================================================================================================
enum { ADJ_THREADS = 256 };
template <bool LIST = false>
__global__ void __launch_bounds__(ADJ_THREADS) k_adjust_stream(const __grid_constant__ PreKParams p, const FrameList fl = {})
{
    int n_list = 0;
    const int* list = nullptr;
    if constexpr (LIST) {
        plist_open(fl, list, n_list);
        if ((int)blockIdx.x >= n_list) return;
    }
    __shared__ __align__(16) uint8_t s_lut[256];
    __shared__ unsigned long long s_red[4 + 16];
    const int tid = threadIdx.x, nthr = blockDim.x, lane = tid & 31;
    const size_t frame_bytes = (size_t)p.h * p.w * 3;
    const int nwords = (int)(frame_bytes >> 2);
    const bool use_lut = p.dynamic || !p.lut_identity;
    const uint32_t a_lut = smem_u32(s_lut);
    const float rcp = 1.0f / 255.0f;
    for (int i = tid; i < 256; i += nthr) s_lut[i] = p.lut[i];
    for (int i = tid; i < 4 + 16; i += nthr) s_red[i] = 0;
    __syncthreads();
    for (int j = blockIdx.x; j < (LIST ? n_list : p.n); j += gridDim.x) {
        const int f = plist_frame<LIST>(list, j);
        const uint8_t* gfr = p.in + (size_t)f * frame_bytes;
        if (p.dynamic) {
            const float fdelta = dynamic_delta_global(p, gfr, s_red, tid, nthr, lane);
            for (int i = tid; i < 256; i += nthr) s_lut[i] = adjust_entry(i, true, fdelta, p.foff, p.fratio);
            __syncthreads();
        }
        const uint32_t* src = reinterpret_cast<const uint32_t*>(gfr);
        uint32_t* du8 = p.out_u8 ? reinterpret_cast<uint32_t*>(p.out_u8 + (size_t)f * frame_bytes) : nullptr;
        float4* df32 = p.out_f32 ? reinterpret_cast<float4*>(p.out_f32 + (size_t)f * frame_bytes) : nullptr;
        for (int i = tid; i < nwords; i += nthr) {
            uint32_t v = __ldg(src + i);
            if (use_lut) v = lut4s(a_lut, v);
            if (du8) du8[i] = v;
            if (df32) {
                float q[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const float x = (float)((v >> (8 * k)) & 0xffu);
                    const float q0 = __fmul_rn(x, rcp);
                    q[k] = __fmaf_rn(__fmaf_rn(-q0, 255.0f, x), rcp, q0);      // x / 255 correctly rounded (all 256 inputs checked)
                }
                df32[i] = make_float4(q[0], q[1], q[2], q[3]);
            }
        }
        if (p.dynamic) __syncthreads();                           // the table is rewritten for the next frame
    }
    if (p.stats) {
        __syncthreads();
        if (tid == 0) {
            const int mine = (int)blockIdx.x < (LIST ? n_list : p.n) ? ((LIST ? n_list : p.n) - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
            if (mine) atomicAdd(&p.stats[0], (unsigned long long)mine);
            if (s_red[4 + 9]) atomicAdd(&p.stats[9], s_red[4 + 9]);
        }
    }
}

}  // namespace trs
