// jpeg_enc_kernels.cuh — batched baseline-JPEG encode of tub records on the GPU (sm_100a); arithmetic in jpeg_enc_core.cuh.
//
// k_jpeg_encode<WRITE>: one CTA per record (grid stride), the record's MCUs in segments of JPE_SEG MCUs in MCU order, with the
// DC predictors, the bit position and the output position carried from one segment to the next.  Per segment:
//   1. the segment's 16 x 16 pixel tiles are loaded once (edge replication by clamped coordinates) and converted to Y / Cb / Cr
//      in shared memory;
//   2. one thread per 8 x 8 block: samples (h2v2 downsampling for chroma), FDCT, quantisation; the 64 zigzag coefficients stay in
//      the thread's registers, the quantised DC goes to shared memory (dummy luma blocks take the DC of the block before them);
//   3. each block's bit count from its coefficients and its predecessor's DC, a CTA-wide exclusive scan gives its bit offset;
//   4. every block ORs its bits into a shared word buffer at that offset (the buffer aliases the tiles);
//   5. the complete bytes are byte-stuffed: per-thread 0xFF counts, a second scan, and each byte (plus its 0x00) goes to its place.
// WRITE = false runs the same steps but only counts: it gives every record's exact file size, the host turns the sizes into
// offsets, and WRITE = true writes header + entropy-coded data + EOI of every record at its offset in one packed blob.  Computing
// twice costs arithmetic the link never sees, and no buffer is ever sized by a guess: the worst case (quality 100, maximum-entropy
// blocks) is about 200 KB per 120 x 160 record, 30 times a typical file.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "jpeg_enc_core.cuh"

namespace trs {

enum { JPE_THREADS = 256, JPE_SEG = 40 };                  // 40 MCUs = 240 blocks, one per thread
enum { JPE_BIT_WORDS = JPE_SEG * 6 * (JPE_MAX_BLOCK_BITS / 32) + 4 };

struct JpeSmem {
    JpeEncTables T;
    union {
        uint8_t tile[JPE_SEG][3][256];                   // Y, Cb, Cr of each MCU at full resolution
        uint32_t bits[JPE_BIT_WORDS];                    // the segment's bits (plus the carried partial byte), stream byte order
    } u;
    int dc[JPE_SEG * 6];
    uint32_t warp_sum[JPE_THREADS / 32];
    int carry_dc[3];
    uint32_t carry_byte, carry_bits;
    uint64_t out_pos;                                    // entropy-coded bytes of the record written so far (stuffing included)
};

// sink of jpe_encode_block: bits go to their offset in the shared buffer (MSB first; a word's bytes in stream order)
struct JpeSmemSink {
    uint32_t* w;
    uint32_t pos;
    __device__ __forceinline__ void put(uint32_t v, int len)
    {
        const uint64_t t = (uint64_t)v << (64 - (int)(pos & 31) - len);
        const uint32_t hi = (uint32_t)(t >> 32), lo = (uint32_t)t;
        if (hi) atomicOr(&w[pos >> 5], __byte_perm(hi, 0, 0x0123));
        if (lo) atomicOr(&w[(pos >> 5) + 1], __byte_perm(lo, 0, 0x0123));
        pos += (uint32_t)len;
    }
};

// exclusive scan over the CTA; returns this thread's prefix, *total the sum (all threads)
__device__ __forceinline__ uint32_t jpe_cta_scan(uint32_t v, uint32_t* warp_sum, uint32_t* total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    uint32_t x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) warp_sum[wid] = x;
    __syncthreads();
    uint32_t before = 0, all = 0;
#pragma unroll
    for (int k = 0; k < JPE_THREADS / 32; ++k) {
        const uint32_t s = warp_sum[k];
        before += k < wid ? s : 0;
        all += s;
    }
    __syncthreads();                                       // warp_sum may be reused by the next scan
    *total = all;
    return before + x - v;
}

template <bool WRITE>
__global__ void __launch_bounds__(JPE_THREADS) k_jpeg_encode(const uint8_t* __restrict__ frames, int n, int h, int w,
                                                             const JpeEncTables* __restrict__ tables, const uint8_t* __restrict__ header,
                                                             unsigned long long* __restrict__ sizes, const unsigned long long* __restrict__ offsets,
                                                             uint8_t* __restrict__ blob)
{
    extern __shared__ __align__(16) uint8_t smem_raw[];
    JpeSmem& S = *reinterpret_cast<JpeSmem*>(smem_raw);
    const int tid = threadIdx.x;
    for (int i = tid; i < (int)(sizeof(JpeEncTables) / 4); i += JPE_THREADS)
        reinterpret_cast<uint32_t*>(&S.T)[i] = reinterpret_cast<const uint32_t*>(tables)[i];
    const JpeGeom g = jpe_geom(h, w);
    const int n_mcu = g.mw * g.mh;
    uint8_t* const sbytes = reinterpret_cast<uint8_t*>(S.u.bits);

#pragma unroll 1
    for (int r = blockIdx.x; r < n; r += gridDim.x) {
        const uint8_t* img = frames + (size_t)r * h * w * 3;
        uint8_t* data = nullptr;
        if (WRITE) {
            uint8_t* file = blob + offsets[r];
            for (int i = tid; i < JPE_HEADER_BYTES; i += JPE_THREADS) file[i] = header[i];
            data = file + JPE_HEADER_BYTES;
        }
        if (tid == 0) { S.carry_dc[0] = S.carry_dc[1] = S.carry_dc[2] = 0; S.carry_byte = 0; S.carry_bits = 0; S.out_pos = 0; }
        __syncthreads();                                   // (also: the tables, and the previous record's last reads of the buffer)
#pragma unroll 1
        for (int m0 = 0; m0 < n_mcu; m0 += JPE_SEG) {
            const int nm = n_mcu - m0 < JPE_SEG ? n_mcu - m0 : JPE_SEG;
            const bool last = m0 + nm == n_mcu;
            // 1. tiles: clamped pixel loads, colour conversion once per pixel
            for (int i = tid; i < nm * 256; i += JPE_THREADS) {
                const int ml = i >> 8, p = i & 255, mcu = m0 + ml;
                const int my = mcu / g.mw, mx = mcu - my * g.mw;
                const int y = min(my * 16 + (p >> 4), h - 1), x = min(mx * 16 + (p & 15), w - 1);
                const uint8_t* px = img + ((size_t)y * w + x) * 3;
                int Y, Cb, Cr;
                jpe_rgb_to_ycc(__ldg(px), __ldg(px + 1), __ldg(px + 2), Y, Cb, Cr);
                S.u.tile[ml][0][p] = (uint8_t)Y; S.u.tile[ml][1][p] = (uint8_t)Cb; S.u.tile[ml][2][p] = (uint8_t)Cr;
            }
            __syncthreads();
            // 2. coefficients, one block per thread
            const bool mine = tid < nm * 6;
            const int ml = tid / 6, sub = tid - ml * 6, mcu = m0 + ml;
            const int my = mcu / g.mw, mx = mcu - my * g.mw;
            const int t = sub < 4 ? 0 : 1;
            int zz[64];
            bool dummy = false;
            if (mine) {
                dummy = jpe_dummy(g, my, mx, sub);
                if (dummy) {
#pragma unroll
                    for (int k = 0; k < 64; ++k) zz[k] = 0;
                } else {
                    int d[64];
                    jpe_block_samples(S.u.tile[ml][0], S.u.tile[ml][1], S.u.tile[ml][2], 16, g, my, sub, d);
                    jpe_block_coefficients(d, S.T.div[t], S.T.recip[t], zz);
                    S.dc[tid] = zz[0];
                }
            }
            __syncthreads();
            if (tid < nm)                                  // dummy luma blocks carry the DC of the block before them (never Y0)
                for (int s = 1; s < 4; ++s)
                    if (jpe_dummy(g, (m0 + tid) / g.mw, (m0 + tid) % g.mw, s)) S.dc[tid * 6 + s] = S.dc[tid * 6 + s - 1];
            __syncthreads();
            // 3. bit counts and offsets; the word buffer (no longer needed as tiles) is cleared meanwhile
            uint32_t len = 0;
            int diff = 0;
            if (mine) {
                const int dc = S.dc[tid];
                const int pred = sub >= 1 && sub <= 3 ? S.dc[tid - 1]
                               : (ml > 0 ? S.dc[sub == 0 ? tid - 3 : tid - 6] : S.carry_dc[sub == 0 ? 0 : sub - 3]);
                diff = dc - pred;
                JpeCountSink cs;
                jpe_encode_block(zz, diff, S.T.dc[t], S.T.ac[t], cs);
                len = cs.bits;
            }
            for (int i = tid; i < JPE_BIT_WORDS; i += JPE_THREADS) S.u.bits[i] = 0;
            uint32_t seg_bits;
            const uint32_t off = jpe_cta_scan(len, S.warp_sum, &seg_bits);     // (its barriers also order the clearing)
            const uint32_t carry_bits = S.carry_bits;
            // 4. bits to their offsets
            if (tid == 0) {
                S.u.bits[0] = S.carry_byte;                                    // the partial byte of the previous segment
                S.carry_dc[0] = S.dc[(nm - 1) * 6 + 3]; S.carry_dc[1] = S.dc[(nm - 1) * 6 + 4]; S.carry_dc[2] = S.dc[(nm - 1) * 6 + 5];
            }
            __syncthreads();
            if (mine) {
                JpeSmemSink sk{S.u.bits, carry_bits + off};
                jpe_encode_block(zz, diff, S.T.dc[t], S.T.ac[t], sk);
            }
            const uint32_t end = carry_bits + seg_bits;
            if (last && (end & 7) && tid == 0) {                               // jchuff.c flush_bits: pad with 1-bits
                JpeSmemSink sk{S.u.bits, end};
                sk.put((1u << (8 - (end & 7))) - 1u, 8 - (int)(end & 7));
            }
            __syncthreads();
            // 5. byte stuffing of the complete bytes: contiguous word ranges per thread, a scan over their 0xFF counts
            const uint32_t nbytes = last ? (end + 7) >> 3 : end >> 3;
            const uint32_t nwords = (nbytes + 3) >> 2, per = (nwords + JPE_THREADS - 1) / JPE_THREADS;
            const uint32_t b0 = min(tid * per * 4, nbytes), b1 = min(b0 + per * 4, nbytes);
            uint32_t ff = 0;
            for (uint32_t b = b0; b < b1; ++b) ff += sbytes[b] == 0xff;
            uint32_t ff_all;
            const uint32_t ff_before = jpe_cta_scan(ff, S.warp_sum, &ff_all);
            const uint64_t pos = S.out_pos;
            if (WRITE) {
                uint8_t* o = data + pos + b0 + ff_before;
                for (uint32_t b = b0; b < b1; ++b) {
                    const uint8_t v = sbytes[b];
                    *o++ = v;
                    if (v == 0xff) *o++ = 0;
                }
            }
            __syncthreads();                                                    // everyone has read out_pos and the bytes
            if (tid == 0) {
                S.out_pos = pos + nbytes + ff_all;
                S.carry_bits = end & 7;
                S.carry_byte = last ? 0u : sbytes[nbytes];
            }
            __syncthreads();
        }
        if (tid == 0) {
            if (WRITE) { data[S.out_pos] = 0xff; data[S.out_pos + 1] = 0xd9; }
            else sizes[r] = JPE_HEADER_BYTES + S.out_pos + 2;
        }
    }
}

}  // namespace trs
