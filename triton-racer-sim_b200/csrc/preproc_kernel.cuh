// preproc_kernel.cuh — the fused per-frame observation kernel (sm_100a).
//
// Replaces ImgPreprocessing.__process (TritonRacerSim/components/img_preprocessing.py:37-102) fused with the
// pilot's /255 normalisation (components/keras_pilot.py:49-50) for N frames.  One CTA owns one frame at a
// time (persistent loop over frames); everything between the single global read of the frame and the single
// global write of the outputs stays in shared memory:
//
//   P0  band of pixel rows (+2 halo rows, +1 halo pixel, borders replicated)  -> smem, through the
//       brightness/contrast table when it is not the identity                  (:81-102)
//   P1  3-channel Sobel, L1 magnitude, strongest channel, direction class      -> smem u16 plane (:79)
//       RGB->HSV fixed point + inRange per colour range                        -> smem bit planes (:65-74)
//   P2  non-maximum suppression                                                -> candidate / strong bit planes
//   P3  hysteresis on the bit planes (word-parallel flood fill to a fixed point)
//   P4  merge (:57-62) + normalise; u8 and/or f32 written once, coalesced
//
// Frames taller than the shared-memory budget are processed in row bands (P0-P2 per band, then P3, P4).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "pixel_math.cuh"
#include "preproc_list.h"

namespace trs {

enum { SRC_PIXEL = 0, SRC_MASK0 = 1, SRC_EDGE = 5 };
enum { PRE_THREADS = 512, HYST_RUN = 8 };

struct PreKParams {
    const uint8_t* in;
    uint8_t* out_u8;
    float* out_f32;
    unsigned long long* stats;
    uint16_t* dbg_mag;      // debug taps: frame 0 only
    uint8_t* dbg_map;
    uint32_t* frame_ctr;    // frame tickets of this launch (store-warp kernels, preproc_fast.cuh draw_frames): zeroed in stream order before it
    int n, h, w;
    int band_h;             // image rows per band
    int row_stride;         // bytes per smem pixel row (16-byte multiple; pixels start at +16)
    int mag_stride;         // u16 elements per smem magnitude row (w + 2, rounded up to even)
    int wwords;             // 32-pixel words per row
    int word_io;            // 1: frame bytes and row bytes are multiples of 4 and bases are 4-aligned
    // brightness / contrast
    int lut_identity;
    int dynamic;
    float foff, fratio;
    double baseline;
    uint8_t lut[256];       // static table (dynamic == 0)
    // colour ranges that can reach the output (host drops overwritten ones)
    int n_ranges;
    HsvRange ranges[4];
    int range_stat[4];      // original index of each kept range (for the statistics slots)
    // edge filter
    int edge_enabled;
    int low, high;
    // merge: source of each output channel
    int src[3];
    int need_pixels;        // some channel keeps the adjusted pixel
};

struct PreSmemLayout {
    int pix_off, mag_off, cand_off, edge_off, mask_off, tab_off, lut_off, red_off, total;
};

__host__ __device__ inline PreSmemLayout pre_smem_layout(int h, int w, int band_h, int row_stride, int mag_stride,
                                                        int wwords, int n_ranges)
{
    PreSmemLayout L;
    int o = 0;
    L.pix_off = o;  o += (band_h + 4) * row_stride + 32;
    L.mag_off = o;  o += ((band_h + 2) * mag_stride * 2 + 15) & ~15;
    const int plane = ((h * wwords * 4) + 15) & ~15;
    L.cand_off = o; o += plane;
    L.edge_off = o; o += plane;
    L.mask_off = o; o += plane * n_ranges;
    L.tab_off = o;  o += 2048;
    L.lut_off = o;  o += 256;
    L.red_off = o;  o += 256;
    L.total = o;
    return L;
}

// Flood the seed bits along the runs of ones of `c` (seeds must be a subset of c), both directions, O(1).
__device__ __forceinline__ uint32_t flood_word(uint32_t seeds, uint32_t c)
{
    const uint32_t up = (c & ~(c + seeds)) | seeds;          // carry ripples up through each run
    const uint32_t cr = __brev(c), sr = __brev(seeds);
    const uint32_t dn = __brev((cr & ~(cr + sr)) | sr);
    return up | dn;
}

__device__ __forceinline__ uint32_t lut4(const uint8_t* lut, uint32_t v)
{
    return (uint32_t)lut[v & 0xff] | ((uint32_t)lut[(v >> 8) & 0xff] << 8) | ((uint32_t)lut[(v >> 16) & 0xff] << 16) |
           ((uint32_t)lut[v >> 24] << 24);
}

// LIST (trs_preprocess_configs): the launch works on the frames of one bucket (preproc_list.h), the frame count read from fl; the CTAs
// without a first frame leave at once.
template <bool LIST = false>
__global__ void __launch_bounds__(PRE_THREADS, 1) k_preprocess(const __grid_constant__ PreKParams p, const FrameList fl = {})
{
    int n_list = 0;
    const int* list = nullptr;
    if constexpr (LIST) {
        plist_open(fl, list, n_list);
        if ((int)blockIdx.x >= n_list) return;
    }
    extern __shared__ __align__(16) uint8_t smem[];
    const PreSmemLayout L = pre_smem_layout(p.h, p.w, p.band_h, p.row_stride, p.mag_stride, p.wwords, p.n_ranges);
    uint8_t* s_pix = smem + L.pix_off;
    uint16_t* s_mag = reinterpret_cast<uint16_t*>(smem + L.mag_off);
    uint32_t* s_cand = reinterpret_cast<uint32_t*>(smem + L.cand_off);
    uint32_t* s_edge = reinterpret_cast<uint32_t*>(smem + L.edge_off);
    uint32_t* s_mask = reinterpret_cast<uint32_t*>(smem + L.mask_off);
    int32_t* s_sdiv = reinterpret_cast<int32_t*>(smem + L.tab_off);
    int32_t* s_hdiv = s_sdiv + 256;
    uint8_t* s_lut = smem + L.lut_off;
    unsigned long long* s_red = reinterpret_cast<unsigned long long*>(smem + L.red_off);

    const int tid = threadIdx.x, nthr = blockDim.x;
    const int lane = tid & 31, warp = tid >> 5, nwarps = nthr >> 5;
    const int h = p.h, w = p.w, wwords = p.wwords;
    const int row_bytes = w * 3;
    const size_t frame_bytes = (size_t)h * row_bytes;
    const int plane_words = h * wwords;

    // tables that do not change per frame
    for (int i = tid; i < 256; i += nthr) {
        // rint((255<<12)/i) and rint((180<<12)/(6 i)): IEEE double division + round-half-even, as OpenCV builds them
        s_sdiv[i] = i ? __double2int_rn((double)(255 << 12) / (double)i) : 0;
        s_hdiv[i] = i ? __double2int_rn((double)(180 << 12) / (6.0 * (double)i)) : 0;
        s_lut[i] = p.lut[i];
    }
    unsigned long long st_mask[4] = {0, 0, 0, 0};
    unsigned long long st_edge = 0, st_strong = 0, st_cand = 0, st_sweeps = 0, st_roi = 0, st_frames = 0;
    __syncthreads();

    for (int j = blockIdx.x; j < (LIST ? n_list : p.n); j += gridDim.x) {
        const int f = LIST ? list[j] : j;
        const uint8_t* __restrict__ gin = p.in + (size_t)f * frame_bytes;

        // ---- dynamic brightness: ROI sums (rows 40..118) -> per-frame table -------------------------------
        if (p.dynamic) {
            const int y0 = min(40, h), y1 = min(119, h);
            unsigned long long s0 = 0, s1 = 0, s2 = 0;
            const int npix = (y1 - y0) * w;
            const uint8_t* roi = gin + (size_t)y0 * row_bytes;
            for (int i = tid; i < npix; i += nthr) {
                s0 += roi[3 * i]; s1 += roi[3 * i + 1]; s2 += roi[3 * i + 2];
            }
            for (int o = 16; o; o >>= 1) {
                s0 += __shfl_xor_sync(0xffffffffu, s0, o);
                s1 += __shfl_xor_sync(0xffffffffu, s1, o);
                s2 += __shfl_xor_sync(0xffffffffu, s2, o);
            }
            if (tid < 3) s_red[tid] = 0;
            __syncthreads();
            if (lane == 0) { atomicAdd(&s_red[0], s0); atomicAdd(&s_red[1], s1); atomicAdd(&s_red[2], s2); }
            __syncthreads();
            const double delta = brightness_delta(s_red[0], s_red[1], s_red[2], (double)npix, p.baseline);
            const float fdelta = (float)delta;
            if (tid == 0) st_roi += s_red[0] + s_red[1] + s_red[2];
            __syncthreads();
            for (int i = tid; i < 256; i += nthr) s_lut[i] = adjust_entry(i, true, fdelta, p.foff, p.fratio);
            __syncthreads();
        }
        const bool use_lut = p.dynamic || !p.lut_identity;

        // mask planes are written word by word in P1; cand/edge in P2 — no clearing needed.
        for (int by0 = 0; by0 < h; by0 += p.band_h) {
            const int by1 = min(h, by0 + p.band_h);
            const int prow0 = by0 - 2;                    // image row of smem pixel row 0
            const int nprow = (by1 - by0) + 4;
            const int mrow0 = by0 - 1;                    // image row of smem magnitude row 0
            const int nmrow = (by1 - by0) + 2;

            // ---- P0: pixels -> smem (rows replicated at the frame border), zero the magnitude plane --------
            if (p.edge_enabled || p.n_ranges > 0) {
                if (p.word_io) {
                    const int wpr = row_bytes >> 2;
                    for (int i = tid; i < nprow * wpr; i += nthr) {
                        const int r = i / wpr, j = i - r * wpr;
                        const int yy = min(max(prow0 + r, 0), h - 1);
                        uint32_t v = __ldg(reinterpret_cast<const uint32_t*>(gin + (size_t)yy * row_bytes) + j);
                        if (use_lut) v = lut4(s_lut, v);
                        *reinterpret_cast<uint32_t*>(s_pix + r * p.row_stride + 16 + 4 * j) = v;
                    }
                } else {
                    for (int i = tid; i < nprow * row_bytes; i += nthr) {
                        const int r = i / row_bytes, j = i - r * row_bytes;
                        const int yy = min(max(prow0 + r, 0), h - 1);
                        uint8_t v = gin[(size_t)yy * row_bytes + j];
                        if (use_lut) v = s_lut[v];
                        s_pix[r * p.row_stride + 16 + j] = v;
                    }
                }
                for (int i = tid; i < nprow * 6; i += nthr) {   // 1-pixel replicated halo left and right
                    const int r = i / 6, k = i - r * 6;
                    const int yy = min(max(prow0 + r, 0), h - 1);
                    const int c = k % 3;
                    const bool right = k >= 3;
                    uint8_t v = gin[(size_t)yy * row_bytes + (right ? (w - 1) * 3 : 0) + c];
                    if (use_lut) v = s_lut[v];
                    s_pix[r * p.row_stride + (right ? 16 + row_bytes : 13) + c] = v;
                }
                if (p.edge_enabled) {
                    uint32_t* z = reinterpret_cast<uint32_t*>(s_mag);
                    for (int i = tid; i < (nmrow * p.mag_stride) >> 1; i += nthr) z[i] = 0;
                }
            }
            __syncthreads();

            // ---- P1: Sobel + magnitude/direction for rows [by0-1, by1+1); colour masks for rows [by0, by1) ----
            {
                const int ya = p.edge_enabled ? max(mrow0, 0) : by0;
                const int yb = p.edge_enabled ? min(by1 + 1, h) : by1;
                const int ntask = (p.edge_enabled || p.n_ranges > 0) ? (yb - ya) * wwords : 0;
                for (int t = warp; t < ntask; t += nwarps) {
                    const int y = ya + t / wwords, wi = t % wwords;
                    const int x = wi * 32 + lane;
                    const bool valid = x < w;
                    const int xs = valid ? x : w - 1;
                    const uint8_t* c1 = s_pix + (y - prow0) * p.row_stride + 16 + xs * 3;   // centre pixel
                    const uint8_t* c0 = c1 - p.row_stride;
                    const uint8_t* c2 = c1 + p.row_stride;
                    if (p.edge_enabled) {
                        int bm = -1, bdx = 0, bdy = 0;
#pragma unroll
                        for (int c = 0; c < 3; ++c) {
                            const int a0 = c0[c - 3], a1 = c0[c], a2 = c0[c + 3];
                            const int m0 = c1[c - 3], m2 = c1[c + 3];
                            const int b0 = c2[c - 3], b1 = c2[c], b2 = c2[c + 3];
                            const int dx = (a2 - a0) + 2 * (m2 - m0) + (b2 - b0);
                            const int dy = (b0 - a0) + 2 * (b1 - a1) + (b2 - a2);
                            const int m = abs(dx) + abs(dy);
                            if (m > bm) { bm = m; bdx = dx; bdy = dy; }
                        }
                        if (valid) s_mag[(y - mrow0) * p.mag_stride + x + 1] = pack_mag(bm, canny_dir(bdx, bdy));
                        if (p.dbg_mag && f == 0 && valid && y >= by0 && y < by1) p.dbg_mag[y * w + x] = (uint16_t)bm;
                    }
                    if (p.n_ranges > 0 && y >= by0 && y < by1) {
                        int hh, ss, vv;
                        rgb2hsv_px(c1[0], c1[1], c1[2], s_sdiv, s_hdiv, hh, ss, vv);
                        for (int k = 0; k < p.n_ranges; ++k) {
                            const uint32_t bits = __ballot_sync(0xffffffffu, valid && in_range_px(hh, ss, vv, p.ranges[k]));
                            if (lane == 0) s_mask[k * plane_words + y * wwords + wi] = bits;
                        }
                    }
                }
            }
            __syncthreads();

            // ---- P2: non-maximum suppression for rows [by0, by1) -----------------------------------------
            if (p.edge_enabled) {
                const int ntask = (by1 - by0) * wwords;
                for (int t = warp; t < ntask; t += nwarps) {
                    const int y = by0 + t / wwords, wi = t % wwords;
                    const int x = wi * 32 + lane;
                    const bool valid = x < w;
                    const uint16_t* mc = s_mag + (y - mrow0) * p.mag_stride + (valid ? x : 0) + 1;
                    const uint16_t cw = *mc;
                    const int m = mag_of(cw);
                    bool is_cand = false;
                    if (valid && m > p.low) {
                        const uint16_t* mu = mc - p.mag_stride;
                        const uint16_t* md = mc + p.mag_stride;
                        is_cand = canny_is_max(m, dir_of(cw), mag_of(mc[-1]), mag_of(mc[1]), mag_of(mu[0]), mag_of(md[0]),
                                               mag_of(mu[-1]), mag_of(mu[1]), mag_of(md[-1]), mag_of(md[1]));
                    }
                    const bool is_strong = is_cand && m > p.high;
                    const uint32_t cb = __ballot_sync(0xffffffffu, is_cand);
                    const uint32_t sb = __ballot_sync(0xffffffffu, is_strong);
                    if (lane == 0) {
                        s_cand[y * wwords + wi] = cb;
                        s_edge[y * wwords + wi] = sb;
                        st_cand += __popc(cb);
                        st_strong += __popc(sb);
                    }
                    if (p.dbg_map && f == 0 && valid) p.dbg_map[y * w + x] = is_strong ? 2 : (is_cand ? 1 : 0);
                }
            }
            __syncthreads();
        }

        // ---- P3: hysteresis — grow the strong set through candidates until nothing changes -----------------
        if (p.edge_enabled) {
            volatile uint32_t* E = s_edge;
            const int nruns = (h + HYST_RUN - 1) / HYST_RUN;
            const int ntask = nruns * wwords;
            int any;
            do {
                int changed = 0;
                for (int t = tid; t < ntask; t += nthr) {
                    const int wi = t % wwords, run = t / wwords;
                    const int ylo = run * HYST_RUN, yhi = min(h, ylo + HYST_RUN);
                    for (int pass = 0; pass < 2; ++pass) {
                        for (int k = 0; k < yhi - ylo; ++k) {
                            const int y = pass == 0 ? ylo + k : yhi - 1 - k;
                            const uint32_t c = s_cand[y * wwords + wi];
                            if (!c) continue;
                            const uint32_t e = E[y * wwords + wi];
                            if (e == c) continue;
                            uint32_t mid = e, lft = 0, rgt = 0;
                            for (int dy = -1; dy <= 1; ++dy) {
                                const int yy = y + dy;
                                if (yy < 0 || yy >= h) continue;
                                mid |= E[yy * wwords + wi];
                                if (wi > 0) lft |= E[yy * wwords + wi - 1];
                                if (wi + 1 < wwords) rgt |= E[yy * wwords + wi + 1];
                            }
                            const uint32_t spread = mid | (mid << 1) | (mid >> 1) | (lft >> 31) | (rgt << 31);
                            const uint32_t ne = flood_word((spread & c) | e, c);
                            if (ne != e) { E[y * wwords + wi] = ne; changed = 1; }
                        }
                    }
                }
                any = __syncthreads_or(changed);
                if (tid == 0) ++st_sweeps;
            } while (any);
        }

        // ---- P4: merge + normalise, written once -------------------------------------------------------
        {
            uint8_t* __restrict__ gout = p.out_u8 ? p.out_u8 + (size_t)f * frame_bytes : nullptr;
            float* __restrict__ gf32 = p.out_f32 ? p.out_f32 + (size_t)f * frame_bytes : nullptr;
            const uint32_t* planes[3];
            for (int c = 0; c < 3; ++c)
                planes[c] = p.src[c] == SRC_EDGE ? s_edge : (p.src[c] >= SRC_MASK0 ? s_mask + (p.src[c] - SRC_MASK0) * plane_words : nullptr);
            if (p.word_io && (w & 3) == 0) {
                const int gpr = w >> 2;                     // groups of 4 pixels per row
                for (int g = tid; g < h * gpr; g += nthr) {
                    const int y = g / gpr, x0 = (g - y * gpr) * 4;
                    uint32_t wv[3] = {0, 0, 0};
                    if (p.need_pixels) {
                        const uint32_t* src = reinterpret_cast<const uint32_t*>(gin + (size_t)y * row_bytes + x0 * 3);
                        wv[0] = __ldg(src); wv[1] = __ldg(src + 1); wv[2] = __ldg(src + 2);
                        if (use_lut) { wv[0] = lut4(s_lut, wv[0]); wv[1] = lut4(s_lut, wv[1]); wv[2] = lut4(s_lut, wv[2]); }
                    }
                    uint8_t b[12];
#pragma unroll
                    for (int k = 0; k < 12; ++k) b[k] = (uint8_t)(wv[k >> 2] >> ((k & 3) * 8));
                    const int wi = x0 >> 5, sh = x0 & 31;
#pragma unroll
                    for (int c = 0; c < 3; ++c) {
                        if (planes[c]) {
                            const uint32_t bits = planes[c][y * wwords + wi] >> sh;
#pragma unroll
                            for (int q = 0; q < 4; ++q) b[q * 3 + c] = ((bits >> q) & 1u) ? 255 : 0;
                        }
                    }
                    if (gout) {
                        uint32_t* dst = reinterpret_cast<uint32_t*>(gout + (size_t)y * row_bytes + x0 * 3);
#pragma unroll
                        for (int k = 0; k < 3; ++k)
                            dst[k] = (uint32_t)b[4 * k] | ((uint32_t)b[4 * k + 1] << 8) | ((uint32_t)b[4 * k + 2] << 16) | ((uint32_t)b[4 * k + 3] << 24);
                    }
                    if (gf32) {
                        float4* dst = reinterpret_cast<float4*>(gf32 + (size_t)y * row_bytes + x0 * 3);
#pragma unroll
                        for (int k = 0; k < 3; ++k)
                            dst[k] = make_float4(__fdiv_rn((float)b[4 * k], 255.0f), __fdiv_rn((float)b[4 * k + 1], 255.0f),
                                                 __fdiv_rn((float)b[4 * k + 2], 255.0f), __fdiv_rn((float)b[4 * k + 3], 255.0f));
                    }
                }
            } else {
                for (int i = tid; i < h * w; i += nthr) {
                    const int y = i / w, x = i - y * w;
                    for (int c = 0; c < 3; ++c) {
                        uint8_t v;
                        if (planes[c]) v = ((planes[c][y * wwords + (x >> 5)] >> (x & 31)) & 1u) ? 255 : 0;
                        else { v = gin[(size_t)i * 3 + c]; if (use_lut) v = s_lut[v]; }
                        if (gout) gout[(size_t)i * 3 + c] = v;
                        if (gf32) gf32[(size_t)i * 3 + c] = __fdiv_rn((float)v, 255.0f);
                    }
                }
            }
        }
        // ---- statistics (plane population counts) ------------------------------------------------------
        if (p.stats) {
            for (int i = tid; i < plane_words; i += nthr) {
                if (p.edge_enabled) st_edge += __popc(s_edge[i]);
                for (int k = 0; k < p.n_ranges; ++k) st_mask[k] += __popc(s_mask[k * plane_words + i]);
            }
            if (tid == 0) ++st_frames;
        }
        __syncthreads();      // planes and the table are reused by the next frame
    }

    if (p.stats) {
        unsigned long long v[10] = {st_frames, 0, 0, 0, 0, st_edge, st_strong, st_cand, st_sweeps, st_roi};
        for (int k = 0; k < p.n_ranges; ++k) v[1 + p.range_stat[k]] = st_mask[k];
#pragma unroll
        for (int k = 0; k < 10; ++k) {
            unsigned long long x = v[k];
            for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if (lane == 0 && x) atomicAdd(&p.stats[k], x);
        }
    }
}

// trs_preprocess_configs: the frames of bucket fl.cfg = K, whose configuration index is outside [0, K), get u8 0 and f32 NaN (the -1 / NaN of
// trs_locate_tracks' out-of-range cars), a CTA per frame at a time.
enum { UNCFG_THREADS = 256 };
__global__ void __launch_bounds__(UNCFG_THREADS) k_preprocess_unconfigured(const FrameList fl, size_t frame_bytes, uint8_t* __restrict__ out_u8,
                                                                          float* __restrict__ out_f32)
{
    const int* list;
    int n;
    plist_open(fl, list, n);
    for (int j = blockIdx.x; j < n; j += gridDim.x) {
        const size_t base = (size_t)list[j] * frame_bytes;
        for (size_t i = threadIdx.x; i < frame_bytes; i += UNCFG_THREADS) {
            if (out_u8) out_u8[base + i] = 0;
            if (out_f32) out_f32[base + i] = __int_as_float(0x7fc00000);
        }
    }
}

}  // namespace trs
