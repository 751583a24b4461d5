// misc_kernels.cuh — normalise/crop/resize, waypoint lookup, speed control (sm_100a).
#pragma once
#include "loc_grid.h"
#include <cuda_runtime.h>
#include <stdint.h>

namespace trs {

// ------------------------------------------------------------------------------------------------------
// K1a: pure streaming normalise, u8 -> f32 (keras_pilot.py:49-50; keras_train.py:41-42).
// One thread converts one 32-bit word (4 bytes) into one 128-bit store, so consecutive lanes read consecutive
// words (128 B per warp load) and write consecutive 16-byte chunks (512 contiguous bytes per warp store); UNROLL
// independent words per thread keep enough loads in flight.  (A 16-bytes-in / 64-bytes-out per thread mapping
// makes every store instruction touch 32 half-written sectors and was measured at 47 % of the HBM roofline.)
// 1/255 is not exactly representable: the quotient must be correctly rounded (126 of 256 inputs differ otherwise).
// x / 255 = q0 + (x - 255 q0) / 255 with q0 = x * fl(1/255): one fused residual correction gives the correctly
// rounded quotient for every x in 0..255 (checked exhaustively: tests/test_oracle_golden.py, tests/test_gpu_parity.py).
// The byte -> float conversion avoids the quarter-rate I2F: 0x4B000000 | b is the float 2^23 + b.
// ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float norm255(uint32_t b) { return __fdiv_rn((float)b, 255.0f); }

__device__ __forceinline__ float norm255_fast(uint32_t word, uint32_t sel)
{
    const float x = __fsub_rn(__uint_as_float(__byte_perm(word, 0x4B000000u, sel)), 8388608.0f);
    const float rcp = 1.0f / 255.0f;
    const float q0 = __fmul_rn(x, rcp);
    return __fmaf_rn(__fmaf_rn(-q0, 255.0f, x), rcp, q0);
}

__device__ __forceinline__ uint32_t ldg_stream32(const uint32_t* p)
{
    uint32_t r;
    asm volatile("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ void stg_stream(float4* p, float4 v)
{
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

__device__ __forceinline__ float4 norm_word(uint32_t w)
{
    // selectors: output byte 0 = source byte k, bytes 1..3 = bytes 5,6,7 of the pair = 0x00,0x00,0x4B
    return make_float4(norm255_fast(w, 0x7650), norm255_fast(w, 0x7651), norm255_fast(w, 0x7652), norm255_fast(w, 0x7653));
}

template <int UNROLL>
__global__ void __launch_bounds__(256) k_normalise_stream(const uint32_t* __restrict__ in, float4* __restrict__ out, size_t n_words)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (; i + (UNROLL - 1) * stride < n_words; i += UNROLL * stride) {
        uint32_t v[UNROLL];
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) v[u] = ldg_stream32(in + i + u * stride);
#pragma unroll
        for (int u = 0; u < UNROLL; ++u) stg_stream(out + i + u * stride, norm_word(v[u]));
    }
    for (; i < n_words; i += stride) stg_stream(out + i, norm_word(ldg_stream32(in + i)));
}

// tail / unaligned fallback: one byte per thread
__global__ void k_normalise_bytes(const uint8_t* __restrict__ in, float* __restrict__ out, size_t n)
{
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) out[i] = norm255(in[i]);
}

// ------------------------------------------------------------------------------------------------------
// K1b: window crop + nearest resize (camera.py:36: src = floor(dst * size_src / size_dst)) + normalise.
// One thread per output pixel; lanes walk along the output row so the source reads of a warp fall in one
// or two source rows (2:1 down-scale touches every other pixel: half of each fetched sector is used).
// ------------------------------------------------------------------------------------------------------
struct ResizeParams {
    const uint8_t* in;
    float* out_f32;
    uint8_t* out_u8;
    int n, h_in, w_in, y0, x0, hs, ws, h_out, w_out;
};

__global__ void __launch_bounds__(256) k_crop_resize(const __grid_constant__ ResizeParams p)
{
    const size_t total = (size_t)p.n * p.h_out * p.w_out;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        const int x = (int)(i % p.w_out);
        const size_t t = i / p.w_out;
        const int y = (int)(t % p.h_out);
        const size_t f = t / p.h_out;
        const int sy = p.y0 + (int)(((long long)y * p.hs) / p.h_out);
        const int sx = p.x0 + (int)(((long long)x * p.ws) / p.w_out);
        const uint8_t* s = p.in + ((f * p.h_in + sy) * p.w_in + sx) * 3;
        const uint8_t r = s[0], g = s[1], b = s[2];
        if (p.out_u8) { uint8_t* o = p.out_u8 + i * 3; o[0] = r; o[1] = g; o[2] = b; }
        if (p.out_f32) { float* o = p.out_f32 + i * 3; o[0] = norm255(r); o[1] = norm255(g); o[2] = norm255(b); }
    }
}

// K1c: the same, one output WORD per thread (output rows a multiple of 4 bytes, outputs 16-byte aligned): the source
// column / row of every output pixel comes from two small shared-memory tables built once per CTA (no division per
// pixel), a thread gathers the 4 source bytes of its word (L1-resident sectors) and writes one 16-byte f32 chunk and one
// 4-byte u8 word, so a warp's stores are 512 / 128 contiguous bytes.  A CTA walks whole output rows.
enum { RESIZE_THREADS = 128, RESIZE_MAX_TAB = 8192, RESIZE_DEPTH = 8 };

__global__ void __launch_bounds__(RESIZE_THREADS) k_crop_resize_words(const __grid_constant__ ResizeParams p)
{
    extern __shared__ int s_tab[];                 // [w_out] source byte offset of column x, then [h_out] source row of row y
    int* s_sx = s_tab;
    int* s_sy = s_tab + p.w_out;
    for (int x = threadIdx.x; x < p.w_out; x += blockDim.x) s_sx[x] = 3 * (p.x0 + (int)(((long long)x * p.ws) / p.w_out));
    for (int y = threadIdx.x; y < p.h_out; y += blockDim.x) s_sy[y] = p.y0 + (int)(((long long)y * p.hs) / p.h_out);
    __syncthreads();
    const int wpr = (p.w_out * 3) >> 2;            // output words per row
    const size_t rows = (size_t)p.n * p.h_out;
    const size_t src_row_bytes = (size_t)p.w_in * 3;
    const float rcp = 1.0f / 255.0f;
    for (size_t R = blockIdx.x; R < rows; R += gridDim.x) {
        const size_t f = R / p.h_out;
        const int y = (int)(R - f * p.h_out);
        const uint8_t* __restrict__ src = p.in + (f * p.h_in + s_sy[y]) * src_row_bytes;
        for (int c = threadIdx.x; c < wpr; c += blockDim.x) {
            uint32_t word = 0;
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const int o = 4 * c + j, px = o / 3, ch = o - 3 * px;
                const uint32_t b = __ldg(src + s_sx[px] + ch);
                word |= b << (8 * j);
                const float xf = __fsub_rn(__uint_as_float(0x4B000000u | b), 8388608.0f);
                const float q0 = __fmul_rn(xf, rcp);
                v[j] = __fmaf_rn(__fmaf_rn(-q0, 255.0f, xf), rcp, q0);          // correctly rounded x / 255 (see norm255_fast)
            }
            if (p.out_f32) stg_stream(reinterpret_cast<float4*>(p.out_f32) + R * wpr + c, make_float4(v[0], v[1], v[2], v[3]));
            if (p.out_u8) reinterpret_cast<uint32_t*>(p.out_u8)[R * wpr + c] = word;
        }
    }
}

// K1d: the same with the source row staged in shared memory.  K1c gathers its bytes with one byte load each; here the part of the
// source row the window needs arrives by 16-byte asynchronous copies (LDGSTS), double-buffered across the rows a CTA walks, and
// the gather runs on shared memory with the four source offsets of an output word in one 16-byte table entry.  No division per
// row either: (frame, output row) advance by the grid stride with a carry.  Needs 16-byte aligned source rows.
__global__ void __launch_bounds__(RESIZE_THREADS) k_crop_resize_rows(const __grid_constant__ ResizeParams p, int col_lo, int span)
{
    extern __shared__ __align__(16) uint8_t s_dyn[];
    const int wpr = (p.w_out * 3) >> 2;            // output words per row
    int4* s_off = reinterpret_cast<int4*>(s_dyn);                                   // [wpr] source offsets (within the staged span) of a word's bytes
    int* s_sy = reinterpret_cast<int*>(s_dyn + sizeof(int4) * wpr);                 // [h_out] source row of row y
    uint8_t* s_row = s_dyn + ((sizeof(int4) * wpr + sizeof(int) * p.h_out + 15) & ~(size_t)15);   // 2 x span
    for (int c = threadIdx.x; c < wpr; c += blockDim.x) {
        int o[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int b = 4 * c + j, px = b / 3, ch = b - 3 * px;
            o[j] = 3 * (p.x0 + (int)(((long long)px * p.ws) / p.w_out)) + ch - col_lo;
        }
        s_off[c] = make_int4(o[0], o[1], o[2], o[3]);
    }
    for (int y = threadIdx.x; y < p.h_out; y += blockDim.x) s_sy[y] = p.y0 + (int)(((long long)y * p.hs) / p.h_out);
    __syncthreads();
    const size_t rows = (size_t)p.n * p.h_out;
    const size_t src_row_bytes = (size_t)p.w_in * 3;
    const int chunks = span >> 4;
    const float rcp = 1.0f / 255.0f;
    const int gq = (int)(gridDim.x / p.h_out), gr = (int)(gridDim.x % p.h_out);
    size_t f = blockIdx.x / p.h_out;
    int y = (int)(blockIdx.x - f * p.h_out);
    auto stage = [&](size_t ff, int yy, int buf) {
        const uint8_t* src = p.in + (ff * p.h_in + s_sy[yy]) * src_row_bytes + col_lo;
        const uint32_t dst = (uint32_t)__cvta_generic_to_shared(s_row + (size_t)buf * span);
        for (int i = threadIdx.x; i < chunks; i += blockDim.x)
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst + 16u * i), "l"(src + 16 * (size_t)i) : "memory");
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    // RESIZE_DEPTH rows in flight per CTA: the row being gathered and the next RESIZE_DEPTH - 1 being staged (one commit group per
    // row, empty past the end, so that "all but the newest RESIZE_DEPTH - 1 groups" always means "this row has landed")
    auto advance = [&](size_t& ff, int& yy) {
        ff += gq; yy += gr;
        if (yy >= p.h_out) { yy -= p.h_out; ++ff; }
    };
    size_t fs = f;                                                          // (frame, row) of the next row to stage
    int ys = y;
    size_t Rs = blockIdx.x;
    for (int d = 0; d < RESIZE_DEPTH - 1; ++d) {
        if (Rs < rows) stage(fs, ys, d);
        else asm volatile("cp.async.commit_group;" ::: "memory");
        Rs += gridDim.x; advance(fs, ys);
    }
    size_t R = blockIdx.x;
    for (uint32_t it = 0; R < rows; R += gridDim.x, ++it) {
        if (Rs < rows) stage(fs, ys, (it + RESIZE_DEPTH - 1) % RESIZE_DEPTH);
        else asm volatile("cp.async.commit_group;" ::: "memory");
        Rs += gridDim.x; advance(fs, ys);
        asm volatile("cp.async.wait_group %0;" ::"n"(RESIZE_DEPTH - 1) : "memory");
        __syncthreads();
        const uint8_t* row = s_row + (size_t)(it % RESIZE_DEPTH) * span;
        for (int c = threadIdx.x; c < wpr; c += blockDim.x) {
            const int4 o = s_off[c];
            const uint32_t b[4] = {row[o.x], row[o.y], row[o.z], row[o.w]};
            float v[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const float xf = __fsub_rn(__uint_as_float(0x4B000000u | b[j]), 8388608.0f);
                const float q0 = __fmul_rn(xf, rcp);
                v[j] = __fmaf_rn(__fmaf_rn(-q0, 255.0f, xf), rcp, q0);          // correctly rounded x / 255 (see norm255_fast)
            }
            if (p.out_f32) stg_stream(reinterpret_cast<float4*>(p.out_f32) + R * wpr + c, make_float4(v[0], v[1], v[2], v[3]));
            if (p.out_u8) reinterpret_cast<uint32_t*>(p.out_u8)[R * wpr + c] = b[0] | (b[1] << 8) | (b[2] << 16) | (b[3] << 24);
        }
        __syncthreads();                                                    // this buffer is restaged in the next iteration
    }
}

// ------------------------------------------------------------------------------------------------------
// K6: nearest waypoint, L1 distance in float64, first index wins ties, running minimum starts at 100
// (track_data_process.py:89-107).  The centre line sits in shared memory as (x,y,z,pad) f64 quads; every lane
// of a warp reads the same waypoint (broadcast), each thread carries CARS cars so one shared-memory read
// feeds CARS distance evaluations.  Distances are summed left to right exactly as the reference does.
// Recorded centre lines repeat points (generated_track: 917 distinct of 1,185; mountain_track: 1,260 of 2,664): a repeat can never win
// the strict `<` against its first occurrence, so the host uploads only the first occurrences, in order, as (x, y, z, original index)
// quads, and the kernels return the original index: fewer evaluations, the reference's argmin bit for bit.  n_wp = points the reference
// loops over (the divisor of the segment map), n_u = distinct points evaluated here.
// ------------------------------------------------------------------------------------------------------
enum { LOC_THREADS = 256, LOC_CARS = 2, LOC_TILE = 1024 };

__global__ void __launch_bounds__(LOC_THREADS) k_locate(const double4* __restrict__ wp, int n_u, int n_wp, double min_map, double max_map,
                                                       const double* __restrict__ xyz, int n, int32_t* __restrict__ idx_out,
                                                       double* __restrict__ seg_out)
{
    __shared__ double4 s_wp[LOC_TILE];
    const int base = (blockIdx.x * LOC_THREADS + threadIdx.x) * LOC_CARS;
    double px[LOC_CARS], py[LOC_CARS], pz[LOC_CARS], best[LOC_CARS];
    double sel[LOC_CARS];                                        // original index of the best point so far, as carried in the quad
#pragma unroll
    for (int c = 0; c < LOC_CARS; ++c) {
        const int k = min(base + c, n - 1);
        px[c] = xyz[3 * (size_t)k]; py[c] = xyz[3 * (size_t)k + 1]; pz[c] = xyz[3 * (size_t)k + 2];
        best[c] = 100.0; sel[c] = 0.0;
    }
    for (int t0 = 0; t0 < n_u; t0 += LOC_TILE) {
        const int tn = min(LOC_TILE, n_u - t0);
        __syncthreads();
        for (int i = threadIdx.x; i < tn; i += LOC_THREADS) s_wp[i] = wp[t0 + i];
        __syncthreads();
#pragma unroll 4
        for (int i = 0; i < tn; ++i) {
            const double4 q = s_wp[i];
#pragma unroll
            for (int c = 0; c < LOC_CARS; ++c) {
                const double d = __dadd_rn(__dadd_rn(fabs(__dsub_rn(px[c], q.x)), fabs(__dsub_rn(py[c], q.y))), fabs(__dsub_rn(pz[c], q.z)));
                if (d < best[c]) { best[c] = d; sel[c] = q.w; }
            }
        }
    }
#pragma unroll
    for (int c = 0; c < LOC_CARS; ++c) {
        const int k = base + c;
        if (k < n) {
            if (idx_out) idx_out[k] = (int)sel[c];
            if (seg_out) seg_out[k] = loct_segment((int)sel[c], n_wp, min_map, max_map);
        }
    }
}

// Measurement aid for K6's roofline (bench.py): the box's FP64 pipe rate.  ILP independent chains per thread of one fp64 instruction
// each (FMA = true: DFMA, 2 flops; false: DADD, 1 flop), 256 threads per CTA, enough CTAs to fill every SM.
enum { PROBE64_ILP = 8, PROBE64_THREADS = 256 };
template <bool FMA>
__global__ void __launch_bounds__(PROBE64_THREADS) k_probe_fp64(double* __restrict__ out, int iters, double a, double b)
{
    double r[PROBE64_ILP];
#pragma unroll
    for (int i = 0; i < PROBE64_ILP; ++i) r[i] = (double)(threadIdx.x + 1) * 1e-3 + i;
#pragma unroll 1
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int i = 0; i < PROBE64_ILP; ++i) r[i] = FMA ? __fma_rn(r[i], a, b) : __dadd_rn(r[i], b);
    }
    double acc = 0;
#pragma unroll
    for (int i = 0; i < PROBE64_ILP; ++i) acc = __dadd_rn(acc, r[i]);
    out[(size_t)blockIdx.x * blockDim.x + threadIdx.x] = acc;
}

// K6b: the same for SMALL batches (N = 1 drop-in, a few thousand cars): one WARP per car, the lanes split the centre line
// (lane l takes waypoints l, l + 32, ...: ascending, so a lane keeps the first index of its own minimum) and a warp-shuffle
// reduction on the pair (distance, index) — smaller distance, then smaller index — yields the reference's first-index argmin.
// A thread per car would leave the GPU empty at these sizes.
//
// K6b and K6c serve one centre line (MULTI = false: trs_locate, the track's LocTrack `one` in the constant bank, no track index) and several
// (MULTI = true: trs_locate_tracks, car i on track trk[i] with the descriptors `desc` and the scan table `scan` of loc_grid.h's loct_build).
enum { LOCW_THREADS = 256 };

// list == nullptr: cars 0 .. n (with MULTI an out-of-range track index gets -1 / NaN); otherwise the cars list[0 .. *count) that k_locate_grid
// put off (all in range).
template <bool MULTI>
__global__ void __launch_bounds__(LOCW_THREADS) k_locate_warp(const __grid_constant__ LocTrack one, const LocTrack* __restrict__ desc, int k,
                                                              const double* __restrict__ scan, const double* __restrict__ xyz,
                                                              const int32_t* __restrict__ trk, int n, int32_t* __restrict__ idx_out,
                                                              double* __restrict__ seg_out, const int* __restrict__ list = nullptr,
                                                              const int* __restrict__ count = nullptr)
{
    const int lane = threadIdx.x & 31;
    const int warps_per_grid = (gridDim.x * blockDim.x) >> 5;
    if (list) n = *count;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n; w += warps_per_grid) {
        const int car = list ? list[w] : w;
        const int t = MULTI ? trk[car] : 0;
        if (MULTI && (uint32_t)t >= (uint32_t)k) {
            if (lane == 0) {
                if (idx_out) idx_out[car] = -1;
                if (seg_out) seg_out[car] = loct_nan();
            }
            continue;
        }
        const LocTrack& d = MULTI ? desc[t] : one;
        const int n_u = d.n_u;
        const double4* wp = reinterpret_cast<const double4*>(scan) + (MULTI ? d.scan_off : 0);     // (one track: scan_off is 0)
        const double px = xyz[3 * (size_t)car], py = xyz[3 * (size_t)car + 1], pz = xyz[3 * (size_t)car + 2];
        double best = 100.0;                                     // track_data_process.py:93: the running minimum starts at 100
        int sel = 0x7fffffff;                                    // "nothing closer than 100 yet"
        for (int i = lane; i < n_u; i += 32) {
            const double2 qa = __ldg(reinterpret_cast<const double2*>(wp + i)), qb = __ldg(reinterpret_cast<const double2*>(wp + i) + 1);
            const double dd = __dadd_rn(__dadd_rn(fabs(__dsub_rn(px, qa.x)), fabs(__dsub_rn(py, qa.y))), fabs(__dsub_rn(pz, qb.x)));
            if (dd < best) { best = dd; sel = (int)qb.y; }       // original indices ascend with i: a lane keeps the first index of its own minimum
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int os = __shfl_xor_sync(0xffffffffu, sel, o);
            if (ob < best || (ob == best && os < sel)) { best = ob; sel = os; }
        }
        if (lane == 0) {
            const int idx = sel == 0x7fffffff ? 0 : sel;        // nothing closer than 100: index 0 (:91-92)
            if (idx_out) idx_out[car] = idx;
            if (seg_out) seg_out[car] = loct_segment(idx, d.n_wp, d.min_map, d.max_map);
        }
    }
}

// K6c: the same argmin through a uniform grid over (x, z): LARGE batches.  The algorithm and why it returns the reference's index bit for bit are in
// loc_grid.h (host / device functions, also compiled by the CPU-side tests): ~40 distance evaluations per car instead of ~1,000.  A car that has not
// settled after the 3 x 3 block and LOCG_MAX_RINGS rings (far from the line but inside its bounding box) is appended to a list for k_locate_warp,
// so one such car never holds its warp for a scan of the whole grid.  Persistent CTAs; each stages the track's table (quads in cell order + cell
// starts) in dynamic shared memory, sized for the largest table of the set.
// One track: the cars 0 .. n by grid stride (contiguous slices per CTA measured 1-2 % slower on the shipped lines: neighbouring cars cost
// alike, so one CTA can draw the expensive part of the line), the table is staged once and the LocTrack is read from the constant bank.  No
// minimum-CTA bound (0): its 40 registers give 6 CTAs per SM anyway, and a bound of 6 makes ptxas move the cell-start base and the grid width
// out of uniform registers, which measured 1 % slower on mountain_track.
// Several tracks: CTA b takes positions loct_slice(start[k], b, gridDim.x) of the bucketed cars perm (k_loct_scatter, loc_tracks.cuh), splits its
// slice at track boundaries and restages a track's table when the slice moves on to it; cars of a track without a grid go to the list whole.
// The track's LocTrack lives in shared memory and ptxas keeps its fields in registers: bounded at 3 CTAs per SM it takes 74 registers without
// spilling (by default it stops at 64 and spills).
// ------------------------------------------------------------------------------------------------------
enum { LOCG_THREADS = 256 };

template <bool MULTI>
__global__ void __launch_bounds__(LOCG_THREADS, MULTI ? 3 : 0) k_locate_grid(const __grid_constant__ LocTrack one, const LocTrack* __restrict__ desc,
                                                                          int k, const double* __restrict__ grid, const int* __restrict__ cells,
                                                                          const int* __restrict__ start, const int* __restrict__ perm, int n,
                                                                          const double* __restrict__ xyz, int32_t* __restrict__ idx_out,
                                                                          double* __restrict__ seg_out, int* __restrict__ defer_list,
                                                                          int* __restrict__ defer_count)
{
    extern __shared__ __align__(16) uint8_t locg_smem[];
    __shared__ LocTrack s_d;
    double* s_q = reinterpret_cast<double*>(locg_smem);
    const int* s_cs = nullptr;
    int lo, hi;
    if (MULTI) loct_slice(start[k], blockIdx.x, gridDim.x, lo, hi);
    else { lo = blockIdx.x * LOCG_THREADS; hi = n; }
    const int stride = MULTI ? LOCG_THREADS : gridDim.x * LOCG_THREADS;
    int staged = -1;
    while (lo < hi) {
        const int t = MULTI ? loct_track_of(start, k, lo) : 0;
        const int end = MULTI ? min(hi, start[t + 1]) : hi;
        const LocTrack& d = MULTI ? desc[t] : one;
        if (MULTI && d.grid_off < 0) {                           // no grid for this track: every car to the scan
            for (int p = lo + threadIdx.x; p < end; p += LOCG_THREADS) defer_list[atomicAdd(defer_count, 1)] = perm[p];
            lo = end;
            continue;
        }
        if (t != staged) {
            if (MULTI) __syncthreads();                          // every thread is done with the previous table (one track: there is none)
            const int nu = d.g.n_u, ncell = d.g.nx * d.g.nz;
            const double4* src = reinterpret_cast<const double4*>(grid) + (MULTI ? d.grid_off : 0);      // (one track: the offsets are 0)
            for (int i = threadIdx.x; i < nu; i += LOCG_THREADS) reinterpret_cast<double4*>(s_q)[i] = src[i];
            int* cs = reinterpret_cast<int*>(locg_smem + sizeof(double) * 4 * (size_t)nu);
            for (int i = threadIdx.x; i <= ncell; i += LOCG_THREADS) cs[i] = cells[(MULTI ? d.cell_off : 0) + i];
            if (MULTI && threadIdx.x == 0) s_d = d;
            s_cs = cs;
            staged = t;
            __syncthreads();
        }
        const LocTrack& e = MULTI ? s_d : one;
        for (int p = lo + threadIdx.x; p < end; p += stride) {
            const int car = MULTI ? perm[p] : p;
            const int idx = locg_walk(e.g, s_q, s_cs, xyz[3 * (size_t)car], xyz[3 * (size_t)car + 1], xyz[3 * (size_t)car + 2]);
            if (idx == LOCG_DEFERRED) {
                defer_list[atomicAdd(defer_count, 1)] = car;
                continue;
            }
            if (idx_out) idx_out[car] = idx;
            if (seg_out) seg_out[car] = loct_segment(idx, e.n_wp, e.min_map, e.max_map);
        }
        lo = end;
    }
}

// ------------------------------------------------------------------------------------------------------
// K7: speed-control tail of the pilots (keras_pilot.py:80-95 == 99-118, 142-153; utils/mapping.py:23-35).
// Types follow numpy >= 2 promotion with np.float32 model outputs by default: the products and the speed difference are
// float32, atan and everything after it float64.  legacy_f64 selects NumPy 1.x promotion instead (np.float32 * 20 is already
// float64 there), which moves results only at the dead-band cut-offs (-0.2, 0, 0.4) and at the `predicted - real > 0` test.
// ------------------------------------------------------------------------------------------------------
struct SpdKParams {
    double threshold, reverse_multiplier, break_multiplier, smooth_threshold;
    int use_break, smooth_steering;
    int legacy_f64;               // NumPy 1.x scalar promotion: the model's float32 speed is widened before the first multiply
};

__global__ void __launch_bounds__(256) k_speed_control(const double* __restrict__ cur, const float* __restrict__ model_spd,
                                                      const float* __restrict__ model_steer, int n, const SpdKParams p,
                                                      double* __restrict__ steer_out, double* __restrict__ thr_out,
                                                      double* __restrict__ brk_out, float* __restrict__ feat_out)
{
    const double half_pi = 3.141592653589793 / 2.0;
    const int stride = gridDim.x * blockDim.x;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const double real_spd = cur[k];
        const float steer_f = model_steer[k];
        double steering = (double)steer_f;
        if (steer_f < -1.0f) steering = -1.0; else if (steer_f > 1.0f) steering = 1.0;
        double delta, delta2;          // predicted * threshold - current, and twice that, in the promotion the caller asked for
        bool faster;                    // predicted - current > 0
        if (p.legacy_f64) {
            const double predicted = __dmul_rn((double)model_spd[k], 20.0);
            delta = __dsub_rn(__dmul_rn(predicted, p.threshold), real_spd);
            delta2 = __dmul_rn(delta, 2.0);
            faster = __dsub_rn(predicted, real_spd) > 0.0;
        } else {
            const float predicted = __fmul_rn(model_spd[k], 20.0f);
            const float target = __fmul_rn(predicted, (float)p.threshold);
            const float real_f = (float)real_spd;
            const float delta_f = __fsub_rn(target, real_f);
            delta = (double)delta_f;
            delta2 = (double)__fmul_rn(delta_f, 2.0f);
            faster = __fsub_rn(predicted, real_f) > 0.0f;
        }
        double throttle = __ddiv_rn(__dmul_rn(p.reverse_multiplier, atan(delta2)), half_pi);
        if (-0.2 < throttle && throttle < 0.0) throttle = 0.0;
        double breaking = 0.0;
        if (p.use_break) {
            throttle = faster ? 1.0 : 0.0;
            breaking = __ddiv_rn(__dmul_rn(__dmul_rn(-1.0, p.break_multiplier), atan(delta)), half_pi);
            if (breaking < 0.4) breaking = 0.0;
        }
        if (p.smooth_steering) {
            if (steering > p.smooth_threshold) steering = 1.0;
            else if (steering < p.smooth_threshold * -1.0) steering = -1.0;
        }
        steer_out[k] = steering; thr_out[k] = throttle; brk_out[k] = breaking;
        if (feat_out) feat_out[k] = (float)__ddiv_rn(real_spd, 20.0);
    }
}

// ------------------------------------------------------------------------------------------------------
// K9: per-car control post-processing, the step after the speed controller (SURVEY.md 8(f) rank 3):
//   ControlMultiplexer.step      components/controlmultiplexer.py:24-43 (launch locks: 48-70)
//   DriverAssistance.step        components/driver_assistance.py:13-31 (fused when a speed vector is given)
// Launch locks: the reference sets a flag at every AI launch and clears it from a thread that sleeps `duration` seconds,
// so a re-launch is cut short by an older thread that is still sleeping.  State per car: the last CTL_LAUNCH_SLOTS
// launch times; the flag is set at the latest launch L and cleared at the earliest t_i + duration that lies after L.
// ------------------------------------------------------------------------------------------------------
enum { CTL_LAUNCH_SLOTS = 4, CTL_MODE_HUMAN = 0, CTL_MODE_AI_STEERING = 1, CTL_MODE_AI = 2 };
#define CTL_NEVER (-1.0e300)

struct CtlKParams {
    int thr_en, st_en, assist_mode;        // assist_mode: 0 off, 1 'steering', 2 'speed'
    double thr_val, thr_dur, st_val, st_dur, assist_k;
};

__device__ __forceinline__ bool ctl_lock_active(const double (&t)[CTL_LAUNCH_SLOTS], double now, double duration)
{
    double latest = t[0];
#pragma unroll
    for (int i = 1; i < CTL_LAUNCH_SLOTS; ++i) latest = fmax(latest, t[i]);
    double first_end = __longlong_as_double(0x7ff0000000000000LL);
#pragma unroll
    for (int i = 0; i < CTL_LAUNCH_SLOTS; ++i) {
        const double end = __dadd_rn(t[i], duration);
        if (t[i] > CTL_NEVER && end > latest) first_end = fmin(first_end, end);
    }
    return latest > CTL_NEVER && now < first_end;
}

__global__ void __launch_bounds__(256) k_control_mux(const int* __restrict__ mode, const double* __restrict__ usr, const double* __restrict__ ai,
                                                    const double* __restrict__ speed, int n, const CtlKParams p, double now,
                                                    int* __restrict__ last_mode, double* __restrict__ launch, double* __restrict__ out)
{
    const int stride = gridDim.x * blockDim.x;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        const int m = mode[k];
        const bool full = m == CTL_MODE_AI;
        double steering = m == CTL_MODE_HUMAN ? usr[k] : ai[k];                           // :26-31
        double throttle = full ? ai[n + k] : usr[n + k];
        double breaking = full ? ai[2 * (size_t)n + k] : usr[2 * (size_t)n + k];
        double t[CTL_LAUNCH_SLOTS];
#pragma unroll
        for (int i = 0; i < CTL_LAUNCH_SLOTS; ++i) t[i] = launch[(size_t)i * n + k];
        if (last_mode[k] != CTL_MODE_AI && full) {                                        // :33-35: the oldest remembered launch drops out
            int oldest = 0;
#pragma unroll
            for (int i = 1; i < CTL_LAUNCH_SLOTS; ++i)
                if (t[i] < t[oldest]) oldest = i;
#pragma unroll
            for (int i = 0; i < CTL_LAUNCH_SLOTS; ++i)
                if (i == oldest) { t[i] = now; launch[(size_t)i * n + k] = now; }
        }
        if (p.st_en && ctl_lock_active(t, now, p.st_dur)) steering = p.st_val;            // :37-38
        if (p.thr_en && ctl_lock_active(t, now, p.thr_dur)) throttle = p.thr_val;         // :39-40
        last_mode[k] = m;                                                                 // :42
        if (speed && p.assist_mode) {                                                     // driver_assistance.py:15-29
            const double sp = speed[k];
            if (p.assist_mode == 1 && sp != 0.0) {
                const double mx = __ddiv_rn(p.assist_k, sp);
                if (steering > mx) { steering = mx; throttle = -0.1; }
                else if (steering < __dmul_rn(mx, -1.0)) { steering = __dmul_rn(mx, -1.0); throttle = -0.1; }
            } else if (p.assist_mode == 2 && steering != 0.0) {
                const double mx = __ddiv_rn(p.assist_k, steering);
                if (sp > mx) { throttle = 0.0; breaking = 0.0; }
            }
        }
        out[k] = steering; out[n + k] = throttle; out[2 * (size_t)n + k] = breaking;
    }
}

// three_segment_map (utils/mapping.py:9-16; cap: 18-21): the [-1, 1] command to a PWM value around a neutral point
__global__ void __launch_bounds__(256) k_pwm_map(const double* __restrict__ val, int n, double min_map, double mid_map, double max_map,
                                                double* __restrict__ out)
{
    const int stride = gridDim.x * blockDim.x;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += stride) {
        double v = val[k];
        v = v < -1.0 ? -1.0 : (v > 1.0 ? 1.0 : v);
        double r = mid_map;
        if (v < 0.0) r = __dadd_rn(mid_map, __dmul_rn(__dsub_rn(mid_map, min_map), v));
        else if (v > 0.0) r = __dadd_rn(mid_map, __dmul_rn(__dsub_rn(max_map, mid_map), v));
        out[k] = r;
    }
}

}  // namespace trs
