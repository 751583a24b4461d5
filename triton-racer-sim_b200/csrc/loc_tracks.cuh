// loc_tracks.cuh — nearest waypoint for cars on several centre lines in one batch (sm_100a).  Car i names its track t_i; its (idx, segment) is
// what trs_locate returns for it with that track alone: the reference's L1 float64 first-index argmin (track_data_process.py:89-107).  A car
// whose index is outside [0, K) gets idx -1 and segment NaN.
//
// Large batches (trs_locate_tracks, from sm_count x 256 cars):
//   k_loct_hist      per-block histogram of the cars' buckets (track, or K for an out-of-range index, whose outputs it writes)
//   k_loct_scan      one block: exclusive scan of the (bucket-major, block-minor) counts -> every block's first slot in every bucket, and the
//                    bucket starts
//   k_loct_scatter   stable scatter of the car indices into bucket order (a permutation; cars of a track stay in their original order)
//   k_locate_tracks_grid  persistent CTAs, each on a contiguous slice of the bucketed cars: the grid walk of loc_grid.h, restaging the track's
//                    table in shared memory whenever the slice moves on to another track; cars the walk puts off, and cars of tracks without a
//                    grid, go on a list for
//   k_locate_tracks_warp  warp per car over the car's own track (also the whole of a small batch, straight from the cars' order).
// TRS_LOCATE=thread replaces the walk with k_locate_tracks_scan, a thread per bucketed car scanning its track.
#pragma once
#include "loc_grid.h"
#include <cuda_runtime.h>
#include <stdint.h>

namespace trs {

enum { LOCT_THREADS = 256, LOCT_SCAN_THREADS = 1024 };

__device__ __forceinline__ double loct_nan() { return __longlong_as_double(0x7ff8000000000000LL); }

// the reference's __map (track_data_process.py:105-107): idx / N * (max - min) + min, one rounding per operation
__device__ __forceinline__ double loct_segment(int idx, int n_wp, double min_map, double max_map)
{
    return __dadd_rn(__dmul_rn(__ddiv_rn((double)idx, (double)n_wp), __dsub_rn(max_map, min_map)), min_map);
}

// Block b counts the buckets of cars [b chunk, (b + 1) chunk) into counts[bucket * nblk + b], and writes the outputs of out-of-range cars.
__global__ void __launch_bounds__(LOCT_THREADS) k_loct_hist(const int32_t* __restrict__ trk, int n, int k, int chunk, int nblk, int* __restrict__ counts,
                                                           int32_t* __restrict__ idx_out, double* __restrict__ seg_out)
{
    extern __shared__ int s_cnt[];                                   // k + 1 buckets
    for (int i = threadIdx.x; i <= k; i += LOCT_THREADS) s_cnt[i] = 0;
    __syncthreads();
    const int lo = blockIdx.x * chunk, hi = min(n, lo + chunk);
    const int lane = threadIdx.x & 31;
    for (int base = lo; base < hi; base += LOCT_THREADS) {
        const int i = base + threadIdx.x;
        const int b = i < hi ? loct_bucket(trk[i], k) : k + 1;
        if (b == k) {
            if (idx_out) idx_out[i] = -1;
            if (seg_out) seg_out[i] = loct_nan();
        }
        const unsigned same = __match_any_sync(0xffffffffu, b);      // one shared atomic per bucket and warp (all cars on one track is common)
        if (b <= k && lane == __ffs(same) - 1) atomicAdd(&s_cnt[b], __popc(same));
    }
    __syncthreads();
    for (int i = threadIdx.x; i <= k; i += LOCT_THREADS) counts[(size_t)i * nblk + blockIdx.x] = s_cnt[i];
}

// One block: counts[0 .. (k + 1) nblk) -> its exclusive prefix sum in place; start[b] = first bucketed position of bucket b (start[k] = the
// in-range cars), start[k + 1] = n.  Also clears the list counter of the walk.
__global__ void __launch_bounds__(LOCT_SCAN_THREADS) k_loct_scan(int* __restrict__ counts, int nblk, int k, int n, int* __restrict__ start,
                                                                int* __restrict__ defer_count)
{
    __shared__ int s_warp[LOCT_SCAN_THREADS / 32];
    const int entries = (k + 1) * nblk;
    const int per = (entries + LOCT_SCAN_THREADS - 1) / LOCT_SCAN_THREADS;
    const int a = min(entries, threadIdx.x * per), b = min(entries, a + per);
    int sum = 0;
    for (int i = a; i < b; ++i) sum += counts[i];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        int w = s_warp[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += v;
        }
        s_warp[lane] = w;                                            // inclusive over warps
    }
    __syncthreads();
    int run = incl - sum + (warp ? s_warp[warp - 1] : 0);
    for (int i = a; i < b; ++i) {
        const int v = counts[i];
        counts[i] = run;
        run += v;
    }
    __syncthreads();                                                 // (global writes of the block are visible to the block after the barrier)
    for (int t = threadIdx.x; t <= k; t += LOCT_SCAN_THREADS) start[t] = counts[(size_t)t * nblk];
    if (threadIdx.x == 0) { start[k + 1] = n; *defer_count = 0; }
}

// Block b writes the indices of its cars to perm[offs[bucket * nblk + b] ...], in order within every bucket: rounds of LOCT_THREADS cars; in a
// round a car's slot is the bucket's running base + the same bucket's cars in the warps before its own + its rank inside its warp.
__global__ void __launch_bounds__(LOCT_THREADS) k_loct_scatter(const int32_t* __restrict__ trk, int n, int k, int chunk, int nblk,
                                                              const int* __restrict__ offs, int* __restrict__ perm)
{
    enum { WARPS = LOCT_THREADS / 32 };
    extern __shared__ int s_sc[];
    int* s_base = s_sc;                                              // k + 1: next slot of every bucket
    int* s_wcnt = s_sc + (k + 1);                                    // WARPS x (k + 1): cars of every bucket in every warp of this round
    for (int i = threadIdx.x; i <= k; i += LOCT_THREADS) s_base[i] = offs[(size_t)i * nblk + blockIdx.x];
    for (int i = threadIdx.x; i < WARPS * (k + 1); i += LOCT_THREADS) s_wcnt[i] = 0;
    __syncthreads();
    const int lo = blockIdx.x * chunk, hi = min(n, lo + chunk);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = lo; base < hi; base += LOCT_THREADS) {
        const int i = base + threadIdx.x;
        const int b = i < hi ? loct_bucket(trk[i], k) : k + 1;
        const unsigned same = __match_any_sync(0xffffffffu, b);
        const bool leader = lane == __ffs(same) - 1, valid = b <= k;
        if (valid && leader) s_wcnt[warp * (k + 1) + b] = __popc(same);
        __syncthreads();
        if (valid) {
            int pos = s_base[b] + __popc(same & ((1u << lane) - 1));
            for (int w = 0; w < warp; ++w) pos += s_wcnt[w * (k + 1) + b];
            perm[pos] = i;
        }
        __syncthreads();
        if (valid && leader) { atomicAdd(&s_base[b], __popc(same)); s_wcnt[warp * (k + 1) + b] = 0; }
        __syncthreads();
    }
}

// The walk.  CTA b takes bucketed positions loct_slice(start[k], b, gridDim.x) and splits them at track boundaries; dynamic shared memory: the
// largest grid table of the tracks (trs_set_tracks sets the attribute).  The track's LocGrid lives in shared memory, not in the constant bank as
// k_locate_grid's does, and ptxas keeps its fields in registers: bounded at 3 CTAs per SM it takes 74 registers without spilling (by default it
// stops at 64 and spills).
__global__ void __launch_bounds__(LOCG_THREADS, 3) k_locate_tracks_grid(const LocTrack* __restrict__ desc, int k, const double* __restrict__ grid,
                                                                    const int* __restrict__ cells, const int* __restrict__ start,
                                                                    const int* __restrict__ perm, const double* __restrict__ xyz,
                                                                    int32_t* __restrict__ idx_out, double* __restrict__ seg_out,
                                                                    int* __restrict__ defer_list, int* __restrict__ defer_count)
{
    extern __shared__ __align__(16) uint8_t loct_smem[];
    __shared__ LocTrack s_d;
    double* s_q = reinterpret_cast<double*>(loct_smem);
    const int* s_cs = nullptr;
    int lo, hi;
    loct_slice(start[k], blockIdx.x, gridDim.x, lo, hi);
    int staged = -1;
    while (lo < hi) {
        const int t = loct_track_of(start, k, lo);
        const int end = min(hi, start[t + 1]);
        if (desc[t].grid_off < 0) {                                  // no grid for this track: every car to the scan
            for (int p = lo + threadIdx.x; p < end; p += LOCG_THREADS) defer_list[atomicAdd(defer_count, 1)] = perm[p];
            lo = end;
            continue;
        }
        if (t != staged) {
            __syncthreads();                                         // every thread is done with the previous table
            const LocTrack& d = desc[t];
            const int nu = d.g.n_u, ncell = d.g.nx * d.g.nz;
            const double4* src = reinterpret_cast<const double4*>(grid) + d.grid_off;
            for (int i = threadIdx.x; i < nu; i += LOCG_THREADS) reinterpret_cast<double4*>(s_q)[i] = src[i];
            int* cs = reinterpret_cast<int*>(loct_smem + sizeof(double) * 4 * (size_t)nu);
            for (int i = threadIdx.x; i <= ncell; i += LOCG_THREADS) cs[i] = cells[d.cell_off + i];
            if (threadIdx.x == 0) s_d = d;
            s_cs = cs;
            staged = t;
            __syncthreads();
        }
        for (int p = lo + threadIdx.x; p < end; p += LOCG_THREADS) {
            const int car = perm[p];
            const int idx = locg_walk(s_d.g, s_q, s_cs, xyz[3 * (size_t)car], xyz[3 * (size_t)car + 1], xyz[3 * (size_t)car + 2]);
            if (idx == LOCG_DEFERRED) {
                defer_list[atomicAdd(defer_count, 1)] = car;
                continue;
            }
            if (idx_out) idx_out[car] = idx;
            if (seg_out) seg_out[car] = loct_segment(idx, s_d.n_wp, s_d.min_map, s_d.max_map);
        }
        lo = end;
    }
}

// Warp per car over its track's distinct points (k_locate_warp with the table chosen per car).  list == nullptr: cars 0 .. n, an out-of-range
// index gets -1 / NaN; otherwise the cars list[0 .. *count) (all in range).
__global__ void __launch_bounds__(LOCW_THREADS) k_locate_tracks_warp(const LocTrack* __restrict__ desc, int k, const double* __restrict__ scan,
                                                                    const double* __restrict__ xyz, const int32_t* __restrict__ trk, int n,
                                                                    int32_t* __restrict__ idx_out, double* __restrict__ seg_out,
                                                                    const int* __restrict__ list = nullptr, const int* __restrict__ count = nullptr)
{
    const int lane = threadIdx.x & 31;
    const int warps_per_grid = (gridDim.x * blockDim.x) >> 5;
    if (list) n = *count;
    for (int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; w < n; w += warps_per_grid) {
        const int car = list ? list[w] : w;
        const int t = trk[car];
        if ((uint32_t)t >= (uint32_t)k) {
            if (lane == 0) {
                if (idx_out) idx_out[car] = -1;
                if (seg_out) seg_out[car] = loct_nan();
            }
            continue;
        }
        const int n_u = desc[t].n_u;
        const double4* wp = reinterpret_cast<const double4*>(scan) + desc[t].scan_off;
        const double px = xyz[3 * (size_t)car], py = xyz[3 * (size_t)car + 1], pz = xyz[3 * (size_t)car + 2];
        double best = 100.0;                                         // track_data_process.py:93
        int sel = 0x7fffffff;
        for (int i = lane; i < n_u; i += 32) {
            const double2 qa = __ldg(reinterpret_cast<const double2*>(wp + i)), qb = __ldg(reinterpret_cast<const double2*>(wp + i) + 1);
            const double d = __dadd_rn(__dadd_rn(fabs(__dsub_rn(px, qa.x)), fabs(__dsub_rn(py, qa.y))), fabs(__dsub_rn(pz, qb.x)));
            if (d < best) { best = d; sel = (int)qb.y; }
        }
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            const double ob = __shfl_xor_sync(0xffffffffu, best, o);
            const int os = __shfl_xor_sync(0xffffffffu, sel, o);
            if (ob < best || (ob == best && os < sel)) { best = ob; sel = os; }
        }
        if (lane == 0) {
            const int idx = sel == 0x7fffffff ? 0 : sel;
            if (idx_out) idx_out[car] = idx;
            if (seg_out) seg_out[car] = loct_segment(idx, desc[t].n_wp, desc[t].min_map, desc[t].max_map);
        }
    }
}

// TRS_LOCATE=thread: a thread per bucketed car scans its track's distinct points in order of first occurrence (strict `<`, as k_locate).
__global__ void __launch_bounds__(LOCT_THREADS) k_locate_tracks_scan(const LocTrack* __restrict__ desc, int k, const double* __restrict__ scan,
                                                                    const int* __restrict__ start, const int* __restrict__ perm,
                                                                    const double* __restrict__ xyz, const int32_t* __restrict__ trk,
                                                                    int32_t* __restrict__ idx_out, double* __restrict__ seg_out)
{
    const int nv = start[k];
    for (int p = blockIdx.x * LOCT_THREADS + threadIdx.x; p < nv; p += gridDim.x * LOCT_THREADS) {
        const int car = perm[p];
        const int t = trk[car];
        const int n_u = desc[t].n_u;
        const double4* wp = reinterpret_cast<const double4*>(scan) + desc[t].scan_off;
        const double px = xyz[3 * (size_t)car], py = xyz[3 * (size_t)car + 1], pz = xyz[3 * (size_t)car + 2];
        double best = 100.0;
        int sel = 0;
        for (int i = 0; i < n_u; ++i) {
            const double2 qa = __ldg(reinterpret_cast<const double2*>(wp + i)), qb = __ldg(reinterpret_cast<const double2*>(wp + i) + 1);
            const double d = __dadd_rn(__dadd_rn(fabs(__dsub_rn(px, qa.x)), fabs(__dsub_rn(py, qa.y))), fabs(__dsub_rn(pz, qb.x)));
            if (d < best) { best = d; sel = (int)qb.y; }
        }
        if (idx_out) idx_out[car] = sel;
        if (seg_out) seg_out[car] = loct_segment(sel, desc[t].n_wp, desc[t].min_map, desc[t].max_map);
    }
}

}  // namespace trs
