// trs_api.cu — the C ABI declared in include/trs_b200.h, over the sm_100a kernels.
//
// Host-side mirror of what the reference's Python does around its library calls: parameter validation and
// derivation (threshold swap/floor, bound rounding, merge order), launch geometry, and the host-buffer pipeline.
// No CPU implementation of any stage lives here: if there is no sm_100 device the calls fail.
#include <cuda_runtime.h>
#include <math.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <atomic>
#include <mutex>
#include <new>
#include <thread>
#include <vector>

#include "../../include/trs_b200.h"
#include "jpeg_host.h"
#include "jpeg_kernels.cuh"
#include "jpeg_enc_kernels.cuh"
#include "misc_kernels.cuh"
#include "preproc_kernel.cuh"
#include "preproc_fast.cuh"
#include "preproc_bsw.cuh"
#include "trs_internal.h"

namespace {

thread_local char g_err[512] = "";
std::atomic<unsigned long long> g_launches{0};

int fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

int cuda_fail(cudaError_t e, const char* what)
{
    snprintf(g_err, sizeof g_err, "%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return (int)e > 0 ? (int)e : 1;
}

#define CU(call)                                              \
    do {                                                      \
        cudaError_t _e = (call);                              \
        if (_e != cudaSuccess) return cuda_fail(_e, #call);   \
    } while (0)

// cvRound semantics of OpenCV's scalar -> int32 conversion (half-to-even; out of range -> INT_MIN)
int32_t round_bound(double v)
{
    if (!(v > -2147483648.5 && v < 2147483647.5)) return INT32_MIN;
    return (int32_t)nearbyint(v);
}

enum { HOST_STREAMS = 3 };

}  // namespace

// Test-only switches (tests/test_gpu_parity.py forces every kernel variant through the same goldens): read from the environment ONCE,
// when the context is created, so no call on the N = 1 latency path pays a getenv.
struct TrsSwitches {
    bool force_generic = false, no_banded = false, no_store_warp = false, resize_scalar = false, resize_gather = false;
    int locate = 0;                    // 0 = by batch size, 1 = warp per car, 2 = thread per car, 3 = grid
    size_t host_chunk_bytes = (size_t)48 << 20;      // ~48 MB of frames per chunk of the host pipeline (the link saturates from ~16 MB up)
};

struct trs_ctx {
    int device = 0;
    TrsSwitches sw;
    int sm_count = 0;
    int smem_optin = 0;
    int cc_major = 0, cc_minor = 0;
    std::mutex mu;
    // preprocessing
    bool have_params = false;
    trs_preproc_params user{};
    trs::PreKParams kp{};              // derived, geometry fields filled per call
    // track
    double* wp_dev = nullptr;          // distinct waypoints in order of first occurrence: (x, y, z, original index) quads
    int n_wp = 0, n_wp_distinct = 0;
    double* wp_grid_dev = nullptr;     // the same quads sorted by grid cell (k_locate_grid), nullptr: no grid for this centre line
    int* wp_cells_dev = nullptr;       // start of every cell in wp_grid_dev, ncell + 1 entries
    trs::LocGrid grid{};
    int* defer_dev = nullptr;          // [0] = count, [1 ..] = cars k_locate_grid left to the warp-per-car kernel
    size_t defer_cap = 0;              // cars the list can hold
    double min_map = 0, max_map = 10;
    // host pipeline
    cudaStream_t hs[HOST_STREAMS] = {nullptr, nullptr, nullptr};
    uint8_t* st_in[HOST_STREAMS] = {nullptr, nullptr, nullptr};
    uint8_t* st_u8[HOST_STREAMS] = {nullptr, nullptr, nullptr};
    float* st_f32[HOST_STREAMS] = {nullptr, nullptr, nullptr};
    size_t st_in_cap = 0, st_u8_cap = 0, st_f32_cap = 0;
    unsigned long long* stats_dev = nullptr;
    cudaEvent_t host_entry = nullptr;  // orders the internal streams after the caller's stream at entry of the *_host calls
    // tub ingestion staging (grown on demand)
    uint8_t* jpg_blob = nullptr;   size_t jpg_blob_cap = 0;
    uint8_t* jpg_planes = nullptr; size_t jpg_planes_cap = 0;
    void* jpg_meta = nullptr;      size_t jpg_meta_cap = 0;
    // tub recording (trs_jpeg_encode): tables + header of the last (h, w, quality), per-record sizes / offsets, the packed files
    uint8_t* jpe_meta = nullptr;   int jpe_meta_key[3] = {0, 0, 0};
    unsigned long long* jpe_sizes = nullptr; size_t jpe_sizes_cap = 0;         // records; the offsets buffer holds one more
    unsigned long long* jpe_offs = nullptr;
    uint8_t* jpe_blob = nullptr;   size_t jpe_blob_cap = 0;
    long long jpe_last_bytes = -1;                                             // bytes of the last encode, -1: none yet
    std::vector<unsigned long long> jpe_host_offs;
};

int trs_i_fail(int code, const char* fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
int trs_i_cuda_fail(cudaError_t e, const char* what) { return cuda_fail(e, what); }
void trs_i_count_launches(int k) { g_launches.fetch_add((unsigned long long)k, std::memory_order_relaxed); }
int trs_i_ctx_device(const trs_ctx* ctx) { return ctx->device; }
int trs_i_ctx_sm_count(const trs_ctx* ctx) { return ctx->sm_count; }

namespace {

void default_params(trs_preproc_params* p)
{
    memset(p, 0, sizeof *p);
    p->contrast_ratio = 1.0;
    p->contrast_offset = 125;
    p->brightness_baseline = 550;
    p->edge_dest = 2;
    p->canny_a = 60;
    p->canny_b = 100;
}

int derive_params(trs_ctx* ctx, const trs_preproc_params* u)
{
    trs::PreKParams k{};
    if (u->color_filter_enabled && (u->n_hsv < 0 || u->n_hsv > TRS_MAX_HSV))
        return fail(TRS_E_ARG, "n_hsv=%d outside [0,%d]", u->n_hsv, TRS_MAX_HSV);
    // brightness / contrast (img_preprocessing.py:81-102)
    k.dynamic = u->dynamic_brightness ? 1 : 0;
    k.foff = (float)u->contrast_offset;
    k.fratio = (float)u->contrast_ratio;
    k.baseline = u->brightness_baseline;
    k.lut_identity = 1;
    for (int i = 0; i < 256; ++i) {
        k.lut[i] = trs::adjust_entry(i, false, 0.0f, k.foff, k.fratio);
        if (k.lut[i] != i) k.lut_identity = 0;
    }
    // merge order (img_preprocessing.py:44-53,57-62): colour layers in list order, then the edge layer; later wins
    int src[3] = {trs::SRC_PIXEL, trs::SRC_PIXEL, trs::SRC_PIXEL};
    const int n_hsv = u->color_filter_enabled ? u->n_hsv : 0;
    for (int i = 0; i < n_hsv; ++i) {
        int ch = u->color_dest[i];
        if (ch < -3 || ch > 2) return fail(TRS_E_ARG, "colour destination channel %d out of range for an RGB frame", ch);
        if (ch < 0) ch += 3;                        // numpy negative index
        src[ch] = trs::SRC_MASK0 + i;
    }
    k.edge_enabled = u->edge_enabled ? 1 : 0;
    if (k.edge_enabled) {
        int ch = u->edge_dest;
        if (ch < -3 || ch > 2) return fail(TRS_E_ARG, "edge destination channel %d out of range for an RGB frame", ch);
        if (ch < 0) ch += 3;
        src[ch] = trs::SRC_EDGE;
    }
    // keep only colour ranges that still reach the output
    k.n_ranges = 0;
    for (int i = 0; i < n_hsv; ++i) {
        bool used = false;
        for (int c = 0; c < 3; ++c) used |= (src[c] == trs::SRC_MASK0 + i);
        if (!used) continue;
        const int slot = k.n_ranges++;
        for (int c = 0; c < 3; ++c) {
            k.ranges[slot].lo[c] = round_bound(u->hsv_lo[i][c]);
            k.ranges[slot].hi[c] = round_bound(u->hsv_hi[i][c]);
            if (src[c] == trs::SRC_MASK0 + i) src[c] = -(slot + 1);      // temporary marker
        }
        k.range_stat[slot] = i;
    }
    k.need_pixels = 0;
    for (int c = 0; c < 3; ++c) {
        if (src[c] < 0) src[c] = trs::SRC_MASK0 + (-src[c] - 1);
        k.src[c] = src[c];
        if (src[c] == trs::SRC_PIXEL) k.need_pixels = 1;
    }
    // cv2.Canny(img, a, b): swap if a > b, then floor (L1 norm)
    double a = u->canny_a, b = u->canny_b;
    if (a > b) { double t = a; a = b; b = t; }
    if (!(a > -2e9 && b < 2e9)) return fail(TRS_E_ARG, "edge thresholds out of range");
    k.low = (int)floor(a);
    k.high = (int)floor(b);
    ctx->kp = k;
    ctx->user = *u;
    ctx->have_params = true;
    return 0;
}

struct Geometry {
    int band_h, row_stride, mag_stride, wwords, smem, ctas_per_sm;
};

int plan_geometry(trs_ctx* ctx, int h, int w, int n_ranges, Geometry* g)
{
    g->wwords = (w + 31) / 32;
    g->row_stride = ((w * 3 + 15) & ~15) + 16;
    g->mag_stride = (w + 3) & ~1;
    const int budget2 = (ctx->smem_optin + 1024) / 2 - 1024;       // two CTAs per SM (1 KB per-CTA reserve)
    auto fits = [&](int band_h, int budget) {
        return trs::pre_smem_layout(h, w, band_h, g->row_stride, g->mag_stride, g->wwords, n_ranges).total <= budget;
    };
    auto largest = [&](int budget) {
        int lo = 0, hi = h;
        while (lo < hi) { int mid = (lo + hi + 1) / 2; if (fits(mid, budget)) lo = mid; else hi = mid - 1; }
        return lo;
    };
    int band = largest(budget2);
    if (band < (h < 16 ? h : 16)) band = largest(ctx->smem_optin);
    if (band < 1) return fail(TRS_E_RANGE, "frame %dx%d does not fit the on-chip working set (%d B shared memory)", h, w, ctx->smem_optin);
    const int nb = (h + band - 1) / band;
    g->band_h = (h + nb - 1) / nb;
    g->smem = trs::pre_smem_layout(h, w, g->band_h, g->row_stride, g->mag_stride, g->wwords, n_ranges).total;
    return 0;
}

// Frame-resident fast path (preproc_fast.cuh): whole frame + magnitude plane + bit planes in one CTA's shared memory,
// width a multiple of 32, everything 16-byte aligned.  Returns 1 if launched, 0 if not eligible, <0 / >1 on error.
template <int NR, bool EDGE, int F0, int F1>
int launch_fast_tf(const trs::FastParams& fp, int grid, cudaStream_t st)
{
    if (EDGE && fp.use_store_warp) {
        // the reference's camera size with its default colour ranges (core/config.py:8-9,23) gets the variant with compile-time dimensions
        if (NR == 2 && F0 >= 0 && trs::sw_static_geometry_ok<120, 160>(fp.g, fp.k.h, fp.k.w)) {
            auto kern = trs::k_preprocess_sw<NR, F0, F1, (NR == 2 && F0 >= 0 ? 120 : 0), (NR == 2 && F0 >= 0 ? 160 : 0)>;
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, fp.g.total);
            if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(sw 120x160)");
            kern<<<grid, trs::SW_THREADS, fp.g.total, st>>>(fp);
            return 0;
        }
        cudaError_t e = cudaFuncSetAttribute(trs::k_preprocess_sw<NR, F0, F1>, cudaFuncAttributeMaxDynamicSharedMemorySize, fp.g.total);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(sw)");
        trs::k_preprocess_sw<NR, F0, F1><<<grid, trs::SW_THREADS, fp.g.total, st>>>(fp);
        return 0;
    }
    if (fp.g.n_bands > 1) {
        cudaError_t e = cudaFuncSetAttribute(trs::k_preprocess_banded<NR, EDGE, F0, F1>, cudaFuncAttributeMaxDynamicSharedMemorySize, fp.g.total);
        if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(banded)");
        trs::k_preprocess_banded<NR, EDGE, F0, F1><<<grid, fp.g.threads, fp.g.total, st>>>(fp);
        return 0;
    }
    cudaError_t e = cudaFuncSetAttribute(trs::k_preprocess_fast<NR, EDGE, F0, F1>, cudaFuncAttributeMaxDynamicSharedMemorySize, fp.g.total);
    if (e != cudaSuccess) return cuda_fail(e, "cudaFuncSetAttribute(fast)");
    trs::k_preprocess_fast<NR, EDGE, F0, F1><<<grid, fp.g.threads, fp.g.total, st>>>(fp);
    return 0;
}

// The reference's default colour ranges (core/config.py:23: white = S <= 64 & V >= 130, yellow = 25 <= H <= 43 & S >= 180 & V >= 155)
// get a variant with the live-bound words baked in; every other configuration reads them at run time.
enum { DEFAULT_F0 = 8 | 16, DEFAULT_F1 = 1 | 2 | 4 | 16 };

template <int NR, bool EDGE>
int launch_fast_t(const trs::FastParams& fp, int grid, cudaStream_t st)
{
    // (the baked variant turns the hue bounds of range 1 into per-delta numerator thresholds and skips the blue-max hue formula, which
    // needs an upper bound below 60: preproc_fast.cuh HueThresholds / hsv_masks_of)
    if (NR == 2 && fp.fr[0].flags == DEFAULT_F0 && fp.fr[1].flags == DEFAULT_F1 && fp.k.ranges[1].hi[0] <= 59)
        return launch_fast_tf<NR, EDGE, (NR == 2 ? (int)DEFAULT_F0 : -1), (NR == 2 ? (int)DEFAULT_F1 : -1)>(fp, grid, st);
    return launch_fast_tf<NR, EDGE, -1, -1>(fp, grid, st);
}

// Banded store-warp kernel (preproc_bsw.cuh) for one compile-time geometry.  Returns 1 if launched, 0 if it does not fit, < 0 on error.
// LUT: a brightness / contrast table that is not the identity.
template <int H, int W, int R, int NSW, int MAXREG = trs::SW_MAXREG, bool LUT = false>
int launch_bsw(trs_ctx* ctx, const trs::FastParams& fp, int n, cudaStream_t st)
{
    using L = trs::BswLayout<H, W, R, 2, NSW>;
    auto kern = trs::k_preprocess_bsw<2, (int)DEFAULT_F0, (int)DEFAULT_F1, H, W, R, NSW, MAXREG, LUT>;
    if (L::TOTAL > (ctx->smem_optin + 1024) / 2 - 1024) return 0;
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, L::TOTAL);
    if (e != cudaSuccess) { cuda_fail(e, "cudaFuncSetAttribute(bsw)"); return -100 - (int)e; }
    int per_sm = 0;
    e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, L::THREADS, L::TOTAL);
    if (e != cudaSuccess) { cuda_fail(e, "occupancy(bsw)"); return -100 - (int)e; }
    if (per_sm < 1) return 0;
    int grid = ctx->sm_count * per_sm;
    if (grid > n) grid = n;
    kern<<<grid, L::THREADS, L::TOTAL, st>>>(fp);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    e = cudaGetLastError();
    if (e != cudaSuccess) { cuda_fail(e, "k_preprocess_bsw launch"); return -100 - (int)e; }
    return 1;
}

int try_launch_fast(trs_ctx* ctx, const trs::PreKParams& k, int n, int h, int w, cudaStream_t st)
{
    if (ctx->sw.force_generic) return 0;
    if (!k.edge_enabled && k.n_ranges == 0) {
        // no filter at all (the reference's defaults): the brightness / contrast table + /255 as a pure stream
        if (!k.word_io || ctx->sw.no_banded) return 0;
        int grid = ctx->sm_count * 8;
        if (grid > n) grid = n;
        trs::k_adjust_stream<<<grid, trs::ADJ_THREADS, 0, st>>>(k);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) { cuda_fail(e, "k_adjust_stream launch"); return -100 - (int)e; }
        return 1;
    }
    if (!k.word_io || (w % 32) != 0 || (((size_t)h * w * 3) % 16) != 0) return 0;
    const int nsg = w / 32;
    trs::FastParams fp;
    memset(&fp, 0, sizeof fp);
    fp.k = k;
    {
        // resident kernel: one frame per CTA, two CTAs per SM; frames that do not fit whole go band by band (k_preprocess_banded) when
        // nothing of the pixels is needed after the strip walk
        const int max_warps = trs::FAST_MAX_THREADS / 32;
        if (nsg > max_warps) return 0;
        const int quads = max_warps / nsg;
        const int budget2 = (ctx->smem_optin + 1024) / 2 - 1024;
        trs::FastGeom g = trs::fast_geometry(h, w, k.n_ranges, 0, nsg * quads, nsg * quads);
        if (g.threads > trs::FAST_MAX_THREADS) return 0;
        if (g.total > budget2) {
            if (ctx->sw.no_banded) return 0;
            bool found = false;
            for (int nb = 2; nb <= h / 4 && !found; ++nb) {
                const int bh = (h + nb - 1) / nb;
                g = trs::fast_geometry(h, w, k.n_ranges, 0, nsg * quads, nsg * quads, 1, bh);
                found = g.n_bands > 1 && g.total <= budget2;
            }
            if (!found) return 0;
        }
        fp.g = g;
    }
    // integer bounds -> fp16-subnormal bit patterns for the packed compares (values live in [0, 2047];
    // anything below 0 compares like -1, anything above like 2047, which keeps every outcome unchanged)
    auto pat = [](long long v) -> uint32_t {
        const uint32_t q = v < 0 ? 0x8001u : (v > 2047 ? 2047u : (uint32_t)v);
        return q | (q << 16);
    };
    fp.need_hue = 0;
    for (int r = 0; r < k.n_ranges && r < 3; ++r) {
        const int top[3] = {179, 255, 255};
        uint32_t flags = 0;
        for (int c = 0; c < 3; ++c) {
            fp.fr[r].lo[c] = pat(k.ranges[r].lo[c]);
            fp.fr[r].hi[c] = pat(k.ranges[r].hi[c]);
            if (k.ranges[r].lo[c] > 0) flags |= 1u << (2 * c);
            if (k.ranges[r].hi[c] < top[c]) flags |= 2u << (2 * c);
        }
        fp.fr[r].flags = flags;
        if (flags & 3u) fp.need_hue = 1;
    }
    // store-warp variant (k_preprocess_sw): edge filter on, every output channel a bit plane, ten compute warps, and the
    // double-buffered mask planes still fit two CTAs per SM
    fp.use_store_warp = 0;
    if (fp.g.n_bands == 1 && k.edge_enabled && !k.need_pixels && fp.g.threads == trs::SW_COMPUTE_THREADS && !ctx->sw.no_store_warp) {
        const trs::FastGeom g2 = trs::fast_geometry(h, w, k.n_ranges, 0, fp.g.front_warps, fp.g.back_warps, 2);
        const int budget2 = (ctx->smem_optin + 1024) / 2 - 1024;
        if (g2.total <= budget2) {
            fp.g = g2;
            fp.use_store_warp = 1;
        }
    }
    fp.low2 = pat(k.low);
    fp.high2 = pat(k.high);
    int grid = ctx->sm_count * 2;
    if (grid > n) grid = n;
    int rc;
    // 240x320 (BASELINE.json configs[2]) with the reference's default ranges: banded store-warp kernel with compile-time geometry
    // (any brightness / contrast setting: the table is applied as the strip walk loads its words.  Ranges whose live bounds are only known at
    // run time stay on k_preprocess_banded: measured at 240x320 with the reference-generated "exotic" configuration, 1.50 M frames/s there
    // against 1.36 M here - the run-time colour tests take twice the instructions and the table on top of them costs more per loaded word than
    // the banded kernel's in-place pass)
    const bool bsw_ok = k.n_ranges == 2 && k.edge_enabled && !k.need_pixels && !ctx->sw.no_store_warp &&
                        fp.fr[0].flags == DEFAULT_F0 && fp.fr[1].flags == DEFAULT_F1 && k.ranges[1].hi[0] <= 59;
    if (bsw_ok && h == 240 && w == 320) {
        rc = (k.dynamic || !k.lut_identity) ? launch_bsw<240, 320, 24, 2, trs::SW_MAXREG, true>(ctx, fp, n, st) : launch_bsw<240, 320, 24, 2>(ctx, fp, n, st);
        if (rc) return rc;
    }
    switch (k.n_ranges * 2 + (k.edge_enabled ? 1 : 0)) {
    case 1: rc = launch_fast_t<0, true>(fp, grid, st); break;
    case 2: rc = launch_fast_t<1, false>(fp, grid, st); break;
    case 3: rc = launch_fast_t<1, true>(fp, grid, st); break;
    case 4: rc = launch_fast_t<2, false>(fp, grid, st); break;
    case 5: rc = launch_fast_t<2, true>(fp, grid, st); break;
    case 6: rc = launch_fast_t<3, false>(fp, grid, st); break;
    default: return 0;
    }
    if (rc) return rc < 0 ? rc : -100 - rc;
    g_launches.fetch_add(1, std::memory_order_relaxed);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) { cuda_fail(e, "k_preprocess_fast launch"); return -100 - (int)e; }
    return 1;
}

int launch_preprocess(trs_ctx* ctx, const uint8_t* in, int n, int h, int w, uint8_t* out_u8, float* out_f32,
                      unsigned long long* stats, uint16_t* dbg_mag, uint8_t* dbg_map, bool force_edge, cudaStream_t st)
{
    trs::PreKParams k = ctx->kp;
    if (force_edge && !k.edge_enabled) { k.edge_enabled = 1; }
    if (!dbg_mag && !dbg_map) {
        trs::PreKParams kf = k;
        kf.in = in; kf.out_u8 = out_u8; kf.out_f32 = out_f32; kf.stats = stats; kf.dbg_mag = nullptr; kf.dbg_map = nullptr;
        kf.n = n; kf.h = h; kf.w = w;
        kf.word_io = ((w * 3) % 4 == 0) && (((uintptr_t)in & 15) == 0) && (!out_u8 || ((uintptr_t)out_u8 & 15) == 0) &&
                     (!out_f32 || ((uintptr_t)out_f32 & 15) == 0) && (((size_t)h * w * 3) % 4 == 0);
        const int fr = try_launch_fast(ctx, kf, n, h, w, st);
        if (fr == 1) return 0;
        if (fr < 0) return fr <= -100 ? -(fr + 100) : fr;
    }
    Geometry g;
    int rc = plan_geometry(ctx, h, w, k.n_ranges, &g);
    if (rc) return rc;
    k.in = in; k.out_u8 = out_u8; k.out_f32 = out_f32; k.stats = stats; k.dbg_mag = dbg_mag; k.dbg_map = dbg_map;
    k.n = n; k.h = h; k.w = w;
    k.band_h = g.band_h; k.row_stride = g.row_stride; k.mag_stride = g.mag_stride; k.wwords = g.wwords;
    const size_t frame_bytes = (size_t)h * w * 3;
    k.word_io = ((w * 3) % 4 == 0) && (((uintptr_t)in & 15) == 0) && (!out_u8 || ((uintptr_t)out_u8 & 15) == 0) &&
                (!out_f32 || ((uintptr_t)out_f32 & 15) == 0) && (frame_bytes % 4 == 0);
    CU(cudaFuncSetAttribute(trs::k_preprocess, cudaFuncAttributeMaxDynamicSharedMemorySize, g.smem));
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trs::k_preprocess, trs::PRE_THREADS, g.smem));
    if (per_sm < 1) return fail(TRS_E_RANGE, "kernel does not fit an SM with %d B shared memory", g.smem);
    int grid = ctx->sm_count * per_sm;
    if (grid > n) grid = n;
    trs::k_preprocess<<<grid, trs::PRE_THREADS, g.smem, st>>>(k);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    return 0;
}

// staging buffers of the host pipeline grow on demand; the capacity is only recorded once all buffers of a kind exist, so a failed
// allocation can never leave a stale capacity next to a null pointer
template <class T>
int grow_staging(T* (&bufs)[HOST_STREAMS], size_t& cap, size_t bytes)
{
    if (cap >= bytes) return 0;
    cap = 0;
    for (int i = 0; i < HOST_STREAMS; ++i) { cudaFree(bufs[i]); bufs[i] = nullptr; }
    for (int i = 0; i < HOST_STREAMS; ++i) CU(cudaMalloc(&bufs[i], bytes));
    cap = bytes;
    return 0;
}

// first statement of every entry point that touches the device
#define TRS_ENTER(ctx)                                                           \
    if (!(ctx)) return fail(TRS_E_ARG, "null context");                          \
    TrsDeviceGuard trs_guard_((ctx)->device);                                    \
    if (trs_guard_.err != cudaSuccess) return cuda_fail(trs_guard_.err, "cudaSetDevice")

}  // namespace

extern "C" {

int trs_version(void) { return TRS_VERSION; }
const char* trs_last_error(void) { return g_err; }
unsigned long long trs_kernel_launches(void) { return g_launches.load(); }

int trs_ctx_create(int device, trs_ctx** out)
{
    if (!out) return fail(TRS_E_ARG, "null out pointer");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        cudaGetLastError();
        return fail(TRS_E_NODEVICE, "no CUDA device (%s): this library has no CPU path", e == cudaSuccess ? "count=0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= count) return fail(TRS_E_ARG, "device %d of %d", device, count);
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) return fail(TRS_E_NODEVICE, "device %d is sm_%d%d; the kernels are built for sm_100a only", device, prop.major, prop.minor);
    trs_ctx* c = new (std::nothrow) trs_ctx();
    if (!c) return fail(TRS_E_ARG, "out of host memory");
    c->device = device;
    c->sm_count = prop.multiProcessorCount;
    c->smem_optin = (int)prop.sharedMemPerBlockOptin;
    c->cc_major = prop.major; c->cc_minor = prop.minor;
    c->sw.force_generic = getenv("TRS_FORCE_GENERIC") != nullptr;
    c->sw.no_banded = getenv("TRS_NO_BANDED") != nullptr;
    c->sw.no_store_warp = getenv("TRS_NO_STORE_WARP") != nullptr;
    c->sw.resize_scalar = getenv("TRS_RESIZE_SCALAR") != nullptr;
    c->sw.resize_gather = getenv("TRS_RESIZE_GATHER") != nullptr;
    if (const char* e = getenv("TRS_LOCATE")) c->sw.locate = e[0] == 'w' ? 1 : (e[0] == 'g' ? 3 : 2);
    if (const char* e = getenv("TRS_HOST_CHUNK_MB")) { const int mb = atoi(e); if (mb > 0) c->sw.host_chunk_bytes = (size_t)mb << 20; }
    trs_preproc_params d;
    default_params(&d);
    derive_params(c, &d);
    *out = c;
    return 0;
}

int trs_ctx_destroy(trs_ctx* ctx)
{
    if (!ctx) return 0;
    TrsDeviceGuard guard(ctx->device);
    for (int i = 0; i < HOST_STREAMS; ++i) {
        if (ctx->hs[i]) cudaStreamDestroy(ctx->hs[i]);
        cudaFree(ctx->st_in[i]); cudaFree(ctx->st_u8[i]); cudaFree(ctx->st_f32[i]);
    }
    if (ctx->host_entry) cudaEventDestroy(ctx->host_entry);
    cudaFree(ctx->wp_dev); cudaFree(ctx->wp_grid_dev); cudaFree(ctx->wp_cells_dev); cudaFree(ctx->defer_dev);
    cudaFree(ctx->stats_dev);
    cudaFree(ctx->jpg_blob); cudaFree(ctx->jpg_planes); cudaFree(ctx->jpg_meta);
    cudaFree(ctx->jpe_meta); cudaFree(ctx->jpe_sizes); cudaFree(ctx->jpe_offs); cudaFree(ctx->jpe_blob);
    delete ctx;
    return 0;
}

int trs_ctx_device_info(trs_ctx* ctx, int* sm_count, int* smem_optin_bytes, int* cc_major, int* cc_minor)
{
    if (!ctx) return fail(TRS_E_ARG, "null context");
    if (sm_count) *sm_count = ctx->sm_count;
    if (smem_optin_bytes) *smem_optin_bytes = ctx->smem_optin;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    return 0;
}

int trs_set_preproc_params(trs_ctx* ctx, const trs_preproc_params* p)
{
    if (!ctx || !p) return fail(TRS_E_ARG, "null argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    return derive_params(ctx, p);
}

int trs_preprocess(trs_ctx* ctx, const uint8_t* in_dev, int n, int h, int w, uint8_t* out_u8_dev, float* out_f32_dev,
                   unsigned long long* stats_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0 || h < 0 || w < 0) return fail(TRS_E_ARG, "negative size n=%d h=%d w=%d", n, h, w);
    if (n == 0 || h == 0 || w == 0) return 0;
    if (!in_dev) return fail(TRS_E_ARG, "null input");
    if (!out_u8_dev && !out_f32_dev && !stats_dev) return fail(TRS_E_ARG, "no output requested");
    return launch_preprocess(ctx, in_dev, n, h, w, out_u8_dev, out_f32_dev, stats_dev, nullptr, nullptr, false, (cudaStream_t)stream);
}

int trs_debug_canny_stages(trs_ctx* ctx, const uint8_t* in_dev, int h, int w, uint16_t* mag_dev, uint8_t* map_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (!in_dev || h <= 0 || w <= 0) return fail(TRS_E_ARG, "bad argument");
    return launch_preprocess(ctx, in_dev, 1, h, w, nullptr, nullptr, nullptr, mag_dev, map_dev, true, (cudaStream_t)stream);
}

int trs_normalise(trs_ctx* ctx, const uint8_t* in_dev, int n, int h_in, int w_in, int roi_y0, int roi_y1, int roi_x0, int roi_x1,
                  int h_out, int w_out, float* out_f32_dev, uint8_t* out_u8_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0 || h_in < 0 || w_in < 0 || h_out < 0 || w_out < 0) return fail(TRS_E_ARG, "negative size");
    if (roi_y0 < 0 || roi_x0 < 0 || roi_y1 > h_in || roi_x1 > w_in || roi_y1 < roi_y0 || roi_x1 < roi_x0)
        return fail(TRS_E_ARG, "window rows [%d,%d) cols [%d,%d) outside a %dx%d frame", roi_y0, roi_y1, roi_x0, roi_x1, h_in, w_in);
    if (n == 0 || h_out == 0 || w_out == 0) return 0;
    if (roi_y1 == roi_y0 || roi_x1 == roi_x0) return fail(TRS_E_ARG, "empty source window for a non-empty output");
    if (!in_dev || (!out_f32_dev && !out_u8_dev)) return fail(TRS_E_ARG, "null pointer");
    cudaStream_t st = (cudaStream_t)stream;
    const bool identity = roi_y0 == 0 && roi_x0 == 0 && roi_y1 == h_in && roi_x1 == w_in && h_out == h_in && w_out == w_in;
    const size_t total = (size_t)n * h_out * w_out * 3;
    if (identity && out_f32_dev && !out_u8_dev && ((uintptr_t)in_dev & 15) == 0 && ((uintptr_t)out_f32_dev & 15) == 0) {
        const size_t chunks = total / 4;                    // 32-bit words
        if (chunks) {
            size_t want = (chunks + 256 * 8 - 1) / (256 * 8);
            const size_t cap = (size_t)ctx->sm_count * 32;
            const int grid = (int)(want < cap ? want : cap);
            trs::k_normalise_stream<8><<<grid, 256, 0, st>>>(reinterpret_cast<const uint32_t*>(in_dev), reinterpret_cast<float4*>(out_f32_dev), chunks);
            g_launches.fetch_add(1, std::memory_order_relaxed);
        }
        const size_t done = chunks * 4;
        if (done < total) {
            trs::k_normalise_bytes<<<1, 32, 0, st>>>(in_dev + done, out_f32_dev + done, total - done);
            g_launches.fetch_add(1, std::memory_order_relaxed);
        }
        CU(cudaGetLastError());
        return 0;
    }
    trs::ResizeParams p{in_dev, out_f32_dev, out_u8_dev, n, h_in, w_in, roi_y0, roi_x0, roi_y1 - roi_y0, roi_x1 - roi_x0, h_out, w_out};
    if ((w_out * 3) % 4 == 0 && w_out + h_out <= trs::RESIZE_MAX_TAB && (!out_f32_dev || ((uintptr_t)out_f32_dev & 15) == 0) &&
        (!out_u8_dev || ((uintptr_t)out_u8_dev & 3) == 0) && !ctx->sw.resize_scalar) {
        const size_t rows = (size_t)n * h_out;
        const size_t cap = (size_t)ctx->sm_count * 16;
        // source rows staged in shared memory when they are 16-byte aligned (camera.py:36: 320x240 -> 160x120 is)
        const int col_lo = (3 * roi_x0) & ~15, col_hi = (3 * roi_x1 + 15) & ~15;
        const int span = (col_hi < w_in * 3 ? col_hi : w_in * 3) - col_lo;
        const size_t tab = ((sizeof(int) * 4 * (size_t)((w_out * 3) >> 2) + sizeof(int) * (size_t)h_out + 15) & ~(size_t)15);
        if ((w_in * 3) % 16 == 0 && ((uintptr_t)in_dev & 15) == 0 && span % 16 == 0 && tab + trs::RESIZE_DEPTH * (size_t)span <= 48 * 1024 &&
            !ctx->sw.resize_gather) {
            trs::k_crop_resize_rows<<<(int)(rows < cap ? rows : cap), trs::RESIZE_THREADS, tab + trs::RESIZE_DEPTH * (size_t)span, st>>>(p, col_lo, span);
            g_launches.fetch_add(1, std::memory_order_relaxed);
            CU(cudaGetLastError());
            return 0;
        }
        trs::k_crop_resize_words<<<(int)(rows < cap ? rows : cap), trs::RESIZE_THREADS, sizeof(int) * (size_t)(w_out + h_out), st>>>(p);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CU(cudaGetLastError());
        return 0;
    }
    const size_t px = total / 3;
    size_t want = (px + 255) / 256;
    const size_t cap = (size_t)ctx->sm_count * 16;
    trs::k_crop_resize<<<(int)(want < cap ? want : cap), 256, 0, st>>>(p);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    return 0;
}

int trs_set_track(trs_ctx* ctx, const double* wp_xyz_host, int n_wp, double min_map, double max_map)
{
    TRS_ENTER(ctx);
    if (!wp_xyz_host || n_wp <= 0) return fail(TRS_E_ARG, "empty centre line");
    std::lock_guard<std::mutex> lk(ctx->mu);
    // only first occurrences are uploaded, each with its original index (loc_grid.h)
    const std::vector<double> quads = trs::locg_distinct_quads(wp_xyz_host, n_wp);
    cudaFree(ctx->wp_dev);
    ctx->wp_dev = nullptr;
    CU(cudaMalloc(&ctx->wp_dev, sizeof(double) * quads.size()));
    CU(cudaMemcpy(ctx->wp_dev, quads.data(), sizeof(double) * quads.size(), cudaMemcpyHostToDevice));
    ctx->n_wp = n_wp;
    ctx->n_wp_distinct = (int)(quads.size() / 4);
    ctx->min_map = min_map;
    ctx->max_map = max_map;
    // uniform grid over (x, z) for k_locate_grid (loc_grid.h); none for non-finite coordinates, a handful of points or a table beyond shared memory:
    // the scanning kernels serve every batch then
    cudaFree(ctx->wp_grid_dev); ctx->wp_grid_dev = nullptr;
    cudaFree(ctx->wp_cells_dev); ctx->wp_cells_dev = nullptr;
    trs::LocGrid g{};
    std::vector<double> sorted;
    std::vector<int> start;
    if (trs::locg_build(quads, (size_t)ctx->smem_optin - 1024, g, sorted, start)) {
        CU(cudaMalloc(&ctx->wp_grid_dev, sizeof(double) * sorted.size()));
        CU(cudaMemcpy(ctx->wp_grid_dev, sorted.data(), sizeof(double) * sorted.size(), cudaMemcpyHostToDevice));
        CU(cudaMalloc(&ctx->wp_cells_dev, sizeof(int) * start.size()));
        CU(cudaMemcpy(ctx->wp_cells_dev, start.data(), sizeof(int) * start.size(), cudaMemcpyHostToDevice));
        CU(cudaFuncSetAttribute(trs::k_locate_grid, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)trs::locg_table_bytes(g)));
        ctx->grid = g;
    }
    return 0;
}

int trs_locate(trs_ctx* ctx, const double* xyz_dev, int n, int32_t* idx_dev, double* segment_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (!ctx->wp_dev) return fail(TRS_E_STATE, "trs_locate before trs_set_track");
    if (n < 0) return fail(TRS_E_ARG, "negative n");
    if (n == 0) return 0;
    if (!xyz_dev || (!idx_dev && !segment_dev)) return fail(TRS_E_ARG, "null pointer");
    // small batches: a warp per car with a shuffle reduction (a thread per car would not fill the GPU); large ones: the grid walk, with the
    // cars it puts off finished by the warp-per-car kernel; TRS_LOCATE=warp|thread|grid forces one
    const bool warp_per_car = ctx->sw.locate ? ctx->sw.locate == 1 : n < ctx->sm_count * 256;      // measured crossover ~50 k cars (15 us vs 55 us below it)
    if (!warp_per_car && ctx->sw.locate != 2 && ctx->wp_grid_dev) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->defer_cap < (size_t)n) {
            cudaFree(ctx->defer_dev); ctx->defer_dev = nullptr; ctx->defer_cap = 0;
            CU(cudaMalloc(&ctx->defer_dev, sizeof(int) * ((size_t)n + 1)));
            ctx->defer_cap = (size_t)n;
        }
        cudaStream_t st = (cudaStream_t)stream;
        CU(cudaMemsetAsync(ctx->defer_dev, 0, sizeof(int), st));
        const trs::LocGrid& g = ctx->grid;
        const size_t smem = trs::locg_table_bytes(g);
        int per_sm = 0;
        CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trs::k_locate_grid, trs::LOCG_THREADS, smem));
        per_sm = std::max(1, per_sm);
        int grid = (n + trs::LOCG_THREADS - 1) / trs::LOCG_THREADS;
        grid = std::min(grid, ctx->sm_count * per_sm);
        trs::k_locate_grid<<<grid, trs::LOCG_THREADS, smem, st>>>(ctx->wp_grid_dev, ctx->wp_cells_dev, g, ctx->n_wp, ctx->min_map,
                                                                  ctx->max_map, xyz_dev, n, idx_dev, segment_dev, ctx->defer_dev + 1, ctx->defer_dev);
        CU(cudaGetLastError());
        trs::k_locate_warp<<<ctx->sm_count * 2, trs::LOCW_THREADS, 0, st>>>(reinterpret_cast<const double4*>(ctx->wp_dev), ctx->n_wp_distinct, ctx->n_wp, ctx->min_map,
                                                                            ctx->max_map, xyz_dev, n, idx_dev, segment_dev, ctx->defer_dev + 1, ctx->defer_dev);
        g_launches.fetch_add(2, std::memory_order_relaxed);
        CU(cudaGetLastError());
        return 0;
    }
    if (warp_per_car) {
        const int warps_per_block = trs::LOCW_THREADS / 32;
        int grid = (n + warps_per_block - 1) / warps_per_block;
        const int cap = ctx->sm_count * 8;
        if (grid > cap) grid = cap;
        trs::k_locate_warp<<<grid, trs::LOCW_THREADS, 0, (cudaStream_t)stream>>>(reinterpret_cast<const double4*>(ctx->wp_dev), ctx->n_wp_distinct, ctx->n_wp,
                                                                                 ctx->min_map, ctx->max_map, xyz_dev, n, idx_dev, segment_dev);
        g_launches.fetch_add(1, std::memory_order_relaxed);
        CU(cudaGetLastError());
        return 0;
    }
    const int per_block = trs::LOC_THREADS * trs::LOC_CARS;
    const int grid = (n + per_block - 1) / per_block;
    trs::k_locate<<<grid, trs::LOC_THREADS, 0, (cudaStream_t)stream>>>(reinterpret_cast<const double4*>(ctx->wp_dev), ctx->n_wp_distinct, ctx->n_wp, ctx->min_map,
                                                                       ctx->max_map, xyz_dev, n, idx_dev, segment_dev);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    return 0;
}

int trs_probe_fp64(trs_ctx* ctx, double* dfma_tflops, double* dadd_tinst_per_s)
{
    TRS_ENTER(ctx);
    const int grid = ctx->sm_count * 8, iters = 4096;
    double* buf = nullptr;
    CU(cudaMalloc(&buf, sizeof(double) * (size_t)grid * trs::PROBE64_THREADS));
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    double rate[2] = {0, 0};
    cudaError_t err = cudaSuccess;
    for (int which = 0; which < 2 && err == cudaSuccess; ++which) {
        float best = 1e30f;
        for (int rep = 0; rep < 4; ++rep) {                      // rep 0 warms up
            cudaEventRecord(e0, 0);
            if (which == 0) trs::k_probe_fp64<true><<<grid, trs::PROBE64_THREADS>>>(buf, iters, 0.999999, 1e-9);
            else trs::k_probe_fp64<false><<<grid, trs::PROBE64_THREADS>>>(buf, iters, 0.0, 1e-9);
            cudaEventRecord(e1, 0);
            err = cudaEventSynchronize(e1);
            if (err != cudaSuccess) break;
            float ms = 0;
            cudaEventElapsedTime(&ms, e0, e1);
            if (rep && ms < best) best = ms;
        }
        g_launches.fetch_add(4, std::memory_order_relaxed);
        rate[which] = (double)grid * trs::PROBE64_THREADS * trs::PROBE64_ILP * (double)iters / ((double)best * 1e-3);      // lane-instructions per second
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    cudaFree(buf);
    if (err != cudaSuccess) return cuda_fail(err, "fp64 probe");
    if (dfma_tflops) *dfma_tflops = 2.0 * rate[0] / 1e12;
    if (dadd_tinst_per_s) *dadd_tinst_per_s = rate[1] / 1e12;
    return 0;
}

int trs_speed_control(trs_ctx* ctx, const double* cur_spd_dev, const float* model_spd_dev, const float* model_steer_dev, int n,
                      const trs_spd_params* p, double* steering_dev, double* throttle_dev, double* breaking_dev,
                      float* spd_feature_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0 || !p) return fail(TRS_E_ARG, "bad argument");
    if (n == 0) return 0;
    if (!cur_spd_dev || !model_spd_dev || !model_steer_dev || !steering_dev || !throttle_dev || !breaking_dev)
        return fail(TRS_E_ARG, "null pointer");
    trs::SpdKParams k{p->threshold, p->reverse_multiplier, p->break_multiplier, p->smooth_threshold, p->use_break ? 1 : 0,
                      p->smooth_steering ? 1 : 0, p->numpy_legacy_promotion ? 1 : 0};
    int grid = (n + 255) / 256;
    const int cap = ctx->sm_count * 8;
    if (grid > cap) grid = cap;
    trs::k_speed_control<<<grid, 256, 0, (cudaStream_t)stream>>>(cur_spd_dev, model_spd_dev, model_steer_dev, n, k, steering_dev,
                                                                  throttle_dev, breaking_dev, spd_feature_dev);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    return 0;
}

int trs_control_mux(trs_ctx* ctx, const int32_t* mode_dev, const double* usr_dev, const double* ai_dev, const double* speed_dev, int n,
                    const trs_ctl_params* p, double now_s, int32_t* last_mode_dev, double* launch_times_dev, double* out_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0 || !p) return fail(TRS_E_ARG, "bad argument");
    if (n == 0) return 0;
    if (!mode_dev || !usr_dev || !ai_dev || !last_mode_dev || !launch_times_dev || !out_dev) return fail(TRS_E_ARG, "null pointer");
    if (p->assist_mode < 0 || p->assist_mode > 2) return fail(TRS_E_ARG, "assist_mode %d (0 off, 1 steering, 2 speed)", p->assist_mode);
    static_assert(TRS_LAUNCH_SLOTS == trs::CTL_LAUNCH_SLOTS, "header and kernel disagree on the launch slots");
    trs::CtlKParams k{p->throttle_lock_enabled ? 1 : 0, p->steering_lock_enabled ? 1 : 0, p->assist_mode, p->throttle_lock_value,
                      p->throttle_lock_duration, p->steering_lock_value, p->steering_lock_duration, p->assist_k};
    int grid = (n + 255) / 256;
    const int cap = ctx->sm_count * 8;
    if (grid > cap) grid = cap;
    trs::k_control_mux<<<grid, 256, 0, (cudaStream_t)stream>>>(mode_dev, usr_dev, ai_dev, speed_dev, n, k, now_s, last_mode_dev, launch_times_dev,
                                                                out_dev);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    return 0;
}

int trs_pwm_map(trs_ctx* ctx, const double* val_dev, int n, double min_map, double mid_map, double max_map, double* out_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0) return fail(TRS_E_ARG, "negative n");
    if (n == 0) return 0;
    if (!val_dev || !out_dev) return fail(TRS_E_ARG, "null pointer");
    int grid = (n + 255) / 256;
    const int cap = ctx->sm_count * 8;
    if (grid > cap) grid = cap;
    trs::k_pwm_map<<<grid, 256, 0, (cudaStream_t)stream>>>(val_dev, n, min_map, mid_map, max_map, out_dev);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    return 0;
}

int trs_jpeg_decode_host(trs_ctx* ctx, const uint8_t* blob_host, const unsigned long long* offsets_host, int n, int h, int w,
                         uint8_t* out_u8_dev, void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0 || h <= 0 || w <= 0) return fail(TRS_E_ARG, "bad size n=%d h=%d w=%d", n, h, w);
    if (n == 0) return 0;
    if (!blob_host || !offsets_host || !out_u8_dev) return fail(TRS_E_ARG, "null pointer");
    std::lock_guard<std::mutex> lk(ctx->mu);
    cudaStream_t st = (cudaStream_t)stream;
    // ---- the files start crossing the PCIe link first (436 MB for 65,536 records: 8 ms), the headers are parsed meanwhile ----------
    for (int k = 0; k < n; ++k)
        if (offsets_host[k + 1] < offsets_host[k]) return fail(TRS_E_ARG, "offsets not ascending at record %d", k);
    const size_t blob_bytes = (size_t)offsets_host[n];
    if (ctx->jpg_blob_cap < blob_bytes + 32) { cudaFree(ctx->jpg_blob); ctx->jpg_blob = nullptr; ctx->jpg_blob_cap = 0; CU(cudaMalloc(&ctx->jpg_blob, blob_bytes + 32)); ctx->jpg_blob_cap = blob_bytes + 32; }
    CU(cudaMemcpyAsync(ctx->jpg_blob, blob_host, blob_bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(ctx->jpg_blob + blob_bytes, 0, 32, st));                   // the bit reader loads one 8-byte chunk ahead
    // ---- host: parse every file (threads; a file whose header bytes equal the previous file's reuses its tables) -----------------
    std::vector<trs::JpegRecord> recs((size_t)n);
    std::vector<trs::JpegTables> sets;
    std::mutex sets_mu;
    std::atomic<int> first_bad{n};
    std::atomic<int> sampling{0};                                // (hs << 4 | vs) of the batch: every record must agree
    std::vector<int> bad_code((size_t)n, 0);
    unsigned nthreads = std::thread::hardware_concurrency();
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 16) nthreads = 16;
    if ((unsigned)n < 64 * nthreads) nthreads = 1;
    auto work = [&](int k0, int k1) {
        const uint8_t* prev = nullptr;
        uint32_t prev_hdr = 0, prev_set = 0;
        for (int k = k0; k < k1; ++k) {
            const unsigned long long a = offsets_host[k], b = offsets_host[k + 1];
            if (b < a) { bad_code[(size_t)k] = -1; int cur = first_bad.load(); while (k < cur && !first_bad.compare_exchange_weak(cur, k)) {} continue; }
            const uint8_t* f = blob_host + a;
            const size_t len = (size_t)(b - a);
            if (prev && len > prev_hdr && memcmp(prev, f, prev_hdr) == 0) {          // same header bytes: same size, tables and scan parameters
                recs[(size_t)k] = trs::JpegRecord{a + prev_hdr, (uint32_t)(len - prev_hdr), prev_set};
                continue;
            }
            trs::JpegTables T;
            trs::JpegScan S;
            memset(&T, 0, sizeof T);
            int pr = trs::jpg_parse(f, len, &T, &S);
            if (!pr && (S.h != h || S.w != w)) pr = -2;
            if (!pr) {
                int expect = 0;
                const int mine = (S.hs << 4) | S.vs;
                if (!sampling.compare_exchange_strong(expect, mine) && expect != mine) pr = -4;
            }
            if (pr) { bad_code[(size_t)k] = pr; int cur = first_bad.load(); while (k < cur && !first_bad.compare_exchange_weak(cur, k)) {} continue; }
            size_t si = 0;
            {
                std::lock_guard<std::mutex> g(sets_mu);
                for (; si < sets.size(); ++si)
                    if (memcmp(&sets[si], &T, sizeof T) == 0) break;
                if (si == sets.size()) {
                    if (sets.size() >= 64) { bad_code[(size_t)k] = -3; int cur = first_bad.load(); while (k < cur && !first_bad.compare_exchange_weak(cur, k)) {} continue; }
                    sets.push_back(T);
                }
            }
            recs[(size_t)k] = trs::JpegRecord{a + S.data_off, S.data_len, (uint32_t)si};
            prev = f; prev_hdr = S.data_off; prev_set = (uint32_t)si;
        }
    };
    if (nthreads == 1) {
        work(0, n);
    } else {
        std::vector<std::thread> pool;
        const int per = (n + (int)nthreads - 1) / (int)nthreads;
        for (unsigned t = 0; t < nthreads; ++t) {
            const int k0 = (int)t * per, k1 = k0 + per < n ? k0 + per : n;
            if (k0 < k1) pool.emplace_back(work, k0, k1);
        }
        for (auto& th : pool) th.join();
    }
    if (first_bad.load() < n) {
        cudaStreamSynchronize(st);                                                // the upload reads the caller's buffer: let it finish
        const int k = first_bad.load(), c = bad_code[(size_t)k];
        if (c == -1) return fail(TRS_E_ARG, "offsets not ascending at record %d", k);
        if (c == -2) return fail(TRS_E_RANGE, "record %d does not have the stated size %dx%d", k, h, w);
        if (c == -3) return fail(TRS_E_RANGE, "more than 64 distinct quantisation / Huffman table sets in one batch");
        if (c == -4) return fail(TRS_E_RANGE, "record %d has another chroma subsampling than the records before it (one per batch)", k);
        return fail(TRS_E_RANGE, "record %d: %s", k, c == trs::JPG_E_UNSUPPORTED ? "not a baseline 8-bit YCbCr (4:2:0 / 4:2:2 / 4:4:4) single-scan JPEG" : "malformed JPEG");
    }
    // ---- device staging: chunks of records through coefficient and plane buffers ----------------------------------------------
    const int hs = sampling.load() >> 4, vs = sampling.load() & 15;
    const int mw = (w + 8 * hs - 1) / (8 * hs), mh = (h + 8 * vs - 1) / (8 * vs);
    const size_t ybytes = (size_t)mw * 8 * hs * mh * 8 * vs, cbytes = (size_t)mw * 8 * mh * 8;
    // Entropy decoding is one thread per record and latency bound: the more records in flight the better, so chunks are as large as
    // ~8 GB of plane staging allows (290 k records of 120x160)
    size_t chunk = ((size_t)8 << 30) / (ybytes + 2 * cbytes);
    if (chunk < 1) chunk = 1;
    if (chunk > (size_t)n) chunk = (size_t)n;
    const size_t planes_bytes = chunk * (ybytes + 2 * cbytes);
    const size_t meta_bytes = sets.size() * sizeof(trs::JpegTables) + (size_t)n * sizeof(trs::JpegRecord) + 16;
    if (ctx->jpg_planes_cap < planes_bytes) { cudaFree(ctx->jpg_planes); ctx->jpg_planes = nullptr; ctx->jpg_planes_cap = 0; CU(cudaMalloc(&ctx->jpg_planes, planes_bytes)); ctx->jpg_planes_cap = planes_bytes; }
    if (ctx->jpg_meta_cap < meta_bytes) { cudaFree(ctx->jpg_meta); ctx->jpg_meta = nullptr; ctx->jpg_meta_cap = 0; CU(cudaMalloc(&ctx->jpg_meta, meta_bytes)); ctx->jpg_meta_cap = meta_bytes; }
    trs::JpegTables* d_sets = reinterpret_cast<trs::JpegTables*>(ctx->jpg_meta);
    trs::JpegRecord* d_recs = reinterpret_cast<trs::JpegRecord*>(reinterpret_cast<uint8_t*>(ctx->jpg_meta) + sets.size() * sizeof(trs::JpegTables));
    int* d_status = reinterpret_cast<int*>(reinterpret_cast<uint8_t*>(d_recs) + (size_t)n * sizeof(trs::JpegRecord));
    uint8_t* d_planes = ctx->jpg_planes;
    CU(cudaMemcpyAsync(d_sets, sets.data(), sets.size() * sizeof(trs::JpegTables), cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_recs, recs.data(), (size_t)n * sizeof(trs::JpegRecord), cudaMemcpyHostToDevice, st));
    CU(cudaMemsetAsync(d_status, 0, sizeof(int), st));
    for (size_t c0 = 0; c0 < (size_t)n; c0 += chunk) {
        const int cn = (int)((size_t)n - c0 < chunk ? (size_t)n - c0 : chunk);
        trs::JpegPlanes P{d_planes, d_planes + (size_t)cn * ybytes, d_planes + (size_t)cn * (ybytes + cbytes), mw, mh, hs, vs};
        trs::k_jpeg_entropy<<<(cn + trs::JPG_THREADS - 1) / trs::JPG_THREADS, trs::JPG_THREADS, 0, st>>>(ctx->jpg_blob, d_recs + c0, d_sets, cn, P, d_status);
        const size_t groups = (size_t)cn * h * ((w + 3) / 4);
        size_t want = (groups + 255) / 256;
        const size_t cap = (size_t)ctx->sm_count * 32;
        trs::k_jpeg_upsample_rgb<<<(int)(want < cap ? want : cap), 256, 0, st>>>(P, cn, h, w, out_u8_dev + c0 * (size_t)h * w * 3);
        g_launches.fetch_add(2, std::memory_order_relaxed);
        CU(cudaGetLastError());
    }
    int status = 0;
    CU(cudaMemcpyAsync(&status, d_status, sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));                              // recs / sets (host vectors) and the staging buffers are reused
    if (status) return fail(TRS_E_RANGE, "corrupt entropy-coded data in at least one record (decoder status %d)", status);
    return 0;
}

int trs_jpeg_encode(trs_ctx* ctx, const uint8_t* frames_dev, int n, int h, int w, int quality, unsigned long long* offsets_host,
                    void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0) return fail(TRS_E_ARG, "negative record count %d", n);
    if (h < 1 || h > 65535 || w < 1 || w > 65535) return fail(TRS_E_ARG, "frame size %dx%d outside 1..65535", h, w);
    if (quality < 1 || quality > 100) return fail(TRS_E_ARG, "quality %d outside 1..100", quality);
    if (!offsets_host) return fail(TRS_E_ARG, "null offsets_host");
    if (n > 0 && !frames_dev) return fail(TRS_E_ARG, "null frames_dev");
    std::lock_guard<std::mutex> lk(ctx->mu);
    ctx->jpe_last_bytes = -1;
    offsets_host[0] = 0;
    if (n == 0) { ctx->jpe_last_bytes = 0; return 0; }
    cudaStream_t st = (cudaStream_t)stream;
    // tables and headers depend only on (h, w, quality): built on the host, uploaded when they change
    const size_t meta_bytes = sizeof(trs::JpeEncTables) + trs::JPE_HEADER_BYTES;
    if (!ctx->jpe_meta) { CU(cudaMalloc(&ctx->jpe_meta, meta_bytes)); ctx->jpe_meta_key[0] = 0; }
    if (ctx->jpe_meta_key[0] != h || ctx->jpe_meta_key[1] != w || ctx->jpe_meta_key[2] != quality) {
        std::vector<uint8_t> meta(meta_bytes);
        trs::JpeEncTables T;
        trs::jpe_make_tables(quality, T);
        memcpy(meta.data(), &T, sizeof T);
        trs::jpe_build_header(h, w, quality, meta.data() + sizeof T);
        ctx->jpe_meta_key[0] = 0;
        CU(cudaMemcpyAsync(ctx->jpe_meta, meta.data(), meta_bytes, cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));                                              // `meta` is a local vector
        ctx->jpe_meta_key[0] = h; ctx->jpe_meta_key[1] = w; ctx->jpe_meta_key[2] = quality;
    }
    const trs::JpeEncTables* d_tables = reinterpret_cast<const trs::JpeEncTables*>(ctx->jpe_meta);
    const uint8_t* d_header = ctx->jpe_meta + sizeof(trs::JpeEncTables);
    if (ctx->jpe_sizes_cap < (size_t)n) {
        cudaFree(ctx->jpe_sizes); cudaFree(ctx->jpe_offs);
        ctx->jpe_sizes = ctx->jpe_offs = nullptr; ctx->jpe_sizes_cap = 0;
        CU(cudaMalloc(&ctx->jpe_sizes, (size_t)n * sizeof(unsigned long long)));
        CU(cudaMalloc(&ctx->jpe_offs, ((size_t)n + 1) * sizeof(unsigned long long)));
        ctx->jpe_sizes_cap = (size_t)n;
    }
    const int smem = (int)sizeof(trs::JpeSmem);
    CU(cudaFuncSetAttribute(trs::k_jpeg_encode<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    CU(cudaFuncSetAttribute(trs::k_jpeg_encode<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    int per_sm = 0;
    CU(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, trs::k_jpeg_encode<true>, trs::JPE_THREADS, smem));
    if (per_sm < 1) return fail(TRS_E_RANGE, "encoder does not fit an SM with %d B shared memory", smem);
    const int grid = n < ctx->sm_count * per_sm ? n : ctx->sm_count * per_sm;
    // pass 1: exact file sizes (the same arithmetic as pass 2, nothing written but the sizes)
    trs::k_jpeg_encode<false><<<grid, trs::JPE_THREADS, smem, st>>>(frames_dev, n, h, w, d_tables, d_header, ctx->jpe_sizes, nullptr, nullptr);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    std::vector<unsigned long long>& offs = ctx->jpe_host_offs;
    offs.assign((size_t)n + 1, 0);
    CU(cudaMemcpyAsync(offs.data() + 1, ctx->jpe_sizes, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    for (size_t k = 1; k <= (size_t)n; ++k) offs[k] += offs[k - 1];
    const size_t total = (size_t)offs[(size_t)n];
    if (ctx->jpe_blob_cap < total) {
        cudaFree(ctx->jpe_blob); ctx->jpe_blob = nullptr; ctx->jpe_blob_cap = 0;
        CU(cudaMalloc(&ctx->jpe_blob, total));
        ctx->jpe_blob_cap = total;
    }
    // pass 2: every file at its offset
    CU(cudaMemcpyAsync(ctx->jpe_offs, offs.data(), ((size_t)n + 1) * sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
    trs::k_jpeg_encode<true><<<grid, trs::JPE_THREADS, smem, st>>>(frames_dev, n, h, w, d_tables, d_header, nullptr, ctx->jpe_offs, ctx->jpe_blob);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CU(cudaGetLastError());
    memcpy(offsets_host, offs.data(), ((size_t)n + 1) * sizeof(unsigned long long));
    ctx->jpe_last_bytes = (long long)total;
    return 0;
}

int trs_jpeg_encode_copy(trs_ctx* ctx, uint8_t* blob_host, unsigned long long bytes, void* stream)
{
    TRS_ENTER(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->jpe_last_bytes < 0) return fail(TRS_E_STATE, "no successful trs_jpeg_encode on this context");
    if (bytes != (unsigned long long)ctx->jpe_last_bytes)
        return fail(TRS_E_ARG, "bytes = %llu, but the last trs_jpeg_encode produced %lld", bytes, ctx->jpe_last_bytes);
    if (bytes == 0) return 0;
    if (!blob_host) return fail(TRS_E_ARG, "null blob_host");
    cudaStream_t st = (cudaStream_t)stream;
    CU(cudaMemcpyAsync(blob_host, ctx->jpe_blob, (size_t)bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return 0;
}

int trs_telemetry_decode_host(trs_ctx* ctx, const char* text_host, const unsigned long long* offsets_host, int n, int h, int w,
                              uint8_t* out_u8_dev, void* stream)
{
    if (!ctx) return fail(TRS_E_ARG, "null context");
    if (n < 0 || h <= 0 || w <= 0) return fail(TRS_E_ARG, "bad size n=%d h=%d w=%d", n, h, w);
    if (n == 0) return 0;
    if (!text_host || !offsets_host || !out_u8_dev) return fail(TRS_E_ARG, "null pointer");
    // base64 -> bytes on the host: output offsets from the text lengths (an upper bound per string), decoded by up to 16 threads
    std::vector<unsigned long long> offs((size_t)n + 1);
    offs[0] = 0;
    for (int k = 0; k < n; ++k) {
        if (offsets_host[k + 1] < offsets_host[k]) return fail(TRS_E_ARG, "offsets not ascending at packet %d", k);
        offs[(size_t)k + 1] = offs[(size_t)k] + ((offsets_host[k + 1] - offsets_host[k]) / 4 + 1) * 3;
    }
    std::vector<uint8_t> blob((size_t)offs[(size_t)n] + 16);
    std::vector<unsigned long long> lens((size_t)n, 0);
    std::atomic<int> first_bad{n};
    static const struct B64Table {
        int8_t v[256];
        B64Table() {
            for (int i = 0; i < 256; ++i) v[i] = -1;
            const char* a = "ABCDEFGHIJKLMNOPQRSTUVWXYZabcdefghijklmnopqrstuvwxyz0123456789+/";
            for (int i = 0; i < 64; ++i) v[(unsigned char)a[i]] = (int8_t)i;
            v[(unsigned char)'='] = -2;
            v[(unsigned char)' '] = v[(unsigned char)'\n'] = v[(unsigned char)'\r'] = v[(unsigned char)'\t'] = -3;
        }
    } B64;
    auto work = [&](int k0, int k1) {
        for (int k = k0; k < k1; ++k) {
            const unsigned char* s = reinterpret_cast<const unsigned char*>(text_host) + offsets_host[k];
            const size_t len = (size_t)(offsets_host[k + 1] - offsets_host[k]);
            uint8_t* o = blob.data() + offs[(size_t)k];
            uint32_t acc = 0;
            int nb = 0;
            size_t out = 0;
            bool bad = false;
            for (size_t i = 0; i < len; ++i) {
                const int v = B64.v[s[i]];
                if (v >= 0) {
                    acc = (acc << 6) | (uint32_t)v;
                    if (++nb == 4) { o[out++] = (uint8_t)(acc >> 16); o[out++] = (uint8_t)(acc >> 8); o[out++] = (uint8_t)acc; nb = 0; acc = 0; }
                } else if (v == -2) {
                    break;                                           // padding: the rest is '='
                } else if (v != -3) {
                    bad = true;
                    break;
                }
            }
            if (nb == 3) { o[out++] = (uint8_t)(acc >> 10); o[out++] = (uint8_t)(acc >> 2); }
            else if (nb == 2) { o[out++] = (uint8_t)(acc >> 4); }
            else if (nb == 1) bad = true;
            if (bad) { int cur = first_bad.load(); while (k < cur && !first_bad.compare_exchange_weak(cur, k)) {} }
            lens[(size_t)k] = out;
        }
    };
    unsigned nthreads = std::thread::hardware_concurrency();
    if (nthreads < 1) nthreads = 1;
    if (nthreads > 16) nthreads = 16;
    if ((unsigned)n < 64 * nthreads) nthreads = 1;
    if (nthreads == 1) {
        work(0, n);
    } else {
        std::vector<std::thread> pool;
        const int per = (n + (int)nthreads - 1) / (int)nthreads;
        for (unsigned t = 0; t < nthreads; ++t) {
            const int k0 = (int)t * per, k1 = k0 + per < n ? k0 + per : n;
            if (k0 < k1) pool.emplace_back(work, k0, k1);
        }
        for (auto& th : pool) th.join();
    }
    if (first_bad.load() < n) return fail(TRS_E_RANGE, "packet %d: the image string is not valid base64", first_bad.load());
    // compact the files (the slots were sized by the upper bound) and hand them to the JPEG path
    std::vector<unsigned long long> foffs((size_t)n + 1);
    foffs[0] = 0;
    for (int k = 0; k < n; ++k) {
        if (foffs[(size_t)k] != offs[(size_t)k]) memmove(blob.data() + foffs[(size_t)k], blob.data() + offs[(size_t)k], (size_t)lens[(size_t)k]);
        foffs[(size_t)k + 1] = foffs[(size_t)k] + lens[(size_t)k];
    }
    return trs_jpeg_decode_host(ctx, blob.data(), foffs.data(), n, h, w, out_u8_dev, stream);
}

int trs_host_alloc(void** out, unsigned long long bytes)
{
    if (!out) return fail(TRS_E_ARG, "null out pointer");
    CU(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return 0;
}

int trs_host_free(void* p)
{
    if (p) CU(cudaFreeHost(p));
    return 0;
}

int trs_preprocess_host(trs_ctx* ctx, const uint8_t* in_host, int n, int h, int w, uint8_t* out_u8_host, float* out_f32_host,
                        float* keep_f32_dev, unsigned long long* stats_host, void* stream)
{
    TRS_ENTER(ctx);
    if (n < 0 || h < 0 || w < 0) return fail(TRS_E_ARG, "negative size");
    if (stats_host) memset(stats_host, 0, sizeof(unsigned long long) * TRS_STAT_COUNT);
    if (n == 0 || h == 0 || w == 0) return 0;
    if (!in_host) return fail(TRS_E_ARG, "null input");
    if (!out_u8_host && !out_f32_host && !keep_f32_dev && !stats_host) return fail(TRS_E_ARG, "no output requested");
    std::lock_guard<std::mutex> lk(ctx->mu);
    const size_t fb = (size_t)h * w * 3;
    size_t chunk = ctx->sw.host_chunk_bytes / fb;
    if (chunk < 1) chunk = 1;
    if (chunk > (size_t)n) chunk = n;
    chunk = (chunk + 3) & ~(size_t)3;                          // keeps every chunk base 16-byte aligned when fb % 4 == 0
    for (int i = 0; i < HOST_STREAMS; ++i)
        if (!ctx->hs[i]) CU(cudaStreamCreateWithFlags(&ctx->hs[i], cudaStreamNonBlocking));
    if (!ctx->host_entry) CU(cudaEventCreateWithFlags(&ctx->host_entry, cudaEventDisableTiming));
    const bool need_f32 = out_f32_host != nullptr;
    // staging buffers grow on demand; a capacity is only recorded once all three buffers of its kind exist
    int rc = grow_staging(ctx->st_in, ctx->st_in_cap, chunk * fb);
    if (!rc && out_u8_host) rc = grow_staging(ctx->st_u8, ctx->st_u8_cap, chunk * fb);
    if (!rc && need_f32 && !keep_f32_dev) rc = grow_staging(ctx->st_f32, ctx->st_f32_cap, chunk * fb * 4);
    if (rc) return rc;
    // the internal streams start after everything the caller has queued on ITS stream (a consumer of keep_f32_dev from the previous
    // step, the producer of a device-resident stats buffer, ...)
    CU(cudaEventRecord(ctx->host_entry, (cudaStream_t)stream));
    for (int i = 0; i < HOST_STREAMS; ++i) CU(cudaStreamWaitEvent(ctx->hs[i], ctx->host_entry, 0));
    // from here on copies into the caller's host buffers may be in flight: every exit drains the internal streams first
    auto drain = [&](int code) {
        for (int i = 0; i < HOST_STREAMS; ++i) cudaStreamSynchronize(ctx->hs[i]);
        return code;
    };
#define CUD(call)                                                       \
    do {                                                                \
        cudaError_t _e = (call);                                        \
        if (_e != cudaSuccess) return drain(cuda_fail(_e, #call));      \
    } while (0)
    if (stats_host) {
        if (!ctx->stats_dev) CUD(cudaMalloc(&ctx->stats_dev, sizeof(unsigned long long) * TRS_STAT_COUNT));
        CUD(cudaMemsetAsync(ctx->stats_dev, 0, sizeof(unsigned long long) * TRS_STAT_COUNT, ctx->hs[0]));
        CUD(cudaStreamSynchronize(ctx->hs[0]));
    }
    int ci = 0;
    for (size_t f0 = 0; f0 < (size_t)n; f0 += chunk, ++ci) {
        const int s = ci % HOST_STREAMS;
        const size_t cn = (size_t)n - f0 < chunk ? (size_t)n - f0 : chunk;
        cudaStream_t st = ctx->hs[s];
        CUD(cudaMemcpyAsync(ctx->st_in[s], in_host + f0 * fb, cn * fb, cudaMemcpyHostToDevice, st));
        uint8_t* du8 = out_u8_host ? ctx->st_u8[s] : nullptr;
        float* df32 = keep_f32_dev ? keep_f32_dev + f0 * fb : (need_f32 ? ctx->st_f32[s] : nullptr);
        rc = launch_preprocess(ctx, ctx->st_in[s], (int)cn, h, w, du8, df32, stats_host ? ctx->stats_dev : nullptr, nullptr, nullptr, false, st);
        if (rc) return drain(rc);
        if (out_u8_host) CUD(cudaMemcpyAsync(out_u8_host + f0 * fb, du8, cn * fb, cudaMemcpyDeviceToHost, st));
        if (need_f32) CUD(cudaMemcpyAsync(out_f32_host + f0 * fb, df32, cn * fb * 4, cudaMemcpyDeviceToHost, st));
    }
    cudaError_t first = cudaSuccess;
    for (int i = 0; i < HOST_STREAMS; ++i) { const cudaError_t e = cudaStreamSynchronize(ctx->hs[i]); if (first == cudaSuccess) first = e; }
    if (first != cudaSuccess) return cuda_fail(first, "cudaStreamSynchronize(host pipeline)");
    if (stats_host) CU(cudaMemcpy(stats_host, ctx->stats_dev, sizeof(unsigned long long) * TRS_STAT_COUNT, cudaMemcpyDeviceToHost));
#undef CUD
    return 0;
}

}  // extern "C"
