// pixel_math.cuh — per-pixel arithmetic of the observation path, written once for host and device.
//
// Every function here is pure (no memory, no threads) so the same source is compiled by nvcc into the
// kernels and by g++ into tests/host_math_check (a CPU-side check of this header against the oracle).
// The arithmetic specifications are SURVEY.md Appendix A; each function names the reference call site.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define TRS_HD __host__ __device__ __forceinline__
#else
#define TRS_HD inline
#endif

namespace trs {

// ---- RGB -> HSV, OpenCV 8-bit integer path (img_preprocessing.py:66, cv2.cvtColor RGB2HSV) -------------
// 12-bit fixed point; sdiv[i] = rint(255*4096/i), hdiv[i] = rint(180*4096/(6 i)), both 0 at i = 0.
struct HsvTables {
    int32_t sdiv[256];
    int32_t hdiv[256];
};

TRS_HD void rgb2hsv_px(int r, int g, int b, const int32_t* sdiv, const int32_t* hdiv, int& h, int& s, int& v)
{
    v = r > g ? r : g; v = b > v ? b : v;
    int vmin = r < g ? r : g; vmin = b < vmin ? b : vmin;
    const int d = v - vmin;
    s = (d * sdiv[v] + 2048) >> 12;
    int h0 = (v == r) ? (g - b) : ((v == g) ? (b - r + 2 * d) : (r - g + 4 * d));
    h = (h0 * hdiv[d] + 2048) >> 12;      // arithmetic shift = floor for negative h0
    h += (h < 0) ? 180 : 0;
}

// The two division tables of the 8-bit RGB -> HSV path, entry i (0 at i = 0).
TRS_HD int hsv_sdiv_entry(int i)
{
#if defined(__CUDA_ARCH__)
    return i ? __double2int_rn((double)(255 << 12) / (double)i) : 0;
#else
    return i ? (int)__builtin_rint((double)(255 << 12) / (double)i) : 0;
#endif
}
TRS_HD int hsv_hdiv_entry(int i)
{
#if defined(__CUDA_ARCH__)
    return i ? __double2int_rn((double)(180 << 12) / (6.0 * (double)i)) : 0;
#else
    return i ? (int)__builtin_rint((double)(180 << 12) / (6.0 * (double)i)) : 0;
#endif
}

// Saturation bounds without computing the saturation (preproc_fast.cuh, SatThresholds): s = (d sdiv[v] + 2048) >> 12 is monotone in the delta d, so
// "s <= K" is "d <= T_K[v]".  Returns T_K[v] as the 16-bit pattern the packed compares use: 0x8001 compares as -1 (no delta qualifies).
// A lower bound "s >= L" is "d > T_{L-1}[v]": pass K = L - 1.
TRS_HD uint32_t sat_threshold_entry(long long K, int v, int sd)
{
    if (K < 0) return 0x8001u;                                    // no d qualifies (compares as -1)
    if (v == 0) return 0u;                                        // v = 0: d = 0, s = 0
    const long long q = (4096 * K + 2047) / sd;
    return (uint32_t)(q < v ? q : v);
}

// ... with the value bounds [vlo, vhi] of the same range folded in (the table is indexed by v already): a value outside them gets a threshold no
// delta passes, 0x8001 (-1) for an upper saturation bound "d <= T" and 255 for a lower one "d > T" (d <= v <= 255).  `upper`: which of the two the
// entry serves; K as for sat_threshold_entry.
TRS_HD uint32_t sat_threshold_entry_folded(long long K, bool upper, int v, int sd, long long vlo, long long vhi)
{
    if (v < vlo || v > vhi) return upper ? 0x8001u : 255u;
    return sat_threshold_entry(K, v, sd);
}

// Hue bounds without computing the hue (preproc_fast.cuh, HueThresholds): h = (h0 hdiv[d] + 2048) >> 12 is monotone in the numerator h0, and a
// wrapped hue (h0 < 0: h + 180 >= 150) cannot pass an upper bound <= 149, so "lo <= h <= hi" is "a_lo <= h0 <= a_hi" for such a bound: the smallest
// numerator with h0 hd + 2048 >= 4096 lo and the largest with h0 hd + 2048 <= 4096 hi + 4095.  Returned biased by 2048 like the packed numerators, as
// (a_lo + 2048) | (a_hi + 2048) << 16.  Needs lo >= 0 as well (a negative lower bound would admit the unwrapped values lo .. -1, whose hue is 177 .. 179):
// the variant is only used when the lower bound can fail, i.e. is positive.
TRS_HD uint32_t hue_threshold_entry(long long lo, long long hi, int hd)
{
    long long a_lo, a_hi;
    if (hd == 0) {                                                // grey pixel: h = 0
        const bool pass = lo <= 0 && 0 <= hi;
        a_lo = pass ? -2048 : 1; a_hi = pass ? 4000 : 0;
    } else {
        const long long nl = 4096 * lo - 2048, nh = 4096 * hi + 2047;
        a_lo = nl >= 0 ? (nl + hd - 1) / hd : -((-nl) / hd);      // ceiling
        a_hi = nh >= 0 ? nh / hd : -((-nh + hd - 1) / hd);        // floor
    }
    a_lo = a_lo < -2048 ? -2048 : (a_lo > 20000 ? 20000 : a_lo);
    a_hi = a_hi < -2048 ? -2048 : (a_hi > 20000 ? 20000 : a_hi);
    return (uint32_t)(a_lo + 2048) | ((uint32_t)(a_hi + 2048) << 16);
}

// ---- inRange with pre-rounded integer bounds (img_preprocessing.py:71, cv2.inRange) --------------------
// OpenCV rounds each scalar bound to int32 (half-to-even; out of range -> INT_MIN) before comparing.
struct HsvRange {
    int32_t lo[3];
    int32_t hi[3];
};

TRS_HD bool in_range_px(int h, int s, int v, const HsvRange& r)
{
    return (r.lo[0] <= h) & (h <= r.hi[0]) & (r.lo[1] <= s) & (s <= r.hi[1]) & (r.lo[2] <= v) & (v <= r.hi[2]);
}

// ---- Canny pieces (img_preprocessing.py:79, cv2.Canny 3-channel, aperture 3, L1) ----------------------
// Direction class of a gradient for the non-maximum suppression:
//   0 horizontal (compare left / right), 1 vertical (up / down),
//   2 diagonal with s = +1 (compare (y-1,x-1) and (y+1,x+1)), 3 diagonal with s = -1 ((y-1,x+1) and (y+1,x-1)).
TRS_HD int canny_dir(int dx, int dy)
{
    const int ax = dx < 0 ? -dx : dx;
    const int ay = (dy < 0 ? -dy : dy) << 15;
    const int tg22x = ax * 13573;
    if (ay < tg22x) return 0;
    const int tg67x = tg22x + (ax << 16);
    if (ay > tg67x) return 1;
    return ((dx ^ dy) < 0) ? 3 : 2;
}

// mag word stored in shared memory: bits 0..10 magnitude (<= 2040), bits 11..12 direction class.
TRS_HD uint16_t pack_mag(int mag, int dir) { return (uint16_t)(mag | (dir << 11)); }
TRS_HD int mag_of(uint16_t w) { return w & 0x7ff; }
TRS_HD int dir_of(uint16_t w) { return (w >> 11) & 3; }

// NMS decision given the centre magnitude m (> low already tested by the caller), its direction class and
// the 8 neighbouring magnitudes (zero outside the image): the comparisons are asymmetric on purpose.
TRS_HD bool canny_is_max(int m, int dir, int left, int right, int up, int down, int ul, int ur, int dl, int dr)
{
    switch (dir) {
    case 0: return (m > left) & (m >= right);
    case 1: return (m > up) & (m >= down);
    case 2: return (m > ul) & (m > dr);
    default: return (m > ur) & (m > dl);
    }
}

// ---- brightness / contrast table (img_preprocessing.py:81-102) -----------------------------------------
// One rounding per float32 operation, as numpy's in-place ops do; truncating cast.
TRS_HD uint8_t adjust_entry(int i, bool dynamic, float fdelta, float foff, float fratio)
{
#if defined(__CUDA_ARCH__)
    float v = (float)i;
    if (dynamic) v = __fadd_rn(v, fdelta);
    v = __fsub_rn(v, foff);
    v = __fmul_rn(v, fratio);
    v = __fadd_rn(v, foff);
#else
    volatile float v = (float)i;
    if (dynamic) v = v + fdelta;
    v = v - foff;
    v = v * fratio;
    v = v + foff;
#endif
    float c = v;
    c = c < 0.0f ? 0.0f : c;
    c = c > 255.0f ? 255.0f : c;
    return (uint8_t)(int)c;
}

// mean / delta of the dynamic-brightness statistic: sums are exact integers over rows 40..118.
TRS_HD double brightness_delta(unsigned long long s0, unsigned long long s1, unsigned long long s2, double npx, double baseline)
{
    const double m0 = npx > 0 ? (double)s0 / npx : 0.0;
    const double m1 = npx > 0 ? (double)s1 / npx : 0.0;
    const double m2 = npx > 0 ? (double)s2 / npx : 0.0;
    const double cur = ((m0 + m1) + m2) + 0.0;
    return (baseline - cur) / 3.0;
}

}  // namespace trs
