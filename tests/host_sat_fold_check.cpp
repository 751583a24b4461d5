// Host build of the folded saturation / value threshold entries (csrc/pixel_math.cuh sat_threshold_entry_folded, the function init_tables calls for
// the default-range kernels) for the CPU-side exhaustive check in tests/test_sat_fold_host.py.  Test infrastructure.
#include "../triton-racer-sim_b200/csrc/pixel_math.cuh"
using namespace trs;

// Number of (v, d) pairs, d <= v, for which the kernel's compare against the folded entry disagrees with "the saturation bound holds and
// vlo <= v <= vhi".  K as sat_threshold_entry takes it: upper bound "s <= K" (compare d <= T), lower bound "s >= K + 1" (compare d > T).
extern "C" long long fold_check(long long K, int upper, long long vlo, long long vhi)
{
    long long bad = 0;
    for (int v = 0; v < 256; ++v) {
        const int sd = hsv_sdiv_entry(v);
        const uint32_t T = sat_threshold_entry_folded(K, upper != 0, v, sd, vlo, vhi);
        const int t = T == 0x8001u ? -1 : (int)T;                       // the packed compare reads 0x8001 as -1
        const bool v_in = vlo <= v && v <= vhi;
        for (int d = 0; d <= v; ++d) {
            const int s = (d * sd + 2048) >> 12;
            const bool want = (upper ? s <= K : s > K) && v_in;
            const bool got = upper ? d <= t : d > t;
            bad += want != got;
        }
    }
    return bad;
}

// every value bound from -1 to 256 on either side (the other side open) against the saturation bounds in ks[0..nk), both directions
extern "C" long long fold_check_all_value_bounds(const long long* ks, int nk)
{
    long long bad = 0;
    for (int i = 0; i < nk; ++i)
        for (int upper = 0; upper < 2; ++upper)
            for (long long b = -1; b <= 256; ++b) {
                bad += fold_check(ks[i], upper, b, 255);
                bad += fold_check(ks[i], upper, 0, b);
            }
    return bad;
}
