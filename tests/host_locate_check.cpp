// Host build of the product's nearest-waypoint grid walk (csrc/loc_grid.h: the same source k_locate_grid and trs_set_track / trs_set_tracks
// compile) for the CPU-side parity test against the oracle (tests/test_host_logic.py).  Test infrastructure: mirrors one track's table (the
// distinct points and the grid loct_build makes of them for every track) + the walk + the warp-per-car scan that finishes the cars the walk
// puts off, one car at a time; tests/host_locate_tracks_check.cpp runs the same walk over several tracks.
#include "../triton-racer-sim_b200/csrc/loc_grid.h"
using namespace trs;

// wp (n_wp, 3) f64, xyz (n, 3) f64 -> idx (n) i32.  stats: [0] 1 if a grid was built, [1] cells along x, [2] along z, [3] cars put off,
// [4] distinct points, [5] log2 of the cell side.  Returns 0.
extern "C" int locate_grid_host(const double* wp, int n_wp, const double* xyz, int n, int32_t* idx, long long* stats)
{
    const std::vector<double> quads = locg_distinct_quads(wp, n_wp);
    const int nu = (int)(quads.size() / 4);
    LocGrid g{};
    std::vector<double> sorted;
    std::vector<int> start;
    const bool have = locg_build(quads, 227 * 1024, g, sorted, start);
    long long deferred = 0;
    for (int k = 0; k < n; ++k) {
        const double x = xyz[3 * k], y = xyz[3 * k + 1], z = xyz[3 * k + 2];
        int r = have ? locg_walk(g, sorted.data(), start.data(), x, y, z) : LOCG_DEFERRED;
        if (r == LOCG_DEFERRED) {                               // the scan: distinct points in order of first occurrence, strict `<`
            ++deferred;
            double best = 100.0;
            r = 0;
            for (int i = 0; i < nu; ++i) {
                const double d = locg_add(locg_add(fabs(locg_sub(x, quads[4 * i])), fabs(locg_sub(y, quads[4 * i + 1]))), fabs(locg_sub(z, quads[4 * i + 2])));
                if (d < best) { best = d; r = (int)quads[4 * i + 3]; }
            }
        }
        idx[k] = r;
    }
    if (stats) {
        stats[0] = have; stats[1] = g.nx; stats[2] = g.nz; stats[3] = have ? deferred : 0; stats[4] = nu;
        stats[5] = have ? (long long)std::lround(std::log2(g.c)) : 0;
    }
    return 0;
}
