// loc_grid.h — nearest waypoint through a uniform grid (track_data_process.py:89-107: L1 distance in float64, first index wins ties, the running
// minimum starts at 100).  Pure host / device functions: k_locate_grid (misc_kernels.cuh) runs locg_walk per car, trs_set_track (trs_api.cu)
// builds the table with locg_build, and tests/host_locate_check.cpp compiles the same source with g++ for the CPU-side parity test.
//
// The distinct points are bucketed into square cells of side c over (x, z).  c is a power of two, so floor(x / c) is exact and a point's and a
// car's cell are decided by the same exact rule.  The points are sorted by cell (row-major, rows along z) behind a prefix array of cell starts.
// A car looks at the 3 x 3 cells around its own, then at rings of growing Chebyshev radius.  Every point in a ring beyond r is at least
// r c + m away in L1 (m = the car's distance to the nearest edge of its own cell), and so is its COMPUTED distance: the bound is representable
// or shrunk below the exact value, rounding is monotone, and the three terms are summed in the reference's order.  The walk stops as soon as the
// best distance so far is strictly below that bound (at equality a tie with a smaller index could still hide out there) or the bound reaches
// 100.  Inside the visited set the argmin is taken on the pair (distance, original index), which is the reference's first-index rule, and every
// evaluated distance is the same three subtractions and two additions as in the scanning kernels: the reference's result bit for bit.
#pragma once
#include <math.h>
#include <stdint.h>

#include <algorithm>
#include <cmath>
#include <utility>
#include <vector>

#if defined(__CUDACC__)
#define LOCG_HD __host__ __device__ __forceinline__
#else
#define LOCG_HD inline
#endif

namespace trs {

enum { LOCG_MAX_RINGS = 6,            // rings after the 3 x 3 block before a car is put off to the warp-per-car scan
       LOCG_MIN_POINTS = 64,          // fewer distinct points: no grid
       LOCG_TARGET_CELLS = 32,        // cells along the longer side of the bounding box (side 4 for the shipped centre lines)
       LOCG_DEFERRED = -1 };

struct LocGrid {
    double c, inv_c;                   // cell side (2^k) and its reciprocal
    double ox, oz;                     // floor(min x / c), floor(min z / c) as doubles (exact integers)
    double x0, x1, y0, y1, z0, z1;     // bounding box of the points
    int nx, nz;                        // cells along x and z
    int n_u;                           // points
};

// one rounding per operation on either side (the device build also runs with -fmad=false; g++ on x86-64 does not contract without -mfma)
#if defined(__CUDA_ARCH__)
LOCG_HD double locg_add(double a, double b) { return __dadd_rn(a, b); }
LOCG_HD double locg_sub(double a, double b) { return __dsub_rn(a, b); }
LOCG_HD double locg_mul(double a, double b) { return __dmul_rn(a, b); }
#else
LOCG_HD double locg_add(double a, double b) { volatile double r = a + b; return r; }
LOCG_HD double locg_sub(double a, double b) { volatile double r = a - b; return r; }
LOCG_HD double locg_mul(double a, double b) { volatile double r = a * b; return r; }
#endif
// max / min that drop a NaN operand like CUDA's fmax / fmin (and C's)
LOCG_HD double locg_max(double a, double b) { return fmax(a, b); }
LOCG_HD double locg_min(double a, double b) { return fmin(a, b); }

// Points [a, b) of the table against one car.  A quad is (x, z, y, original index): the first 16 bytes give |dx| + |dz|, which can only be smaller
// than the distance (rounding is monotone and |dy| >= 0), so a point that already loses on it is dropped before its second half is read.
LOCG_HD void locg_eval(const double* q, int a, int b, double x, double y, double z, double& best, int& sel)
{
    for (int k = a; k < b; ++k) {
#if defined(__CUDA_ARCH__)
        const double2 xz = reinterpret_cast<const double2*>(q + 4 * k)[0];
        const double qx = xz.x, qz = xz.y;
#else
        const double qx = q[4 * k], qz = q[4 * k + 1];
#endif
        const double ax = fabs(locg_sub(x, qx)), az = fabs(locg_sub(z, qz));
        if (locg_add(ax, az) > best) continue;
#if defined(__CUDA_ARCH__)
        const double2 yi = reinterpret_cast<const double2*>(q + 4 * k)[1];
        const double qy = yi.x, qw = yi.y;
#else
        const double qy = q[4 * k + 2], qw = q[4 * k + 3];
#endif
        const double d = locg_add(locg_add(ax, fabs(locg_sub(y, qy))), az);      // (|dx| + |dy|) + |dz|, as the reference sums it
        const int qi = (int)qw;
        // (a distance of exactly 100 never wins: the reference's minimum starts there and its test is strict)
        if (d < best || (d == best && qi < sel && best < 100.0)) { best = d; sel = qi; }
    }
}

// The reference's index for one car, or LOCG_DEFERRED if the car has not settled after the 3 x 3 block and LOCG_MAX_RINGS rings (far from the
// line but inside the bounding box: the caller scans the table for it).  q: quads in cell order, cs: cell starts (nx nz + 1 entries).
LOCG_HD int locg_walk(const LocGrid& G, const double* q, const int* cs, double x, double y, double z)
{
    double best = 100.0;                                         // track_data_process.py:93
    int sel = 0x7fffffff;
    // L1 distance to the points' bounding box, summed like a distance: nothing can be closer than that
    const double bx = locg_max(locg_max(locg_sub(G.x0, x), locg_sub(x, G.x1)), 0.0), by = locg_max(locg_max(locg_sub(G.y0, y), locg_sub(y, G.y1)), 0.0),
                 bz = locg_max(locg_max(locg_sub(G.z0, z), locg_sub(z, G.z1)), 0.0);
    if (!(locg_add(locg_add(bx, by), bz) < 100.0)) return 0;     // (an infinite coordinate ends here; a NaN one fails every `<` below: index 0 either way)
    const int nx = G.nx, nz = G.nz;
    const double fx = floor(locg_mul(x, G.inv_c)), fz = floor(locg_mul(z, G.inv_c));
    const double lim = 536870912.0;                              // (2^29: cx +- r stays inside int for every ring up to r_end)
    const int cx = (int)locg_min(locg_max(locg_sub(fx, G.ox), -lim), lim), cz = (int)locg_min(locg_max(locg_sub(fz, G.oz), -lim), lim);
    // distance to the nearest edge of the car's own cell, shrunk so that rounding can only make the bound smaller
    const double ex = locg_mul(fx, G.c), ez = locg_mul(fz, G.c);
    double m = locg_min(locg_min(locg_sub(x, ex), locg_sub(locg_add(ex, G.c), x)), locg_min(locg_sub(z, ez), locg_sub(locg_add(ez, G.c), z)));
    m = locg_max(locg_mul(m, 0.999), 0.0);
    const int cxm = cx < 0 ? -cx : 0, czm = cz < 0 ? -cz : 0;
    int r_out = cxm > cx - (nx - 1) ? cxm : cx - (nx - 1);       // rings nearer than this lie outside the grid
    const int r_oz = czm > cz - (nz - 1) ? czm : cz - (nz - 1);
    r_out = r_out > r_oz ? r_out : r_oz;
    const int r_ex = cx > nx - 1 - cx ? cx : nx - 1 - cx, r_ez = cz > nz - 1 - cz ? cz : nz - 1 - cz;
    const int r_end = r_ex > r_ez ? r_ex : r_ez;                 // the last ring that touches the grid
    // rings 0 and 1 together, row by row (three contiguous point ranges): with cells this size that settles nearly every car on the line, and a warp
    // runs three long loops instead of five short ones
    if (r_out <= 1) {
        const int i0 = cx - 1 > 0 ? cx - 1 : 0, i1 = cx + 1 < nx - 1 ? cx + 1 : nx - 1;
        const int j0 = cz - 1 > 0 ? cz - 1 : 0, j1 = cz + 1 < nz - 1 ? cz + 1 : nz - 1;
        if (i0 <= i1)
            for (int j = j0; j <= j1; ++j) locg_eval(q, cs[j * nx + i0], cs[j * nx + i1 + 1], x, y, z, best, sel);
        const double bound = locg_add(G.c, m);                   // every point in a ring beyond 1 is at least this far
        if (best < bound || bound >= 100.0) return sel == 0x7fffffff ? 0 : sel;
    }
    int r = r_out > 2 ? r_out : 2, rings = 0;
    while (r <= r_end) {
        const int i0 = cx - r > 0 ? cx - r : 0, i1 = cx + r < nx - 1 ? cx + r : nx - 1;
        if (i0 <= i1) {                                          // the ring's two full rows of cells: contiguous point ranges
            const int jt = cz - r, jb = cz + r;
            if (jt >= 0 && jt < nz) locg_eval(q, cs[jt * nx + i0], cs[jt * nx + i1 + 1], x, y, z, best, sel);
            if (jb >= 0 && jb < nz) locg_eval(q, cs[jb * nx + i0], cs[jb * nx + i1 + 1], x, y, z, best, sel);
        }
        const int j0 = cz - r + 1 > 0 ? cz - r + 1 : 0, j1 = cz + r - 1 < nz - 1 ? cz + r - 1 : nz - 1;
        for (int j = j0; j <= j1; ++j) {                         // ... and the two cells at its sides in every row between
            const int il = cx - r, ir = cx + r;
            if (il >= 0 && il < nx) locg_eval(q, cs[j * nx + il], cs[j * nx + il + 1], x, y, z, best, sel);
            if (ir >= 0 && ir < nx) locg_eval(q, cs[j * nx + ir], cs[j * nx + ir + 1], x, y, z, best, sel);
        }
        const double bound = locg_add(locg_mul((double)r, G.c), m);      // every point in a ring beyond r is at least this far
        ++r;
        if (best < bound || bound >= 100.0) break;
        if (++rings >= LOCG_MAX_RINGS && r <= r_end) return LOCG_DEFERRED;
    }
    return sel == 0x7fffffff ? 0 : sel;
}

// Host: the table for locg_walk from the distinct points (x, y, z, original index quads in order of first occurrence).  Returns false (no grid:
// the scanning kernels serve every batch) for non-finite coordinates, fewer than LOCG_MIN_POINTS points, or a table beyond `smem_limit` bytes.
// sorted: (x, z, y, original index) quads in cell order; start: nx nz + 1 cell starts.
inline bool locg_build(const std::vector<double>& quads, size_t smem_limit, LocGrid& g, std::vector<double>& sorted, std::vector<int>& start)
{
    const int nu = (int)(quads.size() / 4);
    if (nu < LOCG_MIN_POINTS) return false;
    for (double v : quads)
        if (!std::isfinite(v)) return false;
    g = LocGrid{};
    g.x0 = g.x1 = quads[0]; g.y0 = g.y1 = quads[1]; g.z0 = g.z1 = quads[2];
    for (int i = 0; i < nu; ++i) {
        g.x0 = std::min(g.x0, quads[4 * i]); g.x1 = std::max(g.x1, quads[4 * i]);
        g.y0 = std::min(g.y0, quads[4 * i + 1]); g.y1 = std::max(g.y1, quads[4 * i + 1]);
        g.z0 = std::min(g.z0, quads[4 * i + 2]); g.z1 = std::max(g.z1, quads[4 * i + 2]);
    }
    const double ext = std::max(g.x1 - g.x0, g.z1 - g.z0);
    int k = ext > 0 ? (int)std::ceil(std::log2(ext / (double)LOCG_TARGET_CELLS)) : 0;
    k = std::max(-60, std::min(60, k));
    g.c = std::ldexp(1.0, k); g.inv_c = std::ldexp(1.0, -k);
    g.ox = std::floor(g.x0 * g.inv_c); g.oz = std::floor(g.z0 * g.inv_c);
    const double dnx = std::floor(g.x1 * g.inv_c) - g.ox + 1, dnz = std::floor(g.z1 * g.inv_c) - g.oz + 1;
    if (!(dnx >= 1 && dnz >= 1 && dnx <= 80 && dnz <= 80 && std::fabs(g.ox) < 1e9 && std::fabs(g.oz) < 1e9)) return false;
    if (sizeof(double) * 4 * (size_t)nu + sizeof(int) * ((size_t)(dnx * dnz) + 1) > smem_limit) return false;
    g.nx = (int)dnx; g.nz = (int)dnz; g.n_u = nu;
    const int ncell = g.nx * g.nz;
    std::vector<int> cell((size_t)nu), order((size_t)nu);
    start.assign((size_t)ncell + 1, 0);
    for (int i = 0; i < nu; ++i) {
        const int ci = (int)(std::floor(quads[4 * i] * g.inv_c) - g.ox), cj = (int)(std::floor(quads[4 * i + 2] * g.inv_c) - g.oz);
        cell[i] = cj * g.nx + ci;
        ++start[(size_t)cell[i] + 1];
    }
    for (int c = 0; c < ncell; ++c) start[(size_t)c + 1] += start[c];
    std::vector<int> fill(start.begin(), start.end() - 1);
    for (int i = 0; i < nu; ++i) order[(size_t)fill[cell[i]]++] = i;
    sorted.resize(4 * (size_t)nu);
    for (int t = 0; t < nu; ++t) {
        const double* p = &quads[4 * (size_t)order[t]];
        sorted[4 * (size_t)t] = p[0]; sorted[4 * (size_t)t + 1] = p[2]; sorted[4 * (size_t)t + 2] = p[1]; sorted[4 * (size_t)t + 3] = p[3];
    }
    return true;
}

inline size_t locg_table_bytes(const LocGrid& g) { return sizeof(double) * 4 * (size_t)g.n_u + sizeof(int) * ((size_t)g.nx * g.nz + 1); }

// Host: first occurrences of the points of a centre line as (x, y, z, original index) quads (compared by value: -0.0 == 0.0, a NaN is never a repeat).
// A repeated point can never beat its first occurrence under the reference's strict `<` (track_data_process.py:95).
inline std::vector<double> locg_distinct_quads(const double* wp, int n_wp)
{
    std::vector<double> quads;
    quads.reserve(4 * (size_t)n_wp);
    struct Key { double x, y, z; };
    auto norm = [](double v) { return v == 0.0 ? 0.0 : v; };
    std::vector<std::pair<Key, int>> seen;                            // sorted by (x, y, z) among comparable values
    seen.reserve((size_t)n_wp);
    auto less = [](const Key& a, const Key& b) { return a.x != b.x ? a.x < b.x : (a.y != b.y ? a.y < b.y : a.z < b.z); };
    for (int i = 0; i < n_wp; ++i) {
        const Key k{norm(wp[3 * i]), norm(wp[3 * i + 1]), norm(wp[3 * i + 2])};
        bool repeat = false;
        if (k.x == k.x && k.y == k.y && k.z == k.z) {                  // (points with a NaN are always kept)
            auto it = std::lower_bound(seen.begin(), seen.end(), k, [&](const std::pair<Key, int>& a, const Key& b) { return less(a.first, b); });
            repeat = it != seen.end() && it->first.x == k.x && it->first.y == k.y && it->first.z == k.z;
            if (!repeat) seen.insert(it, std::make_pair(k, i));
        }
        if (!repeat) { quads.push_back(wp[3 * i]); quads.push_back(wp[3 * i + 1]); quads.push_back(wp[3 * i + 2]); quads.push_back((double)i); }
    }
    return quads;
}

// ---- several centre lines in one batch (trs_set_tracks / trs_locate_tracks, loc_tracks.cuh) ------------------------------------------------------
// Every track keeps what trs_set_track builds for one: its distinct quads in order of first occurrence (the scan table) and, when locg_build gives
// one, its cell-sorted quads and cell starts (the grid table).  The tracks' tables are concatenated; a descriptor per track holds the offsets.
// Car i names its track t_i; the cars are bucketed by track (a stable counting sort) and each CTA of the walk takes a contiguous slice of the
// bucketed cars, staging a track's grid table whenever its slice moves on to another track.
struct LocTrack {
    LocGrid g;                         // valid when grid_off >= 0
    double min_map, max_map;
    int n_wp;                          // points of the centre line (the divisor of the segment map)
    int n_u;                           // distinct points
    int scan_off;                      // first quad of its distinct points in the scan table
    int grid_off;                      // first quad of its cell-sorted points in the grid table; -1: no grid (every car goes to the scan)
    int cell_off;                      // first entry of its cell starts in the cell table
    int pad_;
};

struct LocTracksHost {
    std::vector<LocTrack> desc;
    std::vector<double> scan, grid;    // quads
    std::vector<int> cells;
    size_t smem = 0;                   // the largest grid table in bytes (the walk's dynamic shared memory)
};

// Host: the tables of `k` centre lines (wp[t]: n_wp[t] x 3 f64).  A track whose grid would not fit `smem_limit` bytes, has non-finite
// coordinates or fewer than LOCG_MIN_POINTS distinct points gets grid_off = -1.  Returns false when the concatenated tables would not be
// addressable with int offsets.
inline bool loct_build(const double* const* wp, const int* n_wp, const double* min_map, const double* max_map, int k, size_t smem_limit,
                       LocTracksHost& out)
{
    out = LocTracksHost{};
    out.desc.resize((size_t)k);
    for (int t = 0; t < k; ++t) {
        LocTrack& d = out.desc[(size_t)t];
        d = LocTrack{};
        const std::vector<double> quads = locg_distinct_quads(wp[t], n_wp[t]);
        d.min_map = min_map[t]; d.max_map = max_map[t];
        d.n_wp = n_wp[t]; d.n_u = (int)(quads.size() / 4);
        if (out.scan.size() / 4 + quads.size() / 4 > (size_t)0x1fffffff) return false;
        d.scan_off = (int)(out.scan.size() / 4);
        out.scan.insert(out.scan.end(), quads.begin(), quads.end());
        std::vector<double> sorted;
        std::vector<int> start;
        d.grid_off = -1;
        if (locg_build(quads, smem_limit, d.g, sorted, start)) {
            d.grid_off = (int)(out.grid.size() / 4);
            d.cell_off = (int)out.cells.size();
            out.grid.insert(out.grid.end(), sorted.begin(), sorted.end());
            out.cells.insert(out.cells.end(), start.begin(), start.end());
            out.smem = std::max(out.smem, locg_table_bytes(d.g));
        } else {
            d.g = LocGrid{};
        }
    }
    return true;
}

// Bucket of a car's track index: t itself, or k for an index outside [0, k) (those cars get idx -1 / segment NaN and are not walked).
LOCG_HD int loct_bucket(int32_t t, int k) { return (uint32_t)t < (uint32_t)k ? (int)t : k; }

// Cars [b chunk, (b + 1) chunk) go to block b of the histogram and scatter passes: chunk a multiple of `step`, at most `max_blocks` blocks.
LOCG_HD void loct_chunking(int n, int max_blocks, int step, int& chunk, int& nblk)
{
    const long long per = ((long long)n + max_blocks - 1) / max_blocks;
    chunk = (int)((per + step - 1) / step * step);
    if (chunk < step) chunk = step;
    nblk = (int)(((long long)n + chunk - 1) / chunk);
}

// Positions [lo, hi) of the bucketed cars for CTA b of g, out of nv in-range cars.
LOCG_HD void loct_slice(int nv, int b, int g, int& lo, int& hi)
{
    lo = (int)((long long)nv * b / g);
    hi = (int)((long long)nv * (b + 1) / g);
}

// The track of bucketed position p < start[k]: the largest t < k with start[t] <= p (start: k + 1 bucket starts, ascending).
LOCG_HD int loct_track_of(const int* start, int k, int p)
{
    int a = 0, b = k - 1;
    while (a < b) {
        const int m = (a + b + 1) >> 1;
        if (start[m] <= p) a = m; else b = m - 1;
    }
    return a;
}

}  // namespace trs
