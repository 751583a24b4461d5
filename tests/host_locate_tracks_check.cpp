// Host build of the multi-track nearest-waypoint path (csrc/loc_grid.h: the per-track tables trs_set_tracks uploads, the bucketing rules and the
// slice / track selection of k_locate_tracks_grid) for the CPU-side tests (tests/test_locate_tracks_host.py).  Test infrastructure: restates the
// histogram / scan / scatter passes and the walk one car at a time, with the cars the walk puts off finished by the scan, as the kernels do.
#include "../triton-racer-sim_b200/csrc/loc_grid.h"
using namespace trs;

namespace {

const size_t SMEM_LIMIT = 227 * 1024 - 1024;        // sharedMemPerBlockOptin of a B200 less the margin trs_set_tracks keeps

std::vector<const double*> split(const double* wp_cat, const int* n_wp, int k)
{
    std::vector<const double*> wp((size_t)k);
    size_t off = 0;
    for (int t = 0; t < k; ++t) { wp[(size_t)t] = wp_cat + 3 * off; off += (size_t)n_wp[t]; }
    return wp;
}

double segment(int idx, int n_wp, double min_map, double max_map)
{
    volatile double q = (double)idx / (double)n_wp;
    return locg_add(locg_mul(q, locg_sub(max_map, min_map)), min_map);
}

}  // namespace

// wp_cat: the k centre lines one after the other (n_wp[t] x 3 f64 each).  info (k x 7): n_u, scan_off, grid_off, cell_off, cells (nx nz), nx,
// nz.  sizes: quads in the scan table, quads in the grid table, cell starts, the largest grid table in bytes.  scan (4 x sizes[0]) and grid
// (4 x sizes[1]) are written when not null.  Returns 0, or 1 when loct_build refuses.
extern "C" int tracks_build_host(const double* wp_cat, const int* n_wp, int k, const double* min_map, const double* max_map, long long* info,
                                 long long* sizes, double* scan, double* grid)
{
    LocTracksHost h;
    if (!loct_build(split(wp_cat, n_wp, k).data(), n_wp, min_map, max_map, k, SMEM_LIMIT, h)) return 1;
    for (int t = 0; t < k; ++t) {
        const LocTrack& d = h.desc[(size_t)t];
        long long* r = info + 7 * t;
        r[0] = d.n_u; r[1] = d.scan_off; r[2] = d.grid_off; r[3] = d.grid_off >= 0 ? d.cell_off : -1;
        r[4] = (long long)d.g.nx * d.g.nz; r[5] = d.g.nx; r[6] = d.g.nz;
    }
    sizes[0] = (long long)(h.scan.size() / 4); sizes[1] = (long long)(h.grid.size() / 4); sizes[2] = (long long)h.cells.size(); sizes[3] = (long long)h.smem;
    if (scan) std::copy(h.scan.begin(), h.scan.end(), scan);
    if (grid) std::copy(h.grid.begin(), h.grid.end(), grid);
    return 0;
}

// k_loct_hist + k_loct_scan + k_loct_scatter: perm (n) = car indices in bucket order, start (k + 2) = bucket starts and n.
extern "C" void tracks_bucket_host(const int32_t* trk, int n, int k, int max_blocks, int step, int* perm, int* start)
{
    int chunk = 0, nblk = 0;
    loct_chunking(n, max_blocks, step, chunk, nblk);
    std::vector<int> counts((size_t)(k + 1) * nblk, 0);
    for (int b = 0; b < nblk; ++b)
        for (int i = b * chunk; i < std::min(n, (b + 1) * chunk); ++i) ++counts[(size_t)loct_bucket(trk[i], k) * nblk + b];
    int run = 0;
    for (int& c : counts) { const int v = c; c = run; run += v; }
    for (int t = 0; t <= k; ++t) start[t] = counts[(size_t)t * nblk];
    start[k + 1] = n;
    for (int b = 0; b < nblk; ++b) {
        std::vector<int> base((size_t)k + 1);
        for (int t = 0; t <= k; ++t) base[(size_t)t] = counts[(size_t)t * nblk + b];
        for (int i = b * chunk; i < std::min(n, (b + 1) * chunk); ++i) perm[base[(size_t)loct_bucket(trk[i], k)]++] = i;
    }
}

// The whole large-batch path for n cars on k tracks with `ctas` CTAs in the walk.  idx / seg (n).  stats: [0] cars put off or on a track
// without a grid, [1] tracks with a grid, [2] cars with an in-range track.  Returns 0, or 1 when loct_build refuses.
extern "C" int locate_tracks_host(const double* wp_cat, const int* n_wp, int k, const double* min_map, const double* max_map, const double* xyz,
                                  const int32_t* trk, int n, int ctas, int32_t* idx, double* seg, long long* stats)
{
    LocTracksHost h;
    if (!loct_build(split(wp_cat, n_wp, k).data(), n_wp, min_map, max_map, k, SMEM_LIMIT, h)) return 1;
    std::vector<int> perm((size_t)n), start((size_t)k + 2);
    tracks_bucket_host(trk, n, k, 2 * ctas, 256, perm.data(), start.data());
    for (int p = start[(size_t)k]; p < n; ++p) { idx[perm[(size_t)p]] = -1; seg[perm[(size_t)p]] = std::nan(""); }
    std::vector<int> list;
    const int nv = start[(size_t)k];
    for (int b = 0; b < ctas; ++b) {
        int lo, hi;
        loct_slice(nv, b, ctas, lo, hi);
        while (lo < hi) {
            const int t = loct_track_of(start.data(), k, lo);
            const int end = std::min(hi, start[(size_t)t + 1]);
            const LocTrack& d = h.desc[(size_t)t];
            for (int p = lo; p < end; ++p) {
                const int car = perm[(size_t)p];
                const int r = d.grid_off < 0 ? LOCG_DEFERRED
                                             : locg_walk(d.g, h.grid.data() + 4 * (size_t)d.grid_off, h.cells.data() + d.cell_off, xyz[3 * (size_t)car],
                                                         xyz[3 * (size_t)car + 1], xyz[3 * (size_t)car + 2]);
                if (r == LOCG_DEFERRED) { list.push_back(car); continue; }
                idx[car] = r;
                seg[car] = segment(r, d.n_wp, d.min_map, d.max_map);
            }
            lo = end;
        }
    }
    for (int car : list) {                                  // k_locate_tracks_warp: the track's distinct points in order of first occurrence, strict `<`
        const LocTrack& d = h.desc[(size_t)trk[car]];
        const double* q = h.scan.data() + 4 * (size_t)d.scan_off;
        const double x = xyz[3 * (size_t)car], y = xyz[3 * (size_t)car + 1], z = xyz[3 * (size_t)car + 2];
        double best = 100.0;
        int r = 0;
        for (int i = 0; i < d.n_u; ++i) {
            const double dd = locg_add(locg_add(fabs(locg_sub(x, q[4 * i])), fabs(locg_sub(y, q[4 * i + 1]))), fabs(locg_sub(z, q[4 * i + 2])));
            if (dd < best) { best = dd; r = (int)q[4 * i + 3]; }
        }
        idx[car] = r;
        seg[car] = segment(r, d.n_wp, d.min_map, d.max_map);
    }
    if (stats) {
        stats[0] = (long long)list.size(); stats[2] = nv;
        stats[1] = 0;
        for (const LocTrack& d : h.desc) stats[1] += d.grid_off >= 0;
    }
    return 0;
}
