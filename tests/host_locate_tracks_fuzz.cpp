// Sanitizer fuzz of the multi-track path (csrc/loc_grid.h through host_locate_tracks_check.cpp) against the reference's loop per track: 200 random
// batches of 1-9 centre lines (circles, flat and vertical lines, heavy repeats, lines too short for a grid, a NaN point; scales 1e-4 .. 1e4, shifts
// up to 1e7) x 600 cars each (near, far, NaN, infinite, huge; track indices in order, shuffled, and out of range), walked by 1-13 CTAs, built with
// -fsanitize=address,undefined: every index and segment must match and no offset, cell or bucket index may leave its array.
// (tests/test_locate_tracks_host.py)
#include <stdio.h>
#include <string.h>
#include <random>
#include <vector>
#include "host_locate_tracks_check.cpp"
int main()
{
    std::mt19937_64 rng(11);
    std::uniform_real_distribution<double> U(0, 1);
    long total = 0;
    for (int trial = 0; trial < 200; ++trial) {
        const int k = 1 + (int)(rng() % 9);
        std::vector<int> n_wp((size_t)k);
        std::vector<double> wp, mn((size_t)k), mx((size_t)k);
        for (int t = 0; t < k; ++t) {
            const int nw = rng() % 7 == 0 ? 5 + (int)(rng() % 50) : 64 + (int)(rng() % 400);
            n_wp[(size_t)t] = nw;
            mn[(size_t)t] = (double)(rng() % 5) - 2.5; mx[(size_t)t] = mn[(size_t)t] + 1 + (double)(rng() % 20);
            const double scale = std::pow(10.0, (int)(rng() % 9) - 4), shift = (U(rng) - 0.5) * std::pow(10.0, (int)(rng() % 8));
            const int shape = (int)(rng() % 4);
            for (int i = 0; i < nw; ++i) {
                const double a = 6.283185307 * i / nw;
                double x = std::cos(a) * 40, z = std::sin(a) * (shape == 1 ? 0.0 : 30), y = 0.5 + 0.01 * U(rng);
                if (shape == 2) { x = 0; }
                if (shape == 3) { x = (double)(rng() % 5); z = (double)(rng() % 5); }
                wp.push_back(x * scale + shift); wp.push_back(y); wp.push_back(z * scale - shift);
            }
            if (rng() % 11 == 0) wp[wp.size() - 3 * (size_t)(1 + rng() % nw) + 1] = std::nan("");
        }
        std::vector<size_t> off((size_t)k + 1, 0);
        for (int t = 0; t < k; ++t) off[(size_t)t + 1] = off[(size_t)t] + (size_t)n_wp[(size_t)t];
        const int n = 600;
        std::vector<double> xyz(3 * (size_t)n);
        std::vector<int32_t> trk((size_t)n);
        const int order = (int)(rng() % 3);
        for (int c = 0; c < n; ++c) {
            int t = order == 0 ? (int)((long)c * k / n) : (int)(rng() % k);
            if (order == 2 && rng() % 17 == 0) t = rng() % 2 ? -1 - (int)(rng() % 3) : k + (int)(rng() % 3);
            trk[(size_t)c] = t;
            const int tt = t < 0 || t >= k ? 0 : t;
            const double* w = &wp[3 * (off[(size_t)tt] + rng() % (size_t)n_wp[(size_t)tt])];
            const double spread = std::pow(10.0, (int)(rng() % 7) - 3) * 100;
            xyz[3 * c] = w[0] + (U(rng) - 0.5) * spread; xyz[3 * c + 1] = w[1] + (U(rng) - 0.5) * 3; xyz[3 * c + 2] = w[2] + (U(rng) - 0.5) * spread;
            if (c % 97 == 0) xyz[3 * c] = std::nan("");
            if (c % 89 == 0) xyz[3 * c + 2] = (c & 1) ? INFINITY : -INFINITY;
            if (c % 83 == 0) xyz[3 * c] = 1e308;
        }
        std::vector<int32_t> idx((size_t)n);
        std::vector<double> seg((size_t)n);
        long long stats[3];
        const int ctas = 1 + (int)(rng() % 13);
        if (locate_tracks_host(wp.data(), n_wp.data(), k, mn.data(), mx.data(), xyz.data(), trk.data(), n, ctas, idx.data(), seg.data(), stats)) {
            printf("loct_build refused trial %d\n", trial);
            return 1;
        }
        for (int c = 0; c < n; ++c) {
            const int t = trk[(size_t)c];
            if (t < 0 || t >= k) {
                if (idx[(size_t)c] != -1 || seg[(size_t)c] == seg[(size_t)c]) { printf("MISMATCH trial %d car %d: out-of-range track %d\n", trial, c, t); return 1; }
                continue;
            }
            double best = 100.0; int r = 0;                  // the reference's loop over the whole centre line
            for (int i = 0; i < n_wp[(size_t)t]; ++i) {
                const double* w = &wp[3 * (off[(size_t)t] + (size_t)i)];
                const double d = (std::fabs(xyz[3 * c] - w[0]) + std::fabs(xyz[3 * c + 1] - w[1])) + std::fabs(xyz[3 * c + 2] - w[2]);
                if (d < best) { best = d; r = i; }
            }
            const double s = (double)r / n_wp[(size_t)t] * (mx[(size_t)t] - mn[(size_t)t]) + mn[(size_t)t];
            if (r != idx[(size_t)c] || memcmp(&s, &seg[(size_t)c], sizeof s) != 0) {
                printf("MISMATCH trial %d car %d track %d: %d vs %d\n", trial, c, t, idx[(size_t)c], r);
                return 1;
            }
        }
        total += n;
    }
    printf("ok %ld cars\n", total);
    return 0;
}
