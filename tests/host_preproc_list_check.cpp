// Host build of the frame bucketing of trs_preprocess_configs (csrc/loc_grid.h: loct_bucket / loct_chunking; csrc/preproc_list.h: the
// slice of every bucket and the frame at each position) for tests/test_preproc_configs_host.py, built with the address and UB sanitizers.
// Test infrastructure: restates the histogram / scan / scatter passes of k_loct_hist / k_loct_scan / k_loct_scatter block by block.
//   usage: host_preproc_list_check <in> <out>
//   in:  int32 n, k, max_blocks, then n int32 configuration indices
//   out: for every bucket b = 0 .. k (k: indices outside [0, k)): int32 count, then the frames of the bucket in launch order
#include <stdio.h>
#include <stdlib.h>

#include <vector>

#include "../triton-racer-sim_b200/csrc/loc_grid.h"
#include "../triton-racer-sim_b200/csrc/preproc_list.h"
using namespace trs;

int main(int argc, char** argv)
{
    if (argc != 3) return 2;
    FILE* fi = fopen(argv[1], "rb");
    if (!fi) return 2;
    int32_t hdr[3];
    if (fread(hdr, sizeof(int32_t), 3, fi) != 3) return 2;
    const int n = hdr[0], k = hdr[1], max_blocks = hdr[2];
    std::vector<int32_t> cfg((size_t)n);
    if (n && fread(cfg.data(), sizeof(int32_t), (size_t)n, fi) != (size_t)n) return 2;
    fclose(fi);

    int chunk = 0, nblk = 0;
    loct_chunking(n, max_blocks, 256, chunk, nblk);
    std::vector<int> counts((size_t)(k + 1) * nblk, 0), start((size_t)k + 2), perm((size_t)n, -1);
    for (int b = 0; b < nblk; ++b)
        for (int i = b * chunk; i < std::min(n, (b + 1) * chunk); ++i) ++counts.at((size_t)loct_bucket(cfg[(size_t)i], k) * nblk + b);
    int run = 0;
    for (int& c : counts) { const int v = c; c = run; run += v; }
    for (int t = 0; t <= k; ++t) start.at((size_t)t) = nblk ? counts.at((size_t)t * nblk) : 0;
    start.at((size_t)k + 1) = n;
    for (int b = 0; b < nblk; ++b) {
        std::vector<int> base((size_t)k + 1);
        for (int t = 0; t <= k; ++t) base.at((size_t)t) = counts.at((size_t)t * nblk + b);
        for (int i = b * chunk; i < std::min(n, (b + 1) * chunk); ++i) perm.at((size_t)base.at((size_t)loct_bucket(cfg[(size_t)i], k))++) = i;
    }

    FILE* fo = fopen(argv[2], "wb");
    if (!fo) return 2;
    for (int c = 0; c <= k; ++c) {
        const FrameList fl{perm.data(), start.data(), c};
        const int* list = nullptr;
        int cnt = 0;
        plist_open(fl, list, cnt);
        fwrite(&cnt, sizeof cnt, 1, fo);
        for (int j = 0; j < cnt; ++j) {
            const int f = plist_frame<true>(list, j);
            if (plist_frame<false>(list, j) != j || f < 0 || f >= n) return 3;
            fwrite(&f, sizeof f, 1, fo);
        }
    }
    fclose(fo);
    return 0;
}
