// preproc_list.h — which frames a launch of trs_preprocess_configs works on (host / device; the CPU-side tests build it with g++).
//
// The batch is bucketed by configuration with the histogram / scan / scatter passes of loc_tracks.cuh (k_loct_hist, k_loct_scan,
// k_loct_scatter over loc_grid.h's loct_bucket / loct_chunking): perm holds the frame indices in bucket order, a stable sort by the
// frame's configuration index, with every index outside [0, K) in bucket K; start[b] is the first position of bucket b, start[K + 1] = n.
// The launch for configuration c walks positions 0 .. count of its slice and processes frame list[j] at the frame's own position in the
// input and the outputs.  The slice is read from device memory, so the host never learns the group sizes.
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define PLIST_HD __host__ __device__ __forceinline__
#else
#define PLIST_HD inline
#endif

namespace trs {

struct FrameList {
    const int* perm;        // frames in bucket order (n)
    const int* start;       // bucket starts (K + 2)
    int cfg;                // the bucket of this launch: a configuration, or K for the frames with an index outside [0, K)
};

// the slice of bucket fl.cfg: frames list[0 .. n)
PLIST_HD void plist_open(const FrameList& fl, const int*& list, int& n)
{
    const int lo = fl.start[fl.cfg];
    n = fl.start[fl.cfg + 1] - lo;
    list = fl.perm + lo;
}

// the frame at position j of the launch: list[j] in list mode, j itself otherwise
template <bool LIST, class T>
PLIST_HD T plist_frame(const int* list, T j)
{
    if constexpr (LIST) return (T)list[j];
    else return j;
}

}  // namespace trs
