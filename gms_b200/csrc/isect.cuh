// isect.cuh — warp-cooperative sorted-list intersection primitives (device side of SortedSet::intersect*).
//
//   vec_set_intersect_count     gms/representations/sets/sorted_set_operations.h:45-71
//   vec_set_intersect           gms/representations/sets/sorted_set_operations.h:37-42
//
// Two strategies, both for ascending duplicate-free int32 ranges and both called by a full warp:
//   warp_gallop_*  — lanes take elements of the shorter list and binary-search the longer one;
//                    O(min * log max), right for skewed pairs.
//   warp_merge_count — merge path: the merged sequence is cut into tiles, each tile's slices of A and B are
//                    staged in shared memory with coalesced loads and every lane walks an equal share of the
//                    tile's diagonal; O((|A|+|B|)/32) steps per lane, right for balanced pairs.
// warp_intersect_count picks one of the two by the length ratio (kGallopRatio).
#pragma once
#include "common.cuh"

namespace gmsb {

constexpr int kMergeTile = 512;     // merged elements per staged tile (per warp: (kMergeTile+2)*4 bytes)

__device__ __forceinline__ int lower_bound_dev(const vid_t *__restrict__ b, int nb, vid_t x) {
    int lo = 0, hi = nb;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (b[mid] < x) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// per-lane partial count; caller reduces
__device__ __forceinline__ uint32_t warp_gallop_count(const vid_t *__restrict__ a, int na, const vid_t *__restrict__ b,
                                                      int nb, int lane) {
    if (na > nb) { const vid_t *t = a; a = b; b = t; int tn = na; na = nb; nb = tn; }
    uint32_t hits = 0;
    for (int j = lane; j < na; j += 32) {
        const vid_t x = a[j];
        int lo = lower_bound_dev(b, nb, x);
        hits += (lo < nb && b[lo] == x);
    }
    return hits;
}

// number of A elements among the first d elements of merge(A,B) with A winning ties
__device__ __forceinline__ int diag_split(const vid_t *a, int na, const vid_t *b, int nb, int d) {
    int lo = d > nb ? d - nb : 0, hi = d < na ? d : na;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (a[mid] <= b[d - 1 - mid]) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// per-lane partial count; `buf` is this warp's shared staging area of kMergeTile + 2 ints
__device__ __forceinline__ uint32_t warp_merge_count(const vid_t *__restrict__ a, int na, const vid_t *__restrict__ b,
                                                     int nb, int lane, vid_t *buf) {
    uint32_t hits = 0;
    const int T = na + nb;
    if (na == 0 || nb == 0) return 0;
    for (int t0 = 0; t0 < T; t0 += kMergeTile) {
        const int t1 = min(t0 + kMergeTile, T);
        const int a0 = diag_split(a, na, b, nb, t0), a1 = diag_split(a, na, b, nb, t1);
        const int b0 = t0 - a0, b1 = t1 - a1;
        const int ta = a1 - a0, tb = b1 - b0;
        __syncwarp();
        // buf[0] = predecessor of the A slice (or -1, which equals no vertex id)
        if (lane == 0) buf[0] = a0 > 0 ? a[a0 - 1] : -1;
        for (int j = lane; j < ta; j += 32) buf[1 + j] = a[a0 + j];
        for (int j = lane; j < tb; j += 32) buf[1 + ta + j] = b[b0 + j];
        __syncwarp();
        const vid_t *sa = buf + 1, *sb = buf + 1 + ta;
        const int tt = ta + tb;
        const int per = (tt + 31) >> 5;
        const int d0 = min(lane * per, tt), d1 = min(d0 + per, tt);
        int ai = diag_split(sa, ta, sb, tb, d0), bi = d0 - ai;
        for (int s = d0; s < d1; ++s) {
            const bool takeA = bi >= tb || (ai < ta && sa[ai] <= sb[bi]);
            if (takeA) ++ai;
            else { hits += (sa[ai - 1] == sb[bi]); ++bi; }     // a B element right after its equal A element
        }
    }
    return hits;
}

// Galloping pays off once the longer list is this many times the shorter one (the set-algebra and ADG pull kernels;
// the triangle schedule takes its ratio from gmsb_tc_options.gallop_ratio instead).
constexpr int kGallopRatio = 8;

// |A ∩ B| as a per-lane partial count (caller reduces): galloping for skewed pairs, merge path for balanced ones
__device__ __forceinline__ uint32_t warp_intersect_count(const vid_t *__restrict__ a, int na, const vid_t *__restrict__ b,
                                                         int nb, int lane, vid_t *buf) {
    const int lo = na < nb ? na : nb, hi = na < nb ? nb : na;
    if (lo == 0) return 0;
    if ((long long)hi >= (long long)kGallopRatio * lo) return warp_gallop_count(a, na, b, nb, lane);
    return warp_merge_count(a, na, b, nb, lane, buf);
}

__device__ __forceinline__ unsigned long long warp_sum(unsigned long long x) {
    for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

__device__ __forceinline__ unsigned long long block_sum(unsigned long long x, unsigned long long *red) {
    x = warp_sum(x);
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    if (lane == 0) red[warp] = x;
    __syncthreads();
    if (warp == 0) {
        x = lane < nw ? red[lane] : 0ull;
        x = warp_sum(x);
    }
    return x;      // valid in thread 0
}

inline int grid_for(int64_t items, int block) {
    int64_t g = ceil_div(items, block);
    int64_t cap = (int64_t)rt().sm_count * 32;
    return (int)std::max<int64_t>(1, std::min(g, cap));
}

}  // namespace gmsb
