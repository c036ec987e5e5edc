// kclique.cu — k-clique counting on an oriented DAG.
//
// Replaces:
//   KClique::KcListing / Parallelize::{node,edge}     gms/algorithms/non_set_based/k_clique_list/kernels/kclisting.h:19-189,
//                                                     parallelizationStrategy/parallelize.h:39-121
//   Builders::SubGraphBuilder::buildSubGraph          parallelizationStrategy/SubGraphBuilder.h:42-123
//   CliqueCount<Set,SGraph,Set2> (k! * C_k)           gms/algorithms/set_based/k_clique_count/k_clique_count_set_based.h:6-31
//
// The reference builds, per vertex or per edge, an induced sub-DAG as a fresh CSR (new NodeId[c*c]) and walks it
// with label arrays, counting the last level one clique at a time.  Here the induced sub-DAG on S = N+(u) is a
// |S| x |S| BIT MATRIX held on chip (row i = members of S that are out-neighbours of S[i]); a recursion level is one
// AND of a candidate bitset with a row, and the last level is a popcount, so the cost is proportional to the number
// of (k-1)-cliques rather than k-cliques and no memory is allocated per sub-problem.
//   d+(u) <= 32 : one warp per u, the matrix lives in 32 registers' worth of shared words, every lane runs the
//                 depth-first search of one first-level member with single 32-bit masks;
//   d+(u)  > 32 : one CTA per u, matrix in shared memory (rows built by streaming N+(S[i]) and binary-searching S);
//                 two kernel families search it:
//                   * warp-cooperative (this file): warps pull first-level members from a ticket and search with
//                     lane-distributed bitsets — used for k <= 4 and k > 10;
//                   * lane-parallel (kclique_lane.cuh, kclique_lane_core.cuh): every lane searches its own subtree
//                     of a compact matrix with its candidate sets in registers — used for 5 <= k <= 10, 4x faster at
//                     k = 6 on Kronecker scale 22 (139 s -> 35 s).
// Every acyclic orientation counts each clique exactly once, so the result equals the reference's for any
// ranking (degree, degeneracy, ...).
#include "common.cuh"
#include "sort.cuh"
#include "isect.cuh"
#include "orient.cuh"
#include "ops.cuh"
#include "kclique_lane.cuh"
#include <cstdlib>
#include <algorithm>
#include <vector>

namespace gmsb {

namespace {

constexpr int kMaxK = 16;

// bit-matrix geometry: rows of an even number of 32-bit words (so they can be walked as 64-bit words)
__host__ __device__ inline int row_words(int D) { return ((D + 63) >> 6) << 1; }
__host__ __device__ inline size_t matrix_words(int D) {
    return (size_t)((D + 1) & ~1) + (size_t)D * (size_t)row_words(D);
}

// ---- d+(u) <= 32 -----------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long dfs32(const uint32_t *rows, uint32_t cand, int need) {
    // number of `need`-cliques inside `cand` (bit i = member i), rows[i] = out-neighbours of member i inside S
    if (need == 1) return __popc(cand);
    unsigned long long total = 0;
    uint32_t it[kMaxK], cur[kMaxK];
    int level = 0;
    cur[0] = cand; it[0] = cand;
    for (;;) {
        if (it[level] == 0) {
            if (level == 0) break;
            --level;
            continue;
        }
        const int i = __ffs(it[level]) - 1;
        it[level] &= it[level] - 1;
        const uint32_t nxt = cur[level] & rows[i];
        const int left = need - level - 1;          // vertices still to pick after choosing i
        if (left == 1) total += __popc(nxt);
        else if (__popc(nxt) >= left) { ++level; cur[level] = nxt; it[level] = nxt; }
    }
    return total;
}

__global__ void __launch_bounds__(256)
k_kclique_small(const vid_t *__restrict__ verts, int64_t count, const eid_t *__restrict__ off,
                const vid_t *__restrict__ nbr, int k, unsigned long long *__restrict__ total, int pi, int P) {
    __shared__ uint32_t rows_s[8][32];
    __shared__ unsigned long long red[8];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    uint32_t *rows = rows_s[wib];
    unsigned long long acc = 0;
    for (int64_t t = pi + warp * P; t < count; t += nwarps * P) {
        const vid_t u = verts[t];
        const eid_t ob = off[u];
        const int D = (int)(off[u + 1] - ob);                 // <= 32
        const vid_t mine = lane < D ? nbr[ob + lane] : -1;    // member `lane` of S
        // row of member `lane`: for every later member j, is S[j] in N+(S[lane]) ?
        uint32_t row = 0;
        if (lane < D) {
            const eid_t mb = off[mine];
            const int md = (int)(off[mine + 1] - mb);
            const vid_t *ml = nbr + mb;
            for (int j = lane + 1; j < D; ++j) {
                const vid_t w = nbr[ob + j];
                const int p = lower_bound_dev(ml, md, w);
                if (p < md && ml[p] == w) row |= 1u << j;
            }
        }
        __syncwarp();
        rows[lane] = row;
        __syncwarp();
        // member `lane` is the second clique vertex; k-2 more are picked inside its row
        if (lane < D) acc += k == 2 ? 1ull : dfs32(rows, row, k - 2);
    }
    unsigned long long s = block_sum(acc, red);
    if (threadIdx.x == 0 && s) atomicAdd(total, s);
}

// ---- d+(u) > 32 --------------------------------------------------------------------------------------------------------
// Bitsets of W words are spread over the warp: word w lives in lane (w & 31), slot (w >> 5); WPL slots per lane.
template <int WPL>
struct WarpSet {
    uint32_t w[WPL];
};

template <int WPL>
__device__ __forceinline__ int first_bit(const WarpSet<WPL> &s, int lane) {
    // index of the lowest set bit over the whole warp-distributed bitset, or -1
#pragma unroll
    for (int slot = 0; slot < WPL; ++slot) {
        const unsigned m = __ballot_sync(0xffffffffu, s.w[slot] != 0);
        if (m) {
            const int L = __ffs(m) - 1;
            const uint32_t word = __shfl_sync(0xffffffffu, s.w[slot], L);
            return ((slot << 5) + L) * 32 + (__ffs(word) - 1);
        }
    }
    return -1;
}

// ---- compaction: once a candidate set has <= 64 members, re-index it to 64-bit masks and finish per lane ---------
struct WarpScratch {
    int list[64];                    // positions (in S) of the candidates, ascending
    unsigned long long cm[64];       // cm[a] bit b = candidate b is an out-neighbour of candidate a
};

__device__ unsigned long long dfs64(const unsigned long long *cm, unsigned long long cand, int need) {
    if (need == 1) return __popcll(cand);
    unsigned long long total = 0, it[kMaxK], cur[kMaxK];
    int level = 0;
    cur[0] = cand; it[0] = cand;
    for (;;) {
        if (it[level] == 0) {
            if (level == 0) break;
            --level;
            continue;
        }
        const int i = __ffsll((long long)it[level]) - 1;
        it[level] &= it[level] - 1;
        const unsigned long long nxt = cur[level] & cm[i];
        const int left = need - level - 1;
        if (left == 1) total += __popcll(nxt);
        else if (__popcll(nxt) >= left) { ++level; cur[level] = nxt; it[level] = nxt; }
    }
    return total;
}

// `need`-cliques inside the warp-distributed set `cand` of c <= 64 members (need >= 2); per-lane partial count.
// The recursion below this point never touches the big matrix again: each lane runs the search of one (or two)
// first members with register masks, which is ~30x cheaper per clique than a warp-wide step.
// ascending list of the positions of a warp-distributed set's members (<= 64 of them) in ws->list.
// word w = lane + 32*slot, so the order is slot-major, then lane, then bit.
template <int WPL>
__device__ __forceinline__ void list_members(const WarpSet<WPL> &cand, int lane, WarpScratch *ws) {
    int base = 0;
    __syncwarp();
#pragma unroll
    for (int s = 0; s < WPL; ++s) {
        uint32_t word = cand.w[s];
        const int pc = __popc(word);
        int incl = pc;
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        int pos = base + incl - pc;
        const int wbase = (lane + (s << 5)) << 5;
        while (word) {
            ws->list[pos++] = wbase + __ffs(word) - 1;
            word &= word - 1;
        }
        base += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
}

// Last two levels for a SMALL candidate set (c <= 64 members): the members are listed once, lane t takes members
// t and t+32, and each walks only the 64-bit words between its own position and the set's last member — candidate
// sets deep in the search cluster at the hub end of S, so that is usually two or three words.
template <int WPL>
__device__ unsigned long long pair_count_small(const uint32_t *rows, int W, const WarpSet<WPL> &cset, int c, int lane,
                                               WarpScratch *ws) {
    list_members<WPL>(cset, lane, ws);
    uint32_t *cw = reinterpret_cast<uint32_t *>(ws->cm);
#pragma unroll
    for (int s = 0; s < WPL; ++s) {
        const int w = lane + (s << 5);
        if (w < W) cw[w] = cset.w[s];
    }
    __syncwarp();
    const unsigned long long *cw64 = reinterpret_cast<const unsigned long long *>(cw);
    const int last = ws->list[c - 1] >> 6;
    unsigned long long total = 0;
    for (int a = lane; a < c; a += 32) {
        const int l = ws->list[a];
        const unsigned long long *row64 = reinterpret_cast<const unsigned long long *>(rows + (size_t)l * W);
        uint32_t cnt = 0;
        for (int x = l >> 6; x <= last; ++x) cnt += __popcll(cw64[x] & row64[x]);
        total += cnt;
    }
    __syncwarp();
    return total;
}

template <int WPL>
__device__ unsigned long long compact_count(const uint32_t *rows, int W, const WarpSet<WPL> &cand, int c, int need,
                                            int lane, WarpScratch *ws) {
    // 1. ascending list of member positions
    list_members<WPL>(cand, lane, ws);
    // 2. compact adjacency: only later members can be out-neighbours (positions ascend with vertex id)
    for (int a = lane; a < c; a += 32) {
        const uint32_t *row = rows + (size_t)ws->list[a] * W;
        unsigned long long mask = 0;
        for (int b = a + 1; b < c; ++b) {
            const int p = ws->list[b];
            mask |= (unsigned long long)((row[p >> 5] >> (p & 31)) & 1u) << b;
        }
        ws->cm[a] = mask;
    }
    __syncwarp();
    // 3. member a is the next clique vertex; need-1 more inside its compact row.  With two or more levels left the
    //    work is dealt out as (a, b) PAIRS — lane t takes the t-th out-neighbour b of a — so that 32 lanes share one
    //    member's subtree instead of each lane owning a whole (and very unequal) subtree.
    unsigned long long total = 0;
    if (need - 1 == 1) {
        for (int a = lane; a < c; a += 32) total += __popcll(ws->cm[a]);
        return total;
    }
    for (int a = 0; a < c; ++a) {
        const unsigned long long ra = ws->cm[a];
        const int na = __popcll(ra);
        if (na < need - 1) continue;
        const unsigned lo = (unsigned)ra, hi = (unsigned)(ra >> 32);
        const int nlo = __popc(lo);
        for (int t = lane; t < na; t += 32) {
            const int b = t < nlo ? (int)__fns(lo, 0, t + 1) : 32 + (int)__fns(hi, 0, t - nlo + 1);
            total += dfs64(ws->cm, ra & ws->cm[b], need - 2);
        }
    }
    return total;
}

// Last two levels for a LARGE candidate set c (2-cliques inside c = sum over l in c of |c ∩ row_l|): c is parked in
// the warp's scratch and every lane walks the rows of the members found in its own words, so a warp retires 32
// members per pass instead of one per shuffle/ballot round.
template <int WPL>
__device__ unsigned long long pair_count(const uint32_t *rows, int W, const WarpSet<WPL> &c, int lane,
                                         WarpScratch *ws) {
    uint32_t *cw = reinterpret_cast<uint32_t *>(ws->cm);          // 512 B = 128 words >= W
    __syncwarp();
#pragma unroll
    for (int s = 0; s < WPL; ++s) {
        const int w = lane + (s << 5);
        if (w < W) cw[w] = c.w[s];
    }
    __syncwarp();
    unsigned long long total = 0;
#pragma unroll
    for (int s = 0; s < WPL; ++s) {
        const int w = lane + (s << 5);
        uint32_t word = c.w[s];
        while (word) {
            const int l = (w << 5) + __ffs(word) - 1;
            word &= word - 1;
            // row_l only has members after l; rows are 8-byte aligned with an even word count -> 64-bit steps
            const unsigned long long *row64 = reinterpret_cast<const unsigned long long *>(rows + (size_t)l * W);
            const unsigned long long *cw64 = reinterpret_cast<const unsigned long long *>(cw);
            uint32_t cnt = 0;
            for (int x = w >> 1; x < (W >> 1); ++x) cnt += __popcll(cw64[x] & row64[x]);
            total += cnt;
        }
    }
    __syncwarp();
    return total;
}

template <int WPL>
__device__ unsigned long long dfs_warp(const uint32_t *rows, int W, WarpSet<WPL> cand, int need, int lane,
                                       WarpScratch *ws) {
    // per-lane partial count of `need`-cliques inside cand; caller reduces over the warp
    unsigned long long total = 0;
    int pc0 = 0;
#pragma unroll
    for (int s = 0; s < WPL; ++s) pc0 += __popc(cand.w[s]);
    if (need == 1) return pc0;
    {
        int all = pc0;
        for (int o = 16; o; o >>= 1) all += __shfl_xor_sync(0xffffffffu, all, o);
        if (all < need) return 0;
        if (all <= 64)
            return need == 2 ? pair_count_small<WPL>(rows, W, cand, all, lane, ws)
                             : compact_count<WPL>(rows, W, cand, all, need, lane, ws);
        if (need == 2) return pair_count<WPL>(rows, W, cand, lane, ws);
    }
    WarpSet<WPL> it[kMaxK - 2], cur[kMaxK - 2];
    int level = 0;
    cur[0] = cand; it[0] = cand;
    for (;;) {
        const int i = first_bit<WPL>(it[level], lane);
        if (i < 0) {
            if (level == 0) break;
            --level;
            continue;
        }
        {   // clear bit i in the iterator
            const int w = i >> 5;
            if ((w & 31) == lane) it[level].w[w >> 5] &= ~(1u << (i & 31));
        }
        WarpSet<WPL> nxt;
        int pc = 0;
#pragma unroll
        for (int s = 0; s < WPL; ++s) {
            const int w = lane + (s << 5);
            nxt.w[s] = w < W ? (cur[level].w[s] & rows[(size_t)i * W + w]) : 0u;
            pc += __popc(nxt.w[s]);
        }
        const int left = need - level - 1;
        if (left == 1) total += pc;
        else {
            // descend only if enough candidates remain (warp-wide popcount); small sets finish in registers
            int all = pc;
            for (int o = 16; o; o >>= 1) all += __shfl_xor_sync(0xffffffffu, all, o);
            if (all >= left) {
                if (all <= 64)
                    total += left == 2 ? pair_count_small<WPL>(rows, W, nxt, all, lane, ws)
                                       : compact_count<WPL>(rows, W, nxt, all, left, lane, ws);
                else if (left == 2) total += pair_count<WPL>(rows, W, nxt, lane, ws);
                else { ++level; cur[level] = nxt; it[level] = nxt; }
            }
        }
    }
    return total;
}

template <int WPL, int BLOCK, int MINB>
__global__ void __launch_bounds__(BLOCK, MINB)
k_kclique_big(const vid_t *__restrict__ verts, const int64_t *__restrict__ item_base, int64_t nverts, int64_t count,
              const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int k, int maxD,
              unsigned long long *__restrict__ total, unsigned int *__restrict__ ticket,
              uint32_t *__restrict__ spill, int pi, int P) {
    extern __shared__ uint32_t smem[];
    // member list + bit matrix live in shared memory, or — when max d+ makes them larger than an SM's shared
    // memory — in this CTA's slice of a global scratch buffer (L2-resident for the sizes that occur)
    uint32_t *store = spill ? spill + (size_t)blockIdx.x * matrix_words(maxD) : smem;
    vid_t *S = reinterpret_cast<vid_t *>(store);           // maxD members (padded to an even count)
    uint32_t *rows = store + ((maxD + 1) & ~1);            // D x W bit matrix, W even so rows are 8-byte aligned
    __shared__ unsigned long long red[BLOCK / 32];
    __shared__ WarpScratch scratch[BLOCK / 32];
    __shared__ unsigned int s_item;
    __shared__ int s_next;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int NW = BLOCK / 32;
    unsigned long long acc = 0;
    for (;;) {
        __syncthreads();
        if (tid == 0) { s_item = atomicAdd(ticket, 1u); s_next = 0; }
        __syncthreads();
        const int64_t item = pi + (int64_t)s_item * P;          // this process's share: items pi, pi+P, ...
        if (item >= count) break;
        // item -> (vertex t, part of its second-level members): heavy vertices are cut into several items so that
        // one dense neighbourhood does not serialise on a single CTA (item_base = exclusive scan of parts)
        const int64_t t = lane::item_vertex(item_base, nverts, item);
        const int part = (int)(item - item_base[t]), nparts = (int)(item_base[t + 1] - item_base[t]);
        const vid_t u = verts[t];
        const eid_t ob = off[u];
        const int D = (int)(off[u + 1] - ob);
        const int W = row_words(D);
        for (int j = tid; j < D; j += BLOCK) S[j] = nbr[ob + j];
        for (int j = tid; j < D * W; j += BLOCK) rows[j] = 0u;
        __syncthreads();
        // rows: warp per member i streams N+(S[i]) and looks every element up in S
        for (int i = warp; i < D; i += NW) {
            const vid_t vi = S[i];
            const eid_t mb = off[vi];
            const int md = (int)(off[vi + 1] - mb);
            for (int j = lane; j < md; j += 32) {
                const vid_t w = nbr[mb + j];
                int lo = i + 1, hi = D;                     // members after i only (ids ascend with position)
                while (lo < hi) {
                    const int mid = (lo + hi) >> 1;
                    if (S[mid] < w) lo = mid + 1; else hi = mid;
                }
                if (lo < D && S[lo] == w) atomicOr(&rows[(size_t)i * W + (lo >> 5)], 1u << (lo & 31));
            }
        }
        __syncthreads();
        // search: a warp takes first-level member i; its row is the candidate set for the other k-2 vertices
        for (;;) {
            int i = 0;
            if (lane == 0) i = atomicAdd(&s_next, 1);
            i = part + __shfl_sync(0xffffffffu, i, 0) * nparts;      // members part, part+nparts, ... (interleaved)
            if (i >= D) break;
            WarpSet<WPL> cand;
#pragma unroll
            for (int s = 0; s < WPL; ++s) {
                const int w = lane + (s << 5);
                cand.w[s] = w < W ? rows[(size_t)i * W + w] : 0u;
            }
            acc += dfs_warp<WPL>(rows, W, cand, k - 2, lane, &scratch[warp]);
        }
    }
    unsigned long long s = block_sum(acc, red);
    if (tid == 0 && s) atomicAdd(total, s);
}

// vertices with enough out-neighbours for a k-clique, split by d+ <= 32
__global__ void k_bucket_flags(const eid_t *__restrict__ off, int64_t n, int k, uint8_t *__restrict__ small,
                               uint8_t *__restrict__ big, int *__restrict__ maxd) {
    int mx = 0;
    for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < n; u += (int64_t)gridDim.x * blockDim.x) {
        const int64_t d = off[u + 1] - off[u];
        const bool ok = d >= k - 1;
        small[u] = ok && d <= 32;
        big[u] = ok && d > 32;
        if (ok && d > 32) mx = max(mx, (int)d);
    }
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0 && mx) atomicMax(maxd, mx);
}
__global__ void k_bucket_fill(int64_t n, const uint8_t *__restrict__ flag, const int64_t *__restrict__ pos,
                              vid_t *__restrict__ out) {
    for (int64_t u = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; u < n; u += (int64_t)gridDim.x * blockDim.x)
        if (flag[u]) out[pos[u]] = (vid_t)u;
}

// big vertices sorted by descending out-degree so that the heaviest sub-problems start first
__global__ void k_degree_key(const vid_t *__restrict__ verts, int64_t cnt, const eid_t *__restrict__ off,
                             uint64_t *__restrict__ keys) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
        const vid_t u = verts[i];
        keys[i] = ((uint64_t)(off[u + 1] - off[u]) << 32) | (uint32_t)u;
    }
}
// parts[t] = number of work items vertex t is cut into (parts[cnt] = 0 ends the list for the exclusive scan)
constexpr int kMidD = 512;
__global__ void k_parts(const vid_t *__restrict__ verts, int64_t cnt, const eid_t *__restrict__ off,
                        int k, int part_rows, int64_t *__restrict__ parts) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i <= cnt; i += (int64_t)gridDim.x * blockDim.x) {
        if (i == cnt) { parts[i] = 0; continue; }
        const vid_t u = verts[i];
        const int64_t d = off[u + 1] - off[u];
        // for k <= 4 building the matrix dominates, so a vertex stays whole; deeper searches are cut finer
        // (every part rebuilds the vertex's matrix, so parts are kept few: the split is only there to spread the
        // handful of densest neighbourhoods over several SMs)
        parts[i] = k <= 4 ? 1 : (d > kMidD ? (d + part_rows - 1) / part_rows : 1);
    }
}
__global__ void k_key_vertex(const uint64_t *__restrict__ keys, int64_t cnt, vid_t *__restrict__ verts) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x)
        verts[i] = (vid_t)(uint32_t)keys[i];
}

// number of vertices (of the descending-degree list) above each class boundary: d+ > 512, 256, 128, 64
__global__ void k_class_counts(const vid_t *__restrict__ verts, int64_t cnt, const eid_t *__restrict__ off,
                               int *__restrict__ counts) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
        const vid_t u = verts[i];
        const int64_t d = off[u + 1] - off[u];
        if (d > 512) atomicAdd(&counts[0], 1);
        if (d > 256) atomicAdd(&counts[1], 1);
        if (d > 128) atomicAdd(&counts[2], 1);
        if (d > 64) atomicAdd(&counts[3], 1);
    }
}

__global__ void k_list_degrees(const vid_t *__restrict__ verts, int64_t cnt, const eid_t *__restrict__ off,
                               int *__restrict__ deg) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * blockDim.x) {
        const vid_t u = verts[i];
        deg[i] = (int)(off[u + 1] - off[u]);
    }
}

// The d+ > 32 vertices in descending out-degree order, and what every class launch needs.
struct BigVerts {
    const vid_t *verts;
    int64_t count;
    int64_t bound[4];              // how many of them have d+ > 512, 256, 128, 64
    int maxD;
    const eid_t *off;
    const vid_t *nbr;
    int k, pi, P;
    DevBuf<unsigned long long> &total;
};

// k = 3, 4, 11..16: the warp-cooperative kernel in two launches, so that the many mid-size neighbourhoods get a small
// matrix and several CTAs per SM.  Work items: (vertex, interleaved part of its second-level members).
void count_warp(const BigVerts &b) {
    Runtime &r = rt();
    DevBuf<int64_t> parts(b.count + 1), item_base(b.count + 1);
    k_parts<<<grid_for(b.count, 256), 256, 0, r.stream>>>(b.verts, b.count, b.off, b.k, 256, parts.p); launched();
    auto run_class = [&](int64_t first, int64_t cnt, int classD, bool huge) {
        if (cnt == 0) return;
        exclusive_sum(parts.p + first, item_base.p, cnt + 1);
        const int64_t n_items = item_base.get(cnt);
        const int W = row_words(classD);
        const size_t need = matrix_words(classD) * 4;
        const bool in_smem = need + 28 * 1024 <= r.smem_optin;    // static scratch (WarpScratch etc.) is <= 25 KB
        const size_t smem = in_smem ? need : 0;
        DevBuf<unsigned int> ticket(1);
        ticket.zero();
        DevBuf<uint32_t> spill;
        auto launch = [&](auto kern, int block) {
            // set on every launch: without it the dynamic part may only take 48 KB minus the static scratch (24.8 KB
            // for the 1024-thread builds), and a larger value left by an earlier call must not decide what fits
            GMSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            int resident = 0;
            GMSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, block, smem));
            GMSB_REQUIRE(resident >= 1, "kclique_count: kernel does not fit on an SM");
            if (!in_smem) resident = 1;
            const int grid = (int)std::min<int64_t>(n_items, (int64_t)r.sm_count * resident);
            if (!in_smem) spill.alloc((size_t)grid * (need / 4));
            kern<<<grid, block, smem, r.stream>>>(b.verts + first, item_base.p, cnt, n_items, b.off, b.nbr, b.k, classD,
                                                  b.total.p, ticket.p, in_smem ? nullptr : spill.p, b.pi, b.P);
            launched();
            GMSB_CUDA(cudaStreamSynchronize(r.stream));
        };
        // the search is a chain of dependent shared-memory steps, so resident warps are what hides its latency:
        // a big matrix fills the SM's shared memory -> one CTA of 1024 threads; mid-size ones -> 2 x 512
        if (huge) {
            if (W <= 32) launch(k_kclique_big<1, 1024, 1>, 1024);
            else if (W <= 64) launch(k_kclique_big<2, 1024, 1>, 1024);
            else launch(k_kclique_big<4, 1024, 1>, 1024);
        } else {
            launch(k_kclique_big<1, 512, 2>, 512);        // kMidD = 512 -> W = 16
        }
    };
    run_class(0, b.bound[0], b.maxD, true);
    run_class(b.bound[0], b.count - b.bound[0], kMidD, false);
}

// Launches of the lane kernels' classes.  The class kernels are independent (own ticket, atomics on one total), so
// each k_kclique_lane_mid class goes to its own stream: its CTAs fill the SMs that the previous class's last items
// leave idle, and with the sub-problems split over several GPUs those tails are a visible share of a launch.
// GMSB_KCLIQUE_TRACE=1 (profiling aid) serialises the launches and prints the device time and clique count of every
// class on stderr.
class LaneClasses {
  public:
    explicit LaneClasses(const BigVerts &b) : b_(b), r_(rt()), trace_(std::getenv("GMSB_KCLIQUE_TRACE") != nullptr) {
        tickets_.zero();
        mark(nullptr, 0);
        if (!trace_) {
            GMSB_CUDA(cudaEventCreateWithFlags(&own_.ready, cudaEventDisableTiming));
            GMSB_CUDA(cudaEventRecord(own_.ready, r_.stream));
            for (auto &st : own_.aux) {
                GMSB_CUDA(cudaStreamCreateWithFlags(&st, cudaStreamNonBlocking));
                GMSB_CUDA(cudaStreamWaitEvent(st, own_.ready, 0));
            }
        }
    }

    // ticket of the d+ > 512 (k = 5, 6) or pair (k >= 7) kernel
    unsigned int *first_ticket() { return tickets_.p; }

    // end of class `name` (`vertices` vertices), launched on the library stream
    void mark(const char *name, int64_t vertices) {
        if (!trace_) return;
        Mark m{nullptr, 0, name, vertices};
        cudaEventCreate(&m.ev);
        own_.events.push_back(m.ev);
        cudaEventRecord(m.ev, r_.stream);
        m.seen = b_.total.get(0);          // synchronises: per-class counts for the trace
        marks_.push_back(m);
    }

    // vertices [first, end) of the list through k_kclique_lane_mid<NWB, BLOCK, MINB>; with rows of 3 or more words
    // every warp gets a box for its third-level matrices
    template <int NWB, int BLOCK, int MINB>
    void mid(int64_t first, int64_t end, const char *name) {
        const int cls = next_++;
        if (end > first) {
            auto kern = lane::k_kclique_lane_mid<NWB, BLOCK, MINB>;
            const size_t dyn = NWB >= 3 ? (size_t)(BLOCK / 32) * sizeof(lane::WarpBox) : 0;
            GMSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
            int resident = 0;
            GMSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, BLOCK, dyn));
            GMSB_REQUIRE(resident >= 1, "kclique_count: kernel does not fit on an SM");
            const int grid = (int)std::min<int64_t>(end - first, (int64_t)r_.sm_count * resident);
            cudaStream_t st = trace_ ? r_.stream : own_.aux[cls];
            kern<<<grid, BLOCK, dyn, st>>>(b_.verts + first, end - first, b_.off, b_.nbr, b_.k, b_.total.p,
                                           tickets_.p + 1 + cls, b_.pi, b_.P);
            launched();
        }
        mark(name, std::max<int64_t>(end - first, 0));
    }

    // the library stream continues after every class
    void join() {
        if (!trace_) {
            for (auto &st : own_.aux) {
                GMSB_CUDA(cudaEventRecord(own_.ready, st));
                GMSB_CUDA(cudaStreamWaitEvent(r_.stream, own_.ready, 0));
            }
        }
        GMSB_CUDA(cudaStreamSynchronize(r_.stream));
        for (size_t i = 1; i < marks_.size(); ++i) {
            float ms = 0;
            cudaEventElapsedTime(&ms, marks_[i - 1].ev, marks_[i].ev);
            std::fprintf(stderr, "[gmsb kclique k=%d] %-13s vertices=%lld ms=%.3f cliques=%llu\n", b_.k, marks_[i].name,
                         (long long)marks_[i].vertices, ms, marks_[i].seen - marks_[i - 1].seen);
        }
    }

  private:
    struct Mark {
        cudaEvent_t ev;
        unsigned long long seen;
        const char *name;
        int64_t vertices;
    };
    const BigVerts &b_;
    Runtime &r_;
    const bool trace_;
    DevBuf<unsigned int> tickets_{5};          // [0] first_ticket(), [1..4] the mid classes in launch order
    struct Owned {                             // released also when the constructor throws half-way
        cudaStream_t aux[4] = {nullptr, nullptr, nullptr, nullptr};
        cudaEvent_t ready = nullptr;
        std::vector<cudaEvent_t> events;
        ~Owned() {
            for (auto st : aux) if (st) cudaStreamDestroy(st);
            if (ready) cudaEventDestroy(ready);
            for (auto ev : events) cudaEventDestroy(ev);
        }
    } own_;
    int next_ = 0;
    std::vector<Mark> marks_;
};

// k = 5, 6: d+ > 512 through k_kclique_lane_huge, one CTA per SM on vertex parts of 64 rows (CTA-wide top of the tree,
// compact matrices below); the four classes <= 512 / 256 / 128 / 64 through k_kclique_lane_mid.
void count_lane_huge(const BigVerts &b) {
    Runtime &r = rt();
    const int64_t n_huge = b.bound[0];
    DevBuf<int64_t> parts, item_base;
    DevBuf<lane::u64> spill;
    LaneClasses classes(b);
    if (n_huge) {
        parts.alloc(n_huge + 1);
        item_base.alloc(n_huge + 1);
        k_parts<<<grid_for(n_huge, 256), 256, 0, r.stream>>>(b.verts, n_huge, b.off, b.k, 64, parts.p); launched();
        exclusive_sum(parts.p, item_base.p, n_huge + 1);
        const int64_t n_items = item_base.get(n_huge);
        // 512 threads cap the kernel at 128 registers and it spills; 384 threads (168 registers, no spills) were 6 %
        // faster at scale 22, k = 6
        constexpr int BLOCK = 384;
        auto kern = lane::k_kclique_lane_huge<BLOCK>;
        const size_t full = lane::huge_smem_words(b.maxD, true) * 8;
        const bool in_smem = full + 2048 <= r.smem_optin;
        const size_t smem = in_smem ? full : lane::huge_smem_words(b.maxD, false) * 8;
        GMSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int grid = (int)std::min<int64_t>(n_items, (int64_t)r.sm_count);
        if (!in_smem) spill.alloc((size_t)grid * (size_t)b.maxD * (size_t)lane::huge_pitch(b.maxD));
        kern<<<grid, BLOCK, smem, r.stream>>>(b.verts, item_base.p, n_huge, n_items, b.off, b.nbr, b.k, b.maxD,
                                              b.total.p, classes.first_ticket(), in_smem ? nullptr : spill.p, b.pi, b.P);
        launched();
    }
    classes.mark("huge(d+>512)", n_huge);
    classes.mid<8, 384, 2>(b.bound[0], b.bound[1], "mid8(<=512)");
    classes.mid<4, 256, 4>(b.bound[1], b.bound[2], "mid4(<=256)");
    classes.mid<2, 128, 8>(b.bound[2], b.bound[3], "mid2(<=128)");
    classes.mid<1, 128, 8>(b.bound[3], b.count, "mid1(<=64)");
    classes.join();
}

// k = 7..10: d+ > 128 decoupled — M1 of every such vertex to global memory (k_kclique_m1_build), then (vertex, member)
// work items through k_kclique_lane_pair, which searches through third-level matrices; those pay when five or more
// vertices are left below u and S[i].  The classes <= 128 / 64 go through k_kclique_lane_mid.  Smallest class of the
// pair kernel, k = 7 at scale 20: d+ > 512 85.7 s, > 256 67.5 s, > 128 64.5 s.
void count_lane_pair(const BigVerts &b) {
    Runtime &r = rt();
    const int64_t n_pair = b.bound[2];
    LaneClasses classes(b);
    if (n_pair) {
        // Sizes come from the (few thousand) out-degrees on the host; the vertices are processed in batches whose
        // matrices fit kM1Budget bytes.
        std::vector<vid_t> hv((size_t)n_pair);
        GMSB_CUDA(cudaMemcpyAsync(hv.data(), b.verts, sizeof(vid_t) * n_pair, cudaMemcpyDeviceToHost, r.stream));
        GMSB_CUDA(cudaStreamSynchronize(r.stream));
        std::vector<int> hd((size_t)n_pair);
        {
            // out-degrees of the listed vertices (descending): two offsets each
            DevBuf<int> dd((size_t)n_pair);
            k_list_degrees<<<grid_for(n_pair, 256), 256, 0, r.stream>>>(b.verts, n_pair, b.off, dd.p); launched();
            dd.download(hd.data(), (size_t)n_pair);
        }
        constexpr size_t kM1Budget = size_t(12) << 30;
        constexpr int PBLOCK = 256;
        const size_t smem2 = lane::pair_smem_words(b.maxD, PBLOCK / 32) * 8;
        GMSB_REQUIRE(smem2 + 4096 <= r.smem_optin, "kclique_count: out-degree too large for the pair kernel");
        auto kern2 = lane::k_kclique_lane_pair<PBLOCK>;
        GMSB_CUDA(cudaFuncSetAttribute(kern2, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2));
        int resident2 = 0;
        GMSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident2, kern2, PBLOCK, smem2));
        GMSB_REQUIRE(resident2 >= 1, "kclique_count: pair kernel does not fit on an SM");
        constexpr int BBLOCK = 256;
        const size_t smem1 = ((size_t)(BBLOCK / 32) * lane::huge_pitch(b.maxD) + (size_t)((b.maxD + 1) >> 1)) * 8;
        auto kern1 = lane::k_kclique_m1_build<BBLOCK>;
        GMSB_CUDA(cudaFuncSetAttribute(kern1, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
        DevBuf<int64_t> pair_base, m1_off;
        DevBuf<lane::u64> m1;
        unsigned int *ticket = classes.first_ticket();
        int64_t t0 = 0;
        int64_t item0 = 0;                       // global numbering of the items, for the multi-GPU deal
        while (t0 < n_pair) {
            std::vector<int64_t> h_m1((size_t)0), h_items((size_t)0);
            size_t words = 0;
            int64_t items = 0, t1 = t0;
            while (t1 < n_pair) {
                const size_t w = (size_t)hd[t1] * (size_t)lane::huge_pitch(hd[t1]);
                if (t1 > t0 && (words + w) * 8 > kM1Budget) break;
                h_m1.push_back((int64_t)words); h_items.push_back(items);
                words += w; items += hd[t1]; ++t1;
            }
            h_items.push_back(items);
            const int64_t nv = t1 - t0;
            m1.alloc(words);
            m1_off.alloc((size_t)nv); pair_base.alloc((size_t)nv + 1);
            m1_off.upload(h_m1.data(), (size_t)nv);
            pair_base.upload(h_items.data(), (size_t)nv + 1);
            const int grid1 = (int)std::min<int64_t>(nv, (int64_t)r.sm_count * 4);
            kern1<<<grid1, BBLOCK, smem1, r.stream>>>(b.verts, t0, nv, b.off, b.nbr, m1_off.p, m1.p, b.maxD); launched();
            // this process's items of the batch: global item numbers congruent to pi modulo P
            const int shift = (int)(((int64_t)b.pi - item0 % b.P + b.P) % b.P);
            const int64_t mine = items > shift ? (items - shift + b.P - 1) / b.P : 0;
            if (mine) {
                GMSB_CUDA(cudaMemsetAsync(ticket, 0, sizeof(unsigned int), r.stream));
                const int grid2 = (int)std::min<int64_t>(mine, (int64_t)r.sm_count * resident2);
                kern2<<<grid2, PBLOCK, smem2, r.stream>>>(b.verts, t0, pair_base.p, nv, items, b.off, m1_off.p, m1.p,
                                                          b.k, b.maxD, b.total.p, ticket, shift, b.P);
                launched();
            }
            GMSB_CUDA(cudaStreamSynchronize(r.stream));      // host vectors / batch buffers are reused
            item0 += items;
            t0 = t1;
        }
    }
    classes.mark("pair(d+>128)", n_pair);
    classes.mid<2, 128, 8>(b.bound[2], b.bound[3], "mid2(<=128)");
    classes.mid<1, 128, 8>(b.bound[3], b.count, "mid1(<=64)");
    classes.join();
}

uint64_t count_on_dag(int64_t n, int64_t m, const eid_t *off, const vid_t *nbr, int k, int pi, int P) {
    Runtime &r = rt();
    if (k == 1) return pi == 0 ? (uint64_t)n : 0;  // parallelize.h:43
    if (k == 2) return pi == 0 ? (uint64_t)m : 0;  // parallelize.h:44
    GMSB_REQUIRE(k <= kMaxK, "kclique_count: clique size above 16 is not supported");
    if (n == 0 || m == 0) return 0;
    DevBuf<uint8_t> fs(n), fb(n);
    DevBuf<int64_t> ps(n + 1), pb(n + 1);
    DevBuf<int> maxd(1);
    maxd.zero();
    k_bucket_flags<<<grid_for(n, 256), 256, 0, r.stream>>>(off, n, k, fs.p, fb.p, maxd.p); launched();
    exclusive_sum(fs.p, ps.p, n);
    exclusive_sum(fb.p, pb.p, n);
    const int64_t ns = ps.get(n - 1) + fs.get(n - 1), nb = pb.get(n - 1) + fb.get(n - 1);
    const int maxD = maxd.get(0);
    DevBuf<unsigned long long> total(1);
    total.zero();
    if (ns) {
        DevBuf<vid_t> vs(ns);
        k_bucket_fill<<<grid_for(n, 256), 256, 0, r.stream>>>(n, fs.p, ps.p, vs.p); launched();
        int grid = (int)std::min<int64_t>(ceil_div(ns, 8), (int64_t)r.sm_count * 16);
        k_kclique_small<<<grid, 256, 0, r.stream>>>(vs.p, ns, off, nbr, k, total.p, pi, P); launched();
    }
    if (nb) {
        DevBuf<vid_t> vb(nb);
        k_bucket_fill<<<grid_for(n, 256), 256, 0, r.stream>>>(n, fb.p, pb.p, vb.p); launched();
        DevBuf<uint64_t> keys(nb), alt(nb);
        k_degree_key<<<grid_for(nb, 256), 256, 0, r.stream>>>(vb.p, nb, off, keys.p); launched();
        uint64_t *sorted = radix_sort_keys(keys.p, alt.p, nb, 0, 64, /*descending=*/true);
        k_key_vertex<<<grid_for(nb, 256), 256, 0, r.stream>>>(sorted, nb, vb.p); launched();
        if (row_words(maxD) > 128)
            throw Error(GMSB_ERR_UNSUPPORTED, "kclique_count: max out-degree " + std::to_string(maxD) +
                                                  " exceeds 4096; orient by degree or degeneracy first");
        DevBuf<int> cc(4);
        cc.zero();
        k_class_counts<<<grid_for(nb, 256), 256, 0, r.stream>>>(vb.p, nb, off, cc.p); launched();
        int bound[4];
        cc.download(bound, 4);
        const BigVerts b{vb.p, nb, {bound[0], bound[1], bound[2], bound[3]}, maxD, off, nbr, k, pi, P, total};
        // lane-parallel kernels where they are faster (B200 measurements, DESIGN.md §3.4) and their path register
        // holds the search (k - 1 <= lane::kMaxNeed); warp-cooperative otherwise
        if (k < 5 || k - 1 > lane::kMaxNeed) count_warp(b);
        else if (k < 7) count_lane_huge(b);
        else count_lane_pair(b);
    }
    return total.get(0);
}

}  // namespace

namespace {
__global__ void k_expand_sources(const eid_t *__restrict__ off, int64_t n, vid_t *__restrict__ src) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t u = warp; u < n; u += nwarps)
        for (eid_t e = off[u] + lane; e < off[u + 1]; e += 32) src[e] = (vid_t)u;
}
// out[0] = largest out-degree; out[1] = 1 when some arc does not go from a lower to a higher id.  The matrix builders
// only look for out-neighbours among the LATER members of S (ids ascend with position), which is right exactly when
// every arc ascends — what gmsb_orient and InduceDirectedGraph produce; any other directed input is re-oriented.
__global__ void k_max_out(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n, int *out) {
    int mx = 0;
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x) {
        const eid_t b = off[v], e = off[v + 1];
        mx = max(mx, (int)(e - b));
        if (e > b && nbr[b] <= (vid_t)v) out[1] = 1;          // lists ascend: the first entry is the smallest
    }
    for (int o = 16; o; o >>= 1) mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, mx);
}
}  // namespace

// part_index / part_count: this process counts share part_index of part_count of the per-vertex sub-problems
// (multi-GPU: graph replicated, sub-problems dealt out round-robin in descending-size order, counts summed by the
// caller with one all-reduce); the shares add up to the full count.
void kclique_count(Graph &g, int k, uint64_t *out, int pi, int P) {
    GMSB_REQUIRE(P >= 1 && pi >= 0 && pi < P, "kclique_count: bad partition");
    if (g.directed) {
        Runtime &r = rt();
        if (k <= 2 || g.n == 0 || g.slots == 0) {
            *out = count_on_dag(g.n, g.slots, g.off.p, g.nbr.p, k, pi, P);
            return;
        }
        DevBuf<int> mx(2);
        mx.zero();
        k_max_out<<<grid_for(g.n, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, g.n, mx.p); launched();
        int h_mx[2];
        mx.download(h_mx, 2);
        const int D = h_mx[0];
        if (h_mx[1] == 0 && matrix_words(D) * 4 + 28 * 1024 <= r.smem_optin) {
            *out = count_on_dag(g.n, g.slots, g.off.p, g.nbr.p, k, pi, P);
            return;
        }
        // The reference's own degeneracy pipeline orients from later- to earlier-removed vertices, which leaves
        // out-degrees unbounded (SURVEY.md §3.2), and a directed graph from a file or an edge list may have arcs in
        // both id directions.  Clique counts do not depend on the orientation (KcListing accepts any DAG), so
        // re-orient the underlying undirected graph by degree and count there.
        DevBuf<vid_t> src(g.slots);
        k_expand_sources<<<grid_for(g.n * 32, 256), 256, 0, r.stream>>>(g.off.p, g.n, src.p); launched();
        Graph *und = graph_from_edgelist_device(g.slots, src.p, g.nbr.p, true);
        try {
            und->dag = build_degree_dag(*und);
            *out = count_on_dag(und->dag->n, und->dag->m, und->dag->off.p, und->dag->nbr.p, k, pi, P);
        } catch (...) { delete und; throw; }
        delete und;
        return;
    }
    if (k == 1) { *out = pi == 0 ? (uint64_t)g.n : 0; return; }
    if (!g.dag) g.dag = build_degree_dag(g);
    *out = count_on_dag(g.dag->n, g.dag->m, g.dag->off.p, g.dag->nbr.p, k, pi, P);
}

// CliqueCount on the unoriented graph counts ordered tuples: k! * C_k, with size_t wrap-around.
void kclique_count_ordered(Graph &g, int k, uint64_t *out) {
    GMSB_REQUIRE(!g.directed, "kclique_count_ordered: graph must be undirected");
    uint64_t c = 0;
    kclique_count(g, k, &c);
    uint64_t f = 1;
    for (int i = 2; i <= k; ++i) f *= (uint64_t)i;
    *out = c * f;
}

}  // namespace gmsb
