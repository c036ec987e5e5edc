// truss.cu — truss number of every undirected edge by level-synchronous peeling of triangle support.
//
// truss(e) = the largest k such that e lies in the k-truss, the maximal subgraph in which every edge closes at least
// k-2 triangles of the subgraph; 2 for an edge in no triangle.  GMS has no truss decomposition; the output follows
// gmsb_edge_similarity's convention (one value per undirected edge a<b, in CSR order), so the edge id of (a,b) is its
// position there: base[a] + (index of b among the neighbours of a that are > a), base = upper_edge_base (setops.cu).
//
// The peel (PKT, Kabir & Madduri, "Parallel k-truss decomposition on multicore systems", HPEC 2017):
//   support    the initial support of every edge comes from one pass of the oriented triangle schedule (tc_support.cu);
//   level k    every live edge with support <= k joins the frontier; an empty level jumps k to the least live support,
//              which the same pass finds, so an empty level costs one pass over the edges, not one per skipped value;
//   sub-round  the frontier is marked in_curr; one lane group per frontier edge e = (a,b) walks the shorter row and
//              binary-searches the longer one; every common w whose edges e1 = (a,w), e2 = (b,w) are both live closes
//              a triangle that leaves with e.  The triangle is accounted once: with neither e1 nor e2 in the frontier
//              both lose one unit of support; with exactly one of them in the frontier, the other loses one unit, taken
//              by whichever of the two frontier edges has the smaller id; with both in the frontier nothing is left to
//              decrement.  An edge whose support falls from k+1 to k joins the next frontier of the same level; support
//              never goes below k (a decrement that would is undone).  The frontier then retires with truss = k + 2.
// Both results are graph invariants, so they do not depend on the order in which the atomics land.
//
// The rows keep their retired entries: a retired (a,w) costs one flag read and no search.
#include "common.cuh"
#include "isect.cuh"
#include "ops.cuh"
#include <algorithm>
#include <climits>

namespace gmsb {

namespace {

// Frontier edges whose shorter row has at least this many entries are peeled by a whole CTA instead of one warp.
constexpr int kLongRow = 1024;
constexpr int kLongBlock = 256;

// edge id of every CSR slot; warp per row.  A lower slot (b < a) takes the id of (b,a): a binary search for a in the
// upper part of row b.  Also counts the edges whose shorter row has >= kLongRow entries (the CTA class's queue size).
__global__ void k_slot_edge_ids(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n,
                                const int64_t *__restrict__ base, int32_t *__restrict__ eid,
                                unsigned long long *__restrict__ nlong) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    unsigned long long longs = 0;
    for (int64_t a = warp; a < n; a += nwarps) {
        const eid_t b0 = off[a], e = off[a + 1];
        const eid_t s0 = e - (base[a + 1] - base[a]);              // first neighbour > a
        for (eid_t s = b0 + lane; s < e; s += 32) {
            const vid_t b = nbr[s];
            if (s >= s0) {
                eid[s] = (int32_t)(base[a] + (s - s0));
                longs += min(e - b0, off[b + 1] - off[b]) >= kLongRow;
            } else {
                const int64_t cb = base[b + 1] - base[b];
                const eid_t ub = off[b + 1] - cb;
                eid[s] = (int32_t)(base[b] + lower_bound_dev(nbr + ub, (int)cb, (vid_t)a));
            }
        }
    }
    longs = warp_sum(longs);
    if (lane == 0 && longs) atomicAdd(nlong, longs);
}

// frontier of level k: every live edge with support <= k (warp-aggregated pushes); *min_above = least support > k
__global__ void k_truss_collect(int64_t m, int k, const int *__restrict__ sup, const uint8_t *__restrict__ gone,
                                int32_t *__restrict__ queue, int *__restrict__ qsize, int *__restrict__ min_above) {
    const int lane = threadIdx.x & 31;
    int mn = INT_MAX;
    for (int64_t w0 = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) - lane; w0 < m;
         w0 += (int64_t)gridDim.x * blockDim.x) {
        const int64_t e = w0 + lane;
        bool take = false;
        if (e < m && !gone[e]) {
            const int s = sup[e];
            if (s <= k) take = true; else mn = min(mn, s);
        }
        const unsigned mask = __ballot_sync(0xffffffffu, take);
        if (!mask) continue;
        int at = 0;
        if (lane == 0) at = atomicAdd(qsize, __popc(mask));
        at = __shfl_sync(0xffffffffu, at, 0);
        if (take) queue[at + __popc(mask & ((1u << lane) - 1))] = (int32_t)e;
    }
    for (int o = 16; o; o >>= 1) mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
    if (lane == 0 && mn != INT_MAX) atomicMin(min_above, mn);
}

__global__ void k_truss_mark(const int32_t *__restrict__ queue, int qs, uint8_t *__restrict__ in_curr) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < qs; i += gridDim.x * blockDim.x) in_curr[queue[i]] = 1;
}

__global__ void k_truss_retire(const int32_t *__restrict__ queue, int qs, int k, uint8_t *__restrict__ gone,
                               uint8_t *__restrict__ in_curr, int32_t *__restrict__ truss) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < qs; i += gridDim.x * blockDim.x) {
        const int32_t e = queue[i];
        gone[e] = 1;
        in_curr[e] = 0;
        truss[e] = k + 2;
    }
}

// endpoints a < b of edge e: a is the row whose id range [base[a], base[a+1]) holds e
__device__ __forceinline__ void edge_ends(int32_t e, const int64_t *__restrict__ base, int64_t n,
                                          const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, vid_t &a,
                                          vid_t &b) {
    int64_t lo = 0, hi = n;                  // first row with base > e, minus one
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (base[mid] <= e) lo = mid + 1; else hi = mid;
    }
    a = (vid_t)(lo - 1);
    b = nbr[off[a + 1] - (base[a + 1] - base[a]) + (e - base[a])];
}

__device__ __forceinline__ void decrement(int32_t x, int k, int *__restrict__ sup, int32_t *__restrict__ next,
                                          int *__restrict__ nsize) {
    const int old = atomicSub(&sup[x], 1);
    if (old == k + 1) next[atomicAdd(nsize, 1)] = x;
    else if (old <= k) atomicAdd(&sup[x], 1);
}

// thread t of a group of G peels frontier edge e = (a,b): the triangles through the shorter row's live entries
template <int G>
__device__ __forceinline__ void peel_edge(int32_t e, vid_t a, vid_t b, int t, int k, const eid_t *__restrict__ off,
                                          const vid_t *__restrict__ nbr, const int32_t *__restrict__ eid,
                                          const uint8_t *__restrict__ gone, const uint8_t *__restrict__ in_curr,
                                          int *__restrict__ sup, int32_t *__restrict__ next, int *__restrict__ nsize) {
    const eid_t sa = off[a], sb = off[b];
    const int da = (int)(off[a + 1] - sa), db = (int)(off[b + 1] - sb);
    const eid_t ss = da <= db ? sa : sb, sl = da <= db ? sb : sa;
    const int ns = da <= db ? da : db, nl = da <= db ? db : da;
    for (int j = t; j < ns; j += G) {
        const int32_t e1 = eid[ss + j];
        if (gone[e1]) continue;
        const vid_t w = nbr[ss + j];
        const int p = lower_bound_dev(nbr + sl, nl, w);
        if (p == nl || nbr[sl + p] != w) continue;
        const int32_t e2 = eid[sl + p];
        if (gone[e2]) continue;
        const bool c1 = in_curr[e1], c2 = in_curr[e2];
        if (!c1 && !c2) {
            decrement(e1, k, sup, next, nsize);
            decrement(e2, k, sup, next, nsize);
        } else if (c1 != c2 && e < (c1 ? e1 : e2)) {
            decrement(c1 ? e2 : e1, k, sup, next, nsize);
        }
    }
}

// warp per frontier edge; edges whose shorter row has >= kLongRow entries go to the CTA class's queue instead
__global__ void __launch_bounds__(256)
k_truss_peel(const int32_t *__restrict__ queue, int qs, int k, const int64_t *__restrict__ base, int64_t n,
             const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const int32_t *__restrict__ eid,
             const uint8_t *__restrict__ gone, const uint8_t *__restrict__ in_curr, int *__restrict__ sup,
             int32_t *__restrict__ next, int *__restrict__ nsize, int32_t *__restrict__ long_queue,
             int *__restrict__ long_size) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < qs; i += nwarps) {
        const int32_t e = queue[i];
        vid_t a, b;
        edge_ends(e, base, n, off, nbr, a, b);
        if (min(off[a + 1] - off[a], off[b + 1] - off[b]) >= kLongRow) {
            if (lane == 0) long_queue[atomicAdd(long_size, 1)] = e;
            continue;
        }
        peel_edge<32>(e, a, b, lane, k, off, nbr, eid, gone, in_curr, sup, next, nsize);
    }
}

// CTA per frontier edge of the long-row queue (its size is read on the device: no host round trip)
__global__ void __launch_bounds__(kLongBlock)
k_truss_peel_long(const int32_t *__restrict__ long_queue, const int *__restrict__ long_size, int k,
                  const int64_t *__restrict__ base, int64_t n, const eid_t *__restrict__ off,
                  const vid_t *__restrict__ nbr, const int32_t *__restrict__ eid, const uint8_t *__restrict__ gone,
                  const uint8_t *__restrict__ in_curr, int *__restrict__ sup, int32_t *__restrict__ next,
                  int *__restrict__ nsize) {
    const int count = *long_size;
    for (int i = blockIdx.x; i < count; i += gridDim.x) {
        const int32_t e = long_queue[i];
        vid_t a, b;
        edge_ends(e, base, n, off, nbr, a, b);
        peel_edge<kLongBlock>(e, a, b, threadIdx.x, k, off, nbr, eid, gone, in_curr, sup, next, nsize);
    }
}

}  // namespace

void truss_numbers(Graph &g, int32_t *out, int64_t *m_out) {
    GMSB_REQUIRE(!g.directed, "truss_numbers: graph must be undirected");
    Runtime &r = rt();
    const int64_t n = g.n;
    int64_t m = 0;
    DevBuf<int64_t> base;
    upper_edge_base(g, base, &m);
    GMSB_REQUIRE(m < (int64_t(1) << 31), "truss_numbers: edge ids are int32, the graph has too many edges");
    if (m_out) *m_out = m;
    if (!out || m == 0) return;

    DevBuf<int32_t> eid(g.slots), truss(m), qa(m), qb(m);
    DevBuf<uint32_t> support(m);
    DevBuf<uint8_t> gone(m), in_curr(m);
    DevBuf<unsigned long long> nlong(1);
    DevBuf<int> ctr(4);                   // [0], [1]: sizes of the two queues, [2]: long-row queue, [3]: least support > k
    gone.zero();
    in_curr.zero();
    nlong.zero();
    k_slot_edge_ids<<<grid_for(n * 32, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, n, base.p, eid.p, nlong.p);
    launched();
    edge_support(g, base.p, support.p);
    // signed from here on: a decrement below the level is undone, and must read as <= k while it is in flight
    int *sup = reinterpret_cast<int *>(support.p);
    const int64_t n_long = (int64_t)nlong.get(0);
    DevBuf<int32_t> ql(n_long);
    const int long_grid = (int)std::min<int64_t>(n_long, (int64_t)r.sm_count * 8);

    int64_t done = 0;
    for (int k = 0; done < m;) {
        const int init[4] = {0, 0, 0, INT_MAX};
        ctr.upload(init, 4);
        k_truss_collect<<<grid_for(m, 256), 256, 0, r.stream>>>(m, k, sup, gone.p, qa.p, ctr.p, ctr.p + 3); launched();
        int h[4];
        ctr.download(h, 4);
        if (h[0] == 0) {                               // empty level: jump to the least live support
            GMSB_REQUIRE(h[3] != INT_MAX, "truss_numbers: no progress");
            k = h[3];
            continue;
        }
        int32_t *cur = qa.p, *nxt = qb.p;
        int *cs = ctr.p, *ns = ctr.p + 1;
        for (int qs = h[0]; qs;) {
            k_truss_mark<<<grid_for(qs, 256), 256, 0, r.stream>>>(cur, qs, in_curr.p); launched();
            GMSB_CUDA(cudaMemsetAsync(ns, 0, sizeof(int), r.stream));
            GMSB_CUDA(cudaMemsetAsync(ctr.p + 2, 0, sizeof(int), r.stream));
            k_truss_peel<<<grid_for((int64_t)qs * 32, 256), 256, 0, r.stream>>>(cur, qs, k, base.p, n, g.off.p, g.nbr.p,
                                                                               eid.p, gone.p, in_curr.p, sup, nxt, ns,
                                                                               ql.p, ctr.p + 2);
            launched();
            if (n_long) {
                k_truss_peel_long<<<long_grid, kLongBlock, 0, r.stream>>>(ql.p, ctr.p + 2, k, base.p, n, g.off.p,
                                                                          g.nbr.p, eid.p, gone.p, in_curr.p, sup, nxt,
                                                                          ns);
                launched();
            }
            k_truss_retire<<<grid_for(qs, 256), 256, 0, r.stream>>>(cur, qs, k, gone.p, in_curr.p, truss.p); launched();
            done += qs;
            std::swap(cur, nxt);
            std::swap(cs, ns);
            GMSB_CUDA(cudaMemcpyAsync(&qs, cs, sizeof(int), cudaMemcpyDeviceToHost, r.stream));
            GMSB_CUDA(cudaStreamSynchronize(r.stream));
        }
        ++k;
    }
    truss.download(out, m);
}

}  // namespace gmsb
