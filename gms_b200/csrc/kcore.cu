// kcore.cu — degeneracy ordering and core numbers by parallel k-core peeling.
//
// Replaces  PpSequential::getDegeneracyOrderingDanischHeap   gms/algorithms/preprocessing/sequential/degeneracy_danisch.h:12-56
//
// The reference pops one minimum-degree vertex at a time from a heap (O(m log n), sequential) and its tie-breaking
// is not reproducible (testing/preprocessing.cpp:6-7).  Here all vertices whose residual degree is <= k leave
// together, their neighbours' degrees drop with atomics, and vertices that fall to <= k join the same level's next
// frontier.  The result is a valid degeneracy order by the reference's own verifier
// (verifiers/degeneracy_verifier.h:69-85: every vertex has at most `degeneracy` neighbours that are removed after
// it), in the reference's ranking convention: the r-th removed vertex (r = 1..n) gets rank n - r.
#include "common.cuh"
#include "sort.cuh"
#include "isect.cuh"
#include "ops.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

namespace gmsb {

namespace {

__global__ void k_init_degrees(const eid_t *__restrict__ off, int64_t n, int *__restrict__ deg) {
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x)
        deg[v] = (int)(off[v + 1] - off[v]);
}

// frontier of level k: every live vertex with residual degree <= k
__global__ void k_collect(int64_t n, int k, const int *__restrict__ deg, int *__restrict__ gone,
                          vid_t *__restrict__ queue, int *__restrict__ qsize) {
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x)
        if (!gone[v] && deg[v] <= k) {
            gone[v] = 1;
            queue[atomicAdd(qsize, 1)] = (vid_t)v;
        }
}

// removal rank (when rank != nullptr) and core number (when core != nullptr) of the frontier's vertices
__global__ void k_assign_level(const vid_t *__restrict__ queue, int qs, int64_t n, int64_t done, int k,
                               vid_t *__restrict__ rank, int32_t *__restrict__ core) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < qs; i += gridDim.x * blockDim.x) {
        if (rank) rank[queue[i]] = (vid_t)(n - 1 - (done + i));
        if (core) core[queue[i]] = k;
    }
}

// one warp per frontier vertex: decrement live neighbours; those that reach <= k join the next frontier
__global__ void k_relax(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const vid_t *__restrict__ queue,
                        int qs, int k, int *__restrict__ deg, int *__restrict__ gone, vid_t *__restrict__ next,
                        int *__restrict__ nsize) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < qs; i += nwarps) {
        const vid_t v = queue[i];
        for (eid_t e = off[v] + lane; e < off[v + 1]; e += 32) {
            const vid_t w = nbr[e];
            if (gone[w]) continue;
            const int old = atomicSub(&deg[w], 1);
            if (old - 1 <= k && atomicExch(&gone[w], 1) == 0) next[atomicAdd(nsize, 1)] = w;
        }
    }
}

}  // namespace

// The level-by-level peel.  A vertex that leaves at level k has core number k: after level k-1 has drained, every
// remaining vertex has residual degree >= k, so the remaining graph is the k-core.  Writes the removal rank and/or
// the core number of every vertex (device arrays; either may be null).
static void peel_levels(Graph &g, vid_t *rank, int32_t *core) {
    Runtime &r = rt();
    const int64_t n = g.n;
    DevBuf<int> deg(n), gone(n), sizes(2);
    DevBuf<vid_t> qa(n), qb(n);
    gone.zero();
    k_init_degrees<<<grid_for(n, 256), 256, 0, r.stream>>>(g.off.p, n, deg.p); launched();
    int64_t done = 0;
    for (int k = 0; done < n; ++k) {
        sizes.zero();
        k_collect<<<grid_for(n, 256), 256, 0, r.stream>>>(n, k, deg.p, gone.p, qa.p, sizes.p); launched();
        vid_t *cur = qa.p, *nxt = qb.p;
        int *cs = sizes.p, *ns = sizes.p + 1;
        for (;;) {
            int qs = 0;
            GMSB_CUDA(cudaMemcpyAsync(&qs, cs, sizeof(int), cudaMemcpyDeviceToHost, r.stream));
            GMSB_CUDA(cudaStreamSynchronize(r.stream));
            if (qs == 0) break;
            k_assign_level<<<grid_for(qs, 256), 256, 0, r.stream>>>(cur, qs, n, done, k, rank, core); launched();
            done += qs;
            GMSB_CUDA(cudaMemsetAsync(ns, 0, sizeof(int), r.stream));
            k_relax<<<grid_for((int64_t)qs * 32, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, cur, qs, k, deg.p, gone.p,
                                                                           nxt, ns);
            launched();
            std::swap(cur, nxt);
            std::swap(cs, ns);
        }
    }
}

void degeneracy_rank(Graph &g, vid_t *out_rank) {
    GMSB_REQUIRE(!g.directed, "order_degeneracy: graph must be undirected");
    const int64_t n = g.n;
    if (n == 0) return;
    GMSB_REQUIRE(n < (int64_t(1) << 31), "order_degeneracy: too many vertices");
    DevBuf<vid_t> rank(n);
    peel_levels(g, rank.p, nullptr);
    rank.download(out_rank, n);
}

void core_numbers(Graph &g, int32_t *out_core) {
    GMSB_REQUIRE(!g.directed, "core_numbers: graph must be undirected");
    const int64_t n = g.n;
    if (n == 0) return;
    GMSB_REQUIRE(n < (int64_t(1) << 31), "core_numbers: too many vertices");
    DevBuf<int32_t> core(n);
    peel_levels(g, nullptr, core.p);
    core.download(out_core, n);
}

// ---- approximate degeneracy order (ADG) ---------------------------------------------------------------------------------
// Replaces  PpParallel::getDegeneracyOrderingApproxCGraph<boundary_function::averageDegree, useRankFormat>
//           gms/algorithms/preprocessing/parallel/degeneracy_approx_csr.h:13-78, boundary_function.h:15-25
// Every round removes ALL vertices whose residual degree is <= (1+eps) * average residual degree, ordered inside the
// round by that degree (ties by id here; the reference's parallel partition + sort leave ties unspecified), and
// decrements the degrees of their neighbours.  O(log n) rounds; a (2+2eps)-approximation of the degeneracy order.
namespace {
__global__ void k_live_degree_sum(int64_t n, const int *__restrict__ deg, const int *__restrict__ gone,
                                  unsigned long long *__restrict__ acc /* [0]=sum [1]=count */) {
    unsigned long long s = 0, c = 0;
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x)
        if (!gone[v]) { s += (unsigned long long)deg[v]; c++; }
    s = warp_sum(s); c = warp_sum(c);
    if ((threadIdx.x & 31) == 0 && c) { atomicAdd(&acc[0], s); atomicAdd(&acc[1], c); }
}
__global__ void k_collect_keys(int64_t n, unsigned int border, const int *__restrict__ deg, int *__restrict__ gone,
                               uint64_t *__restrict__ keys, int *__restrict__ qsize) {
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x)
        if (!gone[v] && (long long)deg[v] <= (long long)border) {
            gone[v] = 1;
            keys[atomicAdd(qsize, 1)] = ((uint64_t)(uint32_t)deg[v] << 32) | (uint32_t)v;
        }
}
__global__ void k_adg_assign(const uint64_t *__restrict__ sorted, int qs, int64_t done, int rank_format,
                             vid_t *__restrict__ out, vid_t *__restrict__ queue) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < qs; i += gridDim.x * blockDim.x) {
        const vid_t v = (vid_t)(uint32_t)sorted[i];
        queue[i] = v;
        if (rank_format) out[v] = (vid_t)(done + i); else out[done + i] = v;
    }
}
// PUSH-style update: every neighbour's counter drops, removed or not (degeneracy_approx_csr.h:62-66)
__global__ void k_adg_relax(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const vid_t *__restrict__ queue,
                            int qs, int *__restrict__ deg) {
    const int lane = threadIdx.x & 31;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < qs; i += nwarps) {
        const vid_t v = queue[i];
        for (eid_t e = off[v] + lane; e < off[v + 1]; e += 32) atomicSub(&deg[nbr[e]], 1);
    }
}
}  // namespace

namespace {
// live[i] for the vertices that are still in the graph, ascending (the reference's vArray after its partition)
__global__ void k_collect_live(int64_t n, const int *__restrict__ gone, vid_t *__restrict__ live, int *__restrict__ nlive) {
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x)
        if (!gone[v]) live[atomicAdd(nlive, 1)] = (vid_t)v;
}
__global__ void k_live_degree_min(int64_t n, const int *__restrict__ deg, const int *__restrict__ gone, int *__restrict__ mn) {
    int m = 0x7fffffff;
    for (int64_t v = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; v < n; v += (int64_t)gridDim.x * blockDim.x)
        if (!gone[v]) m = min(m, deg[v]);
    for (int o = 16; o; o >>= 1) m = min(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMin(mn, m);
}
__global__ void k_gather_degrees(const vid_t *__restrict__ live, const int *__restrict__ picks, int npick,
                                 const int *__restrict__ deg, int *__restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < npick; i += gridDim.x * blockDim.x) out[i] = deg[live[picks[i]]];
}
// PULL-style update (degeneracy_approx_set.h:73-78): every remaining vertex v subtracts |N(v) ∩ X| where X is the set
// removed in this round — the hot path's intersect_count with one shared right-hand set.  One warp per remaining
// vertex; X is ascending; galloping when one side is much shorter, else merge path (isect.cuh).
__global__ void __launch_bounds__(256)
k_adg_pull(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const vid_t *__restrict__ live, int nlive,
           const int *__restrict__ gone, const vid_t *__restrict__ X, int nx, int *__restrict__ deg) {
    __shared__ vid_t stage[8][kMergeTile + 2];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int nwarps = (gridDim.x * blockDim.x) >> 5;
    for (int i = warp; i < nlive; i += nwarps) {
        const vid_t v = live[i];
        if (gone[v]) continue;                         // removed in this round: it is in X itself
        const eid_t b = off[v];
        const int dv = (int)(off[v + 1] - b);
        if (dv == 0) continue;
        const unsigned long long c = warp_sum(warp_intersect_count(nbr + b, dv, X, nx, lane, stage[wib]));
        if (lane == 0 && c) deg[v] -= (int)c;
    }
}
__global__ void k_low_ids(const uint64_t *__restrict__ sorted, int qs, vid_t *__restrict__ out) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < qs; i += gridDim.x * blockDim.x) out[i] = (vid_t)(uint32_t)sorted[i];
}
inline uint64_t wyrand_next(uint64_t &s) {           // gms/third_party/fast_statistics.h:92-97
    s += 0xa0761d6478bd642full;
    __uint128_t t = (__uint128_t)s * (s ^ 0xe7037ed1a0b428dbull);
    return (uint64_t)(t >> 64) ^ (uint64_t)t;
}
}  // namespace

// Replaces  PpParallel::getDegeneracyOrderingApprox{CGraph,SGraph}<boundary, useRankFormat>
//           gms/algorithms/preprocessing/parallel/degeneracy_approx_csr.h:13-78 (push), degeneracy_approx_set.h:14-85 (pull),
//           boundary_function.h:15-91 (averageDegree, minDegree, probMinDegree, probMedianDegree)
// boundary: 0 average, 1 min, 2 sampled min, 3 sampled median.  The two sampled rules draw their vertices with WyRand
// like the reference, which seeds it from the clock and the OpenMP thread number (not reproducible there); here the
// stream starts from `seed`, so a call is repeatable.  pull != 0 runs the Set form of the update.
void degeneracy_order_approx_ex(Graph &g, double epsilon, bool rank_format, int boundary, bool pull, uint64_t seed,
                                vid_t *out_host) {
    GMSB_REQUIRE(!g.directed, "order_degeneracy_approx: graph must be undirected");
    GMSB_REQUIRE(epsilon >= 0, "order_degeneracy_approx: epsilon must be non-negative");
    GMSB_REQUIRE(boundary >= 0 && boundary <= 3, "order_degeneracy_approx: unknown boundary function");
    Runtime &r = rt();
    const int64_t n = g.n;
    if (n == 0) return;
    GMSB_REQUIRE(n < (int64_t(1) << 31), "order_degeneracy_approx: too many vertices");
    DevBuf<int> deg(n), gone(n), qsize(1), nlive(1), mn(1);
    DevBuf<vid_t> out(n), queue(n), live(n), X(n);
    DevBuf<uint64_t> keys(n), alt(n);
    DevBuf<unsigned long long> acc(2);
    gone.zero();
    k_init_degrees<<<grid_for(n, 256), 256, 0, r.stream>>>(g.off.p, n, deg.p); launched();
    uint64_t rng = seed;
    int64_t done = 0;
    while (done < n) {
        acc.zero(); qsize.zero();
        const int64_t remaining = n - done;
        const bool need_live = pull || boundary >= 2;
        int h_live = 0;
        if (need_live) {
            nlive.zero();
            k_collect_live<<<grid_for(n, 256), 256, 0, r.stream>>>(n, gone.p, live.p, nlive.p); launched();
            h_live = nlive.get(0);
            // atomics fill the list in arbitrary order: make it ascending (the sampled rules index into it)
            if (h_live > 1) {
                size_t bytes = 0;
                GMSB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, live.p, queue.p, h_live, 0, bits_for((uint64_t)n), r.stream));
                DevBuf<uint8_t> tmp(bytes);
                GMSB_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, bytes, live.p, queue.p, h_live, 0, bits_for((uint64_t)n), r.stream));
                GMSB_CUDA(cudaMemcpyAsync(live.p, queue.p, sizeof(vid_t) * (size_t)h_live, cudaMemcpyDeviceToDevice, r.stream));
                r.launches += 4;
                GMSB_CUDA(cudaStreamSynchronize(r.stream));
            }
        }
        unsigned int border = 0;
        if (boundary == 0) {
            k_live_degree_sum<<<grid_for(n, 256), 256, 0, r.stream>>>(n, deg.p, gone.p, acc.p); launched();
            unsigned long long h[2];
            acc.download(h, 2);
            border = (unsigned int)((1 + epsilon) * ((double)(long long)h[0] / (double)h[1]));     // boundary_function.h:15-25
        } else if (boundary == 1) {
            const int big = 0x7fffffff;
            GMSB_CUDA(cudaMemcpyAsync(mn.p, &big, sizeof(int), cudaMemcpyHostToDevice, r.stream));
            k_live_degree_min<<<grid_for(n, 256), 256, 0, r.stream>>>(n, deg.p, gone.p, mn.p); launched();
            border = (unsigned int)(2 * (1 + epsilon) * mn.get(0));                                   // :27-35
        } else {
            // :37-91 — size <= 3 special cases, else max(4, size^(0.5 (0.001 + 1 - eps))) draws
            std::vector<int> picks;
            const int size = (int)remaining;
            if (size <= 3) { for (int i = 0; i < size; ++i) picks.push_back(i); }
            else {
                const int trials = std::max(4, (int)std::pow((double)size, 0.5 * (0.001 + (1 - epsilon))));
                for (int i = 0; i < trials; ++i)
                    picks.push_back((int)(((uint64_t)(uint32_t)wyrand_next(rng) * (uint64_t)(uint32_t)size) >> 32));   // fastrange32
            }
            DevBuf<int> dp((size_t)picks.size()), dd((size_t)picks.size());
            dp.upload(picks.data(), picks.size());
            k_gather_degrees<<<grid_for((int64_t)picks.size(), 256), 256, 0, r.stream>>>(live.p, dp.p, (int)picks.size(),
                                                                                        deg.p, dd.p);
            launched();
            std::vector<int> draws(picks.size());
            dd.download(draws.data(), draws.size());
            std::sort(draws.begin(), draws.end());
            if (boundary == 2) border = (unsigned int)draws.front();
            else border = (unsigned int)(size <= 2 ? draws.front() : (size == 3 ? draws[1] : draws[draws.size() / 2]));
            // the sampled rules may pick a border below every remaining counter's ... no: the border IS some
            // remaining vertex's counter, so at least that vertex leaves and the loop makes progress
        }
        k_collect_keys<<<grid_for(n, 256), 256, 0, r.stream>>>(n, border, deg.p, gone.p, keys.p, qsize.p); launched();
        const int qs = qsize.get(0);
        GMSB_REQUIRE(qs > 0, "order_degeneracy_approx: no progress");
        uint64_t *sorted = radix_sort_keys(keys.p, alt.p, qs, 0, 64);
        k_adg_assign<<<grid_for(qs, 256), 256, 0, r.stream>>>(sorted, qs, done, rank_format ? 1 : 0, out.p, queue.p);
        launched();
        if (!pull) {
            k_adg_relax<<<grid_for((int64_t)qs * 32, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, queue.p, qs, deg.p);
            launched();
        } else if (qs < h_live) {
            // X = this round's batch as an ascending set (Set X(start_index, mid), :59)
            size_t bytes = 0;
            GMSB_CUDA(cub::DeviceRadixSort::SortKeys(nullptr, bytes, queue.p, X.p, qs, 0, bits_for((uint64_t)n), r.stream));
            DevBuf<uint8_t> tmp(bytes);
            GMSB_CUDA(cub::DeviceRadixSort::SortKeys(tmp.p, bytes, queue.p, X.p, qs, 0, bits_for((uint64_t)n), r.stream));
            r.launches += 4;
            const int grid = (int)std::min<int64_t>(ceil_div(h_live, 8), (int64_t)r.sm_count * 16);
            k_adg_pull<<<grid, 256, 0, r.stream>>>(g.off.p, g.nbr.p, live.p, h_live, gone.p, X.p, qs, deg.p); launched();
            GMSB_CUDA(cudaStreamSynchronize(r.stream));
        }
        done += qs;
    }
    out.download(out_host, n);
}

void degeneracy_order_approx(Graph &g, double epsilon, bool rank_format, vid_t *out_host) {
    GMSB_REQUIRE(!g.directed, "order_degeneracy_approx: graph must be undirected");
    GMSB_REQUIRE(epsilon >= 0, "order_degeneracy_approx: epsilon must be non-negative");
    Runtime &r = rt();
    const int64_t n = g.n;
    if (n == 0) return;
    GMSB_REQUIRE(n < (int64_t(1) << 31), "order_degeneracy_approx: too many vertices");
    DevBuf<int> deg(n), gone(n), qsize(1);
    DevBuf<vid_t> out(n), queue(n);
    DevBuf<uint64_t> keys(n), alt(n);
    DevBuf<unsigned long long> acc(2);
    gone.zero();
    k_init_degrees<<<grid_for(n, 256), 256, 0, r.stream>>>(g.off.p, n, deg.p); launched();
    int64_t done = 0;
    while (done < n) {
        acc.zero(); qsize.zero();
        k_live_degree_sum<<<grid_for(n, 256), 256, 0, r.stream>>>(n, deg.p, gone.p, acc.p); launched();
        unsigned long long h[2];
        acc.download(h, 2);
        const double res = (double)(long long)h[0];
        const unsigned int border = (unsigned int)((1 + epsilon) * (res / (double)h[1]));   // boundary_function.h:24
        k_collect_keys<<<grid_for(n, 256), 256, 0, r.stream>>>(n, border, deg.p, gone.p, keys.p, qsize.p); launched();
        const int qs = qsize.get(0);
        GMSB_REQUIRE(qs > 0, "order_degeneracy_approx: no progress");
        uint64_t *sorted = radix_sort_keys(keys.p, alt.p, qs, 0, 64);
        k_adg_assign<<<grid_for(qs, 256), 256, 0, r.stream>>>(sorted, qs, done, rank_format ? 1 : 0, out.p, queue.p);
        launched();
        k_adg_relax<<<grid_for((int64_t)qs * 32, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, queue.p, qs, deg.p);
        launched();
        done += qs;
    }
    out.download(out_host, n);
}

}  // namespace gmsb
