// tc_support.cu — per-edge triangle support on the degree-oriented DAG, and what is derived from it.
//
// support[e] = number of triangles containing edge e = |N(a) ∩ N(b)| for e = {a,b}.  One pass of the triangle
// schedule (tc.cu) finds every triangle {u<v<w} exactly once and credits its three edges, which replaces
//   TriangleCount::{Seq,Par}::vertex_count2        gms/algorithms/set_based/triangle_count/parallel/vertex.h:15-49
//       counts[x] = 2 t(x) = sum of support over the edges at x
//   VertexSim::vertex_similarity<Jaccard|Overlap|CommNeigh|TotalNeigh|PrefAtt> per edge
//                                                  gms/algorithms/set_based/vertex_similarity/vertex_similarity.h:30-170
//       whose only graph-dependent input is the common-neighbour count of the edge's endpoints
// at the oriented cost (B_TC) instead of one symmetric-list intersection per edge (B_sim, ~12x more at scale 22).
// All accumulation is integer atomics, so results are exact and order-independent.
#include "common.cuh"
#include "sort.cuh"
#include "isect.cuh"
#include "tc_plan.cuh"
#include "ops.cuh"

namespace gmsb {

namespace {

// position of w in the ascending shared-memory copy of N+(v)
__device__ __forceinline__ int smem_pos(const vid_t *nl, int dv, vid_t w) {
    int lo = 0, hi = dv;
    while (lo < hi) {
        int mid = (lo + hi) >> 1;
        if (nl[mid] < w) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// G lanes per descriptor (32 / 8 / 1 as in tc.cu); every hit credits (u,w) in global memory and (v,w) in the
// CTA's shared counters; the descriptor's own edge (u,v) gets the group's hit total.
template <int G>
__device__ __forceinline__ void support_class(const uint64_t *__restrict__ dptr, int lo, int hi, int *ticket,
                                              const vid_t *__restrict__ nbr, const uint32_t *bm, const vid_t *nl,
                                              uint32_t *cn, int dv, uint32_t base, uint32_t cap_words, int lane,
                                              uint32_t *__restrict__ sup) {
    if (lo >= hi) return;
    constexpr int PER = 32 / G;
    for (;;) {
        int d0 = 0;
        if (lane == 0) d0 = atomicAdd(ticket, PER);
        d0 = __shfl_sync(0xffffffffu, d0, 0) + lo;
        if (d0 >= hi) break;
        const int idx = d0 + lane / G, sub = lane % G;
        const uint64_t ds = idx < hi ? dptr[idx] : 0ull;
        const int64_t start = (int64_t)(ds >> kLenBits);
        const vid_t *__restrict__ p = nbr + start;
        const int len = (int)(ds & kLenMask);
        uint32_t hits = 0;
        for (int j = sub; j < len; j += G) {
            const vid_t w = p[j];
            if (probe(bm, (uint32_t)w - base, cap_words)) {
                ++hits;
                atomicAdd(&sup[start + j], 1u);
                atomicAdd(&cn[smem_pos(nl, dv, w)], 1u);
            }
        }
        // reduce inside the G-lane group (all 32 lanes take part in the shuffles)
        for (int o = G >> 1; o; o >>= 1) hits += __shfl_xor_sync(0xffffffffu, hits, o);
        if (sub == 0 && hits) atomicAdd(&sup[start - 1], hits);
    }
}

template <int BLOCK>
__global__ void __launch_bounds__(BLOCK)
k_support_bitmap(const Item *__restrict__ items, int64_t count, uint32_t cap_words,
                 int max_dplus,
                 const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, const uint64_t *__restrict__ desc,
                 uint32_t *__restrict__ sup, unsigned int *__restrict__ ticket) {
    extern __shared__ uint32_t smem[];
    uint32_t *bm = smem;                                        // cap_words + 1
    vid_t *nl = reinterpret_cast<vid_t *>(smem + cap_words + 1);  // max_dplus
    uint32_t *cn = smem + cap_words + 1 + max_dplus;              // max_dplus
    __shared__ unsigned int s_item;
    __shared__ int s_next[3];
    const int tid = threadIdx.x, lane = tid & 31;
    for (uint32_t i = tid; i <= cap_words; i += BLOCK) bm[i] = 0u;
    for (int i = tid; i < max_dplus; i += BLOCK) cn[i] = 0u;
    for (;;) {
        if (tid == 0) { s_item = atomicAdd(ticket, 1u); s_next[0] = 0; s_next[1] = 0; s_next[2] = 0; }
        __syncthreads();
        const int64_t it = (int64_t)s_item;
        if (it >= count) break;
        const Item item = items[it];
        const vid_t v = item.v;
        const eid_t ob = off[v];
        const int dv = (int)(off[v + 1] - ob);
        const uint32_t base = (uint32_t)v + 1u;
        for (int j = tid; j < dv; j += BLOCK) {
            const vid_t w = nbr[ob + j];
            nl[j] = w;
            const uint32_t x = (uint32_t)w - base;
            atomicOr(&bm[x >> 5], 1u << (x & 31));
        }
        __syncthreads();
        const uint64_t *__restrict__ dptr = desc + item.begin;
        support_class<32>(dptr, item.n1, item.count, &s_next[2], nbr, bm, nl, cn, dv, base, cap_words, lane, sup);
        support_class<8>(dptr, item.n0, item.n1, &s_next[1], nbr, bm, nl, cn, dv, base, cap_words, lane, sup);
        support_class<1>(dptr, 0, item.n0, &s_next[0], nbr, bm, nl, cn, dv, base, cap_words, lane, sup);
        __syncthreads();
        for (int j = tid; j < dv; j += BLOCK) {
            bm[((uint32_t)nl[j] - base) >> 5] = 0u;
            const uint32_t c = cn[j];
            if (c) { atomicAdd(&sup[ob + j], c); cn[j] = 0u; }
        }
    }
}

// Light edges: one warp per edge, lanes binary-search elements of the shorter list in the longer one.
__global__ void __launch_bounds__(256)
k_support_light(const uint64_t *__restrict__ desc, const vid_t *__restrict__ vs,
                int64_t count, const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, uint32_t *__restrict__ sup) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t i = warp; i < count; i += nwarps) {
        const uint64_t ds = desc[i];
        const vid_t v = vs[i];
        const int64_t sa = (int64_t)(ds >> kLenBits), sb = off[v];
        const int na = (int)(ds & kLenMask), nb = (int)(off[v + 1] - sb);
        const bool a_short = na <= nb;
        const int64_t ss = a_short ? sa : sb, sl = a_short ? sb : sa;     // short / long list starts
        const int ns = a_short ? na : nb, nl = a_short ? nb : na;
        uint32_t hits = 0;
        for (int j = lane; j < ns; j += 32) {
            const vid_t x = nbr[ss + j];
            const int lo = lower_bound_dev(nbr + sl, nl, x);
            if (lo < nl && nbr[sl + lo] == x) {
                ++hits;
                atomicAdd(&sup[ss + j], 1u);
                atomicAdd(&sup[sl + lo], 1u);
            }
        }
        hits = (uint32_t)warp_sum(hits);
        if (lane == 0 && hits) atomicAdd(&sup[sa - 1], hits);
    }
}

// counts[rank] = sum of support over the out-edges of the vertex (warp per vertex) ...
__global__ void k_vertex_out_sum(const eid_t *__restrict__ off, int64_t n, const uint32_t *__restrict__ sup,
                                 unsigned long long *__restrict__ t2) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t u = warp; u < n; u += nwarps) {
        unsigned long long s = 0;
        for (eid_t e = off[u] + lane; e < off[u + 1]; e += 32) s += sup[e];
        s = warp_sum(s);
        if (lane == 0 && s) atomicAdd(&t2[u], s);
    }
}
// ... plus the support of every in-edge
__global__ void k_vertex_in_sum(const vid_t *__restrict__ nbr, int64_t m, const uint32_t *__restrict__ sup,
                                unsigned long long *__restrict__ t2) {
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < m; e += (int64_t)gridDim.x * blockDim.x) {
        const uint32_t s = sup[e];
        if (s) atomicAdd(&t2[nbr[e]], (unsigned long long)s);
    }
}
__global__ void k_unrank(const unsigned long long *__restrict__ t2, const vid_t *__restrict__ order, int64_t n,
                         int64_t *__restrict__ out) {
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < n; r += (int64_t)gridDim.x * blockDim.x)
        out[order[r]] = (int64_t)t2[r];
}

// support of the undirected edge between rank-space vertices ra and rb, read from its oriented copy
__device__ __forceinline__ uint32_t oriented_support(vid_t ra, vid_t rb, const eid_t *__restrict__ doff,
                                                     const vid_t *__restrict__ dnbr, const uint32_t *__restrict__ sup) {
    const vid_t lo = ra < rb ? ra : rb, hi = ra < rb ? rb : ra;
    const eid_t lb = doff[lo];
    return sup[lb + lower_bound_dev(dnbr + lb, (int)(doff[lo + 1] - lb), hi)];
}

// Score of every undirected edge a<b (CSR order of the ORIGINAL graph) from the support of its oriented copy.
__global__ void k_edge_scores(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t a_begin, int64_t n,
                              const int64_t *__restrict__ base, const vid_t *__restrict__ rank,
                              const eid_t *__restrict__ doff, const vid_t *__restrict__ dnbr,
                              const uint32_t *__restrict__ sup, int metric, double *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t a = a_begin + warp; a < n; a += nwarps) {
        const eid_t e1 = off[a + 1];
        const int64_t c = base[a + 1] - base[a];
        const eid_t s0 = e1 - c;
        const unsigned long long da = (unsigned long long)(e1 - off[a]);
        const vid_t ra = rank[a];
        for (int64_t j = lane; j < c; j += 32) {
            const vid_t b = nbr[s0 + j];
            const unsigned long long db = (unsigned long long)(off[b + 1] - off[b]);
            const unsigned long long cnt = oriented_support(ra, rank[b], doff, dnbr, sup);
            const double cd = (double)cnt;
            double score;
            if (metric == GMSB_SIM_JACCARD) score = (da == 0 && db == 0) ? 1.0 : cd / (double)(da + db + cd);
            else if (metric == GMSB_SIM_OVERLAP) score = cd / (double)(da < db ? da : db);
            else if (metric == GMSB_SIM_COMM_NEIGH) score = cd;
            else if (metric == GMSB_SIM_TOTAL_NEIGH) score = (double)(da + db - cnt);
            else score = (double)(da * db);
            out[base[a] + j] = score;
        }
    }
}

// Support of every undirected edge a<b, indexed like k_edge_scores' output (the edge ids of truss.cu).
__global__ void k_edge_support(const eid_t *__restrict__ off, const vid_t *__restrict__ nbr, int64_t n,
                               const int64_t *__restrict__ base, const vid_t *__restrict__ rank,
                               const eid_t *__restrict__ doff, const vid_t *__restrict__ dnbr,
                               const uint32_t *__restrict__ sup, uint32_t *__restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t warp = (blockIdx.x * (int64_t)blockDim.x + threadIdx.x) >> 5;
    const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t a = warp; a < n; a += nwarps) {
        const int64_t c = base[a + 1] - base[a];
        const eid_t s0 = off[a + 1] - c;
        const vid_t ra = rank[a];
        for (int64_t j = lane; j < c; j += 32) out[base[a] + j] = oriented_support(ra, rank[nbr[s0 + j]], doff, dnbr, sup);
    }
}

}  // namespace

// support of every oriented edge, in the DAG's CSR order (rank space).  part_index / part_count: this device credits
// the triangles of its share of the schedule only (the edges into the vertices it owns, as in tc_total); the shares
// add up to the full support (multi-GPU: one all-reduce, mgpu.cu).
void tc_support(Graph &g, DevBuf<uint32_t> &sup, int pi, int P) {
    Runtime &r = rt();
    gmsb_tc_options opt = normalise_tc_options(nullptr);
    GMSB_REQUIRE(P >= 1 && pi >= 0 && pi < P, "tc_support: bad partition");
    opt.reuse_plan = 1;
    opt.part_index = pi; opt.part_count = P;          // the schedule is built for this device's share
    TcPlan &p = ensure_plan(g, opt);
    Dag &d = *g.dag;
    sup.alloc(d.m);
    sup.zero();
    if (d.m == 0) return;
    const int64_t my_items = p.n_items;
    if (my_items) {
        constexpr int BLOCK = 512;
        auto kern = k_support_bitmap<BLOCK>;
        const size_t smem = ((size_t)p.max_span_words + 1 + 2 * (size_t)p.max_hub_dplus) * 4;   // only hubs are staged
        GMSB_REQUIRE(smem <= r.smem_optin, "tc_support: neighbourhood too large for shared memory");
        if (smem > 48 * 1024)
            GMSB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int resident = 0;
        GMSB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&resident, kern, BLOCK, smem));
        GMSB_REQUIRE(resident >= 1, "tc_support: kernel does not fit on an SM");
        const int grid = (int)std::min<int64_t>(my_items, (int64_t)r.sm_count * resident);
        DevBuf<unsigned int> ticket(1);
        ticket.zero();
        kern<<<grid, BLOCK, smem, r.stream>>>(p.items.p, my_items, (uint32_t)p.max_span_words, p.max_hub_dplus,
                                              d.off.p, d.nbr.p, p.desc.p, sup.p, ticket.p);
        launched();
        GMSB_CUDA(cudaStreamSynchronize(r.stream));
    }
    const int64_t my_merge = p.n_merge, my_gallop = p.n_gallop;
    if (my_merge) {
        int grid = (int)std::min<int64_t>(ceil_div(my_merge, 8), (int64_t)r.sm_count * 16);
        k_support_light<<<grid, 256, 0, r.stream>>>(p.m_desc.p, p.m_v.p, my_merge, d.off.p, d.nbr.p, sup.p);
        launched();
    }
    if (my_gallop) {
        int grid = (int)std::min<int64_t>(ceil_div(my_gallop, 8), (int64_t)r.sm_count * 16);
        k_support_light<<<grid, 256, 0, r.stream>>>(p.g_desc.p, p.g_v.p, my_gallop, d.off.p, d.nbr.p, sup.p);
        launched();
    }
}

// t2[r] += support of the edges at rank-space vertex r (t2 zeroed by the caller); linear in sup
void support_to_vertex2(Graph &g, const uint32_t *sup, unsigned long long *t2) {
    Runtime &r = rt();
    Dag &d = *g.dag;
    if (d.m == 0) return;
    k_vertex_out_sum<<<grid_for(g.n * 32, 256), 256, 0, r.stream>>>(d.off.p, g.n, sup, t2); launched();
    k_vertex_in_sum<<<grid_for(d.m, 256), 256, 0, r.stream>>>(d.nbr.p, d.m, sup, t2); launched();
}
void vertex2_unrank(Graph &g, const unsigned long long *t2, int64_t *out_dev) {
    Runtime &r = rt();
    k_unrank<<<grid_for(g.n, 256), 256, 0, r.stream>>>(t2, g.dag->order.p, g.n, out_dev); launched();
}

void tc_vertex2(Graph &g, int64_t *out_n) {
    GMSB_REQUIRE(!g.directed, "vertex_count2: graph must be undirected");
    const int64_t n = g.n;
    if (n == 0) return;
    DevBuf<uint32_t> sup;
    tc_support(g, sup);
    DevBuf<unsigned long long> t2(n);
    DevBuf<int64_t> out(n);
    t2.zero();
    support_to_vertex2(g, sup.p, t2.p);
    vertex2_unrank(g, t2.p, out.p);
    out.download(out_n, n);
}

// scores of the undirected edges a<b owned by the vertices [a_begin, a_end) from a complete support array
void edge_scores_range(Graph &g, int metric, const int64_t *base_dev, const uint32_t *sup, int64_t a_begin, int64_t a_end,
                       double *out_dev) {
    Runtime &r = rt();
    Dag &d = *g.dag;
    if (a_end <= a_begin) return;
    k_edge_scores<<<grid_for((a_end - a_begin) * 32, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, a_begin, a_end, base_dev,
                                                                             d.rank.p, d.off.p, d.nbr.p, sup, metric,
                                                                             out_dev);
    launched();
}

// triangle support of every undirected edge a<b in edge-id order (out_dev: uint32[m]); `base` as below
void edge_support(Graph &g, const int64_t *base_dev, uint32_t *out_dev) {
    Runtime &r = rt();
    DevBuf<uint32_t> sup;
    tc_support(g, sup);
    Dag &d = *g.dag;
    k_edge_support<<<grid_for(g.n * 32, 256), 256, 0, r.stream>>>(g.off.p, g.nbr.p, g.n, base_dev, d.rank.p, d.off.p,
                                                                d.nbr.p, sup.p, out_dev);
    launched();
}

// edge_similarity for the metrics that depend on the graph only through the common-neighbour count.
// `base` = exclusive scan of the per-vertex count of neighbours > vertex (setops.cu builds it).
void edge_scores_from_support(Graph &g, int metric, const int64_t *base_dev, double *out_dev) {
    DevBuf<uint32_t> sup;
    tc_support(g, sup);
    edge_scores_range(g, metric, base_dev, sup.p, 0, g.n, out_dev);
    GMSB_CUDA(cudaStreamSynchronize(rt().stream));
}

}  // namespace gmsb
