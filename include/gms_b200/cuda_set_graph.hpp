// cuda_set_graph.hpp — C++ host facade over the C ABI (include/gmsb.h).
//
// CudaSetGraph models the reference's SGraph concept (gms/representations/graphs/set_graph.h:87-118: `FromCGraph`,
// `num_nodes`, `out_degree`, `out_neigh`) for the algorithms of the set-intersection hot path, but the
// neighbourhoods live in HBM and the set algebra runs in batched CUDA kernels.  There is no host implementation of
// intersect / intersect_count here on purpose: this library has no CPU fallback.
//
// Like SetGraph<Set> it is move-only; use clone() for a copy (set_graph.h:28-39).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdlib>
#include <iostream>
#include <stdexcept>
#include <string>
#include <utility>
#include <vector>

#include "../gmsb.h"

namespace gms_b200 {

using NodeId = int32_t;          // gms/common/types.h:9

struct Error : std::runtime_error {
    int code;
    Error(int c, const std::string &msg) : std::runtime_error(msg), code(c) {}
};

inline void check(int code) {
    if (code == GMSB_OK) return;
    // the reference reports a directed input to InduceDirectedGraph with std::invalid_argument (apply_order.h:14-16)
    if (code == GMSB_ERR_INVALID) throw std::invalid_argument(gmsb_last_error());
    throw Error(code, gmsb_last_error());
}

// Read-only view of one neighbourhood in the host mirror: iteration and size, for callers such as verifiers.
class NeighborhoodView {
public:
    using SetElement = NodeId;
    NeighborhoodView(const NodeId *b, const NodeId *e) : b_(b), e_(e) {}
    const NodeId *begin() const { return b_; }
    const NodeId *end() const { return e_; }
    size_t cardinality() const { return static_cast<size_t>(e_ - b_); }
private:
    const NodeId *b_, *e_;
};

enum class Metric { Jaccard, Overlap, AdamicAdar, Resource, CommNeigh, TotalNeigh, PrefAtt };   // vertex_similarity.h:18

class CudaSetGraph {
public:
    using Set = NeighborhoodView;
    using SetElement = NodeId;

    CudaSetGraph() = default;
    explicit CudaSetGraph(gmsb_graph_t h) : h_(h) {}
    CudaSetGraph(CudaSetGraph &&o) noexcept { swap(o); }
    CudaSetGraph &operator=(CudaSetGraph &&o) noexcept { if (this != &o) { release(); swap(o); } return *this; }
    CudaSetGraph(const CudaSetGraph &) = delete;
    CudaSetGraph &operator=(const CudaSetGraph &) = delete;
    ~CudaSetGraph() { release(); }

    // SetGraph<Set>::FromCGraph (set_graph.h:87-89): any graph type with num_nodes(), out_degree(u), out_neigh(u)
    // and directed(); the lists must be ascending and duplicate-free, as Builder::SquishGraph leaves them.
    // RemoveIsolated = true mirrors cgraph_to_neighborhoods_remove_isolated (set_graph.h:190-232): vertices without
    // neighbours are dropped, the others keep their order and are renumbered 0..n'-1 (and the reference's notice is
    // printed); per-vertex results are then indexed by the new ids, exactly as in the reference.
    template <class CGraph, bool RemoveIsolated = false>
    static CudaSetGraph FromCGraph(const CGraph &g) {
        const int64_t n = g.num_nodes();
        std::vector<NodeId> label;
        int64_t isolated = 0;
        if (RemoveIsolated) {
            label.resize(static_cast<size_t>(n));
            for (int64_t u = 0; u < n; ++u) {
                if (g.out_degree(static_cast<NodeId>(u)) == 0) { label[u] = -1; ++isolated; }
                else label[u] = static_cast<NodeId>(u - isolated);
            }
        }
        const bool relabel = RemoveIsolated && isolated > 0;
        const int64_t kept = n - isolated;
        std::vector<int64_t> off(static_cast<size_t>(kept) + 1, 0);
        for (int64_t u = 0, k = 0; u < n; ++u) {
            if (relabel && label[u] < 0) continue;
            off[k + 1] = off[k] + static_cast<int64_t>(g.out_degree(static_cast<NodeId>(u)));
            ++k;
        }
        std::vector<NodeId> nbr(static_cast<size_t>(off[kept]));
        for (int64_t u = 0, k = 0; u < n; ++u) {
            if (relabel && label[u] < 0) continue;
            int64_t p = off[k++];
            for (NodeId v : g.out_neigh(static_cast<NodeId>(u))) nbr[p++] = relabel ? label[v] : v;
        }
        if (relabel)
            std::cout << "Removed " << isolated
                      << " isolated vertices from the graph, the graph got relabeled and shrunk!" << std::endl;
        return FromCSR(kept, off.data(), nbr.data(), g.directed());
    }
    // SetGraph<Set>::FromEL (set_graph.h:54-78): neighbourhood of u = the second entries of the pairs whose first is u;
    // the list is sorted in place unless is_sorted, and — like the reference — NOT symmetrised.  The device handle
    // needs to know whether the result is symmetric (SetGraph::directed() computes that on demand, set_graph.h:128-137).
    template <class EL>
    static CudaSetGraph FromEL(EL &edge_list, size_t num_nodes, bool is_sorted) {
        if (!is_sorted) std::sort(edge_list.begin(), edge_list.end());
        std::vector<int64_t> off(num_nodes + 1, 0);
        std::vector<NodeId> nbr;
        nbr.reserve(edge_list.size());
        auto it = edge_list.begin();
        for (size_t u = 0; u < num_nodes; ++u) {
            while (it != edge_list.end() && static_cast<size_t>(it->first) == u) { nbr.push_back(it->second); ++it; }
            off[u + 1] = static_cast<int64_t>(nbr.size());
        }
        bool directed = false;
        for (size_t u = 0; u < num_nodes && !directed; ++u)
            for (int64_t p = off[u]; p < off[u + 1] && !directed; ++p) {
                const NodeId v = nbr[p];
                directed = !std::binary_search(nbr.begin() + off[v], nbr.begin() + off[v + 1], static_cast<NodeId>(u));
            }
        return FromCSR(static_cast<int64_t>(num_nodes), off.data(), nbr.data(), directed);
    }
    static CudaSetGraph FromCSR(int64_t n, const int64_t *offsets, const NodeId *nbrs, bool directed = false) {
        gmsb_graph_t h = nullptr;
        check(gmsb_graph_from_csr(n, offsets, nbrs, directed ? 1 : 0, &h));
        return CudaSetGraph(h);
    }
    // Builder::MakeGraphFromEL + SquishGraph on the GPU (gapbs/builder.h:279-298,237-251)
    static CudaSetGraph FromEdgeList(const NodeId *src, const NodeId *dst, int64_t m, bool symmetrize = true) {
        gmsb_graph_t h = nullptr;
        check(gmsb_graph_from_edgelist(m, src, dst, symmetrize ? 1 : 0, &h));
        return CudaSetGraph(h);
    }
    // Generator + Builder::MakeGraph for `-g kronecker <scale> --deg <degree>` (cli/cli.h:83-118)
    static CudaSetGraph Kronecker(int scale, int degree = 16, float a = 0.57f, float b = 0.19f, float c = 0.19f) {
        const int64_t m = (int64_t(1) << scale) * degree;
        std::vector<NodeId> s(static_cast<size_t>(m)), d(static_cast<size_t>(m));
        check(gmsb_generate_rmat(scale, m, a, b, c, 1, s.data(), d.data()));
        return FromEdgeList(s.data(), d.data(), m, true);
    }

    CudaSetGraph clone() const {
        ensure_mirror();
        return FromCSR(num_nodes(), off_.data(), nbr_.data(), directed());
    }
    CudaSetGraph RelabelByDegree() const {       // Builder::RelabelByDegree (gapbs/builder.h:1699-1735)
        gmsb_graph_t h = nullptr;
        check(gmsb_graph_relabel_by_degree(h_, &h));
        return CudaSetGraph(h);
    }

    int64_t num_nodes() const { int64_t n = 0; check(gmsb_graph_num_nodes(h_, &n)); return n; }
    int64_t num_edges() const { int64_t s = slots(); return directed() ? s : s / 2; }
    int64_t num_edges_directed() const { return slots(); }
    bool directed() const { int d = 0; check(gmsb_graph_is_directed(h_, &d)); return d != 0; }
    int64_t out_degree(NodeId v) const { ensure_mirror(); return off_[v + 1] - off_[v]; }
    NeighborhoodView out_neigh(NodeId v) const {
        ensure_mirror();
        return NeighborhoodView(nbr_.data() + off_[v], nbr_.data() + off_[v + 1]);
    }
    gmsb_graph_t handle() const { return h_; }

    // ---- batched Set algebra on the device (SortedSet::intersect_count / intersect, sorted_set.h:160-182)
    std::vector<uint64_t> intersect_count(const std::vector<NodeId> &a, const std::vector<NodeId> &b) const {
        if (a.size() != b.size()) throw std::invalid_argument("intersect_count: pair arrays differ in length");
        std::vector<uint64_t> out(a.size());
        check(gmsb_intersect_count_batch(h_, static_cast<int64_t>(a.size()), a.data(), b.data(), out.data()));
        return out;
    }
    // returns (offsets, elements): the intersection of pair i is elements[offsets[i] .. offsets[i+1])
    std::pair<std::vector<int64_t>, std::vector<NodeId>> intersect(const std::vector<NodeId> &a,
                                                                   const std::vector<NodeId> &b) const {
        if (a.size() != b.size()) throw std::invalid_argument("intersect: pair arrays differ in length");
        const int64_t np = static_cast<int64_t>(a.size());
        std::vector<int64_t> off(a.size() + 1);
        check(gmsb_intersect_batch(h_, np, a.data(), b.data(), off.data(), nullptr, 0));
        std::vector<NodeId> el(static_cast<size_t>(off[np]));
        check(gmsb_intersect_batch(h_, np, a.data(), b.data(), off.data(), el.data(), off[np]));
        return {std::move(off), std::move(el)};
    }
    // N(a[i]) \ N(b[i]) and N(a[i]) ∪ N(b[i]) (SortedSet::difference / union_with, sorted_set.h:184-189,104-109), same layout
    std::pair<std::vector<int64_t>, std::vector<NodeId>> difference(const std::vector<NodeId> &a,
                                                                    const std::vector<NodeId> &b) const {
        return two_pass(&gmsb_difference_batch, "difference", a, b);
    }
    std::pair<std::vector<int64_t>, std::vector<NodeId>> union_with(const std::vector<NodeId> &a,
                                                                    const std::vector<NodeId> &b) const {
        return two_pass(&gmsb_union_batch, "union_with", a, b);
    }
    std::vector<uint64_t> union_count(const std::vector<NodeId> &a, const std::vector<NodeId> &b) const {   // :140
        if (a.size() != b.size()) throw std::invalid_argument("union_count: pair arrays differ in length");
        std::vector<uint64_t> out(a.size());
        check(gmsb_union_count_batch(h_, static_cast<int64_t>(a.size()), a.data(), b.data(), out.data()));
        return out;
    }

private:
    gmsb_graph_t h_ = nullptr;
    mutable std::vector<int64_t> off_;
    mutable std::vector<NodeId> nbr_;
    mutable bool mirrored_ = false;

    using BatchFn = int (*)(gmsb_graph_t, int64_t, const int32_t *, const int32_t *, int64_t *, int32_t *, int64_t);
    std::pair<std::vector<int64_t>, std::vector<NodeId>> two_pass(BatchFn fn, const char *what, const std::vector<NodeId> &a,
                                                                  const std::vector<NodeId> &b) const {
        if (a.size() != b.size()) throw std::invalid_argument(std::string(what) + ": pair arrays differ in length");
        const int64_t np = static_cast<int64_t>(a.size());
        std::vector<int64_t> off(a.size() + 1);
        check(fn(h_, np, a.data(), b.data(), off.data(), nullptr, 0));
        std::vector<NodeId> el(static_cast<size_t>(off[np]));
        check(fn(h_, np, a.data(), b.data(), off.data(), el.data(), off[np]));
        return {std::move(off), std::move(el)};
    }
    int64_t slots() const { int64_t s = 0; check(gmsb_graph_num_slots(h_, &s)); return s; }
    void release() { if (h_) gmsb_graph_free(h_); h_ = nullptr; mirrored_ = false; }
    void swap(CudaSetGraph &o) {
        std::swap(h_, o.h_); off_.swap(o.off_); nbr_.swap(o.nbr_); std::swap(mirrored_, o.mirrored_);
    }
    void ensure_mirror() const {
        if (mirrored_) return;
        off_.assign(static_cast<size_t>(num_nodes()) + 1, 0);
        nbr_.assign(static_cast<size_t>(std::max<int64_t>(slots(), 1)), 0);
        check(gmsb_graph_export_csr(h_, off_.data(), nbr_.data()));
        mirrored_ = true;
    }
};

// ---- several GPUs in one process -----------------------------------------------------------------------------------
// UseDevices({0,1,...,7}) once (or the environment variable GMSB_DEVICES="0,1,2,3", read by UseDevicesFromEnv): the
// entry points below then spread every call over those devices (gmsb_*_multi: CSR replicated over NVLink, partitioned
// kernels, NCCL all-reduce for array results).  Handles live on the first listed device.
inline int &multi_device_count() { static int n = 0; return n; }
inline void UseDevices(const std::vector<int> &ids) {
    check(gmsb_set_devices(static_cast<int>(ids.size()), ids.data()));
    multi_device_count() = static_cast<int>(ids.size());
}
inline bool UseDevicesFromEnv() {
    const char *e = std::getenv("GMSB_DEVICES");
    if (!e || !*e) return false;
    std::vector<int> ids;
    for (const char *p = e; *p;) {
        ids.push_back(std::atoi(p));
        while (*p && *p != ',') ++p;
        if (*p == ',') ++p;
    }
    UseDevices(ids);
    return true;
}

// ---- algorithm entry points, plain names (gms_api.hpp maps the reference's names onto these) ---------------------
inline size_t count_total(const CudaSetGraph &g) {
    uint64_t t = 0;
    check(multi_device_count() > 1 ? gmsb_tc_total_multi(g.handle(), &t) : gmsb_tc_total(g.handle(), &t));
    return static_cast<size_t>(t);
}
template <class Output = std::vector<int64_t>>
inline void vertex_count2(const CudaSetGraph &g, Output &counts) {
    const int64_t n = g.num_nodes();
    counts.resize(n);
    std::vector<int64_t> tmp(static_cast<size_t>(std::max<int64_t>(n, 1)));
    check(multi_device_count() > 1 ? gmsb_tc_vertex2_multi(g.handle(), tmp.data()) : gmsb_tc_vertex2(g.handle(), tmp.data()));
    for (int64_t i = 0; i < n; ++i) counts[i] = tmp[i];
}
template <bool useRankFormat = false, class Output = std::vector<NodeId>>
inline void degree_ordering(const CudaSetGraph &g, Output &res) {
    const int64_t n = g.num_nodes();
    res.resize(n);
    std::vector<NodeId> tmp(static_cast<size_t>(std::max<int64_t>(n, 1)));
    check(gmsb_order_degree(g.handle(), useRankFormat ? 1 : 0, tmp.data()));
    for (int64_t i = 0; i < n; ++i) res[i] = tmp[i];
}
template <class Output = std::vector<NodeId>>
inline void degeneracy_ordering(const CudaSetGraph &g, Output &ranking) {
    const int64_t n = g.num_nodes();
    ranking.resize(n);
    std::vector<NodeId> tmp(static_cast<size_t>(std::max<int64_t>(n, 1)));
    check(gmsb_order_degeneracy(g.handle(), tmp.data()));
    for (int64_t i = 0; i < n; ++i) ranking[i] = tmp[i];
}
// core number of every vertex (the largest k whose k-core holds it); the maximum is the degeneracy
inline std::vector<int32_t> core_numbers(const CudaSetGraph &g) {
    std::vector<int32_t> out(static_cast<size_t>(g.num_nodes()));
    check(gmsb_core_numbers(g.handle(), out.data()));
    return out;
}
// truss number of every undirected edge u<v, in the edge order of edge_similarity
inline std::vector<int32_t> truss_numbers(const CudaSetGraph &g) {
    int64_t cnt = 0;
    check(gmsb_truss_numbers(g.handle(), nullptr, &cnt));
    std::vector<int32_t> out(static_cast<size_t>(cnt));
    if (cnt) check(gmsb_truss_numbers(g.handle(), out.data(), &cnt));
    return out;
}
// approximate degeneracy order, averageDegree boundary (degeneracy_approx_csr.h:13-78); ascending convention
template <bool useRankFormat = false, class Output = std::vector<NodeId>>
inline void degeneracy_ordering_approx(const CudaSetGraph &g, Output &res, double epsilon) {
    const int64_t n = g.num_nodes();
    res.resize(n);
    std::vector<NodeId> tmp(static_cast<size_t>(std::max<int64_t>(n, 1)));
    check(gmsb_order_degeneracy_approx(g.handle(), epsilon, useRankFormat ? 1 : 0, tmp.data()));
    for (int64_t i = 0; i < n; ++i) res[i] = tmp[i];
}
// the CLI's auto-relabel heuristic (gapbs/benchmark.h:158-176)
inline bool WorthRelabelling(const CudaSetGraph &g) {
    int w = 0;
    check(gmsb_graph_worth_relabelling(g.handle(), &w));
    return w != 0;
}
inline CudaSetGraph induce_directed_graph(const CudaSetGraph &g, const std::vector<NodeId> &ranking) {
    if (static_cast<int64_t>(ranking.size()) != g.num_nodes()) throw std::invalid_argument("ranking has wrong length");
    gmsb_graph_t h = nullptr;
    check(gmsb_orient(g.handle(), ranking.data(), &h));
    return CudaSetGraph(h);
}
inline unsigned long long kclique_count(const CudaSetGraph &g, int clique_size) {
    uint64_t c = 0;
    check(multi_device_count() > 1 ? gmsb_kclique_count_multi(g.handle(), clique_size, &c)
                                   : gmsb_kclique_count(g.handle(), clique_size, &c));
    return c;
}
inline size_t kclique_count_ordered(const CudaSetGraph &g, size_t k) {
    uint64_t c = 0;
    check(gmsb_kclique_count_ordered(g.handle(), static_cast<int>(k), &c));
    return static_cast<size_t>(c);
}
inline std::vector<double> pair_similarity(Metric m, const CudaSetGraph &g, const std::vector<NodeId> &a,
                                           const std::vector<NodeId> &b) {
    if (a.size() != b.size()) throw std::invalid_argument("pair_similarity: pair arrays differ in length");
    std::vector<double> out(a.size());
    check(gmsb_pair_similarity(g.handle(), static_cast<int>(m), static_cast<int64_t>(a.size()), a.data(), b.data(),
                               out.data()));
    return out;
}
// one score per undirected edge u<v in CSR order
inline std::vector<double> edge_similarity(Metric m, const CudaSetGraph &g) {
    int64_t cnt = 0;
    const bool multi = multi_device_count() > 1;
    check(gmsb_edge_similarity(g.handle(), static_cast<int>(m), nullptr, &cnt));
    std::vector<double> out(static_cast<size_t>(cnt));
    if (cnt) check(multi ? gmsb_edge_similarity_multi(g.handle(), static_cast<int>(m), out.data(), &cnt)
                         : gmsb_edge_similarity(g.handle(), static_cast<int>(m), out.data(), &cnt));
    return out;
}

}  // namespace gms_b200
