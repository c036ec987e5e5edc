// capi.cu — the extern "C" boundary declared in include/gmsb.h.  Every entry point catches C++ exceptions,
// records the message for gmsb_last_error() and maps it to a negative status; nothing here computes on the CPU.
#include "common.cuh"
#include "orient.cuh"
#include "ops.cuh"
#include "sets.cuh"

#include <algorithm>
#include <cstring>
#include <mutex>
#include <random>
#include <unordered_map>
#include <vector>

namespace gmsb {

namespace {
thread_local std::string g_last_error;
// One Runtime per device.  A host thread works on its bound device (bind_device: the workers of the multi-GPU entry
// points, mgpu.cu) or, by default, on the process's primary device (gmsb_set_device).
constexpr int kMaxDevices = 64;
Runtime g_rts[kMaxDevices];
bool g_rt_ready[kMaxDevices] = {};
int g_device = 0;
thread_local int t_device = -1;
std::mutex g_rt_mutex;
}  // namespace

void set_last_error(const std::string &msg) { g_last_error = msg; }
const std::string &last_error_message() { return g_last_error; }

int current_device() { return t_device >= 0 ? t_device : g_device; }
void bind_device(int device) {
    t_device = device;
    if (device >= 0) cudaSetDevice(device);
}

Runtime &rt() {
    const int dev = current_device();
    if (dev < 0 || dev >= kMaxDevices) throw Error(GMSB_ERR_INVALID, "device index out of range");
    if (!g_rt_ready[dev]) {
        std::lock_guard<std::mutex> lock(g_rt_mutex);
        if (!g_rt_ready[dev]) {
            int count = 0;
            cudaError_t e = cudaGetDeviceCount(&count);
            if (e != cudaSuccess || count == 0)
                throw Error(GMSB_ERR_CUDA, std::string("no usable CUDA device (") +
                                               (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                               "); gms-b200 has no CPU fallback");
            GMSB_REQUIRE(dev < count, "device index beyond the visible devices");
            GMSB_CUDA(cudaSetDevice(dev));
            cudaDeviceProp prop{};
            GMSB_CUDA(cudaGetDeviceProperties(&prop, dev));
            g_rts[dev].device = dev;
            g_rts[dev].sm_count = prop.multiProcessorCount;
            g_rts[dev].smem_optin = prop.sharedMemPerBlockOptin;
            g_rt_ready[dev] = true;
        }
    }
    return g_rts[dev];
}

// ---- caching device arena ------------------------------------------------------------------------------------------
// Free lists are kept per device: a block cached by one device is never handed to a kernel on another one.
namespace {
std::mutex g_arena_mutex;
std::unordered_map<size_t, std::vector<void *>> g_arena_free[kMaxDevices];     // size class -> cached blocks
struct LiveBlock { size_t cls; int device; };
std::unordered_map<void *, LiveBlock> g_arena_live;                            // block -> size class, owner device

// classes are spaced 12.5 % apart (and at least 512 B), so a block is at most 1/8 larger than requested
size_t arena_class(size_t bytes) {
    if (bytes <= 512) return 512;
    int top = 63 - __builtin_clzll((unsigned long long)bytes);
    size_t step = size_t(1) << (top > 3 ? top - 3 : 0);
    if (step < 512) step = 512;
    return (bytes + step - 1) / step * step;
}
}  // namespace

void *arena_alloc(size_t bytes) {
    const int dev = rt().device;
    const size_t cls = arena_class(bytes);
    std::lock_guard<std::mutex> lock(g_arena_mutex);
    auto &bin = g_arena_free[dev][cls];
    void *p = nullptr;
    if (!bin.empty()) {
        p = bin.back();
        bin.pop_back();
    } else {
        cudaSetDevice(dev);
        cudaError_t e = cudaMalloc(&p, cls);
        if (e == cudaErrorMemoryAllocation) {           // give this device's cache back and retry once
            cudaGetLastError();
            for (auto &kv : g_arena_free[dev]) { for (void *q : kv.second) cudaFree(q); kv.second.clear(); }
            e = cudaMalloc(&p, cls);
        }
        if (e != cudaSuccess)
            throw Error(e == cudaErrorMemoryAllocation ? GMSB_ERR_OOM : GMSB_ERR_CUDA,
                        std::string("cudaMalloc(") + std::to_string(cls) + " bytes): " + cudaGetErrorString(e));
    }
    g_arena_live[p] = LiveBlock{cls, dev};
    return p;
}

void arena_free(void *p) {
    std::lock_guard<std::mutex> lock(g_arena_mutex);
    auto it = g_arena_live.find(p);
    if (it == g_arena_live.end()) return;
    g_arena_free[it->second.device][it->second.cls].push_back(p);
    g_arena_live.erase(it);
}

void arena_trim() {
    std::lock_guard<std::mutex> lock(g_arena_mutex);
    int prev = 0;
    cudaGetDevice(&prev);
    for (int dev = 0; dev < kMaxDevices; ++dev) {
        if (g_arena_free[dev].empty()) continue;
        cudaSetDevice(dev);
        cudaDeviceSynchronize();
        for (auto &kv : g_arena_free[dev]) { for (void *q : kv.second) cudaFree(q); kv.second.clear(); }
    }
    cudaSetDevice(prev);
}

template <typename F>
int guarded(F &&f) {
    try {
        f();
        return GMSB_OK;
    } catch (const Error &e) {
        set_last_error(e.what());
        return e.code;
    } catch (const std::bad_alloc &) {
        set_last_error("host allocation failed");
        return GMSB_ERR_OOM;
    } catch (const std::exception &e) {
        set_last_error(e.what());
        return GMSB_ERR_INVALID;
    }
}

// any handle: entry points that work on the oriented representation alone (or on the handle's metadata)
inline Graph &Gdag(gmsb_graph_t h) {
    GMSB_REQUIRE(h != nullptr, "null graph handle");
    return *reinterpret_cast<Graph *>(h);
}
// handles with complete symmetric lists: everything else
inline Graph &G(gmsb_graph_t h) {
    Graph &g = Gdag(h);
    GMSB_REQUIRE(!g.dag_only, "this handle comes from a sharded build and holds the oriented representation only "
                              "(triangle counts); build it with gmsb_graph_from_csr for the other operators");
    return g;
}

}  // namespace gmsb

using namespace gmsb;

extern "C" {

GMSB_API const char *gmsb_last_error(void) { return g_last_error.c_str(); }
GMSB_API int gmsb_version(void) { return 100; }

GMSB_API int gmsb_device_count(int *count) {
    return guarded([&] {
        GMSB_REQUIRE(count, "null argument");
        cudaError_t e = cudaGetDeviceCount(count);
        if (e != cudaSuccess) { *count = 0; throw Error(GMSB_ERR_CUDA, cudaGetErrorString(e)); }
    });
}

GMSB_API int gmsb_set_device(int device) {
    return guarded([&] {
        GMSB_REQUIRE(device >= 0 && device < kMaxDevices, "bad device index");
        g_device = device;
        t_device = -1;
        GMSB_CUDA(cudaSetDevice(device));
        rt();
    });
}

GMSB_API int gmsb_set_devices(int n, const int *ids) {
    return guarded([&] {
        mg_set_devices(n, ids);
        g_device = ids[0];
        t_device = -1;
        GMSB_CUDA(cudaSetDevice(ids[0]));
        rt();
    });
}
GMSB_API int gmsb_tc_total_multi(gmsb_graph_t g, uint64_t *out) { return guarded([&] { mg_tc_total(G(g), out); }); }
GMSB_API int gmsb_tc_vertex2_multi(gmsb_graph_t g, int64_t *out_n) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(out_n || gr.n == 0, "null output");
        mg_tc_vertex2(gr, out_n);
    });
}
GMSB_API int gmsb_kclique_count_multi(gmsb_graph_t g, int k, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out && k >= 1, "kclique_count: bad arguments");
        mg_kclique_count(G(g), k, out);
    });
}
GMSB_API int gmsb_edge_similarity_multi(gmsb_graph_t g, int metric, double *out, int64_t *m_out) {
    return guarded([&] {
        GMSB_REQUIRE(metric >= 0 && metric <= GMSB_SIM_PREF_ATT, "invalid similarity measure");
        mg_edge_similarity(G(g), metric, out, m_out);
    });
}

GMSB_API int gmsb_set_stream(void *s) {
    return guarded([&] {
        GMSB_CUDA(cudaStreamSynchronize(rt().stream));     // pool memory freed on the old stream must be quiescent
        rt().stream = reinterpret_cast<cudaStream_t>(s);
    });
}
GMSB_API int gmsb_trim_memory(void) { return guarded([&] { arena_trim(); }); }
GMSB_API int gmsb_synchronize(void) { return guarded([&] { GMSB_CUDA(cudaStreamSynchronize(rt().stream)); }); }
GMSB_API int gmsb_launch_count(uint64_t *count) {
    return guarded([&] {
        GMSB_REQUIRE(count, "null argument");
        uint64_t total = 0;                      // over all devices this process has used
        for (int d = 0; d < kMaxDevices; ++d) if (g_rt_ready[d]) total += g_rts[d].launches;
        *count = total;
    });
}

// ---- generators (host) -----------------------------------------------------------------------------------------
GMSB_API int gmsb_generate_rmat(int scale, int64_t m, float a, float b, float c, int permute, int32_t *src,
                                int32_t *dst) {
    return guarded([&] { generate_rmat(scale, m, a, b, c, permute != 0, src, dst); });
}
GMSB_API int gmsb_generate_uniform(int scale, int64_t m, int32_t *src, int32_t *dst) {
    return guarded([&] { generate_uniform(scale, m, src, dst); });
}

// ---- graphs ----------------------------------------------------------------------------------------------------
GMSB_API int gmsb_graph_from_csr(int64_t n, const int64_t *off, const int32_t *nbr, int directed, gmsb_graph_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        *out = reinterpret_cast<gmsb_graph_t>(graph_from_csr_device(n, off, nbr, directed != 0, true));
    });
}
GMSB_API int gmsb_graph_from_csr_ex(int64_t n, const int64_t *off, const int32_t *nbr, int directed, int flags,
                                    gmsb_graph_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        GMSB_REQUIRE((flags & ~GMSB_BUILD_ORIENT) == 0, "graph_from_csr_ex: unknown flag");
        if ((flags & GMSB_BUILD_ORIENT) && !directed)
            *out = reinterpret_cast<gmsb_graph_t>(graph_from_csr_host_pipelined(n, off, nbr));
        else
            *out = reinterpret_cast<gmsb_graph_t>(graph_from_csr_device(n, off, nbr, directed != 0, true));
    });
}
GMSB_API int gmsb_graph_from_csr_device(int64_t n, const int64_t *off, const int32_t *nbr, int directed, gmsb_graph_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        *out = reinterpret_cast<gmsb_graph_t>(graph_from_csr_device(n, off, nbr, directed != 0, false));
    });
}
// sharded construction of the oriented representation (graph_build.cu: shard_*)
GMSB_API int gmsb_shard_begin(int64_t n, const int64_t *off, const int32_t *nbr, const int64_t *off_dev, int part_index,
                              int part_count, gmsb_shard_t *out, int64_t *piece_len) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        *out = reinterpret_cast<gmsb_shard_t>(shard_begin(n, off, nbr, off_dev, part_index, part_count, piece_len));
    });
}
GMSB_API int gmsb_shard_export(gmsb_shard_t s, int32_t *piece_dev, int32_t *dplus_all_dev) {
    return guarded([&] {
        GMSB_REQUIRE(s, "null shard handle");
        shard_export(*reinterpret_cast<Shard *>(s), piece_dev, dplus_all_dev);
    });
}
GMSB_API int gmsb_shard_finish(gmsb_shard_t s, const int32_t *pieces_dev, int64_t piece_stride, const int32_t *dplus_all_dev,
                               gmsb_graph_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(s && out, "null handle");
        *out = reinterpret_cast<gmsb_graph_t>(shard_finish(*reinterpret_cast<Shard *>(s), pieces_dev, piece_stride,
                                                           dplus_all_dev));
    });
}
GMSB_API int gmsb_shard_free(gmsb_shard_t s) { return guarded([&] { delete reinterpret_cast<Shard *>(s); }); }
GMSB_API int gmsb_graph_from_edgelist(int64_t m, const int32_t *src, const int32_t *dst, int symmetrize, gmsb_graph_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        GMSB_REQUIRE(m >= 0 && (m == 0 || (src && dst)), "graph_from_edgelist: bad arguments");
        DevBuf<vid_t> s(m), d(m);
        s.upload(src, m);
        d.upload(dst, m);
        *out = reinterpret_cast<gmsb_graph_t>(graph_from_edgelist_device(m, s.p, d.p, symmetrize != 0));
    });
}
GMSB_API int gmsb_graph_from_edgelist_device(int64_t m, const int32_t *src, const int32_t *dst, int symmetrize,
                                    gmsb_graph_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        *out = reinterpret_cast<gmsb_graph_t>(graph_from_edgelist_device(m, src, dst, symmetrize != 0));
    });
}
GMSB_API int gmsb_graph_relabel_by_degree(gmsb_graph_t g, gmsb_graph_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        *out = reinterpret_cast<gmsb_graph_t>(graph_relabel_by_degree(G(g)));
    });
}
GMSB_API int gmsb_graph_num_nodes(gmsb_graph_t g, int64_t *n) {
    return guarded([&] { GMSB_REQUIRE(n, "null argument"); *n = Gdag(g).n; });
}
GMSB_API int gmsb_graph_num_slots(gmsb_graph_t g, int64_t *s) {
    return guarded([&] { GMSB_REQUIRE(s, "null argument"); *s = Gdag(g).slots; });
}
GMSB_API int gmsb_graph_is_directed(gmsb_graph_t g, int *d) {
    return guarded([&] { GMSB_REQUIRE(d, "null argument"); *d = Gdag(g).directed ? 1 : 0; });
}
GMSB_API int gmsb_graph_export_csr(gmsb_graph_t g, int64_t *off, int32_t *nbr) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(off && (nbr || gr.slots == 0), "null output");
        gr.off.download(off, gr.n + 1);
        gr.nbr.download(nbr, gr.slots);
    });
}
GMSB_API int gmsb_graph_free(gmsb_graph_t g) {
    return guarded([&] { delete reinterpret_cast<Graph *>(g); });
}

// ---- orderings -----------------------------------------------------------------------------------------------------
GMSB_API int gmsb_order_degree(gmsb_graph_t g, int rank_format, int32_t *out) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(out || gr.n == 0, "null output");
        DevBuf<vid_t> order, rank;
        degree_order(gr, order, rank);
        (rank_format ? rank : order).download(out, gr.n);
    });
}
GMSB_API int gmsb_order_degeneracy(gmsb_graph_t g, int32_t *out_rank) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(out_rank || gr.n == 0, "null output");
        degeneracy_rank(gr, out_rank);
    });
}
GMSB_API int gmsb_core_numbers(gmsb_graph_t g, int32_t *out_n) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(out_n || gr.n == 0, "null output");
        core_numbers(gr, out_n);
    });
}
GMSB_API int gmsb_truss_numbers(gmsb_graph_t g, int32_t *out, int64_t *m_out) {
    return guarded([&] { truss_numbers(G(g), out, m_out); });
}
GMSB_API int gmsb_order_degeneracy_approx(gmsb_graph_t g, double epsilon, int rank_format, int32_t *out) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(out || gr.n == 0, "null output");
        degeneracy_order_approx(gr, epsilon, rank_format != 0, out);
    });
}
GMSB_API int gmsb_order_degeneracy_approx_ex(gmsb_graph_t g, double epsilon, int rank_format, int boundary, int pull,
                                             uint64_t seed, int32_t *out) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(out || gr.n == 0, "null output");
        degeneracy_order_approx_ex(gr, epsilon, rank_format != 0, boundary, pull != 0, seed, out);
    });
}
GMSB_API int gmsb_graph_worth_relabelling(gmsb_graph_t g, int *out) {
    return guarded([&] {
        Graph &gr = G(g);
        GMSB_REQUIRE(out, "null output");
        // host-side heuristic on the degree array (gapbs/benchmark.h:158-176); same libstdc++ RNG stream as the reference
        *out = 0;
        const int64_t n = gr.n;
        if (n == 0 || (gr.directed ? gr.slots : gr.slots / 2) / n < 10) return;      // CSRGraph::num_edges() / num_nodes()
        std::vector<eid_t> off(n + 1);
        gr.off.download(off.data(), n + 1);
        std::mt19937 rng(27491095);
        std::uniform_int_distribution<vid_t> pick(0, (vid_t)(n - 1));
        const int64_t ns = std::min<int64_t>(1000, n);
        std::vector<int64_t> s(ns);
        int64_t total = 0;
        for (int64_t t = 0; t < ns; ++t) {
            vid_t v;
            do { v = pick(rng); } while (off[v + 1] == off[v]);
            s[t] = off[v + 1] - off[v];
            total += s[t];
        }
        std::sort(s.begin(), s.end());
        const double avg = static_cast<double>(total) / ns, med = static_cast<double>(s[ns / 2]);
        *out = avg / 1.3 > med ? 1 : 0;
    });
}
GMSB_API int gmsb_orient(gmsb_graph_t g, const int32_t *ranking, gmsb_graph_t *dag) {
    return guarded([&] {
        GMSB_REQUIRE(dag, "null output handle");
        *dag = reinterpret_cast<gmsb_graph_t>(induce_directed(G(g), ranking));
    });
}

// ---- triangles -------------------------------------------------------------------------------------------------------
GMSB_API int gmsb_tc_total_ex(gmsb_graph_t g, const gmsb_tc_options *opt, uint64_t *out, gmsb_tc_stats *stats) {
    return guarded([&] {
        gmsb_tc_options o{};
        if (opt) o = *opt;
        tc_total(Gdag(g), o, out, stats);
    });
}
GMSB_API int gmsb_tc_total(gmsb_graph_t g, uint64_t *out) {
    gmsb_tc_options o{};
    o.reuse_plan = 1;
    return gmsb_tc_total_ex(g, &o, out, nullptr);
}
GMSB_API int gmsb_tc_vertex2(gmsb_graph_t g, int64_t *out_n) {
    return guarded([&] {
        Graph &gr = Gdag(g);
        GMSB_REQUIRE(out_n || gr.n == 0, "null output");
        tc_vertex2(gr, out_n);
    });
}

// ---- set algebra / similarity --------------------------------------------------------------------------------------------
GMSB_API int gmsb_intersect_count_batch(gmsb_graph_t g, int64_t np, const int32_t *a, const int32_t *b, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(np >= 0 && (np == 0 || (a && b && out)), "intersect_count_batch: bad arguments");
        intersect_count_batch(G(g), np, a, b, out);
    });
}
GMSB_API int gmsb_intersect_batch(gmsb_graph_t g, int64_t np, const int32_t *a, const int32_t *b, int64_t *out_offsets,
                         int32_t *out_elems, int64_t cap) {
    return guarded([&] {
        GMSB_REQUIRE(np >= 0 && out_offsets && (np == 0 || (a && b)), "intersect_batch: bad arguments");
        intersect_batch(G(g), np, a, b, out_offsets, out_elems, cap);
    });
}
GMSB_API int gmsb_difference_batch(gmsb_graph_t g, int64_t np, const int32_t *a, const int32_t *b, int64_t *out_offsets,
                                   int32_t *out_elems, int64_t cap) {
    return guarded([&] {
        GMSB_REQUIRE(np >= 0 && out_offsets && (np == 0 || (a && b)), "difference_batch: bad arguments");
        difference_batch(G(g), np, a, b, out_offsets, out_elems, cap);
    });
}
GMSB_API int gmsb_union_batch(gmsb_graph_t g, int64_t np, const int32_t *a, const int32_t *b, int64_t *out_offsets,
                              int32_t *out_elems, int64_t cap) {
    return guarded([&] {
        GMSB_REQUIRE(np >= 0 && out_offsets && (np == 0 || (a && b)), "union_batch: bad arguments");
        union_batch(G(g), np, a, b, out_offsets, out_elems, cap);
    });
}
GMSB_API int gmsb_union_count_batch(gmsb_graph_t g, int64_t np, const int32_t *a, const int32_t *b, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(np >= 0 && (np == 0 || (a && b && out)), "union_count_batch: bad arguments");
        union_count_batch(G(g), np, a, b, out);
    });
}
GMSB_API int gmsb_pair_similarity(gmsb_graph_t g, int metric, int64_t np, const int32_t *a, const int32_t *b, double *out) {
    return guarded([&] {
        GMSB_REQUIRE(np >= 0 && (np == 0 || (a && b && out)), "pair_similarity: bad arguments");
        GMSB_REQUIRE(metric >= 0 && metric <= GMSB_SIM_PREF_ATT, "invalid similarity measure");
        pair_similarity(G(g), metric, np, a, b, out);
    });
}
GMSB_API int gmsb_edge_similarity(gmsb_graph_t g, int metric, double *out, int64_t *m_out) {
    return guarded([&] {
        GMSB_REQUIRE(metric >= 0 && metric <= GMSB_SIM_PREF_ATT, "invalid similarity measure");
        edge_similarity(G(g), metric, out, m_out);
    });
}

// ---- device-resident sets -------------------------------------------------------------------------------------------------
namespace {
inline DevSet &S(gmsb_set_t h) {
    GMSB_REQUIRE(h != nullptr, "null set handle");
    return *reinterpret_cast<DevSet *>(h);
}
inline gmsb_set_op_kind check_op(int op) {
    GMSB_REQUIRE(op >= GMSB_SET_INTERSECT && op <= GMSB_SET_DIFFERENCE, "unknown set operation");
    return static_cast<gmsb_set_op_kind>(op);
}
}  // namespace
GMSB_API int gmsb_set_from_host(const int32_t *elems, int64_t count, gmsb_set_t *out) {
    return guarded([&] { GMSB_REQUIRE(out, "null output handle"); rt(); *out = reinterpret_cast<gmsb_set_t>(set_from_host(elems, count)); });
}
GMSB_API int gmsb_set_range(int64_t bound, gmsb_set_t *out) {
    return guarded([&] { GMSB_REQUIRE(out, "null output handle"); *out = reinterpret_cast<gmsb_set_t>(set_range(bound)); });
}
GMSB_API int gmsb_set_neighbourhood(gmsb_graph_t g, int32_t v, gmsb_set_t *out) {
    return guarded([&] { GMSB_REQUIRE(out, "null output handle"); *out = reinterpret_cast<gmsb_set_t>(set_neighbourhood(G(g), v)); });
}
GMSB_API int gmsb_set_clone(gmsb_set_t a, gmsb_set_t *out) {
    return guarded([&] { GMSB_REQUIRE(out, "null output handle"); *out = reinterpret_cast<gmsb_set_t>(set_clone(S(a))); });
}
GMSB_API int gmsb_set_free(gmsb_set_t a) { return guarded([&] { delete reinterpret_cast<DevSet *>(a); }); }
GMSB_API int gmsb_set_cardinality(gmsb_set_t a, int64_t *n) {
    return guarded([&] { GMSB_REQUIRE(n, "null argument"); *n = S(a).n; });
}
GMSB_API int gmsb_set_to_host(gmsb_set_t a, int32_t *out) { return guarded([&] { set_to_host(S(a), out); }); }
GMSB_API int gmsb_set_contains(gmsb_set_t a, int32_t x, int *flag) {
    return guarded([&] { GMSB_REQUIRE(flag, "null argument"); *flag = set_contains(S(a), x) ? 1 : 0; });
}
GMSB_API int gmsb_set_add(gmsb_set_t a, int32_t x) { return guarded([&] { set_add(S(a), x); }); }
GMSB_API int gmsb_set_remove(gmsb_set_t a, int32_t x) { return guarded([&] { set_remove(S(a), x); }); }
GMSB_API int gmsb_set_equal(gmsb_set_t a, gmsb_set_t b, int *flag) {
    return guarded([&] { GMSB_REQUIRE(flag, "null argument"); *flag = set_equal(S(a), S(b)) ? 1 : 0; });
}
GMSB_API int gmsb_set_op(int op, gmsb_set_t a, gmsb_set_t b, gmsb_set_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output handle");
        const gmsb_set_op_kind kind = check_op(op);
        DevSet *bs[1] = {&S(b)}, *res[1] = {nullptr};
        set_op_many(kind, S(a), 1, bs, res);
        *out = reinterpret_cast<gmsb_set_t>(res[0]);
    });
}
GMSB_API int gmsb_set_op_inplace(int op, gmsb_set_t a, gmsb_set_t b) {
    return guarded([&] {
        const gmsb_set_op_kind kind = check_op(op);
        DevSet *bs[1] = {&S(b)}, *res[1] = {nullptr};
        set_op_many(kind, S(a), 1, bs, res);
        DevSet &dst = S(a);
        dst.own = std::move(res[0]->own);
        dst.p = dst.own.p;
        dst.n = res[0]->n;
        delete res[0];
    });
}
GMSB_API int gmsb_set_op_count(int op, gmsb_set_t a, gmsb_set_t b, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out, "null output");
        const gmsb_set_op_kind kind = check_op(op);
        DevSet *bs[1] = {&S(b)};
        set_op_count_many(kind, S(a), 1, bs, out);
    });
}
GMSB_API int gmsb_set_op_count_many(int op, gmsb_set_t a, int64_t count, const gmsb_set_t *bs, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(count >= 0 && (count == 0 || (bs && out)), "set_op_count_many: bad arguments");
        const gmsb_set_op_kind kind = check_op(op);
        set_op_count_many(kind, S(a), count, reinterpret_cast<DevSet *const *>(bs), out);
    });
}
GMSB_API int gmsb_set_op_many(int op, gmsb_set_t a, int64_t count, const gmsb_set_t *bs, gmsb_set_t *outs) {
    return guarded([&] {
        GMSB_REQUIRE(count >= 0 && (count == 0 || (bs && outs)), "set_op_many: bad arguments");
        const gmsb_set_op_kind kind = check_op(op);
        set_op_many(kind, S(a), count, reinterpret_cast<DevSet *const *>(bs), reinterpret_cast<DevSet **>(outs));
    });
}
GMSB_API int gmsb_set_op_count_neighbourhoods(int op, gmsb_set_t a, gmsb_graph_t g, gmsb_set_t members, uint64_t *out) {
    return guarded([&] {
        const gmsb_set_op_kind kind = check_op(op);
        GMSB_REQUIRE(out || S(members).n == 0, "null output");
        set_op_count_members(kind, S(a), G(g), S(members), out);
    });
}

// ---- cliques -----------------------------------------------------------------------------------------------------------------
GMSB_API int gmsb_kclique_count(gmsb_graph_t g, int k, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out && k >= 1, "kclique_count: bad arguments");
        kclique_count(G(g), k, out);
    });
}
GMSB_API int gmsb_kclique_count_ex(gmsb_graph_t g, int k, int part_index, int part_count, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out && k >= 1, "kclique_count: bad arguments");
        kclique_count(G(g), k, out, part_index, part_count <= 0 ? 1 : part_count);
    });
}
GMSB_API int gmsb_kclique_count_ordered(gmsb_graph_t g, int k, uint64_t *out) {
    return guarded([&] {
        GMSB_REQUIRE(out && k >= 1, "kclique_count_ordered: bad arguments");
        kclique_count_ordered(G(g), k, out);
    });
}

}  // extern "C"
