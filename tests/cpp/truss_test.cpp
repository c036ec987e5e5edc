// C++ facade test for core and truss numbers (gms_b200::core_numbers / truss_numbers) on closed forms and a generated
// graph.  Exit code 0 = all checks passed; 3 = no usable CUDA device (loud failure).
#include <algorithm>
#include <cstdio>
#include <stdexcept>
#include <vector>

#include <gms_b200/cuda_set_graph.hpp>

#define EXPECT(cond)                                                             \
    do {                                                                         \
        if (!(cond)) { std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); return 1; } \
    } while (0)

using gms_b200::CudaSetGraph;
using gms_b200::NodeId;

static CudaSetGraph from_pairs(const std::vector<std::pair<int, int>> &el) {
    std::vector<NodeId> s, d;
    for (auto &e : el) { s.push_back(e.first); d.push_back(e.second); }
    return CudaSetGraph::FromEdgeList(s.data(), d.data(), (int64_t)s.size(), true);
}

static bool all_equal(const std::vector<int32_t> &v, int32_t x) {
    return std::all_of(v.begin(), v.end(), [x](int32_t y) { return y == x; });
}

static int run() {
    // K6: every edge has truss 6, every vertex core 5
    std::vector<std::pair<int, int>> k6;
    for (int i = 0; i < 6; ++i) for (int j = i + 1; j < 6; ++j) k6.push_back({i, j});
    CudaSetGraph k = from_pairs(k6);
    auto kt = gms_b200::truss_numbers(k);
    EXPECT(kt.size() == 15 && all_equal(kt, 6));
    EXPECT(all_equal(gms_b200::core_numbers(k), 5));
    // two K5 joined by the edge 4-5: the bridge (edge id 10 in CSR order u<v) has truss 2, the rest 5; core 4
    std::vector<std::pair<int, int>> two;
    for (int i = 0; i < 5; ++i) for (int j = i + 1; j < 5; ++j) { two.push_back({i, j}); two.push_back({i + 5, j + 5}); }
    two.push_back({4, 5});
    auto tt = gms_b200::truss_numbers(from_pairs(two));
    EXPECT(tt.size() == 21);
    for (size_t e = 0; e < tt.size(); ++e) EXPECT(tt[e] == (e == 10 ? 2 : 5));
    // triangles_3 (testing/testGraphs): vertex 4 is isolated, core 0
    CudaSetGraph t3 = from_pairs({{0, 1}, {0, 2}, {1, 2}, {1, 3}, {2, 3}, {5, 6}, {5, 7}, {6, 7}, {6, 8}, {7, 9}, {8, 9}});
    EXPECT((gms_b200::core_numbers(t3) == std::vector<int32_t>{2, 2, 2, 2, 0, 2, 2, 2, 2, 2}));
    EXPECT((gms_b200::truss_numbers(t3) == std::vector<int32_t>{3, 3, 3, 3, 3, 3, 3, 3, 2, 2, 2}));
    // kronecker-12: degeneracy 65, max truss 47 (networkx gives the same)
    CudaSetGraph kron = CudaSetGraph::Kronecker(12);
    auto kc = gms_b200::core_numbers(kron);
    auto ktr = gms_b200::truss_numbers(kron);
    EXPECT(*std::max_element(kc.begin(), kc.end()) == 65);
    EXPECT(ktr.size() == 48386 && *std::max_element(ktr.begin(), ktr.end()) == 47);
    // a directed handle is refused (GMSB_ERR_INVALID -> std::invalid_argument)
    bool thrown = false;
    std::vector<int64_t> off = {0, 1, 1};
    std::vector<NodeId> nbr = {1};
    try { gms_b200::truss_numbers(CudaSetGraph::FromCSR(2, off.data(), nbr.data(), true)); }
    catch (const std::invalid_argument &) { thrown = true; }
    EXPECT(thrown);
    std::printf("truss_test: all checks passed\n");
    return 0;
}

int main() {
    try {
        return run();
    } catch (const gms_b200::Error &e) {
        std::fprintf(stderr, "gms-b200 error %d: %s\n", e.code, e.what());
        return e.code == GMSB_ERR_CUDA ? 3 : 1;
    } catch (const std::exception &e) {
        std::fprintf(stderr, "exception: %s\n", e.what());
        return 1;
    }
}
