// TEST INFRASTRUCTURE ONLY — the CPU checkers of gmsb_core_numbers and gmsb_truss_numbers, compiled and loaded by
// tests/truss_oracle.py.  Never linked into the product.
//
// Both are sequential bucket peels over a symmetric CSR (ascending, duplicate-free lists, no self loops), written to be
// independent of the GPU algorithm: no frontiers, no levels, no triangle-once rule.  GMS has neither function.
#include <algorithm>
#include <cstdint>
#include <utility>
#include <vector>

namespace {

using vid = int32_t;

struct Csr {
    int64_t n;
    const int64_t *off;
    const vid *nbr;
    int64_t deg(int64_t v) const { return off[v + 1] - off[v]; }
    const vid *begin(int64_t v) const { return nbr + off[v]; }
    const vid *end(int64_t v) const { return nbr + off[v + 1]; }
};

}  // namespace

extern "C" {

// Core number of every vertex.  Batagelj and Zaversnik, "An O(m) algorithm for cores decomposition of networks"
// (2003): vertices in an array sorted by degree with bucket starts; the next vertex is always one of least residual
// degree, and a neighbour of higher degree moves one bucket down by swapping with the first vertex of its bucket.
void tor_core_numbers(int64_t n, const int64_t *off, const int32_t *nbr, int32_t *core) {
    const Csr g{n, off, nbr};
    if (n == 0) return;
    std::vector<int64_t> deg(n), pos(n), vert(n);
    int64_t md = 0;
    for (int64_t v = 0; v < n; ++v) { deg[v] = g.deg(v); md = std::max(md, deg[v]); }
    std::vector<int64_t> bin(md + 1, 0);
    for (int64_t v = 0; v < n; ++v) bin[deg[v]]++;
    for (int64_t d = 0, start = 0; d <= md; ++d) { const int64_t c = bin[d]; bin[d] = start; start += c; }
    for (int64_t v = 0; v < n; ++v) { pos[v] = bin[deg[v]]; vert[pos[v]] = v; bin[deg[v]]++; }
    for (int64_t d = md; d > 0; --d) bin[d] = bin[d - 1];
    bin[0] = 0;
    for (int64_t i = 0; i < n; ++i) {
        const int64_t v = vert[i];
        for (const vid *p = g.begin(v); p != g.end(v); ++p) {
            const int64_t u = *p;
            if (deg[u] > deg[v]) {
                const int64_t du = deg[u], pu = pos[u], pw = bin[du], w = vert[pw];
                if (u != w) { pos[u] = pw; vert[pu] = w; pos[w] = pu; vert[pw] = u; }
                bin[du]++;
                deg[u]--;
            }
        }
    }
    for (int64_t v = 0; v < n; ++v) core[v] = (int32_t)deg[v];
}

// Truss number of every undirected edge u<v, in CSR order (the order of gmsb_edge_similarity).  Sequential bucket
// peel: repeatedly remove a live edge of least support s, set k = max(k, s), give it truss k + 2, and take one unit of
// support from the two other edges of every triangle it still closes.  Returns m; truss may be NULL to size it.
int64_t tor_truss_numbers(int64_t n, const int64_t *off, const int32_t *nbr, int32_t *truss) {
    const Csr g{n, off, nbr};
    std::vector<int64_t> base(n + 1, 0);
    for (int64_t u = 0; u < n; ++u) base[u + 1] = base[u] + (g.end(u) - std::upper_bound(g.begin(u), g.end(u), (vid)u));
    const int64_t m = base[n];
    if (!truss || m == 0) return m;
    // edge id of every slot: position among the upper entries of the lower endpoint's row
    std::vector<int64_t> eid(off[n]);
    for (int64_t u = 0; u < n; ++u)
        for (const vid *p = g.begin(u); p != g.end(u); ++p) {
            const vid a = std::min<vid>((vid)u, *p), b = std::max<vid>((vid)u, *p);
            const vid *up = std::upper_bound(g.begin(a), g.end(a), a);
            eid[p - nbr] = base[a] + (std::lower_bound(up, g.end(a), b) - up);
        }
    std::vector<vid> ea(m), eb(m);
    for (int64_t u = 0; u < n; ++u)
        for (const vid *p = g.begin(u); p != g.end(u); ++p)
            if (u < *p) { ea[eid[p - nbr]] = (vid)u; eb[eid[p - nbr]] = *p; }
    std::vector<char> gone(m, 0);
    // f(e1, e2) for every triangle (a, b, w) of edge e = (a,b) whose other two edges are live: walk the shorter row,
    // binary-search the longer one
    auto for_live_triangles = [&](int64_t e, auto &&f) {
        vid a = ea[e], b = eb[e];
        if (g.deg(a) > g.deg(b)) std::swap(a, b);
        for (const vid *p = g.begin(a); p != g.end(a); ++p) {
            const vid *q = std::lower_bound(g.begin(b), g.end(b), *p);
            if (q == g.end(b) || *q != *p) continue;
            const int64_t e1 = eid[p - nbr], e2 = eid[q - nbr];
            if (!gone[e1] && !gone[e2]) f(e1, e2);
        }
    };
    std::vector<int64_t> sup(m, 0);
    for (int64_t e = 0; e < m; ++e) for_live_triangles(e, [&](int64_t, int64_t) { ++sup[e]; });
    const int64_t maxs = *std::max_element(sup.begin(), sup.end());
    std::vector<std::vector<int64_t>> bucket(maxs + 1);       // lazy: an entry is stale once its edge's support moved
    for (int64_t e = m - 1; e >= 0; --e) bucket[sup[e]].push_back(e);
    int64_t k = 0, cur = 0;
    for (int64_t removed = 0; removed < m;) {
        while (bucket[cur].empty()) ++cur;
        const int64_t e = bucket[cur].back();
        bucket[cur].pop_back();
        if (gone[e] || sup[e] != cur) continue;
        k = std::max(k, cur);
        truss[e] = (int32_t)(k + 2);
        for_live_triangles(e, [&](int64_t e1, int64_t e2) {
            for (int64_t x : {e1, e2}) { --sup[x]; bucket[sup[x]].push_back(x); cur = std::min(cur, sup[x]); }
        });
        gone[e] = 1;
        ++removed;
    }
    return m;
}

}  // extern "C"
