"""GPU parity (-m gpu): edge cases of the set algebra and of the schedule — empty and ragged neighbourhoods, lists that
span many merge tiles, hubs whose window does not fit the bitmap, isolated vertices, stars, cliques, bipartite
graphs (no triangles), and the degenerate k of the clique entry points."""
import numpy as np
import pytest

from conftest import random_graph_edges

pytestmark = pytest.mark.gpu


def clique_edges(n, base=0):
    s, d = np.triu_indices(n, 1)
    return (s + base).astype(np.int32), (d + base).astype(np.int32)


def comb(n, k):
    from math import comb as c
    return c(n, k)


def test_complete_graphs_have_closed_forms(gms):
    for n in (3, 4, 17, 33, 64, 65, 130):
        s, d = clique_edges(n)
        g = gms.Graph.from_edgelist(s, d, True)
        for v in ("auto", "merge", "gallop", "bitmap"):
            assert g.tc_total_ex(variant=v)[0] == comb(n, 3), (n, v)
        assert g.tc_vertex2().tolist() == [2 * comb(n - 1, 2)] * n
        for k in range(1, 8):
            want = comb(n, k) if k != 1 else n
            assert g.kclique_count(k) == want, (n, k)
        assert (g.edge_similarity("comm_neigh") == n - 2).all()
        assert g.kclique_count_ordered(3) == 6 * comb(n, 3)


def test_triangle_free_graphs(gms):
    # star, path, complete bipartite: no triangles, no k-cliques beyond edges
    star = gms.Graph.from_edgelist(np.zeros(5000, np.int32), np.arange(1, 5001, dtype=np.int32), True)
    assert star.tc_total() == 0 and star.kclique_count(3) == 0 and star.kclique_count(2) == 5000
    assert star.tc_vertex2().sum() == 0
    a, b = np.meshgrid(np.arange(60), np.arange(60, 140))
    bip = gms.Graph.from_edgelist(a.ravel().astype(np.int32), b.ravel().astype(np.int32), True)
    for v in ("auto", "merge", "gallop", "bitmap"):
        assert bip.tc_total_ex(variant=v)[0] == 0
    assert bip.kclique_count(4) == 0
    # common neighbours inside one side are all vertices of the other side
    assert bip.intersect_count_batch([0, 60], [1, 61]).tolist() == [80, 60]


def test_isolated_vertices_and_gaps(gms, orc):
    # ids with large gaps: most vertices are isolated (n = max id + 1)
    s = np.array([5, 5, 9, 100000, 100000, 7], np.int32)
    d = np.array([9, 100000, 100000, 7, 5, 9], np.int32)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    assert g.n == 100001 and g.tc_total() == o.tc_total() == 2
    assert (g.tc_vertex2() == o.tc_vertex2()).all()
    assert (g.degree_order(True) == o.degree_order(True)).all()
    assert g.kclique_count(4) == o.induce_directed(o.degree_order(True)).kclique(4) == 0


def test_ragged_pairs_long_lists_and_empty_sets(gms, orc):
    """Batched intersect over wildly different list lengths, including empty ones and lists of many merge tiles."""
    rng = np.random.default_rng(5)
    n = 6000
    src, dst = [], []
    sizes = {0: 0, 1: 1, 2: 5000, 3: 4999, 4: 37, 5: 2500, 6: 513, 7: 512, 8: 1024, 9: 3}
    for v, k in sizes.items():
        nb = rng.choice(np.arange(10, n), size=k, replace=False)
        src += [v] * k
        dst += nb.tolist()
    g = gms.Graph.from_edgelist(src, dst, False)            # directed: N(v) is exactly what was drawn
    o = orc.from_el(src, dst, False)
    ooff, onbr = o.csr()
    a, b = np.meshgrid(np.arange(10), np.arange(10))
    a, b = a.ravel().astype(np.int32), b.ravel().astype(np.int32)
    cnt = g.intersect_count_batch(a, b)
    off, el = g.intersect_batch(a, b)
    for i in range(len(a)):
        want = np.intersect1d(onbr[ooff[a[i]]:ooff[a[i] + 1]], onbr[ooff[b[i]]:ooff[b[i] + 1]])
        assert cnt[i] == len(want), (a[i], b[i])
        assert el[off[i]:off[i + 1]].tolist() == want.tolist()
    jac = g.pair_similarity("jaccard", a, b)
    assert jac[0] == 1.0                                     # two empty sets (vertex_similarity.h:31-32)
    assert np.isnan(g.pair_similarity("overlap", a[:1], b[:1])[0])     # 0/0 as in the reference
    for m in ("jaccard", "overlap", "comm_neigh", "total_neigh", "pref_att", "resource"):
        x, y = g.pair_similarity(m, a, b), o.pair_similarity(m, a, b)
        assert x.tobytes() == y.tobytes(), m


def test_wide_window_hubs_take_the_light_path(gms, orc):
    """A hub whose out-neighbours span more ids than the bitmap window must still be counted (merge / gallop)."""
    s, d = random_graph_edges(3, 50000, 400000, skew=0.0)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    want = o.tc_total()
    for bits in (64, 1024, 32768):
        c, st = g.tc_total_ex(hub_bitmap_bits=bits, hub_min_work=1)
        assert c == want
    c, st = g.tc_total_ex(variant="bitmap", hub_bitmap_bits=2048)
    assert c == want and st["edges_merge"] + st["edges_gallop"] > 0     # bitmap forced, but windows too wide
    assert (g.tc_vertex2() == o.tc_vertex2()).all()


def test_dense_graph_with_long_oriented_lists(gms, orc):
    """d+ far above 512: exercises the CTA-level list sorter, spill-free clique matrix limits and tiled merges."""
    s, d = random_graph_edges(9, 2500, 1500000, skew=0.3)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    want = o.tc_total()
    for v in ("auto", "merge", "gallop", "bitmap"):
        c, st = g.tc_total_ex(variant=v)
        assert c == want, v
    assert st["max_dplus"] > 512
    assert (g.tc_vertex2() == o.tc_vertex2()).all()
    assert g.edge_similarity("jaccard").tobytes() == o.edge_similarity("jaccard").tobytes()
    assert g.kclique_count(3) == want            # the clique kernels' CTA path agrees with the triangle kernels
    # (the oracle needs minutes for 4-cliques at this density; k >= 4 is covered on sparser graphs)


def test_from_csr_accepts_unsorted_lists_and_rejects_malformed(gms, orc):
    """SortedSet's constructor sorts its input (sorted_set.h:64-66), so FromCGraph works on any list order."""
    s, d = random_graph_edges(12, 800, 9000, skew=0.8)
    o = orc.from_el(s, d, True)
    off, nbr = o.csr()
    rng = np.random.default_rng(0)
    shuffled = nbr.copy()
    for u in range(len(off) - 1):
        rng.shuffle(shuffled[off[u]:off[u + 1]])
    g = gms.Graph.from_csr(off, shuffled)
    eo, en = g.export_csr()
    assert (eo == off).all() and (en == nbr).all() and g.tc_total() == o.tc_total()
    bad = nbr.copy()
    bad[3] = len(off) + 5
    with pytest.raises(gms.GmsbError):
        gms.Graph.from_csr(off, bad)
    bad_off = off.copy()
    bad_off[5], bad_off[6] = bad_off[6], bad_off[5] - 1 if bad_off[5] > 0 else 0
    if (np.diff(bad_off) < 0).any():
        with pytest.raises(gms.GmsbError):
            gms.Graph.from_csr(bad_off, nbr)


def test_degenerate_clique_sizes_and_errors(gms):
    s, d = clique_edges(6)
    g = gms.Graph.from_edgelist(s, d, True)
    dag = g.orient(g.degree_order(True))
    assert dag.kclique_count(1) == dag.n and dag.kclique_count(2) == 15      # parallelize.h:43-44
    assert g.kclique_count(7) == 0 and g.kclique_count(16) == 0
    with pytest.raises(gms.GmsbError):
        g.kclique_count(17)
    with pytest.raises(gms.GmsbError):
        g.kclique_count(0)
    with pytest.raises(gms.GmsbError):
        dag.kclique_count_ordered(3)        # ordered convention is defined on the undirected graph
    with pytest.raises(gms.GmsbError):
        g.pair_similarity("jaccard", [0], [99])


def test_tc_options_reject_unknown_reserved_values(gms):
    """gmsb_tc_options.reserved: [0..2] must be 0 and [3] one of 0, 2, 3; anything else fails instead of running some
    other kernel or the default."""
    import ctypes
    s, d = clique_edges(6)
    g = gms.Graph.from_edgelist(s, d, True)
    lib = gms.capi.lib()
    for reserved in ((0, 0, 7, 0), (0, 0, 0, 1)):
        opt = gms.capi.TcOptions(0, 0, 1, 0, 0, 0, 0, (ctypes.c_int32 * 4)(*reserved))
        out, st = ctypes.c_uint64(0), gms.capi.TcStats()
        assert lib.gmsb_tc_total_ex(g.h, ctypes.byref(opt), ctypes.byref(out), ctypes.byref(st)) == -1, reserved   # GMSB_ERR_INVALID
    assert g.tc_total_ex()[0] == comb(6, 3)


def test_large_host_csr_sorted_unsorted_and_malformed(gms):
    """A host CSR of 31 M slots through gmsb_graph_from_csr: sorted lists, a few reversed lists (the one streaming check
    finds them and only then a sort is paid for), and a malformed id at the very end."""
    s, d = gms.generate_rmat(20)
    g = gms.Graph.from_edgelist(s, d, True)
    off, nbr = g.export_csr()
    assert len(nbr) >= 1 << 24
    assert gms.Graph.from_csr(off, nbr).tc_total() == 423625371            # SURVEY.md 8c, kronecker-20
    rev = nbr.copy()
    for u in (0, 1, 2, len(off) // 2, len(off) - 2):                       # a few lists reversed, one in every region
        rev[off[u]:off[u + 1]] = rev[off[u]:off[u + 1]][::-1]
    big = int(np.argmax(np.diff(off)))
    rev[off[big]:off[big + 1]] = rev[off[big]:off[big + 1]][::-1]
    g2 = gms.Graph.from_csr(off, rev)
    assert g2.tc_total() == 423625371
    o2, n2 = g2.export_csr()
    assert (o2 == off).all() and (n2 == nbr).all()
    bad = nbr.copy()
    bad[-1] = g.n                                                           # id out of range in the last slot
    with pytest.raises(gms.GmsbError):
        gms.Graph.from_csr(off, bad)


def test_pipelined_upload_builds_the_same_representation(gms, orc):
    """gmsb_graph_from_csr_ex(GMSB_BUILD_ORIENT): chunked upload with the ranking / validation / relabel passes running
    on the chunks that have arrived.  Same counts, same exported CSR, same error behaviour as gmsb_graph_from_csr."""
    s, d = gms.generate_rmat(16)
    g = gms.Graph.from_edgelist(s, d, True)
    off, nbr = g.export_csr()
    gp = gms.Graph.from_csr(off, nbr, orient=True)
    assert gp.tc_total_ex(reuse_plan=False)[0] == 15656287                # SURVEY.md 8c, kronecker-16
    assert gp.tc_total_ex(reuse_plan=False)[0] == 15656287                # the pinned DAG survives reuse_plan = 0
    assert (gp.tc_vertex2() == g.tc_vertex2()).all()
    assert gp.kclique_count(4) == 291383976
    eo, en = gp.export_csr()
    assert (eo == off).all() and (en == nbr).all()
    # unsorted lists: sorted on the way in, DAG unaffected
    rng = np.random.default_rng(1)
    shuffled = nbr.copy()
    for u in rng.integers(0, len(off) - 1, 500):
        rng.shuffle(shuffled[off[u]:off[u + 1]])
    gs = gms.Graph.from_csr(off, shuffled, orient=True)
    eo, en = gs.export_csr()
    assert (en == nbr).all() and gs.tc_total() == 15656287
    # malformed inputs are rejected, and the library keeps working afterwards
    bad = nbr.copy()
    bad[len(bad) // 2] = g.n + 7
    with pytest.raises(gms.GmsbError):
        gms.Graph.from_csr(off, bad, orient=True)
    bad[len(bad) // 2] = -3
    with pytest.raises(gms.GmsbError):
        gms.Graph.from_csr(off, bad, orient=True)
    bad_off = off.copy()
    bad_off[7] = bad_off[-1] + 1000
    with pytest.raises(gms.GmsbError):
        gms.Graph.from_csr(bad_off, nbr, orient=True)
    assert gms.Graph.from_csr(off, nbr, orient=True).tc_total() == 15656287
    # small and empty graphs take the plain path
    tri = gms.Graph.from_csr(np.array([0, 2, 4, 6], np.int64), np.array([1, 2, 0, 2, 0, 1], np.int32), orient=True)
    assert tri.tc_total() == 1
    assert gms.Graph.from_csr(np.array([0, 0, 0], np.int64), np.zeros(0, np.int32), orient=True).tc_total() == 0


def test_offsets_beyond_the_neighbour_array_are_rejected(gms):
    """ADVICE r1: offsets such as [0, 1e9, 5] pass 'starts at 0, ends at slots' — every entry has to be bounded."""
    nbr = np.array([1, 0, 2, 1, 0], np.int32)
    for off in ([0, 10**9, 5], [0, 6, 5], [0, -1, 5]):
        with pytest.raises(gms.GmsbError):
            gms.Graph.from_csr(np.array(off, np.int64), nbr)
    g = gms.Graph.from_csr(np.array([0, 2, 4, 6], np.int64), np.array([1, 2, 0, 2, 0, 1], np.int32))
    assert g.tc_total() == 1


def test_cliques_on_a_dag_whose_arcs_descend(gms, orc):
    """ADVICE r1: KcListing accepts any DAG; a directed handle whose arcs go from higher to lower ids (or both ways)
    must give the same counts as the ascending orientation."""
    s, d = random_graph_edges(5, 300, 9000, skew=0.6)
    g = gms.Graph.from_edgelist(s, d, True)
    want = {k: g.kclique_count(k) for k in (3, 4, 5)}
    off, nbr = g.export_csr()
    n = g.n
    src = np.repeat(np.arange(n, dtype=np.int32), np.diff(off))
    down = src > nbr                                         # every edge once, pointing to the lower id
    dag_down = gms.Graph.from_edgelist(src[down], nbr[down], False)
    rng = np.random.default_rng(3)
    order = rng.permutation(n)                               # an arbitrary acyclic orientation
    mixed = order[src] < order[nbr]
    dag_mixed = gms.Graph.from_edgelist(src[mixed], nbr[mixed], False)
    for k, w in want.items():
        assert dag_down.kclique_count(k) == w, k
        assert dag_mixed.kclique_count(k) == w, k
