"""GPU parity suite (-m gpu): the CUDA path, called through the C ABI, against the CPU oracle on the same seeded
inputs, against the committed golden vectors, and through size-independent properties at larger scale.
Bar: bit-exact for every integer output and for the similarity scores computed from integer counts."""
import hashlib

import numpy as np
import pytest

from conftest import random_graph_edges

pytestmark = pytest.mark.gpu

VARIANTS = ["auto", "merge", "gallop", "bitmap"]
EXACT_METRICS = ["jaccard", "overlap", "resource", "comm_neigh", "total_neigh", "pref_att"]


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def same_csr(a, b):
    return all((x == y).all() and len(x) == len(y) for x, y in zip(a, b))


@pytest.fixture(scope="module")
def kron12(gms, orc):
    s, d = gms.generate_rmat(12)
    return gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)


# ---- graph construction ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["micro", "triangles_1", "triangles_3", "smallRandom1", "eppsteinExample",
                                  "tomitaExample"])
def test_reference_test_graphs(gms, golden, name):
    rec = golden["graphs"][name]
    g = gms.Graph.from_edgelist(rec["src"], rec["dst"], True)
    off, nbr = g.export_csr()
    assert off.tolist() == rec["off"] and nbr.tolist() == rec["nbr"]
    for v in VARIANTS:
        assert g.tc_total_ex(variant=v)[0] == rec["tc"], v
    assert g.tc_total() == rec["tc"]
    assert g.degree_order(False).tolist() == rec["order"] and g.degree_order(True).tolist() == rec["rank"]
    dag = g.orient(np.array(rec["rank"], np.int32))
    doff, dnbr = dag.export_csr()
    assert dag.n == rec["dag_n"] and dag.directed
    assert doff[:dag.n + 1].tolist() == rec["dag_off"] and dnbr.tolist() == rec["dag_nbr"]
    rel = g.relabel_by_degree()
    ro, rn = rel.export_csr()
    assert ro.tolist() == rec["relabel_off"] and rn.tolist() == rec["relabel_nbr"]
    for m in EXACT_METRICS:
        assert [x.hex() for x in g.edge_similarity(m)] == rec["sim_hex"][m], m
    # from_csr round trip
    g2 = gms.Graph.from_csr(np.array(rec["off"]), np.array(rec["nbr"], np.int32))
    assert same_csr(g2.export_csr(), (off, nbr)) and g2.tc_total() == rec["tc"]


@pytest.mark.parametrize("key", ["kronecker-8", "kronecker-10", "kronecker-12", "uniform-10", "kronecker-14"])
def test_generated_graphs_against_golden(gms, golden, key):
    kind, scale = key.split("-")
    rec = golden["generated"][key]
    s, d = gms.generate_rmat(int(scale)) if kind == "kronecker" else gms.generate_uniform(int(scale))
    assert sha(s) + sha(d) == rec["el_sha"]
    g = gms.Graph.from_edgelist(s, d, True)
    off, nbr = g.export_csr()
    assert g.n == rec["n"] and g.slots == rec["slots"] and sha(off) + sha(nbr) == rec["csr_sha"]
    for v in VARIANTS:
        assert g.tc_total_ex(variant=v)[0] == rec["tc"], v
    assert sha(g.degree_order(False)) == rec["order_sha"] and sha(g.degree_order(True)) == rec["rank_sha"]
    dag = g.orient(g.degree_order(True))
    doff, dnbr = dag.export_csr()
    assert dag.n == rec["dag_n"] and sha(doff[:dag.n + 1]) + sha(dnbr) == rec["dag_sha"]
    ro, rn = g.relabel_by_degree().export_csr()
    assert sha(ro) + sha(rn) == rec["relabel_sha"]
    for m in EXACT_METRICS:
        assert sha(g.edge_similarity(m)) == rec["sim_sha"][m], m


@pytest.mark.parametrize("seed", range(8))
def test_random_graphs_against_oracle(gms, orc, seed):
    n, m = [(1, 1), (50, 200), (200, 3000), (1000, 8000), (64, 2000), (500, 500), (3000, 60000), (20000, 300000)][seed]
    s, d = random_graph_edges(seed, n, m, skew=(seed % 3) * 0.8)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    assert same_csr(g.export_csr(), o.csr())
    want = o.tc_total()
    for v in VARIANTS:
        got, st = g.tc_total_ex(variant=v)
        assert got == want, (v, st)
    # tuning knobs never change the answer
    for bits, work, ratio in ((64, 1, 2), (4096, 16, 1), (1 << 20, 1, 64)):
        assert g.tc_total_ex(hub_bitmap_bits=bits, hub_min_work=work, gallop_ratio=ratio)[0] == want
    for rf in (False, True):
        assert (g.degree_order(rf) == o.degree_order(rf)).all()
    rank = o.degree_order(True)
    dag, odag = g.orient(rank), o.induce_directed(rank)
    assert dag.n == odag.n and same_csr(dag.export_csr(), odag.csr())
    assert same_csr(g.relabel_by_degree().export_csr(), o.relabel_by_degree().csr())
    # directed build (no symmetrisation)
    gd, od = gms.Graph.from_edgelist(s, d, False), orc.from_el(s, d, False)
    assert gd.directed and same_csr(gd.export_csr(), od.csr())


def test_empty_and_degenerate_inputs(gms):
    g = gms.Graph.from_edgelist(np.zeros(0, np.int32), np.zeros(0, np.int32), True)
    assert g.n == 1 and g.slots == 0 and g.tc_total() == 0          # FindMaxNodeId of an empty list is 0
    g = gms.Graph.from_edgelist([3, 3, 3], [3, 3, 3], True)         # only self loops
    assert g.n == 4 and g.slots == 0 and g.tc_total() == 0
    g = gms.Graph.from_edgelist([0, 0, 0, 1], [1, 1, 1, 0], True)   # duplicates collapse
    assert g.slots == 2
    g = gms.Graph.from_csr(np.zeros(1, np.int64), np.zeros(0, np.int32))
    assert g.n == 0 and g.tc_total() == 0
    with pytest.raises(gms.GmsbError):
        gms.Graph.from_edgelist([0, -1], [1, 2], True)
    gd = gms.Graph.from_edgelist([0, 1], [1, 2], False)
    with pytest.raises(gms.GmsbError):      # the reference throws std::invalid_argument (apply_order.h:14-16)
        gd.orient(np.arange(3, dtype=np.int32))
    with pytest.raises(gms.GmsbError):
        gd.tc_total()
    gu = gms.Graph.from_edgelist([0, 1], [1, 2], True)
    with pytest.raises(gms.GmsbError):
        gu.orient(np.array([0, 0, 1], np.int32))                    # not a permutation


# ---- triangles: partitions, statistics, larger scale ------------------------------------------------------------------
def test_partition_sums_to_total(kron12, golden):
    g, _ = kron12
    want = golden["generated"]["kronecker-12"]["tc"]
    for parts in (2, 3, 8):
        for v in ("auto", "merge", "bitmap"):
            tot, bytes_, edges = 0, 0, [0, 0, 0, 0]
            for p in range(parts):
                c, st = g.tc_total_ex(variant=v, part_index=p, part_count=parts, reuse_plan=True)
                tot += c
                bytes_ += st["algorithmic_bytes"]
                for i, key in enumerate(("edges_bitmap", "edges_merge", "edges_gallop", "bitmap_items")):
                    edges[i] += st[key]
            assert tot == want, (parts, v)
            _, full = g.tc_total_ex(variant=v, reuse_plan=True)
            assert bytes_ == full["algorithmic_bytes"]
            # a device builds only its share of the schedule: the shares cover every edge / hub item exactly once
            assert edges == [full[key] for key in ("edges_bitmap", "edges_merge", "edges_gallop", "bitmap_items")]


def test_schedule_edge_passes_rows_and_slots_agree(gms):
    """The two edge passes of the schedule exist in two forms: walking the rows, and element-wise over the slots (the
    default from 4 parts on; edge_passes = "rows" / "slots" forces one or the other).  Same counts and the same
    statistics, for the whole schedule and for shares of it."""
    s, d = gms.generate_rmat(16)
    g = gms.Graph.from_edgelist(s, d, True)
    keys = ("triangles", "algorithmic_bytes", "wedges_checked", "edges_bitmap", "edges_merge", "edges_gallop",
            "bitmap_items", "bytes_bitmap", "bytes_light", "wedges_bitmap")
    for variant in ("auto", "bitmap", "merge"):
        for parts in (1, 3, 5):
            for p in range(parts):
                a = g.tc_total_ex(variant=variant, part_index=p, part_count=parts, reuse_plan=2, edge_passes="slots")
                b = g.tc_total_ex(variant=variant, part_index=p, part_count=parts, reuse_plan=2, edge_passes="rows")
                c = g.tc_total_ex(variant=variant, part_index=p, part_count=parts, reuse_plan=2)
                assert a[0] == b[0] == c[0], (variant, parts, p)
                assert [a[1][k] for k in keys] == [b[1][k] for k in keys] == [c[1][k] for k in keys], (variant, parts, p)
    assert (g.tc_total_ex(reuse_plan=2, edge_passes="rows")[0] == g.tc_total_ex(reuse_plan=2, edge_passes="slots")[0]
            == 15656287)   # SURVEY.md 8c


def test_algorithmic_bytes_match_definition(kron12, orc):
    g, o = kron12
    b_tc, _, max_dplus = orc.tc_bytes(o)
    _, st = g.tc_total_ex()
    assert st["algorithmic_bytes"] == b_tc and st["max_dplus"] == max_dplus
    assert st["oriented_edges"] == o.slots // 2
    assert st["edges_bitmap"] + st["edges_merge"] + st["edges_gallop"] <= st["oriented_edges"]
    assert st["launches"] > 0


def test_kron16_all_variants(gms, golden):
    s, d = gms.generate_rmat(16)
    g = gms.Graph.from_edgelist(s, d, True)
    rec = golden["generated"]["kronecker-16"]
    assert (g.n, g.slots) == (rec["n"], rec["slots"])
    for v in VARIANTS:
        assert g.tc_total_ex(variant=v)[0] == rec["tc"], v
    # relabelling (what parse_and_load does, cli/cli.h:174-181) never changes the total
    assert g.relabel_by_degree().tc_total() == rec["tc"]


def test_kron18_survey_total(gms):
    s, d = gms.generate_rmat(18)
    g = gms.Graph.from_edgelist(s, d, True)
    assert (g.n, g.slots // 2) == (262143, 3805448)          # SURVEY.md §8c
    assert g.tc_total() == 82728031


def test_properties_at_scale_20(gms):
    """Scale 20: the oracle would take minutes; use invariances instead (and the survey's reference total)."""
    s, d = gms.generate_rmat(20)
    g = gms.Graph.from_edgelist(s, d, True)
    assert (g.n, g.slots // 2) == (1048576, 15699687)
    base, st = g.tc_total_ex()
    assert base == 423625371                                   # SURVEY.md §8c, measured with the reference
    assert g.tc_total_ex(variant="bitmap")[0] == base
    # invariance under vertex relabelling and under edge-list order / duplication
    assert g.relabel_by_degree().tc_total() == base
    perm = np.random.default_rng(1).permutation(len(s))
    g2 = gms.Graph.from_edgelist(np.concatenate([d[perm], s[:1000]]), np.concatenate([s[perm], d[:1000]]), True)
    assert same_csr(g2.export_csr(), g.export_csr())
    # partition additivity
    assert sum(g.tc_total_ex(part_index=p, part_count=4, reuse_plan=True)[0] for p in range(4)) == base


# ---- set algebra / similarity --------------------------------------------------------------------------------------------
def test_set_kats_through_neighbourhoods(gms, golden):
    # the reference's SortedSet KATs (testing/sets.cpp:108-141), as neighbourhoods of a directed graph
    src, dst, pairs = [], [], []
    for i, kat in enumerate(golden["sets"]):
        a_id, b_id = 100 + 2 * i, 101 + 2 * i
        src += [a_id] * len(kat["a"]) + [b_id] * len(kat["b"])
        dst += kat["a"] + kat["b"]
        pairs.append((a_id, b_id))
    src += [200]; dst += [0]
    g = gms.Graph.from_edgelist(src, dst, False)
    a = np.array([p[0] for p in pairs], np.int32)
    b = np.array([p[1] for p in pairs], np.int32)
    for x, y in ((a, b), (b, a)):
        cnt = g.intersect_count_batch(x, y)
        off, elems = g.intersect_batch(x, y)
        for i, kat in enumerate(golden["sets"]):
            assert cnt[i] == len(kat["intersect"])
            assert elems[off[i]:off[i + 1]].tolist() == kat["intersect"]
    # union / difference / union_count of the same KAT sets (testing/sets.cpp union* / difference* cases)
    uoff, uel = g.union_batch(a, b)
    doff, del_ = g.difference_batch(a, b)
    ucnt = g.union_count_batch(a, b)
    for i, kat in enumerate(golden["sets"]):            # golden values produced by the reference's SortedSet
        assert uel[uoff[i]:uoff[i + 1]].tolist() == kat["union"] and ucnt[i] == kat["union_count"]
        assert del_[doff[i]:doff[i + 1]].tolist() == kat["difference"]


@pytest.mark.parametrize("seed", range(3))
def test_pair_ops_against_oracle(gms, orc, seed):
    n, m = [(300, 4000), (5000, 100000), (2000, 150000)][seed]
    s, d = random_graph_edges(10 + seed, n, m, skew=seed * 1.0)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    rng = np.random.default_rng(seed)
    a = rng.integers(0, g.n, 5000, dtype=np.int32)
    b = rng.integers(0, g.n, 5000, dtype=np.int32)
    want = o.pair_similarity("comm_neigh", a, b).astype(np.uint64)
    assert (g.intersect_count_batch(a, b) == want).all()
    ooff, onbr = o.csr()
    off, elems = g.intersect_batch(a[:500], b[:500])
    for i in range(500):
        ref_i = np.intersect1d(onbr[ooff[a[i]]:ooff[a[i] + 1]], onbr[ooff[b[i]]:ooff[b[i] + 1]])
        assert elems[off[i]:off[i + 1]].tolist() == ref_i.tolist()
    # materialising difference / union and union_count against the oracle's restatement of sorted_set.h:104-140,184-189
    doff, delems = g.difference_batch(a[:500], b[:500])
    uoff, uelems = g.union_batch(a[:500], b[:500])
    ucnt = g.union_count_batch(a[:500], b[:500])
    for i in range(500):
        la, lb = onbr[ooff[a[i]]:ooff[a[i] + 1]], onbr[ooff[b[i]]:ooff[b[i] + 1]]
        assert delems[doff[i]:doff[i + 1]].tolist() == orc.difference(la, lb).tolist()
        assert uelems[uoff[i]:uoff[i + 1]].tolist() == orc.union(la, lb).tolist()
        assert int(ucnt[i]) == orc.union_count(la, lb) == uoff[i + 1] - uoff[i]
    for mname in EXACT_METRICS:
        assert g.pair_similarity(mname, a, b).tobytes() == o.pair_similarity(mname, a, b).tobytes(), mname
        assert g.edge_similarity(mname).tobytes() == o.edge_similarity(mname).tobytes(), mname
    # Adamic-Adar goes through log(): a few ulp, not bit-exact (SURVEY.md §8f.1)
    got, ref_ = g.pair_similarity("adamic_adar", a, b), o.pair_similarity("adamic_adar", a, b)
    finite = np.isfinite(ref_)
    assert (np.isfinite(got) == finite).all()
    assert np.allclose(got[finite], ref_[finite], rtol=1e-13, atol=0)
    for call in (g.intersect_count_batch, g.union_count_batch, g.intersect_batch, g.difference_batch, g.union_batch):
        for x, y in (([0, g.n], [0, 0]), ([0, 0], [-1, 0])):
            with pytest.raises(gms.GmsbError, match="vertex id out of range"):
                call(np.array(x, np.int32), np.array(y, np.int32))
    # out-lists of 64, 511 and 512 elements: pairs on both sides of the count kernels' gallop rule (longer >= 8 x
    # shorter), in both orders, through the batch API
    src, dst = [], []
    for v, deg in ((0, 64), (1, 511), (2, 512)):
        src += [v] * deg
        dst += rng.choice(np.arange(3, 1200), deg, replace=False).tolist()
    gb, ob = gms.Graph.from_edgelist(src, dst, False), orc.from_el(src, dst, False)
    boff, bnbr = ob.csr()
    lists = [bnbr[boff[v]:boff[v + 1]] for v in range(3)]
    assert [len(x) for x in lists] == [64, 511, 512]
    pa, pb = np.array([0, 0, 2, 1], np.int32), np.array([2, 1, 0, 0], np.int32)
    assert gb.intersect_count_batch(pa, pb).tolist() == [orc.intersect_count(lists[x], lists[y]) for x, y in zip(pa, pb)]
    assert gb.union_count_batch(pa, pb).tolist() == [orc.union_count(lists[x], lists[y]) for x, y in zip(pa, pb)]
    for batch, op in ((gb.intersect_batch, orc.intersect), (gb.difference_batch, orc.difference),
                      (gb.union_batch, orc.union)):
        boffs, belems = batch(pa, pb)
        for i, (x, y) in enumerate(zip(pa, pb)):
            assert belems[boffs[i]:boffs[i + 1]].tolist() == op(lists[x], lists[y]).tolist()


def test_orientation_fallback_path(gms, orc, monkeypatch):
    """Lists longer than the on-chip sorter take the global radix-sort path; force it with a tiny cap."""
    s, d = random_graph_edges(77, 3000, 80000, skew=1.2)
    o = orc.from_el(s, d, True)
    want = o.tc_total()
    for cap in ("0", "40", "8192"):
        monkeypatch.setenv("GMSB_ORIENT_SORT_CAP", cap)
        g = gms.Graph.from_edgelist(s, d, True)
        assert g.tc_total_ex()[0] == want, cap
        rank = o.degree_order(True)
        dag, odag = g.orient(rank), o.induce_directed(rank)
        assert same_csr(dag.export_csr(), odag.csr()), cap


@pytest.mark.parametrize("scale", [14, 16])
def test_skewed_rmat_against_the_oracle(gms, orc, scale):
    """BASELINE.json configs[4]: R-MAT with a = 0.65 (b = c = 0.15): much heavier hubs than the reference's kronecker.
    Every kernel family against the oracle's count, per-vertex counts, and k-cliques on the same graph."""
    s, d = gms.generate_rmat(scale, a=0.65, b=0.15, c=0.15)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    want = o.tc_total()
    for v in ("auto", "merge", "gallop", "bitmap"):
        c, st = g.tc_total_ex(variant=v)
        assert c == want, (scale, v)
    bt, _, mx = orc.tc_bytes(o)
    c, st = g.tc_total_ex()
    assert st["algorithmic_bytes"] == bt and st["max_dplus"] == mx
    assert (g.tc_vertex2() == o.tc_vertex2()).all()
    assert g.tc_total_ex(hub_bitmap_bits=4096, hub_min_work=1)[0] == want      # narrow windows: hubs fall to the light path
    if scale == 14:
        dag = o.induce_directed(o.degree_order(True))
        for k in (4, 5):
            assert g.kclique_count(k) == dag.kclique(k), k
    off, nbr = g.export_csr()
    gp = gms.Graph.from_csr(off, nbr, orient=True)
    assert gp.tc_total_ex(reuse_plan=False)[0] == want


def test_partition_is_consistent_across_independently_built_schedules(gms):
    """Multi-GPU runs build the schedule once per device; the descriptors inside a hub's segment sit in the order the
    scatter pass's atomics ran in, so ownership must not depend on it: shares taken from DIFFERENT builds of the
    schedule have to add up (this is what goes wrong first when the partition leans on a nondeterministic order)."""
    s, d = gms.generate_rmat(18)
    graphs = [gms.Graph.from_edgelist(s, d, True) for _ in range(4)]
    want = 82728031                                                        # SURVEY.md 8c, kronecker-18
    for variant in ("auto", "bitmap", "gallop"):
        for parts in (2, 4):
            got = sum(graphs[p].tc_total_ex(variant=variant, part_index=p, part_count=parts)[0] for p in range(parts))
            assert got == want, (variant, parts)
    # per-vertex counts over shares from different builds (mgpu.cu path is covered in test_gpu_operators.py)
    got = sum(graphs[p].tc_total_ex(part_index=p, part_count=3, reuse_plan=2)[0] for p in range(3))
    assert got == want
