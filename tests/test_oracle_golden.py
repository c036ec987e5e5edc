"""CPU suite: the oracle (oracle/oracle.cpp) against the golden vectors generated from the unmodified reference
(tests/golden/make_golden.py), against the stored record of the reference's answers on seeded random cases
(oracle/reference_cases.py) and, where the reference library is present, against the reference directly."""
import hashlib

import numpy as np
import pytest

from conftest import random_graph_edges
from oracle import reference_cases as rc
from oracle.binding import METRICS


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def check_record(g, rec, full):
    off, nbr = g.csr()
    assert g.n == rec["n"] and g.slots == rec["slots"]
    assert sha(off) + sha(nbr) == rec["csr_sha"]
    assert g.tc_total(True) == rec["tc"] == g.tc_total(False) == g.tc_verify_total()
    assert g.worth_relabelling() == rec["worth_relabelling"]
    v2 = g.tc_vertex2()
    assert sha(v2) == rec["vertex2_sha"]
    assert int(v2.sum()) == 6 * rec["tc"]
    order, rank = g.degree_order(False), g.degree_order(True)
    assert sha(order) == rec["order_sha"] and sha(rank) == rec["rank_sha"]
    dag = g.induce_directed(rank)
    doff, dnbr = dag.csr()
    assert dag.n == rec["dag_n"] and sha(doff) + sha(dnbr) == rec["dag_sha"]
    for k, want in rec["kclique"].items():
        assert dag.kclique(int(k)) == want, k
    for k, want in rec["ordered"].items():
        assert g.clique_count_set_based(int(k)) == want, k
    rel = g.relabel_by_degree()
    ro, rn = rel.csr()
    assert sha(ro) + sha(rn) == rec["relabel_sha"]
    for m in METRICS:
        assert sha(g.edge_similarity(m)) == rec["sim_sha"][m], m
    if full:
        assert off.tolist() == rec["off"] and nbr.tolist() == rec["nbr"]
        assert v2.tolist() == rec["vertex2"]
        assert order.tolist() == rec["order"] and rank.tolist() == rec["rank"]


def test_set_kats(orc, golden):
    for kat in golden["sets"]:
        a, b = kat["a"], kat["b"]
        assert orc.intersect(a, b).tolist() == kat["intersect"] == orc.intersect(b, a).tolist()
        assert orc.intersect_count(a, b) == len(kat["intersect"]) == orc.intersect_count(b, a)
        assert orc.union(a, b).tolist() == kat["union"]
        assert orc.union_count(a, b) == kat["union_count"]
        assert orc.difference(a, b).tolist() == kat["difference"]


def test_clique_kats(orc, golden):
    for kat in golden["clique_kats"]:
        g = orc.from_el(kat["src"], kat["dst"], True)
        for rank in (g.degree_order(True), orc.degeneracy_rank(g)):
            assert g.induce_directed(rank).kclique(kat["k"]) == kat["count"]


@pytest.mark.parametrize("name", ["micro", "triangles_1", "triangles_3", "smallRandom1", "eppsteinExample",
                                  "tomitaExample"])
def test_reference_test_graphs(orc, golden, name):
    rec = golden["graphs"][name]
    check_record(orc.from_el(rec["src"], rec["dst"], True), rec, True)


def test_survey_goldens(orc, golden):
    # SURVEY.md §8c table
    g = golden["graphs"]
    assert g["triangles_1"]["tc"] == 1 and g["triangles_1"]["vertex2"] == [2, 2, 2]
    assert g["triangles_3"]["tc"] == 3 and g["triangles_3"]["vertex2"] == [2, 4, 4, 2, 0, 2, 2, 2, 0, 0]
    assert g["triangles_3"]["order"] == [4, 0, 3, 5, 8, 9, 1, 2, 6, 7]
    assert g["smallRandom1"]["tc"] == 5 and g["eppsteinExample"]["tc"] == 11 and g["tomitaExample"]["tc"] == 8
    assert g["eppsteinExample"]["kclique"]["4"] == 1 and g["tomitaExample"]["kclique"]["4"] == 1
    assert golden["generated"]["kronecker-12"]["kclique"]["4"] == 4021397
    assert golden["generated"]["kronecker-12"]["ordered"]["3"] == 2900934
    assert golden["generated"]["kronecker-14"]["kclique"]["4"] == 36582679


@pytest.mark.parametrize("key", ["kronecker-8", "kronecker-10", "kronecker-12", "uniform-10", "kronecker-14"])
def test_generated_graphs(orc, golden, key):
    kind, scale = key.split("-")
    rec = golden["generated"][key]
    s, d = orc.generate_el(int(scale), 16, kind == "uniform")
    assert sha(s) + sha(d) == rec["el_sha"]
    check_record(orc.generate(int(scale), 16, kind == "uniform"), rec, False)


def test_kron16_total(orc, golden):
    g = orc.generate(16)
    rec = golden["generated"]["kronecker-16"]
    assert (g.n, g.slots, g.tc_total(True)) == (rec["n"], rec["slots"], rec["tc"])


def test_degeneracy_rank_is_valid(orc):
    for seed in range(4):
        s, d = random_graph_edges(seed, 300, 2000, skew=1.0)
        g = orc.from_el(s, d, True)
        rank = orc.degeneracy_rank(g)
        degen = orc.check_degeneracy_rank(g, rank)
        assert degen >= 0
        bad = rank.copy()
        bad[[0, 1]] = bad[[1, 0]]
        # a random transposition almost always breaks min-degree order; at least it must stay a permutation check
        assert orc.check_degeneracy_rank(g, bad) in (-1, degen)


# ---- comparison with the unmodified reference: its stored answers always, the library itself where it is present -----
@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_reference_random(orc, ref_or_none, reference_cases, seed):
    assert rc.random_record(orc, orc, seed) == reference_cases["random"][seed]
    ref = ref_or_none
    if ref is None:
        return
    s, d, m = rc.random_case(seed)
    go, gr = orc.from_el(s, d, True), ref.from_el(s, d, True)
    for x, y in zip(go.csr(), gr.csr()):
        assert (x == y).all()
    assert go.tc_total() == gr.tc_total()
    assert (go.tc_vertex2() == gr.tc_vertex2(1)).all()
    for rf in (False, True):
        assert (go.degree_order(rf) == gr.degree_order(rf)).all()
    rank = go.degree_order(True)
    do, dr = go.induce_directed(rank), gr.induce_directed(rank)
    assert do.n == dr.n
    for x, y in zip(do.csr(), dr.csr()):
        assert (x == y).all()
    for k in (1, 2, 3, 4, 5):
        assert do.kclique(k) == dr.kclique(k, 2) == dr.kclique(k, 1)
    if m <= 3000:
        assert go.clique_count_set_based(4) == gr.clique_count_set_based(4)
    for mname in METRICS:
        assert go.edge_similarity(mname).tobytes() == gr.edge_similarity(mname).tobytes(), mname
    # a reference degeneracy ranking is valid by the oracle's checker, and orients to the same clique counts
    rr = ref.degeneracy_rank(gr)
    assert orc.check_degeneracy_rank(go, rr) == orc.check_degeneracy_rank(go, orc.degeneracy_rank(go)) >= 0
    assert go.induce_directed(rr).kclique(4) == do.kclique(4)
    rel_o, rel_r = go.relabel_by_degree(), gr.relabel_by_degree()
    for x, y in zip(rel_o.csr(), rel_r.csr()):
        assert (x == y).all()


def test_oracle_sets_match_reference_random(orc, ref_or_none, reference_cases):
    assert rc.set_record(orc) == reference_cases["sets"]
    ref = ref_or_none
    if ref is None:
        return
    for a, b, x in rc.set_cases():
        assert orc.intersect_count(a, b) == ref.intersect_count(a, b)
        assert orc.intersect(a, b).tolist() == ref.intersect(a, b).tolist()
        assert orc.union(a, b).tolist() == ref.union(a, b).tolist()
        assert orc.union_count(a, b) == ref.union_count(a, b)
        assert orc.difference(a, b).tolist() == ref.difference(a, b).tolist()
        assert orc.contains(a, x) == ref.contains(a, x)


def test_clique_recursion_bytes(orc, golden):
    """B_k (SURVEY.md 8d): the instrumented recursion counts the same cliques, and its k = 3 bytes are B_TC."""
    g = orc.generate(12)
    dag = g.induce_directed(g.degree_order(True))
    rec = golden["generated"]["kronecker-12"]["kclique"]
    b_tc, _, _ = orc.tc_bytes(g)
    prev = 0
    for k in (3, 4, 5):
        b, c = orc.kclique_bytes(dag, k)
        assert c == rec[str(k)] == dag.kclique(k)
        assert b > prev
        prev = b
        if k == 3:
            assert b == b_tc
