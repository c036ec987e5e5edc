"""GPU parity (-m gpu): the clique kernels for d+ > 32 against closed forms, the reference's totals (SURVEY.md §8c,
Danisch edge-parallel counts of the unmodified reference) and the oracle.  k picks the kernels: lane-parallel
(kclique_lane.cuh) for 5 <= k <= 10, with the decoupled pair kernel from k = 7 on; warp-cooperative otherwise."""
from math import comb

import numpy as np
import pytest

from conftest import random_graph_edges

pytestmark = pytest.mark.gpu

# reference totals, SURVEY.md §8c (kronecker ef16, reference generator)
KRON14 = {4: 36582679, 5: 383825252, 6: 3276576738, 7: 23152812639, 8: 138220170775}
KRON16 = {4: 291383976, 5: 4609989471, 6: 60115277770}


def complete(gms, n):
    i, j = np.triu_indices(n, 1)
    return gms.Graph.from_edgelist(i.astype(np.int32), j.astype(np.int32), True)


@pytest.mark.parametrize("n,ks", [(40, (4, 5, 6, 7, 8, 9, 10)), (100, (4, 5, 6, 7)), (130, (4, 5)), (300, (4, 5)),
                                  (600, (4, 5)), (700, (5,)), (1100, (4, 5)), (1300, (4, 5))])
def test_complete_graphs_every_class(gms, n, ks):
    """d+ <= 64 / 128 / 256 / 512, > 512 in shared memory, > 512 with CTA-wide levels above the compaction (K_700,
    K_1100) and with the matrix spilled to global memory (K_1300)."""
    g = complete(gms, n)
    for k in ks:
        assert g.kclique_count(k) == comb(n, k), (n, k)


def test_kronecker_against_reference_totals(gms):
    s, d = gms.generate_rmat(14)
    g = gms.Graph.from_edgelist(s, d, True)
    for k, want in KRON14.items():
        assert g.kclique_count(k) == want, k
    s, d = gms.generate_rmat(16)
    g = gms.Graph.from_edgelist(s, d, True)
    for k, want in KRON16.items():
        assert g.kclique_count(k) == want, k


def test_lane_partition_is_additive(gms):
    s, d = gms.generate_rmat(14)
    g = gms.Graph.from_edgelist(s, d, True)
    assert sum(g.kclique_count(6, p, 3) for p in range(3)) == KRON14[6]
    g = complete(gms, 600)
    assert sum(g.kclique_count(5, p, 5) for p in range(5)) == comb(600, 5)


def test_dense_random_graphs(gms, orc):
    s, d = random_graph_edges(61, 600, 60000, skew=0.5)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    dag = o.induce_directed(o.degree_order(True))
    for k in (4, 5, 6):
        assert g.kclique_count(k) == dag.kclique(k), k
    rng = np.random.default_rng(7)
    a = np.triu(rng.random((900, 900)) < 0.35, 1)
    i, j = np.nonzero(a)
    i, j = i.astype(np.int32), j.astype(np.int32)
    g, o = gms.Graph.from_edgelist(i, j, True), orc.from_el(i, j, True)
    dag = o.induce_directed(o.degree_order(True))
    for k in (4, 5, 6):
        assert g.kclique_count(k) == dag.kclique(k), k


def test_complete_multipartite_reaches_the_pair_kernel_above_512(gms):
    """Complete 7-partite graph with parts of 86 vertices: every vertex has degree 516, so in any orientation the
    first-ranked vertex has d+ = 516 > 512, and a 7-clique takes one vertex of every part: C(7, k) * 86^k k-cliques.
    k = 5, 6 run the d+ > 512 and mid-size lane kernels, k = 7 the pair kernel's batch path."""
    parts, size = 7, 86
    part = np.repeat(np.arange(parts), size)
    i, j = np.triu_indices(parts * size, 1)
    keep = part[i] != part[j]
    g = gms.Graph.from_edgelist(i[keep].astype(np.int32), j[keep].astype(np.int32), True)
    for k in (5, 6, 7):
        assert g.kclique_count(k) == comb(parts, k) * size ** k, k


def test_unsupported_sizes_fall_back_to_the_warp_kernels(gms):
    g = complete(gms, 36)          # k > 10 is outside the lane kernels' path register; small n: the warp kernels
    for k in (11, 12):             # enumerate every (k-1)-clique
        assert g.kclique_count(k) == comb(36, k)
