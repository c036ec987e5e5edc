"""CPU suite for core and truss numbers: the two sequential peels of tests/truss_oracle.py against networkx and closed
forms, the Kronecker values they pin, and the C++ facade check failing loudly without a GPU."""
import os
import subprocess

import networkx as nx
import numpy as np
import pytest

import truss_oracle as tor
from conftest import random_graph_edges

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def upper_edges(off, nbr):
    """Undirected edges u<v in CSR order: the index order of truss_numbers' output."""
    return [(u, int(v)) for u in range(len(off) - 1) for v in nbr[off[u]:off[u + 1]] if v > u]


def nx_truss(G, edges):
    """Truss numbers from nx.k_truss for increasing k (2 for an edge in no triangle)."""
    t = {e: 2 for e in edges}
    k, H = 3, G
    while True:
        H = nx.k_truss(H, k)
        if H.number_of_edges() == 0:
            break
        for u, v in H.edges():
            t[(min(u, v), max(u, v))] = k
        k += 1
    return np.array([t[e] for e in edges], np.int32)


def check_against_networkx(orc, s, d):
    o = orc.from_el(s, d, True)
    off, nbr = o.csr()
    G = nx.Graph()
    G.add_nodes_from(range(o.n))
    G.add_edges_from((int(a), int(b)) for a, b in zip(s, d) if a != b)
    core = nx.core_number(G)
    assert tor.core_numbers(off, nbr).tolist() == [core[v] for v in range(o.n)]
    assert (tor.truss_numbers(off, nbr) == nx_truss(G, upper_edges(off, nbr))).all()


@pytest.mark.parametrize("seed", range(6))
def test_oracle_matches_networkx_on_random_graphs(orc, seed):
    n, m = [(30, 150), (60, 700), (80, 1500), (40, 500), (200, 3000), (500, 6000)][seed]
    s, d = random_graph_edges(100 + seed, n, m, skew=(seed % 3) * 0.9)
    check_against_networkx(orc, s, d)


def test_oracle_matches_networkx_on_kronecker_10(orc):
    s, d = orc.generate_el(10)
    check_against_networkx(orc, s, d)


@pytest.mark.parametrize("scale,n,m,degeneracy,max_truss", [
    (10, 1024, 10496, 38, 30), (12, 4096, 48386, 65, 47), (14, 16381, 212930, 123, 78)])
def test_oracle_kronecker_pins(orc, scale, n, m, degeneracy, max_truss):
    """Values networkx gives on generate(scale, 16) (it needs 500 s at scale 14, so that row is pinned here only)."""
    g = orc.generate(scale, 16)
    off, nbr = g.csr()
    core, truss = tor.core_numbers(off, nbr), tor.truss_numbers(off, nbr)
    assert (g.n, len(truss), int(core.max()), int(truss.max())) == (n, m, degeneracy, max_truss)
    rank = orc.degeneracy_rank(g)
    assert orc.check_degeneracy_rank(g, rank) == degeneracy


def closed_forms():
    """(name, src, dst, expected truss per edge u<v or one value for all, expected core per vertex or one value)."""
    cases = []
    for n in (3, 4, 6, 9):
        s, d = zip(*[(i, j) for i in range(n) for j in range(i + 1, n)])
        cases.append((f"K{n}", s, d, n, n - 1))
    cases.append(("star", [0] * 12, list(range(1, 13)), 2, 1))
    pages = 7                                             # spine 0-1, page vertices 2..8
    s = [0] + [0] * pages + [1] * pages
    d = [1] + list(range(2, 2 + pages)) * 2
    cases.append(("book", s, d, 3, 2))
    for rim in (4, 5, 40):                                # hub 0, rim 1..rim
        s = [0] * rim + list(range(1, rim + 1))
        d = list(range(1, rim + 1)) + [i % rim + 1 for i in range(1, rim + 1)]
        cases.append((f"wheel{rim}", s, d, 3, 3))
    k5 = [(i, j) for i in range(5) for j in range(i + 1, 5)]
    edges = k5 + [(i + 5, j + 5) for i, j in k5] + [(4, 5)]
    truss = {e: 5 for e in edges}
    truss[(4, 5)] = 2
    cases.append(("two_K5_bridge", [e[0] for e in edges], [e[1] for e in edges], truss, 4))
    # isolated vertices 3..5 below the highest id 6 (a triangle 0-1-2 and an edge 2-6)
    cases.append(("isolated", [0, 1, 0, 2], [1, 2, 2, 6], {(0, 1): 3, (0, 2): 3, (1, 2): 3, (2, 6): 2},
                  [2, 2, 2, 0, 0, 0, 1]))
    return cases


def expected(case, off, nbr, n):
    _, _, _, truss, core = case
    edges = upper_edges(off, nbr)
    t = [truss[e] for e in edges] if isinstance(truss, dict) else [truss] * len(edges)
    c = list(core) if isinstance(core, list) else [core] * n
    return t, c


@pytest.mark.parametrize("case", closed_forms(), ids=lambda c: c[0])
def test_oracle_closed_forms(orc, case):
    _, s, d, _, _ = case
    o = orc.from_el(np.array(s, np.int32), np.array(d, np.int32), True)
    off, nbr = o.csr()
    t, c = expected(case, off, nbr, o.n)
    assert tor.truss_numbers(off, nbr).tolist() == t
    assert tor.core_numbers(off, nbr).tolist() == c


def test_oracle_graph_without_edges():
    off, nbr = np.zeros(5, np.int64), np.zeros(0, np.int32)
    assert len(tor.truss_numbers(off, nbr)) == 0
    assert tor.core_numbers(off, nbr).tolist() == [0, 0, 0, 0]


def test_truss_facade_compiles_and_fails_loudly_without_gpu(gms):
    from test_cpp_facade import build
    exe = build(os.path.join(ROOT, "tests", "cpp", "truss_test.cpp"), os.path.join(ROOT, "build", "truss_test"))
    import torch
    if not torch.cuda.is_available():
        r = subprocess.run([exe], capture_output=True, text=True)
        assert r.returncode == 3 and "CUDA" in r.stderr        # GMSB_ERR_CUDA, never a CPU fallback
