"""GPU suite (-m gpu) for gmsb_core_numbers and gmsb_truss_numbers: exact equality with the sequential CPU peels of
tests/truss_oracle.py, the two-pass protocol and refusals, determinism, invariants against the existing operators at
scales 20 and 22, and both peel kernel classes on each side of their row-length threshold."""
import os
import subprocess

import numpy as np
import pytest

import truss_oracle as tor
from conftest import random_graph_edges
from test_truss_cpu import closed_forms, expected

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LONG_ROW = 1024          # truss.cu kLongRow: a frontier edge whose shorter row is this long is peeled by a whole CTA


def upper_pairs(off, nbr):
    """Endpoints (a, b), a < b, of every undirected edge in CSR order (= the index order of truss_numbers)."""
    rows = np.repeat(np.arange(len(off) - 1, dtype=np.int32), np.diff(off))
    keep = nbr > rows
    return rows[keep], nbr[keep]


def check_equal(gms, orc, s, d):
    g = gms.Graph.from_edgelist(s, d, True)
    off, nbr = orc.from_el(s, d, True).csr()              # the graph built on the CPU, not the GPU's own CSR
    t = g.truss_numbers()
    assert t.dtype == np.int32 and t.tobytes() == tor.truss_numbers(off, nbr).tobytes()
    assert g.core_numbers().tobytes() == tor.core_numbers(off, nbr).tobytes()
    return g, t


@pytest.mark.parametrize("case", closed_forms(), ids=lambda c: c[0])
def test_closed_forms(gms, case):
    """K_n peels every edge of every triangle in the same sub-round; the wheels' hub meets all rim edges at once."""
    _, s, d, _, _ = case
    g = gms.Graph.from_edgelist(np.array(s, np.int32), np.array(d, np.int32), True)
    off, nbr = g.export_csr()
    t, c = expected(case, off, nbr, g.n)
    assert g.truss_numbers().tolist() == t
    assert g.core_numbers().tolist() == c


@pytest.mark.parametrize("seed", range(6))
def test_random_graphs_against_oracle(gms, orc, seed):
    n, m = [(40, 300), (300, 6000), (2000, 30000), (100, 4000), (5000, 200000), (60, 1700)][seed]
    check_equal(gms, orc, *random_graph_edges(200 + seed, n, m, skew=(seed % 3) * 0.9))


@pytest.mark.parametrize("scale", [10, 12, 14, 16])
def test_kronecker_against_oracle(gms, orc, scale):
    g, t = check_equal(gms, orc, *gms.generate_rmat(scale))
    pins = {10: (38, 30), 12: (65, 47), 14: (123, 78)}
    if scale in pins:
        assert (int(g.core_numbers().max()), int(t.max())) == pins[scale]


def test_uniform_and_skewed_rmat_against_oracle(gms, orc):
    check_equal(gms, orc, *gms.generate_uniform(14))
    check_equal(gms, orc, *gms.generate_rmat(14, a=0.65, b=0.15, c=0.15))       # heavy hubs


def test_hub_with_thousands_of_frontier_edges(gms, orc):
    """A wheel with a 5000-vertex rim: every spoke joins the same frontier and meets the others at the hub; a K_12 on
    rim vertices keeps part of the graph alive at higher levels."""
    rim = 5000
    s = [0] * rim + list(range(1, rim + 1))
    d = list(range(1, rim + 1)) + [i % rim + 1 for i in range(1, rim + 1)]
    clique = list(range(1, 2000, 166))[:12]
    for i in clique:
        for j in clique:
            if i < j:
                s.append(i)
                d.append(j)
    check_equal(gms, orc, np.array(s, np.int32), np.array(d, np.int32))


def hub_graph(seed, degrees, p):
    """Hubs 0..h-1 joined by a seeded G(h, p); hub i gets pendant leaves up to degrees[i] neighbours.  Hub-hub edges
    between two hubs of degree >= LONG_ROW go to the CTA class, the others to the warp class."""
    rng = np.random.default_rng(seed)
    h = len(degrees)
    iu, ju = np.triu_indices(h, 1)
    keep = rng.random(len(iu)) < p
    src, dst = list(iu[keep]), list(ju[keep])
    hub_deg = np.bincount(np.concatenate([iu[keep], ju[keep]]), minlength=h)
    nxt = h
    for i in range(h):
        leaves = degrees[i] - int(hub_deg[i])
        assert leaves >= 0
        src += [i] * leaves
        dst += list(range(nxt, nxt + leaves))
        nxt += leaves
    return np.array(src, np.int32), np.array(dst, np.int32)


@pytest.mark.parametrize("seed,p", [(1, 0.5), (2, 0.8)])
def test_peel_kernel_classes_at_their_threshold(gms, orc, seed, p):
    degrees = [LONG_ROW - 1, LONG_ROW, LONG_ROW + 1, LONG_ROW - 2, 2 * LONG_ROW] * 8
    s, d = hub_graph(seed, degrees, p)
    g, t = check_equal(gms, orc, s, d)
    off, nbr = g.export_csr()
    a, b = upper_pairs(off, nbr)
    deg = np.diff(off)
    hub_edges = (a < len(degrees)) & (b < len(degrees))
    shorter = np.minimum(deg[a], deg[b])
    assert (hub_edges & (shorter == LONG_ROW - 1)).any() and (hub_edges & (shorter == LONG_ROW)).any()
    assert (t[hub_edges] > 3).any()              # the hubs' triangles decide truss numbers above the first levels


def test_two_pass_protocol_and_empty_graph(gms):
    import ctypes as C
    s, d = gms.generate_rmat(10)
    g = gms.Graph.from_edgelist(s, d, True)
    m = C.c_int64(-1)
    assert gms.lib().gmsb_truss_numbers(g.h, None, C.byref(m)) == 0
    assert m.value == g.slots // 2 == 10496
    empty = gms.Graph.from_csr(np.zeros(4, np.int64), np.zeros(0, np.int32))
    assert len(empty.truss_numbers()) == 0
    assert empty.core_numbers().tolist() == [0, 0, 0]


def test_refusals(gms):
    import torch
    off, nbr = np.array([0, 1, 2, 2], np.int64), np.array([1, 0], np.int32)
    directed = gms.Graph.from_csr(off, nbr, directed=True)
    s, d = gms.generate_rmat(8)
    g = gms.Graph.from_edgelist(s, d, True)
    dag = g.orient(g.degree_order(True))
    off, nbr = g.export_csr()
    shard = gms.capi.Shard(off, nbr, 0, 1)
    pieces = torch.zeros(max(shard.piece_len, 1), dtype=torch.int32, device="cuda")
    dplus = torch.zeros(g.n, dtype=torch.int32, device="cuda")
    shard.export(pieces.data_ptr(), dplus.data_ptr())
    torch.cuda.synchronize()
    sharded = shard.finish(pieces.data_ptr(), max(shard.piece_len, 1), dplus.data_ptr())
    assert sharded.tc_total() == g.tc_total()
    for h in (directed, dag, sharded):
        for call in (h.truss_numbers, h.core_numbers):
            with pytest.raises(gms.GmsbError) as e:
                call()
            assert e.value.code == -1                   # GMSB_ERR_INVALID


def test_determinism_and_relabelling(gms):
    s, d = gms.generate_rmat(16)
    g = gms.Graph.from_edgelist(s, d, True)
    t, c = g.truss_numbers(), g.core_numbers()
    assert g.truss_numbers().tobytes() == t.tobytes() and g.core_numbers().tobytes() == c.tobytes()
    rel = g.relabel_by_degree()
    off, nbr = g.export_csr()
    roff, rnbr = rel.export_csr()
    # RelabelByDegree: degree descending, id descending -> new id = position
    deg = np.diff(off)
    new_of = np.empty(g.n, np.int64)
    new_of[np.lexsort((-np.arange(g.n), -deg))] = np.arange(g.n)
    assert (np.diff(roff)[new_of] == deg).all()
    a, b = upper_pairs(off, nbr)
    ra, rb = upper_pairs(roff, rnbr)
    rt = rel.truss_numbers()
    key = np.minimum(new_of[a], new_of[b]) * g.n + np.maximum(new_of[a], new_of[b])
    rkey = ra.astype(np.int64) * g.n + rb
    order = np.argsort(rkey)
    assert (rt[order[np.searchsorted(rkey[order], key)]] == t).all()
    assert (rel.core_numbers()[new_of] == c).all()


@pytest.mark.parametrize("scale", [20, 22])
def test_invariants_at_scale(gms, orc, scale):
    s, d = gms.generate_rmat(scale)
    g = gms.Graph.from_edgelist(s, d, True)
    t, c = g.truss_numbers(), g.core_numbers()
    off, nbr = g.export_csr()
    a, b = upper_pairs(off, nbr)
    assert len(t) == len(a) and t.min() >= 2
    cn = g.edge_similarity("comm_neigh")
    assert (t - 2 <= cn).all()
    assert (t <= np.minimum(c[a], c[b]) + 1).all()
    assert int(c.max()) == orc.core_number_of_rank(orc.from_csr(off, nbr), g.degeneracy_rank())
    for k in sorted({3, int(np.median(t)), int(t.max())}):
        keep = t >= k
        if not keep.any():
            continue
        sub = gms.Graph.from_edgelist(a[keep], b[keep], True)
        assert sub.edge_similarity("comm_neigh").min() >= k - 2, k


def test_truss_facade_on_gpu(gms):
    from test_cpp_facade import build
    exe = build(os.path.join(ROOT, "tests", "cpp", "truss_test.cpp"), os.path.join(ROOT, "build", "truss_test"))
    r = subprocess.run([exe], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "all checks passed" in r.stdout
