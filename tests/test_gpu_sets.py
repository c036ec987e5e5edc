"""GPU parity (-m gpu): device-resident sets (gmsb_set_*, gms_b200.DeviceSet) against the oracle's SortedSet
operations (oracle.cpp restates sorted_set_operations.h:30-106) on random sets of ragged sizes, the batched
"one set against many" forms, and neighbourhood views of a graph."""
import numpy as np
import pytest

from conftest import random_graph_edges

pytestmark = pytest.mark.gpu


def rand_set(rng, n, hi):
    return np.sort(rng.choice(hi, n, replace=False)).astype(np.int32)       # exactly n elements


def test_binary_operations_against_the_oracle(gms, orc):
    rng = np.random.default_rng(11)
    # (64, 512) / (512, 64) sit on the gallop side of the count kernels' rule (longer >= 8 x shorter), (64, 511) /
    # (511, 64) one element below it, on the merge side
    sizes = [(0, 0), (0, 50), (1, 1), (5, 4000), (4000, 5), (700, 900), (3000, 3000), (33, 32), (20000, 150),
             (64, 512), (64, 511), (512, 64), (511, 64)]
    for na, nb in sizes:
        a, b = rand_set(rng, na, 50000), rand_set(rng, nb, 50000)
        A, B = gms.DeviceSet(rng.permutation(a)), gms.DeviceSet(b)        # the constructor sorts
        assert (A.to_array() == a).all()
        assert A.op_count("intersect", B) == orc.intersect_count(a, b)
        assert A.op_count("union", B) == orc.union_count(a, b)
        assert A.op_count("difference", B) == len(orc.difference(a, b))
        assert B.op_count("difference", A) == len(orc.difference(b, a))
        assert list(A.op_count_many("intersect", [B, A])) == [orc.intersect_count(a, b), na]
        assert (A.op("intersect", B).to_array() == orc.intersect(a, b)).all()
        assert (A.op("union", B).to_array() == orc.union(a, b)).all()
        assert (A.op("difference", B).to_array() == orc.difference(a, b)).all()
        assert (B.op("difference", A).to_array() == orc.difference(b, a)).all()
        C = A.clone()
        C.op_inplace("intersect", B)
        assert C == A.op("intersect", B) and A.cardinality() == len(a)
        for x in (0, 17, 49999):
            assert A.contains(x) == orc.contains(a, x)


def test_add_remove_keep_the_set_sorted(gms):
    rng = np.random.default_rng(5)
    want = set()
    s = gms.DeviceSet()
    for x in rng.integers(0, 200, 300):
        if rng.random() < 0.6:
            s.add(int(x)); want.add(int(x))
        else:
            s.remove(int(x)); want.discard(int(x))
    assert list(s.to_array()) == sorted(want)
    assert gms.DeviceSet.range(7) == gms.DeviceSet([0, 1, 2, 3, 4, 5, 6])
    with pytest.raises(gms.GmsbError):
        gms.DeviceSet([3, -1])


def test_one_set_against_many_and_against_neighbourhoods(gms, orc):
    s, d = random_graph_edges(3, 500, 12000, skew=0.7)
    g, o = gms.Graph.from_edgelist(s, d, True), orc.from_el(s, d, True)
    off, nbr = o.csr()
    rng = np.random.default_rng(2)
    p = rand_set(rng, 200, g.n)
    P = gms.DeviceSet(p)
    members = gms.DeviceSet(rand_set(rng, 120, g.n))
    views = [gms.DeviceSet.neighbourhood(g, int(v)) for v in members.to_array()[:40]]
    difference_count = lambda x, y: len(orc.difference(x, y))                # noqa: E731
    for kind, op, count in (("intersect", orc.intersect, orc.intersect_count), ("union", orc.union, orc.union_count),
                            ("difference", orc.difference, difference_count)):
        want = [count(p, nbr[off[v]:off[v + 1]]) for v in members.to_array()]
        assert list(P.op_count_neighbourhoods(kind, g, members)) == want, kind
        assert list(P.op_count_many(kind, views)) == want[:40], kind
        for v, r in zip(members.to_array()[:40], P.op_many(kind, views)):
            assert (r.to_array() == op(p, nbr[off[v]:off[v + 1]])).all(), kind
    # a view turns into an owning set when it is modified; the graph is untouched
    view = gms.DeviceSet.neighbourhood(g, 7)
    before = view.to_array().copy()
    view.add(int(before.max()) + 1 if len(before) else 0)
    assert (gms.DeviceSet.neighbourhood(g, 7).to_array() == before).all()
    with pytest.raises(gms.GmsbError):
        gms.DeviceSet.neighbourhood(g, g.n)
