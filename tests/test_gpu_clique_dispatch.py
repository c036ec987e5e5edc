"""k-clique counting at the boundaries where `count_on_dag` (gms_b200/csrc/kclique.cu) switches kernels, against exact
counts that do not go through the GPU code.

The kernel that counts the cliques below a vertex u depends on k and on its out-degree d+(u):
  d+ <= 32                 k_kclique_small
  k = 3, 4, 11..16         k_kclique_big<1,512,2> up to 512; above, <1,1024,1> / <2,1024,1> / <4,1024,1> for a largest
                           d+ up to 1024 / 2048 / 4096, with the matrix in global memory once it outgrows shared memory
  k = 5, 6                 k_kclique_lane_mid<1,2,4,8> up to 64 / 128 / 256 / 512, k_kclique_lane_huge above
  k = 7..10                k_kclique_lane_mid<1,2> up to 64 / 128, k_kclique_m1_build + k_kclique_lane_pair above
  d+ > 4096                GMSB_ERR_UNSUPPORTED
Complete graphs pass all of these with any bug that keeps every row a full suffix, so the graphs here are joins and
unions of empty blocks and seeded random blocks (with a planted clique for the large k): dense, irregular rows, and
an exact clique polynomial.  Vertex ids are the orientation order (arcs ascend), so `orient(identity)` keeps it and
every chosen vertex gets exactly the out-degree it is built for; above what a custom orientation may use the library
orients by degree, and pendant leaves put the hub first.

References.  For every vertex v the construction keeps perv[v][j] = number of j-cliques of the sub-DAG on N+(v):
    join of blocks B_1..B_m (ids in that order):  perv(v in B_j) = perv_{B_j}(v) * prod_{l > j} C_{B_l}(x)
    disjoint union:                               perv unchanged
    C_G[k] = sum_v perv[v][k - 1]
The per-vertex polynomials of a random block come from the oracle's pivot counter on each vertex's sub-DAG.  They give
the total, and the share of every kernel class that GMSB_KCLIQUE_TRACE reports.  The CPU test checks the whole scheme
against the pivot counter and the Danisch enumeration on scaled-down instances.  Counts are compared modulo 2^64:
the kernels accumulate in u64."""
import re
from functools import lru_cache
from math import comb, factorial

import numpy as np
import pytest

KMAX = 16
U64 = 1 << 64


# ---- clique polynomials (lists of Python ints, index = clique size, truncated at KMAX) ---------------------------------
def pmul(a, b):
    out = [0] * min(len(a) + len(b) - 1, KMAX + 1)
    for i, x in enumerate(a):
        if x:
            for j, y in enumerate(b[:KMAX + 1 - i]):
                out[i + j] += x * y
    return out


def coef(p, k):
    return p[k] if k < len(p) else 0


class Build:
    """Undirected graph whose ids are its orientation order, with perv[v] = clique polynomial of the sub-DAG on N+(v)."""

    def __init__(self, n, src, dst, perv):
        self.n, self.src, self.dst, self.perv = n, np.asarray(src, np.int64), np.asarray(dst, np.int64), perv

    def poly(self):
        p = [0] * (KMAX + 1)
        p[0] = 1
        for q in self.perv:
            for j, x in enumerate(q[:KMAX]):
                p[j + 1] += x
        return p

    def dplus(self):
        return np.bincount(np.minimum(self.src, self.dst), minlength=self.n)

    def edges32(self):
        return self.src.astype(np.int32), self.dst.astype(np.int32)


def empty(s):
    return Build(s, [], [], [[1]] * s)


def sub_dag_polys(orc, A, verts):
    """Clique polynomial of the sub-DAG induced on N+(v) for each v, from the pivot counter (A: upper-triangular
    boolean adjacency, ids ascending along arcs)."""
    out = []
    for v in verts:
        S = np.nonzero(A[v])[0]
        if len(S) == 0:
            out.append([1])
            continue
        i, j = np.nonzero(np.triu(A[np.ix_(S, S)], 1))
        off = np.zeros(len(S) + 1, np.int64)
        np.add.at(off, i + 1, 1)
        dag = orc.from_csr(np.cumsum(off), j.astype(np.int32), True)
        cnt = orc.clique_counts_pivot(dag, KMAX)
        out.append([1] + cnt[1:])
    return out


@lru_cache(maxsize=None)
def _random_block(s, p, seed, plant):
    from oracle import binding
    rng = np.random.default_rng(seed)
    A = np.triu(rng.random((s, s)) < p, 1)
    if plant:
        q = np.sort(rng.choice(s, min(plant, s), replace=False))
        A[np.ix_(q, q)] = True
        A = np.triu(A, 1)
    i, j = np.nonzero(A)
    return i, j, sub_dag_polys(binding.oracle(), A, range(s))


def random_block(s, p=0.2, seed=1, plant=12):
    """G(s, p) with a clique on `plant` random members."""
    i, j, perv = _random_block(s, p, seed, plant)
    return Build(s, i, j, perv)


def join(*blocks):
    """Every vertex of a block adjacent to every vertex of the others; ids block by block."""
    src, dst, perv, base = [], [], [], 0
    starts = np.cumsum([0] + [b.n for b in blocks])
    later = [[1]] * len(blocks)
    for j in range(len(blocks) - 2, -1, -1):
        later[j] = pmul(later[j + 1], blocks[j + 1].poly())
    for j, b in enumerate(blocks):
        src.append(b.src + base)
        dst.append(b.dst + base)
        rest = np.arange(starts[j + 1], starts[-1])
        mine = np.arange(base, base + b.n)
        src.append(np.repeat(mine, len(rest)))
        dst.append(np.tile(rest, b.n))
        perv += [pmul(q, later[j]) for q in b.perv]
        base += b.n
    return Build(base, np.concatenate(src), np.concatenate(dst), perv)


def union(*blocks):
    src, dst, perv, base = [], [], [], 0
    for b in blocks:
        src.append(b.src + base)
        dst.append(b.dst + base)
        perv += b.perv
        base += b.n
    return Build(base, np.concatenate(src), np.concatenate(dst), perv)


def hub(empties, r, p=0.2, seed=1, plant=12):
    """A vertex joined to X = E(e_1) + ... + E(e_m) + R (joins, ids in that order), R = random_block(r): the hub has
    d+ = sum(e) + r, a member of the first empty block has the candidate set E(e_2) + ... + R after (hub, member)."""
    return join(empty(1), *[empty(e) for e in empties], random_block(r, p, seed, plant))


def hub_d(d, seed=1, **kw):
    """hub() with d+ = d: a quarter of X in one empty block, the rest random."""
    return hub((d // 4,), d - d // 4, seed=seed, **kw)


# ---- what the library does with a graph --------------------------------------------------------------------------------
def custom_limit():
    """Largest max d+ for which kclique_count keeps the caller's ascending orientation: the warp kernels' matrix
    (kclique.cu: matrix_words) plus 28 KB of static scratch fits the shared-memory opt-in of one block."""
    import torch
    optin = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    D = 33
    while True:
        nxt = D + 1
        rw = ((nxt + 63) >> 6) << 1
        if (((nxt + 1) & ~1) + nxt * rw) * 4 + 28 * 1024 > optin:
            return D, optin
        D = nxt


def lane_huge_in_smem(D, optin):
    """k_kclique_lane_huge keeps its matrix in shared memory (kclique_lane.cuh: huge_smem_words)."""
    p1 = ((D + 63) >> 6) | 1
    words = D * p1 + 512 * 9 + 16 * p1 + ((D + 1) >> 1) + ((p1 + 2) >> 1) + 512 // 4
    return words * 8 + 2048 <= optin


def on_gpu(gms, b):
    """(undirected handle, DAG handle in the construction's order, exported out-degrees of that DAG)."""
    s, d = b.edges32()
    g = gms.Graph.from_edgelist(s, d, True)
    dag = g.orient(np.arange(b.n, dtype=np.int32))
    off, nbr = dag.export_csr()
    dp = np.diff(off)
    assert np.array_equal(dp, b.dplus())          # the library's DAG is the one the references describe
    return g, dag, dp


TRACE = re.compile(r"\[gmsb kclique k=(\d+)\] (\S+)\s+vertices=(\d+) ms=\S+ cliques=(\d+)")
LANE_CLASSES = {"huge(d+>512)": (512, 1 << 30), "mid8(<=512)": (256, 512), "mid4(<=256)": (128, 256),
                "mid2(<=128)": (64, 128), "mid1(<=64)": (32, 64)}
PAIR_CLASSES = {"pair(d+>128)": (128, 1 << 30), "mid2(<=128)": (64, 128), "mid1(<=64)": (32, 64)}


def check_trace(dag, b, dp, k, capfd, monkeypatch, must_run):
    """Counts once without and once with GMSB_KCLIQUE_TRACE: equal totals, and every class the trace reports has the
    vertices (d+ in its range and >= k - 1) and the cliques (sum of their (k-1)-cliques below) the DAG says."""
    total = dag.kclique_count(k)
    capfd.readouterr()
    monkeypatch.setenv("GMSB_KCLIQUE_TRACE", "1")
    traced = dag.kclique_count(k)
    monkeypatch.delenv("GMSB_KCLIQUE_TRACE")
    lines = [m.groups() for m in TRACE.finditer(capfd.readouterr().err)]
    assert traced == total
    classes = PAIR_CLASSES if k >= 7 else LANE_CLASSES
    assert [name for _, name, _, _ in lines] == list(classes), lines
    for kk, name, nv, cl in lines:
        lo, hi = classes[name]
        vs = np.nonzero((dp > lo) & (dp <= hi) & (dp >= k - 1))[0]
        assert int(kk) == k and int(nv) == len(vs), (k, name, nv, len(vs))
        assert int(cl) == sum(coef(b.perv[v], k - 1) for v in vs) % U64, (k, name)
        if name in must_run:
            assert len(vs) > 0, (k, name)
    return total


# ---- the graphs ------------------------------------------------------------------------------------------------------
# d+ 31 / 32 / 33 on both sides of k_kclique_small, K_15 planted so that every k up to 16 has cliques
def g_small():
    return union(*[join(empty(1), random_block(d, 0.5, seed=d, plant=15)) for d in (31, 32, 33)])


# the k_kclique_big<1,512,2> class on both sides of every lane class boundary, K_15 planted
MID_DS = (33, 64, 65, 128, 129, 256, 257, 512)


def g_warp_mid():
    return union(*[hub_d(d, seed=d, plant=15) for d in MID_DS])


# largest d+ D above 512 with the caller's orientation; a d+ = 40 hub keeps the <= 512 class busy
def g_warp_huge(D):
    return union(hub((16,), D - 16, seed=D, plant=15), hub_d(40, seed=40, plant=15))


# the lane classes of k = 5, 6: below and above 64 / 128 / 256 / 512; the rows of the first empty block's members hold
# 193 (d = 257) and 192 (d = 256) members: one more than the per-warp M3 box takes, and exactly what it takes
LANE_DS = (33, 64, 65, 128, 129, 256, 257, 512, 513, 1024)


def g_lane(extra=()):
    return union(*[hub_d(d, seed=d) for d in LANE_DS + tuple(extra)])


# the pair kernel (k = 7..10): after (hub, member of the first empty block) the candidate set holds
# 97, 128, 129, 192, 193, 256, 257, 448 (40 of whose rows hold 408 > 192 members) and 640 (> 512: the CTA expands it,
# and its children, up to 190 members, are compacted with four padded words)
PAIR_HUBS = (((16,), 48), ((16,), 49), ((32,), 96), ((32,), 97), ((42,), 128), ((42,), 129), ((64,), 192),
             ((64,), 193), ((85,), 256), ((85,), 257), ((32, 40), 408))


def g_pair():
    parts = [hub(e, r, seed=r) for e, r in PAIR_HUBS]
    return union(*parts, hub((60,), 640, p=0.3, seed=640))


def degree_hub(D, seed=7):
    """hub + X, X = E(a) + R (join, a = D // 2, R sparse with a planted K_15) and pendant leaves that lift every member
    of X to degree D + 1: ordering by degree puts the hub (degree D) before all of X, so d+(hub) = D.  Leaves add
    vertices and edges and no clique of size >= 3.  Returns (src, dst, n, clique polynomial)."""
    a = D // 2
    b = hub((a,), D - a, p=0.004, seed=seed, plant=15)
    deg = np.bincount(np.concatenate([b.src, b.dst]), minlength=b.n)
    lift = D + 1 - deg
    lift[0] = 0
    assert (lift[1:] >= 0).all()
    leaves = int(lift.sum())
    owner = np.repeat(np.arange(b.n), lift)
    src = np.concatenate([b.src, owner]).astype(np.int32)
    dst = np.concatenate([b.dst, b.n + np.arange(leaves)]).astype(np.int32)
    p = b.poly()
    p[1] += leaves
    p[2] += leaves
    return src, dst, b.n + leaves, p


def degree_dag_dplus(g):
    off, _ = g.orient(g.degree_order(True)).export_csr()
    return np.diff(off)


# ---- CPU: the references ---------------------------------------------------------------------------------------------
def dag_of(orc, b):
    s, d = np.minimum(b.src, b.dst), np.maximum(b.src, b.dst)
    order = np.lexsort((d, s))
    off = np.zeros(b.n + 1, np.int64)
    np.add.at(off, s + 1, 1)
    return orc.from_csr(np.cumsum(off), d[order].astype(np.int32), True)


def test_references_against_pivot_and_danisch(orc):
    """Scaled-down instances of every construction: the closed form against the pivot counter and the Danisch
    enumeration, and each vertex's polynomial against the pivot counter on its own sub-DAG."""
    cases = [
        union(*[join(empty(1), random_block(d, 0.5, seed=d, plant=15)) for d in (12, 13)]),
        union(*[hub_d(d, seed=d, plant=9) for d in (20, 33, 41)]),
        union(hub((6, 5), 30, seed=3), hub((9,), 40, p=0.3, seed=4)),
        join(empty(3), union(hub((4,), 12, seed=5), empty(2)), random_block(15, 0.5, seed=6, plant=6)),
    ]
    for b in cases:
        dag = dag_of(orc, b)
        want = b.poly()
        got = orc.clique_counts_pivot(dag, KMAX)
        assert [coef(want, k) % U64 for k in range(1, KMAX + 1)] == got[1:], (b.n, want, got)
        for k in range(3, 7):
            assert dag.kclique(k) == coef(want, k)
        A = np.zeros((b.n, b.n), bool)
        A[np.minimum(b.src, b.dst), np.maximum(b.src, b.dst)] = True
        for v, q in zip(range(b.n), sub_dag_polys(orc, A, range(b.n))):
            assert [coef(q, j) for j in range(KMAX)] == [coef(b.perv[v], j) for j in range(KMAX)], v
    # the degree construction: the hub comes first under the degree order and has d+ = D
    for D in (24, 41):
        s, d, n, want = degree_hub(D)
        g = orc.from_el(s, d, True)
        dag = g.induce_directed(g.degree_order(True))
        off, _ = dag.csr()
        assert np.diff(off).max() == D
        got = orc.clique_counts_pivot(dag, KMAX)
        assert [coef(want, k) for k in range(1, KMAX + 1)] == got[1:]
        assert dag.kclique(4) == want[4]


def test_polynomial_algebra():
    # K_4 as a join of four single vertices, K_{2,3} as a join of two empty blocks, C(x) of a union
    k4 = join(*[empty(1)] * 4)
    assert k4.poly()[:5] == [1, 4, 6, 4, 1]
    assert join(empty(2), empty(3)).poly()[:3] == [1, 5, 6]
    assert union(k4, empty(3)).poly()[:5] == [1, 7, 6, 4, 1]
    assert hub((2,), 3, p=0.0, plant=0).poly()[:4] == [1, 6, 2 * 1 + 3 + 2 * 3, 2 * 3]


# ---- GPU ------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu


@gpu
def test_small_kernel_at_32_and_33(gms):
    b = g_small()
    g, dag, dp = on_gpu(gms, b)
    assert sorted(dp)[-3:] == [31, 32, 33]
    want = b.poly()
    assert want[16] > 0
    for k in range(3, KMAX + 1):
        assert g.kclique_count(k) == want[k] % U64, k
        assert dag.kclique_count(k) == want[k] % U64, k


@gpu
def test_warp_kernel_up_to_512(gms):
    b = g_warp_mid()
    g, dag, dp = on_gpu(gms, b)
    assert dp.max() == 512 and {d for d in MID_DS} <= set(dp.tolist())
    want = b.poly()
    for k in (3, 4) + tuple(range(11, KMAX + 1)):
        assert want[k] > 0
        assert dag.kclique_count(k) == want[k] % U64, k


@gpu
@pytest.mark.parametrize("D", [513, 1024, 1025, "limit"])
def test_warp_kernel_above_512_custom_orientation(gms, D):
    """<1,1024,1> (513, 1024), <2,1024,1> (1025 and the largest d+ the caller's orientation may have)."""
    limit, _ = custom_limit()
    assert limit >= 1025
    D = limit if D == "limit" else D
    b = g_warp_huge(D)
    g, dag, dp = on_gpu(gms, b)
    assert dp.max() == D
    want = b.poly()
    for k in (3, 4) + tuple(range(11, KMAX + 1)):
        assert dag.kclique_count(k) == want[k] % U64, k


@gpu
@pytest.mark.parametrize("D", [2048, 2049, 4096])
def test_warp_kernel_degree_orientation(gms, D):
    """<2,1024,1> at 2048 and <4,1024,1> at 2049 and 4096, matrix in global memory; the library orients by degree."""
    s, d, n, want = degree_hub(D)
    g = gms.Graph.from_edgelist(s, d, True)
    dp = degree_dag_dplus(g)
    assert dp.max() == D and np.count_nonzero(dp == D) == 1
    for k in (3, 4) + tuple(range(11, KMAX + 1)):
        assert g.kclique_count(k) == want[k] % U64, k


@gpu
def test_out_degree_above_4096_is_unsupported(gms):
    s, d, n, _ = degree_hub(4097)
    g = gms.Graph.from_edgelist(s, d, True)
    assert degree_dag_dplus(g).max() == 4097
    with pytest.raises(gms.GmsbError) as e:
        g.kclique_count(3)
    assert e.value.code == -4
    dag = g.orient(np.arange(n, dtype=np.int32))       # ascending, but too wide to keep: re-oriented by degree
    with pytest.raises(gms.GmsbError) as e:
        dag.kclique_count(4)
    assert e.value.code == -4
    del g, dag
    # the library keeps answering
    s, d, n, want = degree_hub(4096)
    assert gms.Graph.from_edgelist(s, d, True).kclique_count(3) == want[3]
    b = g_small()
    assert on_gpu(gms, b)[1].kclique_count(5) == b.poly()[5]


@gpu
@pytest.mark.parametrize("which", ["smem", "spilled"])
def test_lane_kernels_k5_k6(gms, capfd, monkeypatch, which):
    """lane_mid 1/2/4/8 on both sides of each boundary, lane_huge with its matrix in shared memory (max d+ 1024) and
    spilled to global memory (the largest d+ the caller's orientation may have)."""
    limit, optin = custom_limit()
    b = g_lane() if which == "smem" else g_lane((limit,))
    g, dag, dp = on_gpu(gms, b)
    assert dp.max() == (1024 if which == "smem" else limit)
    assert lane_huge_in_smem(int(dp.max()), optin) == (which == "smem")
    want = b.poly()
    for k in (5, 6):
        got = check_trace(dag, b, dp, k, capfd, monkeypatch, must_run=set(LANE_CLASSES))
        assert got == want[k] % U64, k


@gpu
def test_pair_kernel_k7_to_k10(gms, capfd, monkeypatch):
    b = g_pair()
    g, dag, dp = on_gpu(gms, b)
    assert dp.max() == 700 and {64, 65, 128, 129, 170, 171, 256, 257, 341, 342, 480} <= set(dp.tolist())
    want = b.poly()
    for k in (7, 8, 9, 10):
        assert want[k] > 0
        got = check_trace(dag, b, dp, k, capfd, monkeypatch, must_run=set(PAIR_CLASSES))
        assert got == want[k] % U64, k


@gpu
def test_partitions_are_additive(gms):
    """sum over part_index of kclique_count(k, part_index, P) is the total, for every family; the lone d+ = 600 hub
    has one work item (k = 4) or fewer than P (k = 5 cuts it into ten parts of 64 rows) in its class."""
    cases = [(g_warp_mid(), (4, 12)), (g_lane(), (5, 6)), (g_pair(), (7, 8, 9, 10)),
             (hub((), 600, p=0.25, seed=600), (4, 5, 7))]
    for b, ks in cases:
        g, dag, dp = on_gpu(gms, b)
        want = b.poly()
        for k in ks:
            for P in (2, 3, 7):
                assert sum(dag.kclique_count(k, p, P) for p in range(P)) == want[k] % U64, (b.n, k, P)


@gpu
def test_ordered_count_wraps_like_size_t(gms):
    i, j = np.triu_indices(30, 1)
    g = gms.Graph.from_edgelist(i.astype(np.int32), j.astype(np.int32), True)
    for k in (14, 15, 16):
        assert g.kclique_count_ordered(k) == factorial(k) * comb(30, k) % U64, k
    assert factorial(16) * comb(30, 16) > U64
