"""Triangle counting at the boundaries of its schedule (gms_b200/csrc/tc.cu: k_classify, k_item_keys, scatter_edge) and
per-edge support (tc_support.cu), against exact counts that do not go through the GPU code.

In rank space (degree ascending, then id) every oriented edge (u,v) with a non-empty suffix of N+(u) after v is a
descriptor of its closing vertex v, and |suffix ∩ N+(v)| = |N+(u) ∩ N+(v)| is what it counts.  The schedule sends it
  to a hub bitmap item when v is a hub (variant bitmap, or auto and work(v) >= hub_min_work; span(v) <= hub_bits),
      in the window class of v: NEAR (the window from (v+1) & ~31 reaches n - 1 in kNearWords words), small
      (span <= 439968 bits) or wide; inside an item by length class: <= 8, <= 96, longer;
  else to the gallop list when max(len, d+(v)) >= ratio * min(len, d+(v)), to the merge list otherwise.
`plan_model` restates that in numpy and gives every statistic of gmsb_tc_stats and the triangles of every class, which
GMSB_TC_TRACE reports per launch.  The graphs put vertices and descriptors on both sides of each boundary:
  g_small  circulants C_n(1..k) (regular, so rank == id; every suffix length 0..k-1, k - 97 class-2 descriptors in
           the one item of a vertex with k <= 102, two items at k = 725), seeded random blocks, and pendant vertices whose
           suffixes reach the last vertex (suffix elements beyond every hub's window)
  g_far    n = 600 k vertices, all of degree 2 (rank == id): triangles {a, v, c} put the closing vertex v at a chosen
           span and NEAR reach, 4-cycles a-v-x-w put a suffix element w far outside v's window
  g_wide   a hub of work 1024 and span 524288 beside small-window hubs: the support kernel's window at its widest
References: per-edge support from a dense A @ A per connected component (exact in float32 at these sizes) or, for
g_far, from the construction (1 on every triangle edge, 0 on the 4-cycles); tc_vertex2 = the row sums; the total from the oracle in the CPU test."""
import re
from functools import lru_cache

import numpy as np
import pytest

SHORT, MID = 8, 96                          # tc_plan.cuh: kShortLen, kMidLen
NEAR_WORDS = 55000 // 4 - 1                 # tc.cu: kNearWords (kSmallWindowBytes / 4 - 1)
ITEM_COST = 262144                          # tc.cu: kItemCost
SMEM_OPTIN = 232448                         # B200: shared memory per block with the opt-in (227 KB)
CLASSES = ("near", "small", "wide", "merge", "gallop")


# ---- graphs ----------------------------------------------------------------------------------------------------------
class G:
    """Undirected simple graph: n, edges (src < dst), no duplicates."""

    def __init__(self, n, src, dst):
        src, dst = np.asarray(src, np.int64), np.asarray(dst, np.int64)
        a, b = np.minimum(src, dst), np.maximum(src, dst)
        assert (a != b).all()
        o = np.lexsort((b, a))
        self.n, self.a, self.b = n, a[o], b[o]
        assert not ((np.diff(self.a) == 0) & (np.diff(self.b) == 0)).any(), "duplicate edge"
        self.deg = np.bincount(np.concatenate([self.a, self.b]), minlength=n)
        self.rank = np.empty(n, np.int64)
        self.rank[np.lexsort((np.arange(n), self.deg))] = np.arange(n)   # degree ascending, then id
        ra, rb = self.rank[self.a], self.rank[self.b]
        lo, hi = np.minimum(ra, rb), np.maximum(ra, rb)
        o = np.lexsort((hi, lo))
        self.dnbr = hi[o]
        self.doff = np.concatenate([[0], np.cumsum(np.bincount(lo, minlength=n))])
        self._tri = self._sup = None

    def edges32(self):
        return self.a.astype(np.int32), self.b.astype(np.int32)

    def slot_triangles(self):
        """|N+(u) ∩ N+(v)| for every slot (u,v) of the rank-space DAG."""
        if self._tri is None:
            u = np.repeat(np.arange(self.n), np.diff(self.doff))
            if self.n <= 20000:
                self._tri = per_component(self.n, u, self.dnbr, lambda D: D @ D.T, upper=True)
            else:                                   # sparse: g_far has in-degrees of at most 2
                from scipy import sparse
                D = sparse.csr_matrix((np.ones(len(u), np.int64), (u, self.dnbr)), shape=(self.n, self.n))
                T = (D @ D.T).tocsr()
                self._tri = np.asarray(T[u, self.dnbr]).ravel().astype(np.int64)
        return self._tri

    def support(self):
        """Triangles through every edge (a < b, in CSR order of the original ids)."""
        if self._sup is None:
            self._sup = (per_component(self.n, self.a, self.b, lambda A: A @ A) if self.n <= 20000
                         else self.closed_support)
        return self._sup


def per_component(n, r, c, product, upper=False):
    """product(X)[r, c] for the 0/1 matrix X of the edges (r, c) (symmetric unless `upper`), one dense float32 block per
    connected component (exact: every entry is below 2^24)."""
    from scipy import sparse
    from scipy.sparse.csgraph import connected_components
    _, lab = connected_components(sparse.csr_matrix((np.ones(len(r)), (r, c)), shape=(n, n)), directed=False)
    out = np.zeros(len(r), np.int64)
    el = lab[r]
    for comp in np.unique(el):
        verts = np.nonzero(lab == comp)[0]
        loc = np.full(n, -1)
        loc[verts] = np.arange(len(verts))
        sel = np.nonzero(el == comp)[0]
        X = np.zeros((len(verts), len(verts)), np.float32)
        X[loc[r[sel]], loc[c[sel]]] = 1
        if not upper:
            X[loc[c[sel]], loc[r[sel]]] = 1
        out[sel] = product(X)[loc[r[sel]], loc[c[sel]]].astype(np.int64)
    return out


def circulant(n, S, base=0):
    """C_n(S): x ~ x + s (mod n); n > 2 max(S) keeps the edges distinct."""
    S = np.asarray(S, np.int64)
    assert n > 2 * S.max()
    x = np.repeat(np.arange(n), len(S))
    return x + base, (x + np.tile(S, n)) % n + base


def circulant_support(n, S):
    """support of an edge at offset s: #{x in ±S : s - x in ±S (mod n)}, for every s in S."""
    pm = np.concatenate([S, -np.asarray(S)]) % n
    mem = np.zeros(n, bool)
    mem[pm] = True
    return {s: int(mem[(s - pm) % n].sum()) for s in S}


CIRC_KS = (98, 99, 100, 101, 102, 258, 725)
SMALL_CIRC_BASE = 1200 + 600 + 103


@lru_cache(maxsize=None)
def g_small():
    """A seeded random block with a planted K_40 (light vertices, gallop and merge pairs), a dense random block,
    C_103(1..50) and C_{3k+2}(1..k) for the k of CIRC_KS; every third vertex x of C_103 has an in-edge from a pendant
    vertex whose suffix after x is the last vertex of the circulants, far past the window of every hub."""
    rng = np.random.default_rng(5)
    R = 1200
    A = np.triu(rng.random((R, R)) < 0.012, 1)
    q = np.sort(rng.choice(R, 40, replace=False))
    A[np.ix_(q, q)] = True
    A = np.triu(A, 1)
    i, j = np.nonzero(A)
    src, dst = [i], [j]
    # a dense random block: merge pairs of 512 and more elements whose common elements fall anywhere in a tile
    B = np.triu(rng.random((600, 600)) < 0.6, 1)
    i, j = np.nonzero(B)
    src.append(i + R)
    dst.append(j + R)
    R += 600
    base = R
    s, d = circulant(103, np.arange(1, 51), base)
    src.append(s)
    dst.append(d)
    long_from = np.arange(base, base + 103, 3)
    base += 103
    for k in CIRC_KS:
        s, d = circulant(3 * k + 2, np.arange(1, k + 1), base)
        src.append(s)
        dst.append(d)
        base += 3 * k + 2
    # pendant vertices p (degree 2, no in-edge) with N+(p) = {x, last vertex}: the suffix of (p, x) is the last vertex
    p = base + np.arange(len(long_from))
    src += [p, p]
    dst += [long_from, np.full(len(p), base - 1)]
    base += len(p)
    s, d = sliced_hub(base)
    src.append(s)
    dst.append(d)
    return G(base + SLICED_N, np.concatenate(src), np.concatenate(dst))


SLICED_S, SLICED_Q, SLICED_L, SLICED_T = 700, 700, 660, 400
SLICED_N = SLICED_S + SLICED_Q + SLICED_L + 1 + SLICED_T


def sliced_hub(base):
    """A hub x whose first item holds class-0 descriptors only: ids S (700), Q (700), L (660), x, T (400).  T is a
    clique joined to x, L and Q; every s in S has N+(s) = {x, one member of T} (700 suffixes of length 1), every l in L
    has N+(l) = {x} + T (660 of length 400).  Q lifts the degree of T to that of x, so x ranks below T.  work(x) =
    660 * 400 + 700 cuts x into two items of 680 descriptors: [0, 680) is all class 0, [680, 1360) has its boundary at
    20."""
    S = base + np.arange(SLICED_S)
    Q = S[-1] + 1 + np.arange(SLICED_Q)
    L = Q[-1] + 1 + np.arange(SLICED_L)
    x = L[-1] + 1
    T = x + 1 + np.arange(SLICED_T)
    ti, tj = np.triu_indices(SLICED_T, 1)
    src = [S, S, np.full(SLICED_L, x), np.full(SLICED_T, x), np.repeat(L, SLICED_T), np.repeat(Q, SLICED_T), T[ti]]
    dst = [np.full(SLICED_S, x), T[np.arange(SLICED_S) % SLICED_T], L, T, np.tile(T, SLICED_L), np.tile(T, SLICED_Q),
           T[tj]]
    return np.concatenate(src), np.concatenate(dst)


WIDE_FILL, WIDE_K = 524256, 120


@lru_cache(maxsize=None)
def g_wide():
    """A hub v of work 1024 whose window is 524288 bits wide, beside hubs with small windows, for the support kernel
    (default options, so its window is as wide as the widest hub's).  Ids: u_1..u_32, v; a triangle-free 34-regular
    filler C_N(1, 3, .., 33) (N even, so every cycle is even); Y = K_32; C_362(1..120).  N+(u_i) = {v} + Y and
    N+(v) = {y_1}: v has 32 in-edges of suffix length 32, and the filler (degree 34 > 33) ranks between v and Y.
    The circulant's hubs have work >= 1024 and suffixes of every length class."""
    u = np.arange(32)
    v = 32
    f0 = 33
    fs, fd = circulant(WIDE_FILL, np.arange(1, 34, 2), f0)
    y = f0 + WIDE_FILL + np.arange(32)
    yi, yj = np.triu_indices(32, 1)
    cs, cd = circulant(3 * WIDE_K + 2, np.arange(1, WIDE_K + 1), y[-1] + 1)
    src = np.concatenate([u, np.repeat(u, 32), [v], y[yi], cs])
    dst = np.concatenate([np.full(32, v), np.tile(y, 32), [y[0]], y[yj], cd])
    n = int(y[-1]) + 1 + 3 * WIDE_K + 2
    g = G(n, np.concatenate([src, fs]), np.concatenate([dst, fd]))
    # the filler has no triangle and touches nothing else: dense products over the rest only
    filler = (g.a >= f0) & (g.a < f0 + WIDE_FILL)
    g.closed_support = np.zeros(len(g.a), np.int64)
    g.closed_support[~filler] = per_component(n, g.a[~filler], g.b[~filler], lambda A: A @ A)
    fr = np.zeros(n, bool)
    fr[g.rank[f0:f0 + WIDE_FILL]] = True
    du = np.repeat(np.arange(n), np.diff(g.doff))
    keep = ~fr[du]
    g._tri = np.zeros(len(du), np.int64)
    g._tri[keep] = per_component(n, du[keep], g.dnbr[keep], lambda D: D @ D.T, upper=True)
    g.wide_hub, g.filler = v, (f0, f0 + WIDE_FILL)
    return g


def far_specials(n):
    """Triangles (a, v, c) and 4-cycles (a, v, x, w) of g_far(n): v is the closing vertex; N+(v) = {c} or {x}."""
    tri, quad = [], []
    # spans on both sides of 64, 4096 (small hub_bits), 439968 (small / wide window) and 524288 (default hub_bits)
    for i, span in enumerate((64, 65, 4096, 4097, 439968, 439969, 524288, 524289)):
        v = 1000 + 10 * i
        tri.append((v - 3, v, v + span))
    # NEAR reach n - 1 - base = 439967 (n = 0 mod 32: NEAR) or 439968 (n = 1 mod 32: not NEAR), where base =
    # (v + 1) & ~31: v + 1 == base and v + 1 == base + 5
    base = n - 1 - (439967 if n % 32 == 0 else 439968)
    assert base % 32 == 0
    for v in (base - 1, base + 4):
        tri.append((v - 2, v, v + 7))
    # an element at id n - 1 in a NEAR item: the suffix of a triangle and of a 4-cycle
    tri.append((n - 200, n - 150, n - 1))
    quad.append((n - 300, n - 250, n - 240, n - 4))
    # suffix elements beyond the small and the wide windows (the probe clamps to the guard word)
    quad.append((2000, 2001, 2003, n - 3))
    quad.append((2010, 2011, 2011 + 500000, n - 2))
    quad.append((2020, 2021, 2021 + 439000, n - 6))
    return tri, quad


@lru_cache(maxsize=None)
def g_far(n):
    """Every vertex of degree 2 (rank == id): the special triangles and 4-cycles, the other ids cut into triangles of
    consecutive free ids."""
    tri, quad = far_specials(n)
    special = np.array([x for t in tri + quad for x in t])
    assert len(set(special.tolist())) == len(special) and special.min() >= 0 and special.max() < n
    free = np.setdiff1d(np.arange(n), special)
    assert len(free) % 3 == 0, n
    t = np.array(tri + [tuple(r) for r in free.reshape(-1, 3)], np.int64)
    qd = np.array(quad, np.int64)
    src = np.concatenate([t[:, 0], t[:, 0], t[:, 1], qd[:, 0], qd[:, 1], qd[:, 2], qd[:, 3]])
    dst = np.concatenate([t[:, 1], t[:, 2], t[:, 2], qd[:, 1], qd[:, 2], qd[:, 3], qd[:, 0]])
    g = G(n, src, dst)
    in_tri = np.zeros(n, bool)
    in_tri[t.ravel()] = True
    g.closed_support = in_tri[g.a].astype(np.int64)     # a triangle edge has both ends in the triangle, 4-cycles none
    return g


FAR_N = (600064, 600001)        # 0 and 1 mod 32, both 0 mod 3 after the special ids


# ---- the schedule, restated ------------------------------------------------------------------------------------------
def snake_owner(d, P):
    r = d % (2 * P)
    return np.where(r < P, r, 2 * P - 1 - r)


def plan_model(g, variant="auto", hub_bitmap_bits=512 * 1024, hub_min_work=1024, gallop_ratio=8, part_index=0,
               part_count=1, smem_optin=SMEM_OPTIN):
    """gmsb_tc_stats of tc_total_ex with these options, the items of every hub and the triangles of every class."""
    n, doff, dnbr = g.n, g.doff, g.dnbr
    dplus = np.diff(doff)
    m = len(dnbr)
    u = np.repeat(np.arange(n), dplus)
    ln = doff[u + 1] - np.arange(m) - 1
    v = dnbr
    own = snake_owner(n - 1 - v, part_count) == part_index if part_count > 1 else np.ones(m, bool)
    du, dv = dplus[u], dplus[v]
    kept = own & (ln > 0) & (dv > 0)
    lcls = np.where(ln <= SHORT, 0, np.where(ln <= MID, 1, 2))
    c = np.stack([np.bincount(v[kept & (lcls == k)], minlength=n) for k in range(3)])
    cnt = c.sum(0)
    work = np.bincount(v[kept], weights=ln[kept], minlength=n).astype(np.int64)
    hub_bits = hub_bitmap_bits
    if hub_bits // 8 > smem_optin - 1024:
        hub_bits = (smem_optin - 1024) * 8
    last = np.where(dplus > 0, dnbr[np.maximum(doff[1:] - 1, 0)], 0)
    ids = np.arange(n)
    span = last - ids
    hub = (cnt > 0) & (variant in ("auto", "bitmap")) & (span <= hub_bits)
    if variant == "auto":
        hub &= work >= hub_min_work
    # items (k_classify)
    target = np.maximum(ITEM_COST, 16 * dplus)
    k = np.clip(-(-(work + 4 * cnt) // target), 1, np.maximum(cnt, 1))
    chunk = -(-cnt // k)
    k = np.where(hub, -(-cnt // np.maximum(chunk, 1)), 0)
    # window classes (k_item_keys)
    words = (span + 31) >> 5
    reach = ((n - 1 - ((ids + 1) & ~31)) >> 5) + 1
    wcls = np.where(reach <= NEAR_WORDS, 0, np.where((words + 1) * 4 > 55000, 2, 1))
    cwords = np.where(wcls == 0, reach, words)
    # light edges (scatter_edge)
    hub_e = kept & hub[v]
    light = kept & ~hub[v]
    lo, hi = np.minimum(ln, dv), np.maximum(ln, dv)
    if variant == "gallop":
        gal = light
    elif variant == "merge":
        gal = np.zeros(m, bool)
    else:
        gal = light & (hi >= gallop_ratio * lo)
    mer = light & ~gal
    t = g.slot_triangles()
    st = dict(
        edges_bitmap=int(cnt[hub].sum()), edges_merge=int(mer.sum()), edges_gallop=int(gal.sum()),
        bitmap_items=int(k.sum()), wedges_bitmap=int(work[hub].sum()),
        wedges_checked=int(ln[kept].sum()), algorithmic_bytes=4 * int((du + dv)[own].sum()),
        bytes_bitmap=4 * int(du[hub_e].sum() + (cnt * dplus)[hub].sum()),
        bitmap_smem_bytes=4 * (int(words[hub].max()) + 1 if hub.any() else 1))
    st["bytes_light"] = 4 * int(du[kept].sum() + (cnt * dplus)[cnt > 0].sum()) - st["bytes_bitmap"]
    tri = {name: int(t[hub_e & (wcls[v] == w)].sum()) for w, name in enumerate(CLASSES[:3])}
    tri["merge"], tri["gallop"] = int(t[mer].sum()), int(t[gal].sum())
    items = {name: int(k[hub & (wcls == w)].sum()) for w, name in enumerate(CLASSES[:3])}
    cw = {name: int(cwords[hub & (wcls == w)].max()) if (hub & (wcls == w)).any() else 0
          for w, name in enumerate(CLASSES[:3])}
    return dict(stats=st, tri=tri, items=items, words=cw, triangles=int(t[own].sum()), hub=hub, cnt=cnt, c=c,
                work=work, span=span, k=k, wcls=wcls, ln=ln, kept=kept, hub_e=hub_e, mer=mer, gal=gal, lo=lo, hi=hi,
                u=u, v=v, max_span_words=int(words[hub].max()) if hub.any() else 0)


def hub_items(model, x):
    """(begin, count, n0, n1) of every item of hub x, relative to its descriptor segment (k_plan_layout)."""
    c0, c1, _ = model["c"][:, x]
    cnt, k = int(model["cnt"][x]), int(model["k"][x])
    chunk = -(-cnt // k)
    out = []
    for j in range(k):
        s = j * chunk
        cc = min(cnt - s, chunk)
        out.append((s, cc, min(max(c0 - s, 0), cc), min(max(c0 + c1 - s, 0), cc)))
    return out


def merge_split_at_tile_edge(a, b, tile=512):
    """A common element of the merge of a and b (a wins ties) whose copy from a ends a tile and whose copy from b
    starts the next."""
    com = np.intersect1d(a, b)
    pos = np.searchsorted(a, com) + np.searchsorted(b, com)        # position of a's copy in the merged sequence
    return bool(((pos % tile) == tile - 1).any())


def edge_scores(g):
    """jaccard, overlap, total_neigh, pref_att as k_edge_scores computes them (float64)."""
    cd = g.support().astype(np.float64)
    da, db = g.deg[g.a], g.deg[g.b]
    return {"jaccard": np.where((da == 0) & (db == 0), 1.0, cd / ((da + db).astype(np.float64) + cd)),
            "overlap": cd / np.minimum(da, db).astype(np.float64),
            "total_neigh": (da + db - g.support()).astype(np.float64),
            "pref_att": (da * db).astype(np.float64)}


# ---- CPU: the constructions land on their boundaries -----------------------------------------------------------------
def small_option_sets(g):
    """Option sets run on g_small: every variant, hub_min_work at and one above a hub's work, ratios 2 / 8 / 64 with
    every vertex light."""
    base = plan_model(g)
    x = g.rank[small_circ_vertex(g, 100)]
    W = int(base["work"][x])
    sets = [dict(variant=v) for v in ("auto", "bitmap", "merge", "gallop")]
    sets += [dict(hub_min_work=W), dict(hub_min_work=W + 1)]
    sets += [dict(hub_min_work=1 << 40, gallop_ratio=r) for r in (2, 8, 64)]
    return sets


def small_circ_vertex(g, k):
    """Id of the vertex 2k of the C_{3k+2}(1..k) block of g_small: neither it nor an in-neighbour has a wrapping edge,
    so its in-edges have the suffix lengths 0 .. k - 1."""
    base = SMALL_CIRC_BASE
    for kk in CIRC_KS:
        if kk == k:
            return base + 2 * k
        base += 3 * kk + 2
    raise KeyError(k)


def far_option_sets():
    return [dict(variant="bitmap"), dict(variant="bitmap", hub_bitmap_bits=64),
            dict(variant="bitmap", hub_bitmap_bits=4096), dict(variant="auto"), dict(variant="merge"),
            dict(variant="gallop"), dict(variant="auto", hub_min_work=1)]


def test_small_graph_boundaries(orc):
    g = g_small()
    a, b = g.edges32()
    assert plan_model(g)["triangles"] == orc.from_el(a, b, True).tc_total()
    o = orc.from_el(a, b, True)
    assert (o.degree_order(True) == g.rank).all()
    for opts in small_option_sets(g):
        M = plan_model(g, **opts)
        assert sum(M["tri"].values()) == M["triangles"], opts
        assert M["stats"]["edges_bitmap"] + M["stats"]["edges_merge"] + M["stats"]["edges_gallop"] == M["kept"].sum()
    M = plan_model(g)
    hub = M["hub"]
    # suffix lengths on both sides of every length class and 128-element block edge, all in hub items
    lens = set(M["ln"][M["hub_e"]].tolist())
    assert {1, 8, 9, 96, 97, 127, 128, 129, 256, 257} <= lens
    # one item per vertex 2k of the C_{3k+2}(1..k) blocks, k <= 102, with k - 97 class-2 descriptors (1..5 mod 4)
    for k in CIRC_KS[:5]:
        x = g.rank[small_circ_vertex(g, k)]
        assert hub[x] and M["k"][x] == 1 and M["c"][2, x] == k - 97, k
    # hubs of two items, with the class boundaries before, inside and at the end of a slice
    x = g.rank[small_circ_vertex(g, 725)]
    assert M["k"][x] == 2
    its = hub_items(M, x)
    assert sum(c for _, c, _, _ in its) == M["cnt"][x]
    assert 0 < its[0][2] < its[0][3] < its[0][1] and its[1][2] == its[1][3] == 0
    # and a hub whose first slice ends before its class boundaries (all class 0), the second holding them
    x = g.rank[g.n - SLICED_T - 1]
    its = hub_items(M, x)
    assert M["hub"][x] and its == [(0, 680, 680, 680), (680, 680, 20, 20)], its
    # every hub's items cover its descriptors exactly once, class boundaries inside [0, count]
    for x in np.nonzero(hub)[0]:
        its = hub_items(M, x)
        assert [s for s, _, _, _ in its] == list(np.cumsum([0] + [c for _, c, _, _ in its])[:-1])
        assert sum(c for _, c, _, _ in its) == M["cnt"][x] and all(0 <= a0 <= a1 <= c for _, c, a0, a1 in its)
    assert M["stats"]["bitmap_items"] == sum(len(hub_items(M, x)) for x in np.nonzero(hub)[0])
    # an in-edge of a hub whose suffix runs past every hub window (k_support_bitmap probes it through the clamp)
    last = g.dnbr[g.doff[M["u"] + 1] - 1]
    assert ((((last - M["v"] - 1) >> 5) > M["max_span_words"]) & M["hub_e"] & (M["hub"][M["v"]])).any()
    # both light kernels run under the default options, and hub_min_work = work(x) / work(x) + 1 moves x's block
    assert M["stats"]["edges_merge"] > 0 and M["stats"]["edges_gallop"] > 0 and M["tri"]["merge"] > 0
    assert M["tri"]["gallop"] > 0 and M["tri"]["near"] > 0
    sets = small_option_sets(g)
    x = g.rank[small_circ_vertex(g, 100)]
    assert plan_model(g, **sets[4])["hub"][x] and not plan_model(g, **sets[5])["hub"][x]
    # gallop ratio: light pairs at hi == ratio * lo and ratio * lo - 1
    for r in (2, 8, 64):
        Mr = plan_model(g, hub_min_work=1 << 40, gallop_ratio=r)
        assert not Mr["hub"].any()
        L = Mr["kept"]
        assert (L & (Mr["hi"] == r * Mr["lo"])).any() and (L & (Mr["hi"] == r * Mr["lo"] - 1)).any(), r
    # merge tiles: combined lengths 511, 512, 513, 1024, 1025, and a common element split by a tile edge
    tot = M["ln"] + np.diff(g.doff)[M["v"]]
    Mm = plan_model(g, variant="merge")
    assert {511, 512, 513, 1024, 1025} <= set(tot[Mm["mer"]].tolist())
    split = 0
    for s in np.nonzero(Mm["mer"] & (tot > 512))[0][::7]:
        uu, vv = M["u"][s], M["v"][s]
        if merge_split_at_tile_edge(g.dnbr[s + 1:g.doff[uu + 1]], g.dnbr[g.doff[vv]:g.doff[vv + 1]]):
            split += 1
            break
    assert split
    # the circulant blocks: support in closed form
    sup = g.support()
    base = SMALL_CIRC_BASE
    for k in CIRC_KS:
        n = 3 * k + 2
        cs = circulant_support(n, np.arange(1, k + 1))
        sel = (g.a >= base) & (g.b < base + n)
        off = np.minimum(g.b[sel] - g.a[sel], n - (g.b[sel] - g.a[sel]))
        assert (sup[sel] == np.array([cs[o] for o in off])).all(), k
        base += n


@pytest.mark.parametrize("n", FAR_N)
def test_far_graph_boundaries(orc, n):
    g = g_far(n)
    assert (g.rank == np.arange(n)).all() and (g.deg == 2).all()
    a, b = g.edges32()
    assert g.support().sum() // 3 == orc.from_el(a, b, True).tc_total() == plan_model(g)["triangles"]
    tri, quad = far_specials(n)
    for opts in far_option_sets():
        M = plan_model(g, **opts)
        assert sum(M["tri"].values()) == M["triangles"], opts
    M = plan_model(g, variant="bitmap")
    # windows: small at span 439968, wide at 439969 and at 524288 == hub_bits, light at 524289
    vs = {span: t[1] for span, t in zip((64, 65, 4096, 4097, 439968, 439969, 524288, 524289), tri)}
    assert M["span"][vs[439968]] == 439968 and M["wcls"][vs[439968]] == 1 and M["hub"][vs[439968]]
    assert M["wcls"][vs[439969]] == 2 and M["hub"][vs[439969]] and M["hub"][vs[524288]]
    assert not M["hub"][vs[524289]] and M["mer"][M["v"] == vs[524289]].any()
    for bits in (64, 4096):
        Mb = plan_model(g, variant="bitmap", hub_bitmap_bits=bits)
        assert Mb["hub"][vs[bits]] and not Mb["hub"][vs[bits + 1]]
    # NEAR reach 439967 (NEAR) or 439968 (not), with v + 1 on and off a multiple of 32
    near = n % 32 == 0
    for v in (tri[8][1], tri[9][1]):
        reach = n - 1 - ((v + 1) & ~31)
        assert reach == (439967 if near else 439968) and (M["wcls"][v] == 0) == near
    assert (tri[8][1] + 1) % 32 == 0 and (tri[9][1] + 1) % 32 != 0
    # an element at n - 1 in a NEAR item
    assert M["wcls"][n - 150] == 0 and M["hub"][n - 150]
    # suffix elements beyond the windows of small and wide items
    for (_, v, x, w) in quad[1:]:
        assert M["hub"][v] and (w - v - 1) >> 5 > M["words"][CLASSES[M["wcls"][v]]]
    assert M["wcls"][quad[1][1]] == 1 and M["wcls"][quad[2][1]] == 2
    # every window class counts triangles
    assert all(M["tri"][c] > 0 for c in ("near", "small", "wide", "merge"))


def test_wide_support_graph_boundaries(orc):
    g = g_wide()
    M = plan_model(g)
    v = g.rank[g.wide_hub]
    # under the default options: v is a hub at work == hub_min_work with span == hub_bits, in the wide class
    assert M["work"][v] == 1024 and M["span"][v] == 512 * 1024 and M["hub"][v] and M["wcls"][v] == 2
    assert M["tri"]["wide"] == 32
    # the support kernel's window is that wide (more than the 48 KB without the opt-in), and hubs with small windows,
    # work >= 1024 and all three length classes close triangles beside it
    assert M["max_span_words"] == 16384 and M["stats"]["bitmap_smem_bytes"] == 4 * 16385
    small = M["hub"] & (M["span"] <= 4096) & (M["work"] >= 1024)
    assert small.sum() > 100 and (M["c"][:, small].sum(1) > 0).all() and M["tri"]["near"] > 0
    # the filler ranks between v and its out-neighbour, has no triangle and no hub
    f0, f1 = g.filler
    assert (g.rank[f0:f1] > v).all() and (g.rank[f0:f1] < v + M["span"][v]).all()
    assert not M["hub"][g.rank[f0:f1]].any() and M["stats"]["edges_merge"] > 0
    # the references against the oracle and a sparse product on the whole graph
    a, b = g.edges32()
    assert g.support().sum() == 3 * M["triangles"] == 3 * orc.from_el(a, b, True).tc_total()
    from scipy import sparse
    D = sparse.csr_matrix((np.ones(len(M["u"]), np.int64), (M["u"], g.dnbr)), shape=(g.n, g.n))
    assert np.array_equal(np.asarray((D @ D.T)[M["u"], g.dnbr]).ravel(), g.slot_triangles())


# ---- GPU ------------------------------------------------------------------------------------------------------------
gpu = pytest.mark.gpu
TRACE = re.compile(r"\[gmsb tc\] class=(\w+) (items|edges)=(\d+)(?: words=(\d+))? triangles=(\d+)")
STAT_KEYS = ("edges_bitmap", "edges_merge", "edges_gallop", "bitmap_items", "wedges_bitmap", "wedges_checked",
             "algorithmic_bytes", "bytes_bitmap", "bytes_light", "bitmap_smem_bytes")


def smem_optin():
    import torch
    return torch.cuda.get_device_properties(0).shared_memory_per_block_optin


def run_and_check(gg, g, opts, capfd, monkeypatch, seen, part_index=0, part_count=1, edge_passes="auto"):
    """One count without and one with GMSB_TC_TRACE: the count, every statistic and every class line equal the
    model's.  Returns the count."""
    M = plan_model(g, part_index=part_index, part_count=part_count, smem_optin=smem_optin(), **opts)
    kw = dict(part_index=part_index, part_count=part_count, edge_passes=edge_passes, **opts)
    got, st = gg.tc_total_ex(**kw)
    where = (opts, part_index, part_count, edge_passes)
    assert got == M["triangles"], where
    assert {k: st[k] for k in STAT_KEYS} == {k: M["stats"][k] for k in STAT_KEYS}, where
    capfd.readouterr()
    monkeypatch.setenv("GMSB_TC_TRACE", "1")
    traced, _ = gg.tc_total_ex(**kw)
    monkeypatch.delenv("GMSB_TC_TRACE")
    lines = [m.groups() for m in TRACE.finditer(capfd.readouterr().err)]
    assert traced == got
    want = []
    for c in CLASSES[:3]:
        if M["items"][c]:
            want.append((c, "items", str(M["items"][c]), str(M["words"][c]), str(M["tri"][c])))
    for c, key in (("merge", "edges_merge"), ("gallop", "edges_gallop")):
        if M["stats"][key]:
            want.append((c, "edges", str(M["stats"][key]), None, str(M["tri"][c])))
    assert lines == want, where
    for c in CLASSES:
        if M["tri"][c]:
            seen.add(c)
    return got


@pytest.fixture(scope="module")
def small_gpu(gms):
    g = g_small()
    gg = gms.Graph.from_edgelist(*g.edges32(), True)
    assert (gg.degree_order(True) == g.rank).all()
    return g, gg


@gpu
def test_small_graph_every_option_set(small_gpu, capfd, monkeypatch):
    g, gg = small_gpu
    seen = set()
    for opts in small_option_sets(g):
        run_and_check(gg, g, opts, capfd, monkeypatch, seen)
    assert seen == set(CLASSES) - {"small", "wide"}


@gpu
@pytest.mark.parametrize("n", FAR_N)
def test_far_graph_window_classes(gms, capfd, monkeypatch, n):
    g = g_far(n)
    gg = gms.Graph.from_edgelist(*g.edges32(), True)
    seen = set()
    for opts in far_option_sets():
        run_and_check(gg, g, opts, capfd, monkeypatch, seen)
    assert seen == set(CLASSES)


@gpu
def test_shares_add_up(gms, small_gpu, capfd, monkeypatch):
    """part_count 2, 3, 8, both forms of the edge passes: every share equals its model, the shares add up."""
    cases = [(small_gpu, dict(variant="auto")), (small_gpu, dict(variant="bitmap"))]
    g = g_far(FAR_N[0])
    cases.append(((g, gms.Graph.from_edgelist(*g.edges32(), True)), dict(variant="bitmap")))
    for (g, gg), opts in cases:
        total = plan_model(g, **opts)["triangles"]
        for P in (2, 3, 8):
            for passes in ("rows", "slots"):
                seen = set()
                got = sum(run_and_check(gg, g, opts, capfd, monkeypatch, seen, p, P, passes) for p in range(P))
                assert got == total, (opts, P, passes)


@gpu
def test_wide_support_graph_counts(gms, capfd, monkeypatch):
    """tc_total on g_wide with the default options: its hub at work == hub_min_work, span == hub_bits goes to the
    wide window class."""
    g = g_wide()
    gg = gms.Graph.from_edgelist(*g.edges32(), True)
    seen = set()
    run_and_check(gg, g, {}, capfd, monkeypatch, seen)
    assert {"near", "wide"} <= seen


@gpu
@pytest.mark.parametrize("which", ["small", "far", "wide"])
def test_support_vertex2_and_scores(gms, which):
    """edge_similarity("comm_neigh") is the support of every edge; the other support metrics are bit-exact against
    numpy's float64; tc_vertex2 (and its several-GPU form) are the row sums of the support.  The support kernels run
    on the default schedule: on g_small its hubs of all length classes, multi-item hubs and both light lists; on g_far
    the light lists only; on g_wide a 524288-bit window shared by the small-window hubs."""
    g = {"small": g_small, "far": lambda: g_far(FAR_N[0]), "wide": g_wide}[which]()
    gg = gms.Graph.from_edgelist(*g.edges32(), True)
    M = plan_model(g)
    if which == "small":
        assert (M["c"][:, M["hub"]].sum(1) > 0).all() and (M["k"] > 1).any()
        assert M["stats"]["edges_merge"] and M["stats"]["edges_gallop"]
    elif which == "far":
        assert not M["hub"].any() and M["tri"]["merge"] > 0
    else:
        assert M["max_span_words"] == 16384 and M["hub"].sum() > 100
    sup = g.support()
    assert np.array_equal(gg.edge_similarity("comm_neigh"), sup.astype(np.float64))
    for metric, want in edge_scores(g).items():
        assert gg.edge_similarity(metric).tobytes() == want.tobytes(), metric
    v2 = np.bincount(np.concatenate([g.a, g.b]), weights=np.concatenate([sup, sup]), minlength=g.n).astype(np.int64)
    assert np.array_equal(gg.tc_vertex2(), v2)
    gms.set_devices([0])          # the several-GPU entry points on device 0 alone (test_gpu_operators leaves it so too)
    assert np.array_equal(gg.tc_vertex2_multi(), v2)
