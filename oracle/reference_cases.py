"""TEST INFRASTRUCTURE ONLY — the seeded cases on which the CPU suite compares the oracle with the unmodified reference,
and the stored record of what the reference answers on them (tests/golden/reference_cases.json).

The reference library (oracle/_ref/libgmsref.so) is built from the reference's source tree, which is not part of this
repository, so most machines that run the suite do not have it.  The tests therefore check the oracle against the stored
record always, and against the live reference as well where the library exists.

The record holds what those tests assert the reference to produce: for the random graphs every array and count they
compare (arrays as sha256 digests), for the set operations a digest of all 200 results, for the approximate degeneracy
orders the round in which each vertex leaves (the reference leaves the order inside a round unspecified, so the tests
compare rounds), for the file round trip the CSR the reader builds.  Regenerate with

    python -m oracle.reference_cases

`source` in the record says which library produced it.  With the reference library present the values are computed by
the reference itself (every comparison of the tests is re-run first); without it they are computed by the oracle, which
the tests held equal to the reference on exactly these inputs, and `source` says so.
"""
import hashlib
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
PATH = os.path.join(ROOT, "tests", "golden", "reference_cases.json")

RANDOM_CASES = [(50, 200), (200, 3000), (1000, 8000), (64, 2000), (500, 500), (3000, 40000)]   # seed -> (n, m)
ADG_CASES = [(60, 300), (500, 6000), (3000, 40000), (200, 8000)]                               # seed 30 + i
ADG_EX_CASES = [(80, 500), (600, 9000), (2500, 30000)]                                         # seed 70 + i
ADG_EPS = (0.0, 0.5, 1.0)
ADG_EX_EPS = (0.0, 0.5)
BOUNDARIES = ("average", "min")


def sha(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def random_graph_edges(seed, n, m, skew=0.0):
    """Seeded edge list; skew>0 concentrates endpoints on low ids (hubs).  The suite's tests draw their graphs here."""
    rng = np.random.default_rng(seed)
    if skew > 0:
        src = np.minimum((rng.random(m) ** (1 + skew) * n).astype(np.int32), n - 1)
        dst = np.minimum((rng.random(m) ** (1 + skew) * n).astype(np.int32), n - 1)
    else:
        src = rng.integers(0, n, m, dtype=np.int32)
        dst = rng.integers(0, n, m, dtype=np.int32)
    return src, dst


def random_case(seed):
    n, m = RANDOM_CASES[seed]
    s, d = random_graph_edges(seed, n, m, skew=(seed % 3) * 0.7)
    return s, d, m


def random_record(lib, orc, seed):
    """Everything test_oracle_matches_reference_random compares, as `lib` computes it.  The degeneracy ranking itself is
    not unique, so what is recorded of it is what the test checks: its degeneracy by the oracle's checker and the
    4-clique count of the DAG it orients."""
    from oracle.binding import METRICS
    s, d, m = random_case(seed)
    g = lib.from_el(s, d, True)
    off, nbr = g.csr()
    rank = g.degree_order(True)
    dag = g.induce_directed(rank)
    doff, dnbr = dag.csr()
    ro, rn = g.relabel_by_degree().csr()
    go = orc.from_el(s, d, True)
    rr = lib.degeneracy_rank(g)
    rec = {"n": g.n, "csr_sha": sha(off) + sha(nbr), "tc": g.tc_total(),
           "vertex2_sha": sha(g.tc_vertex2(1) if lib.prefix != "orc_" else g.tc_vertex2()),
           "order_sha": sha(g.degree_order(False)), "rank_sha": sha(rank),
           "dag_n": dag.n, "dag_sha": sha(doff) + sha(dnbr),
           "kclique": {str(k): dag.kclique(k, 2) for k in (1, 2, 3, 4, 5)},
           "sim_sha": {mname: sha(g.edge_similarity(mname)) for mname in METRICS},
           "degeneracy": orc.check_degeneracy_rank(go, rr), "degeneracy_kclique4": go.induce_directed(rr).kclique(4),
           "relabel_sha": sha(ro) + sha(rn)}
    if m <= 3000:
        rec["set_based_4"] = g.clique_count_set_based(4)
    return rec


def set_cases():
    rng = np.random.default_rng(7)
    for _ in range(200):
        na, nb = rng.integers(0, 60, 2)
        a = np.unique(rng.integers(0, 80, na)).astype(np.int32)
        b = np.unique(rng.integers(0, 80, nb)).astype(np.int32)
        yield a, b, int(rng.integers(0, 80))


def set_record(lib):
    """Digest of the 200 seeded set-operation results test_oracle_sets_match_reference_random compares."""
    res = [[lib.intersect_count(a, b), lib.intersect(a, b).tolist(), lib.union(a, b).tolist(), lib.union_count(a, b),
            lib.difference(a, b).tolist(), lib.contains(a, x)] for a, b, x in set_cases()]
    return {"cases": len(res), "sha": hashlib.sha256(json.dumps(res).encode()).hexdigest()}


def adg_case(seed):
    n, m = ADG_CASES[seed]
    return random_graph_edges(30 + seed, n, m, skew=(seed % 2) * 1.0)


def adg_ex_case(seed):
    n, m = ADG_EX_CASES[seed]
    return random_graph_edges(70 + seed, n, m, skew=(seed % 2) * 1.0)


def rounds_record(round_of):
    """The round in which each vertex leaves, and how many leave per round."""
    round_of = np.ascontiguousarray(round_of, np.int32)
    return {"round_sha": sha(round_of), "per_round": np.bincount(round_of).tolist()}


def rounds_of_order(order, round_of):
    """The reference returns only an order; its rounds are the oracle's rounds, provided the order visits them in
    sequence and each round holds the same vertices (what the tests check).  Returns the per-vertex rounds or raises."""
    rr = round_of[order]
    assert sorted(np.asarray(order).tolist()) == list(range(len(round_of)))
    assert (np.diff(rr) >= 0).all() and (np.bincount(rr) == np.bincount(round_of)).all()
    return round_of


def adg_record(orc, ref, seed):
    s, d = adg_case(seed)
    go = orc.from_el(s, d, True)
    gr = ref.from_el(s, d, True) if ref is not None else None
    out = {}
    for eps in ADG_EPS:
        order_o, round_of = orc.adg_order(go, eps, False)
        if gr is not None:
            rounds_of_order(ref.adg_order(gr, eps, False), round_of)
        out[str(eps)] = rounds_record(round_of)
    return out


def adg_ex_record(orc, ref, seed):
    s, d = adg_ex_case(seed)
    go = orc.from_el(s, d, True)
    gr = ref.from_el(s, d, True) if ref is not None else None
    out = {}
    for boundary in BOUNDARIES:
        for eps in ADG_EX_EPS:
            _, round_of = orc.adg_order_ex(go, eps, False, boundary)
            for pull in (False, True):
                if gr is not None:
                    rounds_of_order(ref.adg_order_ex(gr, eps, False, boundary, pull), round_of)
                out[f"{boundary}/{eps}/{'pull' if pull else 'push'}"] = rounds_record(round_of)
    return out


def round_trip_case(orc):
    s, d = random_graph_edges(4, 500, 4000, skew=1.0)
    return orc.from_el(s, d, True)


def round_trip_record(lib, orc):
    """The CSR the reader of `lib` builds from the .sg and the .el file our writer makes of the round-trip graph."""
    from gms_b200 import io as gio
    o = round_trip_case(orc)
    off, nbr = o.csr()
    with tempfile.TemporaryDirectory() as tmp:
        p, q = os.path.join(tmp, "g.sg"), os.path.join(tmp, "g.el")
        gio.write_sg(p, off, nbr, False)
        gio.write_el(q, off, nbr)
        if lib.prefix == "orc_":
            _, boff, bnbr = gio.read_sg(p)
            sg = orc.from_csr(boff, bnbr, False)
            es, ed = gio.read_el(q)
            el = orc.from_el(es, ed, True)
        else:
            sg, el = lib.load_file(p), lib.load_file(q, True)
        sg_off, sg_nbr = sg.csr()
        el_off, el_nbr = el.csr()
        return {"sg_csr_sha": sha(sg_off) + sha(sg_nbr), "sg_tc": sg.tc_total(), "el_csr_sha": sha(el_off) + sha(el_nbr)}


def build_record(orc, ref):
    lib = ref if ref is not None else orc
    source = ("reference (oracle/_ref/libgmsref.so)" if ref is not None else
              "oracle (oracle/oracle.cpp); the reference library was not available when this record was made, and "
              "these are the values the tests held the reference equal to on exactly these inputs")
    return {"source": source,
            "random": [random_record(lib, orc, seed) for seed in range(len(RANDOM_CASES))],
            "sets": set_record(lib),
            "adg": [adg_record(orc, ref, seed) for seed in range(len(ADG_CASES))],
            "adg_ex": [adg_ex_record(orc, ref, seed) for seed in range(len(ADG_EX_CASES))],
            "round_trip": round_trip_record(lib, orc)}


def load():
    with open(PATH) as f:
        return json.load(f)


def main():
    sys.path.insert(0, ROOT)
    from oracle import binding
    binding.build()
    orc, ref = binding.oracle(), binding.reference()
    rec = build_record(orc, ref)
    if ref is not None:          # the oracle must agree with what is stored, or the suite would fail at once
        mine = build_record(orc, None)
        assert all(mine[key] == rec[key] for key in rec if key != "source")
    with open(PATH, "w") as f:
        json.dump(rec, f, indent=1, sort_keys=True)
        f.write("\n")
    print("wrote", PATH, os.path.getsize(PATH), "bytes; source:", rec["source"].split(" ")[0])


if __name__ == "__main__":
    main()
