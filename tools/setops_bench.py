"""Throughput of the batched Set operations and of the per-edge similarity scores (BASELINE.json configs[3]).

    python tools/setops_bench.py [--scale 22] [--cpu-seconds 10]

One JSON line per measurement:
  * edge_similarity (Jaccard, CommNeigh: from one pass of the oriented triangle schedule; Adamic-Adar: one symmetric-list
    intersection per edge, the batched intersect kernels) over ALL undirected edges, with the bytes that bound each:
    B_TC for the support path, B_sim = sum over edges u<v of 4 (d(u) + d(v)) + 8 m for the pair path (SURVEY.md 8d);
  * gmsb_intersect_count_batch / gmsb_pair_similarity on hub x hub pairs (both lists long and balanced: the merge
    path) and on hub x leaf pairs (skewed: galloping), host arrays in, host arrays out;
  * the reference's CPU loop over vertex_similarity<Jaccard|CommNeigh> on a bounded sample of the same edges."""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gms_b200 as G  # noqa: E402


def emit(**kw):
    print(json.dumps(kw), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=int, default=22)
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    args = ap.parse_args()
    peak = 6550.4
    try:
        peak = float(json.load(open(os.path.join(os.path.dirname(__file__), "..", "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:
        pass
    G.set_device(0)
    src, dst = G.generate_rmat(args.scale)
    g = G.Graph.from_edgelist(src, dst, True)
    off, nbr = g.export_csr()
    deg = np.diff(off)
    n, m = g.n, g.slots // 2
    u = np.repeat(np.arange(n, dtype=np.int32), deg)
    up = u < nbr
    b_sim = int(4 * (deg[u[up]].astype(np.int64) + deg[nbr[up]].astype(np.int64)).sum() + 8 * m)
    _, st = g.tc_total_ex(reuse_plan=True)
    b_tc = st["algorithmic_bytes"]
    for metric in ("jaccard", "comm_neigh", "adamic_adar"):
        g.edge_similarity(metric)
        G.synchronize()
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            out = g.edge_similarity(metric)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        bound = b_sim if metric == "adamic_adar" else b_tc + 8 * m
        emit(what="edge_similarity", metric=metric, scale=args.scale, edges=m, seconds=best, edges_per_s=m / best,
             path="pair kernels (symmetric lists)" if metric == "adamic_adar" else "edge support from the triangle schedule",
             bound_bytes=bound, GBps=bound / best / 1e9, frac_of_hbm_peak=bound / best / 1e9 / peak,
             d2h_bytes=8 * m, checksum=float(np.nansum(out[np.isfinite(out)])))
    # hub x hub and hub x leaf pairs through the host-array batch API
    order = np.argsort(-deg, kind="stable")
    hubs = order[:2000].astype(np.int32)
    leaves = order[n // 2: n // 2 + 2000].astype(np.int32)
    rng = np.random.default_rng(1)
    npairs = 1 << 20
    for name, a, b in (("hub x hub", rng.choice(hubs, npairs), rng.choice(hubs, npairs)),
                       ("hub x leaf", rng.choice(hubs, npairs), rng.choice(leaves, npairs))):
        a, b = a.astype(np.int32), b.astype(np.int32)
        g.intersect_count_batch(a[:1024], b[:1024])
        t0 = time.perf_counter()
        c = g.intersect_count_batch(a, b)
        dt = time.perf_counter() - t0
        bytes_ = int(4 * (deg[a].astype(np.int64) + deg[b].astype(np.int64)).sum())
        emit(what="intersect_count_batch", pairs=name, npairs=npairs, seconds=dt, pairs_per_s=npairs / dt,
             list_bytes=bytes_, GBps=bytes_ / dt / 1e9, frac_of_hbm_peak=bytes_ / dt / 1e9 / peak, checksum=int(c.sum()))
        t0 = time.perf_counter()
        j = g.pair_similarity("jaccard", a, b)
        dt = time.perf_counter() - t0
        emit(what="pair_similarity(jaccard)", pairs=name, npairs=npairs, seconds=dt, pairs_per_s=npairs / dt,
             GBps=bytes_ / dt / 1e9, checksum=float(j.sum()))
    # CPU: the reference's vertex_similarity over a bounded sample of the edges (all host threads)
    if args.cpu_seconds > 0:
        from oracle import binding
        lib = binding.reference() or binding.oracle()
        kind = "reference" if binding.reference() is not None else "port"
        lib.set_threads(len(os.sched_getaffinity(0)))
        cg = lib.from_csr(off, nbr, False)
        ea, eb = u[up], nbr[up]
        elems = float((deg[ea].astype(np.float64) + deg[eb]).sum())
        stride = max(1, int(elems / (0.25e9 * lib.max_threads()) / args.cpu_seconds))
        sa, sb = np.ascontiguousarray(ea[::stride]), np.ascontiguousarray(eb[::stride])
        for metric in ("jaccard", "comm_neigh"):
            t0 = time.perf_counter()
            out = cg.pair_similarity(metric, sa, sb)
            dt = time.perf_counter() - t0
            gpu = g.pair_similarity(metric, sa, sb)
            emit(what="cpu_baseline", kind=kind, cores=lib.max_threads(), metric=metric,
                 sample=f"every {stride}-th undirected edge of the same graph", pairs=len(sa), seconds=dt,
                 edges_per_s=len(sa) / dt, bit_identical_to_gpu=bool(out.tobytes() == gpu.tobytes()))


if __name__ == "__main__":
    main()
