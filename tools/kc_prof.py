"""Profiling helper: one k-clique count on a Kronecker graph (python tools/kc_prof.py <scale> <k> [reps])."""
import sys
import time
import os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gms_b200 as G
scale, k = int(sys.argv[1]), int(sys.argv[2])
reps = int(sys.argv[3]) if len(sys.argv) > 3 else 1
s, d = G.generate_rmat(scale)
g = G.Graph.from_edgelist(s, d, True)
g.kclique_count(3)
for _ in range(reps):
    t = time.time()
    c = g.kclique_count(k)
    print(f"k={k} scale={scale} count={c} seconds={time.time() - t:.3f}", flush=True)
