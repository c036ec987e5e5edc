"""Balance of the multi-device partition, measured on ONE device: every part's share of the schedule is built and counted
in turn (the parts of a real run do exactly this, each on its own GPU), so max over the parts is the step time a run on
P devices would see, without paying for P GPUs.

    python tools/partition_balance.py [--scale 24] [--parts 2,4,8] [--reps 3]
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gms_b200 as G  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", type=int, default=24)
    ap.add_argument("--rmat-a", type=float, default=0.57)
    ap.add_argument("--parts", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--row-walk", action="store_true", help="force the row-walking schedule passes (A/B against the "
                                                            "element-wise ones)")
    args = ap.parse_args()
    G.set_device(0)
    a = args.rmat_a
    src, dst = G.generate_rmat(args.scale, a=a, b=(0.95 - a) / 2, c=(0.95 - a) / 2)
    g = G.Graph.from_edgelist(src, dst, True)
    del src, dst
    total, _ = g.tc_total_ex(reuse_plan=1)
    for P in [int(x) for x in args.parts.split(",")]:
        sched, count, bitmap, tri, edges = [], [], [], 0, 0
        for p in range(P):
            best = None
            for _ in range(args.reps):
                c, st = g.tc_total_ex(part_index=p, part_count=P, reuse_plan=2,
                                      edge_passes="rows" if args.row_walk else "auto")
                if best is None or st["ms_orient"] + st["ms_count"] < best["ms_orient"] + best["ms_count"]:
                    best = st
            tri += c
            edges += best["edges_bitmap"] + best["edges_merge"] + best["edges_gallop"]
            sched.append(round(best["ms_orient"], 3)); count.append(round(best["ms_count"], 3))
            bitmap.append(round(best["ms_bitmap"], 3))
        assert tri == total, (P, tri, total)
        step = [s + c for s, c in zip(sched, count)]
        print(json.dumps({"scale": args.scale, "rmat_a": a, "row_walk": args.row_walk, "parts": P, "triangles": tri, "edges_scheduled": edges,
                          "schedule_ms": sched, "count_ms": count, "bitmap_ms": bitmap,
                          "max_step_ms": round(max(step), 3), "mean_step_ms": round(sum(step) / P, 3),
                          "max_count_ms": max(count), "mean_count_ms": round(sum(count) / P, 3)}), flush=True)


if __name__ == "__main__":
    main()
