"""Core and truss numbers on one GPU, Kronecker graphs (`-g kronecker <scale> --deg 16`).

    python tools/bench_truss.py [--scales 20,22,24] [--oracle-scale 18]

One JSON line per scale: n, m, degeneracy, max truss; the peel's levels (distinct truss values), passes over the edges
(one per level plus one per empty level jumped over) and sub-rounds; launches of one truss_numbers call (difference
of gmsb_launch_count); ms of core_numbers and truss_numbers from a host clock around one call after a warm-up call,
result download included; and a device-time split of one further call, profiled separately (torch.profiler, CUDA
kernels by name) into the edge ids, the initial support and the peel.  The GPU's name and power limit are read in the
same run.  --oracle-scale S adds one line with the sequential time of the CPU checker (tests/truss_oracle.py) for both
peels at scale S (no GPU)."""
import argparse
import json
import os
import re
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SUPPORT_KERNELS = ("k_support_bitmap", "k_support_light", "k_edge_support")
PEEL_KERNELS = ("k_truss_collect", "k_truss_mark", "k_truss_peel", "k_truss_peel_long", "k_truss_retire")


def gpu_identity():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True).stdout.strip()
    name, _, power = out.partition(",")
    return name.strip(), power.strip()


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return r, (time.perf_counter() - t0) * 1e3


def kernel_split(g):
    """Device ms by kernel family and launch counts of one truss_numbers call under torch.profiler."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        g.truss_numbers()
        torch.cuda.synchronize()
    ms, calls = {}, {}
    for ev in prof.key_averages():
        found = re.search(r"\b(k_\w+)", ev.key)      # "void gmsb::(anonymous namespace)::k_truss_peel(...)"
        if not found:
            continue
        base = found.group(1)
        ms[base] = ms.get(base, 0.0) + ev.device_time_total / 1e3
        calls[base] = calls.get(base, 0) + ev.count
    return ms, calls


def bench_scale(G, scale):
    src, dst = G.generate_rmat(scale)
    g = G.Graph.from_edgelist(src, dst, True)
    g.core_numbers()                                     # warm-up: modules, allocator, the cached triangle schedule
    g.truss_numbers()
    core, ms_core = timed(g.core_numbers)
    l0 = G.launch_count()
    truss, ms_truss = timed(g.truss_numbers)
    launches = G.launch_count() - l0
    ms, calls = kernel_split(g)
    name, power = gpu_identity()
    return {"graph": f"kronecker-{scale}", "n": g.n, "m": len(truss), "degeneracy": int(core.max()),
            "max_truss": int(truss.max()), "levels": len(set(truss.tolist())),
            "edge_passes": calls.get("k_truss_collect", 0), "sub_rounds": calls.get("k_truss_peel", 0),
            "long_row_launches": calls.get("k_truss_peel_long", 0), "launches": launches,
            "ms_core_numbers": round(ms_core, 3), "ms_truss_numbers": round(ms_truss, 3),
            "device_ms_edge_ids": round(ms.get("k_slot_edge_ids", 0.0), 3),
            "device_ms_support": round(sum(ms.get(k, 0.0) for k in SUPPORT_KERNELS), 3),
            "device_ms_peel": round(sum(ms.get(k, 0.0) for k in PEEL_KERNELS), 3),
            "device_ms_peel_by_kernel": {k: round(ms.get(k, 0.0), 3) for k in PEEL_KERNELS},
            "gpu": name, "power_limit": power}


def oracle_line(scale):
    import platform
    from oracle import binding
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
    import truss_oracle as tor
    binding.build()
    g = binding.oracle().generate(scale, 16)
    off, nbr = g.csr()
    core, ms_core = timed(lambda: tor.core_numbers(off, nbr))
    truss, ms_truss = timed(lambda: tor.truss_numbers(off, nbr))
    return {"graph": f"kronecker-{scale}",
            "cpu_checker": "sequential bucket peels (tests/cpp/truss_oracle.cpp), one thread", "n": g.n, "m": len(truss), "degeneracy": int(core.max()), "max_truss": int(truss.max()),
            "cpu_ms_core_numbers": round(ms_core, 1), "cpu_ms_truss_numbers": round(ms_truss, 1),
            "cpu": platform.processor() or platform.machine()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scales", default="20,22,24")
    ap.add_argument("--oracle-scale", type=int, default=None)
    args = ap.parse_args()
    if args.oracle_scale is not None:
        print(json.dumps(oracle_line(args.oracle_scale)), flush=True)
    if args.scales:
        import gms_b200 as G
        G.set_device(0)
        for s in [int(x) for x in args.scales.split(",")]:
            print(json.dumps(bench_scale(G, s)), flush=True)


if __name__ == "__main__":
    main()
