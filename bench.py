#!/usr/bin/env python
"""bench.py — triangle counting on Kronecker scale-24 (edge factor 16), BASELINE.json configs[1].

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--scale S] [--variant V]
                    [--dump-outputs DIR]

Our arm (default).  Untimed setup: generate the edge list with the reference generator's semantics, build the
symmetric CSR on the GPU (radix sort), keep a copy of the CSR in PINNED host memory.  Then
  * `value`  : K steps of count_total over the device graph.  The reference harness (gms/common/benchmark.h:96-137)
               builds SGraph::FromCGraph once outside the timed trials; the analogue here is the degree-oriented DAG,
               which is built once (`dag_ms`).  The triangle SCHEDULE (descriptors grouped by closing vertex, hub
               items, light lists) is specific to this kernel, so it is rebuilt INSIDE every timed step
               (gmsb_tc_options.reuse_plan = 2): a step = schedule build + every counting kernel over all oriented
               edges + the count back (checked every step).  `count_only` is the same without the schedule build;
  * `e2e`    : K steps of the call a user makes from host memory: gmsb_graph_from_csr_ex(GMSB_BUILD_ORIENT) (pinned host
               CSR -> HBM, orientation pipelined with the upload) + gmsb_tc_total_ex (schedule + count, nothing
               cached) + the 8-byte result back + free;
  * `roofline`: the dominant kernel (k_tc_bitmap) — its algorithmic bytes / its CUDA-event time, vs MEASURED_PEAKS;
  * `cpu_baseline` (N=1): the reference's own Par::count_total inner loop (oracle/_ref, else the oracle port) on a
               bounded sample of the same graph, all host threads;
  * `kclique` : the other half of BASELINE.json's metric — k-clique counts/s for k = 4,5,6 on configs[2]
               (Kronecker scale-22), sub-problems dealt over the ranks, one all-reduce (--kclique '' skips it); at N=1
               with `kclique.cpu_baseline`: the reference's Par::EP_kclisting on all host threads on Kronecker
               scale-16 and our kernels on that same graph.
N>1 (torchrun): every rank holds the graph, builds and counts only ITS share of the schedule (the edges whose closing
vertex it owns), one all-reduce sums the counts; time = max over ranks.  In the e2e leg rank r uploads 1/N of the offsets
and the neighbour slots of vertex range r, orients that range, and the finished rows are all-gathered over NVLink
(gmsb_shard_*), so h2d_bytes_per_step is still the whole CSR once (summed over ranks).

Reference arm (--impl reference): rank 0 only, the reference's CPU path on bounded samples of the same workload.
"""
import argparse
import atexit
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

REF_FULL_SCALE = 20        # the reference's complete run / our like-for-like check (about a minute of CPU time)
# Largest k of the CPU k-clique baseline when the oracle port stands in for the reference library (kind "port").  On
# Kronecker scale-16 with 16 host threads of a B200 machine the reference took 0.50 / 3.4 / 41 s for k = 4 / 5 / 6
# (profiles/r2r_bench_1gpu.json) and the port 5.4 / 99.6 s for k = 4 / 5; k = 6 would keep the port busy for about
# half an hour, so it is left out (reported in skipped_k).
KCLIQUE_PORT_MAX_K = 5
METRIC = "tc_edges_per_sec"
UNIT = "edges/s"


def log(*a):
    print(*a, file=sys.stderr, flush=True)


# Libraries (NCCL's version banner, the reference's progress lines) write to fd 1; the contract is ONE JSON line on
# stdout, so fd 1 is pointed at stderr for the whole run and the result line goes to the saved descriptor.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


def emit_result(obj):
    os.write(_REAL_STDOUT, (json.dumps(obj) + "\n").encode())


def dump_outputs(path, arrays):
    """--dump-outputs: each result the timed legs returned in their last step, as <path>/<name>.npy in float64."""
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, np.float64))
    log(f"[dump] {', '.join(sorted(arrays))} -> {path}")


def count_words(c):
    """A count as (c >> 32, c & 0xffffffff): both words are exact in float64 whatever the count (the 8-GPU k = 7 count
    on Kronecker scale-22, ~1.4e16, is above 2**53), so dumps of two builds differ exactly when the counts do."""
    return [c >> 32, c & 0xffffffff]


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


def ncu_capture(kernel):
    """The committed, dated `ncu --set full` capture of `kernel` on the scale-24 workload (profiles/traffic.json):
    DRAM bytes per counting step and the issue counters; None when no capture is committed."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)[kernel]
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            atexit.register(self.proc.terminate)        # a run that fails before stop() leaves no sampler behind
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm = [float(r[1]) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 8 for i in range(4) if r[4 + i] == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def cpu_sample_stride(deg, cores, target_seconds):
    """Pick the edge-sampling stride so the reference loop does ~target_seconds of work.
    Work of the reference loop = sum over undirected edges of (d(u)+d(v)) = sum_u d(u)^2 list elements."""
    elems = float((deg.astype(np.float64) ** 2).sum())
    rate = 0.25e9 * max(cores, 1)            # ~elements/s per core of the branchy scalar merge (SURVEY.md §6)
    return max(1, int(np.ceil(elems / rate / target_seconds))), elems


def cpu_lib():
    from oracle import binding
    ref = binding.reference()
    lib, kind = (ref, "reference") if ref is not None else (None, "port")
    if lib is None:
        binding.build()
        lib = binding.oracle()
    # torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU baseline is meant to use every host core
    lib.set_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    return lib, kind


def run_reference(args):
    """The reference's CPU implementation on the host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    lib, kind = cpu_lib()
    cores = lib.max_threads()
    t0 = time.time()
    g = lib.generate(args.scale, 16, False)            # the reference's own generator + builder
    off, _ = g.csr()
    deg = np.diff(off)
    m = g.slots // 2
    log(f"[reference] built kronecker-{args.scale}: n={g.n} m={m} in {time.time() - t0:.1f}s; kind={kind} cores={cores}")
    total = args.steps + args.warmup
    per_step = max(2.0, min(10.0, 150.0 / max(total, 1)))
    stride, elems = cpu_sample_stride(deg, cores, per_step)
    g.tc_total_sample(max(stride * 8, 8), 0)           # builds the SetGraph (FromCGraph) outside the timing
    times, edges = [], 0
    for i in range(total):
        sec, e, _ = g.tc_total_sample(stride, i % stride)
        if i >= args.warmup:
            times.append(sec)
            edges += e
    T = sum(times)
    value = edges / T
    sample = (f"every {stride}-th undirected edge (u<v, CSR order) of kronecker-{args.scale} per step, "
              f"SortedSet::intersect_count over full neighbourhoods, omp dynamic, {cores} threads")
    # one complete run of the reference's Par::count_total at a size it finishes in about a minute, so that one
    # ratio is like for like (bench.py's own arm reports the same graph as `same_config_check`)
    full = None
    if not args.no_full_reference:
        g20 = lib.generate(REF_FULL_SCALE, 16, False)
        g20.tc_total_sample(1 << 20, 0)                 # FromCGraph outside the timing, as the harness does
        sec, tri = g20.tc_total_timed(True)
        full = {"scale": REF_FULL_SCALE, "n": g20.n, "m": g20.slots // 2, "triangles": tri, "seconds": sec,
                "value": (g20.slots // 2) / sec, "unit": UNIT,
                "what": "TriangleCount::Par::count_total<SortedSetGraph>, every edge, all host threads"}
        log(f"[reference] full run kronecker-{REF_FULL_SCALE}: {sec:.1f}s, {tri} triangles")
    emit_result({
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * T / max(args.steps, 1),
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"triangle counting, Kronecker scale-{args.scale} edge factor 16 (n={g.n}, m={m})",
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "full_run": full,
    })


def run_kclique(args, G, gd, rank, world, dev):
    """k-clique counting (Danisch-style, degree-oriented DAG) on Kronecker scale-`kclique_scale`: the per-vertex
    sub-problems are dealt out over the ranks (gmsb_kclique_count_ex), counts summed by one all-reduce; time = max
    over ranks of the wall time around the C-ABI call (it returns the count, i.e. it is synchronous)."""
    import torch
    src, dst = G.generate_rmat(args.kclique_scale)
    g = G.Graph.from_edgelist(src, dst, True)
    del src, dst
    m = g.slots // 2
    g.kclique_count(3, rank, world)                    # builds the oriented DAG, warms the allocator
    rows = []
    for k in kclique_sizes(args, world):
        gd.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        part = g.kclique_count(k, rank, world)
        sec = gd.allreduce_max(time.perf_counter() - t0, device=dev)
        total, = gd.allreduce_counts([part], device=dev)
        rows.append({"k": k, "count": total, "seconds": sec, "cliques_per_s": total / sec, "edges_per_s": m / sec})
        log(f"[rank {rank}] kclique k={k}: {total} in {sec:.3f}s")
    out = {"workload": f"k-clique counting, Kronecker scale-{args.kclique_scale} edge factor 16 (n={g.n}, m={m}), "
                       "degree-oriented DAG (the degeneracy orientation BASELINE.json names was measured and is slower "
                       "here: profiles/r2a_kclique_orientation.jsonl), graph replicated, sub-problems dealt over the ranks",
           "metric": "kclique_counts_per_sec", "unit": "cliques/s", "n_gpus": world, "results": rows,
           "roofline": kclique_roofline(),
           "note": "k = 7 runs by default only at 8 GPUs (one B200 needs about half an hour for it); k = 8 is not run: "
                   "the count grows ~50x per k on this graph (DESIGN.md section 3)"}
    g.free()
    # the reference's Par::EP_kclisting beside it (rank 0, N=1): bounded by running it on a smaller graph of the same
    # family, with our kernels timed on that same graph for a like-for-like ratio
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            out["cpu_baseline"] = kclique_cpu_baseline(args, G)
        except Exception as ex:      # reported, never required
            out["cpu_baseline"] = {"kind": "unavailable", "sample": str(ex)}
    return out


def kclique_sizes(args, world):
    if args.kclique != "auto":
        return [int(x) for x in args.kclique.split(",")]
    return [4, 5, 6, 7] if world >= 8 else [4, 5, 6]


def kclique_roofline():
    """Pipe utilisation of the clique kernels from the committed, dated ncu capture (profiles/kclique_pipes.json): the
    search is AND + popcount over bit-matrix rows, bound by the SM's XU (POPC / FLO, quarter rate) and ALU pipes."""
    try:
        with open(os.path.join(ROOT, "profiles", "kclique_pipes.json")) as f:
            return json.load(f)
    except Exception:
        return None


def kclique_cpu_baseline(args, G, scale=16):
    lib, kind = cpu_lib()
    cores = lib.max_threads()
    cg = lib.generate(scale, 16, False)
    # the reference's own pipeline: getDegeneracyOrderingDanischHeap -> InduceDirectedGraph -> EP_kclisting
    # (gms/algorithms/non_set_based/k_clique_list/bench_helper.h:33-38)
    t0 = time.perf_counter()
    dag = cg.induce_directed(lib.degeneracy_rank(cg))
    pre_s = time.perf_counter() - t0
    src, dst = G.generate_rmat(scale)
    g = G.Graph.from_edgelist(src, dst, True)
    g.kclique_count(3)
    rows = []
    sizes = [k for k in kclique_sizes(args, 1) if k <= 6]
    skipped = [k for k in sizes if kind == "port" and k > KCLIQUE_PORT_MAX_K]
    for k in [k for k in sizes if k not in skipped]:
        sec, cnt = dag.kclique_timed(k, 2)                     # mode 2 = edge-parallel (EP_kclisting)
        best = None
        for _ in range(3):
            t0 = time.perf_counter()
            ours = g.kclique_count(k)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        assert ours == cnt, (k, ours, cnt)
        rows.append({"k": k, "count": cnt, "cpu_seconds": sec, "cpu_cliques_per_s": cnt / sec, "gpu_seconds": best,
                     "gpu_cliques_per_s": cnt / best})
        log(f"[cpu_baseline] kclique k={k} scale {scale}: {kind} {sec:.2f}s on {cores} threads, GPU {best * 1e3:.2f} ms")
    g.free()
    if skipped:
        log(f"[cpu_baseline] kclique k={skipped} scale {scale}: not run on the {kind} (k <= {KCLIQUE_PORT_MAX_K})")
    return {"kind": kind, "cores": cores, "unit": "cliques/s", "preprocess_seconds": pre_s,
            "sample": f"Kronecker scale-{scale} edge factor 16 (same generator), the reference's pipeline: DanischHeap "
                      f"degeneracy order -> InduceDirectedGraph -> KClique::Par::EP_kclisting on all host threads; "
                      f"gpu_seconds = gmsb_kclique_count on the same graph",
            "results": rows, "skipped_k": skipped}


def run_e2e(args, G, gd, off_h, nbr_h, n, slots, m, opts, expect, world, dev):
    """host CSR -> HBM -> orient -> schedule -> count -> result, nothing cached.  N = 1: the C-ABI call on the host
    buffers (gmsb_graph_from_csr_ex, upload pipelined with the orientation).  N > 1: the sharded build (gmsb_shard_*,
    gms_b200/dist.py: ShardedOrientedBuild) — rank r uploads and orients vertex range r of N, the finished rows are
    all-gathered over NVLink, so the host copy is read once and the orientation passes are split N ways."""
    import torch
    sharded = gd.ShardedOrientedBuild(off_h, nbr_h[:slots], dev) if world > 1 else None

    def e2e_step():
        if sharded is None:
            gg = G.Graph.from_csr(off_h.numpy(), nbr_h.numpy()[:slots], orient=True)   # GMSB_BUILD_ORIENT
        else:
            gg = sharded.build()
        c, s2 = gg.tc_total_ex(reuse_plan=False, **opts)
        gg.free()
        return c, s2

    for _ in range(min(args.warmup, 2)):
        e2e_step()
    e2e_steps = args.steps
    gd.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e2e_parts, e2e_orient = [], []
    for _ in range(e2e_steps):
        c, s2 = e2e_step()
        e2e_parts.append(c)
        e2e_orient.append(s2["ms_orient"])
    torch.cuda.synchronize()
    e2e_ms = gd.allreduce_max((time.perf_counter() - t0) * 1e3, device=dev)
    e2e_totals = gd.allreduce_counts(e2e_parts, device=dev)
    assert all(t == expect for t in e2e_totals)
    e2e_value = m * e2e_steps / (e2e_ms * 1e-3)

    return e2e_value, e2e_ms, e2e_steps, e2e_orient, e2e_totals[-1]


def run_ours(args):
    import torch
    import gms_b200 as G
    from gms_b200 import dist as gd

    rank, world, local = gd.init()
    assert world == args.gpus or world == 1, f"--gpus {args.gpus} but WORLD_SIZE={world}"
    torch.cuda.set_device(local)
    G.set_device(local)
    dev = torch.device("cuda", local)

    # ---- untimed setup: edge list (rank 0 generates, shared through /dev/shm), symmetric CSR on the GPU
    t0 = time.time()
    shm = f"/dev/shm/gmsb_kron{args.scale}_{os.environ.get('MASTER_PORT', '0')}.npy"
    if rank == 0:
        src, dst = G.generate_rmat(args.scale, a=args.rmat_a, b=(0.95 - args.rmat_a) / 2, c=(0.95 - args.rmat_a) / 2)
        if world > 1:
            np.save(shm, np.stack([src, dst]))
    gd.barrier()
    if rank != 0:
        el = np.load(shm, mmap_mode="r")
        src, dst = np.ascontiguousarray(el[0]), np.ascontiguousarray(el[1])
    t_gen = time.time() - t0
    t0 = time.time()
    g = G.Graph.from_edgelist(src, dst, True)
    G.synchronize()
    t_build = time.time() - t0
    del src, dst
    gd.barrier()
    if rank == 0 and world > 1:
        os.remove(shm)
    n, slots = g.n, g.slots
    m = slots // 2
    family = "Kronecker" if abs(args.rmat_a - 0.57) < 1e-9 else f"R-MAT(a={args.rmat_a})"
    log(f"[rank {rank}] {family}-{args.scale}: n={n} m={m} generate {t_gen:.1f}s build-on-gpu {t_build:.2f}s")

    # pinned host copy of the CSR: the e2e leg's input
    off_h = nbr_h = None
    if not args.no_e2e:
        off_h = torch.empty(n + 1, dtype=torch.int64).pin_memory()
        nbr_h = torch.empty(max(slots, 1), dtype=torch.int32).pin_memory()
        G.capi._check(G.lib().gmsb_graph_export_csr(g.h, off_h.numpy(), nbr_h.numpy()))

    opts = dict(variant=args.variant, part_index=rank, part_count=world)
    # ---- representation build (FromCGraph analogue): ranking + oriented DAG; the schedule is rebuilt in every step
    g.tc_total_ex(reuse_plan=False, **opts)            # warms the device-memory arena (first-ever cudaMalloc of GBs)
    _, st_cold = g.tc_total_ex(reuse_plan=False, **opts)
    prep_ms = st_cold["ms_orient"]                     # ranking + DAG + schedule, steady state
    part, st0 = g.tc_total_ex(reuse_plan=1, **opts)    # leaves the DAG cached on the handle
    expect, = gd.allreduce_counts([part], device=dev)

    def step():
        c, st = g.tc_total_ex(reuse_plan=2, **opts)    # keep the DAG, rebuild the schedule, count
        return c, st

    sampler = ClockSampler(local)
    if rank == 0 and not args.no_clocks:
        sampler.start()          # nvidia-smi's own start-up stalls the driver for a moment: keep it out of the timing
        time.sleep(1.5)
    for _ in range(args.warmup):
        step()
    if rank == 0:
        sampler.rows.clear()     # keep only samples taken under load
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = G.launch_count()
    gd.barrier()
    torch.cuda.synchronize()
    ev0.record()
    ms_bitmap, ms_count, ms_sched, parts, wall = [], [], [], [], []
    for _ in range(args.steps):
        tw = time.perf_counter()
        c, st = step()
        wall.append((time.perf_counter() - tw) * 1e3)
        parts.append(c)
        ms_bitmap.append(st["ms_bitmap"])
        ms_count.append(st["ms_count"])
        ms_sched.append(st["ms_orient"])
    ev1.record()
    torch.cuda.synchronize()
    gd.barrier()
    ms_total = gd.allreduce_max(ev0.elapsed_time(ev1), device=dev)
    launches = G.launch_count() - l0
    clocks = sampler.stop() if rank == 0 else None
    totals = gd.allreduce_counts(parts, device=dev)
    assert all(t == expect for t in totals), (totals, expect)
    outputs = {"triangles": count_words(totals[-1])}
    st = st0
    value = m * args.steps / (ms_total * 1e-3)

    # ---- e2e: host CSR -> HBM -> orient -> schedule -> count -> result, nothing cached
    # N = 1: the plain C-ABI call on the host buffers; N > 1: the sharded build (every rank uploads 1/N of the offsets and
    # its own vertex range of the neighbour array; h2d counts all ranks)
    e2e_value, e2e_ms, e2e_steps, e2e_orient, h2d = None, float("nan"), 1, [float("nan")], 8 * (n + 1) + 4 * slots
    if not args.no_e2e:
        e2e_value, e2e_ms, e2e_steps, e2e_orient, e2e_last = run_e2e(args, G, gd, off_h, nbr_h, n, slots, m, opts, expect,
                                                                     world, dev)
        outputs["e2e_triangles"] = count_words(e2e_last)

    # ---- roofline of the dominant kernel (k_tc_bitmap2), three views of the same launch:
    #   frac            what the formulation has to pull through the memory system — 4 B per probed list element (only the
    #                   suffix after v is read), 8 B per descriptor, N+(v) once per item — over the measured HBM peak;
    #   frac_dram       DRAM bytes of the dated ncu capture of this workload over the same peak;
    #   frac_algorithmic  SURVEY.md 8(d): 4*(d+(u)+d+(v)) per oriented edge, i.e. both full lists streamed per edge, which
    #                   the suffix + on-chip-bitmap formulation does not do (hence > 1; kept for comparison with round 1).
    peak, peak_src = peaks()
    bm_ms = float(np.mean(ms_bitmap))
    count_ms = float(np.mean(ms_count))
    sched_ms = float(np.mean(ms_sched))
    # (N > 1: every statistic of the schedule is this rank's share, like the kernel time beside it)
    alg_bytes = st["bytes_bitmap"]
    min_traffic = 4.0 * st["wedges_bitmap"] + 8.0 * st["edges_bitmap"] + 32.0 * st["bitmap_items"]
    cap = ncu_capture("k_tc_bitmap2") if world == 1 else None
    achieved = min_traffic / (bm_ms * 1e-3) / 1e9 if bm_ms > 0 else 0.0
    roofline = {
        "bound": "hbm", "kernel": "k_tc_bitmap2", "achieved": achieved, "peak": peak, "unit": "GB/s",
        "frac": achieved / peak, "traffic": cap["dram_bytes_per_launch"] if cap else None, "peak_source": peak_src,
        "kernel_ms": bm_ms, "min_traffic_bytes": min_traffic,
        "frac_dram": (cap["dram_bytes_per_launch"] / (bm_ms * 1e-3) / 1e9 / peak) if cap and bm_ms else None,
        "algorithmic_bytes_per_launch": alg_bytes,
        "frac_algorithmic": alg_bytes / (bm_ms * 1e-3) / 1e9 / peak if bm_ms else None,
        "issue": ({"warp_inst_per_32_probes": 32.0 * cap["smsp_inst_executed"] / cap["probes"],
                   "issue_active_pct": cap["issue_active_pct"], "l2_hit_pct": cap["lts_hit_pct"],
                   "capture": cap["capture"]} if cap and "smsp_inst_executed" in cap else None),
        "all_count_kernels": {"algorithmic_bytes": st["algorithmic_bytes"], "ms": count_ms},
        "note": "frac = bytes the suffix + on-chip-bitmap formulation must request / kernel time / measured HBM peak; "
                "about half of them are served by the L2 (frac_dram); the kernel is latency- and issue-bound, see "
                "profiles/r2d_bitmap_ncu.txt",
    }

    out = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": f"triangle counting, {family} scale-{args.scale} edge factor 16 (n={n}, m={m})",
                   "variant": args.variant, "parallelism": f"edge-partition x{world} by closing vertex, schedule built per share",
                   "l2": "inputs_exceed_L2 (oriented CSR %.2f GB vs 126 MB L2)" % (st["oriented_edges"] * 4 / 1e9),
                   "step": "schedule build + count_total over the oriented device graph (DAG built once, dag_ms); "
                           "everything from the host CSR on is in e2e"},
        "triangles": expect, "prep_ms": prep_ms, "dag_ms": prep_ms - sched_ms, "schedule_ms": sched_ms,
        "count_ms": count_ms, "step_wall_ms": [round(w, 2) for w in wall],
        "count_only": {"value": m / (count_ms * 1e-3) if count_ms else None, "unit": UNIT, "ms_per_step": count_ms,
                       "note": "counting kernels alone over a cached schedule (round-1 definition of value)"},
        "kernel_ms": {"bitmap": bm_ms, "merge": st["ms_merge"], "gallop": st["ms_gallop"]},
        "edges_by_kernel": {"bitmap": st["edges_bitmap"], "merge": st["edges_merge"], "gallop": st["edges_gallop"]},
        "roofline": roofline, "clocks": clocks, "gpu_launches": int(launches),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                "ms_per_step": e2e_ms / e2e_steps, "schedule_and_rest_ms": float(np.mean(e2e_orient)),
                "note": ("gmsb_graph_from_csr_ex(GMSB_BUILD_ORIENT) from pinned host memory (upload pipelined with the "
                         "ranking / validation / orientation passes) + gmsb_tc_total_ex with nothing cached + result"
                         if world == 1 else
                         "gmsb_shard_begin / export / finish from pinned host memory (each rank uploads 1/N of the offsets "
                         "and one vertex range of the neighbour array and orients that range; offsets and finished rows "
                         "all-gathered over NVLink) + gmsb_tc_total_ex with nothing cached + result")},
    }

    if args.no_e2e:
        out["e2e"] = {"value": None, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 8,
                      "note": "skipped (--no-e2e)"}
    # ---- CPU baseline beside it (rank 0, N=1 only): bounded sample of the same graph
    if rank == 0 and world == 1 and not args.no_cpu_baseline and off_h is not None:
        try:
            lib, kind = cpu_lib()
            cores = lib.max_threads()
            off_np = off_h.numpy()
            stride, _ = cpu_sample_stride(np.diff(off_np), cores, 12.0)
            t0 = time.time()
            cg = lib.from_csr(off_np, nbr_h.numpy()[:slots], False)
            cg.tc_total_sample(max(stride * 16, 16), 1)       # FromCGraph outside the timing
            sec, e, _ = cg.tc_total_sample(stride, 0)
            log(f"[cpu_baseline] {kind} {cores} threads: setup {time.time() - t0 - sec:.1f}s, sample {sec:.1f}s")
            out["cpu_baseline"] = {
                "value": e / sec, "unit": UNIT, "cores": cores, "kind": kind, "seconds": sec,
                "sample": f"every {stride}-th undirected edge (u<v, CSR order) of the same graph, "
                          f"SortedSet::intersect_count over full neighbourhoods, omp dynamic"}
        except Exception as ex:      # the baseline is reported, never required
            out["cpu_baseline"] = {"value": None, "unit": UNIT, "cores": 0, "kind": "unavailable", "sample": str(ex)}
    g.free()
    # ---- like-for-like size for the reference arm's complete run (--impl reference reports `full_run` at this scale)
    if rank == 0 and world == 1 and abs(args.rmat_a - 0.57) < 1e-9:
        s20, d20 = G.generate_rmat(REF_FULL_SCALE)
        g20 = G.Graph.from_edgelist(s20, d20, True)
        g20.tc_total_ex(reuse_plan=False)
        t0 = time.perf_counter()
        tri20, st20 = g20.tc_total_ex(reuse_plan=False)
        wall20 = time.perf_counter() - t0
        out["same_config_check"] = {"scale": REF_FULL_SCALE, "m": g20.slots // 2, "triangles": tri20,
                                    "seconds": wall20, "value": (g20.slots // 2) / wall20, "unit": UNIT,
                                    "what": "gmsb_tc_total_ex with nothing cached (ranking + DAG + schedule + count), "
                                            "device graph resident; compare with --impl reference full_run"}
        g20.free()
    # ---- the other half of BASELINE.json's metric: k-clique counts/s on configs[2] (Kronecker scale-22 ef16)
    if args.kclique:
        out["kclique"] = run_kclique(args, G, gd, rank, world, dev)
        outputs["kclique_counts"] = [[r["k"]] + count_words(r["count"]) for r in out["kclique"]["results"]]
    if rank == 0:
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
        emit_result(out)
    gd.barrier()
    if torch.distributed.is_initialized():
        torch.distributed.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--scale", type=int, default=24)
    ap.add_argument("--variant", default="auto", choices=["auto", "merge", "gallop", "bitmap"])
    ap.add_argument("--rmat-a", type=float, default=0.57,
                    help="R-MAT a (b = c = (0.95 - a) / 2); 0.57 is the reference's kronecker, 0.65 BASELINE.json configs[4]")
    ap.add_argument("--kclique", default="auto",
                    help="clique sizes timed on configs[2] after the TC legs ('' = skip; auto = 4,5,6 and 7 at 8 GPUs)")
    ap.add_argument("--kclique-scale", type=int, default=22)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-clocks", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-CSR end-to-end leg (scale-26 runs: 8.6 GB pinned per rank)")
    ap.add_argument("--no-full-reference", action="store_true", help="reference arm: skip the complete scale-20 run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the run, write what the timed legs computed in their last step to DIR/<name>.npy "
                         "in float64, every count c as the words (c >> 32, c & 0xffffffff): triangles, e2e_triangles, "
                         "kclique_counts as rows of (k, high word, low word); ours only")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
