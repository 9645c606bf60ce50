#!/usr/bin/env python
"""bench.py — the measurement contract for the PageRank hot path.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W
    python bench.py --gpus 1 --scale 27                      (the single-GPU denominator of the scale-27 configuration)
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   (also writes the last timed step's result as .npy)

Workload (BASELINE.json configs[1]): PageRank on RMAT scale-24 edge-factor-16 (Graph500 a,b,c,
multi-edges and self-loops kept, scrambled ids, unweighted, int32 ids / float32 scores), alpha 0.85,
epsilon 0 (never converges), 100 iterations, graph stored transposed.  N>1: weak scaling with 2^28 edge
draws per GPU (scale 24 + log2 N; N = 8 is BASELINE's scale-27 configuration), 2D edge partition.

A STEP is one call of `cugraph_pagerank_allow_nonconvergence` (100 iterations) through the C-ABI.
  value  = MTEPS = E * iterations * steps / time, graph already resident in HBM (graph creation is
           staging, excluded exactly as the reference's own harness does, pagerank_test.cpp:221-236)
  e2e    = the same metric for the whole reference-facing call sequence with HOST buffers inside the
           timed region: pinned edge list -> H2D -> cugraph_graph_create_with_times_sg -> pagerank ->
           D2H of (vertices, scores)
  roofline = the pull-SpMV sweep (kernels k_sweep + k_sweep_finish = one per_v_transform_reduce_incoming_e)
           timed alone with CUDA events on the handle's stream; algorithmic bytes per sweep =
           4E + 4(V+1) + 4V + 4V (SURVEY.md §8d); traffic = DRAM bytes of the two kernels from the ncu capture
           of the same kernels on the same workload (profiles/spmv_traffic.json names the capture)
  config.bfs_* / config.sssp_* = BASELINE.json configs[2], [3]: BFS (direction-optimising, 64 random sources) and SSSP
           (8 sources) on the symmetrised RMAT-24 graph, Graph500 TEPS (undirected edges of the source's component /
           time of the C-ABI call), harmonic + arithmetic mean, with size-independent result checks
  cpu_baseline = the CPU port of the same algorithm (oracle/bench_ref.c, float32, OpenMP on the physical cores) on a
           bounded sample; cpu_baseline.networkx_mteps = nx.pagerank (BASELINE's named baseline) on a small sample
  timing = CUDA events recorded on the handle's stream (the stream the library launches on) around the K calls;
           the wall-clock time of the same region is reported next to it
Synthetic data, random seed 0.  Inputs (1.2 GB per sweep) exceed the 126 MB L2, so no explicit L2 flush
is needed between timed iterations (stated in config.l2).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ALPHA, ITERS = 0.85, 100


def metric_name(scale, n_gpus=1):
    m = f"MTEPS (million traversed edges/sec) PageRank RMAT-{scale} ef-16, 100 iterations"
    return m if n_gpus == 1 else m + f", {n_gpus} GPUs (2D edge partition)"


def physical_cores():
    """physical cores this process may run on (cgroup / affinity aware)"""
    try:
        allowed = os.sched_getaffinity(0)
    except Exception:
        allowed = set(range(os.cpu_count() or 1))
    cores = set()
    try:
        for cpu in allowed:
            with open(f"/sys/devices/system/cpu/cpu{cpu}/topology/thread_siblings_list") as f:
                cores.add(f.read().strip())
        return max(1, len(cores))
    except Exception:
        return max(1, len(allowed))


def pin_host_threads():
    """OpenMP settings of the CPU arms, fixed BEFORE any OpenMP runtime is loaded: one thread per physical core, bound.
    (torchrun exports OMP_NUM_THREADS=1 and an unpinned 128-thread run once performed like a single thread: the CPU arm
    wandered 6.5x between boxes, VERDICT r01.)"""
    n = physical_cores()
    os.environ["OMP_NUM_THREADS"] = str(n)
    os.environ["OMP_PROC_BIND"] = "close"
    os.environ["OMP_PLACES"] = "cores"
    os.environ.setdefault("OMP_WAIT_POLICY", "active")
    return n


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = float(r[1])
                for k, nm in enumerate(names):
                    if r[3 + k].lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def _cpu_port_pagerank(scale, budget_s, steps=1, warmup=0):
    """The CPU port (oracle/bench_ref.c: float32 PageRank, OpenMP) on RMAT-`scale` ef-16: `steps` timed steps after
    `warmup` untimed ones.  A step is 100 iterations unless that cannot fit the time budget, then fewer (said so)."""
    import oracle
    V, E = 1 << scale, 16 << scale
    t0 = time.perf_counter()
    src, dst = oracle.bench_rmat_edges(scale, E, seed=0)
    off, idx, deg = oracle.bench_build_csc(src, dst, V)
    del src, dst
    setup_s = time.perf_counter() - t0
    pr = oracle.BenchPageRank(off, idx, deg, ALPHA)
    pr.run(1)                                   # page in, warm the caches
    t0 = time.perf_counter()
    pr.run(2)
    per_it = (time.perf_counter() - t0) / 2
    its = ITERS
    total = (steps + warmup) * ITERS * per_it
    if total > budget_s:
        its = max(2, int(budget_s / ((steps + warmup) * per_it)))
    for _ in range(warmup):
        pr.reset()
        pr.run(its)
    t0 = time.perf_counter()
    for _ in range(steps):
        pr.reset()
        pr.run(its)
    dt = time.perf_counter() - t0
    return {"value": E * its * steps / dt / 1e6, "ms_per_step": dt / steps * 1e3, "iterations_per_step": its,
            "cores": oracle.num_threads(), "setup_s": setup_s, "scale": scale, "edges": E}


def _cpu_baseline(sample_scale=22, target_s=12.0):
    """cpu_baseline of the GPU arm: the same port as `--impl reference` on a bounded sample (rank 0, N = 1 only).  Runs in a
    CHILD process: the OpenMP settings of the CPU arm (one bound, actively waiting thread per physical core) must not leak
    into the process that drives the GPU — with them set here the host thread could not keep the GPU fed (PageRank measured
    100 ms per step instead of 39)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "cpu-sample", "--scale", str(sample_scale)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    if r.returncode != 0 or not lines:
        raise RuntimeError(f"cpu-sample child failed ({r.returncode}): {r.stderr[-300:]}")
    return json.loads(lines[-1])


def run_cpu_sample(args, target_s=12.0):
    """child of _cpu_baseline (threads already pinned by main): prints the cpu_baseline object"""
    scale = args.scale or 22
    r = _cpu_port_pagerank(scale, target_s, steps=1, warmup=0)
    out = {"value": r["value"], "unit": "MTEPS", "cores": r["cores"], "kind": "port",
           "sample": f"{r['iterations_per_step']} float32 PageRank iterations (oracle/bench_ref.c, OpenMP, threads bound to "
                     f"physical cores) on RMAT scale-{scale} ef-16; graph set-up ({r['setup_s']:.1f} s) not timed"}
    nx = _networkx_baseline(min(scale, 16))
    out["networkx_mteps"] = nx.get("value")
    out["networkx_sample"] = nx.get("sample") or nx.get("error")
    print(json.dumps(out), flush=True)


def _networkx_baseline(scale):
    """NetworkX (BASELINE.json's named CPU baseline): nx.pagerank, 100 power iterations (tol = 0 never converges; the
    PowerIterationFailedConvergence after max_iter marks the end), on a small RMAT sample — building a NetworkX graph at
    benchmark scale is prohibitive.  Graph construction is not timed."""
    try:
        import networkx as nx
        import oracle
        src, dst = oracle.bench_rmat_edges(scale, 16 << scale, seed=0)
        G = nx.MultiDiGraph()
        G.add_edges_from(zip(src.tolist(), dst.tolist()))
        t0 = time.perf_counter()
        try:
            nx.pagerank(G, alpha=ALPHA, tol=0.0, max_iter=ITERS)
        except nx.PowerIterationFailedConvergence:
            pass
        dt = time.perf_counter() - t0
        return {"value": src.shape[0] * ITERS / dt / 1e6, "unit": "MTEPS", "cores": 1, "version": nx.__version__,
                "sample": f"nx.pagerank {nx.__version__}, {ITERS} iterations, RMAT scale-{scale} ef-16 MultiDiGraph (SciPy-backed, 1 thread)"}
    except Exception as ex:
        return {"value": None, "error": f"{type(ex).__name__}: {ex}"[:200]}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  libcugraph cannot be built here (DESIGN.md §4), so
    this is the port of its algorithm (oracle/bench_ref.c) — on the BENCHMARK configuration itself: RMAT scale-24 ef-16,
    float32, 100 iterations per step, all physical cores.  Rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    scale = args.scale or 24
    r = _cpu_port_pagerank(scale, budget_s=float(os.environ.get("CUGRAPH_B200_REF_BUDGET_S", "150")), steps=args.steps,
                           warmup=args.warmup)
    its = r["iterations_per_step"]
    sample = (f"PageRank on RMAT scale-{scale} ef-16, float32, {its} iterations per step"
              + ("" if its == ITERS else f" (of the {ITERS} of a full step: time-bounded sample, MTEPS is per iteration)")
              + f", oracle/bench_ref.c, OpenMP {r['cores']} threads bound to physical cores")
    out = {"impl": "reference", "metric": metric_name(scale), "value": r["value"], "unit": "MTEPS", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"pagerank_rmat{scale}_ef16_100it", "scale": scale, "edge_factor": 16, "num_edges": r["edges"],
                      "alpha": ALPHA, "iterations": ITERS, "iterations_timed_per_step": its, "vertex_type": "int32"},
           "cpu_baseline": {"value": r["value"], "unit": "MTEPS", "cores": r["cores"], "kind": "port", "sample": sample},
           "e2e": {"value": r["value"], "unit": "MTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def run_single(args):
    import torch
    from cugraph_b200 import _capi
    from cugraph_b200 import pylibcugraph as plc
    from cugraph_b200.generators import rmat_edgelist
    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(0)
    scale = args.scale
    L = _capi.lib()
    src, dst = rmat_edgelist(scale, 16 << scale, seed=0)
    E = src.numel()
    h = plc.ResourceHandle()
    props = plc.GraphProperties(is_symmetric=False, is_multigraph=True)
    G = plc.SGGraph(h, props, src, dst, store_transposed=True, renumber=True)
    # pinned host copy of the edge list for the e2e arm (the scale-27 denominator run is device-resident only: 17 GB of host
    # staging per step says nothing about the hot path)
    big = scale >= 26
    h_src = h_dst = None
    if not big:
        h_src = torch.empty(E, dtype=torch.int32).pin_memory()
        h_dst = torch.empty(E, dtype=torch.int32).pin_memory()
        h_src.copy_(src)
        h_dst.copy_(dst)
    del src, dst

    def step():
        return plc.pagerank(h, G, None, None, None, None, ALPHA, 0.0, ITERS, False, fail_on_nonconvergence=False)

    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(0)
    torch.cuda.synchronize()
    sampler.start()
    l0 = h.launch_count()
    # CUDA events on the stream the library launches on (the handle's own stream, not torch's current stream)
    hstream = torch.cuda.ExternalStream(int(L.cugraph_b200_handle_stream(h.ptr) or 0))
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(hstream)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v, p, _ = step()  # synchronous on return (the C-ABI syncs the handle's stream)
    e1.record(hstream)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    nv = v.numel()
    if args.dump_outputs:
        dump_pagerank(args.dump_outputs, v, p)
    del v, p
    launches = h.launch_count() - l0
    clocks = sampler.stop()
    dev_s = e0.elapsed_time(e1) * 1e-3  # device time between the two events; wall is the host's view of the same region
    # the calls are synchronous, so the two clocks must agree; if the events saw something else (wrong stream), fall back
    events_ok = 0.5 * wall <= dev_s <= 1.05 * wall
    timed_s = dev_s if events_ok else wall
    ms_step = timed_s / args.steps * 1e3
    value = E * ITERS * args.steps / timed_s / 1e6

    # roofline: the pull sweep alone, CUDA events on the handle's stream inside the library
    # three repeats of 50 back-to-back sweeps each; the fastest repeat counts (the same protocol as the Python-free probe
    # scripts/cbench.cu), all three are reported
    ms, by, err = C.c_double(), C.c_double(), C.c_void_p()
    sweep_runs = []
    for _ in range(3):
        code = L.cugraph_b200_time_pull_spmv(h.ptr, G.ptr, 50, C.byref(ms), C.byref(by), C.byref(err))
        _capi.check(code, err, "cugraph_b200_time_pull_spmv")
        sweep_runs.append(ms.value)
    ms.value = min(sweep_runs)
    peak, peak_src = _peaks()
    achieved = by.value / (ms.value * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "spmv_traffic.json")
    if os.path.exists(tpath) and scale == 24:
        try:
            tj = json.load(open(tpath))
            traffic, traffic_src = tj.get("dram_bytes_per_sweep"), tj.get("source")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                "kernel": "pull sweep: k_sweep + k_sweep_finish",
                "ms_per_sweep": ms.value, "ms_per_sweep_repeats": sweep_runs, "sweeps_per_repeat": 50,
                "algorithmic_bytes_per_sweep": by.value,
                "sweep_mteps": E / (ms.value * 1e-3) / 1e6}
    # the same ratio for a whole PageRank iteration (SURVEY.md §8d: B_iter = B_spmv + 4 V-sized streams of the vertex pass)
    b_iter = by.value + 16.0 * nv
    ms_iter = ms_step / ITERS
    roofline["iteration"] = {"algorithmic_bytes": b_iter, "ms": ms_iter, "achieved": b_iter / (ms_iter * 1e-3) / 1e9,
                             "frac": b_iter / (ms_iter * 1e-3) / 1e9 / peak}

    # the device-resident numbers go to stderr right away: should anything below take the process down, the log has them
    sys.stderr.write("[bench provisional] " + json.dumps({"value": value, "unit": "MTEPS", "ms_per_step": ms_step,
                                                          "gpu_launches": launches, "roofline": roofline}) + "\n")
    sys.stderr.flush()

    # e2e: host edge list -> H2D -> graph create -> pagerank -> D2H
    del G
    torch.cuda.empty_cache()
    e2e_steps = max(1, min(args.steps, 5))
    e2e_warmup = 3  # the stream-ordered memory pool reaches its steady state after a few graph-sized allocate / free rounds
    # pinned host buffers for the result (a pageable .cpu() costs 20-30 ms for 134 MB)
    h_v = torch.empty(nv, dtype=torch.int32).pin_memory()
    h_p = torch.empty(nv, dtype=torch.float32).pin_memory()

    def e2e_step():
        s = h_src.cuda(non_blocking=True)
        d = h_dst.cuda(non_blocking=True)
        g = plc.SGGraph(h, props, s, d, store_transposed=True, renumber=True)  # waits for the two copies first
        vv, pp, _ = plc.pagerank(h, g, None, None, None, None, ALPHA, 0.0, ITERS, False, fail_on_nonconvergence=False)
        assert vv.numel() == nv, f"e2e graph has {vv.numel()} vertices, the resident one {nv}"
        h_v.copy_(vv, non_blocking=True)
        h_p.copy_(pp, non_blocking=True)
        torch.cuda.synchronize()
        return h_v, h_p

    try:
        if big:
            raise RuntimeError(f"not measured at scale {scale} (device-resident denominator run)")
        for _ in range(e2e_warmup):
            e2e_step()
        torch.cuda.synchronize()
        per_step = []
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            t1 = time.perf_counter()
            e2e_step()
            per_step.append((time.perf_counter() - t1) * 1e3)
        torch.cuda.synchronize()
        e2e_wall = time.perf_counter() - t0
        e2e = {"value": E * ITERS * e2e_steps / e2e_wall / 1e6, "unit": "MTEPS", "h2d_bytes_per_step": 2 * E * 4,
               "d2h_bytes_per_step": nv * 8, "steps": e2e_steps, "warmup": e2e_warmup, "ms_per_step": e2e_wall / e2e_steps * 1e3,
               "ms_per_step_min": min(per_step), "ms_per_step_max": max(per_step),
               "includes": "pinned H2D of edge list, graph staging, 100 iterations, D2H of vertices+scores into pinned buffers"}
    except Exception as ex:  # keep the device-resident measurement even if the host-buffer arm fails
        e2e = {"value": None, "unit": "MTEPS", "h2d_bytes_per_step": 2 * E * 4, "d2h_bytes_per_step": nv * 8,
               "error": f"{type(ex).__name__}: {ex}"[:300]}

    del h_src, h_dst, h_v, h_p
    torch.cuda.empty_cache()
    trav = {}
    if os.environ.get("CUGRAPH_B200_BENCH_TRAVERSAL", "1") != "0" and not big:
        try:
            trav = _traversal(scale, int(os.environ.get("CUGRAPH_B200_BENCH_BFS_SOURCES", "64")),
                              int(os.environ.get("CUGRAPH_B200_BENCH_SSSP_SOURCES", "8")))
        except Exception as ex:  # the PageRank line must survive a failure here
            trav = {"traversal_error": f"{type(ex).__name__}: {ex}"[:300]}
        torch.cuda.empty_cache()

    try:
        if big:
            raise RuntimeError("skipped in the scale-27 denominator run")
        cpu = _cpu_baseline(sample_scale=args.cpu_sample_scale)
    except Exception as ex:  # the GPU measurements above must still be reported
        cpu = {"value": None, "unit": "MTEPS", "cores": None, "kind": "port", "error": f"{type(ex).__name__}: {ex}"[:300]}
    config = {"workload": f"pagerank_rmat{scale}_ef16_100it", "scale": scale, "edge_factor": 16,
              "num_vertices": nv, "num_edges": E, "alpha": ALPHA, "iterations": ITERS, "vertex_type": "int32",
              "l2": "inputs (1.2 GB/sweep) exceed the 126 MB L2; no explicit flush"}
    config.update(trav)
    config["networkx_mteps"] = cpu.get("networkx_mteps")
    out = {"metric": metric_name(scale), "value": value, "unit": "MTEPS", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
           "data": "synthetic", "config": config,
           "timing": {"device_ms_per_step": dev_s / args.steps * 1e3, "wall_ms_per_step": wall / args.steps * 1e3,
                      "value_from": "device events" if events_ok else "wall clock (events disagreed)",
                      "how": "CUDA events recorded on the handle's stream around the K synchronous C-ABI calls"},
           "clocks": clocks, "e2e": e2e, "gpu_launches": launches, "roofline": roofline, "cpu_baseline": cpu}
    print(json.dumps(out), flush=True)


DUMP_SAMPLE = 1 << 20


def dump_pagerank(out_dir, verts, scores):
    """The result of the last timed step, as its caller receives it (vertex ids, PageRank scores), sorted by vertex id so
    that two builds that order their result rows differently compare row for row.  Above DUMP_SAMPLE vertices a fixed,
    seeded sample of the sorted rows is written (8 + 4 bytes per row: at most 12 MB)."""
    import numpy as np
    import torch
    order = torch.argsort(verts)
    vs, ps = verts[order], scores[order]
    if vs.numel() > DUMP_SAMPLE:
        keep = np.sort(np.random.default_rng(0).choice(vs.numel(), DUMP_SAMPLE, replace=False))
        idx = torch.as_tensor(keep, device=vs.device)
        vs, ps = vs[idx], ps[idx]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pagerank_vertices.npy"), vs.cpu().numpy().astype(np.float64))
    np.save(os.path.join(out_dir, "pagerank_scores.npy"), ps.cpu().numpy().astype(np.float32))


def _harmonic(xs):
    return len(xs) / sum(1.0 / x for x in xs) if xs else None


def _traversal(scale, n_bfs, n_sssp):
    """BASELINE.json configs[2] and [3] on the symmetrised RMAT graph (weights U[0,1) for SSSP, symmetric): one warm-up +
    n timed random sources each (Graph500 protocol, mg_graph500_bfs_test.cu:113-114, 757-764).  TEPS per source = undirected
    edges of the source's component / time of the C-ABI call (wall clock, device synchronised on both sides, view creation
    and result read-back outside).  Returns FLAT keys (they go into `config`, which the driver keeps)."""
    import torch
    from cugraph_b200 import _capi
    from cugraph_b200 import pylibcugraph as plc
    from cugraph_b200.generators import rmat_edgelist
    from cugraph_b200.pylibcugraph.utils import View
    L = _capi.lib()
    V = 1 << scale
    src, dst = rmat_edgelist(scale, 16 << scale, seed=0)
    s2, d2 = torch.cat([src, dst]), torch.cat([dst, src])
    del src, dst
    g = torch.Generator(device="cuda")
    g.manual_seed(2)
    w = torch.rand(s2.numel() // 2, device="cuda", generator=g)
    w2 = torch.cat([w, w])
    del w
    h = plc.ResourceHandle()
    G = plc.SGGraph(h, plc.GraphProperties(is_symmetric=True, is_multigraph=True), s2, d2, weight_array=w2,
                    store_transposed=False, renumber=True)
    deg = torch.bincount(s2.long(), minlength=V)
    e_sym = int(s2.numel())
    del s2, d2, w2
    cand = torch.nonzero(deg > 0).flatten()
    torch.manual_seed(1)
    sources = cand[torch.randperm(cand.numel(), device="cuda")[:max(n_bfs, n_sssp) + 1]].to(torch.int32)
    out = {"traversal_graph": f"RMAT-{scale} ef-16 symmetrised, {e_sym} directed edges, weights U[0,1) symmetric"}
    INT_MAX, FLT_MAX = 2**31 - 1, 3.0e38

    def c_call(name, s_t):
        res, err = C.c_void_p(), C.c_void_p()
        if name == "bfs":
            sv = View(s_t)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            code = L.cugraph_bfs(h.ptr, G.ptr, sv.ptr, 1, INT_MAX - 1, 1, 0, C.byref(res), C.byref(err))
            dt = time.perf_counter() - t0      # the C-ABI call is synchronous: the result is complete on return
            sv.free()
        else:
            s_host = int(s_t.item())
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            code = L.cugraph_sssp(h.ptr, G.ptr, s_host, float("inf"), 1, 0, C.byref(res), C.byref(err))
            dt = time.perf_counter() - t0
        _capi.check(code, err, f"cugraph_{name}")
        from cugraph_b200.pylibcugraph.utils import copy_to_torch
        verts = copy_to_torch(h, L.cugraph_paths_result_get_vertices(res))
        dist = copy_to_torch(h, L.cugraph_paths_result_get_distances(res))
        pred = copy_to_torch(h, L.cugraph_paths_result_get_predecessors(res))
        L.cugraph_paths_result_free(res)
        return dt, verts, dist, pred

    ok_all = True
    for name, n in (("bfs", n_bfs), ("sssp", n_sssp)):
        teps, ms = [], []
        for i in range(n + 1):  # source 0 is the warm-up (and the checked one)
            s_t = sources[i:i + 1].contiguous()
            dt, verts, dist, pred = c_call(name, s_t)
            reached = (dist != INT_MAX) if name == "bfs" else (dist < FLT_MAX)
            ne = int(deg[verts.long()][reached].sum().item()) // 2
            if i == 0:  # size-independent properties of the full-size result (external ids)
                d_ext = torch.empty(V, dtype=dist.dtype, device="cuda")
                d_ext[verts.long()] = dist
                has_pred = pred >= 0
                dp, dv = d_ext[pred[has_pred].long()], dist[has_pred]
                ok = bool(((dp + 1 == dv) if name == "bfs" else (dp <= dv)).all().item())
                ok = ok and bool((d_ext[int(s_t.item())] == 0).item())
                ok = ok and int(has_pred.sum().item()) == int(reached.sum().item()) - 1
                ok_all = ok_all and ok
            else:
                teps.append(ne / dt)
                ms.append(dt * 1e3)
        out[f"{name}_sources"] = n
        out[f"{name}_harmonic_mteps"] = _harmonic(teps) / 1e6 if teps else None
        out[f"{name}_mean_mteps"] = sum(teps) / len(teps) / 1e6 if teps else None
        out[f"{name}_ms_per_source"] = sum(ms) / len(ms) if ms else None
        out[f"{name}_ms_min_max"] = [min(ms), max(ms)] if ms else None
    out["traversal_checks_ok"] = ok_all
    out["traversal_timing"] = "wall clock around the synchronous C-ABI call (cugraph_bfs / cugraph_sssp), device synchronised before"
    return out


def run_multi(args):
    from cugraph_b200.mg_bench import run_mg_pagerank
    run_mg_pagerank(args, metric_name, ALPHA, ITERS, ClockSampler, _peaks)


def _protect_stdout():
    """Libraries (NCCL's version banner, torchrun children) write to fd 1; the contract is ONE JSON line on
    stdout.  Route fd 1 to stderr for the run and keep the real stdout for the final line."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w", buffering=1)


def main():
    _protect_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--scale", type=int, default=None, help="override RMAT scale (development only)")
    ap.add_argument("--cpu-sample-scale", type=int, default=22, help="RMAT scale of the cpu_baseline sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the vertices and scores of the last timed step to DIR/*.npy (single GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl in ("reference", "cpu-sample"):
        pin_host_threads()  # before numpy / the oracle load an OpenMP runtime; ONLY in the CPU arms (see _cpu_baseline)
        return run_reference(args) if args.impl == "reference" else run_cpu_sample(args)
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 or world > 1:
        if args.dump_outputs:
            ap.error("--dump-outputs is implemented for --gpus 1")
        return run_multi(args)  # weak scaling: scale 24 + log2(N); N = 8 is BASELINE's scale-27 configuration
    if args.scale is None:
        args.scale = 24
    return run_single(args)


if __name__ == "__main__":
    main()
