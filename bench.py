#!/usr/bin/env python
"""bench.py — benchmark of the B200 backend for VGL's frontier-processing hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload pr|bfs|sssp|cc|bfs20|config5] [--scaling weak|strong] [--no-extras] [--dump-outputs DIR]

Headline (default) = BASELINE.json configs[1]: PageRank pull, 20 iterations fp32, RMAT scale-24 edge-factor 16 on one
B200; a "step" is one complete PageRank run (20 sweeps) over the resident graph. Metric = GTEPS in the reference's
convention: iterations x graph edges / time / 1e9 (performance_stats.hpp:272-275, pr.hpp:147).

  value        device-timed (CUDA events on the library's stream), graph resident in HBM, max over ranks
  e2e          the same metric through the C ABI with HOST buffers: every step copies the VectCSR arrays the reference
               host build owns (row pointers, adjacency, id map; pinned memory) to HBM (vglb_graph_from_csr =
               VGL_Graph::move_to_device; the host announces PageRank with vglb_set_upload_hint), runs the algorithm, reorders the
               result to the caller's ORIGINAL numbering on the device (N = 1) and copies it back
  roofline     dominant kernel(s) (PageRank: the four kernels of one sweep): algorithmic bytes per launch (SURVEY §8d formulas evaluated with the library's counters) /
               average launch duration, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline the reference's own multicore (OpenMP) implementation (oracle/_ref: unmodified VGL, timing build) on this
               box's host cores, on the SAME graph when it fits the time budget (configs 1 and 2 do), else a bounded sample
  parity_check every rank runs the four algorithms on the golden fixtures (outputs of the unmodified reference,
               tests/golden/) through the same (partitioned, at N > 1) code path before anything is timed
  extras.workloads   after the headline, outside its timed region: the other BASELINE configs with the same measurements —
               bfs (config 4: DO-BFS Kronecker s26 ef16), sssp (config 3: uniform s24 ef32), cc (RMAT s24 ef16 symmetrised),
               bfs20 (config 1: BFS RMAT s20 ef16, N = 1, with the CPU reference on the same graph and sources);
               at N > 1 also bfs_strong (config 4 strong scaling: the same s26 graph at every N); config 5 (CC + PageRank on
               RMAT scale-28 ef16, 8 GPUs) is `--workload config5`

`--impl reference` times the reference's CPU path alone (same metric / config / unit). Under torchrun (N > 1) every rank
owns a 1D vertex range of the graph (DESIGN.md §5); `--scaling strong` keeps the graph fixed as N grows.

`--dump-outputs DIR` writes what the headline's last timed step computed, in ORIGINAL vertex numbering, to DIR/<name>.npy
(PageRank ranks and SSSP distances as float32, BFS levels and CC labels as float64). An output larger than 64 MB is
written at 2^22 seeded positions (sorted; the same positions for the same vertex count). The graph, the sources and the
sample depend only on the arguments, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "GTEPS"
WORKLOADS = {
    # name: (generator kind, scale, edge factor, description)   — BASELINE.json configs
    "pr": (0, 24, 16, "PageRank pull, 20 iters fp32, RMAT scale-24 ef16"),                                # configs[1]
    "sssp": (2, 24, 32, "SSSP frontier Bellman-Ford, fp32 weights, uniform-random scale-24 ef32"),         # configs[2]
    "bfs": (1, 26, 16, "Direction-optimising BFS, Graph500 Kronecker scale-26 ef16"),                     # configs[3]
    "cc": (0, 24, 16, "CC min-label hook + jump, RMAT scale-24 ef16 symmetrised"),                        # one GPU's share of configs[4]
    "bfs20": (0, 20, 16, "BFS, RMAT scale-20 ef16"),                                                      # configs[0]
}
PR_ITERS = 20
GOLDEN = ("rmat_s8_ef4", "kron_s10_ef16", "ru_s10_ef32", "rmat_s11_ef8")
OUTPUT_NAMES = {"pr": "pagerank_ranks", "bfs": "bfs_levels", "sssp": "sssp_distances", "cc": "cc_labels"}
DUMP_BUDGET_BYTES = 64 * 10 ** 6
DUMP_SAMPLE = 1 << 22
T0 = time.perf_counter()


def algo_of(workload: str) -> str:
    return "bfs" if workload == "bfs20" else workload


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def ncu_traffic(workload: str, world: int):
    """DRAM bytes (read + write) of one launch of the dominant kernel from the committed `ncu --set full` summary of the
    same command (profiles/, B200_PROFILING.md recipe); None where no capture of the configuration exists."""
    if world != 1:
        return None
    names = {"pr": ["r2_pr_sweep_ncu_full.txt"]}.get(workload, [])  # (first line of that kind = the four kernels of a sweep together)
    for name in names:
        try:
            for line in open(os.path.join(ROOT, "profiles", name)):
                if line.strip().startswith("traffic (dram read + write) bytes:"):
                    return int(line.split(":")[1])
        except OSError:
            continue
    return None


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
        except Exception:
            pass
    return 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def workload_config(workload: str, scale: int, world: int, weak: bool):
    """The `config` object both arms print for a workload: the same dict for the repo arm and the reference arm."""
    kind, base_scale, ef, desc = WORKLOADS[workload]
    total_scale = scale + (int(np.log2(world)) if (weak and world > 1) else 0)
    name = desc.replace(f"scale-{base_scale}", f"scale-{total_scale}")
    if world > 1:
        name += (f" (weak scaling: scale-{scale} per GPU x {world} GPUs)" if weak else f" (strong scaling: the same graph on {world} GPUs)")
    V = 1 << total_scale
    E = (ef << total_scale) * (2 if algo_of(workload) == "cc" else 1)
    adj_gb = 4 * E / world / 1e9
    return {"workload": name, "vertices": V, "edges": E, "iterations_per_step": PR_ITERS if workload == "pr" else 1,
            "l2": (("L2 flushed before every timed step (adjacency %.2f GB per GPU < 2 x L2)" if adj_gb < 0.252 else
                    "inputs larger than L2 (adjacency %.2f GB per GPU, L2 126 MB)") % adj_gb), "seed": hex(0xB200)}


# ---------------------------------------------------------------------------------------------------------------------
# reference arm / cpu baseline: the unmodified reference (oracle/_ref) or, where it is not built, the C oracle port.
# The only place where bench.py executes anything under oracle/.
# ---------------------------------------------------------------------------------------------------------------------

def cpu_reference_run(workload: str, sample_scale: int, steps: int, warmup: int, budget_s: float = 240.0):
    """Times the reference's own CPU implementation of `workload` at `sample_scale`. Returns (gteps, info dict)."""
    threads = max(2, host_threads())  # the reference segfaults with one OpenMP thread (SURVEY App. A.1)
    os.environ["OMP_NUM_THREADS"] = str(threads)
    os.environ.setdefault("OMP_PROC_BIND", "close")
    import oracle as O
    algo = algo_of(workload)
    kind, config_scale, ef, _ = WORKLOADS[workload]
    V = 1 << sample_scale
    t_setup = time.perf_counter()
    src, dst = O.generate_edges(kind, sample_scale, ef)
    if algo == "cc":
        src, dst = O.symmetrize(src, dst)
    E = len(src)
    outdeg = np.bincount(src, minlength=V)
    sources = O.pick_sources(V, outdeg, max(1, steps + warmup))
    times = []
    timing = O.ref_available(algo, timing=True)
    if O.ref_available(algo, timing=timing):
        kind_s = "reference"
        build = ("timing build: -O3 -march=x86-64-v3 -ffast-math -funroll-loops -ftree-vectorize" if timing else "parity build: -O2")
        rg = O.RefGraph(V, src, dst, algo, timing=timing)
        del src, dst
        t_setup = time.perf_counter() - t_setup
        t_loop = time.perf_counter()
        for i in range(warmup + steps):
            if algo == "pr":
                _, t = rg.pagerank(PR_ITERS)
            elif algo == "bfs":
                _, t = rg.bfs(sources[i], 0)
            elif algo == "sssp":
                _, t = rg.sssp(sources[i], O.MASTER_SEED ^ 0x5555, 2)  # PARTIAL_ACTIVE PUSH (timing only: racy)
            else:
                _, t = rg.cc()
            if i >= warmup:
                times.append(t)
            if len(times) >= 2 and time.perf_counter() - t_loop > budget_s:  # bounded: stop once the budget is spent
                break
        rg.close()
    else:
        kind_s, build = "port", "C restatement, -O2"
        og = O.OracleGraph(V, src, dst)
        t_setup = time.perf_counter() - t_setup
        t_loop = time.perf_counter()
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            if algo == "pr":
                og.pagerank_f32(PR_ITERS, threads)
            elif algo == "bfs":
                og.bfs(sources[i])
            elif algo == "sssp":
                og.sssp_frontier_bf(sources[i], O.MASTER_SEED ^ 0x5555)
            else:
                og.cc()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
            if len(times) >= 2 and time.perf_counter() - t_loop > budget_s:
                break
    mult = PR_ITERS if algo == "pr" else 1
    t_mean = float(np.mean(times))
    gteps = mult * E / t_mean / 1e9
    gen = {0: "RMAT", 1: "Kronecker", 2: "uniform-random"}[kind]
    same = sample_scale == config_scale
    info = {"value": gteps, "unit": METRIC, "cores": threads, "kind": kind_s,
            "sample": ("the whole workload: " if same else "bounded sample: ") + f"{gen} scale-{sample_scale} ef{ef}"
                      + (" symmetrised" if algo == "cc" else "")
                      + (f", {PR_ITERS} iterations" if algo == "pr" else ", one seeded source per run" if algo != "cc" else "")
                      + f", {len(times)} timed runs, VGL multicore (OpenMP), {build}",
            "same_config": same, "seconds_per_run": t_mean, "setup_seconds": t_setup,
            "min_max_gteps": [mult * E / max(times) / 1e9, mult * E / min(times) / 1e9]}
    return gteps, info


def cpu_scale_for(workload: str, requested: int) -> int:
    """Scale of the CPU arm's graph: the workload's own scale when the reference can import it within the time budget
    (import is minutes beyond scale 24; E must stay below 2^31: SURVEY App. A.5), else the largest that does."""
    if requested:
        return requested
    _, scale, ef, _ = WORKLOADS[workload]
    cap = {"pr": 24, "bfs20": 20, "bfs": 23, "sssp": 22, "cc": 22}[workload]
    return min(scale, cap)


def reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    workload = "pr" if args.workload == "config5" else args.workload
    _, scale, _, _ = WORKLOADS[workload]
    weak = args.scaling == "weak"
    t0 = time.perf_counter()
    sample_scale = cpu_scale_for(workload, args.cpu_scale)
    gteps, info = cpu_reference_run(workload, sample_scale, args.steps, args.warmup)
    cfg = workload_config(workload, scale, args.gpus, weak)
    info["same_config"] = bool(info["same_config"] and args.gpus == 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": gteps, "unit": METRIC, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": info["seconds_per_run"] * 1e3, "higher_is_better": True,
        "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f32" if workload in ("pr", "sssp") else "int32",
        "data": "synthetic", "config": cfg, "cpu_baseline": info,
        "e2e": {"value": gteps, "unit": METRIC, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)
    return 0


# ---------------------------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------------------------

class Bench:
    def __init__(self, args):
        import torch
        import vectorgraphlibrary_b200 as vgl
        from vectorgraphlibrary_b200 import dist as vdist
        self.torch, self.vgl, self.vdist, self.args = torch, vgl, vdist, args
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if self.world != args.gpus:
            raise SystemExit(f"bench.py --gpus {args.gpus} but WORLD_SIZE={self.world}: launch with torchrun --nproc-per-node {args.gpus}")
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; libvgl_b200 has no CPU fallback (use --impl reference for the CPU arm)")
        torch.cuda.set_device(self.local_rank)
        self.tcomm = vdist.Communicator.from_env(self.local_rank) if self.world > 1 else None
        self.ctx = vgl.Context(self.local_rank)
        # one NCCL communicator of the library for the whole process (every partitioned graph of this run uses it)
        self.vcomm = None
        if self.world > 1:
            self.vcomm = vgl.Comm(self.ctx, self.rank, self.world,
                                  exchange=lambda b: self.tcomm.broadcast_bytes(b, vgl.UNIQUE_ID_BYTES, 0))
        self.peak, self.peak_src = measured_peak()
        self.stream = torch.cuda.ExternalStream(self.ctx.stream, device=self.local_rank)

    def barrier(self):
        if self.tcomm is not None:
            self.tcomm.barrier()
        self.ctx.synchronize()
        self.torch.cuda.synchronize()

    def max_float(self, x):
        return self.tcomm.max_float(x) if self.tcomm is not None else x

    # ---- pre-timing correctness gate (golden fixtures = outputs of the unmodified reference) ----
    def parity_check(self):
        vgl, ctx = self.vgl, self.ctx
        t0 = time.perf_counter()
        checked, failures = 0, []
        for name in GOLDEN:
            g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
            src, dst = vgl.generate_edges_host(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))
            V = 1 << int(g["scale"])
            if self.world > 1:
                G = vgl.Graph.from_edges_partitioned(ctx, self.vcomm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
            else:
                G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
            fwd = G.orig_to_sorted()

            def check(what, ok):
                nonlocal checked
                checked += 1
                if not ok:
                    failures.append(f"{name}:{what}")

            for i, s in enumerate(g["sources"]):
                for dopt in (False, True):
                    lv, _ = G.bfs(int(fwd[int(s)]), direction_optimising=dopt)
                    check(f"bfs[{i}]{'do' if dopt else 'td'}", np.array_equal(G.to_original(lv), g["bfs_levels"][i]))
                    lv.free()
            w = G.synthetic_weights(int(g["weight_seed"]))
            for i, s in enumerate(g["sources"]):
                d, _ = G.sssp(w, int(fwd[int(s)]))
                check(f"sssp[{i}]", np.array_equal(G.to_original(d).view(np.uint32), g["sssp_dist"][i].view(np.uint32)))
                d.free()
            w.free()
            lab, _ = G.cc()
            check("cc", np.array_equal(G.to_original(lab), g["cc_directed"]))
            lab.free()
            if self.world == 1:  # the contract number: reference-order dangling sum at the fixture's thread count
                ranks, _ = G.pagerank(int(g["pr_iters"]), reference_threads=int(g["pr_threads"]))
            else:
                ranks, _ = G.pagerank(int(g["pr_iters"]))
            r, ref = G.to_original(ranks).astype(np.float64), g["pr_ranks"].astype(np.float64)
            check("pagerank<=1e-6", float(np.abs(r - ref).sum() / np.abs(ref).sum()) <= 1e-6)
            ranks.free()
            G.free()
        bad = len(failures)
        if self.tcomm is not None:
            bad = self.tcomm.sum_int(bad)
        return {"status": "ok" if bad == 0 else "FAILED", "checks_per_rank": checked, "ranks": self.world,
                "failed_checks_all_ranks": bad, "failures_rank0": failures[:8],
                "what": "BFS (TD + DO) levels, SSSP distances, CC labels bit-exact and PageRank <= 1e-6 rel. L1 against tests/golden/ "
                        "(outputs of the unmodified reference), on every rank through the " + ("partitioned" if self.world > 1 else "single-GPU") + " path",
                "seconds": time.perf_counter() - t0}

    def dump_outputs(self, runner, algo, out_dir):
        """--dump-outputs: the result array of the runner's last step in ORIGINAL numbering -> out_dir/<name>.npy.
        Collective on a partitioned graph (every rank takes part in the reorder); rank 0 writes."""
        full = runner.g.to_original(runner.out)
        if self.rank != 0:
            return None
        dtype = np.dtype(np.float32 if full.dtype == np.float32 else np.float64)  # int32 labels / levels stay exact
        sampled = full.size * dtype.itemsize > DUMP_BUDGET_BYTES
        if sampled:
            full = full[np.sort(np.random.default_rng(self.vgl.MASTER_SEED).choice(full.size, DUMP_SAMPLE, replace=False))]
        os.makedirs(out_dir, exist_ok=True)
        name = OUTPUT_NAMES[algo]
        np.save(os.path.join(out_dir, name + ".npy"), full.astype(dtype))
        return {name: {"dtype": dtype.name, "values": int(full.size), "sampled": sampled}}

    # ---- one workload: device-timed value, roofline, e2e ----
    def run_workload(self, workload, scale, steps, warmup, weak=True, sample_clocks=False, e2e_steps=None, td_only=False,
                     dump_dir=None):
        vgl, ctx, torch = self.vgl, self.ctx, self.torch
        kind, _, ef, _ = WORKLOADS[workload]
        algo = algo_of(workload)
        runner = self.vdist.make_runner(vgl, ctx, self.tcomm, algo, kind, scale, ef, PR_ITERS, weak=weak, vcomm=self.vcomm)
        if td_only:
            runner.bfs_direction_optimising = False
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(warmup):
            runner.step(i)
        self.barrier()
        sampler = ClockSampler(self.local_rank) if (sample_clocks and self.rank == 0) else None
        if sampler:
            sampler.start()
        stats = []
        # timing rule: inputs larger than L2, or L2 flushed between timed iterations. Small graphs (config 1: 67 MB of
        # adjacency < 126 MB L2) get a flush before every step and are timed by the library's own per-call CUDA events
        # (the flush kernel stays outside the timed intervals)
        flush = runner.adj_bytes_per_gpu < 2 * 126e6
        ev0.record(self.stream)
        for i in range(steps):
            if flush:
                ctx.flush_l2()
            stats.append(runner.step(warmup + i))
        ev1.record(self.stream)
        self.barrier()
        clocks = sampler.stop() if sampler else None
        if flush:
            ms_per_step = self.max_float(float(np.mean([s["seconds"] for s in stats])) * 1e3)
        else:
            ms_per_step = self.max_float(ev0.elapsed_time(ev1)) / steps
        dumped = self.dump_outputs(runner, algo, dump_dir) if dump_dir else None
        edges_per_step = runner.edges_per_step  # whole job, all ranks
        value = edges_per_step / (ms_per_step * 1e-3) / 1e9
        # dominant kernel(s): duration from the library's own CUDA events around the algorithm loop
        kern_s = float(np.mean([s["seconds"] / max(1, s["dominant_launches"]) for s in stats]))
        kern_bytes = float(np.mean([s["dominant_bytes"] / max(1, s["dominant_launches"]) for s in stats]))
        achieved = kern_bytes / kern_s / 1e9
        e2e = runner.e2e(e2e_steps if e2e_steps is not None else max(2, min(steps, 5)))
        e2e["seconds"] = self.max_float(e2e["seconds"])
        cfg = workload_config(workload, scale, self.world, weak)
        cfg["vertices"], cfg["edges"] = runner.V_total, runner.E_total
        cfg["l2"] = (("L2 flushed before every timed step (adjacency %.2f GB per GPU < 2 x L2)" if flush else
                      "inputs larger than L2 (adjacency %.2f GB per GPU, L2 126 MB)") % (runner.adj_bytes_per_gpu / 1e9))
        res = {
            "value": value, "unit": METRIC, "ms_per_step": ms_per_step, "steps": steps, "warmup": warmup,
            "scaling": ("weak" if weak else "strong") if self.world > 1 else "weak",
            "dtype": runner.dtype, "config": cfg, "partition": runner.partition,
            "roofline": {"bound": "hbm", "kernel": runner.dominant_kernel, "achieved": achieved, "peak": self.peak, "unit": "GB/s",
                         "frac": achieved / self.peak, "traffic": ncu_traffic(workload, self.world) if scale == WORKLOADS[workload][1] else None,
                         "traffic_source": "profiles/r2_pr_sweep_ncu_full.txt: dram__bytes_read + dram__bytes_write of the four kernels of one sweep, "
                                           "one `ncu --set full` capture of this command (committed; not re-measured in this run)"
                         if workload == "pr" and self.world == 1 and scale == WORKLOADS[workload][1] else None,
                         "peak_source": self.peak_src, "bytes_per_launch": kern_bytes, "ms_per_launch": kern_s * 1e3},
            "e2e": {"value": edges_per_step / e2e["seconds"] / 1e9, "unit": METRIC, "h2d_bytes_per_step": e2e["h2d"],
                    "d2h_bytes_per_step": e2e["d2h"], "ms_per_step": e2e["seconds"] * 1e3},
            "gpu_launches": int(sum(s["kernel_launches"] for s in stats)),
            # the reference's own "total bandwidth" line: edges x INT_ELEMENTS_PER_EDGE x 4 bytes / time
            # (apps/bfs/bfs.cpp:3 -> 16 B per edge, apps/pr/pr.cpp:3 etc. -> 20 B; performance_stats.hpp:272-275)
            "reference_accounting_gbs": edges_per_step * (16 if algo == "bfs" else 20) / (ms_per_step * 1e-3) / 1e9,
            # BFS / SSSP: one seeded source per step (SURVEY §8d); `value` = edges / mean time over the timed sources (events around
            # the whole loop, host gaps included); min / max come from the library's per-call device timers
            "per_source_gteps": ({"min": edges_per_step / max(s["seconds"] for s in stats) / 1e9,
                                  "max": edges_per_step / min(s["seconds"] for s in stats) / 1e9, "sources": len(stats)}
                                 if algo in ("bfs", "sssp") else None),
            "iterations_per_run": float(np.mean([s["iterations"] for s in stats])),
            "edges_inspected_per_run": float(np.mean([s["edges_inspected"] for s in stats])),
            "runner_extras": runner.extras(),
        }
        if clocks is not None:
            res["clocks"] = clocks
        if dumped is not None:
            res["dumped_outputs"] = dumped
        runner.close()
        return res


def compact(res):
    """What an extras.workloads entry carries."""
    keep = ("value", "unit", "ms_per_step", "steps", "warmup", "scaling", "dtype", "config", "roofline", "e2e", "gpu_launches",
            "per_source_gteps", "iterations_per_run", "edges_inspected_per_run", "cpu_baseline", "top_down_only")
    return {k: res[k] for k in keep if k in res}


def ours(args):
    B = Bench(args)
    rank, world = B.rank, B.world
    weak = args.scaling == "weak"
    line_holder = {}

    def emit_and_exit(note):
        """Watchdog: extras must never cost the headline its line. Prints what there is and leaves."""
        if rank == 0 and "line" in line_holder and not line_holder.get("printed"):
            line_holder["line"]["extras"]["note"] = note
            print(json.dumps(line_holder["line"]), flush=True)
        os._exit(0)

    parity = B.parity_check()
    if parity["status"] != "ok":
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": None, "unit": METRIC, "n_gpus": world, "parity_check": parity,
                              "error": "parity gate failed: nothing was timed"}), flush=True)
        return 1

    config5 = args.workload == "config5"
    headline = "pr" if config5 else args.workload
    scale = args.scale or (28 if config5 else WORKLOADS[headline][1])
    head_weak = weak and not config5
    res = B.run_workload(headline, scale, args.steps, args.warmup, weak=head_weak, sample_clocks=True, td_only=args.top_down_only,
                         dump_dir=args.dump_outputs)

    line = None
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:  # the CPU baseline is reported at N = 1 only
            try:
                _, cpu = cpu_reference_run(headline, cpu_scale_for(headline, args.cpu_scale), 3, 1, budget_s=60.0)
            except Exception as ex:  # the checker must not take the product's number down with it
                cpu = {"value": None, "unit": METRIC, "cores": host_threads(), "kind": "unavailable", "sample": repr(ex)}
        line = {
            "metric": METRIC, "value": res["value"], "unit": METRIC, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": res["ms_per_step"], "higher_is_better": True, "scaling": res["scaling"], "vs_baseline": None,
            "dtype": res["dtype"], "data": "synthetic", "config": res["config"], "partition": res["partition"],
            "roofline": res["roofline"], "cpu_baseline": cpu, "e2e": res["e2e"], "gpu_launches": res["gpu_launches"],
            "clocks": res.get("clocks"), "reference_accounting_gbs": res["reference_accounting_gbs"],
            "per_source_gteps": res["per_source_gteps"], "parity_check": parity,
            "extras": {"workloads": {}, "runner": res["runner_extras"]},
        }
        if "dumped_outputs" in res:
            line["dumped_outputs"] = {"dir": os.path.abspath(args.dump_outputs), "files": res["dumped_outputs"]}
        line_holder["line"] = line

    # ---- the other BASELINE configs, after (and outside) the headline's timed region ----
    if not args.no_extras and (args.workload == "pr" or config5) and not args.scale:
        deadline = T0 + args.extras_budget
        watchdog = threading.Timer(max(1.0, deadline + 240.0 - time.perf_counter()), emit_and_exit,
                                   args=("extras stopped by the watchdog (a workload overran its budget)",))
        watchdog.daemon = True
        watchdog.start()
        plan = []
        if config5:
            plan.append(("cc_s28", "cc", 28, False, 3, False))
        else:
            plan += [("bfs", "bfs", WORKLOADS["bfs"][1], weak, 16, False), ("sssp", "sssp", WORKLOADS["sssp"][1], weak, 16, False),
                     ("cc", "cc", WORKLOADS["cc"][1], weak, 5, False)]
            if world == 1:
                plan.append(("bfs20", "bfs20", 20, True, 16, False))
                plan.append(("bfs20_top_down", "bfs20", 20, True, 16, True))
            else:
                plan.append(("bfs_strong", "bfs", WORKLOADS["bfs"][1], False, 16, False))
            # (config 5 — CC + PageRank on RMAT scale-28, 8 GPUs — is `--workload config5`: 4.3 G edges take minutes to
            # generate and partition, too long for the default line)
        for key, wl, sc, wk, steps, td_only in plan:
            # every rank takes the same decision (the clock of rank 0 is broadcast through the max)
            over = B.max_float(1.0 if time.perf_counter() > deadline else 0.0) > 0.0
            if over:
                if rank == 0:
                    line["extras"]["workloads"][key] = {"skipped": "time budget of the default run spent"}
                continue
            try:
                r = B.run_workload(wl, sc, steps, 3, weak=wk, e2e_steps=2, td_only=td_only)
                if td_only:
                    r["top_down_only"] = True
                if rank == 0 and world == 1 and wl == "bfs20" and not args.no_cpu_baseline and not td_only:
                    # config 1 fits both arms at full size: same graph, same seeded sources, the reference's own top-down BFS
                    try:
                        _, r["cpu_baseline"] = cpu_reference_run("bfs20", 20, 16, 2, budget_s=30.0)
                    except Exception as ex:
                        r["cpu_baseline"] = {"value": None, "kind": "unavailable", "sample": repr(ex)}
                if rank == 0:
                    line["extras"]["workloads"][key] = compact(r)
            except Exception as ex:
                if world > 1:
                    raise  # ranks must not diverge inside collectives
                line["extras"]["workloads"][key] = {"error": repr(ex)}
        watchdog.cancel()

    if rank == 0:
        line["wall_s"] = time.perf_counter() - T0
        print(json.dumps(line), flush=True)
        line_holder["printed"] = True
    if B.vcomm is not None:
        B.vcomm.close()
    if B.tcomm is not None:
        B.tcomm.close()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pr", choices=sorted(WORKLOADS) + ["config5"])
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = scale + log2 N (per-GPU work fixed); strong = the same graph at every N")
    ap.add_argument("--scale", type=int, default=0, help="override the workload's scale (parity/dev runs only)")
    ap.add_argument("--cpu-scale", type=int, default=0, help="scale of the CPU arm's graph (default: the workload's own where it fits)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="headline only (profiling runs)")
    ap.add_argument("--top-down-only", action="store_true", help="BFS workloads: no direction switch (the reference's BFS::vgl_top_down)")
    ap.add_argument("--extras-budget", type=float, default=420.0, help="seconds after which no further extra workload is started")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the headline's result of its last timed step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the GPU path computed: it needs --impl ours")
    if args.warmup < 3 and args.impl == "ours":
        args.warmup = 3  # timing rule: W >= 3
    if args.impl == "reference":
        return reference_arm(args)
    return ours(args)


if __name__ == "__main__":
    sys.exit(main())
