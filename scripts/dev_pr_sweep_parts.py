"""dev (GPU): where the PageRank sweep at RMAT scale 24 ef16 spends its time.

    python scripts/dev_pr_sweep_parts.py [reps]

ms per sweep from the library's CUDA events over `reps` runs of 20 sweeps (median, min, max), then one torch.profiler run (CUDA
activities) of 2 x 20 sweeps with every kernel's mean duration per sweep (the passes run one after another on one stream, so
each duration is the time of that pass by itself). VGLB_PR_TRACE=1 is set for the first run, so the library prints each
kernel's resident CTAs per SM before and after it sets the shared-memory carve-outs. With VGLB_LIB_PATH it times a developer
A/B build (scripts/dev_build_variant.sh); the kernels a build does not have (pr_finish_kernel ran as a pass of its own until
pr_sweep_kernel<false> took its blocks) are left out of the per-kernel line."""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

import vectorgraphlibrary_b200 as vgl

KERNELS = ["pr_bin_kernel", "pr_cold_bin_kernel", "pr_sweep_kernel", "pr_finish_kernel"]  # the passes of a sweep, in order
ITERS = 20
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 7

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"GPU: {gpu[0] if gpu else 'unknown'}", flush=True)
torch.cuda.init()
with vgl.Context(0) as ctx:
    dsrc, ddst = ctx.generate_edges(vgl.GEN_RMAT, 24, 16)
    g = vgl.Graph.from_edges(ctx, 1 << 24, dsrc, ddst, 0)
    out = ctx.empty(g.V, np.float32)
    print(f"RMAT s24 ef16: V={g.V} E={g.E}, {ITERS} sweeps per run", flush=True)
    os.environ["VGLB_PR_TRACE"] = "1"
    g.pagerank(ITERS, 0.85, out)  # module load, bins build
    os.environ.pop("VGLB_PR_TRACE", None)
    t = []
    for r in range(reps):
        _, st = g.pagerank(ITERS, 0.85, out)
        t.append(st.seconds * 1e3 / ITERS)
    med = statistics.median(t)
    print(f"ms per sweep: median {med:.4f}  min {min(t):.4f}  max {max(t):.4f}  ({reps} runs; {g.E / med / 1e6:.1f} GTEPS at the median)",
          flush=True)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(2):
            g.pagerank(ITERS, 0.85, out)
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        for k in KERNELS:
            if e.key.split("(")[0].split(" ")[-1].split("<")[0] == k:
                per[k] = per.get(k, 0.0) + e.device_time_total
    sweeps = 2 * ITERS
    parts = "  ".join(f"{k} {per[k] / sweeps:.1f}" for k in KERNELS if k in per)
    print(f"us per sweep per kernel (torch.profiler): {parts}  sum {sum(per.values()) / sweeps:.1f}", flush=True)
    out.free()
    g.free()
