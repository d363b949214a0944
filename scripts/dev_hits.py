"""dev (GPU): vglb_hits on one B200, with vglb_pagerank on the same graph as the yardstick (both gather one fp32 per edge).

    python scripts/dev_hits.py [reps]

Graphs: RMAT scale 24 ef16 (the gathered vectors fit the L2) and Kronecker scale 26 ef16 (they do not), 20 steps / sweeps per
call, uploaded without the incoming CSR (the warm-up call derives it). After one warm-up call of each, `reps` HITS calls and
`reps` PageRank calls alternate; times are the library's CUDA events (stats.seconds). Printed: ms per step (median, min, max),
GTEPS = steps * E / time (the reference's HITS convention), algorithmic bytes / time against the 6539 GB/s copy bandwidth
DESIGN measured, then one torch.profiler run (CUDA activities) with the mean time of each pass per step: the authority pass
pulls over the incoming CSR (rows in SCATTER order, not degree-sorted), the hub pass over the outgoing CSR (degree-sorted).
Last, the outputs of the timed calls are checked against the fp64 restatement of include/vgl_b200.h (computed with torch on
the GPU in fp64, in ORIGINAL numbering). The card's name and power limit are read in the same run."""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

import vectorgraphlibrary_b200 as vgl

STEPS = 20
COPY_GBPS = 6539.0  # DESIGN: measured device copy bandwidth of the B200
GRAPHS = [("RMAT s24 ef16", vgl.GEN_RMAT, 24, 16), ("Kronecker s26 ef16", vgl.GEN_KRONECKER, 26, 16)]
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5


def restatement(V, src, dst, steps):
    """fp64 HITS on the GPU (torch): h_0 = 1, authority step then hub step, each normalised; a zero vector stays zero."""
    h = torch.ones(V, dtype=torch.float64, device="cuda")
    a = torch.zeros_like(h)
    for _ in range(steps):
        a = torch.zeros_like(h).index_add_(0, dst, h[src])
        n = torch.linalg.vector_norm(a)
        a = a / n if n > 0 else a
        h = torch.zeros_like(a).index_add_(0, src, a[dst])
        n = torch.linalg.vector_norm(h)
        h = h / n if n > 0 else h
    return a.cpu().numpy(), h.cpu().numpy()


def rel_l1(x, ref):
    return float(np.abs(x.astype(np.float64) - ref).sum() / np.abs(ref).sum())


gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"GPU: {gpu[0] if gpu else 'unknown'}", flush=True)
torch.cuda.init()
with vgl.Context(0) as ctx:
    for name, kind, scale, ef in GRAPHS:
        V = 1 << scale
        dsrc, ddst = ctx.generate_edges(kind, scale, ef)
        g = vgl.Graph.from_edges(ctx, V, dsrc, ddst, 0)
        E = g.E
        auth, hub, ranks = ctx.empty(V, np.float32), ctx.empty(V, np.float32), ctx.empty(V, np.float32)
        g.hits(STEPS, auth, hub)        # derives the incoming CSR, module load
        g.pagerank(STEPS, 0.85, ranks)  # builds what the sweep needs
        th, tp, bytes_ = [], [], 0
        for _ in range(reps):
            _, _, st = g.hits(STEPS, auth, hub)
            th.append(st.seconds * 1e3 / STEPS)
            bytes_ = st.algorithmic_bytes
            _, st = g.pagerank(STEPS, 0.85, ranks)
            tp.append(st.seconds * 1e3 / STEPS)
        mh, mp = statistics.median(th), statistics.median(tp)
        print(f"{name}: V={V} E={E}, {STEPS} steps per call, {reps} calls each, alternated", flush=True)
        print(f"  HITS     ms per step: median {mh:.4f}  min {min(th):.4f}  max {max(th):.4f}  "
              f"{E / mh / 1e6:.2f} GTEPS  {bytes_ / (mh * 1e-3 * STEPS) / 1e9:.0f} GB/s algorithmic "
              f"({bytes_ / (mh * 1e-3 * STEPS) / 1e9 / COPY_GBPS * 100:.0f} % of {COPY_GBPS:.0f} GB/s)", flush=True)
        print(f"  PageRank ms per sweep: median {mp:.4f}  min {min(tp):.4f}  max {max(tp):.4f}  "
              f"{E / mp / 1e6:.2f} GTEPS;  HITS step / PageRank sweep = {mh / mp:.2f}", flush=True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            g.hits(STEPS, auth, hub)
            torch.cuda.synchronize()
        per = {}
        for e in prof.key_averages():
            k = e.key.split("(")[0].split(" ")[-1]
            if k.startswith("hits_"):
                per[k] = per.get(k, 0.0) + e.device_time_total
        parts = "  ".join(f"{k} {v / STEPS:.1f}" for k, v in sorted(per.items()))
        print(f"  us per step per kernel (torch.profiler, one call): {parts}", flush=True)
        a = g.to_original(auth)
        h = g.to_original(hub)
        src = torch.from_numpy(dsrc.to_numpy()).cuda().long()
        dst = torch.from_numpy(ddst.to_numpy()).cuda().long()
        dsrc.free(); ddst.free()
        ra, rh = restatement(V, src, dst, STEPS)
        del src, dst
        torch.cuda.empty_cache()
        print(f"  vs fp64 restatement: auth rel L1 {rel_l1(a, ra):.2e}  hub rel L1 {rel_l1(h, rh):.2e}", flush=True)
        auth.free(); hub.free(); ranks.free()
        g.free()
