"""dev (GPU): one multi-source BFS call (vglb_bfs_multi) against the same k vglb_bfs calls in a loop.

    python scripts/dev_bfs_multi.py [reps]

Graphs: Kronecker scale 26 ef16 (BASELINE configs[3], bench `bfs`) and RMAT scale 20 ef16 (configs[0], bench `bfs20`; its
adjacency is under 2 x L2, so L2 is flushed before every timed call, batched or single, as bench.py does). Sources: the first k
of dist.pick_sources(V, out-degrees, 64, MASTER_SEED), whose first 16 are the bench's. For k in {1, 16, 32, 64} and both
direction modes the batched call and the loop run alternately `reps` times (default 3); times are the library's CUDA-event
times (median; a loop's time is the sum of its calls). Every row of the batched output is compared on the device with the
single-source result of the same source. GTEPS are the bench's convention, k * E / time."""
import ctypes as C
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np

import vectorgraphlibrary_b200 as vgl
from vectorgraphlibrary_b200 import dist

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
GRAPHS = [("Kronecker s26 ef16", vgl.GEN_KRONECKER, 26, 16), ("RMAT s20 ef16", vgl.GEN_RMAT, 20, 16)]
KS = [1, 16, 32, 64]

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"GPU: {gpu[0] if gpu else 'unknown'}", flush=True)
L = vgl.lib()
with vgl.Context(0) as ctx:
    for name, kind, scale, ef in GRAPHS:
        V = 1 << scale
        dsrc, ddst = ctx.generate_edges(kind, scale, ef)
        g = vgl.Graph.from_edges(ctx, V, dsrc, ddst, vgl.GRAPH_WITH_INCOMING)
        dsrc.free(); ddst.free()
        ptr, _ = g.layout()
        fwd = g.orig_to_sorted()
        sources = [int(fwd[s]) for s in dist.pick_sources(V, np.diff(ptr)[fwd], 64, vgl.MASTER_SEED)]
        del ptr
        flush = 4 * g.E < 2 * 126e6
        print(f"\n{name}: V={g.V} E={g.E}; L2 {'flushed before every timed call' if flush else 'not flushed (adjacency > 2 x L2)'}",
              flush=True)
        print(f"{'mode':<4} {'k':>3} | {'batched ms':>10} {'ms/src':>7} {'GTEPS':>7} {'levels':>6} {'BU':>3} {'edges insp.':>12} "
              f"{'GB/s':>6} | {'loop ms':>9} {'ms/src':>7} {'GTEPS':>7} {'edges insp.':>12} | speed-up", flush=True)
        out = ctx.empty(64 * V, np.int32)
        one = ctx.empty(V, np.int32)
        for dopt in (True, False):
            g.bfs(sources[0], direction_optimising=dopt, levels=one)  # warm-up: module load, scratch, incoming CSR
            g.bfs_multi(sources[:2], direction_optimising=dopt, levels=out)
            g.bfs_multi(sources[:33], direction_optimising=dopt, levels=out)
            for k in KS:
                src = sources[:k]
                tb, tl, stb, loop_edges = [], [], None, 0
                for r in range(reps):
                    if flush:
                        ctx.flush_l2()
                    _, stb = g.bfs_multi(src, direction_optimising=dopt, levels=out)
                    tb.append(stb.seconds)
                    total, loop_edges, bad = 0.0, 0, 0
                    for i, s in enumerate(src):
                        if flush:
                            ctx.flush_l2()
                        _, st = g.bfs(s, direction_optimising=dopt, levels=one)
                        total += st.seconds
                        loop_edges += st.edges_inspected
                        err = C.c_int64()
                        vgl._check(L.vglb_verify_i32(ctx.h, out.ptr + i * V * 4, one.ptr, V, C.byref(err)))
                        bad += err.value
                    tl.append(total)
                    if bad:
                        raise SystemExit(f"{name} k={k} dopt={dopt}: {bad} levels differ between the batched call and the loop")
                b, l = statistics.median(tb), statistics.median(tl)
                print(f"{'DO' if dopt else 'TD':<4} {k:>3} | {b * 1e3:>10.3f} {b * 1e3 / k:>7.3f} {k * g.E / b / 1e9:>7.1f} "
                      f"{stb.iterations:>6} {stb.bottom_up_levels:>3} {stb.edges_inspected:>12} {stb.algorithmic_bytes / b / 1e9:>6.0f} | "
                      f"{l * 1e3:>9.3f} {l * 1e3 / k:>7.3f} {k * g.E / l / 1e9:>7.1f} {loop_edges:>12} | {l / b:>5.2f}x", flush=True)
        print("outputs: every row of every batched call equals its vglb_bfs result", flush=True)
        out.free(); one.free()
        g.free()
