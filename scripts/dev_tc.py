"""dev (GPU): vglb_tc on one B200, with the PageRank sweep on the same graph as the yardstick.

    python scripts/dev_tc.py [reps]   -> prints, and writes profiles/r8_tc.txt unless the tree is read-only

Graphs: RMAT scale 24 ef16, uniform scale 24 ef32 and Kronecker scale 26 ef16, generated on the device and uploaded without the
incoming CSR. Per graph: one warm-up call, then `reps` timed calls (stats.seconds: the library's CUDA events around the whole
call, oriented-CSR build included) reported as median, min and max; the timed calls' outputs must equal the warm-up call's,
and 3 * total must equal the sum of the counts. One torch.profiler run (CUDA activities) splits a call into the build (key
kernel, radix sort, dedupe, scans, ids and cost kernels, memsets) and tc_count_kernel. Printed: E+ (edges of the oriented
CSR), the list elements the intersections read, the longest oriented row, the triangles, and three rates: GTEPS = E / time
(the reference's convention), list elements per second, and algorithmic bytes / time against the 6539 GB/s copy bandwidth
DESIGN measured. Then 20 PageRank sweeps on the same graph (ms per sweep). The card's name and power limit are read in the
same run."""
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch
from torch.profiler import ProfilerActivity, profile

import vectorgraphlibrary_b200 as vgl

COPY_GBPS = 6539.0  # DESIGN: measured device copy bandwidth of the B200
GRAPHS = [("RMAT s24 ef16", vgl.GEN_RMAT, 24, 16), ("uniform s24 ef32", vgl.GEN_UNIFORM, 24, 32),
          ("Kronecker s26 ef16", vgl.GEN_KRONECKER, 26, 16)]
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
lines = []


def out(s=""):
    print(s, flush=True)
    lines.append(s)


def longest_oriented_row(G):
    """the oriented CSR restated with torch on the GPU from the downloaded layout: the longest row N+(u) = {w < u}"""
    ptr, adj = G.layout()
    V = G.V
    rows = torch.repeat_interleave(torch.arange(V, device="cuda"), torch.from_numpy(np.diff(ptr)).cuda())
    a = torch.from_numpy(adj).cuda().long()
    keep = rows != a
    key = torch.unique(torch.maximum(rows, a)[keep] * V + torch.minimum(rows, a)[keep])
    return int(torch.bincount(key // V, minlength=V).max())


def main():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    out(f"GPU: {q[0] if q else 'unknown'}")
    with vgl.Context(0) as ctx:
        for name, kind, scale, ef in GRAPHS:
            V = 1 << scale
            dsrc, ddst = ctx.generate_edges(kind, scale, ef)
            G = vgl.Graph.from_edges(ctx, V, dsrc, ddst)
            dsrc.free(); ddst.free()
            E = G.E
            c0, total, st0 = G.tc()
            ref = c0.to_numpy()
            assert 3 * total == int(ref.sum()), "3 * total != sum(counts)"
            times, same = [], True
            for _ in range(reps):
                c, t, st = G.tc(c0)
                times.append(st.seconds)
                same &= t == total and np.array_equal(c.to_numpy(), ref)
            med = statistics.median(times)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                G.tc(c0)
                torch.cuda.synchronize()
            count_us = build_us = 0.0
            per = {}
            for ev in prof.key_averages():
                us = ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
                if us <= 0:
                    continue
                per[ev.key] = us
                if "tc_count_kernel" in ev.key:
                    count_us += us
                else:
                    build_us += us
            e_plus = (st0.algorithmic_bytes - 8 * E - 4 * st0.edges_inspected - 16 * V) // 12
            longest = longest_oriented_row(G)
            out(f"{name}: V={V} E={E} E+={e_plus} list elements read={st0.edges_inspected} longest oriented row={longest} "
                f"rows with entries={st0.vertices_processed} triangles={total}")
            out(f"  vglb_tc ms per call: median {med * 1e3:.2f}  min {min(times) * 1e3:.2f}  max {max(times) * 1e3:.2f}  "
                f"({reps} calls; outputs equal the warm-up call's: {same}; 3 * total == sum(counts): True)")
            out(f"  {E / med / 1e9:.2f} GTEPS (E / time)  {st0.edges_inspected / med / 1e9:.2f} G list elements/s  "
                f"{st0.algorithmic_bytes / med / 1e9:.0f} GB/s algorithmic ({st0.algorithmic_bytes / med / 1e9 / COPY_GBPS * 100:.1f} % of "
                f"{COPY_GBPS:.0f} GB/s)")
            out(f"  torch.profiler, one call: build {build_us / 1e3:.2f} ms, tc_count_kernel {count_us / 1e3:.2f} ms; "
                f"count kernel {st0.edges_inspected / (count_us * 1e-6) / 1e9:.2f} G list elements/s")
            for k, us in sorted(per.items(), key=lambda kv: -kv[1])[:8]:
                out(f"    {us / 1e3:9.3f} ms  {k[:110]}")
            c0.free()
            ranks, _ = G.pagerank(20)
            pr = []
            for _ in range(3):
                _, sp = G.pagerank(20, ranks=ranks)
                pr.append(sp.seconds / 20)
            ranks.free()
            out(f"  PageRank sweep on the same graph: {statistics.median(pr) * 1e3:.3f} ms;  vglb_tc / sweep = "
                f"{med / statistics.median(pr):.1f}")
            assert same, "a timed call's output differs from the warm-up call's"
            G.free()
            torch.cuda.empty_cache()
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "profiles", "r8_tc.txt")
    try:
        with open(path, "w") as f:
            f.write("\n".join(lines) + "\n")
    except OSError:
        pass


if __name__ == "__main__":
    main()
