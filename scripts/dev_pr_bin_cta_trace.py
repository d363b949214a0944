"""dev (GPU): how evenly pr_bin_kernel's persistent CTAs, and the warps inside them, share the shared-memory bins at RMAT scale 24.

    scripts/dev_build_variant.sh ctatrace -DPRB_CTA_TRACE
    VGLB_LIB_PATH=dev/lib_ctatrace.so python scripts/dev_pr_bin_cta_trace.py [reps]

A PRB_CTA_TRACE build records, for the last pr_bin_kernel launch, %globaltimer at the start and end of every CTA, its chunks,
runs and bins, the time its slice loads take between their two barriers, and per warp the time inside its units, their steps and
runs. After each of `reps` runs of 20 sweeps this prints the CTA times (min / avg / max), their correlation with the cost
estimate 2048 per chunk + 1 per run, the spread of the warps inside a CTA, and a least-squares fit of the warps' unit times
to steps and runs (ns per step, ns per run), which is what the cost estimate of the chunks and the warp pieces should weigh."""
import ctypes as C
import os
import subprocess
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
import numpy as np
import torch

import vectorgraphlibrary_b200 as vgl

ITERS = 20
WARPS = 32
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 3

gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print(f"GPU: {gpu[0] if gpu else 'unknown'}  library: {os.path.basename(vgl.LIB_PATH)}", flush=True)
torch.cuda.init()
L = vgl.lib()
if not hasattr(L, "vglb_dev_prb_cta_trace"):
    sys.exit("this library was built without -DPRB_CTA_TRACE")
ctas = torch.cuda.get_device_properties(0).multi_processor_count  # pr_bin_kernel's grid: one CTA per SM


def stats(x):
    return f"min {x.min():7.1f} avg {x.mean():7.1f} max {x.max():7.1f}"


with vgl.Context(0) as ctx:
    dsrc, ddst = ctx.generate_edges(vgl.GEN_RMAT, 24, 16)
    g = vgl.Graph.from_edges(ctx, 1 << 24, dsrc, ddst, 0)
    out = ctx.empty(g.V, np.float32)
    print(f"RMAT s24 ef16: V={g.V} E={g.E}, {ctas} CTAs; trace of the last pr_bin_kernel of a run of {ITERS} sweeps", flush=True)
    for r in range(reps):
        g.pagerank(ITERS, 0.85, out)
        cta = np.zeros((ctas, 8), np.uint64)
        warp = np.zeros((ctas, WARPS, 4), np.uint64)
        rc = L.vglb_dev_prb_cta_trace(cta.ctypes.data_as(C.c_void_p), warp.ctypes.data_as(C.c_void_p), C.c_int(ctas))
        assert rc == 0, rc
        t0, t1 = cta[:, 0].astype(np.float64), cta[:, 1].astype(np.float64)
        dur = (t1 - t0) / 1e3  # us
        chunks, runs, nbins, load = (cta[:, i].astype(np.float64) for i in (2, 3, 4, 5))
        busy = warp[:, :, 0].astype(np.float64) / 1e3
        steps, wruns = warp[:, :, 1].astype(np.float64), warp[:, :, 2].astype(np.float64)
        est = 2048 * chunks + runs
        print(f"--- run {r}: kernel span {(t1.max() - t0.min()) / 1e3:.1f} us; CTA start spread {(t0.max() - t0.min()) / 1e3:.1f} us", flush=True)
        print(f"CTA us:              {stats(dur)}  (max / avg {dur.max() / dur.mean():.3f})")
        print(f"CTA cost estimate:   {stats(est / 1e3)} k  corr(time, estimate) {np.corrcoef(dur, est)[0, 1]:.3f}; "
              f"corr(time, chunks) {np.corrcoef(dur, chunks)[0, 1]:.3f}; corr(time, runs) {np.corrcoef(dur, runs)[0, 1]:.3f}")
        print(f"CTA bins:            {stats(nbins)}; slice loads us {stats(load / 1e3)}")
        wmax, wavg = busy.max(axis=1), busy.mean(axis=1)
        print(f"warp unit us per CTA: slowest {stats(wmax)}; mean {stats(wavg)}; slowest / mean: {stats(wmax / wavg)}")
        # unit time of a warp ~ a * steps + b * runs (the 32 warps of an SM share its pipes, so a and b are shares of the SM)
        A = np.stack([steps.ravel(), wruns.ravel()], axis=1)
        y = busy.ravel() * 1e3
        coef, *_ = np.linalg.lstsq(A, y, rcond=None)
        pred = A @ coef
        r2 = 1 - ((y - pred) ** 2).sum() / ((y - y.mean()) ** 2).sum()
        print(f"fit over {y.size} warps: unit ns = {coef[0]:.1f} * steps + {coef[1]:.2f} * runs  (R^2 {r2:.3f}; step / run = {coef[0] / coef[1]:.1f}); "
              f"runs per step: {stats(wruns.ravel() / np.maximum(steps.ravel(), 1))}", flush=True)
        cest = coef[0] * 8 * chunks + coef[1] * runs
        print(f"corr(CTA time, fitted estimate) {np.corrcoef(dur, cest)[0, 1]:.3f}")
        if r == reps - 1:
            print("CTA us by block (the chunk ranges in bin order): " + " ".join(f"{d:.0f}" for d in dur))
    out.free()
    g.free()
