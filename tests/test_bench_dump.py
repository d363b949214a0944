"""bench.py --dump-outputs: the headline's result of its last timed step, in ORIGINAL numbering, equals what the oracle
computes on the same seeded graph (BFS: for the source of the last step; every step takes the next seeded source)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          timeout=900, cwd=ROOT)


def test_bench_refuses_what_it_cannot_do(tmp_path):
    p = _bench("--steps", "0")
    assert p.returncode == 2 and "--steps must be at least 1" in p.stderr
    p = _bench("--impl", "reference", "--dump-outputs", str(tmp_path))
    assert p.returncode == 2 and "--dump-outputs" in p.stderr
    assert not os.listdir(tmp_path)


@pytest.mark.gpu
@pytest.mark.parametrize("workload,name,dtype", [("pr", "pagerank_ranks", np.float32), ("bfs", "bfs_levels", np.float64)])
def test_bench_dumps_the_last_step(oracle, tmp_path, workload, name, dtype):
    O = oracle
    scale, warmup, steps = 12, 3, 2
    kind, ef = {"pr": (O.GEN_RMAT, 16), "bfs": (O.GEN_KRONECKER, 16)}[workload]
    out = tmp_path / "out"
    p = _bench("--workload", workload, "--scale", str(scale), "--steps", str(steps), "--warmup", str(warmup),
               "--no-cpu-baseline", "--dump-outputs", str(out))
    assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    assert line["dumped_outputs"]["files"] == {name: {"dtype": np.dtype(dtype).name, "values": 1 << scale, "sampled": False}}
    assert sorted(os.listdir(out)) == [name + ".npy"]
    got = np.load(out / (name + ".npy"))
    assert got.dtype == dtype and got.shape == (1 << scale,)
    V = 1 << scale
    src, dst = O.generate_edges(kind, scale, ef)
    og = O.OracleGraph(V, src, dst)
    if workload == "pr":
        assert O.rel_l1(got, og.pagerank_f64(20)) <= 1e-6
    else:
        last = O.pick_sources(V, np.bincount(src, minlength=V), warmup + steps)[-1]
        assert np.array_equal(got, og.bfs(last)[0].astype(np.float64))
