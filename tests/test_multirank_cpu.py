"""CPU tests of the multi-GPU host logic: partition arithmetic (mirror of csrc/partition.cu) and the torch.distributed
plumbing with the gloo backend at world_size 2 (the N > 1 path of bench.py minus the CUDA calls)."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_round_robin_deal_arithmetic():
    from vectorgraphlibrary_b200 import multi
    for V in (1, 2, 33, 1 << 10, 12345):
        for P in (1, 2, 3, 4, 8):
            vp = multi.rows_per_rank(V, P)
            assert vp % 32 == 0 and vp * P >= V and vp >= -(-V // P)
            s = np.arange(V)
            c = multi.column_of_sorted(s, P, vp)
            assert len(np.unique(c)) == V and c.max() < vp * P
            assert np.array_equal(multi.sorted_of_column(c, P, vp), s)
            assert np.array_equal(multi.owner_of_column(c, vp), s % P)
            assert sum(multi.local_rows(V, P, r) for r in range(P)) == V
            # every rank's rows keep the sorted (degree-descending) order
            for r in range(P):
                mine = c[(s % P) == r]
                assert np.array_equal(mine, r * vp + np.arange(len(mine)))


def test_gloo_world_size_2():
    port = 29700 + (os.getpid() % 2000)
    env = dict(os.environ, OMP_NUM_THREADS="1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "gloo_worker.py")]
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stdout[-3000:] + p.stderr[-3000:]
    assert p.stdout.count("GLOO_WORKER_OK") == 2


def test_bench_requires_matching_world_size():
    """bench.py --gpus N outside torchrun must refuse to run rather than silently measure one GPU."""
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "2", "--steps", "1"], capture_output=True,
                       text=True, timeout=300, cwd=ROOT)
    assert p.returncode != 0 and "WORLD_SIZE" in (p.stdout + p.stderr)


def test_bench_reference_arm_contract(vgl):
    """`bench.py --impl reference` (the CPU arm that runs beside ours) prints one JSON line with the contract's keys;
    and our own arm refuses to run without a CUDA device instead of falling back to anything."""
    import json
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1",
                        "--cpu-scale", "12"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "GTEPS" and line["unit"] == "GTEPS" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["gpu_launches"] == 0 and line["config"]["workload"].startswith("PageRank pull")
    assert line["cpu_baseline"]["kind"] in ("reference", "port") and line["cpu_baseline"]["cores"] >= 1 and "sample" in line["cpu_baseline"]
    assert line["e2e"] == {"value": line["value"], "unit": "GTEPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    # the device count of the library, not `import torch`: once an earlier test in this process has created a library
    # communicator, the NCCL that dlopen() found first is loaded, and torch cannot load the newer one it links against
    if vgl.lib().vglb_device_count() == 0:
        q = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert q.returncode != 0 and "no CUDA device" in (q.stdout + q.stderr)


def test_source_picker_twins_agree():
    """dist.pick_sources (bench / runners), oracle.pick_sources (tests) and vglb_source_candidate (include/vglb_synth.h) are the
    same seeded sequence."""
    import oracle as O
    from vectorgraphlibrary_b200 import dist as vdist
    rng = np.random.default_rng(3)
    for V in (64, 1000, 1 << 14):
        deg = rng.integers(0, 3, V)
        deg[rng.integers(0, V)] = 5
        for seed in (0xB200, 7):
            assert vdist.pick_sources(V, deg, 8, seed) == [int(x) for x in O.pick_sources(V, deg, 8, seed)]
