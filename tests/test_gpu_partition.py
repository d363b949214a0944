"""GPU parity of the 1D-partitioned path (csrc/partition.cu and the *_partitioned drivers).

* the partitioned builder, for every rank of P = 1, 2, 3, 4 (detached communicators: the build is collective-free),
  against the reference layout frozen in tests/golden/;
* the four partitioned algorithm drivers with a live single-rank NCCL communicator on one GPU (every collective runs);
* the same on 2 GPUs (torchrun, one process per GPU) when the box has them: results must be identical for any P.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PR_TOL = 1e-6


def _edges(O, g):
    return O.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))


@pytest.mark.parametrize("P", [1, 2, 3, 4])
def test_partitioned_build_matches_reference_layout(vgl, ctx, oracle, golden, P):
    from vectorgraphlibrary_b200 import multi
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    vp = multi.rows_per_rank(V, P)
    ref_ptr, ref_adj, ref_fwd = g["out_ptr"], g["out_adj"], g["out_fwd"]
    in_src_sorted = np.repeat(np.arange(V, dtype=np.int64), np.diff(ref_ptr))  # source (sorted id) of every out-CSR position
    total_e = 0
    for rank in range(P):
        comm = vgl.Comm(ctx, rank, P, detached=True)
        G = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
        assert (G.rank, G.world, G.vp, G.cols, G.V_global, G.E_global) == (rank, P, vp, vp * P, V, len(src))
        assert G.V == multi.local_rows(V, P, rank) and G.col0 == rank * vp
        # numbering: ORIGINAL -> column is the reference's ORIGINAL -> sorted map composed with the round-robin deal
        fwd = G.orig_to_sorted()
        assert np.array_equal(fwd, multi.column_of_sorted(ref_fwd, P, vp))
        bwd = G.sorted_to_orig()
        assert np.array_equal(bwd[fwd], np.arange(V)) and int((bwd < 0).sum()) == vp * P - V
        ptr, adj = G.layout()
        iptr, iadj = G.layout(incoming=True)
        total_e += G.E
        for r in range(G.V):
            s = r * P + rank  # sorted id of local row r
            want = np.sort(multi.column_of_sorted(ref_adj[ref_ptr[s]:ref_ptr[s + 1]], P, vp))
            got = adj[ptr[r]:ptr[r + 1]]
            assert np.array_equal(np.sort(got), want), (rank, r)
            # rows list their neighbours hubs-first (ascending sorted id)
            assert np.all(np.diff(multi.sorted_of_column(got, P, vp)) >= 0)
        want_in = [np.sort(multi.column_of_sorted(in_src_sorted[ref_adj == (r * P + rank)], P, vp)) for r in range(G.V)]
        for r in range(G.V):
            assert np.array_equal(np.sort(iadj[iptr[r]:iptr[r + 1]]), want_in[r]), (rank, r)
        deg = np.diff(ptr)
        assert np.all(np.diff(deg) <= 0)  # every part is degree-sorted: tiers stay contiguous
        td, tb = G.tiers()
        for t in range(vgl.NUM_TIERS - 1):
            assert tb[t] == int((deg >= td[t]).sum())
        G.free()
        comm.close()
    assert total_e == len(src)


def test_partitioned_build_from_generator_and_symmetrize(vgl, ctx, oracle):
    from vectorgraphlibrary_b200 import multi
    scale, ef, P = 10, 8, 2
    V = 1 << scale
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, scale, ef)
    s2, d2 = oracle.symmetrize(src, dst)
    for rank in range(P):
        comm = vgl.Comm(ctx, rank, P, detached=True)
        A = vgl.Graph.from_generator_partitioned(ctx, comm, vgl.GEN_RMAT, scale, ef, 0, symmetrize=True)
        B = vgl.Graph.from_edges_partitioned(ctx, comm, V, s2, d2, 0)
        C_ = vgl.Graph.from_edges_partitioned(ctx, comm, V, ctx.from_numpy(src), ctx.from_numpy(dst), 0, symmetrize=True)
        for X in (B, C_):
            pa, aa = A.layout()
            px, ax = X.layout()
            assert np.array_equal(pa, px) and np.array_equal(aa, ax)
            assert np.array_equal(A.orig_to_sorted(), X.orig_to_sorted())
        assert A.E_global == 2 * len(src)
        for X in (A, B, C_):
            X.free()
        comm.close()


def _check_algorithms(vgl, ctx, oracle, comm, g, G):
    """All four algorithms on a partitioned graph G against the golden outputs of the unmodified reference."""
    fwd = G.orig_to_sorted()
    for i, s in enumerate(g["sources"]):
        for dopt in (False, True):
            lv, st = G.bfs(int(fwd[int(s)]), direction_optimising=dopt)
            assert np.array_equal(G.to_original(lv), g["bfs_levels"][i]), ("bfs", i, dopt)
            lv.free()
    w = G.synthetic_weights(int(g["weight_seed"]))
    for i, s in enumerate(g["sources"]):
        d, st = G.sssp(w, int(fwd[int(s)]))
        assert np.array_equal(G.to_original(d).view(np.uint32), g["sssp_dist"][i].view(np.uint32)), ("sssp", i)
        d.free()
    lab, st = G.cc()
    assert np.array_equal(G.to_original(lab), g["cc_directed"])
    ranks, st = G.pagerank(int(g["pr_iters"]))
    assert oracle.rel_l1(G.to_original(ranks), g["pr_ranks"]) <= PR_TOL
    assert st.iterations == int(g["pr_iters"])


def test_partitioned_drivers_single_rank_nccl(vgl, ctx, oracle, golden):
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    comm = vgl.Comm(ctx, 0, 1)
    G = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    _check_algorithms(vgl, ctx, oracle, comm, g, G)
    # the upload path of an already-built part (VGL_Graph::move_to_device twin) gives the same PageRank
    ptr, adj = G.layout()
    iptr, iadj = G.layout(incoming=True)
    H = vgl.Graph.from_csr_partitioned(ctx, comm, V, ptr, adj, G.orig_to_sorted(), iptr, iadj)
    _check_algorithms(vgl, ctx, oracle, comm, g, H)
    s2, d2 = oracle.symmetrize(src, dst)
    G2 = vgl.Graph.from_edges_partitioned(ctx, comm, V, s2, d2)
    lab2, _ = G2.cc()
    assert np.array_equal(G2.to_original(lab2), g["cc_symmetric"])
    for X in (G, H, G2):
        X.free()
    comm.close()


@pytest.mark.parametrize("world,dense", [(2, False), (2, True)])
def test_partitioned_drivers_multi_gpu(vgl, world, dense):
    """torchrun, one process per GPU; every rank checks the whole result against the golden fixtures — with the CUDA IPC
    exchanges (default) and with the NCCL-only fallbacks."""
    if vgl.lib().vglb_device_count() < world:
        pytest.skip(f"needs {world} GPUs")
    port = 29500 + (os.getpid() % 2000) + (7 if dense else 0)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={world}", "--master-addr", "127.0.0.1",
           "--master-port", str(port), os.path.join(ROOT, "tests", "part_worker.py")]
    env = dict(os.environ)
    if dense:
        env["VGLB_DENSE_EXCHANGE"] = "1"
    p = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert p.returncode == 0, p.stdout[-4000:] + p.stderr[-4000:]
    assert p.stdout.count("PART_WORKER_OK") == world, p.stdout[-4000:] + p.stderr[-4000:]


def test_partitioned_ragged_and_empty(vgl, ctx, oracle):
    """V not a multiple of 32 or of the rank count, self loops, duplicates, isolated vertices; and a graph without edges."""
    from vectorgraphlibrary_b200 import multi
    V = 77
    rng = np.random.default_rng(5)
    src = np.concatenate([np.zeros(60, np.int32), rng.integers(1, 50, 90).astype(np.int32), np.array([3, 3, 9], np.int32)])
    dst = np.concatenate([rng.integers(0, 70, 60).astype(np.int32), rng.integers(0, 50, 90).astype(np.int32), np.array([3, 3, 9], np.int32)])
    og = oracle.OracleGraph(V, src, dst)
    for P in (3, 8):
        vp = multi.rows_per_rank(V, P)
        seen_rows = 0
        for rank in range(P):
            comm = vgl.Comm(ctx, rank, P, detached=True)
            G = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
            assert G.V == multi.local_rows(V, P, rank) and G.vp == vp and G.cols == vp * P
            assert np.array_equal(G.orig_to_sorted(), multi.column_of_sorted(og.fwd, P, vp))
            ptr, adj = G.layout()
            for r in range(G.V):
                s = r * P + rank
                want = np.sort(multi.column_of_sorted(og.adj[og.row_ptr[s]:og.row_ptr[s + 1]], P, vp))
                assert np.array_equal(np.sort(adj[ptr[r]:ptr[r + 1]]), want)
            seen_rows += G.V
            G.free()
            comm.close()
        assert seen_rows == V
    # live single-rank communicator: the algorithms on the ragged graph and on a graph without edges
    comm = vgl.Comm(ctx, 0, 1)
    G = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    fwd = G.orig_to_sorted()
    w = G.synthetic_weights(11)
    for s in (0, 3, 76):
        for dopt in (False, True):
            lv, _ = G.bfs(int(fwd[s]), dopt)
            assert np.array_equal(G.to_original(lv), og.bfs(s)[0])
        d, _ = G.sssp(w, int(fwd[s]))
        assert np.array_equal(G.to_original(d).view(np.uint32), og.sssp(s, 11)[0].view(np.uint32))
    lab, _ = G.cc()
    assert np.array_equal(G.to_original(lab), og.cc()[0])
    ranks, _ = G.pagerank(20)
    assert oracle.rel_l1(G.to_original(ranks), og.pagerank_f32(20, 2)) <= PR_TOL
    G.free()
    e = np.empty(0, np.int32)
    G0 = vgl.Graph.from_edges_partitioned(ctx, comm, 40, e, e, vgl.GRAPH_WITH_INCOMING)
    assert G0.E == 0 and G0.V == 40
    lv, _ = G0.bfs(7, True)
    exp = np.full(40, -1, np.int32)
    exp[G0.sorted_to_orig()[7]] = 1
    assert np.array_equal(G0.to_original(lv), exp)
    lab, _ = G0.cc()
    assert np.array_equal(np.sort(G0.to_original(lab)), np.arange(40))
    ranks, _ = G0.pagerank(3)
    assert abs(float(ranks.to_numpy().astype(np.float64).sum()) - 1.0) < 1e-5
    G0.free()
    comm.close()


def test_partitioned_fallback_exchanges(vgl, ctx, oracle, golden, monkeypatch):
    """Without CUDA IPC the partitioned BFS / SSSP fall back to NCCL-only exchanges (candidate-bitmap all-to-all,
    allreduce(min) of the distance vector); VGLB_DENSE_EXCHANGE forces that path."""
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    monkeypatch.setenv("VGLB_DENSE_EXCHANGE", "1")
    comm = vgl.Comm(ctx, 0, 1)
    G = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    _check_algorithms(vgl, ctx, oracle, comm, g, G)
    G.free()
    comm.close()
