"""Rows without out-edges in the one-GPU PageRank sweep. They all get the same rank, so from PrParams::zero_kept on their
contributions are stored only by the sweep that stores the ranks: the other sweeps compute them where they are gathered
(rank0 of the previous sweep times inv[v]) and add their dangling share as one count. The ranks must be those of the
oracle, the same bits in two runs, and the same bits as with every row stored in every sweep (VGLB_PR_STORE_ZERO_ROWS).

The graphs cover zero rows with and without in-edges (inv != 0 and inv == 0); zero rows past the column bins, so the cold bin
gathers computed values (RMAT s22 ef8); zero rows that start inside the bins' columns, so only those past them are skipped
(RMAT s21); bins that cover every column, so nothing is skipped (RMAT s16); the warp-task sweep (VGLB_PR_NO_BINS); a graph
without heavy rows whose row count is no multiple of a zero-row block; a graph without zero rows; a graph without edges."""
import contextlib
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PR_TOL = 1e-6  # relative L1, as in the other PageRank tests


@contextlib.contextmanager
def _env(**kv):
    old = {k: os.environ.get(k) for k in kv}
    try:
        for k, v in kv.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _tail_only(O):
    # sources in the first third, 1..20 edges each (no heavy rows, no bins); about 2/3 of the rows have no out-edges, most
    # of them with in-edges
    V = 3 * (1 << 14) + 123
    rng = np.random.default_rng(0x2E01)
    deg = rng.integers(1, 21, V // 3)
    src = np.repeat(np.arange(V // 3, dtype=np.int32), deg)
    dst = rng.integers(0, V, src.shape[0]).astype(np.int32)
    return V, src, dst


def _no_zero_rows(O):
    V = 1 << 14
    rng = np.random.default_rng(0x2E02)
    ring = np.arange(V, dtype=np.int32)
    extra = rng.integers(0, V, (2, 8 * V)).astype(np.int32)
    return V, np.concatenate([ring, extra[0]]), np.concatenate([(ring + 1) % V, extra[1]]).astype(np.int32)


def _rmat(scale, ef):
    def make(O):
        src, dst = O.generate_edges(O.GEN_RMAT, scale, ef, 0x2E0 + scale)
        return 1 << scale, src, dst
    return make


def _no_edges(O):
    e = np.empty(0, np.int32)
    return 5000, e, e


# name: (edge maker, VGLB_PR_NO_BINS)
GRAPHS = {
    "tail_only": (_tail_only, False),
    "rmat16_bins_cover_all": (_rmat(16, 4), False),
    "rmat16_warp_tasks": (_rmat(16, 4), True),
    "rmat21_zero_rows_inside_bins": (_rmat(21, 16), False),
    "rmat22_zero_rows_past_bins": (_rmat(22, 8), False),
    "no_zero_rows": (_no_zero_rows, False),
    "no_edges": (_no_edges, False),
}


@pytest.fixture(scope="module")
def graphs(vgl, ctx, oracle):
    cache = {}

    def get(name):
        if name not in cache:
            make, no_bins = GRAPHS[name]
            V, src, dst = make(oracle)
            with _env(VGLB_PR_NO_BINS="1" if no_bins else None):
                G = vgl.Graph.from_edges(ctx, V, src, dst, 0)
            cache[name] = (G, oracle.OracleGraph(V, src, dst), no_bins)
        return cache[name]

    yield get
    for G, _, _ in cache.values():
        G.free()


def _run(G, no_bins, iters, store_zero_rows=False, reference_threads=0):
    with _env(VGLB_PR_NO_BINS="1" if no_bins else None, VGLB_PR_STORE_ZERO_ROWS="1" if store_zero_rows else None):
        r, _ = G.pagerank(iters, reference_threads=reference_threads)
    out = G.to_original(r)
    r.free()
    return out


def _bits(a):
    return a.view(np.uint32)


@pytest.mark.parametrize("iters", [0, 1, 2, 20])
@pytest.mark.parametrize("name", list(GRAPHS))
def test_zero_rows_match_oracle_and_stored_pass(graphs, oracle, name, iters):
    G, og, no_bins = graphs(name)
    got = _run(G, no_bins, iters)
    err = oracle.rel_l1(got, og.pagerank_f64(iters))
    assert err <= PR_TOL, (name, iters, err)
    assert np.array_equal(_bits(got), _bits(_run(G, no_bins, iters))), "two runs differ"
    stored = _run(G, no_bins, iters, store_zero_rows=True)
    assert np.array_equal(_bits(got), _bits(stored)), "computed zero-row contributions differ from stored ones"


@pytest.mark.parametrize("iters", [1, 20])
@pytest.mark.parametrize("name", ["tail_only", "rmat16_warp_tasks", "no_edges"])
def test_zero_rows_reference_order(graphs, oracle, name, iters):
    """reference_threads: the dangling mass is summed in the reference's order from every rank, each sweep stores them all"""
    G, og, no_bins = graphs(name)
    T = 8
    got = _run(G, no_bins, iters, reference_threads=T)
    err = oracle.rel_l1(got, og.pagerank_f32(iters, T))
    assert err <= PR_TOL, (name, iters, err)
    assert np.array_equal(_bits(got), _bits(_run(G, no_bins, iters, reference_threads=T)))
