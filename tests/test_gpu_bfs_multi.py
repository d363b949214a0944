"""Multi-source BFS (vglb_bfs_multi): row i of one batched call must equal vglb_bfs(sources[i]) bit for bit, in both
direction modes, for both word widths (k <= 32: 32-bit words, k > 32: 64-bit words), with repeated sources, sources
without out-edges, isolated sources and rows of several CTA chunks; plus the argument checks."""
import ctypes as C

import numpy as np
import pytest

gpu = pytest.mark.gpu


def _edges(O, g):
    return O.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))


def _rows(G, lv, k):
    return lv.to_numpy()[: k * G.V].reshape(k, G.V)


def _single(G, sources, dopt):
    """vglb_bfs for every distinct source: {sorted id: levels in SCATTER numbering}"""
    out = {}
    for s in sorted(set(int(x) for x in sources)):
        lv, _ = G.bfs(s, direction_optimising=dopt)
        out[s] = lv.to_numpy()
        lv.free()
    return out


def test_null_arguments_fail_without_device(vgl):
    L = vgl.lib()
    src = np.zeros(1, np.int32)
    assert L.vglb_bfs_multi(None, None, 1, src.ctypes.data, None, None, None) == 1  # VGLB_EINVAL
    assert b"NULL" in L.vglb_last_error()
    assert L.vglb_bfs_multi(None, None, 1, None, None, None, None) == 1
    assert b"NULL" in L.vglb_last_error()
    assert vgl.BFS_MULTI_MAX_SOURCES == 64


@gpu
@pytest.mark.parametrize("dopt", [False, True])
def test_golden_fixtures(vgl, ctx, oracle, golden, dopt):
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    fwd = G.orig_to_sorted()
    base = [int(fwd[int(s)]) for s in g["sources"]]
    for k in (len(base), 33, 32):
        sources = [base[i % len(base)] for i in range(k)]
        lv, st = G.bfs_multi(sources, direction_optimising=dopt)
        rows = G.to_original_rows(lv, k)
        for i in range(k):
            assert np.array_equal(rows[i], g["bfs_levels"][i % len(base)]), (name, k, i)
        assert st.iterations == int(rows.max()) and st.kernel_launches >= st.iterations
        lv.free()
    G.free()


@gpu
@pytest.mark.parametrize("kind,scale,ef", [(0, 12, 16), (1, 14, 16), (2, 16, 8)])
def test_equivalence_with_single_source(vgl, ctx, oracle, kind, scale, ef):
    O = oracle
    V = 1 << scale
    src, dst = O.generate_edges(kind, scale, ef, 0x5EED + scale)
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    fwd, bwd = G.orig_to_sorted(), G.sorted_to_orig()
    outdeg = np.bincount(src, minlength=V)
    indeg = np.bincount(dst, minlength=V)
    seeded = [int(fwd[s]) for s in O.pick_sources(V, outdeg, 40)]
    special = []
    no_out = np.flatnonzero((outdeg == 0) & (indeg > 0))
    if len(no_out):
        special.append(int(fwd[no_out[0]]))  # reachable, but expands nothing
    isolated = np.flatnonzero((outdeg == 0) & (indeg == 0))
    if len(isolated):
        special.append(int(fwd[isolated[0]]))  # its row is the source alone
    pool = special + seeded
    og = O.OracleGraph(V, src, dst)
    for dopt in (False, True):
        for k in (1, 2, 31, 32, 33, 63, 64):
            sources = [pool[i % len(pool)] for i in range(k)]
            if k >= 31:
                sources[5] = sources[3]  # duplicates inside the batch as well as from the wrap-around
            ref = _single(G, sources, dopt)
            lv, st = G.bfs_multi(sources, direction_optimising=dopt)
            rows = _rows(G, lv, k)
            for i, s in enumerate(sources):
                assert np.array_equal(rows[i], ref[s]), (kind, scale, dopt, k, i)
            assert st.iterations == int(rows.max()) and st.kernel_launches >= st.iterations
            assert dopt or st.bottom_up_levels == 0
            if k == 33:
                orig_rows = G.to_original_rows(lv, k)
                for i in (0, k - 1):
                    assert np.array_equal(orig_rows[i], og.bfs(int(bwd[sources[i]]))[0]), (kind, dopt, i)
            lv.free()
    G.free()


@gpu
def test_hubs_and_long_chain(vgl, ctx, oracle):
    """The graph of test_gpu_parity.test_hubs_and_long_chain: two hubs with > 8192 out-edges (several CTA chunks per row) and
    a 3000-vertex chain hanging off a hub; sources on the hubs, the chain and the filler."""
    O = oracle
    V = 1 << 15
    rng = np.random.default_rng(17)
    hub_a = np.full(20000, 5, np.int32)
    hub_b = np.full(9000, 6, np.int32)
    chain = np.arange(20000, 23000, dtype=np.int32)
    src = np.concatenate([hub_a, hub_b, np.array([5], np.int32), chain[:-1], rng.integers(0, V, 60000).astype(np.int32)])
    dst = np.concatenate([rng.integers(0, V, 20000).astype(np.int32), rng.integers(0, V, 9000).astype(np.int32),
                          chain[:1], chain[1:], rng.integers(0, V, 60000).astype(np.int32)])
    og = O.OracleGraph(V, src, dst)
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    assert G.info.max_degree > 8192
    fwd = G.orig_to_sorted()
    orig = [5, 6, 20000, 21500, 22990, 100, 31000, 7]
    want = {s: og.bfs(s)[0] for s in orig}
    for dopt in (False, True):
        for k in (len(orig), 40):
            sources = [orig[i % len(orig)] for i in range(k)]
            lv, st = G.bfs_multi([int(fwd[s]) for s in sources], direction_optimising=dopt)
            rows = G.to_original_rows(lv, k)
            for i, s in enumerate(sources):
                assert np.array_equal(rows[i], want[s]), (dopt, k, s)
            assert st.iterations == int(rows.max()) and st.kernel_launches >= st.iterations
            lv.free()
    G.free()


@gpu
def test_edge_cases(vgl, ctx):
    V = 40
    e = np.empty(0, np.int32)
    G = vgl.Graph.from_edges(ctx, V, e, e, vgl.GRAPH_WITH_INCOMING)
    sources = [7, 3, 7, 39]
    for dopt in (False, True):
        lv, st = G.bfs_multi(sources, direction_optimising=dopt)
        rows = _rows(G, lv, len(sources))
        for i, s in enumerate(sources):
            exp = np.full(V, -1, np.int32)
            exp[s] = 1
            assert np.array_equal(rows[i], exp)
        assert st.iterations == 1 and st.edges_inspected == 0
    G.free()
    # no incoming CSR: the direction-optimising call derives it, and the rows are the single-source ones
    V = 1 << 12
    src = np.arange(V, dtype=np.int32)
    dst = np.concatenate([(src[: V // 2] + 1) % (V // 2), np.random.default_rng(3).integers(0, V, V // 2).astype(np.int32)])
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    assert not G.info.has_incoming
    sources = [0, 1, V - 1, V // 2 + 7, 0]
    lv, st = G.bfs_multi(sources, direction_optimising=True)
    ref = _single(G, sources, False)
    rows = _rows(G, lv, len(sources))
    for i, s in enumerate(sources):
        assert np.array_equal(rows[i], ref[s]), i
    assert st.iterations == int(rows.max()) and st.kernel_launches >= st.iterations
    G.free()


@gpu
def test_shared_scratch_with_bfs_and_sssp(vgl, ctx, oracle):
    O = oracle
    scale = 13
    V = 1 << scale
    src, dst = O.generate_edges(O.GEN_RMAT, scale, 8, 0xBEEF)
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    fwd = G.orig_to_sorted()
    s = [int(fwd[x]) for x in O.pick_sources(V, np.bincount(src, minlength=V), 3)]
    w = G.synthetic_weights(11)
    lv0, _ = G.bfs(s[0], direction_optimising=True)
    d0, _ = G.sssp(w, s[1])
    before = (lv0.to_numpy(), d0.to_numpy().view(np.uint32))
    ms, _ = G.bfs_multi(s + s[:1], direction_optimising=True)
    rows = _rows(G, ms, 4)
    lv1, _ = G.bfs(s[0], direction_optimising=True)
    d1, _ = G.sssp(w, s[1])
    assert np.array_equal(lv1.to_numpy(), before[0]) and np.array_equal(d1.to_numpy().view(np.uint32), before[1])
    assert np.array_equal(rows[0], before[0]) and np.array_equal(rows[3], before[0])
    G.free()


@gpu
def test_argument_errors_on_device(vgl, ctx):
    V = 16
    src = np.arange(V, dtype=np.int32)
    dst = (src + 1) % V
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    for k in (0, 65):
        with pytest.raises(vgl.VglbError, match="num_sources"):
            G.bfs_multi([0] * k)
    with pytest.raises(vgl.VglbError, match="out of range"):
        G.bfs_multi([0, V])
    with pytest.raises(vgl.VglbError, match="out of range"):
        G.bfs_multi([-1])
    lv, _ = G.bfs_multi([0, 3])  # the graph is still usable
    assert np.array_equal(_rows(G, lv, 2)[1], (np.arange(V) - 3) % V + 1)
    G.free()
    comm = vgl.Comm(ctx, 0, 2, detached=True)
    P = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    with pytest.raises(vgl.VglbError, match="partitioned"):
        P.bfs_multi([0])
    P.free()
    comm.close()


@gpu
def test_kronecker_s26_bench_sources(vgl, ctx):
    """The bench's BFS graph (Kronecker scale 26, edge factor 16) and its 16 sources: every row of one direction-optimising
    batched call equals its vglb_bfs row (compared on the device)."""
    from vectorgraphlibrary_b200 import dist
    scale, ef = 26, 16
    V = 1 << scale
    dsrc, ddst = ctx.generate_edges(vgl.GEN_KRONECKER, scale, ef)
    G = vgl.Graph.from_edges(ctx, V, dsrc, ddst, vgl.GRAPH_WITH_INCOMING)
    dsrc.free(); ddst.free()
    ptr, _ = G.layout()
    fwd = G.orig_to_sorted()
    sources = [int(fwd[s]) for s in dist.pick_sources(V, np.diff(ptr)[fwd], 16, vgl.MASTER_SEED)]
    del ptr
    ms, st = G.bfs_multi(sources, direction_optimising=True)
    one = ctx.empty(V, np.int32)
    L = vgl.lib()
    for i, s in enumerate(sources):
        G.bfs(s, direction_optimising=True, levels=one)
        err = C.c_int64()
        vgl._check(L.vglb_verify_i32(ctx.h, ms.ptr + i * V * 4, one.ptr, V, C.byref(err)))
        assert err.value == 0, (i, s, err.value)
    assert st.iterations >= 2 and st.bottom_up_levels >= 1
    ms.free(); one.free()
    G.free()
