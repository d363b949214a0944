"""HITS (vglb_hits): hub and authority scores against an fp64 numpy restatement of the contract in include/vgl_b200.h,

    a_raw[v] = sum_{u->v} h[u],  a = a_raw / ||a_raw||;   h_raw[u] = sum_{u->v} a[v],  h = h_raw / ||h_raw||,   h_0 = 1,

compared in ORIGINAL numbering. The restatement itself is checked against the principal singular vectors of the adjacency
matrix. Covered on the GPU: the golden fixtures and three generators at 1, 2 and 20 steps, RMAT scale 24, duplicate edges,
self loops and vertices without in- or out-edges, rows long enough to be cut into pieces in both directions, bitwise
reproducibility, the four ways a graph gets its incoming CSR, a graph without edges, argument errors and the stats."""
import numpy as np
import pytest

gpu = pytest.mark.gpu
TOL = 1e-6  # relative L1, the PageRank bar


def hits_f64(V, src, dst, steps):
    """fp64 restatement: (authorities, hubs) after `steps` steps; a zero vector stays zero."""
    src = np.asarray(src, np.int64)
    dst = np.asarray(dst, np.int64)
    h = np.ones(V)
    a = np.zeros(V)
    for _ in range(steps):
        a = np.bincount(dst, weights=h[src], minlength=V)
        n = np.sqrt((a * a).sum())
        a = a / n if n > 0 else a
        h = np.bincount(src, weights=a[dst], minlength=V)
        n = np.sqrt((h * h).sum())
        h = h / n if n > 0 else h
    return a, h


def _rel(O, got, ref):
    return O.rel_l1(got, ref)


def _run(vgl, G, steps):
    a, h, st = G.hits(steps)
    out = G.to_original(a), G.to_original(h), st
    a.free()
    h.free()
    return out


def _check_parity(vgl, O, G, V, src, dst, steps, what):
    ga, gh, _ = _run(vgl, G, steps)
    ra, rh = hits_f64(V, src, dst, steps)
    assert np.isfinite(ga).all() and np.isfinite(gh).all()
    ea, eh = _rel(O, ga, ra), _rel(O, gh, rh)
    assert ea <= TOL and eh <= TOL, (what, steps, ea, eh)


# ---- CPU --------------------------------------------------------------------------------------------------------------

def test_null_arguments_fail_without_device(vgl):
    L = vgl.lib()
    buf = np.zeros(4, np.float32)
    assert L.vglb_hits(None, None, 1, None, None, None) == 1  # VGLB_EINVAL
    assert b"NULL" in L.vglb_last_error()
    assert L.vglb_hits(None, None, 1, buf.ctypes.data, buf.ctypes.data, None) == 1
    assert b"NULL" in L.vglb_last_error()


def test_restatement_converges_to_the_principal_singular_vectors():
    """After 200 steps the authorities are the principal eigenvector of A^T A and the hubs that of A A^T."""
    rng = np.random.default_rng(11)
    V = 24
    src = rng.integers(0, V, 90)
    dst = rng.integers(0, V, 90)
    # a dense core gives a clear eigengap
    core = np.array([(u, v) for u in range(4) for v in range(4, 9)])
    src = np.concatenate([src, core[:, 0], core[:, 0]])
    dst = np.concatenate([dst, core[:, 1], core[:, 1]])
    A = np.zeros((V, V))
    np.add.at(A, (src, dst), 1.0)
    for M, which in ((A.T @ A, 0), (A @ A.T, 1)):
        w, vec = np.linalg.eigh(M)
        assert w[-2] / w[-1] < 0.5, "the test graph needs a clear eigengap"
        got = hits_f64(V, src, dst, 200)[which]
        cos = abs(got @ vec[:, -1]) / (np.linalg.norm(got) * np.linalg.norm(vec[:, -1]))
        assert cos >= 1 - 1e-9, (which, cos)


# ---- GPU --------------------------------------------------------------------------------------------------------------

@gpu
@pytest.mark.parametrize("steps", [1, 2, 20])
def test_golden_fixtures(vgl, ctx, oracle, golden, steps):
    name, g = golden
    src, dst = oracle.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))
    V = 1 << int(g["scale"])
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    _check_parity(vgl, oracle, G, V, src, dst, steps, name)
    G.free()


@gpu
@pytest.mark.parametrize("kind,scale,ef", [(0, 14, 16), (1, 14, 16), (2, 12, 32)])
@pytest.mark.parametrize("steps", [1, 2, 20])
def test_generators(vgl, ctx, oracle, kind, scale, ef, steps):
    V = 1 << scale
    src, dst = oracle.generate_edges(kind, scale, ef, 0x4175 + scale)
    G = vgl.Graph.from_edges(ctx, V, src, dst)  # no incoming CSR: the first call derives it
    _check_parity(vgl, oracle, G, V, src, dst, steps, (kind, scale, ef))
    G.free()


@gpu
def test_rmat_s24(vgl, ctx, oracle):
    """RMAT scale 24 ef16, 20 steps, against the restatement on the CSR the builder produced (SCATTER numbering)."""
    scale, ef, steps = 24, 16, 20
    V = 1 << scale
    dsrc, ddst = ctx.generate_edges(vgl.GEN_RMAT, scale, ef)
    G = vgl.Graph.from_edges(ctx, V, dsrc, ddst)
    dsrc.free(); ddst.free()
    ptr, adj = G.layout()
    rows = np.repeat(np.arange(V, dtype=np.int32), np.diff(ptr))
    a, h, st = G.hits(steps)
    ga, gh = a.to_numpy(), h.to_numpy()
    ra, rh = hits_f64(V, rows, adj, steps)
    del rows
    ea, eh = oracle.rel_l1(ga, ra), oracle.rel_l1(gh, rh)
    assert ea <= TOL and eh <= TOL, (ea, eh)
    assert st.edges_inspected == 2 * G.E * steps
    G.free()


def _structure_graph():
    """Duplicate edges, self loops, an isolated vertex, vertices with only in-edges and only out-edges."""
    edges = [(0, 1), (0, 1), (0, 2), (1, 1), (1, 2), (2, 0), (2, 0), (3, 2), (3, 3), (6, 0), (6, 2), (0, 7), (1, 7),
             (8, 8), (9, 10), (9, 10), (9, 10), (4, 11), (11, 4)]
    src = np.array([e[0] for e in edges], np.int32)
    dst = np.array([e[1] for e in edges], np.int32)
    return 13, src, dst  # vertices 5 and 12 are isolated


@gpu
@pytest.mark.parametrize("steps", [1, 2, 20])
def test_exact_structure(vgl, ctx, oracle, steps):
    V, src, dst = _structure_graph()
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    ga, gh, _ = _run(vgl, G, steps)
    ra, rh = hits_f64(V, src, dst, steps)
    assert oracle.rel_l1(ga, ra) <= TOL and oracle.rel_l1(gh, rh) <= TOL
    indeg, outdeg = np.bincount(dst, minlength=V), np.bincount(src, minlength=V)
    assert np.all(ga[indeg == 0] == 0.0) and np.all(ga[indeg > 0] > 0.0)
    assert np.all(gh[outdeg == 0] == 0.0) and np.all(gh[outdeg > 0] > 0.0)
    G.free()


def _long_rows_graph():
    """Vertex 0 has 150,000 out-edges, vertex 1 has 130,000 in-edges, next to 6,000 rows of one edge."""
    rng = np.random.default_rng(5)
    V = 1 << 18
    s = [np.zeros(150_000, np.int64), np.arange(2, 130_002), rng.integers(2, V, 6_000)]
    d = [rng.integers(0, V, 150_000), np.ones(130_000, np.int64), rng.integers(0, V, 6_000)]
    return V, np.concatenate(s).astype(np.int32), np.concatenate(d).astype(np.int32)


@gpu
def test_long_rows_and_reproducibility(vgl, ctx, oracle):
    V, src, dst = _long_rows_graph()
    assert np.bincount(src).max() >= 100_000 and np.bincount(dst).max() >= 100_000
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    for steps in (1, 2, 20):
        _check_parity(vgl, oracle, G, V, src, dst, steps, "long rows")
    a1, h1, _ = G.hits(20)
    a2, h2, _ = G.hits(20)
    assert a1.to_numpy().tobytes() == a2.to_numpy().tobytes()
    assert h1.to_numpy().tobytes() == h2.to_numpy().tobytes()
    G.free()


@gpu
def test_reproducible_bits_rmat(vgl, ctx, oracle):
    V = 1 << 16
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, 16, 16, 0x4176)
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    a1, h1, _ = G.hits(20)
    a2, h2, _ = G.hits(20)
    assert a1.to_numpy().tobytes() == a2.to_numpy().tobytes()
    assert h1.to_numpy().tobytes() == h2.to_numpy().tobytes()
    G.free()


@gpu
def test_incoming_csr_four_ways(vgl, ctx, oracle):
    """from_edges with and without GRAPH_WITH_INCOMING, from_csr with and without incoming arrays: identical bits."""
    V = 1 << 14
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, 14, 16, 0x4177)
    G0 = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    ptr, adj = G0.layout()
    iptr, iadj = G0.layout(incoming=True)
    fwd = G0.orig_to_sorted()
    graphs = [G0, vgl.Graph.from_edges(ctx, V, src, dst), vgl.Graph.from_csr(ctx, ptr, adj, fwd, iptr, iadj),
              vgl.Graph.from_csr(ctx, ptr, adj, fwd)]
    outs = []
    for G in graphs:
        a, h, _ = G.hits(20)
        outs.append((a.to_numpy().tobytes(), h.to_numpy().tobytes()))
        G.free()
    assert all(o == outs[0] for o in outs[1:])


@gpu
def test_graph_without_edges(vgl, ctx):
    V = 64
    e = np.empty(0, np.int32)
    G = vgl.Graph.from_edges(ctx, V, e, e, vgl.GRAPH_WITH_INCOMING)
    a, h, st = G.hits(3)
    ga, gh = a.to_numpy(), h.to_numpy()
    assert np.all(ga == 0.0) and np.all(gh == 0.0)
    assert st.iterations == 3 and st.edges_inspected == 0
    G.free()


@gpu
def test_argument_errors(vgl, ctx, oracle):
    V = 1 << 10
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, 10, 8, 0x4178)
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    for steps in (0, -1, 1 << 20):
        with pytest.raises(vgl.VglbError, match=r"\[vglb error 1\].*steps"):
            G.hits(steps)
    G.free()
    comm = vgl.Comm(ctx, 0, 2, detached=True)
    P = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    with pytest.raises(vgl.VglbError, match=r"\[vglb error 1\].*partitioned"):
        P.hits(1)
    P.free()
    comm.close()


@gpu
def test_stats(vgl, ctx, oracle):
    V = 1 << 12
    src, dst = oracle.generate_edges(oracle.GEN_KRONECKER, 12, 16, 0x4179)
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    for steps in (1, 7):
        _, _, st = G.hits(steps)
        E = G.E
        assert st.iterations == steps
        assert st.edges_inspected == 2 * E * steps
        assert st.vertices_processed == 2 * V * steps
        assert st.algorithmic_bytes == 2 * steps * (8 * E + 12 * V) + 16 * V
        assert st.kernel_launches >= 2 * steps and st.seconds > 0
    G.free()


@gpu
def test_against_reference_seq_hits(vgl, ctx, oracle):
    """The reference's own HITS::seq_hits (oracle/ref_gpu_harness.cu) on the drop-in test's 5-step RMAT scale-13 case."""
    O = oracle
    if not O.gpu_ref_available("dropin"):
        pytest.skip("oracle/_ref/libvgl_dropin.so not built: it needs the reference's sources")
    V = 1 << 13
    src, dst = O.generate_edges(O.GEN_RMAT, 13, 16, 0xE1)
    R = O.GpuRefGraph(V, src, dst, "dropin")
    _, _, sa, sh, _ = R.hits(5)
    R.close()
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    ga, gh, _ = _run(vgl, G, 5)
    G.free()
    assert O.rel_l1(ga, sa) <= 1e-5 and O.rel_l1(gh, sh) <= 1e-5, (O.rel_l1(ga, sa), O.rel_l1(gh, sh))
