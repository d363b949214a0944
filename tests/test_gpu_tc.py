"""Triangle counting (vglb_tc) against the C oracle vglo_tc (tests/tc_oracle.c, compiled here into a temporary directory),
which is pinned here against scipy and closed forms.

Counted: the triangles of the undirected simple graph under the outgoing CSR (duplicates once, self loops ignored, direction
ignored). The GPU counts are int64 in SCATTER numbering; the tests compare them in ORIGINAL numbering, permuted on the host
with Graph.orig_to_sorted(). Covered on the GPU: the golden fixtures, the three generators at scales 14-16, RMAT scale 20 and
uniform scale 20, a clique whose last rows are longer than a warp's staging buffer (the global-memory path), a wheel with 10^6
spokes (every triangle's smallest id is the hub), graphs without triangles or edges, V = 1 and V not a multiple of 32, six
inputs that describe the same graph, determinism, argument errors and the stats."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest

gpu = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))

# tc.cu: a warp stages its window's slice of the oriented CSR in TC_STAGE = 2048 entries of shared memory; a row with more
# entries than that always has windows that read their prefixes from global memory
TC_STAGE = 2048


def _scipy_tc(V, src, dst):
    import scipy.sparse as sp
    A = sp.coo_matrix((np.ones(len(src)), (src, dst)), shape=(V, V)).tocsr()
    A = A + A.T
    A.setdiag(0)
    A.eliminate_zeros()
    A.data[:] = 1.0
    per_vertex = np.asarray(((A @ A).multiply(A)).sum(axis=1)).ravel() / 2
    total = (A @ A @ A).diagonal().sum() / 6
    return per_vertex.astype(np.int64), int(round(total))


@pytest.fixture(scope="session")
def tc_oracle(tmp_path_factory):
    """vglo_tc(V, row_ptr, adj, counts, &total) from tests/tc_oracle.c"""
    lib_path = str(tmp_path_factory.mktemp("tc_oracle") / "libtc_oracle.so")
    cc = shutil.which("gcc") or "/usr/bin/gcc"
    subprocess.run([cc, "-O2", "-fopenmp", "-fPIC", "-shared", "-std=c11", "-o", lib_path, os.path.join(HERE, "tc_oracle.c")],
                   check=True)
    L = C.CDLL(lib_path)
    i64p = np.ctypeslib.ndpointer(np.int64, flags="C_CONTIGUOUS")
    L.vglo_tc.argtypes = [C.c_int32, i64p, np.ctypeslib.ndpointer(np.int32, flags="C_CONTIGUOUS"), i64p, C.POINTER(C.c_int64)]
    return L


def _oracle_tc(L, V, src, dst):
    """(int64 triangles per vertex, total) of the edge list, in its own numbering"""
    s = np.asarray(src, np.int64)
    row_ptr = np.zeros(V + 1, np.int64)
    np.cumsum(np.bincount(s, minlength=V), out=row_ptr[1:])
    adj = np.ascontiguousarray(np.asarray(dst, np.int32)[np.argsort(s, kind="stable")])
    counts = np.empty(max(V, 1), np.int64)
    total = C.c_int64()
    assert L.vglo_tc(V, row_ptr, adj, counts, C.byref(total)) == 0, "vglo_tc: out of memory"
    return counts[:V], total.value


def clique(n):
    u, v = np.triu_indices(n, 1)
    return n, u.astype(np.int32), v.astype(np.int32)


def wheel(n):
    """hub 0 with spokes to the rim 1..n, and the rim cycle"""
    rim = np.arange(1, n + 1, dtype=np.int32)
    src = np.concatenate([np.zeros(n, np.int32), rim])
    dst = np.concatenate([rim, np.roll(rim, -1)])
    return n + 1, src, dst


def random_tree(V, seed):
    rng = np.random.default_rng(seed)
    child = np.arange(1, V, dtype=np.int32)
    parent = (rng.random(V - 1) * child).astype(np.int32)
    return V, parent, child


def bipartite(a, b, E, seed):
    rng = np.random.default_rng(seed)
    src = rng.integers(0, a, E).astype(np.int32)
    dst = (a + rng.integers(0, b, E)).astype(np.int32)
    flip = rng.random(E) < 0.5
    return a + b, np.where(flip, dst, src), np.where(flip, src, dst)


def messy(V, E, seed):
    """random edges plus duplicates, self loops and reversed copies"""
    rng = np.random.default_rng(seed)
    src = rng.integers(0, V, E).astype(np.int32)
    dst = rng.integers(0, V, E).astype(np.int32)
    k = E // 4
    loops = rng.integers(0, V, k).astype(np.int32)
    src = np.concatenate([src, src[:k], dst[k:2 * k], loops])
    dst = np.concatenate([dst, dst[:k], src[k:2 * k], loops])
    return V, src, dst


# ---- CPU --------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("V,E,seed", [(1, 3, 1), (7, 20, 2), (40, 300, 3), (200, 3000, 4), (500, 20000, 5)])
def test_oracle_matches_scipy(tc_oracle, V, E, seed):
    V, src, dst = messy(V, E, seed)
    counts, total = _oracle_tc(tc_oracle, V, src, dst)
    ref, ref_total = _scipy_tc(V, src, dst)
    assert np.array_equal(counts, ref) and total == ref_total
    assert 3 * total == counts.sum()


@pytest.mark.parametrize("n", [3, 4, 10, 57])
def test_oracle_clique(tc_oracle, n):
    V, src, dst = clique(n)
    counts, total = _oracle_tc(tc_oracle, V, src, dst)
    assert total == n * (n - 1) * (n - 2) // 6
    assert np.all(counts == (n - 1) * (n - 2) // 2)


@pytest.mark.parametrize("n", [4, 5, 100])
def test_oracle_wheel(tc_oracle, n):
    V, src, dst = wheel(n)
    counts, total = _oracle_tc(tc_oracle, V, src, dst)
    assert total == n and counts[0] == n and np.all(counts[1:] == 2)


def test_oracle_no_triangles(tc_oracle):
    for V, src, dst in (random_tree(1000, 6), bipartite(300, 200, 5000, 7)):
        counts, total = _oracle_tc(tc_oracle, V, src, dst)
        assert total == 0 and not counts.any()


def test_null_arguments_fail_without_device(vgl):
    L = vgl.lib()
    buf = np.zeros(4, np.int64)
    assert L.vglb_tc(None, None, None, None, None) == 1  # VGLB_EINVAL
    assert b"NULL" in L.vglb_last_error()
    assert L.vglb_tc(None, None, buf.ctypes.data, buf.ctypes.data_as(vgl.C.POINTER(vgl.C.c_int64)), None) == 1
    assert b"NULL" in L.vglb_last_error()


# ---- GPU --------------------------------------------------------------------------------------------------------------

def _run(G):
    """(counts in ORIGINAL numbering, total, stats)"""
    c, total, st = G.tc()
    counts = c.to_numpy()[G.orig_to_sorted()]
    c.free()
    assert 3 * total == counts.sum()
    return counts, total, st


def _check(vgl, ctx, L, V, src, dst, flags=0):
    G = vgl.Graph.from_edges(ctx, V, src, dst, flags)
    counts, total, _ = _run(G)
    G.free()
    ref, ref_total = _oracle_tc(L, V, src, dst)
    assert total == ref_total and np.array_equal(counts, ref), (total, ref_total, int(np.abs(counts - ref).max()))
    return counts, total


@gpu
def test_golden_fixtures(vgl, ctx, oracle, tc_oracle, golden):
    name, g = golden
    src, dst = oracle.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))
    _check(vgl, ctx, tc_oracle, 1 << int(g["scale"]), src, dst)


@gpu
@pytest.mark.parametrize("kind,scale,ef", [(0, 16, 16), (1, 15, 16), (2, 14, 32)])
def test_generators(vgl, ctx, oracle, tc_oracle, kind, scale, ef):
    src, dst = oracle.generate_edges(kind, scale, ef, 0x7C00 + scale)
    _, total = _check(vgl, ctx, tc_oracle, 1 << scale, src, dst)
    assert total > 0


@gpu
@pytest.mark.parametrize("kind,ef", [(0, 16), (2, 32)])
def test_scale_20(vgl, ctx, oracle, tc_oracle, kind, ef):
    src, dst = oracle.generate_edges(kind, 20, ef)
    _check(vgl, ctx, tc_oracle, 1 << 20, src, dst)


@gpu
def test_clique_past_the_staging_buffer(vgl, ctx):
    n = TC_STAGE + 52  # rows 2049 .. 2099 of the oriented CSR hold more entries than a staging buffer
    V, src, dst = clique(n)
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    counts, total, st = _run(G)
    G.free()
    assert total == n * (n - 1) * (n - 2) // 6
    assert np.all(counts == (n - 1) * (n - 2) // 2)  # 2.2 million per vertex


@gpu
def test_wheel_hub(vgl, ctx):
    n = 1_000_000
    V, src, dst = wheel(n)
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    assert G.orig_to_sorted()[0] == 0  # the hub is SCATTER id 0: its oriented row is empty, it is every triangle's w
    counts, total, _ = _run(G)
    G.free()
    assert total == n and counts[0] == n and np.all(counts[1:] == 2)


@gpu
def test_no_triangles_and_no_edges(vgl, ctx):
    for V, src, dst in (random_tree(100_000, 8), bipartite(30_000, 20_000, 400_000, 9)):
        G = vgl.Graph.from_edges(ctx, V, src, dst)
        counts, total, st = _run(G)
        G.free()
        assert total == 0 and not counts.any() and st.edges_inspected > 0
    e = np.empty(0, np.int32)
    G = vgl.Graph.from_edges(ctx, 64, e, e, vgl.GRAPH_WITH_INCOMING)
    counts, total, st = _run(G)
    G.free()
    assert total == 0 and not counts.any()
    assert st.iterations == 1 and st.edges_inspected == 0 and st.vertices_processed == 0 and st.algorithmic_bytes == 16 * 64


@gpu
def test_small_vertex_counts(vgl, ctx, tc_oracle):
    one = np.zeros(2, np.int32)  # V = 1: two self loops
    G = vgl.Graph.from_edges(ctx, 1, one, one)
    counts, total, _ = _run(G)
    G.free()
    assert total == 0 and counts.tolist() == [0]
    for V, E, seed in ((3, 3, 10), (1000, 30_000, 11), (4099, 200_000, 12)):
        V, src, dst = messy(V, E, seed)
        _check(vgl, ctx, tc_oracle, V, src, dst)
    _check(vgl, ctx, tc_oracle, *clique(3))


@gpu
def test_same_graph_six_ways(vgl, ctx, oracle, tc_oracle, tmp_path):
    """(src, dst), (dst, src), the symmetrised list, extra duplicates and self loops, WITH_INCOMING, from_csr, load_vgl"""
    V = 1 << 14
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, 14, 16, 0x7C11)
    ref, ref_total = _check(vgl, ctx, tc_oracle, V, src, dst)
    rng = np.random.default_rng(13)
    pick = rng.integers(0, len(src), len(src) // 3)
    loops = rng.integers(0, V, 5000).astype(np.int32)
    variants = [(dst, src, 0), (np.concatenate([src, dst]), np.concatenate([dst, src]), 0),
                (np.concatenate([src, dst[pick], src[pick], loops]), np.concatenate([dst, src[pick], dst[pick], loops]), 0),
                (src, dst, vgl.GRAPH_WITH_INCOMING)]
    for s, d, flags in variants:
        G = vgl.Graph.from_edges(ctx, V, s, d, flags)
        counts, total, _ = _run(G)
        G.free()
        assert total == ref_total and np.array_equal(counts, ref)
    G0 = vgl.Graph.from_edges(ctx, V, src, dst)
    ptr, adj = G0.layout()
    G = vgl.Graph.from_csr(ctx, ptr, adj, G0.orig_to_sorted())
    G0.free()
    counts, total, _ = _run(G)
    G.free()
    assert total == ref_total and np.array_equal(counts, ref)
    path = str(tmp_path / "g.vgl")
    vgl.save_vgl(ctx, path, V, src, dst)
    G = vgl.Graph.load_vgl(ctx, path)
    counts, total, _ = _run(G)
    G.free()
    assert total == ref_total and np.array_equal(counts, ref)


@gpu
def test_determinism(vgl, ctx, oracle):
    V = 1 << 16
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, 16, 16, 0x7C12)
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    c1, t1, _ = G.tc()
    c2, t2, _ = G.tc()
    assert t1 == t2 and c1.to_numpy().tobytes() == c2.to_numpy().tobytes()
    G.free()


@gpu
def test_partitioned_graph_rejected(vgl, ctx, oracle):
    V = 1 << 10
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, 10, 8, 0x7C13)
    comm = vgl.Comm(ctx, 0, 2, detached=True)
    P = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst)
    with pytest.raises(vgl.VglbError, match=r"\[vglb error 1\].*partitioned"):
        P.tc()
    P.free()
    comm.close()


def oriented_stats(V, ptr, adj):
    """numpy restatement of the oriented CSR and the kernel's per-edge rule on a SCATTER-numbered CSR:
    (E+, rows with entries, list elements read = sum over oriented edges (u, v) at position j of j when 2 j < |N+(v)|,
    else |N+(v)|)"""
    rows = np.repeat(np.arange(V, dtype=np.int64), np.diff(ptr))
    a = np.asarray(adj, np.int64)
    keep = rows != a
    hi, lo = np.maximum(rows, a)[keep], np.minimum(rows, a)[keep]
    key = np.unique(hi * V + lo)
    u, v = key // V, key % V
    n_plus = np.bincount(u, minlength=V)
    start = np.zeros(V + 1, np.int64)
    np.cumsum(n_plus, out=start[1:])
    j = np.arange(len(key)) - start[u]
    return len(key), int((n_plus > 0).sum()), int(np.where(2 * j < n_plus[v], j, n_plus[v]).sum())


@gpu
@pytest.mark.parametrize("kind,scale,ef", [(0, 14, 16), (2, 13, 32)])
def test_stats(vgl, ctx, oracle, kind, scale, ef):
    V = 1 << scale
    src, dst = oracle.generate_edges(kind, scale, ef, 0x7C14)
    src = np.concatenate([src, src[:100]])  # duplicates and self loops
    dst = np.concatenate([dst, src[:100]])
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    ptr, adj = G.layout()
    e_plus, rows, elems = oriented_stats(V, ptr, adj)
    _, _, st = G.tc()
    assert st.iterations == 1
    assert st.edges_inspected == elems and st.vertices_processed == rows
    assert st.algorithmic_bytes == 8 * G.E + 12 * e_plus + 4 * elems + 16 * V
    assert st.kernel_launches >= 1 and st.seconds > 0
    G.free()
