"""The reference's on-disk formats (csrc/graph_io.cu): files written by libvgl_b200 must be byte-identical to the ones
the unmodified reference writes, and load into the reference; files written by the reference must load into the device
layout and give the reference's results. (.el_container: edges_container.h:58-99; .vgl: vgl_graph.hpp:109-161,
vect_csr_graph.hpp:141-180.) The reference's files are compared with as the reference writes them where oracle/_ref is
built, and otherwise as assembled from its layouts frozen in tests/golden/; the reference reading our files needs
oracle/_ref."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _have_ref(oracle):
    """oracle/_ref (the reference built with its file-format entry points) is present: its writer and reader run live."""
    return oracle.ref_available("bfs") and hasattr(oracle.ref_lib("bfs"), "vglref_graph_save")


def _reference_el_container(V, src, dst):
    """The bytes EdgesContainer::save_to_binary_file writes (edges_container.h:58-76): int32 V, int64 E, int32 4
    (EDGES_CONTAINER), int32 src[E], int32 dst[E]."""
    return (np.int32(V).tobytes() + np.int64(len(src)).tobytes() + np.int32(4).tobytes()
            + np.ascontiguousarray(src, "<i4").tobytes() + np.ascontiguousarray(dst, "<i4").tobytes())


def _reference_vgl_file(oracle, g, V, src, dst):
    """The bytes VGL_Graph::save_to_binary_file writes for a golden case (vgl_graph.hpp:109-161, vect_csr_graph.hpp:141-180),
    assembled from the reference's own layouts stored in the fixture (row pointers, adjacency and ORIGINAL -> sorted maps of
    both containers). The per-edge order arrays are the oracle's import order, which test_io_cpu.py pins against a file the
    reference wrote: the outgoing import of the edge list, and the incoming import of its transpose in outgoing-CSR order."""
    E = len(src)
    og = oracle.OracleGraph(V, src, dst, want_edge_order=True)
    assert np.array_equal(og.row_ptr, g["out_ptr"]) and np.array_equal(og.adj, g["out_adj"]) and np.array_equal(og.fwd, g["out_fwd"])
    rows = np.repeat(np.arange(V, dtype=np.int32), np.diff(og.row_ptr))
    ig = oracle.OracleGraph(V, og.bwd[og.adj], og.bwd[rows], want_edge_order=True)
    assert np.array_equal(ig.row_ptr, g["in_ptr"]) and np.array_equal(ig.adj, g["in_adj"]) and np.array_equal(ig.fwd, g["in_fwd"])

    def container(ptr, adj, fwd, edge_order):
        bwd = np.empty(V, np.int32)
        bwd[fwd] = np.arange(V, dtype=np.int32)
        return (np.int32(V).tobytes() + np.int64(E).tobytes() + np.int32(1).tobytes() + np.ascontiguousarray(ptr, "<i8").tobytes()
                + np.ascontiguousarray(adj, "<i4").tobytes() + np.ascontiguousarray(fwd, "<i4").tobytes() + bwd.tobytes()
                + np.ascontiguousarray(edge_order, "<i8").tobytes())

    return (np.int32(V).tobytes() + np.int64(E).tobytes() + np.int32(1).tobytes()
            + container(g["out_ptr"], g["out_adj"], g["out_fwd"], og.edge_order)
            + container(g["in_ptr"], g["in_adj"], g["in_fwd"], ig.edge_order))


def test_el_container_round_trip(vgl, ctx, oracle, golden, tmp_path):
    name, g = golden
    src, dst = oracle.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))
    V = 1 << int(g["scale"])
    ours = str(tmp_path / "ours.el_container")
    vgl.save_el_container(ours, V, src, dst)
    raw = open(ours, "rb").read()
    assert len(raw) == 16 + 8 * len(src)
    assert np.frombuffer(raw[:4], "<i4")[0] == V and np.frombuffer(raw[4:12], "<i8")[0] == len(src) and np.frombuffer(raw[12:16], "<i4")[0] == 4
    G = vgl.Graph.import_el_container(ctx, ours, vgl.GRAPH_WITH_INCOMING)
    ptr, adj = G.layout()
    assert np.array_equal(ptr, g["out_ptr"]) and np.array_equal(adj, g["out_adj"]) and np.array_equal(G.orig_to_sorted(), g["out_fwd"])
    fwd = G.orig_to_sorted()
    lv, _ = G.bfs(int(fwd[int(g["sources"][0])]), True)
    assert np.array_equal(G.to_original(lv), g["bfs_levels"][0])
    G.free()
    with pytest.raises(vgl.VglbError):
        vgl.Graph.import_el_container(ctx, str(tmp_path / "missing.el_container"))
    bad = str(tmp_path / "bad.el_container")
    open(bad, "wb").write(raw[:12] + np.int32(1).tobytes() + raw[16:])
    with pytest.raises(vgl.VglbError, match="incorrect type of graph"):
        vgl.Graph.import_el_container(ctx, bad)
    open(bad, "wb").write(raw[:-8])
    with pytest.raises(vgl.VglbError, match="truncated"):
        vgl.Graph.import_el_container(ctx, bad)


def test_el_container_matches_reference_writer_and_reader(vgl, ctx, oracle, golden, tmp_path):
    name, g = golden
    src, dst = oracle.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))
    V = 1 << int(g["scale"])
    ours, theirs = str(tmp_path / "ours.el_container"), str(tmp_path / "ref.el_container")
    vgl.save_el_container(ours, V, src, dst)
    expected = _reference_el_container(V, src, dst)
    if _have_ref(oracle):
        oracle.ref_save_edges(theirs, V, src, dst)
        assert open(theirs, "rb").read() == expected
    assert open(ours, "rb").read() == expected
    if not _have_ref(oracle):
        return
    rg = oracle.RefGraph.from_edges_file(ours)  # the reference imports OUR file
    ptr, adj, fwd, _, _ = rg.layout(0)
    assert np.array_equal(ptr, g["out_ptr"]) and np.array_equal(adj, g["out_adj"]) and np.array_equal(fwd, g["out_fwd"])
    rg.close()


def test_vgl_graph_file_byte_identical_and_loadable_both_ways(vgl, ctx, oracle, golden, tmp_path):
    name, g = golden
    src, dst = oracle.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))
    V = 1 << int(g["scale"])
    ours, theirs = str(tmp_path / "ours.vgl"), str(tmp_path / "ref.vgl")
    vgl.save_vgl(ctx, ours, V, src, dst)
    expected = _reference_vgl_file(oracle, g, V, src, dst)
    if _have_ref(oracle):
        rg = oracle.RefGraph(V, src, dst, "bfs")
        rg.save(theirs)
        rg.close()
        assert open(theirs, "rb").read() == expected
    else:
        open(theirs, "wb").write(expected)
    a, b = open(ours, "rb").read(), open(theirs, "rb").read()
    assert len(a) == len(b) == 16 + 2 * (16 + 8 * (V + 1) + 4 * len(src) + 8 * V + 8 * len(src))
    assert a == b, "VGL graph file differs from the reference's at byte %d" % next(i for i in range(len(a)) if a[i] != b[i])
    s0 = int(g["sources"][0])
    if _have_ref(oracle):
        # the reference loads OUR file and runs its own BFS on it
        rl = oracle.RefGraph.load(ours)
        assert (rl.V, rl.E) == (V, len(src))
        assert np.array_equal(rl.bfs(s0, 0)[0], g["bfs_levels"][0])
        rl.close()
    # we load THEIR file (and one written with device-resident edges) into the device layout
    also = str(tmp_path / "ours_dev.vgl")
    vgl.save_vgl(ctx, also, V, ctx.from_numpy(src), ctx.from_numpy(dst))
    assert open(also, "rb").read() == b
    G = vgl.Graph.load_vgl(ctx, theirs, vgl.GRAPH_WITH_INCOMING)
    ptr, adj = G.layout()
    assert np.array_equal(ptr, g["out_ptr"]) and np.array_equal(adj, g["out_adj"]) and np.array_equal(G.orig_to_sorted(), g["out_fwd"])
    H = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    for x, y in zip(G.layout(incoming=True), H.layout(incoming=True)):
        assert np.array_equal(x, y)  # the derived incoming direction equals the builder's
    fwd = G.orig_to_sorted()
    for dopt in (False, True):
        lv, _ = G.bfs(int(fwd[s0]), dopt)
        assert np.array_equal(G.to_original(lv), g["bfs_levels"][0])
    ranks, _ = G.pagerank(int(g["pr_iters"]))
    assert oracle.rel_l1(G.to_original(ranks), g["pr_ranks"]) <= 1e-6
    G.free(); H.free()
    with pytest.raises(vgl.VglbError):
        vgl.Graph.load_vgl(ctx, str(tmp_path / "ours.el_container"))
