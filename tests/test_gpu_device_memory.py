"""Device memory of graph set-up, preparation and verification: every temporary block goes back to the allocation cache,
when a call succeeds and when it rejects its input. The count of live blocks comes from `vglb_dev_live_blocks`, a test hook
of context.cu that is not part of the public header."""
import ctypes as C
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _live(vgl):
    gc.collect()  # DeviceArrays of earlier tests free their blocks when they are collected
    blocks, nbytes = C.c_int64(), C.c_int64()
    assert vgl.lib().vglb_dev_live_blocks(C.byref(blocks), C.byref(nbytes)) == 0
    return blocks.value, nbytes.value


def _rejected(vgl, baseline, call, match, repeats=3):
    for _ in range(repeats):
        with pytest.raises(vgl.VglbError, match=match):
            call()
        assert _live(vgl) == baseline


def test_rejected_input_leaves_no_block_behind(vgl, ctx, oracle):
    scale, ef = 10, 8
    V = 1 << scale
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, scale, ef)
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    ptr, adj = G.layout()
    fwd = G.orig_to_sorted()
    G.free()
    assert ptr[1] < ptr[2]
    bad_ptr = ptr.copy()
    bad_ptr[1], bad_ptr[2] = ptr[2], ptr[1]
    bad_adj = adj.copy()
    bad_adj[0] = V
    bad_fwd = fwd.copy()
    bad_fwd[1] = fwd[0]
    bad_dst = dst.copy()
    bad_dst[len(dst) // 2] = V
    # a CSR that passes every check but is not degree-sorted: rejected after the whole upload
    unsorted_ptr = np.array([0, 1, 3, 3], np.int64)
    unsorted_adj = np.array([1, 0, 2], np.int32)
    labels = ctx.from_numpy(np.arange(V, dtype=np.int32))
    bad_labels = ctx.from_numpy(np.full(V, V + 5, np.int32))
    comm = vgl.Comm(ctx, 0, 1)
    P = vgl.Graph.from_edges_partitioned(ctx, comm, V, src, dst)
    pptr, padj = P.layout()
    pfwd = P.orig_to_sorted()
    P.free()
    bad_padj = padj.copy()
    bad_padj[0] = P.cols

    baseline = _live(vgl)
    _rejected(vgl, baseline, lambda: vgl.Graph.from_edges(ctx, V, src, bad_dst), "out of range")
    _rejected(vgl, baseline, lambda: vgl.Graph.from_edges(ctx, V, src, bad_dst, vgl.GRAPH_WITH_INCOMING), "out of range")
    for p, a, f in ((bad_ptr, adj, fwd), (ptr, bad_adj, fwd), (ptr, adj, bad_fwd)):
        _rejected(vgl, baseline, lambda: vgl.Graph.from_csr(ctx, p, a, f), "not a CSR")
    _rejected(vgl, baseline, lambda: vgl.Graph.from_csr(ctx, ptr, adj, fwd, bad_ptr, adj), "not a CSR")
    _rejected(vgl, baseline, lambda: vgl.Graph.from_csr(ctx, unsorted_ptr, unsorted_adj), "not sorted by degree")
    _rejected(vgl, baseline, lambda: vgl.Graph.from_csr_partitioned(ctx, comm, V, pptr, bad_padj, pfwd),
              "this rank's part is not a CSR")
    _rejected(vgl, baseline, lambda: vgl.equal_components(ctx, labels, bad_labels), "labels must lie")

    # the partitioned upload that succeeds, and its reorder (which allgathers through a temporary)
    H = vgl.Graph.from_csr_partitioned(ctx, comm, V, pptr, padj, pfwd)
    rows = ctx.from_numpy(np.arange(H.V, dtype=np.int32))
    orig = H.reorder(rows, vgl.SCATTER, vgl.ORIGINAL)
    assert sorted(orig.to_numpy().tolist()) == list(range(V))
    for x in (orig, rows):
        x.free()
    H.free()
    assert _live(vgl) == baseline
    comm.close()
    labels.free()
    bad_labels.free()


def test_graph_lifetime_leaves_no_block_behind(vgl, ctx, oracle, tmp_path):
    scale, ef = 12, 8
    V = 1 << scale
    src, dst = oracle.generate_edges(oracle.GEN_RMAT, scale, ef, 0x5E)
    s2, d2 = oracle.symmetrize(src, dst)
    path = str(tmp_path / "g.vgl")
    baseline = _live(vgl)
    for flags in (0, vgl.GRAPH_WITH_INCOMING):
        G = vgl.Graph.from_edges(ctx, V, s2, d2, flags)
        arrays = [G.pagerank(5)[0], G.pagerank(5, reference_threads=8)[0], G.bfs(0)[0], G.bfs(0, False)[0],
                  G.bfs_multi([0, 1, 2])[0], G.cc()[0]]
        w = G.synthetic_weights(7)
        arrays += [w, G.sssp(w, 0)[0], G.mirror_out_to_in(w)]
        arrays.append(G.reorder(arrays[0], vgl.SCATTER, vgl.ORIGINAL))
        arrays.append(G.reorder(arrays[-1], vgl.ORIGINAL, vgl.SCATTER))
        for a in arrays:
            a.free()
        G.free()
        assert _live(vgl) == baseline
    vgl.save_vgl(ctx, path, V, src, dst)
    assert _live(vgl) == baseline
    L = vgl.Graph.load_vgl(ctx, path, vgl.GRAPH_WITH_INCOMING)
    ranks = L.pagerank(5)[0]
    ranks.free()
    L.free()
    assert _live(vgl) == baseline
