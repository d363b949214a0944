"""The drop-in boundary, tested the way north_star states it: "the user-lambda operator API and the algorithms/* call sites
stay unchanged".

oracle/_ref/libvgl_dropin.so is oracle/ref_gpu_harness.cu compiled (by build() where the reference tree is present,
oracle/Makefile REF) with `-D __USE_GPU__` against the UNMODIFIED reference tree — its graph_library.h, its data structures and its
algorithms/bfs/bfs.hpp, pr/gpu_pr.hpp, sssp/gpu_shortest_paths.hpp, cc/gpu_shiloach_vishkin.hpp, hits/hits.hpp — with
include/vgl_b200/overlay first on the include path, so that `vgl_compute_api/gpu/graph_abstractions_gpu.h` resolves to this
repo's B200 backend. Every result below is therefore produced by the reference's own algorithm source running on
libvgl_b200's operators (advance / compute / reduce / generate_new_frontier), and is compared with the CPU oracle.
libvgl_refgpu.so is the same harness on the reference's own CUDA backend (recompiled for sm_100a): a cross-check and a baseline.
The reference's sources are not part of this repository, so without a checkout of them these tests skip.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

CASES = [(0, 14, 16, 0xD1), (1, 13, 16, 0xD2), (2, 12, 32, 0xD3)]  # RMAT, Kronecker, uniform


def _textbook_pagerank_f64(V, src, dst, iters, push):
    """gpu_pr.hpp:7-175 restated in fp64. PULL (the reference's default): r'[v] = k + d (sum_{u->v, u != v} r[u] / outdeg_nl(u) + D),
    D = sum_{outdeg_nl(u) = 0} r[u] / V. PUSH: the same with the in-degree without loops as the normaliser (SURVEY App. A.12)."""
    keep = src != dst
    s, t = src[keep], dst[keep]
    norm = np.bincount(t if push else s, minlength=V).astype(np.float64)
    inv = np.divide(1.0, norm, out=np.zeros(V), where=norm > 0)
    d = float(np.float32(0.85))
    k = (1.0 - d) / V
    r = np.full(V, 1.0 / V)
    for _ in range(iters):
        dangling = r[norm == 0].sum() / V
        acc = np.bincount(t, weights=(r * inv)[s], minlength=V)
        r = k + d * (acc + dangling)
    return r


@pytest.fixture(scope="module")
def dropin(oracle):
    if not oracle.gpu_ref_available("dropin"):
        pytest.skip("oracle/_ref/libvgl_dropin.so not built: it compiles the reference's algorithm sources against "
                    "include/vgl_b200/overlay, and build() makes it only where the reference tree (oracle/Makefile REF) is present")
    return oracle


@pytest.mark.parametrize("kind,scale,ef,seed", CASES)
def test_reference_algorithms_on_b200_backend(dropin, kind, scale, ef, seed):
    O = dropin
    V = 1 << scale
    src, dst = O.generate_edges(kind, scale, ef, seed)
    og = O.OracleGraph(V, src, dst)
    G = O.GpuRefGraph(V, src, dst, "dropin")
    outdeg = np.bincount(src, minlength=V)
    for s in O.pick_sources(V, outdeg, 2, seed):
        lv, _ = G.bfs(s)                                         # BFS::vgl_top_down (bfs.hpp), scatter + generate_new_frontier
        assert np.array_equal(lv, og.bfs(s)[0]), "BFS levels"
        ref_d = og.sssp(s, seed ^ 0x5555)[0].view(np.uint32)
        for mode in (2, 0, 1):                                   # partial-active (GNF + add_vertex), all-active push, all-active pull
            d, _ = G.sssp(s, seed ^ 0x5555, mode)
            assert np.array_equal(d.view(np.uint32), ref_d), f"SSSP mode {mode}"
    lab, _ = G.cc()                                              # gpu_shiloach_vishkin.hpp: scatter + compute, host-read managed flags
    assert np.array_equal(lab, og.cc()[0]), "CC labels"
    for push in (False, True):                                   # gpu_pr.hpp: compute, reduce<double>, gather / scatter with atomics
        r, _ = G.pagerank(20, push)
        ref = _textbook_pagerank_f64(V, src, dst, 20, push)
        assert O.rel_l1(r, ref) <= 1e-6, ("PageRank", push, O.rel_l1(r, ref))
    G.close()


def test_non_core_algorithm_hits_on_b200_backend(dropin):
    """HITS (algorithms/hits/hits.hpp) is not one of the four: 8-functor gather and scatter with vertex pre-ops, both traversal
    directions inside one run, reduce<float> and compute — checked against the reference's own HITS::seq_hits."""
    O = dropin
    V = 1 << 13
    src, dst = O.generate_edges(O.GEN_RMAT, 13, 16, 0xE1)
    G = O.GpuRefGraph(V, src, dst, "dropin")
    a, h, sa, sh, _ = G.hits(5)
    assert np.isfinite(a).all() and np.isfinite(h).all()
    assert O.rel_l1(a, sa) <= 1e-5 and O.rel_l1(h, sh) <= 1e-5, (O.rel_l1(a, sa), O.rel_l1(h, sh))
    G.close()


def test_add_group_of_vertices_on_b200_backend(dropin):
    """frontier.add_group_of_vertices (modification.hpp:88-145) is the reference's own host code; the backend has to pick the
    list up (tiers, neighbour count) — compute and reduce over it."""
    O = dropin
    V = 1 << 12
    src, dst = O.generate_edges(O.GEN_RMAT, 12, 8, 0xE2)
    G = O.GpuRefGraph(V, src, dst, "dropin")
    rng = np.random.default_rng(3)
    outdeg = np.bincount(src, minlength=V)
    ids = rng.choice(V, 700, replace=False).astype(np.int32)
    ids[:3] = np.argsort(-outdeg)[:3]  # the hubs are part of the group
    ids = np.unique(ids)
    marks, total = G.group_mark(ids)
    expect = np.zeros(V, np.int32)
    expect[ids] = 7
    assert np.array_equal(marks, expect)
    assert total == int(outdeg[ids].sum())
    G.close()


def test_b200_backend_next_to_reference_cuda_backend(dropin):
    """The same harness on the reference's own CUDA backend (recompiled for sm_100a, oracle/_ref/libvgl_refgpu.so). Its sparse
    path is sound, so BFS levels must be identical. Its ALL_ACTIVE VectorCSR advance processes the wrong vertices for the vc and
    collective tiers (`_sparse_mode = false` makes src_id start at 0 instead of the tier offset, gpu/advance_vect_csr.hpp:96-122;
    SURVEY §2.3) — PageRank from it is therefore NOT the recurrence of gpu_pr.hpp, which is why the B200 backend is checked
    against the fp64 restatement and the reference backend's distance from it is only reported."""
    O = dropin
    if not O.gpu_ref_available("refgpu"):
        pytest.skip("oracle/_ref/libvgl_refgpu.so not built")
    V = 1 << 13
    src, dst = O.generate_edges(O.GEN_KRONECKER, 13, 16, 0xE3)
    A, B = O.GpuRefGraph(V, src, dst, "dropin"), O.GpuRefGraph(V, src, dst, "refgpu")
    s = O.pick_sources(V, np.bincount(src, minlength=V), 1, 0xE3)[0]
    assert np.array_equal(A.bfs(s)[0], B.bfs(s)[0])
    truth = _textbook_pagerank_f64(V, src, dst, 10, False)
    ra, rb = A.pagerank(10)[0], B.pagerank(10)[0]
    print("PageRank rel-L1 vs the fp64 restatement of gpu_pr.hpp: B200 backend %.2e, reference CUDA backend %.2e"
          % (O.rel_l1(ra, truth), O.rel_l1(rb, truth)))
    assert O.rel_l1(ra, truth) <= 1e-6
    A.close(); B.close()
