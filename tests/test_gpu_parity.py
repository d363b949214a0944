"""GPU parity (through the C ABI of libvgl_b200.so) against the frozen reference fixtures (tests/golden/, produced by
the unmodified reference) and against the C oracle on fresh seeded inputs.

Bars (BASELINE.json north_star): bit-exact VectCSR layout, BFS levels, SSSP distances (uint32 view) and CC labels;
PageRank <= 1e-6 relative L1 against the reference's multicore result (and the fp64 restatement for attribution)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

PR_TOL = 1e-6  # north_star: "PageRank within 1e-6 relative L1"


def _edges(O, g):
    return O.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))


def _incoming_on_scatter_numbering(ptr, adj):
    """Expected in-CSR on the SAME numbering as the out-CSR: stable sort of the out-CSR positions by destination."""
    V = len(ptr) - 1
    row_of_pos = np.repeat(np.arange(V, dtype=np.int32), np.diff(ptr))
    order = np.argsort(adj, kind="stable")
    in_ptr = np.zeros(V + 1, np.int64)
    np.cumsum(np.bincount(adj, minlength=V), out=in_ptr[1:])
    return in_ptr, row_of_pos[order]


# ---------------------------------------------------------------------------------------------------------------------
# golden fixtures (outputs of the unmodified reference)
# ---------------------------------------------------------------------------------------------------------------------

def test_builder_layout_matches_reference(vgl, ctx, oracle, golden):
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    for on_device in (False, True):
        if on_device:
            dsrc, ddst = ctx.generate_edges(int(g["kind"]), int(g["scale"]), int(g["edge_factor"]), int(g["seed"]))
            assert np.array_equal(dsrc.to_numpy(), src) and np.array_equal(ddst.to_numpy(), dst)
            G = vgl.Graph.from_edges(ctx, V, dsrc, ddst, vgl.GRAPH_WITH_INCOMING | vgl.GRAPH_WITH_EDGE_ORDER)
        else:
            G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING | vgl.GRAPH_WITH_EDGE_ORDER)
        ptr, adj = G.layout()
        assert np.array_equal(ptr, g["out_ptr"])
        assert np.array_equal(adj, g["out_adj"])
        assert np.array_equal(G.orig_to_sorted(), g["out_fwd"])
        assert np.array_equal(G.sorted_to_orig()[g["out_fwd"]], np.arange(V))
        iptr, iadj = G.layout(incoming=True)
        eptr, eadj = _incoming_on_scatter_numbering(ptr, adj)
        assert np.array_equal(iptr, eptr) and np.array_equal(iadj, eadj)
        eo = G._d2h(G.info.d_edge_order, G.E, np.int64)
        og = oracle.OracleGraph(V, src, dst, want_edge_order=True)
        assert np.array_equal(eo, og.edge_order)
        # tiers: border[t] = number of rows with degree >= tier_degree[t]
        deg = np.diff(ptr)
        td, tb = G.tiers()
        for t in range(vgl.NUM_TIERS - 1):
            assert tb[t] == int((deg >= td[t]).sum())
        assert tb[-1] == V
        assert G.threshold_vertex(64) == og.thresholds(1 << 30, 64)[1]
        G.free()


@pytest.mark.parametrize("dopt", [False, True])
def test_bfs_levels_bit_exact(vgl, ctx, oracle, golden, dopt):
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    fwd = G.orig_to_sorted()
    for i, s in enumerate(g["sources"]):
        lv, st = G.bfs(int(fwd[int(s)]), direction_optimising=dopt)
        assert np.array_equal(G.to_original(lv), g["bfs_levels"][i])
        assert st.iterations >= 1 and st.kernel_launches >= st.iterations
        lv.free()
    G.free()


def test_sssp_bit_exact(vgl, ctx, oracle, golden):
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    og = oracle.OracleGraph(V, src, dst)
    w = G.synthetic_weights(int(g["weight_seed"]))
    assert np.array_equal(w.to_numpy().view(np.uint32), og.weights(int(g["weight_seed"])).view(np.uint32))
    fwd = G.orig_to_sorted()
    for i, s in enumerate(g["sources"]):
        d, st = G.sssp(w, int(fwd[int(s)]))
        assert np.array_equal(G.to_original(d).view(np.uint32), g["sssp_dist"][i].view(np.uint32))
        d.free()
    G.free()


def test_cc_labels_bit_exact(vgl, ctx, oracle, golden):
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    lab, st = G.cc()
    assert np.array_equal(G.to_original(lab), g["cc_directed"])
    G.free()
    s2, d2 = oracle.symmetrize(src, dst)
    G2 = vgl.Graph.from_edges(ctx, V, s2, d2)
    lab2, st2 = G2.cc()
    assert np.array_equal(G2.to_original(lab2), g["cc_symmetric"])
    G2.free()


def test_pagerank_within_tolerance(vgl, ctx, oracle, golden):
    name, g = golden
    src, dst = _edges(oracle, g)
    V = 1 << int(g["scale"])
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    ranks, st = G.pagerank(int(g["pr_iters"]))
    r = G.to_original(ranks)
    og = oracle.OracleGraph(V, src, dst)
    assert oracle.rel_l1(r, g["pr_ranks"]) <= PR_TOL                      # the contract: vs the reference's own output
    assert oracle.rel_l1(r, og.pagerank_f64(int(g["pr_iters"]))) <= PR_TOL  # attribution: vs fp64 truth
    assert st.iterations == int(g["pr_iters"]) and st.kernel_launches >= int(g["pr_iters"]) + 1
    G.free()


# ---------------------------------------------------------------------------------------------------------------------
# fresh seeded inputs against the C oracle (sizes the oracle finishes in seconds)
# ---------------------------------------------------------------------------------------------------------------------

FRESH = [(0, 16, 16, 0xA1), (1, 15, 16, 0xA2), (2, 14, 32, 0xA3), (0, 13, 1, 0xA4)]


@pytest.mark.parametrize("kind,scale,ef,seed", FRESH)
def test_all_algorithms_vs_oracle(vgl, ctx, oracle, kind, scale, ef, seed):
    O = oracle
    V = 1 << scale
    src, dst = O.generate_edges(kind, scale, ef, seed)
    og = O.OracleGraph(V, src, dst)
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    ptr, adj = G.layout()
    assert np.array_equal(ptr, og.row_ptr) and np.array_equal(adj, og.adj)
    fwd = G.orig_to_sorted()
    assert np.array_equal(fwd, og.fwd)
    outdeg = np.bincount(src, minlength=V)
    w = G.synthetic_weights(seed ^ 0x5555)
    for s in O.pick_sources(V, outdeg, 3, seed):
        ref_lv, _ = og.bfs(s)
        for dopt in (False, True):
            lv, st = G.bfs(int(fwd[s]), direction_optimising=dopt)
            assert np.array_equal(G.to_original(lv), ref_lv), (s, dopt)
            lv.free()
        ref_d, _ = og.sssp(s, seed ^ 0x5555)
        d, st = G.sssp(w, int(fwd[s]))
        assert np.array_equal(G.to_original(d).view(np.uint32), ref_d.view(np.uint32))
        d.free()
    lab, _ = G.cc()
    assert np.array_equal(G.to_original(lab), og.cc()[0])
    # PageRank, the three numbers of SURVEY §8c. The reference sums the dangling mass in fp32 over T static chunks, which
    # moves its result away from the exact recurrence by far more than the tolerance (1.6e-5 at scale 16, growing with V);
    # the contract "within 1e-6 of the reference" is met by the reference-order mode (same chunked fp32 dangling sum),
    # the default mode is within 1e-6 of the exact (fp64) recurrence instead.
    T = 8
    r64 = og.pagerank_f64(20)
    r32 = og.pagerank_f32(20, T)                    # C port of the reference's fp32 evaluation order at T threads
    ranks, _ = G.pagerank(20)
    assert O.rel_l1(G.to_original(ranks), r64) <= PR_TOL
    ranks_ref, _ = G.pagerank(20, reference_threads=T)
    r = G.to_original(ranks_ref)
    numbers = {"ours_vs_reference": O.rel_l1(r, r32), "ours_default_vs_fp64": O.rel_l1(G.to_original(ranks), r64),
               "reference_vs_fp64": O.rel_l1(r32, r64)}
    print("PageRank rel-L1", kind, scale, numbers)
    assert numbers["ours_vs_reference"] <= PR_TOL, numbers
    if O.ref_available("pr"):                       # the unmodified reference itself, same thread count
        import os
        assert int(os.environ.get("OMP_NUM_THREADS", "0")) == T
        rg = O.RefGraph(V, src, dst, "pr")
        assert rg.threads() == T
        rr, _ = rg.pagerank(20)
        rg.close()
        assert O.rel_l1(r, rr) <= PR_TOL, ("vs the unmodified reference", O.rel_l1(r, rr), numbers)
    G.free()


def test_cc_symmetric_vs_oracle(vgl, ctx, oracle):
    O = oracle
    V = 1 << 15
    src, dst = O.generate_edges(O.GEN_RMAT, 15, 4, 0xC0)
    s2, d2 = O.symmetrize(src, dst)
    og = O.OracleGraph(V, s2, d2)
    G = vgl.Graph.from_edges(ctx, V, s2, d2)
    lab, st = G.cc()
    got = G.to_original(lab)
    assert np.array_equal(got, og.cc()[0])
    # component minimum in sorted numbering (verify_results.h:197-254 equal_components is implied by label equality)
    assert np.all(lab.to_numpy() <= np.arange(V))
    G.free()


# ---------------------------------------------------------------------------------------------------------------------
# edge cases the reference's checks cover: empty / ragged inputs, isolated sources, self loops, duplicates
# ---------------------------------------------------------------------------------------------------------------------

def test_ragged_small_graph(vgl, ctx, oracle):
    """V not a multiple of 32, self loops, duplicate edges, isolated vertices, one hub."""
    O = oracle
    V = 77
    rng = np.random.default_rng(5)
    src = np.concatenate([np.zeros(60, np.int32), rng.integers(1, 50, 90).astype(np.int32), np.array([3, 3, 9], np.int32)])
    dst = np.concatenate([rng.integers(0, 70, 60).astype(np.int32), rng.integers(0, 50, 90).astype(np.int32),
                          np.array([3, 3, 9], np.int32)])
    og = O.OracleGraph(V, src, dst)
    G = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    assert np.array_equal(G.layout()[0], og.row_ptr) and np.array_equal(G.layout()[1], og.adj)
    fwd = G.orig_to_sorted()
    w = G.synthetic_weights(11)
    for s in (0, 3, 76):  # hub, self-looped vertex, isolated vertex (levels: only the source is reached)
        for dopt in (False, True):
            lv, _ = G.bfs(int(fwd[s]), direction_optimising=dopt)
            assert np.array_equal(G.to_original(lv), og.bfs(s)[0])
        d, _ = G.sssp(w, int(fwd[s]))
        assert np.array_equal(G.to_original(d).view(np.uint32), og.sssp(s, 11)[0].view(np.uint32))
    lab, _ = G.cc()
    assert np.array_equal(G.to_original(lab), og.cc()[0])
    ranks, _ = G.pagerank(20)
    assert O.rel_l1(G.to_original(ranks), og.pagerank_f32(20, 2)) <= PR_TOL
    ranks0, _ = G.pagerank(0)
    assert np.all(ranks0.to_numpy() == np.float32(1.0 / V))
    G.free()


def test_hubs_and_long_chain(vgl, ctx, oracle, monkeypatch):
    """Rows on both sides of every tier border: two hubs with > 8192 out-edges (several CTA chunks per row), a 3000-vertex
    chain (thousands of BFS levels / SSSP rounds with one-vertex frontiers) hanging off a hub, random filler. Also the
    three SSSP schedules (reference's plain schedule, default near/far, a very fine threshold) must give the same bits."""
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
    assert G.info.max_degree > 8192 and G.tiers()[1][0] >= 2
    fwd = G.orig_to_sorted()
    w = G.synthetic_weights(3)
    for s in (5, 20000, 22990):
        for dopt in (False, True):
            lv, st = G.bfs(int(fwd[s]), direction_optimising=dopt)
            assert np.array_equal(G.to_original(lv), og.bfs(s)[0]), (s, dopt)
        ref = og.sssp(s, 3)[0].view(np.uint32)
        for scale in ("0", "4", "0.05"):
            monkeypatch.setenv("VGLB_SSSP_DELTA_SCALE", scale)
            d, st = G.sssp(w, int(fwd[s]))
            assert np.array_equal(G.to_original(d).view(np.uint32), ref), (s, scale)
        monkeypatch.delenv("VGLB_SSSP_DELTA_SCALE")
    lab, _ = G.cc()
    assert np.array_equal(G.to_original(lab), og.cc()[0])
    ranks, _ = G.pagerank(20)
    assert O.rel_l1(G.to_original(ranks), og.pagerank_f64(20)) <= PR_TOL
    G.free()


def test_graph_without_edges(vgl, ctx):
    V = 40
    e = np.empty(0, np.int32)
    G = vgl.Graph.from_edges(ctx, V, e, e, vgl.GRAPH_WITH_INCOMING)
    assert G.E == 0 and np.all(G.layout()[0] == 0)
    lv, st = G.bfs(7, direction_optimising=True)
    exp = np.full(V, -1, np.int32)
    exp[7] = 1
    assert np.array_equal(lv.to_numpy(), exp)
    w = ctx.empty(0, np.float32)
    d, _ = G.sssp(w, 5)
    dn = d.to_numpy()
    assert dn[5] == 0 and np.all(np.delete(dn, 5) == np.finfo(np.float32).max)
    lab, _ = G.cc()
    assert np.array_equal(lab.to_numpy(), np.arange(V, dtype=np.int32))
    ranks, _ = G.pagerank(3)
    assert abs(float(ranks.to_numpy().astype(np.float64).sum()) - 1.0) < 1e-5
    G.free()


def test_argument_errors(vgl, ctx):
    V = 16
    src = np.arange(V, dtype=np.int32)
    dst = (src + 1) % V
    G = vgl.Graph.from_edges(ctx, V, src, dst)  # no incoming CSR: a direction-optimising run derives it on the device
    lv_do, _ = G.bfs(0, direction_optimising=True)
    lv_td, _ = G.bfs(0, direction_optimising=False)
    assert np.array_equal(lv_do.to_numpy(), lv_td.to_numpy())
    with pytest.raises(vgl.VglbError, match="out of range"):
        G.bfs(V, direction_optimising=False)
    with pytest.raises(vgl.VglbError, match="out of range"):
        vgl.Graph.from_edges(ctx, V, src, dst + 100)
    # a CSR whose rows are not degree-sorted is not a VectCSR layout
    ptr = np.array([0, 1, 3], np.int64)
    adj = np.array([1, 0, 1], np.int32)
    with pytest.raises(vgl.VglbError, match="not sorted by degree"):
        vgl.Graph.from_csr(ctx, ptr, adj)
    G.free()


def test_from_csr_borrows_reference_layout(vgl, ctx, oracle, golden):
    """vglb_graph_from_csr: the path a VGL host build takes (VGL_Graph::move_to_device) with ITS arrays."""
    name, g = golden
    V = 1 << int(g["scale"])
    G = vgl.Graph.from_csr(ctx, g["out_ptr"], g["out_adj"], g["out_fwd"])
    fwd = g["out_fwd"]
    s = int(g["sources"][0])
    lv, _ = G.bfs(int(fwd[s]), direction_optimising=False)
    assert np.array_equal(G.to_original(lv), g["bfs_levels"][0])
    ranks, _ = G.pagerank(int(g["pr_iters"]))
    assert oracle.rel_l1(G.to_original(ranks), g["pr_ranks"]) <= PR_TOL
    G.free()


# ---------------------------------------------------------------------------------------------------------------------
# operators: frontier, generate_new_frontier, reduce, reorder
# ---------------------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("scale,density", [(8, 0.3), (13, 0.02), (13, 0.5), (13, 0.9), (15, 1.0), (15, 0.0)])
def test_generate_new_frontier_and_reduce(vgl, ctx, oracle, scale, density):
    O = oracle
    V = (1 << scale) - 5  # ragged tail
    src, dst = O.generate_edges(O.GEN_RMAT, scale, 8, 0x77)
    keep = (src < V) & (dst < V)
    src, dst = src[keep], dst[keep]
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    ptr, _ = G.layout()
    deg = np.diff(ptr)
    rng = np.random.default_rng(scale * 100 + int(density * 10))
    flags = (rng.random(V) < density).astype(np.int32) if 0.0 < density < 1.0 else np.full(V, int(density), np.int32)
    F = vgl.Frontier(G)
    dflags = ctx.from_numpy(flags)
    F.generate_from_flags(dflags)
    fi = F.info()
    ids = np.nonzero(flags)[0].astype(np.int32)
    assert fi.size == len(ids) and fi.neighbours == int(deg[ids].sum())
    _, tb = G.tiers()
    assert list(fi.tier_size) == [int((ids < tb[0]).sum()), int(((ids >= tb[0]) & (ids < tb[1])).sum()), int((ids >= tb[1]).sum())]
    # multicore/generate_new_frontier.hpp:67-91
    exp_type = 0 if len(ids) == V else (1 if len(ids) / V > 0.7 else 2)
    assert fi.sparsity_type == exp_type
    assert np.array_equal(F.ids(), ids), "compaction must be order preserving (copy_if_indexes, copy_if.hpp:127-191)"
    bits = np.unpackbits(F.bitmap().view(np.uint8), bitorder="little")[:V]
    assert np.array_equal(bits, flags.astype(np.uint8))
    vals = rng.integers(-1000, 1000, V).astype(np.int32)
    dvals = ctx.from_numpy(vals)
    fvals = rng.random(V).astype(np.float32)
    dfvals = ctx.from_numpy(fvals)
    assert F.reduce_sum_i32(dvals) == int(vals[ids].astype(np.int64).sum())
    if len(ids):
        assert F.reduce_max_i32(dvals) == int(vals[ids].max())
    assert abs(F.reduce_sum_f32(dfvals) - float(fvals[ids].astype(np.float64).sum())) <= 1e-9 * max(1, len(ids))
    # predicate forms used by BFS (levels == key) and SSSP (dist != prev)
    F.generate_eq(dvals, int(vals[0]))
    assert np.array_equal(F.ids(), np.nonzero(vals == vals[0])[0])
    other = vals.copy()
    other[::3] += 1
    dother = ctx.from_numpy(other)
    F.generate_ne(dvals, dother)
    assert np.array_equal(F.ids(), np.nonzero(vals != other)[0])
    # set_all_active / clear / add_vertex (modification.hpp:5-84)
    F.set_all_active()
    assert F.info().sparsity_type == 0 and F.size() == V and F.info().neighbours == G.E
    assert F.reduce_sum_i32(dvals) == int(vals.astype(np.int64).sum())
    F.clear()
    assert F.size() == 0
    F.add_vertex(3)
    assert F.size() == 1 and F.ids().tolist() == [3] and F.info().neighbours == int(deg[3])
    with pytest.raises(vgl.VglbError, match="non-empty frontier"):
        F.add_vertex(4)
    F.free()
    G.free()


def test_reorder_round_trip(vgl, ctx, oracle):
    O = oracle
    V = 1 << 12
    src, dst = O.generate_edges(O.GEN_KRONECKER, 12, 8, 0x99)
    G = vgl.Graph.from_edges(ctx, V, src, dst)
    fwd = G.orig_to_sorted()
    a = np.arange(V, dtype=np.int32) * 7
    d = ctx.from_numpy(a)
    s = G.reorder(d, vgl.ORIGINAL, vgl.SCATTER)
    assert np.array_equal(s.to_numpy()[fwd], a)          # sorted[fwd[orig]] = original[orig]
    back = G.reorder(s, vgl.SCATTER, vgl.ORIGINAL)
    assert np.array_equal(back.to_numpy(), a)
    with pytest.raises(vgl.VglbError):
        G.reorder(d, vgl.GATHER, vgl.SCATTER)
    G.free()


# ---------------------------------------------------------------------------------------------------------------------
# larger size: properties that do not need the oracle (BFS tree validity, SSSP optimality conditions, PR mass)
# ---------------------------------------------------------------------------------------------------------------------

def test_scale20_properties(vgl, ctx, oracle):
    O = oracle
    scale, ef = 20, 16
    V = 1 << scale
    dsrc, ddst = ctx.generate_edges(vgl.GEN_RMAT, scale, ef)
    G = vgl.Graph.from_edges(ctx, V, dsrc, ddst, vgl.GRAPH_WITH_INCOMING)
    ptr, adj = G.layout()
    row = np.repeat(np.arange(V, dtype=np.int32), np.diff(ptr))
    src_sorted = 0  # the largest hub
    lv_td, st_td = G.bfs(src_sorted, direction_optimising=False)
    lv_do, st_do = G.bfs(src_sorted, direction_optimising=True)
    a, b = lv_td.to_numpy(), lv_do.to_numpy()
    assert np.array_equal(a, b), "levels are direction independent"
    assert st_do.bottom_up_levels >= 1 and st_do.edges_inspected < st_td.edges_inspected
    # BFS validity: every edge out of a reached vertex ends at most one level deeper; every reached non-source vertex
    # has an in-neighbour exactly one level up
    reached = a[row] != -1
    assert np.all(a[adj[reached]] != -1) and np.all(a[adj[reached]] <= a[row[reached]] + 1)
    best_parent = np.full(V, np.iinfo(np.int32).max, np.int32)
    np.minimum.at(best_parent, adj[reached], a[row[reached]])
    nz = (a != -1) & (np.arange(V) != src_sorted)
    assert np.all(best_parent[nz] == a[nz] - 1) and a[src_sorted] == 1
    # SSSP optimality: dist[v] <= dist[u] + w for every edge, with equality for some in-edge of every reached vertex
    w = G.synthetic_weights(3)
    d, st = G.sssp(w, src_sorted)
    dn, wn = d.to_numpy(), w.to_numpy()
    reach = dn[row] < np.finfo(np.float32).max
    cand = (dn[row[reach]] + wn[reach]).astype(np.float32)
    assert np.all(dn[adj[reach]] <= cand)
    best = np.full(V, np.finfo(np.float32).max, np.float32)
    np.minimum.at(best, adj[reach], cand)
    nzs = (dn < np.finfo(np.float32).max) & (np.arange(V) != src_sorted)
    assert np.array_equal(best[nzs].view(np.uint32), dn[nzs].view(np.uint32)) and dn[src_sorted] == 0
    assert np.array_equal(dn < np.finfo(np.float32).max, a != -1), "SSSP and BFS reach the same set"
    # PageRank: mass conservation and agreement with the fp64 restatement
    ranks, st = G.pagerank(20)
    r = ranks.to_numpy()
    assert abs(float(r.astype(np.float64).sum()) - 1.0) < 1e-5
    og = O.OracleGraph(V, dsrc.to_numpy(), ddst.to_numpy())
    assert O.rel_l1(G.to_original(ranks), og.pagerank_f64(20)) <= PR_TOL
    G.free()


def test_baseline_size_properties(vgl, ctx, oracle):
    """BASELINE.json's full single-GPU size (RMAT scale 24, edge factor 16: 268 M edges), checked through properties that
    do not need an oracle run: the BFS / CC results are the unique solutions of their local equations over the incoming
    CSR, SSSP satisfies every edge inequality and reaches the BFS set, PageRank conserves mass and one more sweep of the
    fp64 restatement applied to the 20-sweep result gives the 21-sweep result."""
    scale, ef = 24, 16
    V = 1 << scale
    dsrc, ddst = ctx.generate_edges(vgl.GEN_RMAT, scale, ef)
    G = vgl.Graph.from_edges(ctx, V, dsrc, ddst, vgl.GRAPH_WITH_INCOMING)
    dsrc.free(); ddst.free()
    assert G.E == ef << scale
    iptr, iadj = G.layout(incoming=True)
    has_in = np.diff(iptr) > 0
    starts = iptr[:-1][has_in]  # reduceat over the non-empty in-rows (consecutive non-empty rows are adjacent in iadj)

    def min_over_in_neighbours(values, fill):
        out = np.full(V, fill, values.dtype)
        out[has_in] = np.minimum.reduceat(values[iadj], starts)
        return out

    src_sorted = 0  # the largest hub
    lv, st_do = G.bfs(src_sorted, direction_optimising=True)
    a = lv.to_numpy()
    lv2, st_td = G.bfs(src_sorted, direction_optimising=False)
    assert np.array_equal(a, lv2.to_numpy()), "levels are direction independent"
    assert st_do.bottom_up_levels >= 1 and st_do.edges_inspected < st_td.edges_inspected
    big = np.iinfo(np.int32).max
    parent_level = min_over_in_neighbours(np.where(a == -1, big, a).astype(np.int32), big)
    expect = np.where(parent_level == big, -1, parent_level + 1).astype(np.int32)
    expect[src_sorted] = 1
    assert np.array_equal(a, expect), "every vertex sits one level below its shallowest in-neighbour"
    lv.free(); lv2.free()

    lab, _ = G.cc()
    c = lab.to_numpy()
    ids = np.arange(V, dtype=np.int32)
    assert np.array_equal(c, np.minimum(ids, min_over_in_neighbours(c, big))), "labels = min id over the vertex and its in-neighbours' labels"
    lab.free()

    w = G.synthetic_weights(3)
    d, _ = G.sssp(w, src_sorted)
    dn = d.to_numpy()
    d2, _ = G.sssp(w, src_sorted)
    assert np.array_equal(dn.view(np.uint32), d2.to_numpy().view(np.uint32)), "SSSP is reproducible bit for bit"
    fmax = np.finfo(np.float32).max
    assert np.array_equal(dn < fmax, a != -1), "SSSP and BFS reach the same set"
    ptr, adj = G.layout()
    wn = w.to_numpy()
    for lo in range(0, V, V // 8):  # edge inequalities dist[dst] <= fl(dist[src] + w), an eighth of the rows at a time
        hi = lo + V // 8
        e0, e1 = int(ptr[lo]), int(ptr[hi])
        row = np.repeat(np.arange(lo, hi, dtype=np.int32), np.diff(ptr[lo:hi + 1]))
        ok = dn[row] < fmax
        assert np.all(dn[adj[e0:e1][ok]] <= (dn[row[ok]] + wn[e0:e1][ok]).astype(np.float32))
    del wn
    w.free(); d.free(); d2.free()

    r20, _ = G.pagerank(20)
    x = r20.to_numpy().astype(np.float64)
    assert abs(x.sum() - 1.0) < 1e-5
    r21, _ = G.pagerank(21)
    indeg = G.indegree_noloops().to_numpy().astype(np.float64)
    inv = np.divide(1.0, indeg, out=np.zeros(V), where=indeg > 0)
    contrib = x * inv
    sums = np.zeros(V)
    for lo in range(0, V, V // 8):
        hi = lo + V // 8
        e0, e1 = int(ptr[lo]), int(ptr[hi])
        row = np.repeat(np.arange(lo, hi, dtype=np.int32), np.diff(ptr[lo:hi + 1]))
        col = adj[e0:e1]
        vals = np.where(col != row, contrib[col], 0.0)
        nz = np.diff(ptr[lo:hi + 1]) > 0
        seg = np.add.reduceat(vals, (ptr[lo:hi][nz] - e0)) if e1 > e0 else np.zeros(0)
        sums[lo:hi][nz] = seg
    dangling = x[indeg == 0].sum() / V
    nxt = (1.0 - 0.85) / V + 0.85 * (sums + dangling)
    assert oracle.rel_l1(r21.to_numpy(), nxt) <= PR_TOL, "one fp64 sweep on top of the 20-sweep result gives the 21-sweep result"
    G.free()


def test_direction_optimising_bfs_derives_the_incoming_csr(vgl, ctx, oracle):
    """A graph uploaded without incoming arrays: the first direction-optimising vglb_bfs derives them on the device; the levels
    are those of the graph built with VGLB_GRAPH_WITH_INCOMING (and of the oracle)."""
    O = oracle
    scale, ef = 15, 16
    V = 1 << scale
    src, dst = O.generate_edges(O.GEN_RMAT if hasattr(O, "GEN_RMAT") else 0, scale, ef, 0xD0B)
    G0 = vgl.Graph.from_edges(ctx, V, src, dst, vgl.GRAPH_WITH_INCOMING)
    ptr, adj = G0.layout()
    fwd = G0.orig_to_sorted()
    outdeg = np.bincount(src, minlength=V)
    s = int(O.pick_sources(V, outdeg, 1, 0xD0B)[0])
    want, _ = G0.bfs(int(fwd[s]), direction_optimising=True)
    want = G0.to_original(want)
    G0.free()
    G = vgl.Graph.from_csr(ctx, ptr, adj, fwd)  # outgoing direction only
    got, st = G.bfs(int(fwd[s]), direction_optimising=True)
    got = G.to_original(got)
    G.free()
    assert np.array_equal(got, want)
    assert np.array_equal(got, O.OracleGraph(V, src, dst).bfs(s)[0])
