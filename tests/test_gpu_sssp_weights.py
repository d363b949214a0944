"""SSSP with caller-supplied edge weights: vglb_sssp must return the unique fp32 min-plus fixed point for ANY per-position
non-negative weight array, not only for the uniform [0, 100) weights of vglb_edge_weight.

The near/far schedule of sssp_run depends on the weights: delta comes from a sampled maximum weight (every position up to
E = 2^22, every (E >> 22)-th above), the threshold moves by delta or jumps to the smallest pending distance + delta,
vertices wait in the far bitmap, and the one-CTA drain returns to the host for three reasons (bucket empty, frontier
outgrew one CTA, first round too large to start). Every (weight family, graph shape) pair below must give the oracle's
bits under the default schedule, the plain schedule (delta scale 0), a fine one (0.05), a degenerate one (1e-9: delta below
the spacing of fp32 distances, so every threshold move is a jump) and without the drain.

References: oracle.lib().vglo_sssp (fp32 binary-heap Dijkstra, strict IEEE build) on the GPU graph's own CSR with the same
weight array, compared on the uint32 view; on graphs up to 2^15 vertices also an independent numpy fp32 Bellman-Ford
iterated to its fixed point, which checks the oracle on weights it was never pinned with.

Weights are a function of the ORIGINAL (src, dst) pair, so they are defined on any layout (one GPU or partitioned). The
stall regression is the exception: it places weights by CSR position, against the sample's stride.
"""
import ctypes as C
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

F32 = np.float32
FLT_MAX = F32(np.finfo(F32).max)
FLT_MAX_BITS = int(FLT_MAX.view(np.uint32))
NEG_ZERO_BITS = 0x80000000
WEIGHT_SEED = 0x5EED_B200
KNOBS = ("VGLB_SSSP_DELTA_SCALE", "VGLB_SSSP_NO_DRAIN", "VGLB_SSSP_TRACE", "VGLB_DENSE_EXCHANGE")
SCHEDULES = {
    "default": {},
    "plain": {"VGLB_SSSP_DELTA_SCALE": "0"},
    "fine": {"VGLB_SSSP_DELTA_SCALE": "0.05"},
    "degenerate": {"VGLB_SSSP_DELTA_SCALE": "1e-9"},
    "no_drain": {"VGLB_SSSP_NO_DRAIN": "1"},
}
BF_MAX_VERTICES = 1 << 15
SAMPLE_LIMIT = 1 << 22  # sssp.cu: the weight sample reads every (E >> 22)-th position once E > 2^22

# ---------------------------------------------------------------------------------------------------------------------
# weight families: fp32 weight of the edge between ORIGINAL ids (src, dst)
# ---------------------------------------------------------------------------------------------------------------------


def _mix64(z):
    """splitmix64 finalizer on a uint64 array (wrapping arithmetic)."""
    z = z + np.uint64(0x9E3779B97F4A7C15)
    z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return z ^ (z >> np.uint64(31))


def _bits(x):
    return np.uint32(x).view(F32)


def family_weights(family, osrc, odst):
    key = (osrc.astype(np.uint64) << np.uint64(32)) | odst.astype(np.uint32).astype(np.uint64)
    h = _mix64(key ^ np.uint64(WEIGHT_SEED))
    u = (h >> np.uint64(40)).astype(np.float64) / float(1 << 24)  # [0, 1) in 2^-24 steps
    pick = (h & np.uint64(0xFFFF)).astype(np.int64)
    uniform100 = (100.0 * u).astype(F32)
    if family == "zero":  # +0.0, a quarter of them -0.0
        return np.where(pick % 4 == 0, _bits(NEG_ZERO_BITS), F32(0.0)).astype(F32)
    if family == "ones":
        return np.ones(len(u), F32)
    if family == "small_int":
        return (1 + (h >> np.uint64(20)) % np.uint64(4)).astype(F32)
    if family == "log_uniform":  # 2^-20 .. 2^20
        return np.exp2(-20.0 + 40.0 * u).astype(F32)
    if family == "denormal":  # bit patterns 0 .. 2^23 - 1: zero and the subnormals, an eighth of them exactly zero
        w = ((h >> np.uint64(41)) & np.uint64(0x7FFFFF)).astype(np.uint32).view(F32)
        return np.where(pick % 8 == 0, F32(0.0), w).astype(F32)
    if family == "huge":  # uniform up to 3e38: two-edge sums overflow
        return (3e38 * u).astype(F32)
    if family == "inf_nan":  # +inf, +NaN and -NaN edges among uniform [0, 100)
        m = pick % 64
        w = np.where(m == 0, F32(np.inf), uniform100)
        w = np.where(m == 1, _bits(0x7FC00000), w)
        return np.where(m == 2, _bits(0xFFC00000), w).astype(F32)
    if family == "nan_only":  # +NaN and -NaN edges, no inf: the sampled maximum stays finite
        m = pick % 32
        w = np.where(m == 1, _bits(0x7FC00000), uniform100)
        return np.where(m == 2, _bits(0xFFC00000), w).astype(F32)
    if family == "outliers":  # uniform [0, 100), 1 % at 1e6
        return np.where(pick % 100 == 0, F32(1e6), uniform100).astype(F32)
    raise ValueError(family)


FAMILIES = ["zero", "ones", "small_int", "log_uniform", "denormal", "huge", "inf_nan", "nan_only", "outliers"]

# ---------------------------------------------------------------------------------------------------------------------
# graph shapes: ORIGINAL edge lists, sources, edges forced to +0.0 (by original source), what the drain trace must show
# ---------------------------------------------------------------------------------------------------------------------


def _generated(O, kind, scale, ef):
    src, dst = O.generate_edges(kind, scale, ef)
    V = 1 << scale
    return dict(V=V, src=src, dst=dst, sources=O.pick_sources(V, np.bincount(src, minlength=V), 1))


def _ragged():
    V = 77
    rng = np.random.default_rng(5)  # the graph of test_gpu_parity.py::test_ragged_small_graph
    src = np.concatenate([np.zeros(60, np.int32), rng.integers(1, 50, 90).astype(np.int32), np.array([3, 3, 9], np.int32)])
    dst = np.concatenate([rng.integers(0, 70, 60).astype(np.int32), rng.integers(0, 50, 90).astype(np.int32),
                          np.array([3, 3, 9], np.int32)])
    return dict(V=V, src=src, dst=dst, sources=[0, 3, 76])  # hub, self-looped vertex, isolated vertex


def _big_source():
    """Vertex 0 has 70,000 out-edges: more than one drain round may relax, so its round goes to the regular relax
    (several 8192-edge CTA chunks) without the drain starting."""
    V, n = 80000, 70000
    rng = np.random.default_rng(21)
    src = np.concatenate([np.zeros(n, np.int32), rng.integers(1, V, 80000).astype(np.int32)])
    dst = np.concatenate([np.arange(1, n + 1, dtype=np.int32), rng.integers(0, V, 80000).astype(np.int32)])
    return dict(V=V, src=src, dst=dst, sources=[0], trace="regular_first")


def _star(leaves):
    """Vertex 0 reaches `leaves` distinct leaves over +0.0 edges: the drain's second list has more than 1,024 rows
    (and, at 3,000 leaves, more than its 2,048 slots); the leaves and a random filler carry the family's weights."""
    V = 8192
    rng = np.random.default_rng(leaves)
    leaf = np.arange(1, leaves + 1, dtype=np.int32)
    src = np.concatenate([np.zeros(leaves, np.int32), np.repeat(leaf, 3), rng.integers(1, V, 16000).astype(np.int32)])
    dst = np.concatenate([leaf, rng.integers(1, V, 3 * leaves).astype(np.int32), rng.integers(0, V, 16000).astype(np.int32)])
    return dict(V=V, src=src, dst=dst, sources=[0], zero_src=[0], trace="outgrew")


def _fan():
    """Vertex 0 -> 100 middles over +0.0 edges, each middle -> 1,000 random vertices: the drain's second round holds
    100,000 edges, more than one CTA relaxes."""
    V = 1 << 15
    rng = np.random.default_rng(100)
    mid = np.arange(1, 101, dtype=np.int32)
    src = np.concatenate([np.zeros(100, np.int32), np.repeat(mid, 1000), rng.integers(101, V, 30000).astype(np.int32)])
    dst = np.concatenate([mid, rng.integers(101, V, 100000).astype(np.int32), rng.integers(101, V, 30000).astype(np.int32)])
    return dict(V=V, src=src, dst=dst, sources=[0], zero_src=[0], trace="outgrew")


def _chain():
    """3,000 vertices i -> i + 1, with skip edges i -> i + 5 competing: thousands of one-vertex rounds."""
    V = 3000
    a = np.arange(V - 1, dtype=np.int32)
    b = np.arange(V - 5, dtype=np.int32)
    return dict(V=V, src=np.concatenate([a, b]), dst=np.concatenate([a + 1, b + 5]), sources=[0], trace="bucket_empty")


def make_shape(O, name):
    if name == "rmat_s15":
        return _generated(O, O.GEN_RMAT, 15, 16)
    if name == "kron_s13":
        return _generated(O, O.GEN_KRONECKER, 13, 16)
    if name == "uniform_s12":
        return _generated(O, O.GEN_UNIFORM, 12, 32)
    if name == "ragged77":
        return _ragged()
    if name == "big_source":
        return _big_source()
    if name == "star1500":
        return _star(1500)
    if name == "star3000":
        return _star(3000)
    if name == "fan100x1000":
        return _fan()
    if name == "chain3000":
        return _chain()
    raise ValueError(name)


SHAPES = ["rmat_s15", "kron_s13", "uniform_s12", "ragged77", "big_source", "star1500", "star3000", "fan100x1000", "chain3000"]


def csr_weights(shape, family, ptr, adj, row_to_orig):
    """Weights by CSR position of a layout whose row r is ORIGINAL vertex row_to_orig[r] and whose adj holds ids that
    row_to_orig maps to ORIGINAL ids."""
    rows = np.repeat(np.arange(len(ptr) - 1), np.diff(ptr))
    osrc, odst = row_to_orig[rows], row_to_orig[adj]
    w = family_weights(family, osrc, odst)
    for z in shape.get("zero_src", ()):
        w[osrc == z] = F32(0.0)
    return w

# ---------------------------------------------------------------------------------------------------------------------
# references
# ---------------------------------------------------------------------------------------------------------------------


def _require_gradual_underflow():
    # a fast-math library loaded into this process could have set flush-to-zero / denormals-are-zero
    assert np.float32(1e-45) + np.float32(1e-45) == np.float32(3e-45), "denormals are flushed in this process"


def oracle_sssp(O, ptr, adj, w, source):
    _require_gradual_underflow()
    V = len(ptr) - 1
    ref = np.empty(V, F32)
    relaxed = C.c_int64()
    O.lib().vglo_sssp(V, np.ascontiguousarray(ptr, np.int64), np.ascontiguousarray(adj, np.int32), np.ascontiguousarray(w, F32),
                      int(source), ref, C.byref(relaxed))
    return ref


def bellman_ford(ptr, adj, w, source):
    """fp32 Bellman-Ford to its fixed point: each pass relaxes the out-edges of the rows whose distance changed in the
    previous pass (the other rows' candidates are unchanged), cand = dist[row] + w in fp32, np.fmin ignores NaN."""
    _require_gradual_underflow()
    V = len(ptr) - 1
    deg = np.diff(ptr)
    dist = np.full(V, FLT_MAX, F32)
    dist[source] = F32(0.0)
    active = np.array([source], np.int64)
    while active.size:
        cnt = deg[active]
        total = int(cnt.sum())
        if total == 0:
            break
        first = np.repeat(ptr[active] - (np.cumsum(cnt) - cnt), cnt)
        pos = first + np.arange(total)
        with np.errstate(over="ignore", invalid="ignore"):
            cand = (dist[np.repeat(active, cnt)] + w[pos]).astype(F32)
        new = dist.copy()
        np.fmin.at(new, adj[pos], cand)
        active = np.flatnonzero(new.view(np.uint32) != dist.view(np.uint32))
        dist = new
    return dist


def expected_split(w, E, V, scale=4.0):
    """sssp_run's delta from the sampled maximum weight (fmaxf from 0: NaN skipped, -0.0 counts as 0); True when the
    near/far split is on."""
    stride = E >> 22 if E > SAMPLE_LIMIT else 1
    sample = w[::stride]
    wmax = float(np.fmax.reduce(sample, initial=F32(0.0))) if len(sample) else 0.0
    avg = E / V
    with np.errstate(over="ignore"):
        delta = F32(scale * wmax / (avg if avg > 1.0 else 1.0))
    return bool(delta > 0 and delta < FLT_MAX)


def assert_same_bits(got, ref, what):
    g, r = got.view(np.uint32), ref.view(np.uint32)
    bad = np.flatnonzero(g != r)
    assert bad.size == 0, f"{what}: {bad.size} distances differ, first at {bad[:5].tolist()}: got {got[bad[:5]]} want {ref[bad[:5]]}"


def check_stats(st, ptr, got, source, what):
    deg = np.diff(ptr)
    reached = got.view(np.uint32) != FLT_MAX_BITS
    assert st.edges_inspected >= int(deg[reached].sum()), (what, st.edges_inspected, int(deg[reached].sum()))
    if deg[source] > 0:
        assert st.iterations >= 1, what


def run_sssp(G, w_dev, source, monkeypatch, env):
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    d, st = G.sssp(w_dev, source)
    got = d.to_numpy()
    d.free()
    for k in env:
        monkeypatch.delenv(k)
    return got, st

# ---------------------------------------------------------------------------------------------------------------------
# one GPU: every family on every shape under every schedule
# ---------------------------------------------------------------------------------------------------------------------


@pytest.fixture(scope="module")
def graphs(vgl, ctx, oracle):
    cache = {}

    def get(name):
        if name not in cache:
            sh = make_shape(oracle, name)
            G = vgl.Graph.from_edges(ctx, sh["V"], sh["src"], sh["dst"])
            ptr, adj = G.layout()
            cache[name] = (sh, G, ptr, adj, G.sorted_to_orig(), G.orig_to_sorted())
        return cache[name]

    yield get
    for sh, G, *_ in cache.values():
        G.free()


def _check_trace(kind, err, split, what):
    drains = re.findall(r"^sssp drain: (\d+) rounds, (\d+) rows, (\d+) edges on the device, (.*)$", err, re.M)
    assert ("sssp select" in err), what
    # a far selection runs exactly when the split is on
    assert ("(far)" in err) == split, (what, split)
    if kind == "bucket_empty":
        assert any(r[3] == "bucket empty" for r in drains), (what, drains[:4])
    elif kind == "outgrew":
        # the first drain relaxes the source's row and stops on its second list
        assert drains and drains[0][0] == "1" and drains[0][3] == "frontier outgrew one CTA", (what, drains[:4])
    elif kind == "regular_first":
        # the source's row is too long for the drain's first round: no drain line before the second selection, which
        # reports the regular relax of all of its edges
        head = err.split("sssp select 2 ", 1)[0]
        assert "sssp drain" not in head, what
        m = re.search(r"^sssp select 2 .*previous round relaxed (\d+) edges", err, re.M)
        assert m and int(m.group(1)) > 65536, (what, m and m.group(0))


@pytest.mark.parametrize("family", FAMILIES)
@pytest.mark.parametrize("shape_name", SHAPES)
def test_weight_family_all_schedules(vgl, ctx, oracle, graphs, shape_name, family, monkeypatch, capfd):
    sh, G, ptr, adj, bwd, fwd = graphs(shape_name)
    w = csr_weights(sh, family, ptr, adj, bwd)
    w_dev = ctx.from_numpy(w)
    split = expected_split(w, G.E, G.V)
    for s_orig in sh["sources"]:
        source = int(fwd[s_orig])
        ref = oracle_sssp(oracle, ptr, adj, w, source)
        if G.V <= BF_MAX_VERTICES:
            assert_same_bits(bellman_ford(ptr, adj, w, source), ref, f"{shape_name}/{family}: numpy Bellman-Ford vs the oracle")
        for sched, env in SCHEDULES.items():
            what = f"{shape_name}/{family}/{sched} source {s_orig}"
            if sched == "default":
                capfd.readouterr()
                env = dict(env, VGLB_SSSP_TRACE="1")
            got, st = run_sssp(G, w_dev, source, monkeypatch, env)
            assert_same_bits(got, ref, what)
            assert not np.any(got.view(np.uint32) == NEG_ZERO_BITS), f"{what}: -0.0 distance"
            check_stats(st, ptr, got, source, what)
            if sched == "default":
                _check_trace(sh.get("trace") if s_orig == sh["sources"][0] else None, capfd.readouterr().err, split, what)
    w_dev.free()

# ---------------------------------------------------------------------------------------------------------------------
# the threshold jump through the public API: the sample misses the only heavy edges
# ---------------------------------------------------------------------------------------------------------------------


def test_unsampled_heavy_edges_do_not_stall(vgl, ctx, oracle, monkeypatch):
    """E > 2^22: the weight sample reads every stride-th position only. Every weight is 1.0 (delta = 4 / 16 = 0.25) except
    the source's out-edges, which weigh 2^27 and sit at positions the sample skips. The smallest pending distance is then
    2^27, and 2^27 + 0.25 rounds back to 2^27 in fp32: the threshold jump must still move past it."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    scale, ef = 19, 16
    V = 1 << scale
    dsrc, ddst = ctx.generate_edges(vgl.GEN_RMAT, scale, ef)
    G = vgl.Graph.from_edges(ctx, V, dsrc, ddst)
    dsrc.free(); ddst.free()
    ptr, adj = G.layout()
    E = G.E
    stride = E >> 22 if E > SAMPLE_LIMIT else 1
    assert stride >= 2, E
    deg = np.diff(ptr)
    # rows whose every out-edge sits off the sample (all d positions between two multiples of the stride), not a self
    # loop; take the one whose first neighbour has the most out-edges
    cand = np.flatnonzero((deg >= 1) & (deg < stride))
    p0 = ptr[cand]
    off = (p0 % stride != 0) & ((p0 % stride) + deg[cand] <= stride)
    cand, p0 = cand[off], p0[off]
    cand = cand[adj[p0] != cand]
    assert cand.size, "no row off the sample"
    source = int(cand[np.argmax(deg[adj[ptr[cand]]])])
    s, e = int(ptr[source]), int(ptr[source + 1])
    heavy = F32(2.0 ** 27)
    w = np.ones(E, F32)
    w[s:e] = heavy
    assert np.all(np.arange(s, e) % stride != 0)
    assert float(w[::stride].max()) == 1.0, "the sample sees no heavy edge"
    delta = F32(4.0 * 1.0 / (G.E / V))
    assert heavy + delta == heavy, "the regime where fmaxf(threshold, min_pending) + delta == min_pending"
    ref = oracle_sssp(oracle, ptr, adj, w, source)
    w_dev = ctx.from_numpy(w)
    d, st = G.sssp(w_dev, source)
    got = d.to_numpy()
    assert_same_bits(got, ref, "heavy unsampled source edges")
    assert int((got.view(np.uint32) != FLT_MAX_BITS).sum()) > e - s + 1, "the heavy edges lead somewhere"
    check_stats(st, ptr, got, source, "heavy unsampled source edges")
    d.free(); w_dev.free()
    G.free()

# ---------------------------------------------------------------------------------------------------------------------
# partitioned driver on a live single-rank communicator
# ---------------------------------------------------------------------------------------------------------------------


@pytest.mark.parametrize("family", ["log_uniform", "ones"])
@pytest.mark.parametrize("shape_name", ["rmat_s15", "ragged77", "star3000", "chain3000"])
def test_partitioned_weight_families(vgl, ctx, oracle, shape_name, family, monkeypatch):
    """The default exchange (per-owner update lists, near/far schedule), a degenerate delta on it, and the dense
    exchange (allreduce(min) of the vector, plain schedule)."""
    for k in KNOBS:
        monkeypatch.delenv(k, raising=False)
    sh = make_shape(oracle, shape_name)
    comm = vgl.Comm(ctx, 0, 1)
    runs = [("default exchange", {}, False), ("default exchange, delta scale 1e-9", {"VGLB_SSSP_DELTA_SCALE": "1e-9"}, False),
            ("dense exchange", {}, True)]
    built = {}
    try:
        for what, env, dense in runs:
            if dense not in built:
                if dense:
                    monkeypatch.setenv("VGLB_DENSE_EXCHANGE", "1")  # read once per graph, at its first exchange
                G = vgl.Graph.from_edges_partitioned(ctx, comm, sh["V"], sh["src"], sh["dst"])
                assert (G.world, G.col0, G.V) == (1, 0, sh["V"])
                ptr, adj = G.layout()
                bwd, fwd = G.sorted_to_orig(), G.orig_to_sorted()
                w = csr_weights(sh, family, ptr, adj, bwd)
                built[dense] = (G, ptr, adj, fwd, w, ctx.from_numpy(w))
            G, ptr, adj, fwd, w, w_dev = built[dense]
            for s_orig in sh["sources"]:
                source = int(fwd[s_orig])
                ref = oracle_sssp(oracle, ptr, adj, w, source)
                if dense:
                    env = dict(env, VGLB_DENSE_EXCHANGE="1")
                got, st = run_sssp(G, w_dev, source, monkeypatch, env)
                tag = f"{shape_name}/{family}/{what} source {s_orig}"
                assert_same_bits(got, ref, tag)
                check_stats(st, ptr, got, source, tag)
    finally:
        for G, *_, w_dev in built.values():
            w_dev.free()
            G.free()
        comm.close()
