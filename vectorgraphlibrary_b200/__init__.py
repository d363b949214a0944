"""vectorgraphlibrary_b200 — host-side mirror (Python, ctypes) of the C ABI in include/vgl_b200.h.

The product is ``libvgl_b200.so`` (hand-written sm_100a CUDA behind a C ABI); this module only binds it for tests
and benchmarks and mirrors the reference's object model for the hot path:

    VGL_RUNTIME::init_library      -> Context                       (vgl_runtime/vgl_runtime.hpp:5-16)
    VGL_Graph + import             -> Graph.from_edges / from_csr   (vgl_graph.hpp:57-68)
    VerticesArray<T> / EdgesArray  -> DeviceArray                   (vertices_array.h:16-77)
    BFS::vgl_top_down              -> Graph.bfs                     (algorithms/bfs/bfs.hpp:56-86)
    PageRank::vgl_page_rank        -> Graph.pagerank                (algorithms/pr/pr.hpp:7-148)
    ShortestPaths::vgl_dijkstra    -> Graph.sssp                    (algorithms/sssp/shortest_paths.hpp:298-317)
    ConnectedComponents::vgl_shiloach_vishkin -> Graph.cc           (algorithms/cc/shiloach_vishkin.hpp:7-88)
    HITS::vgl_hits                 -> Graph.hits                    (algorithms/hits/hits.hpp:5-100)

There is no CPU fallback: importing works anywhere (so the symbol table can be checked on a CPU box), but creating a
Context raises VglbError when no CUDA device is usable, and a missing shared object raises at import of `lib()`.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VGLB_LIB_PATH") or os.path.join(_HERE, "libvgl_b200.so")  # env override: developer A/B builds
_LIB = None

GEN_RMAT, GEN_KRONECKER, GEN_UNIFORM = 0, 1, 2
SCATTER, GATHER, ORIGINAL = 0, 1, 2
GRAPH_WITH_INCOMING, GRAPH_WITH_EDGE_ORDER = 1, 2
HINT_PAGERANK = 1  # vglb_set_upload_hint
MASTER_SEED = 0xB200
NUM_TIERS = 8
BFS_MULTI_MAX_SOURCES = 64  # VGLB_BFS_MULTI_MAX_SOURCES: sources of one vglb_bfs_multi call


class VglbError(RuntimeError):
    """Mirrors the reference's `throw "message"` convention (common/advance.hpp:19-26)."""


class GraphInfo(C.Structure):
    _fields_ = [("vertices", C.c_int32), ("edges", C.c_int64), ("has_incoming", C.c_int32), ("max_degree", C.c_int32),
                ("tier_degree", C.c_int32 * NUM_TIERS), ("tier_border", C.c_int32 * NUM_TIERS),
                ("d_out_ptr", C.c_void_p), ("d_out_adj", C.c_void_p), ("d_in_ptr", C.c_void_p), ("d_in_adj", C.c_void_p),
                ("d_orig_to_sorted", C.c_void_p), ("d_sorted_to_orig", C.c_void_p), ("d_edge_order", C.c_void_p),
                ("part_rank", C.c_int32), ("part_world", C.c_int32), ("rows_per_rank", C.c_int32),
                ("col_of_row0", C.c_int32), ("vertices_global", C.c_int32), ("reserved", C.c_int32),
                ("columns", C.c_int64), ("edges_global", C.c_int64)]


class Stats(C.Structure):
    _fields_ = [("seconds", C.c_double), ("iterations", C.c_int64), ("edges_inspected", C.c_int64),
                ("vertices_processed", C.c_int64), ("frontier_bytes", C.c_int64), ("algorithmic_bytes", C.c_int64),
                ("kernel_launches", C.c_int64), ("bottom_up_levels", C.c_int32), ("reserved", C.c_int32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if k != "reserved"}


class PrOpts(C.Structure):
    _fields_ = [("dangling_mode", C.c_int32), ("reference_threads", C.c_int32)]


class BfsOpts(C.Structure):
    _fields_ = [("direction_optimising", C.c_int32), ("alpha", C.c_int32), ("beta", C.c_int32), ("reserved", C.c_int32)]


class FrontierInfo(C.Structure):
    _fields_ = [("sparsity_type", C.c_int32), ("size", C.c_int32), ("neighbours", C.c_int64),
                ("tier_size", C.c_int32 * 3), ("reserved", C.c_int32), ("d_ids", C.c_void_p), ("d_bitmap", C.c_void_p)]


# name -> (restype, argtypes); also the list the CPU test checks against include/vgl_b200.h
_P = C.c_void_p
_SIGNATURES = {
    "vglb_init": (C.c_int, [C.c_int, C.POINTER(_P)]),
    "vglb_finalize": (C.c_int, [_P]),
    "vglb_last_error": (C.c_char_p, []),
    "vglb_device_count": (C.c_int, []),
    "vglb_synchronize": (C.c_int, [_P]),
    "vglb_stream": (_P, [_P]),
    "vglb_malloc": (C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    "vglb_free": (C.c_int, [_P, _P]),
    "vglb_memcpy_h2d": (C.c_int, [_P, _P, _P, C.c_size_t]),
    "vglb_memcpy_d2h": (C.c_int, [_P, _P, _P, C.c_size_t]),
    "vglb_memcpy_d2d": (C.c_int, [_P, _P, _P, C.c_size_t]),
    "vglb_memset": (C.c_int, [_P, _P, C.c_int, C.c_size_t]),
    "vglb_host_alloc_pinned": (C.c_int, [C.c_size_t, C.POINTER(_P)]),
    "vglb_host_free_pinned": (C.c_int, [_P]),
    "vglb_flush_l2": (C.c_int, [_P]),
    "vglb_generate_edges_device": (C.c_int, [_P, C.c_int, C.c_int, C.c_int64, C.c_uint64, C.c_int, C.c_int, C.c_int, _P, _P]),
    "vglb_generate_edges_host": (C.c_int, [C.c_int, C.c_int, C.c_int64, C.c_uint64, C.c_int, C.c_int, C.c_int, _P, _P]),
    "vglb_graph_from_edges": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, C.c_int, C.c_int, C.POINTER(_P)]),
    "vglb_set_upload_hint": (C.c_int, [_P, C.c_int]),
    "vglb_graph_from_csr": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, _P, _P, _P, C.POINTER(_P)]),
    "vglb_graph_free": (C.c_int, [_P, _P]),
    "vglb_el_container_save": (C.c_int, [C.c_char_p, C.c_int32, C.c_int64, _P, _P]),
    "vglb_graph_import_el_container": (C.c_int, [_P, C.c_char_p, C.c_int, C.POINTER(_P)]),
    "vglb_graph_save_vgl": (C.c_int, [_P, C.c_char_p, C.c_int32, C.c_int64, _P, _P, C.c_int]),
    "vglb_graph_load_vgl": (C.c_int, [_P, C.c_char_p, C.c_int, C.POINTER(_P)]),
    "vglb_graph_get_info": (C.c_int, [_P, C.POINTER(GraphInfo)]),
    "vglb_graph_threshold_vertex": (C.c_int, [_P, _P, C.c_int32, C.POINTER(C.c_int32)]),
    "vglb_varray_reorder_u32": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int]),
    "vglb_earray_fill_synthetic_weights": (C.c_int, [_P, _P, C.c_uint64, _P]),
    "vglb_graph_indegree_noloops": (C.c_int, [_P, _P, _P]),
    "vglb_earray_mirror_out_to_in_u32": (C.c_int, [_P, _P, _P, _P]),
    "vglb_verify_i32": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "vglb_verify_f32": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(C.c_int64)]),
    "vglb_verify_ranking_f32": (C.c_int, [_P, _P, _P, C.c_int64, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "vglb_verify_components_i32": (C.c_int, [_P, _P, _P, C.c_int32, C.POINTER(C.c_int64)]),
    "vglb_pagerank": (C.c_int, [_P, _P, C.c_int, C.c_float, _P, C.POINTER(Stats)]),
    "vglb_pagerank_ex": (C.c_int, [_P, _P, C.c_int, C.c_float, C.POINTER(PrOpts), _P, C.POINTER(Stats)]),
    "vglb_bfs": (C.c_int, [_P, _P, C.c_int32, _P, C.POINTER(BfsOpts), C.POINTER(Stats)]),
    "vglb_bfs_multi": (C.c_int, [_P, _P, C.c_int32, _P, _P, C.POINTER(BfsOpts), C.POINTER(Stats)]),
    "vglb_sssp": (C.c_int, [_P, _P, _P, C.c_int32, _P, C.POINTER(Stats)]),
    "vglb_cc": (C.c_int, [_P, _P, _P, C.POINTER(Stats)]),
    "vglb_hits": (C.c_int, [_P, _P, C.c_int, _P, _P, C.POINTER(Stats)]),
    "vglb_frontier_create": (C.c_int, [_P, _P, C.POINTER(_P)]),
    "vglb_frontier_create_borrowed": (C.c_int, [_P, _P, _P, C.POINTER(_P)]),
    "vglb_frontier_set_ids": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int]),
    "vglb_graph_borrow_csr": (C.c_int, [_P, C.c_int32, C.c_int64, _P, _P, C.POINTER(_P)]),
    "vglb_frontier_destroy": (C.c_int, [_P, _P]),
    "vglb_frontier_set_all_active": (C.c_int, [_P, _P]),
    "vglb_frontier_clear": (C.c_int, [_P, _P]),
    "vglb_frontier_add_vertex": (C.c_int, [_P, _P, C.c_int32]),
    "vglb_frontier_get_info": (C.c_int, [_P, _P, C.POINTER(FrontierInfo)]),
    "vglb_gnf_from_flags": (C.c_int, [_P, _P, _P]),
    "vglb_gnf_from_bitmap": (C.c_int, [_P, _P, _P]),
    "vglb_gnf_eq_i32": (C.c_int, [_P, _P, _P, C.c_int32]),
    "vglb_gnf_ne_u32": (C.c_int, [_P, _P, _P, _P]),
    "vglb_reduce_sum_i32": (C.c_int, [_P, _P, _P, C.POINTER(C.c_int64)]),
    "vglb_reduce_sum_f32": (C.c_int, [_P, _P, _P, C.POINTER(C.c_double)]),
    "vglb_reduce_max_i32": (C.c_int, [_P, _P, _P, C.POINTER(C.c_int32)]),
    "vglb_comm_unique_id": (C.c_int, [_P]),
    "vglb_comm_init": (C.c_int, [_P, C.c_int, C.c_int, _P, C.POINTER(_P)]),
    "vglb_comm_init_detached": (C.c_int, [_P, C.c_int, C.c_int, C.POINTER(_P)]),
    "vglb_comm_destroy": (C.c_int, [_P]),
    "vglb_comm_barrier": (C.c_int, [_P]),
    "vglb_comm_allgather": (C.c_int, [_P, _P, C.c_size_t]),
    "vglb_comm_allreduce_sum_i64": (C.c_int, [_P, _P, C.c_int]),
    "vglb_comm_allreduce_max_f64": (C.c_int, [_P, C.POINTER(C.c_double)]),
    "vglb_graph_from_edges_partitioned": (C.c_int, [_P, _P, C.c_int32, C.c_int64, _P, _P, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "vglb_graph_from_generator_partitioned": (C.c_int, [_P, _P, C.c_int, C.c_int, C.c_int64, C.c_uint64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(_P)]),
    "vglb_graph_set_exchange": (C.c_int, [_P, _P, C.c_int]),
    "vglb_graph_from_csr_partitioned": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, C.POINTER(_P)]),
}
UNIQUE_ID_BYTES = 128
EXCHANGE_NCCL, EXCHANGE_P2P = 0, 1
PR_DANGLING_FP64, PR_DANGLING_REFERENCE_ORDER = 0, 1


def lib() -> C.CDLL:
    """Load libvgl_b200.so. Fails loudly when the CUDA extension has not been built (no fallback of any kind)."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise VglbError(f"{LIB_PATH} is missing: build it with `python -m vectorgraphlibrary_b200.build` "
                            "(there is no CPU or PyTorch fallback)")
        L = C.CDLL(LIB_PATH)
        missing = []
        for name, (res, args) in _SIGNATURES.items():
            try:
                fn = getattr(L, name)
            except AttributeError:
                missing.append(name)
                continue
            fn.restype = res
            fn.argtypes = args
        if missing and not os.environ.get("VGLB_ALLOW_PARTIAL_LIB"):
            raise VglbError("libvgl_b200.so does not export: " + ", ".join(missing))
        _LIB = L
    return _LIB


def _check(rc: int):
    if rc != 0:
        raise VglbError(f"[vglb error {rc}] " + lib().vglb_last_error().decode(errors="replace"))


def generate_edges_host(kind: int, scale: int, edge_factor: int, seed: int = MASTER_SEED, abc=(57, 19, 19)):
    """Host twin of the device generator (identical edges; used by CPU-side tests and the reference arm)."""
    E = edge_factor << scale
    src, dst = np.empty(E, np.int32), np.empty(E, np.int32)
    _check(lib().vglb_generate_edges_host(kind, scale, E, seed, abc[0], abc[1], abc[2], src.ctypes.data, dst.ctypes.data))
    return src, dst


def save_el_container(path: str, V: int, src: np.ndarray, dst: np.ndarray):
    """EdgesContainer::save_to_binary_file."""
    src, dst = np.ascontiguousarray(src, np.int32), np.ascontiguousarray(dst, np.int32)
    _check(lib().vglb_el_container_save(os.fsencode(path), V, len(src), src.ctypes.data, dst.ctypes.data))


def save_vgl(ctx: "Context", path: str, V: int, src, dst):
    """VGL_Graph::import + save_to_binary_file: both VectorCSRGraph containers built on the GPU, reference file format."""
    on_device = isinstance(src, DeviceArray)
    E = src.n if on_device else len(src)
    if not on_device:
        src, dst = np.ascontiguousarray(src, np.int32), np.ascontiguousarray(dst, np.int32)
    _check(lib().vglb_graph_save_vgl(ctx.h, os.fsencode(path), V, E, _ptr(src), _ptr(dst), int(on_device)))


def pinned_array(n: int, dtype):
    """numpy view of pinned host memory (vglb_host_alloc_pinned); lives until pinned_free() or the end of the process."""
    dtype = np.dtype(dtype)
    nbytes = max(1, int(n)) * dtype.itemsize
    p = _P()
    _check(lib().vglb_host_alloc_pinned(nbytes, C.byref(p)))
    buf = (C.c_char * nbytes).from_address(p.value)
    return np.frombuffer(buf, dtype=dtype, count=int(n))


def pinned_free(arr: np.ndarray):
    """Release a pinned_array(); the caller must drop every view of it first."""
    if arr is not None:
        _check(lib().vglb_host_free_pinned(_P(arr.ctypes.data)))


class Context:
    def __init__(self, device: int = 0):
        self.h = _P()
        _check(lib().vglb_init(device, C.byref(self.h)))
        self.device = device

    def close(self):
        if self.h:
            lib().vglb_finalize(self.h)
            self.h = _P()

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()

    def synchronize(self):
        _check(lib().vglb_synchronize(self.h))

    def flush_l2(self):
        _check(lib().vglb_flush_l2(self.h))

    @property
    def stream(self) -> int:
        return lib().vglb_stream(self.h) or 0

    def empty(self, n: int, dtype) -> "DeviceArray":
        return DeviceArray(self, n, np.dtype(dtype))

    def from_numpy(self, a: np.ndarray) -> "DeviceArray":
        a = np.ascontiguousarray(a)
        d = DeviceArray(self, a.size, a.dtype)
        d.copy_from_host(a)
        return d

    def generate_edges(self, kind: int, scale: int, edge_factor: int, seed: int = MASTER_SEED, abc=(57, 19, 19)):
        E = edge_factor << scale
        src, dst = self.empty(E, np.int32), self.empty(E, np.int32)
        _check(lib().vglb_generate_edges_device(self.h, kind, scale, E, seed, abc[0], abc[1], abc[2], src.ptr, dst.ptr))
        return src, dst


class Comm:
    """NCCL communicator of this rank inside libvgl_b200 (vgl_mpi_init twin, library_data/init.hpp:5-38). The unique id
    is created on rank 0 and handed to the other ranks by the caller (`exchange`: bytes on rank 0 -> bytes everywhere;
    bench.py / the tests use a torch.distributed broadcast for that plumbing)."""

    def __init__(self, ctx: Context, rank: int, world: int, exchange=None, detached: bool = False):
        self.ctx, self.rank, self.world = ctx, rank, world
        self.h = _P()
        if detached:
            _check(lib().vglb_comm_init_detached(ctx.h, rank, world, C.byref(self.h)))
            return
        uid = C.create_string_buffer(UNIQUE_ID_BYTES)
        if rank == 0:
            _check(lib().vglb_comm_unique_id(uid))
        raw = bytes(uid.raw)
        if world > 1:
            if exchange is None:
                raise VglbError("Comm: world > 1 needs an `exchange` callable to distribute the NCCL unique id")
            raw = exchange(raw if rank == 0 else None)
        _check(lib().vglb_comm_init(ctx.h, rank, world, raw, C.byref(self.h)))

    def barrier(self):
        _check(lib().vglb_comm_barrier(self.h))

    def max_float(self, x: float) -> float:
        v = C.c_double(x)
        _check(lib().vglb_comm_allreduce_max_f64(self.h, C.byref(v)))
        return v.value

    def close(self):
        if self.h:
            lib().vglb_comm_destroy(self.h)
            self.h = _P()


class DeviceArray:
    """HBM-resident flat array (VerticesArray / EdgesArray storage; MemoryAPI::allocate_array, memory_API.hpp:3-15)."""

    def __init__(self, ctx: Context, n: int, dtype: np.dtype):
        self.ctx, self.n, self.dtype = ctx, int(n), np.dtype(dtype)
        p = _P()
        _check(lib().vglb_malloc(ctx.h, self.nbytes, C.byref(p)))
        self.ptr = p.value

    @property
    def nbytes(self) -> int:
        return self.n * self.dtype.itemsize

    def copy_from_host(self, a: np.ndarray):
        a = np.ascontiguousarray(a, dtype=self.dtype)
        assert a.size == self.n
        _check(lib().vglb_memcpy_h2d(self.ctx.h, self.ptr, a.ctypes.data, self.nbytes))

    def to_numpy(self) -> np.ndarray:
        out = np.empty(self.n, self.dtype)
        if self.n:
            _check(lib().vglb_memcpy_d2h(self.ctx.h, out.ctypes.data, self.ptr, self.nbytes))
        return out

    def fill_bytes(self, byte: int):
        _check(lib().vglb_memset(self.ctx.h, self.ptr, byte, self.nbytes))

    def free(self):
        if self.ptr and self.ctx.h:
            lib().vglb_free(self.ctx.h, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def _ptr(x):
    if x is None:
        return None
    if isinstance(x, DeviceArray):
        return x.ptr
    if isinstance(x, np.ndarray):
        return x.ctypes.data
    return int(x)


class Graph:
    """Device VectCSR graph (VGL_Graph with VECTOR_CSR_GRAPH containers)."""

    def __init__(self, ctx: Context, handle):
        self.ctx, self.h = ctx, handle
        self.info = GraphInfo()
        _check(lib().vglb_graph_get_info(self.h, C.byref(self.info)))
        self.V, self.E = self.info.vertices, self.info.edges
        # partitioned graphs: V / E are this rank's rows / edges; vertex state is indexed by column id
        self.V_global, self.E_global, self.cols = self.info.vertices_global, self.info.edges_global, self.info.columns
        self.rank, self.world, self.vp, self.col0 = self.info.part_rank, self.info.part_world, self.info.rows_per_rank, self.info.col_of_row0

    @classmethod
    def from_edges_partitioned(cls, ctx: Context, comm: "Comm", V: int, src, dst, flags: int = 0, symmetrize: bool = False) -> "Graph":
        """This rank's part of the 1D-partitioned graph; every rank passes the same edge list (collective-free build)."""
        on_device = isinstance(src, DeviceArray)
        E = src.n if on_device else int(src.shape[0])
        if not on_device:
            src = np.ascontiguousarray(src, np.int32)
            dst = np.ascontiguousarray(dst, np.int32)
        h = _P()
        _check(lib().vglb_graph_from_edges_partitioned(ctx.h, comm.h, V, E, _ptr(src), _ptr(dst), int(on_device),
                                                       int(symmetrize), flags, C.byref(h)))
        g = cls(ctx, h)
        g.comm = comm
        return g

    @classmethod
    def from_csr_partitioned(cls, ctx: Context, comm: "Comm", V_global: int, out_ptr, out_adj, orig_to_col, in_ptr=None,
                             in_adj=None) -> "Graph":
        """VGL_Graph::move_to_device for this rank's part (host arrays -> HBM)."""
        rows = int(out_ptr.shape[0]) - 1
        keep = [np.ascontiguousarray(out_ptr, np.int64), np.ascontiguousarray(out_adj, np.int32),
                np.ascontiguousarray(orig_to_col, np.int32)]
        for a, t in ((in_ptr, np.int64), (in_adj, np.int32)):
            keep.append(None if a is None else np.ascontiguousarray(a, t))
        h = _P()
        _check(lib().vglb_graph_from_csr_partitioned(ctx.h, comm.h, V_global, rows, *[_ptr(a) for a in keep], C.byref(h)))
        g = cls(ctx, h)
        g.comm = comm
        return g

    @classmethod
    def from_generator_partitioned(cls, ctx: Context, comm: "Comm", kind: int, scale: int, edge_factor: int, flags: int = 0,
                                   symmetrize: bool = False, seed: int = MASTER_SEED, abc=(57, 19, 19)) -> "Graph":
        h = _P()
        _check(lib().vglb_graph_from_generator_partitioned(ctx.h, comm.h, kind, scale, edge_factor << scale, seed, abc[0], abc[1],
                                                           abc[2], int(symmetrize), flags, C.byref(h)))
        g = cls(ctx, h)
        g.comm = comm
        return g

    @classmethod
    def from_edges(cls, ctx: Context, V: int, src, dst, flags: int = 0) -> "Graph":
        on_device = isinstance(src, DeviceArray)
        E = src.n if on_device else int(src.shape[0])
        if not on_device:
            src = np.ascontiguousarray(src, np.int32)
            dst = np.ascontiguousarray(dst, np.int32)
        h = _P()
        _check(lib().vglb_graph_from_edges(ctx.h, V, E, _ptr(src), _ptr(dst), int(on_device), flags, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def import_el_container(cls, ctx: Context, path: str, flags: int = 0) -> "Graph":
        """VGL_Graph::import of an .el_container file (the apps' `-import <file>`)."""
        h = _P()
        _check(lib().vglb_graph_import_el_container(ctx.h, os.fsencode(path), flags, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def load_vgl(cls, ctx: Context, path: str, flags: int = 0) -> "Graph":
        """VGL_Graph::load_from_binary_file + move_to_device."""
        h = _P()
        _check(lib().vglb_graph_load_vgl(ctx.h, os.fsencode(path), flags, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_csr(cls, ctx: Context, out_ptr: np.ndarray, out_adj: np.ndarray, orig_to_sorted=None, in_ptr=None,
                 in_adj=None) -> "Graph":
        V, E = int(out_ptr.shape[0]) - 1, int(out_adj.shape[0])
        keep = [np.ascontiguousarray(out_ptr, np.int64), np.ascontiguousarray(out_adj, np.int32)]
        for a, t in ((orig_to_sorted, np.int32), (in_ptr, np.int64), (in_adj, np.int32)):
            keep.append(None if a is None else np.ascontiguousarray(a, t))
        h = _P()
        _check(lib().vglb_graph_from_csr(ctx.h, V, E, *[_ptr(a) for a in keep], C.byref(h)))
        return cls(ctx, h)

    def free(self):
        if self.h and self.ctx.h:
            lib().vglb_graph_free(self.ctx.h, self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # ---- layout read-back (parity of the builder against VectorCSRGraph) ----
    def _d2h(self, dptr, n, dtype):
        out = np.empty(n, dtype)
        if n:
            _check(lib().vglb_memcpy_d2h(self.ctx.h, out.ctypes.data, dptr, out.nbytes))
        return out

    def layout(self, incoming: bool = False):
        i = self.info
        if incoming:
            ptr = self._d2h(i.d_in_ptr, self.V + 1, np.int64)
            return ptr, self._d2h(i.d_in_adj, int(ptr[-1]), np.int32)
        return self._d2h(i.d_out_ptr, self.V + 1, np.int64), self._d2h(i.d_out_adj, self.E, np.int32)

    def orig_to_sorted(self):
        """ORIGINAL id -> SCATTER id (the column id on a partitioned graph)."""
        return self._d2h(self.info.d_orig_to_sorted, self.V_global, np.int32)

    def sorted_to_orig(self):
        """column id -> ORIGINAL id (-1 for the padding columns of a partitioned graph)."""
        return self._d2h(self.info.d_sorted_to_orig, self.cols, np.int32)

    def tiers(self):
        return list(self.info.tier_degree), list(self.info.tier_border)

    def threshold_vertex(self, degree_threshold: int) -> int:
        out = C.c_int32()
        _check(lib().vglb_graph_threshold_vertex(self.ctx.h, self.h, degree_threshold, C.byref(out)))
        return out.value

    def reorder(self, arr: DeviceArray, from_dir: int, to_dir: int) -> DeviceArray:
        assert arr.dtype.itemsize == 4
        out = self.ctx.empty(self.V_global if to_dir == ORIGINAL else self.V, arr.dtype)
        _check(lib().vglb_varray_reorder_u32(self.ctx.h, self.h, arr.ptr, out.ptr, from_dir, to_dir))
        return out

    def set_exchange(self, mode: int):
        _check(lib().vglb_graph_set_exchange(self.ctx.h, self.h, mode))

    def to_original_rows(self, arr: DeviceArray, k: int) -> np.ndarray:
        """(k, V) array in ORIGINAL numbering of k consecutive V-sized rows in SCATTER numbering (vglb_bfs_multi's output).
        One-GPU graphs only."""
        assert arr.dtype.itemsize == 4 and arr.n >= k * self.V
        row = self.ctx.empty(self.V, arr.dtype)
        out = np.empty((k, self.V), arr.dtype)
        for i in range(k):
            _check(lib().vglb_varray_reorder_u32(self.ctx.h, self.h, arr.ptr + i * self.V * 4, row.ptr, SCATTER, ORIGINAL))
            out[i] = row.to_numpy()
        row.free()
        return out

    def to_original(self, arr: DeviceArray) -> np.ndarray:
        """VerticesArray::reorder(ORIGINAL) + move_to_host (a collective on a partitioned graph: every rank gets the
        whole array)."""
        return self.reorder(arr, SCATTER, ORIGINAL).to_numpy()

    def synthetic_weights(self, seed: int) -> DeviceArray:
        w = self.ctx.empty(self.E, np.float32)
        _check(lib().vglb_earray_fill_synthetic_weights(self.ctx.h, self.h, seed, w.ptr))
        return w

    def mirror_out_to_in(self, out_values: DeviceArray) -> DeviceArray:
        """VGL_Graph::copy_outgoing_to_incoming_edges: per-edge values in outgoing-CSR order -> incoming-CSR order."""
        assert out_values.dtype.itemsize == 4 and out_values.n == self.E
        out = self.ctx.empty(self.E, out_values.dtype)
        _check(lib().vglb_earray_mirror_out_to_in_u32(self.ctx.h, self.h, out_values.ptr, out.ptr))
        return out

    def indegree_noloops(self) -> DeviceArray:
        d = self.ctx.empty(self.V, np.int32)
        _check(lib().vglb_graph_indegree_noloops(self.ctx.h, self.h, d.ptr))
        return d

    # ---- the four algorithms ----
    def pagerank(self, iters: int = 20, damping: float = 0.85, ranks: DeviceArray | None = None,
                 reference_threads: int = 0):
        """`reference_threads` > 0: sum the dangling mass in the reference's order for that OpenMP thread count
        (vglb_pagerank_ex, VGLB_PR_DANGLING_REFERENCE_ORDER); 0: fp64 inside the sweep."""
        ranks = ranks or self.ctx.empty(self.V, np.float32)
        st = Stats()
        if reference_threads > 0:
            opts = PrOpts(PR_DANGLING_REFERENCE_ORDER, reference_threads)
            _check(lib().vglb_pagerank_ex(self.ctx.h, self.h, iters, damping, C.byref(opts), ranks.ptr, C.byref(st)))
        else:
            _check(lib().vglb_pagerank(self.ctx.h, self.h, iters, damping, ranks.ptr, C.byref(st)))
        return ranks, st

    def bfs(self, source_sorted: int, direction_optimising: bool = True, levels: DeviceArray | None = None,
            alpha: int = 0, beta: int = 0):
        levels = levels or self.ctx.empty(self.V, np.int32)
        st = Stats()
        opts = BfsOpts(int(direction_optimising), alpha, beta, 0)
        _check(lib().vglb_bfs(self.ctx.h, self.h, int(source_sorted), levels.ptr, C.byref(opts), C.byref(st)))
        return levels, st

    def bfs_multi(self, sources_sorted, direction_optimising: bool = True, levels: DeviceArray | None = None,
                  alpha: int = 0, beta: int = 0):
        """vglb_bfs_multi: up to BFS_MULTI_MAX_SOURCES BFS runs in one traversal. Returns (k*V int32 levels, row i =
        Graph.bfs(sources_sorted[i]), Stats)."""
        src = np.ascontiguousarray(np.asarray(sources_sorted, np.int32).reshape(-1))
        k = len(src)
        levels = levels or self.ctx.empty(max(1, k) * self.V, np.int32)
        st = Stats()
        opts = BfsOpts(int(direction_optimising), alpha, beta, 0)
        _check(lib().vglb_bfs_multi(self.ctx.h, self.h, k, src.ctypes.data, levels.ptr, C.byref(opts), C.byref(st)))
        return levels, st

    def sssp(self, weights: DeviceArray, source_sorted: int, dist: DeviceArray | None = None):
        dist = dist or self.ctx.empty(self.V, np.float32)
        st = Stats()
        _check(lib().vglb_sssp(self.ctx.h, self.h, weights.ptr, int(source_sorted), dist.ptr, C.byref(st)))
        return dist, st

    def cc(self, labels: DeviceArray | None = None):
        labels = labels or self.ctx.empty(self.V, np.int32)
        st = Stats()
        _check(lib().vglb_cc(self.ctx.h, self.h, labels.ptr, C.byref(st)))
        return labels, st

    def hits(self, steps: int = 20, auth: DeviceArray | None = None, hub: DeviceArray | None = None):
        """vglb_hits: `steps` HITS steps. Returns (authority scores, hub scores, Stats), fp32 in SCATTER numbering."""
        auth = auth or self.ctx.empty(self.V, np.float32)
        hub = hub or self.ctx.empty(self.V, np.float32)
        st = Stats()
        _check(lib().vglb_hits(self.ctx.h, self.h, int(steps), auth.ptr, hub.ptr, C.byref(st)))
        return auth, hub, st


def verify_results(ctx: "Context", a: DeviceArray, b: DeviceArray) -> int:
    """verify_results (verify_results.h:33-93) on the device: the `error count` (0 = equal). int32 arrays compare exactly,
    float32 arrays with the reference's are_same tolerance."""
    assert a.n == b.n and a.dtype == b.dtype
    out = C.c_int64()
    fn = lib().vglb_verify_f32 if a.dtype == np.float32 else lib().vglb_verify_i32
    _check(fn(ctx.h, a.ptr, b.ptr, a.n, C.byref(out)))
    return out.value


def verify_ranking_results(ctx: "Context", a: DeviceArray, ref: DeviceArray):
    """verify_ranking_results (verify_results.h:97-148): (mean |a - ref|, relative L1, error count)."""
    assert a.n == ref.n
    diff, rel, err = C.c_double(), C.c_double(), C.c_int64()
    _check(lib().vglb_verify_ranking_f32(ctx.h, a.ptr, ref.ptr, a.n, C.byref(diff), C.byref(rel), C.byref(err)))
    return diff.value, rel.value, err.value


def equal_components(ctx: "Context", a: DeviceArray, b: DeviceArray) -> int:
    """equal_components (verify_results.h:198-254): error count, 0 = the label arrays describe the same partition."""
    assert a.n == b.n
    out = C.c_int64()
    _check(lib().vglb_verify_components_i32(ctx.h, a.ptr, b.ptr, a.n, C.byref(out)))
    return out.value


class Frontier:
    """VGL_Frontier / FrontierVectorCSR (frontier_vect_csr.h:5-53): sparse id queue or dense bitmap by density."""

    def __init__(self, graph: Graph):
        self.g, self.ctx = graph, graph.ctx
        self.h = _P()
        _check(lib().vglb_frontier_create(self.ctx.h, graph.h, C.byref(self.h)))

    def free(self):
        if self.h and self.ctx.h:
            lib().vglb_frontier_destroy(self.ctx.h, self.h)
        self.h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    def set_all_active(self):
        _check(lib().vglb_frontier_set_all_active(self.ctx.h, self.h))

    def clear(self):
        _check(lib().vglb_frontier_clear(self.ctx.h, self.h))

    def add_vertex(self, v: int):
        _check(lib().vglb_frontier_add_vertex(self.ctx.h, self.h, v))

    def add_group_of_vertices(self, ids):
        """FrontierVectorCSR::add_group_of_vertices: the reference sorts the list ascending first; so does this mirror."""
        ids = np.ascontiguousarray(np.sort(np.asarray(ids, np.int32)))
        _check(lib().vglb_frontier_set_ids(self.ctx.h, self.h, ids.ctypes.data, len(ids), 0))

    def info(self) -> FrontierInfo:
        fi = FrontierInfo()
        _check(lib().vglb_frontier_get_info(self.ctx.h, self.h, C.byref(fi)))
        return fi

    def size(self) -> int:
        return self.info().size

    def ids(self) -> np.ndarray:
        fi = self.info()
        return self.g._d2h(fi.d_ids, fi.size, np.int32)

    def bitmap(self) -> np.ndarray:
        fi = self.info()
        return self.g._d2h(fi.d_bitmap, (self.g.V + 31) // 32, np.uint32)

    def generate_from_flags(self, flags: DeviceArray):
        _check(lib().vglb_gnf_from_flags(self.ctx.h, self.h, flags.ptr))

    def generate_eq(self, values: DeviceArray, key: int):
        _check(lib().vglb_gnf_eq_i32(self.ctx.h, self.h, values.ptr, key))

    def generate_ne(self, a: DeviceArray, b: DeviceArray):
        _check(lib().vglb_gnf_ne_u32(self.ctx.h, self.h, a.ptr, b.ptr))

    def reduce_sum_i32(self, values: DeviceArray) -> int:
        out = C.c_int64()
        _check(lib().vglb_reduce_sum_i32(self.ctx.h, self.h, values.ptr, C.byref(out)))
        return out.value

    def reduce_sum_f32(self, values: DeviceArray) -> float:
        out = C.c_double()
        _check(lib().vglb_reduce_sum_f32(self.ctx.h, self.h, values.ptr, C.byref(out)))
        return out.value

    def reduce_max_i32(self, values: DeviceArray) -> int:
        out = C.c_int32()
        _check(lib().vglb_reduce_max_i32(self.ctx.h, self.h, values.ptr, C.byref(out)))
        return out.value
