"""Host-side drivers for the four algorithms on 1..N GPUs (one process per GPU) — used by bench.py, the smoke test and
the multi-rank tests. The compute is libvgl_b200 (C ABI); torch.distributed is plumbing only (rendezvous, barrier,
exchange of the NCCL unique id / CUDA IPC handles, max-over-ranks of timings).

Reference: the MPI layer of the NEC backend (vgl_compute_api/common/mpi_exchange.hpp:155-271,
vgl_runtime/helpers/library_data/init.hpp:5-38) replicates the graph and exchanges whole vertex arrays; here the graph is
1D-partitioned by vertex range (see DESIGN.md, "Multi-GPU") and only owned slices travel.
"""
from __future__ import annotations

import ctypes as C
import os
import time

import numpy as np

_M64 = (1 << 64) - 1


def mix64(z: int) -> int:
    """vglb_mix64 (include/vglb_synth.h) in Python."""
    z = (z + 0x9E3779B97F4A7C15) & _M64
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return z ^ (z >> 31)


def pick_sources(V: int, out_degree_orig: np.ndarray, count: int, seed: int) -> list[int]:
    """`count` seeded ORIGINAL ids with out-degree > 0 (vglb_source_candidate; reference: select_random_nz_vertex per
    round, apps/bfs/bfs.cpp:38)."""
    out, k = [], 0
    while len(out) < count:
        v = mix64(seed ^ ((0xA5A5A5A5 + k * 0x9E3779B97F4A7C15) & _M64)) % V
        k += 1
        if out_degree_orig[v] > 0:
            out.append(int(v))
        if k > 64 * count + 1024:
            raise RuntimeError("no vertex with out-degree > 0")
    return out


class Communicator:
    """torch.distributed process group (nccl on GPUs, gloo on CPU) used for the plumbing around the library."""

    def __init__(self, backend: str, device=None):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        if not dist.is_initialized():
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            kw = {}
            if backend == "nccl" and device is not None:
                kw["device_id"] = torch.device("cuda", device)
            dist.init_process_group(backend=backend, **kw)
        self.rank, self.world = dist.get_rank(), dist.get_world_size()
        self.device = torch.device("cuda", device) if backend == "nccl" else torch.device("cpu")
        self.backend = backend

    @classmethod
    def from_env(cls, local_rank: int) -> "Communicator":
        return cls("nccl", local_rank)

    def barrier(self):
        if self.backend == "nccl":
            t = self.torch.zeros(1, device=self.device)
            self.dist.all_reduce(t)
            self.torch.cuda.synchronize()
        else:
            self.dist.barrier()

    def max_float(self, x: float) -> float:
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_int(self, x: int) -> int:
        t = self.torch.tensor([x], dtype=self.torch.int64, device=self.device)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return int(t.item())

    def allgather_bytes(self, b: bytes) -> list[bytes]:
        t = self.torch.frombuffer(bytearray(b), dtype=self.torch.uint8).to(self.device)
        out = [self.torch.empty_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [bytes(o.cpu().numpy().tobytes()) for o in out]

    def broadcast_bytes(self, b: bytes | None, n: int, root: int = 0) -> bytes:
        t = self.torch.frombuffer(bytearray(b if self.rank == root else bytes(n)), dtype=self.torch.uint8).to(self.device)
        self.dist.broadcast(t, root)
        return bytes(t.cpu().numpy().tobytes())

    def close(self):
        if self.dist.is_initialized():
            self.dist.destroy_process_group()


def _stats(st, dominant_launches, dominant_bytes):
    d = st.as_dict()
    d["dominant_launches"] = dominant_launches
    d["dominant_bytes"] = dominant_bytes
    return d


class SingleGpuRunner:
    """One GPU, whole graph resident: the N = 1 case of every workload."""

    weak = True
    partition = "single GPU, whole graph"
    ncu_traffic = None
    bfs_direction_optimising = True

    def __init__(self, vgl, ctx, workload, kind, scale, ef, pr_iters):
        self.vgl, self.ctx, self.workload, self.pr_iters = vgl, ctx, workload, pr_iters
        V = 1 << scale
        src, dst = ctx.generate_edges(kind, scale, ef)
        if workload == "cc":  # symmetrised input (SURVEY §8d): append the reversed copy of every edge
            s2, d2 = ctx.empty(2 * src.n, np.int32), ctx.empty(2 * src.n, np.int32)
            L = vgl.lib()
            for dstbuf, a, b in ((s2, src, dst), (d2, dst, src)):
                vgl._check(L.vglb_memcpy_d2d(ctx.h, dstbuf.ptr, a.ptr, a.nbytes))
                vgl._check(L.vglb_memcpy_d2d(ctx.h, dstbuf.ptr + a.nbytes, b.ptr, b.nbytes))
            src.free(); dst.free()
            src, dst = s2, d2
        flags = vgl.GRAPH_WITH_INCOMING if workload == "bfs" else 0
        self.g = vgl.Graph.from_edges(ctx, V, src, dst, flags)
        src.free(); dst.free()
        self.V_total, self.E_total = self.g.V, self.g.E
        self.scale = scale
        self.adj_bytes_per_gpu = 4 * self.g.E
        self.dtype = "f32" if workload in ("pr", "sssp") else "int32"
        self.iters_per_step = pr_iters if workload == "pr" else 1
        self.edges_per_step = self.g.E * self.iters_per_step
        self.out = ctx.empty(V, np.float32 if self.dtype == "f32" else np.int32)
        self.dominant_kernel = {"pr": "pr_bin_kernel + pr_cold_bin_kernel + pr_sweep_kernel + pr_finish_kernel (one sweep)", "bfs": "bfs_td_kernel + bfs_bu_kernel (whole run)",
                                "sssp": "sssp_relax_flat_kernel + sssp_select_kernel (whole run)", "cc": "cc_hook_kernel + cc_jump_kernel (whole run)"}[workload]
        self.weights = self.g.synthetic_weights(vgl.MASTER_SEED ^ 0x5555) if workload == "sssp" else None
        self.sources = None
        if workload in ("bfs", "sssp"):
            ptr, _ = self.g.layout()  # host copy of the row pointers, setup only
            deg_sorted = np.diff(ptr)
            fwd = self.g.orig_to_sorted()
            orig = pick_sources(V, deg_sorted[fwd], 16, vgl.MASTER_SEED)
            self.sources = [int(fwd[s]) for s in orig]
        self.per_step = []
        self._host = None

    def step(self, i):
        w = self.workload
        if w == "pr":
            _, st = self.g.pagerank(self.pr_iters, 0.85, self.out)
            return _stats(st, self.pr_iters, st.algorithmic_bytes)
        if w == "bfs":
            _, st = self.g.bfs(self.sources[i % len(self.sources)], self.bfs_direction_optimising, self.out)
        elif w == "sssp":
            _, st = self.g.sssp(self.weights, self.sources[i % len(self.sources)], self.out)
        else:
            _, st = self.g.cc(self.out)
        return _stats(st, 1, st.algorithmic_bytes)

    # ---- end to end through the C ABI with HOST buffers ----
    def _host_arrays(self):
        """The arrays a VGL host build owns (VectorCSRGraph::get_vertex_pointers / get_adjacent_ids, id map), in pinned
        host memory; setup, outside the timed region."""
        if self._host is None:
            vgl, g = self.vgl, self.g
            pinned_array = lambda _v, n, dt: (vgl.pinned_array(n, dt), None)
            ptr, adj = g.layout()
            h_ptr, _ = pinned_array(vgl, g.V + 1, np.int64)
            h_adj, _ = pinned_array(vgl, g.E, np.int32)
            h_fwd, _ = pinned_array(vgl, g.V, np.int32)
            h_ptr[:], h_adj[:], h_fwd[:] = ptr, adj, g.orig_to_sorted()
            h_out, _ = pinned_array(vgl, g.V, np.float32 if self.dtype == "f32" else np.int32)
            host = {"ptr": h_ptr, "adj": h_adj, "fwd": h_fwd, "out": h_out, "w": None}
            del ptr, adj
            # BFS: the bottom-up levels need the incoming CSR. Only the outgoing direction goes up and vglb_bfs derives the
            # incoming one on the device (a sort of the edges beats a second PCIe upload of the same size).
            if self.workload == "sssp":
                host["w"], _ = pinned_array(vgl, g.E, np.float32)
                host["w"][:] = self.weights.to_numpy()
            self._host = host
        return self._host

    def e2e(self, steps):
        vgl, ctx = self.vgl, self.ctx
        H = self._host_arrays()
        L = vgl.lib()
        h2d = H["ptr"].nbytes + H["adj"].nbytes + H["fwd"].nbytes
        if H["w"] is not None:
            h2d += H["w"].nbytes
        d2h = H["out"].nbytes
        times = []
        # (the caller says what it is going to run: PageRank's preparation then happens behind the upload)
        vgl._check(L.vglb_set_upload_hint(ctx.h, vgl.HINT_PAGERANK if self.workload == "pr" else 0))
        for i in range(steps + 1):
            ctx.synchronize()
            t0 = time.perf_counter()
            g = vgl.Graph.from_csr(ctx, H["ptr"], H["adj"], H["fwd"])
            out = ctx.empty(g.V, H["out"].dtype)
            if self.workload == "pr":
                g.pagerank(self.pr_iters, 0.85, out)
            elif self.workload == "bfs":
                g.bfs(self.sources[i % len(self.sources)], self.bfs_direction_optimising, out)
            elif self.workload == "sssp":
                w = ctx.empty(g.E, np.float32)
                vgl._check(L.vglb_memcpy_h2d(ctx.h, w.ptr, H["w"].ctypes.data, H["w"].nbytes))
                g.sssp(w, self.sources[i % len(self.sources)], out)
                w.free()
            else:
                g.cc(out)
            # the caller gets the result in ITS numbering: VerticesArray::reorder(ORIGINAL) on the device, then the download
            res = g.reorder(out, vgl.SCATTER, vgl.ORIGINAL)
            vgl._check(L.vglb_memcpy_d2h(ctx.h, H["out"].ctypes.data, res.ptr, d2h))
            ctx.synchronize()
            dt = time.perf_counter() - t0
            res.free()
            out.free()
            g.free()
            if i > 0:  # first pass warms the allocator
                times.append(dt)
        vgl._check(L.vglb_set_upload_hint(ctx.h, 0))
        return {"seconds": float(np.mean(times)), "h2d": int(h2d), "d2h": int(d2h)}

    def extras(self):
        return None

    def close(self):
        if self.weights is not None:
            self.weights.free()
        self.out.free()
        self.g.free()
        if self._host:
            for a in self._host.values():
                self.vgl.pinned_free(a)
        self._host = None


def make_runner(vgl, ctx, comm, workload, kind, scale, ef, pr_iters, weak=True, vcomm=None):
    if comm is None or comm.world == 1:
        return SingleGpuRunner(vgl, ctx, workload, kind, scale, ef, pr_iters)
    from .multi import PartitionedRunner
    return PartitionedRunner(vgl, ctx, comm, workload, kind, scale, ef, pr_iters, weak=weak, vcomm=vcomm)
