"""Tensor-level layer over the C ABI (include/graphpope_b200.h).

PyTorch is plumbing here — device memory, streams, ``torch.distributed`` — the
work happens in ``libgraphpope_b200.so``.  Every call passes raw device pointers
and the current CUDA stream; nothing in this module computes on the CPU.
"""
from __future__ import annotations

import ctypes
from ctypes import byref, c_int32, c_int64, c_void_p

import numpy as np
import torch

from . import _lib
from ._lib import CsrInfo, MsbfsStats, check


def _stream() -> c_void_p:
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t: torch.Tensor | None) -> c_void_p:
    return c_void_p(0 if t is None else t.data_ptr())


def launch_count() -> int:
    """Kernels launched by libgraphpope_b200.so in this process so far."""
    return int(_lib.load().gp_launch_count())


def device_info() -> dict:
    lib = _lib.require_cuda()
    sm, major, minor = c_int32(), c_int32(), c_int32()
    name = ctypes.create_string_buffer(128)
    check(lib.gp_device_info(byref(sm), byref(major), byref(minor), name, 128))
    return {"sm_count": sm.value, "cc": (major.value, minor.value), "name": name.value.decode()}


class DeviceCsr:
    """De-duplicated digraph in CSR form on the device (``to_networkx`` replacement, utils.py:121)."""

    def __init__(self, num_nodes: int, edge_capacity: int, symmetrize: bool = False):
        self._lib = _lib.require_cuda()
        self.num_nodes = int(num_nodes)
        self.edge_capacity = int(edge_capacity)
        self.symmetrize = bool(symmetrize)
        self._h = c_void_p()
        flags = _lib.GP_CSR_SYMMETRIZE if symmetrize else 0
        check(self._lib.gp_csr_create(self.num_nodes, self.edge_capacity, flags, byref(self._h)))
        self._edges = None

    def build(self, edge_index: torch.Tensor) -> "DeviceCsr":
        """Enqueue the build on the current stream.  ``edge_index``: cuda int64 ``[2, E]``."""
        if edge_index.dim() != 2 or edge_index.size(0) != 2:
            raise ValueError("edge_index must have shape [2, E]")
        if not edge_index.is_cuda or edge_index.dtype != torch.int64:
            raise TypeError("edge_index must be a cuda int64 tensor")
        edge_index = edge_index.contiguous()
        self._edges = edge_index  # keep alive until the stream has consumed it
        check(self._lib.gp_csr_build(self._h, _ptr(edge_index), edge_index.size(1), _stream()))
        return self

    def info(self) -> dict:
        info = CsrInfo()
        check(self._lib.gp_csr_info(self._h, byref(info), _stream()))
        return {k: int(getattr(info, k)) for k, _ in CsrInfo._fields_ if k != "reserved"}

    def export(self, which: str = "out"):
        """(rowptr int32[N+1], col int32[E']) device tensors; ``which`` in {'out', 'in'}."""
        n_edges = self.info()["num_edges"]
        rowptr = torch.empty(self.num_nodes + 1, dtype=torch.int32, device="cuda")
        col = torch.empty(max(n_edges, 1), dtype=torch.int32, device="cuda")
        check(self._lib.gp_csr_export(self._h, {"out": 0, "in": 1}[which], _ptr(rowptr), _ptr(col), _stream()))
        return rowptr, col[:n_edges]

    def degree(self) -> torch.Tensor:
        """In+out degree over de-duplicated edges (utils.py:38-42 score, unnormalised)."""
        deg = torch.empty(self.num_nodes, dtype=torch.int32, device="cuda")
        check(self._lib.gp_degree(self._h, _ptr(deg), _stream()))
        return deg

    def pagerank(self, alpha: float = 0.85, tol: float = 1.0e-6, max_iter: int = 100):
        """networkx ``pagerank_scipy`` defaults (utils.py:26-30).  Returns (x float64[N], iterations)."""
        x = torch.empty(self.num_nodes, dtype=torch.float64, device="cuda")
        it = c_int32()
        check(self._lib.gp_pagerank(self._h, alpha, tol, max_iter, _ptr(x), byref(it), _stream()), iterations=max_iter)
        return x, it.value

    def closeness(self) -> torch.Tensor:
        """networkx ``closeness_centrality`` defaults (utils.py:50-54): float64[N], bit-equal scores."""
        x = torch.empty(self.num_nodes, dtype=torch.float64, device="cuda")
        check(self._lib.gp_closeness(self._h, _ptr(x), _stream()))
        return x

    def clustering(self) -> torch.Tensor:
        """networkx ``clustering(G)`` on the DiGraph (utils.py:56-60): float64[N], bit-equal scores."""
        x = torch.empty(self.num_nodes, dtype=torch.float64, device="cuda")
        check(self._lib.gp_clustering(self._h, _ptr(x), _stream()))
        return x

    def betweenness(self) -> torch.Tensor:
        """networkx ``betweenness_centrality`` defaults (utils.py:32-36): float64[N]; path counts exact, scores
        within a few ulp of networkx (its summation order follows the BFS queue; ours is fixed by node id)."""
        x = torch.empty(self.num_nodes, dtype=torch.float64, device="cuda")
        check(self._lib.gp_betweenness(self._h, _ptr(x), _stream()))
        return x

    def eigenvector(self, tol: float = 1e-15, max_iter: int = 20000):
        """networkx ``eigenvector_centrality_numpy`` (utils.py:44-48) by power iteration on ``A^T + I``:
        (float64[N] unit-norm positive vector, iterations).  Agrees with ARPACK to rounding, not bit for bit."""
        x = torch.empty(self.num_nodes, dtype=torch.float64, device="cuda")
        it = c_int32(0)
        check(self._lib.gp_eigenvector(self._h, tol, max_iter, _ptr(x), byref(it), _stream()), iterations=max_iter)
        return x, it.value

    def close(self):
        if self._h:
            self._lib.gp_csr_free(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def topk_stable(score: torch.Tensor, k: int) -> torch.Tensor:
    """``sorted(score.items(), key=value)`` then ``[-k:]`` (utils.py:29-30): int64 node ids."""
    lib = _lib.require_cuda()
    n = score.numel()
    take = n if (k == 0 or k > n) else k
    out = torch.empty(take, dtype=torch.int64, device="cuda")
    if n == 0:
        return out
    score = score.contiguous()
    if score.dtype == torch.int32:
        check(lib.gp_topk_stable_i32(_ptr(score), n, k, _ptr(out), _stream()))
    elif score.dtype == torch.float64:
        check(lib.gp_topk_stable_f64(_ptr(score), n, k, _ptr(out), _stream()))
    else:
        raise TypeError("topk_stable takes int32 or float64 scores")
    return out


class MsBfs:
    """Multi-source BFS workspace bound to a :class:`DeviceCsr`."""

    def __init__(self, csr: DeviceCsr, max_anchors: int):
        self._lib = _lib.require_cuda()
        self.csr = csr
        self.max_anchors = int(max_anchors)
        self.num_anchors = 0
        self._h = c_void_p()
        check(self._lib.gp_msbfs_create(csr._h, self.max_anchors, byref(self._h)))
        self._anchors = None

    def run(self, anchors: torch.Tensor) -> "MsBfs":
        if not anchors.is_cuda or anchors.dtype != torch.int64:
            raise TypeError("anchors must be a cuda int64 tensor")
        anchors = anchors.contiguous()
        self._anchors = anchors
        self.num_anchors = anchors.numel()
        check(self._lib.gp_msbfs_run(self._h, _ptr(anchors), anchors.numel(), _stream()))
        return self

    def hops_u16(self, out: torch.Tensor | None = None, col_offset: int = 0) -> torch.Tensor:
        n, k = self.csr.num_nodes, self.num_anchors
        if out is None:
            out = torch.empty((n, k), dtype=torch.uint16, device="cuda")
        check(self._lib.gp_msbfs_hops_u16(self._h, _ptr(out), out.stride(0) if out.dim() == 2 and n else k,
                                          col_offset, _stream()))
        return out

    def features(self, x: torch.Tensor | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
        """Fused normalise + concat epilogue: float32 ``[N, F + K]`` (F = 0 without ``x``)."""
        n, k = self.csr.num_nodes, self.num_anchors
        f = 0 if x is None else x.size(1)
        if x is not None:
            if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.size(0) != n:
                raise TypeError("x must be a cuda float32 tensor of shape [N, F]")
            if x.stride(1) != 1:
                x = x.contiguous()
        if out is None:
            out = torch.empty((n, f + k), dtype=torch.float32, device="cuda")
        ld_out = out.stride(0) if n > 1 else f + k
        check(self._lib.gp_msbfs_features(self._h, _ptr(x), f, x.stride(0) if x is not None and n > 1 else f,
                                          _ptr(out), ld_out, f, _stream()))
        return out

    def stats(self) -> dict:
        st = MsbfsStats()
        check(self._lib.gp_msbfs_stats(self._h, byref(st), _stream()))
        return st.as_dict()

    def kernel_ms(self) -> float:
        """Device time of the last persistent MS-BFS kernel alone (events on its launch stream)."""
        ms = ctypes.c_float()
        check(self._lib.gp_msbfs_kernel_ms(self._h, byref(ms)))
        return float(ms.value)

    def set_stage_events(self, enable: bool):
        """Record event nodes around csr build / MS-BFS / epilogue inside the captured pipeline (each node costs ~4 us of
        the replayed step, so they are off by default); needed by :meth:`pipeline_stage_ms` / :meth:`kernel_ms` after
        a replayed run."""
        check(self._lib.gp_msbfs_set_stage_events(self._h, int(bool(enable))))

    def kernel_device_ms(self) -> float:
        """Duration of the last MS-BFS kernel by the device clock (%globaltimer stamps written by the kernel itself:
        entry of thread 0 to the end of the last level); needs no event nodes.  Syncs."""
        ns = ctypes.c_uint64()
        check(self._lib.gp_msbfs_kernel_device_ns(self._h, byref(ns), _stream()))
        return ns.value / 1e6

    def pipeline_stage_ms(self):
        """(csr build, MS-BFS kernel, epilogue) device milliseconds of the last fused run on this handle,
        from event nodes inside the replayed CUDA graph."""
        ms = (ctypes.c_float * 3)()
        check(self._lib.gp_pipeline_stage_ms(self._h, ms))
        return float(ms[0]), float(ms[1]), float(ms[2])

    def planes(self):
        """(uint64 view [num_planes, words], meta dict) of the bit-sliced result, for the gather."""
        ptr, stride = c_void_p(), c_int64()
        nplanes, batches, wb = c_int32(), c_int32(), c_int32()
        check(self._lib.gp_msbfs_planes(self._h, byref(ptr), byref(stride), byref(nplanes), byref(batches),
                                        byref(wb), _stream()))
        meta = {"plane_stride_words": stride.value, "num_planes": nplanes.value, "batches": batches.value,
                "words_per_batch": wb.value, "ptr": ptr.value}
        return meta

    def close(self):
        if self._h:
            self._lib.gp_msbfs_free(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class GeodesicEngine:
    """CSR + MS-BFS handles for one (N, E, K) shape, reusable across calls."""

    def __init__(self, num_nodes: int, edge_capacity: int, max_anchors: int, symmetrize: bool = False):
        self.csr = DeviceCsr(num_nodes, edge_capacity, symmetrize)
        self.bfs = MsBfs(self.csr, max_anchors)

    def fits(self, num_nodes, num_edges, num_anchors, symmetrize) -> bool:
        return (self.csr.num_nodes == num_nodes and self.csr.edge_capacity >= num_edges
                and self.bfs.max_anchors >= num_anchors and self.csr.symmetrize == bool(symmetrize))

    def run(self, edge_index: torch.Tensor, anchors: torch.Tensor, x: torch.Tensor | None = None,
            out: torch.Tensor | None = None) -> torch.Tensor:
        """edge_index -> [N, F + K] features, all enqueued on the current stream (no host sync).

        One C-ABI call (gp_geodesic_run); from the second call with the same tensors on it replays
        a captured CUDA graph.
        """
        n = self.csr.num_nodes
        if edge_index.dim() != 2 or edge_index.size(0) != 2 or not edge_index.is_cuda or edge_index.dtype != torch.int64:
            raise TypeError("edge_index must be a cuda int64 tensor of shape [2, E]")
        if not anchors.is_cuda or anchors.dtype != torch.int64:
            raise TypeError("anchors must be a cuda int64 tensor")
        edge_index, anchors = edge_index.contiguous(), anchors.contiguous()
        k = anchors.numel()
        f = 0 if x is None else x.size(1)
        if x is not None:
            if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.size(0) != n:
                raise TypeError("x must be a cuda float32 tensor of shape [N, F]")
            if x.stride(1) != 1:
                x = x.contiguous()
        if out is None:
            out = torch.empty((n, f + k), dtype=torch.float32, device="cuda")
        self.csr._edges, self.bfs._anchors, self._x = edge_index, anchors, x  # keep alive for the stream
        self.bfs.num_anchors = k
        check(self.csr._lib.gp_geodesic_run(self.csr._h, self.bfs._h, _ptr(edge_index), edge_index.size(1),
                                            _ptr(anchors), k, _ptr(x), f,
                                            x.stride(0) if x is not None and n > 1 else f, _ptr(out),
                                            out.stride(0) if n > 1 else f + k, f, _stream()))
        return out


class FeatureStore:
    """The ``[N, F + K]`` matrix of ``concat_into_features`` (utils.py:129-135) held compactly on the device: x as
    is, the anchor block as a reached bit plus ``bit_length(max hop)`` hop-bit planes per entry (the format is
    documented in include/graphpope_b200.h, gp_fstore_*).  Rows are produced on demand by a fused gather kernel, so
    ``store[n_id]`` stands in for ``data.x[n_id]`` of the trainer (main.py:120,177) without the dense matrix.

    ``FeatureStore(bfs, x)`` packs the last run of an :class:`MsBfs` (the store does not refer to it afterwards);
    ``num_planes`` packs with more planes than the run needs (the extra hop bits are zero), so that stores of
    different anchor shards share one layout.  :meth:`from_shards` merges such shard stores into one.
    """

    def __init__(self, bfs: MsBfs, x: torch.Tensor | None = None, num_planes: int | None = None):
        self._lib = _lib.require_cuda()
        n = bfs.csr.num_nodes
        x = self._device_x(x, n)
        stats = bfs.stats()  # syncs; surfaces index errors of the run
        planes, words = c_int32(), c_int64()
        check(self._lib.gp_fstore_layout(bfs._h, byref(planes), byref(words), _stream()))
        p = planes.value if num_planes is None else int(num_planes)  # too few planes: GP_ERR_INVALID from the pack
        raw = torch.empty((n, p, words.value), dtype=torch.uint64, device="cuda")
        check(self._lib.gp_fstore_pack(bfs._h, _ptr(raw), p, _stream()))
        self._adopt(raw, bfs.num_anchors, x, stats)

    @staticmethod
    def _device_x(x, n):
        if x is not None:
            if x.dtype != torch.float32 or x.dim() != 2 or x.size(0) != n:
                raise TypeError("x must be a float32 tensor of shape [N, F]")
            x = x.to(device="cuda").contiguous()
        return x

    def _adopt(self, raw, k, x, stats):
        self._raw, self._x, self.stats = raw, x, stats
        self.num_nodes, self.num_anchors = raw.size(0), int(k)
        self.num_features = 0 if x is None else x.size(1)
        self._bad = torch.zeros(1, dtype=torch.int32, device="cuda")

    @classmethod
    def from_shards(cls, shards: torch.Tensor, num_anchors: int, x: torch.Tensor | None = None,
                    stats: dict | None = None) -> "FeatureStore":
        """One store from the stores of S contiguous anchor shards, stacked as a cuda uint64 (or int64) tensor
        ``[S, N, P, Ws]``: shard s holds anchors ``distributed.shard_bounds(K, S, s)``, i.e. columns
        ``[s * ceil(K/S), min((s + 1) * ceil(K/S), K))``, packed with the common P and zero-padded to Ws >=
        ceil(ceil(K/S) / 64) words.  ``raw`` is byte-identical to that of one run over all K anchors packed with P
        planes (``FeatureStore.build`` when P is what the deepest shard needs).  Runs on the current stream."""
        lib = _lib.require_cuda()
        if not shards.is_cuda or shards.dim() != 4 or shards.dtype not in (torch.uint64, torch.int64):
            raise TypeError("shards must be a cuda uint64 tensor [S, N, P, Ws]")
        shards = shards.contiguous()
        s, n, p, ws = shards.shape
        k = int(num_anchors)
        per = -(-k // s) if s else 0
        x = cls._device_x(x, n)
        raw = torch.empty((n, p, -(-k // 64)), dtype=torch.uint64, device="cuda")
        check(lib.gp_fstore_merge(_ptr(shards), s, per, ws, n, p, k, _ptr(raw), _stream()))
        store = cls.__new__(cls)
        store._lib = lib
        store._adopt(raw, k, x, {} if stats is None else dict(stats))
        return store

    @classmethod
    def build(cls, edge_index, num_nodes: int, anchors, x: torch.Tensor | None = None,
              symmetrize: bool = False) -> "FeatureStore":
        """csr build + MS-BFS + pack; the BFS workspace is freed before returning."""
        ei = torch.as_tensor(edge_index).to(device="cuda", dtype=torch.int64)
        if ei.dim() != 2 or ei.size(0) != 2:
            raise ValueError("edge_index must have shape [2, E]")
        a = torch.as_tensor(np.asarray(anchors, dtype=np.int64).reshape(-1)).cuda()
        csr = DeviceCsr(int(num_nodes), ei.size(1), symmetrize).build(ei)
        bfs = MsBfs(csr, max(1, a.numel()))
        try:
            return cls(bfs.run(a), x)
        finally:
            bfs.close()
            csr.close()

    # ---- tensor-like surface
    @property
    def shape(self) -> torch.Size:
        return torch.Size((self.num_nodes, self.num_features + self.num_anchors))

    def size(self, dim: int | None = None):
        return self.shape if dim is None else self.shape[dim]

    @property
    def dtype(self) -> torch.dtype:
        return torch.float32

    @property
    def device(self) -> torch.device:
        return self._raw.device

    def __len__(self) -> int:
        return self.num_nodes

    @property
    def num_planes(self) -> int:
        return self._raw.size(1)

    @property
    def nbytes(self) -> int:
        """Bytes of the anchor block (x is held as given)."""
        return self._raw.numel() * 8

    @property
    def raw(self) -> torch.Tensor:
        """The packed records, uint64 ``[N, P, W]``."""
        return self._raw

    def gather(self, rows: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
        """Rows ``rows`` (cuda integer ids; negative ids wrap once) as a cuda float32 ``[B, F + K]``; no host sync.
        Ids outside ``[-N, N)`` give zero rows and are reported by :meth:`check`."""
        if not rows.is_cuda or rows.dtype == torch.bool or rows.is_floating_point() or rows.is_complex():
            raise TypeError("rows must be a cuda integer tensor")
        rows = rows.reshape(-1).to(torch.int64).contiguous()
        b, f, k = rows.numel(), self.num_features, self.num_anchors
        if out is None:
            out = torch.empty((b, f + k), dtype=torch.float32, device="cuda")
        elif (not out.is_cuda or out.dtype != torch.float32 or out.dim() != 2 or tuple(out.shape) != (b, f + k)
              or (out.stride(1) != 1 and f + k > 1)):
            raise TypeError(f"out must be a cuda float32 [{b}, {f + k}] tensor with unit column stride")
        x = self._x
        check(self._lib.gp_fstore_gather(_ptr(self._raw), self.num_nodes, k, self.num_planes, _ptr(rows), b,
                                         _ptr(x), f, x.stride(0) if x is not None else 0, _ptr(out),
                                         out.stride(0) if b > 1 else f + k, f, _ptr(self._bad), _stream()))
        return out

    def check(self):
        """Syncs.  Raises ``IndexError`` if gathers since the last check met ids outside ``[-N, N)`` (once; the
        counter is reset)."""
        bad = int(self._bad.item())
        if bad:
            self._bad.zero_()
            raise IndexError(f"{bad} gathered row ids were outside [-{self.num_nodes}, {self.num_nodes})")

    def __getitem__(self, index):
        """``store[i]``, ``store[a:b:s]``, ``store[ids]`` with ``ids`` a CPU or cuda integer tensor, a numpy array or
        a list, with torch's result shapes.  A host-side index is range-checked before anything is launched."""
        n = self.num_nodes
        if isinstance(index, tuple):
            raise TypeError("FeatureStore takes one row index (no tuples)")
        if isinstance(index, slice):
            return self.gather(torch.arange(*index.indices(n), device="cuda"))
        if isinstance(index, (int, np.integer)) and not isinstance(index, (bool, np.bool_)):
            index = int(index)
            if not -n <= index < n:
                raise IndexError(f"index {index} is out of bounds for dimension 0 with size {n}")
            return self.gather(torch.tensor([index], device="cuda"))[0]
        if not torch.is_tensor(index):
            if isinstance(index, (bool, np.bool_)):
                raise TypeError("FeatureStore does not take boolean masks")
            index = torch.as_tensor(np.asarray(index))
            if index.numel() == 0:
                index = index.to(torch.int64)  # [] -> an empty batch, as in torch
        if index.dtype == torch.bool:
            raise TypeError("FeatureStore does not take boolean masks")
        if index.is_floating_point() or index.is_complex():
            raise IndexError("tensors used as indices must be integer tensors")
        if not index.is_cuda:
            if index.numel() and (int(index.min()) < -n or int(index.max()) >= n):
                bad = index[(index < -n) | (index >= n)].reshape(-1)[0]
                raise IndexError(f"index {int(bad)} is out of bounds for dimension 0 with size {n}")
            index = index.to("cuda")
        return self.gather(index).reshape(*index.shape, self.num_features + self.num_anchors)

    def to_dense(self) -> torch.Tensor:
        """The dense cuda float32 ``[N, F + K]`` matrix (what ``GRAPHPOPE_OUTPUT=cuda`` returns)."""
        return self.gather(torch.arange(self.num_nodes, device="cuda"))

    def __repr__(self):
        return (f"FeatureStore(shape={tuple(self.shape)}, num_planes={self.num_planes}, "
                f"nbytes={self.nbytes}, device={self.device})")


def normalize_into(dist_u16: torch.Tensor, out: torch.Tensor, col_offset: int = 0) -> torch.Tensor:
    lib = _lib.require_cuda()
    n, k = dist_u16.shape
    check(lib.gp_normalize_into(_ptr(dist_u16), n, k, dist_u16.stride(0) if n > 1 else k, _ptr(out),
                                out.stride(0) if n > 1 else out.size(1), col_offset, _stream()))
    return out


class HostContext:
    """Explicit state of the one-call host entry (``gp_ctx_t``): its own handles, device staging, stream and pinned
    ring.  One call at a time per context; separate contexts (e.g. one per host thread) do not serialise."""

    def __init__(self):
        self._lib = _lib.require_cuda()
        self._h = c_void_p()
        check(self._lib.gp_ctx_create(byref(self._h)))

    def close(self):
        if self._h:
            self._lib.gp_ctx_free(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def geodesic_embed_host(edge_index, num_nodes: int, anchors, x=None, symmetrize: bool = False,
                        want_hops: bool = False, out: torch.Tensor | None = None, ctx: HostContext | None = None):
    """One C-ABI call with HOST buffers: returns (features cpu float32 [N, F+K], hops|None, stats).

    This is the boundary the reference-side stub binds (INTEGRATION.md): host
    ``edge_index`` in, host ``[N, F + K]`` out, host<->device copies inside.
    """
    lib = _lib.require_cuda()
    ei = torch.as_tensor(edge_index)
    if ei.dtype != torch.int64 or ei.is_cuda:
        ei = ei.to(device="cpu", dtype=torch.int64)
    ei = ei.contiguous()
    if ei.dim() != 2 or ei.size(0) != 2:
        raise ValueError("edge_index must have shape [2, E]")
    a = torch.as_tensor(np.asarray(anchors, dtype=np.int64)).contiguous()
    n, k = int(num_nodes), a.numel()
    f = 0
    if x is not None:
        x = torch.as_tensor(x)
        if x.is_cuda or x.dtype != torch.float32 or not x.is_contiguous():
            x = x.to(device="cpu", dtype=torch.float32).contiguous()
        f = x.size(1)
    if out is None:
        out = torch.empty((n, f + k), dtype=torch.float32)
    hops = torch.empty((n, k), dtype=torch.uint16) if want_hops else None
    st = MsbfsStats()
    flags = _lib.GP_CSR_SYMMETRIZE if symmetrize else 0
    if ctx is None:
        check(lib.gp_geodesic_embed_host(_ptr(ei), ei.size(1), n, flags, _ptr(a), k, _ptr(x), f, _ptr(out), f + k, f,
                                         _ptr(hops), byref(st)))
    else:
        check(lib.gp_geodesic_embed_host_ctx(ctx._h, _ptr(ei), ei.size(1), n, flags, _ptr(a), k, _ptr(x), f, _ptr(out),
                                             f + k, f, _ptr(hops), byref(st)))
    return out, hops, st.as_dict()


def cdist_minmax(emb: torch.Tensor, anchor_emb: torch.Tensor, mode: int | str, apply_minmax: bool = True,
                 out: torch.Tensor | None = None, col_offset: int = 0) -> torch.Tensor:
    """Pairwise block of attach_node2vec (utils.py:174-176) on the tensor cores: float32 ``[N, K]``."""
    lib = _lib.require_cuda()
    if isinstance(mode, str):
        mode = _lib.CDIST_MODES[mode]
    emb = emb.to(device="cuda", dtype=torch.float32).contiguous()
    anchor_emb = anchor_emb.to(device="cuda", dtype=torch.float32).contiguous()
    n, d = emb.shape
    k = anchor_emb.size(0)
    if anchor_emb.size(1) != d:
        raise ValueError("embedding dimensions differ")
    if out is None:
        out = torch.empty((n, k), dtype=torch.float32, device="cuda")
        col_offset = 0
    check(lib.gp_cdist_minmax(_ptr(emb), _ptr(anchor_emb), n, k, d, int(mode), int(bool(apply_minmax)),
                              _ptr(out), out.stride(0) if n > 1 else out.size(1), col_offset, _stream()))
    return out


def kmeans(table: torch.Tensor, num_clusters: int, n_init: int = 10, max_iter: int = 300, tol: float = 1.0e-4,
           seed: int | None = None):
    """KMeans cluster centres of the node2vec table on the device (utils.py:168-170 uses scikit-learn's
    ``KMeans(n_clusters=K).fit(table).cluster_centers_`` with its defaults: k-means++, n_init = 10,
    max_iter = 300, tol = 1e-4 scaled by the mean feature variance, unseeded).

    Returns ``(centers float32 [K, D] on the device, inertia, iterations of the best run)``.  Parity with
    scikit-learn is statistical (the reference does not seed it): same objective, same stopping rule.  One known
    divergence: a cluster that loses all its rows keeps its previous centre here, where scikit-learn moves it onto
    the row farthest from its own centre; after a k-means++ start this is rare and only lowers the odds of that run
    being the best of ``n_init`` (the result is still the run with the lowest inertia).  Tables wider than 128
    columns are not clustered on the device (``utils.attach_node2vec`` keeps scikit-learn for those).
    """
    lib = _lib.require_cuda()
    x = table.to(device="cuda", dtype=torch.float32).contiguous()
    n, d_in = x.shape
    if d_in > 128:
        raise ValueError("device k-means covers embedding widths up to 128 (the reference writes 128-d tables)")
    if d_in not in (64, 128):
        # the kernels are instantiated for 64 and 128 columns: zero columns change neither distances nor means
        x = torch.nn.functional.pad(x, (0, (64 if d_in < 64 else 128) - d_in)).contiguous()
    d = x.size(1)
    k = int(num_clusters)
    if k <= 0 or k > n:
        raise ValueError(f"n_clusters={k} must be in [1, {n}]")
    rng = np.random.default_rng(seed)
    tol_abs = float(tol) * float(x.var(dim=0, unbiased=False).mean().item())  # sklearn _tolerance()
    centers = torch.empty((k, d), dtype=torch.float32, device="cuda")
    mind2 = torch.empty(n, dtype=torch.float32, device="cuda")
    chosen = torch.empty(k, dtype=torch.int64, device="cuda")
    best = torch.empty(n, dtype=torch.int64, device="cuda")  # uint64 payload
    sums = torch.empty((k, d), dtype=torch.float32, device="cuda")
    counts = torch.empty(k, dtype=torch.int32, device="cuda")
    scal = torch.zeros(2, dtype=torch.float64, device="cuda")  # [shift2, inertia]
    result = None
    for _ in range(max(1, int(n_init))):
        check(lib.gp_kmeans_plusplus(_ptr(x), n, k, d, int(rng.integers(0, n)), int(rng.integers(0, 2**63 - 1)),
                                     _ptr(centers), _ptr(mind2), _ptr(chosen), _stream()))
        iters = 0
        for it in range(1, int(max_iter) + 1):
            check(lib.gp_kmeans_assign(_ptr(x), _ptr(centers), n, k, d, _ptr(best), _stream()))
            check(lib.gp_kmeans_update(_ptr(x), _ptr(best), n, k, d, _ptr(centers), _ptr(sums), _ptr(counts),
                                       c_void_p(scal.data_ptr()), c_void_p(scal.data_ptr() + 8), _stream()))
            iters = it
            if it % 4 == 0 or it == max_iter:  # the stopping test needs a host round trip: every 4th iteration
                if float(scal[0].item()) <= tol_abs:
                    break
        # inertia of the final centres (the update above measured the assignment to the previous ones)
        check(lib.gp_kmeans_assign(_ptr(x), _ptr(centers), n, k, d, _ptr(best), _stream()))
        inertia = float((best >> 32).to(torch.int32).view(torch.float32).double().sum().item())
        if result is None or inertia < result[1]:
            result = (centers[:, :d_in].clone(), inertia, iters)
    return result
