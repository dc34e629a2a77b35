"""Anchor-sharded multi-GPU geodesic embedding (one process per GPU, torch.distributed / NCCL).

The reference shards its CPU pool by *node slice* (utils.py:99-100) because its unit of work is
a (node, anchor) pair; every DDP rank then recomputes the identical embedding (main.py:88-98).
Here the BFS is sharded by *anchor*: the CSR is replicated, rank r owns anchors
``[r*K/G, (r+1)*K/G)`` as its own bit lanes, and there is no exchange during traversal.  The one
real exchange step is assembling the replicated ``[N, F+K]`` output: ranks all-gather their
bit-sliced result planes (≈ (1 + log2(max hops)) bits per (node, anchor) instead of 16 or 32) and
each rank's epilogue kernel decodes all shards, performing the ``[G][N][K/G] -> [N, F + g*K/G + j]``
column permutation while it writes fp32.

The host-side logic below (shard bounds, plane-count agreement, gather layout) is backend
agnostic so the world_size-2 ``gloo`` tests can drive it with CPU tensors.
"""
from __future__ import annotations

import os
from ctypes import c_void_p

import torch
import torch.distributed as dist


def shard_bounds(num_anchors: int, world_size: int, rank: int) -> tuple[int, int]:
    """Contiguous anchor shards of ``ceil(K / G)`` columns; when G does not divide K the last ranks hold fewer
    (possibly zero) anchors.  The reference accepts any K (utils.py:24, main.py:37: the default is 2)."""
    per = -(-int(num_anchors) // int(world_size))
    return min(num_anchors, rank * per), min(num_anchors, (rank + 1) * per)


def pad_anchors(anchors, world_size: int, multiple: int = 8):
    """The device exchange needs every rank to own the same number of lanes, a multiple of ``multiple`` (a decode
    lane owns 8 columns).  Returns ``(padded anchors, anchors per rank)``: K is padded up to ``G * per`` by repeating
    the last anchor — duplicate anchors are legal (sampling is with replacement, utils.py:24) and the padded columns
    are dropped by the caller."""
    k = len(anchors)
    per = -(-max(k, 1) // world_size)
    per = -(-per // multiple) * multiple
    pad = world_size * per - k
    if pad == 0:
        return anchors, per
    if torch.is_tensor(anchors):
        fill = anchors[-1:].expand(pad) if k else torch.zeros(pad, dtype=anchors.dtype, device=anchors.device)
        return torch.cat([anchors, fill]), per
    import numpy as np

    a = np.asarray(anchors, dtype=np.int64)
    return np.concatenate([a, np.full(pad, a[-1] if k else 0, dtype=np.int64)]), per


def agree_num_planes(local_num_planes: int, group=None, device="cpu") -> int:
    """All ranks must decode the same number of planes: the max over ranks (one tiny all-reduce)."""
    t = torch.tensor([int(local_num_planes)], dtype=torch.int32, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return int(t.item())


def gather_planes(local_planes: torch.Tensor, group=None) -> torch.Tensor:
    """all-gather equal-shaped int64 plane blocks ``[P, words]`` into ``[G, P, words]``."""
    world = dist.get_world_size(group)
    flat = local_planes.contiguous().view(-1)
    out = torch.empty(world * flat.numel(), dtype=flat.dtype, device=flat.device)
    dist.all_gather_into_tensor(out, flat, group=group)  # flat shapes: accepted by both NCCL and gloo
    return out.view((world,) + tuple(local_planes.shape))


def anchor_checksum(anchors) -> int:
    """A 62-bit digest of the anchor list (count and values, in order), non-negative in an int64."""
    import hashlib

    import numpy as np

    a = np.ascontiguousarray(np.asarray(torch.as_tensor(anchors).cpu(), dtype=np.int64).reshape(-1))
    h = hashlib.blake2b(np.int64([a.size]).tobytes() + a.tobytes(), digest_size=8).digest()
    return int.from_bytes(h, "little") >> 2


def check_anchors_agree(anchors, group=None, device="cpu"):
    """Raises ``ValueError`` on every rank unless every rank passed the same anchor list: all-reduce MIN and MAX of
    :func:`anchor_checksum`.  A sharded build from different lists would silently mix columns of different runs."""
    c = anchor_checksum(anchors)
    lo = torch.tensor([c], dtype=torch.int64, device=device)
    hi = lo.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN, group=group)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX, group=group)
    if int(lo.item()) != int(hi.item()):
        raise ValueError("the ranks passed different anchor lists to a collective anchor-sharded build (same seed "
                         "and sampler on every rank are needed)")


def agree_store_layout(local_num_planes: int, local_max_level: int, failed: bool = False, group=None,
                       device="cpu") -> tuple[int, int, bool]:
    """(P, max_level, some rank failed): the max over ranks of each, in one all-reduce.  The largest finite hop over
    all shards is the one-GPU ``max_level``, so the agreed P is the one a single run over all anchors packs with."""
    t = torch.tensor([int(local_num_planes), int(local_max_level), int(bool(failed))], dtype=torch.int64,
                     device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    p, level, bad = t.tolist()
    return int(p), int(level), bool(bad)


def shard_words(num_anchors: int, world_size: int) -> int:
    """Ws: uint64 words per plane of every rank's shard store, enough for the ``ceil(K/G)`` anchors of a full
    shard, so that all ranks' blocks have one shape for the all-gather."""
    per = -(-int(num_anchors) // int(world_size))
    return -(-per // 64)


def pad_shard_store(raw: torch.Tensor | None, num_nodes: int, num_planes: int, words: int,
                    device="cpu") -> torch.Tensor:
    """A shard store ``[N, P_local, W_local]`` (``None``: a rank without anchors) as an int64 ``[N, P, Ws]`` block,
    zero in the planes and words it lacks; the store itself (viewed as int64) when it already has that shape."""
    shape = (int(num_nodes), int(num_planes), int(words))
    if raw is not None and tuple(raw.shape) == shape:
        return raw.view(torch.int64)
    block = torch.zeros(shape, dtype=torch.int64, device=raw.device if raw is not None else device)
    if raw is not None:
        block[:, :raw.size(1), :raw.size(2)].copy_(raw.view(torch.int64))
    return block


def sharded_feature_store(edge_index, num_nodes: int, anchors, x: torch.Tensor | None = None,
                          symmetrize: bool = False, group=None):
    """Collective: every rank calls it with the same arguments and gets the same :class:`device.FeatureStore` of all
    K anchors, whose ``raw`` is byte-identical to ``FeatureStore.build(edge_index, num_nodes, anchors, x)`` on one
    GPU.  Rank r runs the csr build and the MS-BFS for its anchors ``shard_bounds(K, G, r)`` only (a BFS workspace of
    ``ceil(K/G)`` lanes), packs them with the P agreed over the ranks into a zero-padded ``[N, P, Ws]`` block, frees
    the BFS workspace, all-gathers the G blocks and merges them into the one-GPU record layout (gp_fstore_merge).
    Peak device memory is about twice the store plus x.  ``store.stats`` holds this rank's MS-BFS counters with
    ``max_level`` the max over the ranks.  Needs a process group that all-gathers cuda tensors (NCCL)."""
    import numpy as np

    from ._lib import MsbfsStats
    from .device import DeviceCsr, FeatureStore, MsBfs

    backend = str(dist.get_backend(group))
    if "nccl" not in backend:
        raise RuntimeError(f"sharded_feature_store all-gathers cuda tensors and needs an NCCL process group, "
                           f"not {backend!r}")
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    a = np.ascontiguousarray(np.asarray(torch.as_tensor(anchors).cpu(), dtype=np.int64).reshape(-1))
    n, k = int(num_nodes), a.size
    check_anchors_agree(a, group, device="cuda")
    lo, hi = shard_bounds(k, world, rank)
    ws = shard_words(k, world)
    csr = bfs = None
    stats = MsbfsStats().as_dict()  # a rank without anchors: all counters zero
    error = None
    try:
        ei = torch.as_tensor(edge_index).to(device="cuda", dtype=torch.int64)
        if ei.dim() != 2 or ei.size(0) != 2:
            raise ValueError("edge_index must have shape [2, E]")
        if hi > lo:
            csr = DeviceCsr(n, ei.size(1), symmetrize).build(ei)
            bfs = MsBfs(csr, hi - lo).run(torch.from_numpy(a[lo:hi]).cuda())
            stats = bfs.stats()  # syncs; surfaces index errors of the run
    except Exception as e:  # reported to the other ranks below instead of leaving them in a collective
        error = e
    local_planes = 1 + int(stats["max_level"]).bit_length()
    try:
        p, max_level, failed = agree_store_layout(local_planes, stats["max_level"], error is not None, group, "cuda")
        if error is not None:
            raise error
        if failed:
            raise RuntimeError("sharded_feature_store failed on another rank")
        shard = FeatureStore(bfs, num_planes=p).raw if bfs is not None else None
    finally:
        for h in (bfs, csr):
            if h is not None:
                h.close()
    block = pad_shard_store(shard, n, p, ws, device="cuda")
    del shard
    gathered = gather_planes(block, group)  # [G, N, P, Ws] int64
    del block
    stats = dict(stats, max_level=max_level)
    return FeatureStore.from_shards(gathered, k, x, stats)


def _wrap_device_words(ptr: int, nwords: int) -> torch.Tensor:
    """Zero-copy int64 view of library-owned device memory (the bit planes of the last run)."""
    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (nwords,), "typestr": "<i8", "data": (ptr, False), "version": 2}
    return torch.as_tensor(h, device="cuda")


def sharded_geodesic_features(engine, edge_index: torch.Tensor, anchors: torch.Tensor,
                              x: torch.Tensor | None = None, out: torch.Tensor | None = None,
                              group=None) -> torch.Tensor:
    """Every rank returns the full float32 ``[N, F + K]`` block; rank r ran only its K/G anchors.

    ``engine`` is a :class:`graphpope_b200.device.GeodesicEngine` sized for K/G anchors;
    ``anchors`` holds all K anchors (identical on every rank: same seed, same sampler).
    """
    from . import _lib
    from ._lib import check
    from .device import _ptr, _stream

    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    n = engine.csr.num_nodes
    k = anchors.numel()
    f = 0 if x is None else x.size(1)
    if out is None:
        out = torch.empty((n, f + k), dtype=torch.float32, device="cuda")
    if world == 1:
        return engine.run(edge_index, anchors, x, out)
    if k % world:
        raise ValueError(f"the all-gather path needs num_anchor_nodes={k} divisible by the world size {world}; "
                         "PeerAssembly pads a ragged K itself")
    lo, hi = shard_bounds(k, world, rank)
    engine.csr.build(edge_index)
    engine.bfs.run(anchors[lo:hi].contiguous())
    meta = engine.bfs.planes()  # syncs: needs max_level
    stride = meta["plane_stride_words"]
    num_planes = agree_num_planes(meta["num_planes"], group, device="cuda")
    local = _wrap_device_words(meta["ptr"], 32 * stride)[: num_planes * stride].view(num_planes, stride)
    if num_planes > meta["num_planes"]:
        local[meta["num_planes"]:].zero_()  # planes this shard never reached hold stale bits
    gathered = gather_planes(local, group)  # [G, P, words] int64
    lib = _lib.load()
    check(lib.gp_decode_gathered(_ptr(gathered), num_planes * stride, world, n, hi - lo, num_planes,
                                 meta["batches"], meta["words_per_batch"], stride, _ptr(x), f,
                                 x.stride(0) if x is not None and n > 1 else f, _ptr(out),
                                 out.stride(0) if n > 1 else f + k, f, _stream()))
    return out


def sharded_geodesic_embed_host(engine, edge_index: torch.Tensor, anchors, x: torch.Tensor | None,
                                out: torch.Tensor, staging: dict, group=None, peer=None) -> torch.Tensor:
    """Host-buffer form of the sharded path (what a DataModule calls): HOST ``edge_index`` / ``x`` in,
    HOST float32 ``[N, F + K]`` out.  ``staging`` caches the device / pinned scratch between calls."""
    from . import _lib
    from ._lib import check
    from .device import _ptr

    n = engine.csr.num_nodes
    a = torch.as_tensor(anchors)
    k = a.numel()
    f = 0 if x is None else x.size(1)
    if staging.get("shape") != (n, k, edge_index.size(1)):
        staging.clear()
        staging["shape"] = (n, k, edge_index.size(1))
        staging["ei"] = torch.empty_like(edge_index, device="cuda")
        staging["anchors"] = torch.empty(k, dtype=torch.int64, device="cuda")
        staging["block_d"] = torch.empty((n, k), dtype=torch.float32, device="cuda")
        staging["block_h"] = torch.empty((n, k), dtype=torch.float32).pin_memory()
    staging["ei"].copy_(edge_index, non_blocking=True)
    staging["anchors"].copy_(a, non_blocking=True)
    lib = _lib.load()
    direct = out.is_pinned() and out.stride(1) == 1  # strided DMA straight into columns [F, F + K) of `out`

    def device_to_host():
        if direct:
            check(lib.gp_block_to_host(_ptr(staging["block_d"]), n, k, _ptr(out), out.stride(0), f,
                                       c_void_p(torch.cuda.current_stream().cuda_stream)))
        else:
            staging["block_h"].copy_(staging["block_d"], non_blocking=True)  # one contiguous DMA, scattered below

    if peer is not None:
        _, deep = peer.run(staging["ei"], staging["anchors"], None, staging["block_d"])
    else:
        deep = None
        sharded_geodesic_features(engine, staging["ei"], staging["anchors"], None, staging["block_d"], group)
    device_to_host()
    # concat_into_features (utils.py:129-135): x goes into columns [0, F) on the host while the GPU works
    if x is not None:
        check(lib.gp_host_concat(_ptr(x), f, None, 0, n, _ptr(out), out.stride(0)))
    torch.cuda.current_stream().synchronize()
    if deep is not None and int(deep.item()) != 0:  # hops > 15 somewhere: redo through the all-gather path
        sharded_geodesic_features(engine, staging["ei"], staging["anchors"], None, staging["block_d"], group)
        device_to_host()
        torch.cuda.current_stream().synchronize()
    if not direct:
        check(lib.gp_host_concat(None, f, _ptr(staging["block_h"]), k, n, _ptr(out), out.stride(0)))
    return out


class SharedHostMatrix:
    """One float32 ``[rows, cols]`` matrix in POSIX shared memory per node, page-locked in every rank.

    The reference runs ``Graphpope`` in every DDP rank (main.py:88-98) and afterwards only indexes ``data.x[n_id]``
    (main.py:120,177), so all ranks of a node hold identical ``[N, F+K]`` host matrices.  Here there is ONE: rank 0
    creates ``/dev/shm/<name>``, every rank maps the same pages, registers them with CUDA (``cudaHostRegister``) so
    device-to-host DMAs can land in it directly, and wraps the mapping as a torch tensor.  Rank r then writes only
    its own column block (and its row range of ``x``), a barrier later every rank sees the whole matrix.
    """

    def __init__(self, rows: int, cols: int, group=None, name: str | None = None, register: bool = True):
        import mmap
        import uuid

        import numpy as np

        self.rows, self.cols, self.group = int(rows), int(cols), group
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        nbytes = max(4 * self.rows * self.cols, mmap.PAGESIZE)
        self.nbytes = -(-nbytes // mmap.PAGESIZE) * mmap.PAGESIZE
        box = [os.path.basename(name) if name else "graphpope_%s" % uuid.uuid4().hex, None]
        if self.rank == 0:
            # rank 0 creates the file and RESERVES its pages before anyone maps it: a full /dev/shm is an OSError
            # here (reported on every rank), not a SIGBUS at the first touch inside cudaHostRegister
            path = os.path.join("/dev/shm", box[0])
            try:
                fd = os.open(path, os.O_CREAT | os.O_RDWR | os.O_TRUNC, 0o600)
                try:
                    os.posix_fallocate(fd, 0, self.nbytes)
                except OSError:
                    os.close(fd)
                    os.unlink(path)
                    raise
            except OSError as err:
                box[1] = f"{path}: {err}"
        if self.world > 1:
            dist.broadcast_object_list(box, src=0, group=group)  # also orders "created" before the other ranks' open
        if box[1] is not None:
            raise RuntimeError(f"cannot create the node-shared matrix ({self.nbytes} bytes): {box[1]}")
        self.path = os.path.join("/dev/shm", box[0])
        if self.rank != 0:
            fd = os.open(self.path, os.O_RDWR)
        self._mm = mmap.mmap(fd, self.nbytes, mmap.MAP_SHARED, mmap.PROT_READ | mmap.PROT_WRITE)
        os.close(fd)
        if self.world > 1:
            dist.barrier(group=group)
        if self.rank == 0:
            os.unlink(self.path)  # every rank holds its mapping; the name is no longer needed
        arr = np.frombuffer(self._mm, dtype=np.float32, count=self.rows * self.cols).reshape(self.rows, self.cols)
        self.tensor = torch.from_numpy(arr)
        self._registered = False
        self.shard = (0, 0)
        if register and torch.cuda.is_available():
            rc = torch.cuda.cudart().cudaHostRegister(self.tensor.data_ptr(), self.nbytes, 0)
            if int(rc) != 0:
                raise RuntimeError(f"cudaHostRegister of the shared matrix failed with error {int(rc)}")
            self._registered = True

    def barrier(self):
        if self.world > 1:
            dist.barrier(group=self.group)

    def close(self):
        if self._registered:
            torch.cuda.cudart().cudaHostUnregister(self.tensor.data_ptr())
            self._registered = False
        self.tensor = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def row_slice(num_rows: int, world_size: int, rank: int) -> tuple[int, int]:
    """Rank r's share of a row-partitioned host copy (``x`` into columns ``[0, F)``)."""
    per = -(-int(num_rows) // int(world_size))
    return min(num_rows, rank * per), min(num_rows, (rank + 1) * per)


def sharded_embed_host_shared(engine, edge_index: torch.Tensor, anchors, x: torch.Tensor | None,
                              shared: "SharedHostMatrix", staging: dict) -> torch.Tensor:
    """Host contract of the geodesic path for the ranks of one node WITHOUT assembling anything on the device
    (SURVEY §8 f3): HOST ``edge_index`` / ``x`` in, the node-shared HOST ``[N, F + K]`` matrix out.

    Rank r runs the MS-BFS for its anchor shard only, decodes its own ``[N, K/G]`` block and DMAs it straight
    into columns ``[F + lo, F + hi)`` of the shared matrix; the copy of ``x`` (concat_into_features,
    utils.py:129-135) is split by row range across the ranks; one barrier, then every rank returns the same
    tensor.  Per rank and step: H2D = edge_index + its anchors, D2H = N * K/G floats (1/G of what the
    replicated assembly moved), host copy = N/G rows of x.  Bit-equal to the 1-GPU result.
    """
    from . import _lib
    from ._lib import check
    from .device import _ptr

    import numpy as np

    n = engine.csr.num_nodes
    a = torch.as_tensor(np.asarray(anchors, dtype=np.int64))
    k = a.numel()
    f = 0 if x is None else x.size(1)
    out = shared.tensor
    if tuple(out.shape) != (n, f + k):
        raise ValueError(f"shared matrix is {tuple(out.shape)}, expected {(n, f + k)}")
    rank, world = shared.rank, shared.world
    lo, hi = shard_bounds(k, world, rank)
    shared.shard = (lo, hi)  # the anchor columns this rank computed
    kr = hi - lo
    key = (n, kr, edge_index.size(1))
    if staging.get("shape") != key:
        staging.clear()
        staging["shape"] = key
        staging["ei"] = torch.empty_like(edge_index, device="cuda")
        staging["anchors"] = torch.empty(max(kr, 1), dtype=torch.int64, device="cuda")
        staging["block_d"] = torch.empty((n, max(kr, 1)), dtype=torch.float32, device="cuda")
        staging["a_pin"] = torch.empty(max(kr, 1), dtype=torch.int64).pin_memory()
    lib = _lib.load()
    stream = c_void_p(torch.cuda.current_stream().cuda_stream)
    if kr > 0:
        staging["ei"].copy_(edge_index, non_blocking=True)
        staging["a_pin"][:kr].copy_(a[lo:hi])
        staging["anchors"][:kr].copy_(staging["a_pin"][:kr], non_blocking=True)
        engine.run(staging["ei"], staging["anchors"][:kr], None, staging["block_d"][:, :kr])
        check(lib.gp_block_to_host(_ptr(staging["block_d"]), n, kr, _ptr(out), out.stride(0), f + lo, stream))
    if x is not None and f > 0:
        if not x.is_contiguous():
            x = x.contiguous()
        r0, r1 = row_slice(n, world, rank)
        if r1 > r0:  # this rank's rows of x, on the host while the GPU works
            check(lib.gp_host_concat(c_void_p(x.data_ptr() + 4 * r0 * x.stride(0)), f, None, 0, r1 - r0,
                                     c_void_p(out.data_ptr() + 4 * r0 * out.stride(0)), out.stride(0)))
    torch.cuda.current_stream().synchronize()
    engine.bfs.stats() if kr > 0 else None  # surfaces latched device errors (bad index, uint16 overflow)
    shared.barrier()
    return out


class PushExchange:
    """The exchange step as ONE kernel over NVLink peer memory (csrc/gp_exchange.cu): every rank packs its result
    into its own exchange buffer and raises a flag on the peers; its row-streaming epilogue then gathers the peers'
    packed row segments into shared memory with the bulk-copy engine, two row blocks ahead of the rows it writes.
    No collective library call, no host round trip; the whole step (csr build + MS-BFS + exchange / decode) replays
    from one CUDA graph.

    Collective: every rank constructs it together and calls :meth:`run` once per step, in the same order.
    Sharing one process (tests: several "ranks" on one GPU) is supported through ``peers=``.
    """

    def __init__(self, engine, group=None, world=None, rank=None, grid_blocks=0):
        import ctypes

        from . import _lib
        from ._lib import check

        self.engine, self.group = engine, group
        self.lib = _lib.load()
        self.world = dist.get_world_size(group) if world is None else int(world)
        self.rank = dist.get_rank(group) if rank is None else int(rank)
        if self.world > 8:
            raise ValueError("the push exchange covers the GPUs of one NVSwitch node (<= 8 ranks)")
        self._h = c_void_p()
        check(self.lib.gp_exchange_create(engine.bfs._h, self.world, self.rank, ctypes.byref(self._h)))
        if grid_blocks:  # ranks sharing one GPU (tests): partial grids, so that all of them are resident at once
            check(self.lib.gp_exchange_set_grid(self._h, int(grid_blocks)))
        self._opened = []
        self._pad = {}
        if world is None and self.world > 1:  # one process per GPU: CUDA IPC mappings of the other ranks' buffers
            handle = (ctypes.c_uint8 * 64)()
            check(self.lib.gp_exchange_ipc_export(self._h, handle))
            mine = torch.tensor(list(bytes(handle)), dtype=torch.uint8, device="cuda")
            every = torch.empty(self.world * 64, dtype=torch.uint8, device="cuda")
            dist.all_gather_into_tensor(every, mine, group=group)
            every = every.cpu().view(self.world, 64)
            for r in range(self.world):
                if r == self.rank:
                    continue
                buf = (ctypes.c_uint8 * 64)(*every[r].tolist())
                ptr = c_void_p()
                check(self.lib.gp_ipc_open(buf, ctypes.byref(ptr)))
                self._opened.append(ptr.value)
                check(self.lib.gp_exchange_set_peer(self._h, r, ptr))
            dist.barrier(group=group)

    def local_ptr(self) -> int:
        import ctypes

        from ._lib import check
        ptr = c_void_p()
        check(self.lib.gp_exchange_local_ptr(self._h, ctypes.byref(ptr)))
        return ptr.value

    def set_peer(self, rank: int, ptr: int):
        from ._lib import check
        check(self.lib.gp_exchange_set_peer(self._h, int(rank), c_void_p(ptr)))

    def run(self, edge_index, anchors, x=None, out=None):
        """Every rank returns the full float32 ``[N, F + K]`` block; this rank ran only its K/G anchors.
        ``anchors`` holds all K anchors (identical on every rank).  Returns ``(out, self)``; ``self.item()`` is 1 if
        some shard had hops > 15 (then redo the step with :func:`sharded_geodesic_features`)."""
        from ._lib import check
        from .device import _ptr, _stream

        eng = self.engine
        n = eng.csr.num_nodes
        k = anchors.numel()
        f = 0 if x is None else x.size(1)
        if out is None:
            out = torch.empty((n, f + k), dtype=torch.float32, device="cuda")
        # stable tensors = stable graph keys; a ragged K is padded with repeats of the last anchor.  The entry keeps
        # `anchors` itself: its storage cannot be freed and handed to another tensor while the key is live, and an
        # in-place update (version counter) re-derives the padded copy
        key = (anchors.data_ptr(), k, anchors._version)
        if key not in self._pad:
            padded, per = pad_anchors(anchors, self.world)
            shard = padded[self.rank * per:(self.rank + 1) * per].contiguous()
            tmp = None if padded.numel() == k else torch.empty((n, f + padded.numel()), dtype=torch.float32, device="cuda")
            self._pad = {key: (shard, per, tmp, anchors)}
        shard, per, tmp, _ = self._pad[key]
        dst = out if tmp is None else tmp
        edge_index = edge_index.contiguous()
        if x is not None and x.stride(1) != 1:
            x = x.contiguous()
        eng.csr._edges, eng.bfs._anchors, eng.bfs.num_anchors, self._x = edge_index, shard, per, x
        check(self.lib.gp_geodesic_run_exchange(eng.csr._h, eng.bfs._h, self._h, _ptr(edge_index), edge_index.size(1),
                                                _ptr(shard), per, _ptr(x), f, x.stride(0) if x is not None and n > 1 else f,
                                                _ptr(dst), dst.stride(0) if n > 1 else dst.size(1), f, _stream()))
        if tmp is not None:
            out.copy_(tmp[:, :f + k])
        return out, self

    def item(self) -> int:
        """Syncs.  1 if the last step hit hops > 15 somewhere; raises if a peer's data never arrived."""
        import ctypes

        from ._lib import check
        from .device import _stream
        deep = ctypes.c_int32(0)
        check(self.lib.gp_exchange_status(self._h, ctypes.byref(deep), _stream()))
        return int(deep.value)

    trace_events = ()

    def trace(self):
        """Diagnostics: microseconds from the start of the last exchange kernel (block 0) to: its share packed, every
        peer's flag seen, and the last block leaving."""
        import ctypes

        from ._lib import check
        st = (ctypes.c_uint64 * 8)()
        check(self.lib.gp_exchange_trace(self._h, st))
        t0 = st[0]
        return {"packed_us": (st[1] - t0) / 1e3, "flags_seen_us": (st[2] - t0) / 1e3, "end_us": (st[3] - t0) / 1e3}

    def close(self):
        for p in self._opened:
            self.lib.gp_ipc_close(c_void_p(p))
        self._opened = []
        if self._h:
            self.lib.gp_exchange_free(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def PeerAssembly(engine, group=None):
    """The device exchange of the sharded path: the push kernel (default) or round 1's pull-based peer decode
    (``GP_EXCHANGE=pull``: pack + NCCL flag all-reduce + an epilogue that reads the peers' shards over NVLink)."""
    if os.environ.get("GP_EXCHANGE", "push") == "pull":
        return PullAssembly(engine, group)
    return PushExchange(engine, group)


class PullAssembly:
    """NVLink peer-to-peer assembly of the sharded result (the B200-native form of the exchange step).

    Instead of all-gathering result masks into a staging buffer and then decoding, every rank maps the
    other ranks' packed result buffers (CUDA IPC over NVSwitch) once, and the fused epilogue kernel
    reads them *in place* while it writes the fp32 rows: own shard from HBM, peer shards through
    NVLink loads, so the transfer overlaps the HBM-bound output writes tile by tile.  Per step there
    is one tiny NCCL all-reduce (it carries the "hops > 15" flag and doubles as the cross-GPU barrier
    that orders pack before decode); buffers are double-buffered so no second barrier is needed.
    """

    def __init__(self, engine, group=None):
        import ctypes

        from . import _lib
        from ._lib import check

        self.engine, self.group = engine, group
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        if self.world > 8:
            raise ValueError("PeerAssembly covers the GPUs of one NVSwitch node (<= 8 ranks)")
        self.lib = _lib.load()
        handle = (ctypes.c_uint8 * 64)()
        slot_stride = ctypes.c_int64()
        check(self.lib.gp_msbfs_ipc_export(engine.bfs._h, handle, ctypes.byref(slot_stride)))
        self.slot_stride_words = slot_stride.value
        mine = torch.tensor(list(bytes(handle)), dtype=torch.uint8, device="cuda")
        every = torch.empty(self.world * 64, dtype=torch.uint8, device="cuda")
        dist.all_gather_into_tensor(every, mine, group=group)
        every = every.cpu().view(self.world, 64)
        self.base = []
        self._opened = []
        for r in range(self.world):
            if r == self.rank:
                self.base.append(None)  # filled from gp_msbfs_pack (own allocation)
                continue
            buf = (ctypes.c_uint8 * 64)(*every[r].tolist())
            ptr = ctypes.c_void_p()
            check(self.lib.gp_ipc_open(buf, ctypes.byref(ptr)))
            self.base.append(ptr.value)
            self._opened.append(ptr.value)
        self.step = 0
        self.trace_events = []
        self.flag = torch.zeros(1, dtype=torch.int32, device="cuda")

    def close(self):
        for p in self._opened:
            self.lib.gp_ipc_close(c_void_p(p))
        self._opened = []

    def run(self, edge_index, anchors, x=None, out=None):
        """Same contract as :func:`sharded_geodesic_features`; returns (out, deep) where ``deep`` is a
        device int32 that is 1 if some shard had hops > 15 (then the caller must use the gather path)."""
        import ctypes

        from ._lib import check
        from .device import _ptr, _stream

        eng = self.engine
        n = eng.csr.num_nodes
        k = anchors.numel()
        f = 0 if x is None else x.size(1)
        if out is None:
            out = torch.empty((n, f + k), dtype=torch.float32, device="cuda")
        lo, hi = shard_bounds(k, self.world, self.rank)
        slot = self.step & 1
        self.step += 1
        key = (anchors.data_ptr(), lo, hi)
        if getattr(self, "_shard_key", None) != key:  # keep the shard tensor alive and its pointer stable (graph key)
            self._shard_key, self._shard = key, anchors[lo:hi].contiguous()
        edge_index = edge_index.contiguous()
        eng.csr._edges, eng.bfs._anchors, eng.bfs.num_anchors = edge_index, self._shard, hi - lo
        trace = os.environ.get("GP_PEER_TRACE") is not None  # diagnostics: device time of the three phases
        if trace:
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
            ev[0].record()
        check(self.lib.gp_geodesic_run_packed(eng.csr._h, eng.bfs._h, _ptr(edge_index), edge_index.size(1),
                                              _ptr(self._shard), hi - lo, slot, _stream()))
        if trace:
            ev[1].record()
        packed, stride = ctypes.c_void_p(), ctypes.c_int64()
        batches, wb, deep = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_void_p()
        check(self.lib.gp_msbfs_packed_info(eng.bfs._h, slot, ctypes.byref(packed), ctypes.byref(stride),
                                            ctypes.byref(batches), ctypes.byref(wb), ctypes.byref(deep)))
        # flag <- max over ranks of "my shard is deep"; stream-ordered, so it is also the barrier between
        # every rank's pack and every rank's decode
        self.flag.copy_(_wrap_device_words_i32(deep.value), non_blocking=True)
        dist.all_reduce(self.flag, op=dist.ReduceOp.MAX, group=self.group)
        if trace:
            ev[2].record()
        ptrs = (ctypes.c_void_p * self.world)()
        for r in range(self.world):
            base = packed.value - slot * self.slot_stride_words * 8 if r == self.rank else self.base[r]
            ptrs[r] = base + slot * self.slot_stride_words * 8
        check(self.lib.gp_decode_peers(ptrs, self.world, n, hi - lo, batches.value, wb.value, stride.value, _ptr(x), f,
                                       x.stride(0) if x is not None and n > 1 else f, _ptr(out),
                                       out.stride(0) if n > 1 else f + k, f, _stream()))
        if trace:
            ev[3].record()
            self.trace_events.append(ev)
        return out, self.flag

    def trace_summary(self):
        """Median device milliseconds of (csr + bfs + pack, flag all-reduce, peer decode) over the traced steps."""
        import statistics
        torch.cuda.synchronize()
        cols = [[e[i].elapsed_time(e[i + 1]) for e in self.trace_events] for i in range(3)]
        return [statistics.median(c) for c in cols] if self.trace_events else None


def _wrap_device_words_i32(ptr: int) -> torch.Tensor:
    class _Holder:
        pass

    h = _Holder()
    h.__cuda_array_interface__ = {"shape": (1,), "typestr": "<i4", "data": (ptr, False), "version": 2}
    return torch.as_tensor(h, device="cuda")
