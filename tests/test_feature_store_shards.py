"""Anchor-sharded compact feature store, host side (no GPU).

A numpy restatement of gp_fstore_merge: G shard stores of ``ceil(K/G)`` columns each, packed with the agreed P and
padded to Ws words, merge into exactly the store of one run over all K anchors (test_feature_store_format.encode).
The world_size-2 gloo test drives the product's host logic of distributed.sharded_feature_store: plane agreement
across shards of different depth, equal-shape padding of a short or empty tail shard, the gathered layout, and the
refusal of differing anchor lists.
"""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from graphpope_b200 import distributed as gpd
from test_feature_store_format import UNREACHED, _bits, encode


def merge(shards: np.ndarray, k: int) -> np.ndarray:
    """uint64 [S, N, P, Ws] shard stores (shard s = columns [s*per, min((s+1)*per, K)), per = ceil(K/S)) ->
    uint64 [N, P, ceil(K/64)]: the columns of every shard, in shard order, in the one-store layout."""
    s, n, p, _ = shards.shape
    per = -(-k // s)
    cols = [_bits(shards[g])[:, :, :min(per, k - g * per)] for g in range(s) if g * per < k]
    w = -(-k // 64)
    bits = np.zeros((n, p, 64 * w), dtype=bool)
    if cols:
        bits[:, :, :k] = np.concatenate(cols, axis=-1)
    return np.ascontiguousarray(np.packbits(bits, axis=-1, bitorder="little")).view("<u8").reshape(n, p, w)


def shard_stores(hops: np.ndarray, world: int):
    """Each shard encoded on its own (its local P), then padded to the agreed P and to Ws words, as every rank of
    sharded_feature_store does.  Returns (uint64 [G, N, P, Ws], local P of each shard)."""
    n, k = hops.shape
    raws = []
    for r in range(world):
        lo, hi = gpd.shard_bounds(k, world, r)
        raws.append(torch.from_numpy(encode(hops[:, lo:hi])) if hi > lo else None)
    local = [1 if raw is None else raw.shape[1] for raw in raws]
    p, ws = max(local), gpd.shard_words(k, world)
    blocks = [gpd.pad_shard_store(raw, n, p, ws) for raw in raws]
    return torch.stack(blocks).numpy().view(np.uint64), local


def random_hops(n, k, seed):
    """Column depth varies (max hop 1, 15 or 300 per column), so that shards need different plane counts."""
    rng = np.random.default_rng(seed)
    depth = rng.choice([1, 15, 300], size=k)
    hops = (rng.random((n, k)) * (depth + 1)).astype(np.uint16)
    hops[rng.random((n, k)) < 0.3] = UNREACHED
    return hops


@pytest.mark.parametrize("k", [1, 2, 7, 8, 63, 64, 65, 70, 256, 257, 1000])
@pytest.mark.parametrize("world", range(1, 9))
def test_merge_restatement_equals_one_store(world, k):
    hops = random_hops(37, k, seed=k * 11 + world)
    shards, local = shard_stores(hops, world)
    want = encode(hops)
    assert shards.shape == (world, 37, want.shape[1], -(-(-(-k // world)) // 64))
    assert max(local) == want.shape[1]  # the agreed P is the one-store P
    assert np.array_equal(merge(shards, k), want)


def test_shard_words_and_padding():
    assert [gpd.shard_words(k, g) for k, g in ((4096, 8), (4097, 8), (3, 8), (256, 1), (1000, 3))] == [8, 9, 1, 4, 6]
    raw = torch.arange(2 * 3 * 1, dtype=torch.int64).view(2, 3, 1)
    block = gpd.pad_shard_store(raw, 2, 5, 2)
    assert block.shape == (2, 5, 2) and torch.equal(block[:, :3, :1], raw) and not block[:, 3:].any()
    assert not block[:, :, 1:].any()
    assert gpd.pad_shard_store(raw, 2, 3, 1).data_ptr() == raw.data_ptr()  # already the block shape: no copy
    assert not gpd.pad_shard_store(None, 4, 2, 3).any()


def test_anchor_checksum():
    a = np.array([5, 9, 9, 2])
    assert gpd.anchor_checksum(a) == gpd.anchor_checksum([5, 9, 9, 2]) == gpd.anchor_checksum(torch.tensor(a))
    assert 0 <= gpd.anchor_checksum(a) < 1 << 62
    for other in ([5, 9, 2, 9], [5, 9, 9], [5, 9, 9, 2, 0], []):
        assert gpd.anchor_checksum(other) != gpd.anchor_checksum(a)


def _graph(n):
    """A directed path 0 -> 1 -> ... -> 199 (anchor 199 is 199 hops from node 0) plus a random part on 200..n-1."""
    from graphpope_b200 import synth
    path = np.stack([np.arange(199), np.arange(1, 200)])
    rnd = synth.random_digraph(n - 200, 1200, seed=3) + 200
    return np.concatenate([path, rnd], axis=1).astype(np.int64)


def _worker(rank, world, port, k, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from oracle import cbfs
        n = 500
        ei = _graph(n)
        anchors = np.random.default_rng(k).integers(200, n, k)
        anchors[-1] = 199  # the tail shard is the deep one
        gpd.check_anchors_agree(anchors)
        lo, hi = gpd.shard_bounds(k, world, rank)
        hops = cbfs.bfs_hops(cbfs.InCsr(ei, n), anchors[lo:hi]) if hi > lo else np.zeros((n, 0), np.uint16)
        raw = torch.from_numpy(encode(hops)) if hi > lo else None
        reached = hops[hops != UNREACHED]
        level = int(reached.max()) if reached.size else 0
        local_p = 1 + level.bit_length()
        p, max_level, failed = gpd.agree_store_layout(local_p, level)
        block = gpd.pad_shard_store(raw, n, p, gpd.shard_words(k, world))
        gathered = gpd.gather_planes(block)  # [G, N, P, Ws] int64
        full = cbfs.bfs_hops(cbfs.InCsr(ei, n), anchors)
        want = encode(full)
        ok = (not failed and p == want.shape[1] and max_level == int(full[full != UNREACHED].max())
              and tuple(gathered.shape) == (world, n, p, gpd.shard_words(k, world))
              and np.array_equal(merge(gathered.numpy().view(np.uint64), k), want))
        # a failure on one rank reaches every rank through the same all-reduce
        ok &= gpd.agree_store_layout(local_p, level, failed=rank == 1)[2]
        # differing anchor lists are refused on every rank
        try:
            gpd.check_anchors_agree(anchors if rank == 0 else np.append(anchors, 0))
            refused = False
        except ValueError:
            refused = True
        # the device path needs NCCL: a gloo group is refused before anything runs
        try:
            gpd.sharded_feature_store(ei, n, anchors)
            needs_nccl = False
        except RuntimeError as e:
            needs_nccl = "NCCL" in str(e)
        ret[rank] = (bool(ok), refused, needs_nccl, local_p, hi - lo)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("k", [1, 3, 130])
def test_sharded_store_host_logic_world_size_2(k):
    """K = 1: rank 1 holds no anchor; K = 3: a short tail shard; K = 130: full shards of 65 columns in 2 words."""
    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(2, port, k, ret), nprocs=2, join=True)
    ret = dict(ret)
    assert all(ret[r][:3] == (True, True, True) for r in (0, 1)), ret
    per = -(-k // 2)
    assert [ret[r][4] for r in (0, 1)] == [min(per, k), k - min(per, k)]
    if k > 1:
        assert ret[0][3] < ret[1][3], "shards of different depth: the agreement has to raise rank 0's P"
