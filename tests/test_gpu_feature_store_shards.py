"""Anchor-sharded compact feature store on the device (gp_fstore_merge via FeatureStore.from_shards and
distributed.sharded_feature_store): merged records are byte-equal to the one-GPU store and to the numpy encoder of
the C oracle's hops, gathers from them are bit-equal to the dense rows, and a real NCCL job of 2 and up to 8 ranks
returns the one-GPU store on every rank."""
import datetime
import os
import socket

import numpy as np
import pytest
import torch

from conftest import DEEP_HUB_NAMES
from graphpope_b200 import distributed as gpd
from graphpope_b200 import synth
from test_feature_store_format import encode

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from graphpope_b200 import device
    return device


def _oracle_hops(ei, n, anchors):
    from oracle import cbfs
    return cbfs.bfs_hops(cbfs.InCsr(ei, n), anchors)


def virtual_ranks(dev, ei, n, anchors, world, x=None):
    """What `world` ranks of sharded_feature_store do, in one process: per rank a csr + MS-BFS over its anchor shard,
    P agreed as the max of the shards' own P, every shard packed with it and padded to Ws; then the merge."""
    a = torch.as_tensor(np.asarray(anchors, dtype=np.int64)).cuda()
    k = a.numel()
    ei_d = torch.as_tensor(ei).cuda()
    csr = dev.DeviceCsr(n, ei_d.size(1)).build(ei_d)
    runs, local = [], []
    for r in range(world):
        lo, hi = gpd.shard_bounds(k, world, r)
        if hi > lo:
            bfs = dev.MsBfs(csr, hi - lo).run(a[lo:hi])
            local.append(1 + bfs.stats()["max_level"].bit_length())
            runs.append(bfs)
        else:
            local.append(1)
            runs.append(None)
    p, ws = max(local), gpd.shard_words(k, world)
    blocks = []
    for bfs in runs:
        blocks.append(gpd.pad_shard_store(None if bfs is None else dev.FeatureStore(bfs, num_planes=p).raw, n, p, ws,
                                          device="cuda"))
        if bfs is not None:
            bfs.close()
    csr.close()
    return dev.FeatureStore.from_shards(torch.stack(blocks), k, x), local


@pytest.fixture(scope="module")
def digraph():
    n = 3000
    return n, synth.random_digraph(n, 9000, seed=17)


@pytest.mark.parametrize("k", [1, 2, 7, 8, 63, 64, 65, 70, 256, 257, 1000])
@pytest.mark.parametrize("world", range(1, 9))
def test_virtual_ranks_merge_to_the_one_gpu_store(dev, digraph, world, k):
    n, ei = digraph
    anchors = np.random.default_rng(k).integers(0, n, k)  # duplicates allowed
    one = dev.FeatureStore.build(ei, n, anchors)
    merged, _ = virtual_ranks(dev, ei, n, anchors, world)
    assert merged.raw.dtype == torch.uint64 and merged.raw.shape == one.raw.shape
    assert torch.equal(merged.raw.view(torch.int64), one.raw.view(torch.int64))
    assert np.array_equal(merged.raw.cpu().numpy(), encode(_oracle_hops(ei, n, anchors)))


@pytest.mark.parametrize("world", [2, 3])
@pytest.mark.parametrize("name", DEEP_HUB_NAMES)
def test_deep_hub_lollipop_shards(dev, golden_deep_hub, name, world):
    g = golden_deep_hub
    n, ei, anchors = int(g[f"{name}/n"]), g[f"{name}/edge_index"], g[f"{name}/anchors"]
    merged, local = virtual_ranks(dev, ei, n, anchors, world)
    want = encode(_oracle_hops(ei, n, anchors))
    assert np.array_equal(merged.raw.cpu().numpy(), want)
    assert merged.num_planes == max(local) == want.shape[1]
    if name == "deep_chain":
        assert merged.num_planes == 14
    assert np.array_equal(merged.to_dense().cpu().numpy().view(np.uint32), g[f"{name}/embedding"].view(np.uint32))


@pytest.mark.parametrize("k", [256, 70])  # the byte-lane gather kernel (K % 8 == 0) and the scalar one
@pytest.mark.parametrize("f", [0, 500])
def test_gathers_from_the_merged_store(dev, k, f):
    n = 5000
    ei = synth.random_digraph(n, 30000, seed=11)
    anchors = np.random.default_rng(k + f).integers(0, n, k)
    x = torch.as_tensor(np.random.default_rng(f).standard_normal((n, f)).astype(np.float32)) if f else None
    eng = dev.GeodesicEngine(n, ei.shape[1], k)
    dense = eng.run(torch.as_tensor(ei).cuda(), torch.as_tensor(anchors).cuda(), None if x is None else x.cuda())
    merged, _ = virtual_ranks(dev, ei, n, anchors, 3, x)
    assert merged.shape == (n, f + k)
    ids = torch.as_tensor(np.random.default_rng(3).integers(-n, n, 1999)).cuda()
    for rows in (ids, torch.arange(n, device="cuda")):
        got = merged.gather(rows)
        assert torch.equal(got.view(torch.int32), dense[rows].view(torch.int32))
    merged.check()


def test_merge_argument_errors(dev):
    from graphpope_b200 import _lib
    lib = _lib.load()
    buf = torch.zeros(4 * 10 * 2 * 2, dtype=torch.int64, device="cuda")
    out = torch.zeros(10 * 2 * 4, dtype=torch.int64, device="cuda")
    p, o, s = dev._ptr(buf), dev._ptr(out), dev._stream()
    before = dev.launch_count()
    bad = [
        (buf, 4, 64, 1, 10, 0, 200, out),   # P = 0
        (buf, 4, 64, 1, 10, 18, 200, out),  # P = 18
        (buf, 4, 65, 1, 10, 2, 200, out),   # 65 columns do not fit in one word
        (buf, 4, 64, 2, 10, 2, 257, out),   # 4 * 64 < 257 anchors
        (None, 4, 64, 1, 10, 2, 200, out),  # NULL shards while there is work
        (buf, 4, 64, 1, 10, 2, 200, None),  # NULL store while there is work
        (buf, 0, 64, 1, 10, 2, 200, out),   # no shards
    ]
    for sh, ns, per, ws, n, planes, k, st in bad:
        rc = lib.gp_fstore_merge(dev._ptr(sh), ns, per, ws, n, planes, k, dev._ptr(st), s)
        assert rc == _lib.GP_ERR_INVALID, (ns, per, ws, n, planes, k)
    assert lib.gp_fstore_merge(None, 4, 64, 1, 0, 2, 200, None, s) == _lib.GP_OK  # N = 0: nothing to do
    assert dev.launch_count() == before
    assert lib.gp_fstore_merge(p, 4, 64, 1, 10, 2, 200, o, s) == _lib.GP_OK
    torch.cuda.synchronize()
    assert dev.launch_count() == before + 1


# ------------------------------------------------------------------ real ranks: one process per GPU, NCCL
def _rank_worker(rank, world, port, ret):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), GRAPHPOPE_OUTPUT="compact",
                      GRAPHPOPE_SHARED="1", GRAPHPOPE_QUIET="1")
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, timeout=datetime.timedelta(minutes=5),
                            device_id=torch.device("cuda", rank))
    try:
        from graphpope_b200 import device as dev
        from graphpope_b200 import utils

        n = 4000
        ei = synth.random_digraph(n, 16000, seed=23)
        x = torch.as_tensor(np.random.default_rng(1).standard_normal((n, 12)).astype(np.float32))
        good = []
        for k, method in ((100, "stochastic"), (3, "degree_centrality")):

            class D:
                pass

            d = D()
            d.num_nodes, d.edge_index, d.x = n, torch.as_tensor(ei), x
            np.random.seed(7)
            utils.clear_cache()
            store = utils.Graphpope(d, "toy", "geodesic", method, k, None, 4)
            one = dev.FeatureStore.build(ei, n, d.anchor_nodes, x)
            good.append(isinstance(store, dev.FeatureStore) and tuple(store.shape) == (n, 12 + k)
                        and torch.equal(store.raw.view(torch.int64), one.raw.view(torch.int64))
                        and torch.equal(store.to_dense(), one.to_dense())
                        and store.stats["max_level"] == one.stats["max_level"])
        ret[rank] = good
        dist.barrier()
    finally:
        dist.destroy_process_group()


def _world_sizes():
    count = torch.cuda.device_count() if torch.cuda.is_available() else 0
    return [2] + ([min(count, 8)] if count > 2 else [])


@pytest.mark.parametrize("world", _world_sizes())
def test_real_ranks_build_the_one_gpu_store(world):
    if torch.cuda.device_count() < world:
        pytest.skip(f"needs {world} GPUs, {torch.cuda.device_count()} visible")
    import torch.multiprocessing as mp

    s = socket.socket(); s.bind(("127.0.0.1", 0)); port = s.getsockname()[1]; s.close()
    ret = mp.Manager().dict()
    mp.spawn(_rank_worker, args=(world, port, ret), nprocs=world, join=True)
    assert dict(ret) == {r: [True, True] for r in range(world)}
