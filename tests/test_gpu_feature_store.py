"""The compact feature store on the device (gp_fstore.cu via graphpope_b200.device.FeatureStore): the packed records
are byte-equal to the numpy encoder of tests/test_feature_store_format.py on the oracle's hops, and gathered rows are
bit-equal to the rows of the dense path (GeodesicEngine.run)."""
import numpy as np
import pytest
import torch

from conftest import micro_names
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


def _raw(store):
    return store.raw.cpu().numpy()


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


def _dense(dev, ei, n, anchors, x=None):
    eng = dev.GeodesicEngine(n, ei.shape[1], len(anchors))
    out = eng.run(torch.as_tensor(ei).cuda(), torch.as_tensor(np.asarray(anchors, dtype=np.int64)).cuda(),
                  None if x is None else x.cuda())
    torch.cuda.synchronize()
    return out


# ------------------------------------------------------------------ pack: byte-equal to the numpy encoder
def test_micro_graphs_pack_like_the_encoder(dev, golden_small):
    for name in micro_names(golden_small):
        n = int(golden_small[f"micro/{name}/n"])
        ei, anchors = golden_small[f"micro/{name}/edges"], golden_small[f"micro/{name}/anchors"]
        store = dev.FeatureStore.build(ei, n, anchors)
        assert np.array_equal(_raw(store), encode(_oracle_hops(ei, n, anchors))), name


@pytest.mark.parametrize("name,planes", [("deep_chain", 14), ("hub_star", None), ("lollipop", None)])
def test_deep_hub_lollipop_pack_like_the_encoder(dev, golden_deep_hub, name, planes):
    g = golden_deep_hub
    n, ei, anchors = int(g[f"{name}/n"]), g[f"{name}/edge_index"], g[f"{name}/anchors"]
    store = dev.FeatureStore.build(ei, n, anchors)
    want = encode(_oracle_hops(ei, n, anchors))
    assert np.array_equal(_raw(store), want)
    if planes is not None:
        assert store.num_planes == planes
    assert np.array_equal(_bits(store.to_dense().cpu().numpy()), _bits(g[f"{name}/embedding"]))


@pytest.mark.parametrize("k", [1, 2, 63, 64, 65, 256, 257, 1024])
def test_random_digraphs_pack_like_the_encoder(dev, k):
    n = 3000
    ei = synth.random_digraph(n, 9000, seed=k)
    anchors = np.random.default_rng(k).integers(0, n, k)  # duplicates allowed
    store = dev.FeatureStore.build(ei, n, anchors)
    assert np.array_equal(_raw(store), encode(_oracle_hops(ei, n, anchors)))
    assert store.nbytes == n * store.num_planes * (-(-k // 64)) * 8


# ------------------------------------------------------------------ gather: bit-equal to the dense rows
@pytest.fixture(scope="module")
def graph():
    n = 5000
    ei = synth.random_digraph(n, 30000, seed=11)
    return n, ei


@pytest.mark.parametrize("k", [256, 70])
@pytest.mark.parametrize("f", [0, 3, 500])
def test_gather_matches_dense_rows(dev, graph, k, f):
    n, ei = graph
    anchors = np.random.default_rng(k + f).integers(0, n, k)
    x = torch.as_tensor(np.random.default_rng(f).standard_normal((n, f)).astype(np.float32)) if f else None
    dense = _dense(dev, ei, n, anchors, x)
    store = dev.FeatureStore.build(ei, n, anchors, x)
    assert store.shape == (n, f + k) and store.size(1) == f + k and len(store) == n
    assert store.dtype == torch.float32 and store.device.type == "cuda"
    rng = np.random.default_rng(3)
    cases = [rng.integers(0, n, 777), np.array([], dtype=np.int64), np.array([n - 1]), np.arange(n),
             rng.integers(-n, n, 999)]  # unsorted with duplicates, B = 0, B = 1, every row, negative ids
    for ids in cases:
        got = store.gather(torch.as_tensor(ids).cuda())
        want = dense[torch.as_tensor(ids).cuda()]
        assert got.shape == want.shape and torch.equal(got.view(torch.int32), want.view(torch.int32)), ids[:5]
    store.check()
    # a view inside wider rows: aligned (fast path when K % 8 == 0) and unaligned (scalar path)
    ids = torch.as_tensor(rng.integers(0, n, 300)).cuda()
    for lead in (4, 1):
        big = torch.full((300, f + k + 9), float("nan"), device="cuda")
        view = big[:, lead:lead + f + k]
        store.gather(ids, out=view)
        assert torch.equal(view.view(torch.int32), dense[ids].view(torch.int32))
        assert bool(big[:, :lead].isnan().all()) and bool(big[:, lead + f + k:].isnan().all())


def test_indexing_shapes_follow_torch(dev, graph):
    n, ei = graph
    anchors = np.arange(0, n, 97)[:48]
    x = torch.randn(n, 5)
    store = dev.FeatureStore.build(ei, n, anchors, x)
    dense = _dense(dev, ei, n, anchors, x)
    for index in (7, -1, slice(10, 200, 3), slice(None), [4, 4, 1], np.array([[1, 2], [3, -4]]),
                  torch.tensor([9, 8]), torch.tensor([9, 8]).cuda(), torch.tensor(5).cuda(), [], np.int64(3)):
        dense_index = index.cuda() if torch.is_tensor(index) else (torch.as_tensor(index, dtype=torch.int64).cuda()
                                                                  if isinstance(index, (list, np.ndarray)) else index)
        assert torch.equal(store[index], dense[dense_index]), index
    for bad in (torch.tensor([True, False]), (1, 2), True):
        with pytest.raises(TypeError):
            store[bad]
    with pytest.raises(IndexError):
        store[torch.tensor([0.5])]


def test_flickr_shape_k256(dev):
    from oracle import cbfs
    shape = synth.FLICKR_SHAPE
    n = shape.num_nodes
    ei = synth.make_graph(shape)
    anchors = synth.stochastic_anchors(n, 256, 42)
    x = torch.as_tensor(np.random.default_rng(0).standard_normal((n, shape.num_features)).astype(np.float32))
    store = dev.FeatureStore.build(ei, n, anchors, x)
    assert store.nbytes == n * store.num_planes * 4 * 8 and store.raw.shape == (n, store.num_planes, 4)
    assert store.num_planes == 1 + store.stats["max_level"].bit_length()
    rows = np.sort(np.random.default_rng(1).choice(n, 4096, replace=False))
    got = store[torch.as_tensor(rows).cuda()].cpu().numpy()
    want = cbfs.normalise(_oracle_hops(ei, n, anchors)[rows])
    assert np.array_equal(_bits(got[:, shape.num_features:]), _bits(want))
    assert np.array_equal(got[:, : shape.num_features], x.numpy()[rows])


def test_out_of_range_ids(dev, graph):
    n, ei = graph
    anchors = np.arange(64)
    x = torch.randn(n, 4)
    store = dev.FeatureStore.build(ei, n, anchors, x)
    dense = _dense(dev, ei, n, anchors, x)
    ids = torch.tensor([3, n, 17, -n - 1, -1, 1 << 40, -n], device="cuda")
    got = store.gather(ids)
    for i, good in ((0, 3), (2, 17), (4, n - 1), (6, 0)):
        assert torch.equal(got[i], dense[good])
    for i in (1, 3, 5):
        assert not bool(got[i].any())
    with pytest.raises(IndexError):
        store.check()
    store.check()  # reported once
    before = dev.launch_count()
    for bad in (torch.tensor([0, n]), [-n - 1], n, np.array([2, n + 5])):
        with pytest.raises(IndexError):
            store[bad]
    assert dev.launch_count() == before  # a host-side index is checked before anything is launched


def test_store_outlives_its_bfs(dev, graph):
    n, ei = graph
    csr = dev.DeviceCsr(n, ei.shape[1]).build(torch.as_tensor(ei).cuda())
    bfs = dev.MsBfs(csr, 200)
    bfs.run(torch.arange(0, 200, dtype=torch.int64, device="cuda"))
    store = dev.FeatureStore(bfs)
    raw0, dense0 = store.raw.clone(), store.to_dense().clone()
    bfs.run(torch.arange(1000, 1130, dtype=torch.int64, device="cuda"))
    torch.cuda.synchronize()
    assert torch.equal(store.raw, raw0)
    bfs.close()
    csr.close()
    assert torch.equal(store.to_dense(), dense0)


# ------------------------------------------------------------------ GRAPHPOPE_OUTPUT=compact
class _Data:
    pass


def _data(n, ei, x):
    d = _Data()
    d.num_nodes, d.edge_index, d.x = n, torch.as_tensor(ei), x
    return d


@pytest.mark.parametrize("sampling", ["stochastic", "degree_centrality"])
def test_graphpope_compact_equals_default(dev, graph, monkeypatch, sampling):
    from graphpope_b200 import utils
    n, ei = graph
    x = torch.as_tensor(np.random.default_rng(2).standard_normal((n, 6)).astype(np.float32))

    def run():
        d = _data(n, ei, x)
        np.random.seed(7)
        utils.clear_cache()
        return d, utils.Graphpope(d, "toy", "geodesic", sampling, 40, None, 4)

    monkeypatch.delenv("GRAPHPOPE_OUTPUT", raising=False)
    d_host, host = run()
    monkeypatch.setenv("GRAPHPOPE_OUTPUT", "compact")
    d_c, store = run()
    assert isinstance(store, dev.FeatureStore) and tuple(store.shape) == (n, 6 + 40)
    assert np.array_equal(np.asarray(d_c.anchor_nodes), np.asarray(d_host.anchor_nodes))
    assert torch.equal(store.to_dense().cpu().view(torch.int32), host.view(torch.int32))
    assert utils.Graphpope(d_c, "toy", "geodesic", sampling, 40, None, 4) is store  # the memo
    n_id = torch.tensor([5, 0, n - 1, 17, 5], device="cuda")
    assert torch.equal(store[n_id].cpu(), host[n_id.cpu()])
    utils.clear_cache()


def test_compact_distance_vector_and_errors(dev, graph, monkeypatch, tmp_path):
    from graphpope_b200 import utils
    n, ei = graph
    monkeypatch.setenv("GRAPHPOPE_OUTPUT", "compact")
    monkeypatch.setenv("GRAPHPOPE_CACHE_DIR", str(tmp_path))
    d = _data(n, ei, torch.zeros(n, 3, dtype=torch.float64))
    d.anchor_nodes = [4, 9, 4]
    store = utils.get_geodesic_distance_vector(d, 4)
    assert tuple(store.shape) == (n, 3) and store.num_features == 0
    assert not any(tmp_path.iterdir())  # compact mode neither reads nor writes the block cache
    want = _dense(dev, ei, n, d.anchor_nodes)
    assert torch.equal(store.to_dense(), want)
    with pytest.raises(TypeError, match="GRAPHPOPE_OUTPUT=compact"):
        utils.attach_distance_embedding(d, "toy", 8, "stochastic", None, 4)


def test_node2vec_under_compact_is_the_cuda_path(dev, golden_small, tmp_path, monkeypatch):
    from graphpope_b200 import utils
    monkeypatch.setenv("GRAPHPOPE_DATA_DIR", str(tmp_path))
    table = synth.node2vec_table(400, 128, seed=int(golden_small["node2vec/table_seed"]))
    torch.save(torch.as_tensor(table), tmp_path / "toy_node2vec.pt")
    outs = {}
    for mode in ("cuda", "compact"):
        monkeypatch.setenv("GRAPHPOPE_OUTPUT", mode)
        d = _data(400, np.zeros((2, 0), dtype=np.int64), torch.as_tensor(golden_small["node2vec/x"]))
        np.random.seed(5)
        outs[mode] = utils.attach_node2vec(d, "toy", 12, "stochastic", "distance", 2)
    assert outs["compact"].is_cuda and torch.equal(outs["compact"], outs["cuda"])
