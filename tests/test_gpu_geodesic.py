"""Parity of the CUDA geodesic path against the CPU oracle and the frozen reference outputs.

Everything here calls through the C ABI (graphpope_b200.device / graphpope_b200.utils ->
libgraphpope_b200.so).  Bar: bit-exact uint16 hops and bit-exact float32 features.
"""
import hashlib

import numpy as np
import pytest
import torch

from conftest import micro_names
from graphpope_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from graphpope_b200 import device
    return device


def _oracle_hops(ei, n, anchors, symmetrize=False):
    from oracle import cbfs
    return cbfs.bfs_hops(cbfs.InCsr(ei, n, symmetrize), anchors)


def _gpu_hops_and_features(dev, ei, n, anchors, x=None, symmetrize=False):
    eng = dev.GeodesicEngine(n, ei.shape[1], len(anchors), symmetrize)
    ei_d = torch.as_tensor(ei, dtype=torch.int64).cuda()
    a_d = torch.as_tensor(np.asarray(anchors, dtype=np.int64)).cuda()
    x_d = None if x is None else torch.as_tensor(x).cuda()
    feats = eng.run(ei_d, a_d, x_d)
    hops = eng.bfs.hops_u16()
    stats = eng.bfs.stats()
    torch.cuda.synchronize()
    return hops.cpu().numpy(), feats.cpu().numpy(), stats


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint32)


# ------------------------------------------------------------------ CSR builder
@pytest.mark.parametrize("n,e,seed", [(1, 3, 0), (7, 0, 1), (50, 400, 2), (3000, 20000, 3), (70000, 300000, 4)])
@pytest.mark.parametrize("symmetrize", [False, True])
def test_csr_matches_oracle(dev, n, e, seed, symmetrize):
    from oracle import geodesic as g
    ei = synth.random_digraph(n, e, seed=seed)
    csr = dev.DeviceCsr(n, ei.shape[1], symmetrize).build(torch.as_tensor(ei).cuda())
    info = csr.info()
    for which, fn in (("out", g.out_csr), ("in", g.in_csr)):
        rp_want, col_want = fn(ei, n, symmetrize)
        rp, col = csr.export(which)
        assert np.array_equal(rp.cpu().numpy(), rp_want), which
        assert np.array_equal(col.cpu().numpy(), col_want), which
    s, d = g.dedup_edges(ei, n, symmetrize)
    assert info["num_edges"] == s.size
    assert info["num_input_edges"] == ei.shape[1]
    assert info["max_out_degree"] == (np.bincount(s, minlength=n).max() if s.size else 0)
    sym = set(zip(s.tolist(), d.tolist())) == set(zip(d.tolist(), s.tolist()))
    assert bool(info["is_symmetric"]) == sym


@pytest.mark.parametrize("n", [20000, 1_000_000])
def test_csr_row_sort_paths(dev, n):
    """Rows of every length class with repeated edges: the warp register sort (<= 32 / 64 / 128 edges),
    the CTA bitmap sort (graphs whose node bitmap fits in shared memory), the shared-memory sorting
    network and the in-place one (rows above 8192 edges when the bitmap does not fit)."""
    from oracle import geodesic as g
    rng = np.random.default_rng(n)
    lens = [0, 1, 2, 31, 32, 33, 40, 63, 64, 65, 100, 127, 128, 129, 200, 511, 1000, 4097, 8192, 8193, 9000]
    src, dst = [], []
    for r, ln in enumerate(lens):
        row = r * 7 + 3
        cols = rng.choice(n, size=ln, replace=False) if ln else np.zeros(0, dtype=np.int64)
        rep = rng.integers(1, 4, size=ln)  # every edge 1..3 times
        cols = np.repeat(cols, rep)
        src.append(np.full(cols.size, row, dtype=np.int64))
        dst.append(cols.astype(np.int64))
    # background edges, some of them into the heavy rows
    bg = synth.random_digraph(n, 5000, seed=n + 1)
    src.append(bg[0]); dst.append(bg[1])
    ei = np.stack([np.concatenate(src), np.concatenate(dst)])
    ei = np.ascontiguousarray(ei[:, rng.permutation(ei.shape[1])])
    csr = dev.DeviceCsr(n, ei.shape[1]).build(torch.as_tensor(ei).cuda())
    for which, fn in (("out", g.out_csr), ("in", g.in_csr)):
        rp_want, col_want = fn(ei, n, False)
        rp, col = csr.export(which)
        assert np.array_equal(rp.cpu().numpy(), rp_want), which
        assert np.array_equal(col.cpu().numpy(), col_want), which
    info = csr.info()
    s_, d_ = g.dedup_edges(ei, n, False)
    assert info["num_edges"] == s_.size
    assert info["max_out_degree"] == np.bincount(s_, minlength=n).max()
    # and the traversal over that CSR (hub chunks, every slot class) stays bit-exact; at n = 1_000_000 the per-hop
    # bitmaps (125 KB) do not fit in shared memory next to the work cache, so this runs the global-memory map variant
    anchors = rng.integers(0, n, 64)
    hops, _, _ = _gpu_hops_and_features(dev, ei, n, anchors)
    assert np.array_equal(hops, _oracle_hops(ei, n, anchors))


def test_csr_rejects_out_of_range_index(dev):
    ei = torch.tensor([[0, 1, 9], [1, 2, 0]], dtype=torch.int64).cuda()
    csr = dev.DeviceCsr(5, 3).build(ei)
    with pytest.raises(IndexError):
        csr.info()
    ei = torch.tensor([[0, -1], [1, 2]], dtype=torch.int64).cuda()
    with pytest.raises(IndexError):
        dev.DeviceCsr(5, 2).build(ei).info()


# ------------------------------------------------------------------ golden fixtures (reference outputs)
def test_micro_graphs_match_reference(dev, golden_small):
    for name in micro_names(golden_small):
        n = int(golden_small[f"micro/{name}/n"])
        ei = golden_small[f"micro/{name}/edges"]
        anchors = golden_small[f"micro/{name}/anchors"]
        want = golden_small[f"micro/{name}/rows_f64"].astype(np.float32)
        hops, feats, _ = _gpu_hops_and_features(dev, ei, n, anchors)
        assert np.array_equal(_bits(feats), _bits(want)), name
        assert np.array_equal(hops, _oracle_hops(ei, n, anchors)), name


@pytest.mark.parametrize("name", ["deep_chain", "hub_star"])
def test_deep_and_hub_graphs_match_reference(dev, golden_deep_hub, name):
    """Deep bit planes (4999 hops) and hub chunks / CTA row sort (5000- and 300-edge rows) against what the
    unmodified reference returned for these graphs (reference_deep_hub.npz), bit for bit.  (The third graph of the
    fixture, both at once with two lane words, is in tests/test_gpu_shims.py.)"""
    g = golden_deep_hub
    n, ei, anchors = int(g[f"{name}/n"]), g[f"{name}/edge_index"], g[f"{name}/anchors"]
    hops, feats, _ = _gpu_hops_and_features(dev, ei, n, anchors)
    assert np.array_equal(_bits(feats), _bits(g[f"{name}/embedding"]))
    assert np.array_equal(hops, _oracle_hops(ei, n, anchors))


def test_toy_pipeline_matches_reference(dev, golden_small):
    n = int(golden_small["toy/n"])
    ei, x = golden_small["toy/edge_index"], golden_small["toy/x"]
    anchors = golden_small["toy/anchors"]
    want = golden_small["toy/features"]
    _, feats, _ = _gpu_hops_and_features(dev, ei, n, anchors, x)  # F=5, K=8: unaligned scalar epilogue
    assert feats.shape == want.shape
    assert np.array_equal(_bits(feats), _bits(want))
    # duplicate anchor 102 -> identical columns
    assert np.array_equal(feats[:, 5 + 0], feats[:, 5 + 6])


def test_toysym_matches_reference(dev, golden_small):
    ei, anchors = golden_small["toysym/edge_index"], golden_small["toysym/anchors"]
    want = golden_small["toysym/embedding"]
    for sym in (False, True):
        _, feats, _ = _gpu_hops_and_features(dev, ei, 300, anchors, symmetrize=sym)
        assert np.array_equal(_bits(feats), _bits(want))


def test_pubmed_shape_matches_reference_verbatim(dev, golden_pubmed):
    """BASELINE.json configs[0]: the reference's own run (num_workers=6) frozen as a hash."""
    shape = synth.PUBMED_SHAPE
    ei = synth.make_graph(shape)
    anchors = synth.stochastic_anchors(shape.num_nodes, 256, 42)
    assert np.array_equal(anchors, golden_pubmed["anchors"])
    hops, feats, stats = _gpu_hops_and_features(dev, ei, shape.num_nodes, anchors)
    rows = golden_pubmed["sample_rows"]
    assert np.array_equal(_bits(feats[rows]), _bits(golden_pubmed["sample"]))
    assert hashlib.sha256(np.ascontiguousarray(feats).tobytes()).digest() == golden_pubmed["sha256"].tobytes()
    assert np.array_equal(hops, _oracle_hops(ei, shape.num_nodes, anchors))
    assert stats["max_level"] == int(hops[hops != 0xFFFF].max())


# ------------------------------------------------------------------ oracle parity, many shapes
@pytest.mark.parametrize("k", [1, 2, 63, 64, 65, 128, 129, 256, 257, 700])
def test_anchor_counts_and_lane_padding(dev, k):
    n = 2500
    ei = synth.random_digraph(n, 9000, seed=k)
    anchors = np.random.default_rng(k).integers(0, n, k)
    hops, feats, stats = _gpu_hops_and_features(dev, ei, n, anchors)
    want = _oracle_hops(ei, n, anchors)
    assert hops.shape == (n, k) and np.array_equal(hops, want)
    from oracle import cbfs
    assert np.array_equal(_bits(feats), _bits(cbfs.normalise(want)))
    assert stats["num_anchors"] == k


@pytest.mark.parametrize("seed", range(4))
def test_random_asymmetric_multigraphs(dev, seed):
    rng = np.random.default_rng(100 + seed)
    n = int(rng.integers(2, 4000))
    ei = synth.random_digraph(n, int(rng.integers(0, 6 * n)), seed=seed)
    anchors = rng.integers(0, n, int(rng.integers(1, 300)))
    hops, _, _ = _gpu_hops_and_features(dev, ei, n, anchors)
    assert np.array_equal(hops, _oracle_hops(ei, n, anchors))


def test_hub_rows_take_the_cta_and_warp_paths(dev):
    # star with 5000 leaves + a 300-leaf hub + chain: exercises large / medium / small row classes
    n = 6000
    e = [(0, i) for i in range(1, 5001)] + [(i, 0) for i in range(1, 5001)]
    e += [(5001, i) for i in range(5002, 5302)] + [(i, 5001) for i in range(5002, 5302)]
    e += [(i, i + 1) for i in range(5302, 5999)] + [(5001, 0), (5500, 5001)]
    ei = np.asarray(e, dtype=np.int64).T
    anchors = np.array([0, 17, 5001, 5999, 5302, 5100, 17], dtype=np.int64)
    hops, _, stats = _gpu_hops_and_features(dev, ei, n, anchors)
    assert np.array_equal(hops, _oracle_hops(ei, n, anchors))


def test_deep_path_uses_many_distance_planes(dev):
    n = 5000
    ei = np.stack([np.arange(n - 1), np.arange(1, n)]).astype(np.int64)
    anchors = np.array([n - 1, 0, 2500], dtype=np.int64)
    hops, feats, stats = _gpu_hops_and_features(dev, ei, n, anchors)
    want = _oracle_hops(ei, n, anchors)
    assert np.array_equal(hops, want)
    assert stats["max_level"] == n - 1
    from oracle import cbfs
    assert np.array_equal(_bits(feats), _bits(cbfs.normalise(want)))


def test_handle_reuse_after_a_deeper_run(dev):
    """A run of depth ~100 on a handle that earlier saw depth 699: the high deep-hop bit planes of the
    first run must not leak into the second (they are cleared at hop 15 of every deep run)."""
    n = 700
    a = np.arange(n - 1)
    path = np.stack([np.concatenate([a, a + 1]), np.concatenate([a + 1, a])]).astype(np.int64)
    r = np.arange(200)
    ring = np.stack([np.concatenate([r, (r + 1) % 200]), np.concatenate([(r + 1) % 200, r])]).astype(np.int64)
    eng = dev.GeodesicEngine(n, path.shape[1], 64)
    anchors = np.array([0, 5, 699, 100], dtype=np.int64)
    a_d = torch.as_tensor(anchors).cuda()
    for ei in (path, ring, path, ring):
        eng.csr.build(torch.as_tensor(ei).cuda())
        eng.bfs.run(a_d)
        got = eng.bfs.hops_u16().cpu().numpy()
        assert np.array_equal(got, _oracle_hops(ei, n, anchors))
        feats = eng.bfs.features().cpu().numpy()
        want = np.where(got == 0xFFFF, np.float32(0), np.float32(1) / (got.astype(np.float32) + np.float32(1)))
        assert np.array_equal(_bits(feats), _bits(want.astype(np.float32)))


def test_uint16_overflow_is_reported(dev):
    n = 65600
    ei = np.stack([np.arange(n - 1), np.arange(1, n)]).astype(np.int64)
    eng = dev.GeodesicEngine(n, ei.shape[1], 1)
    eng.csr.build(torch.as_tensor(ei).cuda())
    eng.bfs.run(torch.tensor([n - 1], dtype=torch.int64).cuda())
    with pytest.raises(OverflowError):
        eng.bfs.stats()
    # 65534 hops is the largest representable distance
    eng.bfs.run(torch.tensor([65534], dtype=torch.int64).cuda())
    assert eng.bfs.stats()["max_level"] == 65534
    hops = eng.bfs.hops_u16().cpu().numpy()
    assert hops[0, 0] == 65534 and hops[65535, 0] == 0xFFFF


def test_bad_anchor_is_reported(dev):
    ei = synth.random_digraph(100, 300, seed=1)
    eng = dev.GeodesicEngine(100, ei.shape[1], 4)
    eng.csr.build(torch.as_tensor(ei).cuda())
    eng.bfs.run(torch.tensor([1, 100, 3], dtype=torch.int64).cuda())
    with pytest.raises(IndexError):
        eng.bfs.stats()


def test_empty_inputs(dev):
    ei = np.zeros((2, 0), dtype=np.int64)
    hops, feats, _ = _gpu_hops_and_features(dev, ei, 4, np.array([1, 1]))
    assert feats.tolist() == [[0, 0], [1, 1], [0, 0], [0, 0]]
    out, hops, _ = dev.geodesic_embed_host(ei, 3, [], None)
    assert tuple(out.shape) == (3, 0)
    x = np.arange(6, dtype=np.float32).reshape(3, 2)
    out, _, _ = dev.geodesic_embed_host(ei, 3, [], x)
    assert np.array_equal(out.numpy(), x)
    out, _, _ = dev.geodesic_embed_host(ei, 0, [], None)
    assert tuple(out.shape) == (0, 0)


def test_device_run_with_empty_output(dev):
    """GeodesicEngine.run with no anchors: an [N, 0] result has no storage (a NULL d_out), which gp_geodesic_run
    accepts because it has nothing to write; the run still counts for stats().  With x it writes x alone."""
    n = 50
    ei_d = torch.as_tensor(synth.random_digraph(n, 200, seed=4)).cuda()
    none = torch.empty(0, dtype=torch.int64, device="cuda")
    eng = dev.GeodesicEngine(n, ei_d.size(1), 8)
    for _ in range(3):  # eager, then the calls that would capture / replay a graph
        out = eng.run(ei_d, none)
        torch.cuda.synchronize()
        assert tuple(out.shape) == (n, 0)
        assert eng.bfs.stats()["num_anchors"] == 0
    x = torch.randn(n, 3, device="cuda")
    assert torch.equal(eng.run(ei_d, none, x), x)
    a_d = torch.as_tensor([1, 7], device="cuda")
    assert tuple(eng.run(ei_d, a_d).shape) == (n, 2)  # the handle still runs anchors afterwards


# ------------------------------------------------------------------ full-size properties (Flickr shape)
@pytest.fixture(scope="module")
def flickr():
    shape = synth.FLICKR_SHAPE
    ei = synth.make_graph(shape)
    anchors = synth.stochastic_anchors(shape.num_nodes, 256, 42)
    return shape, ei, anchors


def test_flickr_shape_k256_bit_exact(dev, flickr):
    """BASELINE.json configs[1] (the headline workload) against the C oracle."""
    shape, ei, anchors = flickr
    x = np.random.default_rng(0).standard_normal((shape.num_nodes, shape.num_features)).astype(np.float32)
    hops, feats, stats = _gpu_hops_and_features(dev, ei, shape.num_nodes, anchors, x)
    want = _oracle_hops(ei, shape.num_nodes, anchors)
    assert np.array_equal(hops, want)
    from oracle import cbfs
    assert np.array_equal(_bits(feats[:, shape.num_features:]), _bits(cbfs.normalise(want)))
    assert np.array_equal(feats[:, : shape.num_features], x)
    assert stats["lane_words"] == 4


def test_flickr_shape_properties(dev, flickr):
    shape, ei, anchors = flickr
    n = shape.num_nodes
    hops, feats, _ = _gpu_hops_and_features(dev, ei, n, anchors)
    hops2, feats2, _ = _gpu_hops_and_features(dev, ei, n, anchors)
    assert np.array_equal(hops, hops2) and np.array_equal(_bits(feats), _bits(feats2))  # deterministic
    cols = np.arange(anchors.size)
    assert np.all(hops[anchors, cols] == 0) and np.all(feats[anchors, cols] == 1.0)
    # symmetric graph: hops(a_i -> a_j) == hops(a_j -> a_i)
    sub = hops[anchors][:, :]
    assert np.array_equal(sub, sub.T)
    # triangle inequality through anchor 0 on reachable triples (sampled rows)
    r = np.arange(0, n, 37)
    d0 = hops[r, 0].astype(np.int64)
    a0 = hops[anchors[0]].astype(np.int64)  # hops(anchor0 -> anchor_j)
    ok = (hops[r] != 0xFFFF) & (d0[:, None] != 0xFFFF) & (a0[None, :] != 0xFFFF)
    assert np.all((hops[r].astype(np.int64) <= d0[:, None] + a0[None, :]) | ~ok)
    # permuting the anchors permutes the columns
    perm = np.random.default_rng(1).permutation(anchors.size)
    hops_p, _, _ = _gpu_hops_and_features(dev, ei, n, anchors[perm])
    assert np.array_equal(hops_p, hops[:, perm])


def test_normalize_into_matches_convention(dev):
    d = np.array([[0, 1, 2, 0xFFFF], [65534, 7, 0xFFFF, 3]], dtype=np.uint16)
    out = torch.full((2, 6), -1.0, device="cuda")
    dev.normalize_into(torch.as_tensor(d.view(np.int16)).cuda().view(torch.uint16), out, col_offset=2)
    from oracle import cbfs
    got = out.cpu().numpy()
    assert np.array_equal(_bits(got[:, 2:]), _bits(cbfs.normalise(d)))
    assert np.all(got[:, :2] == -1.0)


def test_device_resident_output_equals_host_output(dev, monkeypatch):
    """GRAPHPOPE_OUTPUT=cuda (SURVEY §8f rank 3): same bits, but the [N, F+K] matrix stays in HBM so the
    trainer's x[n_id] gathers (main.py:120,177) run on the device."""
    from graphpope_b200 import utils
    n, f, k = 3000, 12, 40
    ei = synth.random_digraph(n, 20000, seed=5)
    x = torch.as_tensor(np.random.default_rng(1).standard_normal((n, f)).astype(np.float32))

    class D:
        pass

    def run():
        d = D()
        d.num_nodes, d.edge_index, d.x = n, torch.as_tensor(ei), x
        np.random.seed(7)
        return utils.attach_distance_embedding(d, "toy", k, "stochastic", None, 4)

    monkeypatch.delenv("GRAPHPOPE_OUTPUT", raising=False)
    host = run()
    monkeypatch.setenv("GRAPHPOPE_OUTPUT", "cuda")
    devout = run()
    assert not host.is_cuda and devout.is_cuda
    assert torch.equal(devout.cpu(), host)
    n_id = torch.tensor([5, 0, 2999, 17], device="cuda")
    assert torch.equal(devout[n_id].cpu(), host[n_id.cpu()])


@pytest.mark.parametrize("n,f,pad", [(1, 1, 0), (37, 5, 3), (1000, 500, 256), (513, 129, 2)])
def test_concat_x_matches_torch_slicing(dev, n, f, pad):
    """gp_concat_x: the x half of concat_into_features (utils.py:133-134) as one strided device-to-device copy."""
    from ctypes import c_void_p

    from graphpope_b200 import _lib
    lib = _lib.load()
    x = torch.randn(n, f, device="cuda")
    out = torch.full((n, f + pad), float("nan"), device="cuda")
    _lib.check(lib.gp_concat_x(c_void_p(x.data_ptr()), n, f, f, c_void_p(out.data_ptr()), f + pad,
                               c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert torch.equal(out[:, :f], x)
    assert bool(torch.isnan(out[:, f:]).all())
    assert lib.gp_concat_x(None, n, f, f, c_void_p(out.data_ptr()), f + pad, None) == _lib.GP_ERR_INVALID
    assert lib.gp_concat_x(c_void_p(x.data_ptr()), n, f, f - 1, c_void_p(out.data_ptr()), f + pad, None) == \
        _lib.GP_ERR_INVALID


@pytest.mark.parametrize("n,f,ldx,pad", [(1, 4, 4, 4), (4097, 4, 4, 8), (89250, 500, 500, 256), (3001, 500, 512, 256),
                                         (700, 4096, 4096, 64), (300, 4100, 4100, 4), (77, 1028, 1032, 12)])
def test_bulk_copy_engine_x_copy(dev, n, f, ldx, pad):
    """gp_concat_x on 16-byte aligned rows = the TMA bulk-copy pipeline (gp_xcopy.cu): one row per 16 KB stage up to
    1024 rows per stage, contiguous and pitched x, a ragged last block; rows over 16 KB take the strided copy."""
    from ctypes import c_void_p

    from graphpope_b200 import _lib
    lib = _lib.load()
    xb = torch.randn(n, ldx, device="cuda")
    x = xb[:, :f]
    out = torch.full((n, f + pad), float("nan"), device="cuda")
    for _ in range(2):  # twice: the second call reuses the kernel's cached launch attributes
        _lib.check(lib.gp_concat_x(c_void_p(x.data_ptr()), n, f, ldx, c_void_p(out.data_ptr()), f + pad,
                                   c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    assert torch.equal(out[:, :f], x)
    assert bool(torch.isnan(out[:, f:]).all())


def test_wide_feature_rows_take_the_chunked_x_copy(dev):
    """F > 512 floats: the epilogue's x-row copy runs more than one batch of loads per lane; odd F: scalar tail."""
    from oracle import cbfs, geodesic
    n, k = 300, 16
    ei = synth.random_digraph(n, 900, seed=3)
    anchors = np.random.default_rng(1).integers(0, n, k)
    for f in (517, 1030, 2052):
        x = np.random.default_rng(f).standard_normal((n, f)).astype(np.float32)
        _, feats, _ = _gpu_hops_and_features(dev, ei, n, anchors, x)
        want = geodesic.concat_features(x, cbfs.geodesic_features(ei, n, anchors))
        assert np.array_equal(feats.view(np.uint32), want.view(np.uint32)), f


@pytest.mark.parametrize("world,k,f,n,ldx", [
    pytest.param(2, 64, 20, 3000, 20, id="2-64-20"),
    pytest.param(4, 512, 500, 3000, 500, id="4-512-500"),
    pytest.param(3, 48, 8, 3000, 8, id="3-48-8"),
    pytest.param(8, 128, 4, 3000, 4, id="8-128-4"),
    (2, 512, 20, 3000, 20),     # 256 lanes per rank: 4 words per batch, the benchmark's shard
    (4, 1024, 4, 3000, 4),
    (3, 984, 8, 3000, 8),       # 328 lanes: 2 batches, the last one ragged
    (2, 1040, 12, 3000, 12),    # 520 lanes: 3 batches
    (2, 1040, 12, 3001, 12),    # and N not a multiple of the row block
    (2, 64, 20, 3001, 20),      # 8-byte rows, odd N: the last block's segment is rounded up to 16 bytes
    (4, 128, 20, 3000, 21),     # x a column slice with a pitch that is not a multiple of 4: scalar x copy
])
def test_push_exchange_virtual_ranks_on_one_gpu(dev, monkeypatch, world, k, f, n, ldx):
    """gp_exchange.cu with `world` virtual ranks in ONE process on one GPU (plain device pointers instead of IPC
    mappings): every rank runs its anchor shard, then the fused pack / push / decode kernels run side by side on
    their own streams (partial grids so all of them are resident) and every rank's [N, F + K] matrix must equal the
    single-GPU result bit for bit.  Two steps: both slot parities and the epoch protocol."""
    from ctypes import c_void_p

    from graphpope_b200 import _lib, distributed as gpd
    lib = _lib.load()
    ei = synth.chung_lu_symmetric(n, 18000, 2.2, seed=5)
    ei = np.concatenate([ei, synth.random_digraph(n, 700, seed=6)], axis=1)
    per = k // world
    ei_d = torch.as_tensor(ei).cuda()
    x = torch.randn(n, ldx, device="cuda")[:, :f]
    engines = [dev.GeodesicEngine(n, ei.shape[1], per) for _ in range(world)]
    xch = [gpd.PushExchange(engines[r], world=world, rank=r, grid_blocks=24) for r in range(world)]
    for r in range(world):
        for q in range(world):
            if q != r:
                xch[r].set_peer(q, xch[q].local_ptr())
    streams = [torch.cuda.Stream() for _ in range(world)]
    for step in range(2):
        anchors = np.random.default_rng(step).integers(0, n, k)
        a_d = torch.as_tensor(anchors).cuda()
        want = dev.GeodesicEngine(n, ei.shape[1], k).run(ei_d, a_d, x).clone()
        outs = [torch.full((n, f + k), float("nan"), device="cuda") for _ in range(world)]
        for r in range(world):
            engines[r].csr.build(ei_d)
            engines[r].bfs.run(a_d[r * per:(r + 1) * per].contiguous())
        torch.cuda.synchronize()
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                _lib.check(lib.gp_exchange_run(xch[r]._h, c_void_p(x.data_ptr()), f, ldx, c_void_p(outs[r].data_ptr()),
                                               f + k, f, c_void_p(streams[r].cuda_stream)))
        torch.cuda.synchronize()
        for r in range(world):
            assert xch[r].item() == 0
            assert torch.equal(outs[r], want), (step, r)
    for e in xch:
        e.close()


def test_pageable_output_ring_equals_pinned_output(dev):
    """gp_geodesic_embed_host with a PAGEABLE output goes through two pinned 8 MB ring slots (three chunks here);
    the result must equal the strided-DMA path taken for a pinned output, x columns included."""
    n, k, f = 70000, 64, 12
    ei = synth.chung_lu_symmetric(n, 400000, 2.1, seed=11)
    anchors = np.random.default_rng(3).integers(0, n, k)
    x = torch.randn(n, f)
    pinned = torch.empty(n, f + k).pin_memory()
    dev.geodesic_embed_host(torch.as_tensor(ei), n, anchors, x, out=pinned)
    pageable = torch.full((n, f + k), float("nan"))
    dev.geodesic_embed_host(torch.as_tensor(ei), n, anchors, x, out=pageable)
    assert torch.equal(pageable, pinned) and torch.equal(pageable[:, :f], x)


def test_two_host_threads_with_their_own_contexts(dev):
    """gp_ctx_t: two host threads, each with its own context (handles, stream, staging), run the one-call host entry
    at the same time on different graphs; both results equal the oracle.  No state is shared between contexts."""
    import threading
    from oracle import cbfs, geodesic
    jobs = []
    for seed, n, k in ((1, 5000, 40), (2, 9000, 96)):
        ei = np.concatenate([synth.chung_lu_symmetric(n, 6 * n, 2.2, seed=seed), synth.random_digraph(n, n // 4, seed=seed + 7)], axis=1)
        anchors = np.random.default_rng(seed).integers(0, n, k)
        x = np.random.default_rng(seed + 1).standard_normal((n, 9)).astype(np.float32)
        jobs.append((ei, n, anchors, x, geodesic.concat_features(x, cbfs.geodesic_features(ei, n, anchors))))
    results, errors = [None, None], []

    def work(i):
        try:
            ctx = dev.HostContext()
            ei, n, anchors, x, _ = jobs[i]
            for _ in range(5):
                results[i] = dev.geodesic_embed_host(torch.as_tensor(ei), n, anchors, torch.as_tensor(x), ctx=ctx)[0]
            ctx.close()
        except Exception as e:  # noqa: BLE001
            errors.append(e)

    threads = [threading.Thread(target=work, args=(i,)) for i in range(2)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    assert not errors, errors
    for i in range(2):
        assert np.array_equal(results[i].numpy().view(np.uint32), jobs[i][4].view(np.uint32)), i


def test_two_hundred_runs_are_identical(dev, flickr):
    """Stress for the hand-rolled grid barrier and the hub-row hand-off: 200 back-to-back runs on the Flickr-shaped
    graph (graph-replayed pipeline, then eager MS-BFS launches) must give the same hop matrix every time."""
    shape, ei, anchors = flickr
    n = shape.num_nodes
    eng = dev.GeodesicEngine(n, ei.shape[1], 256)
    ei_d, a_d = torch.as_tensor(ei).cuda(), torch.as_tensor(anchors).cuda()
    out = torch.empty(n, 256, device="cuda")
    eng.run(ei_d, a_d, None, out)
    first = eng.bfs.hops_u16().view(torch.int16).clone()
    first_out = out.clone()
    for i in range(100):
        eng.run(ei_d, a_d, None, out)
        assert torch.equal(out, first_out), i
    for i in range(100):
        eng.bfs.run(a_d)
        assert torch.equal(eng.bfs.hops_u16().view(torch.int16), first), i
    assert eng.bfs.stats()["max_level"] >= 5


@pytest.mark.parametrize("symmetrize", [False, True])
@pytest.mark.parametrize("k", [1, 64, 100, 256])
def test_hop1_pull_matches_oracle(dev, k, symmetrize):
    """Hop 1 of the fused pipeline pulls like every other hop, on an asymmetric multigraph with self loops and repeated
    edges, duplicate anchors and anchors adjacent to anchors; with and without GP_CSR_SYMMETRIZE.  Bit-equal to the
    oracle on the eager, captured and replayed runs; the stats report no push level.  gp_msbfs_set_push keeps its ABI
    version 1 symbol: 0 is accepted, 1 is GP_ERR_UNSUPPORTED."""
    from graphpope_b200 import _lib
    n = 5000
    ei = np.concatenate([synth.chung_lu_symmetric(n, 30000, 2.2, seed=13), synth.random_digraph(n, 4000, seed=14)], axis=1)
    rng = np.random.default_rng(k)
    anchors = rng.integers(0, n, k)
    if k > 2:
        anchors[1] = anchors[0]              # duplicate anchor
        anchors[2] = ei[1, ei[0] == anchors[0]][0] if (ei[0] == anchors[0]).any() else anchors[2]  # neighbour of an anchor
    want = _oracle_hops(ei, n, anchors, symmetrize)
    ei_d, a_d = torch.as_tensor(ei).cuda(), torch.as_tensor(anchors).cuda()
    eng = dev.GeodesicEngine(n, ei.shape[1], k, symmetrize)
    lib = _lib.load()
    assert lib.gp_msbfs_set_push(eng.bfs._h, 1) == _lib.GP_ERR_UNSUPPORTED
    assert b"always pulls" in lib.gp_last_error()
    assert lib.gp_msbfs_set_push(eng.bfs._h, 0) == _lib.GP_OK
    for run in ("eager", "captured", "replayed"):
        eng.run(ei_d, a_d)
        hops = eng.bfs.hops_u16().cpu().numpy()
        st = eng.bfs.stats()
        assert np.array_equal(hops, want), run
        assert st["push_levels"] == 0 and st["pull_levels"] + st["push_levels"] == st["levels_run"], run


@pytest.mark.parametrize("k", [50, 3, 64])
def test_exchange_entry_pads_a_ragged_anchor_count(dev, k):
    """PushExchange.run (gp_geodesic_run_exchange) with an anchor count that is not a multiple of 8: the shard is
    padded with repeats of the last anchor, computed into a scratch matrix and the real columns copied out.  One rank
    here (the padding logic is per rank); three calls = eager, captured, replayed."""
    from graphpope_b200 import distributed as gpd
    from oracle import cbfs, geodesic
    n, f = 4000, 12
    ei = np.concatenate([synth.chung_lu_symmetric(n, 24000, 2.2, seed=3), synth.random_digraph(n, 900, seed=4)], axis=1)
    anchors = np.random.default_rng(k).integers(0, n, k)
    x = np.random.default_rng(1).standard_normal((n, f)).astype(np.float32)
    want = geodesic.concat_features(x, cbfs.geodesic_features(ei, n, anchors))
    eng = dev.GeodesicEngine(n, ei.shape[1], -(-k // 8) * 8)
    xch = gpd.PushExchange(eng, world=1, rank=0)
    ei_d, a_d, x_d = torch.as_tensor(ei).cuda(), torch.as_tensor(anchors).cuda(), torch.as_tensor(x).cuda()
    for _ in range(3):
        out, flag = xch.run(ei_d, a_d, x_d)
        assert flag.item() == 0
        assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32))
    xch.close()
