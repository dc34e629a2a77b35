"""The multi-rank assembly paths of the anchor-sharded embedding, with G virtual ranks in one process on one GPU:

- the all-gather decode (distributed.sharded_geodesic_features -> gp_decode_gathered), driven through the real
  wrapper with its two collectives replaced by a thread barrier, and gp_decode_gathered called directly;
- the deep flag of the push exchange (gp_exchange.cu), which must describe the step that raised it and no later one;
- the node-shared host matrix (distributed.sharded_embed_host_shared), rank after rank into one registered matrix.

Every result is bit-equal to the C oracle (cbfs.bfs_hops / cbfs.normalise, x concatenated in front).

The graph is a random digraph whose hops stay below 8, plus a directed path of 40 nodes that only anchors on the
path can see.  An anchor at path position p makes its shard exactly p hops deep, so a test picks each shard's depth
(shallow <= 15 or deep > 15) by where it places one anchor, and checks that premise from the MS-BFS stats.
"""
import threading
from ctypes import c_void_p

import numpy as np
import pytest
import torch

from graphpope_b200 import distributed as gpd
from graphpope_b200 import synth

pytestmark = pytest.mark.gpu

R, L = 2000, 40  # random part, path part
N = R + L
SHALLOW_AT = (15, None, 11, 9, 13, 8, 14, 10)  # path position (= depth) of shard r's path anchor; None: no path anchor
MIXES = ("one_deep", "shallow", "all_deep")


@pytest.fixture(scope="module")
def dev():
    from graphpope_b200 import device
    return device


@pytest.fixture(scope="module")
def graphs():
    """(random part + path, random part alone, a 700-node two-way path) as int64 [2, E] arrays over N nodes."""
    rand = synth.random_digraph(R, 10 * R, seed=31)
    path = np.stack([R + np.arange(L - 1), R + np.arange(1, L)]).astype(np.int64)
    a = np.arange(699)
    long_path = np.stack([np.concatenate([a, a + 1]), np.concatenate([a + 1, a])]).astype(np.int64)
    return np.concatenate([rand, path], axis=1), rand, long_path


def _oracle(ei, anchors, x=None):
    from oracle import cbfs, geodesic
    feats = cbfs.normalise(cbfs.bfs_hops(cbfs.InCsr(ei, N), anchors))
    return feats if x is None else geodesic.concat_features(x, feats)


def _mix_anchors(world, kr, mix, seed):
    """world * kr anchors in the random part; one anchor of every shard moved onto the path to set its depth."""
    a = np.random.default_rng(seed).integers(0, R, world * kr)
    for r in range(world):
        if mix == "all_deep":
            p = L - 1 - r
        elif mix == "one_deep" and r == world - 1:
            p = L - 1
        else:
            p = SHALLOW_AT[r]
        if p is not None:
            a[r * kr + kr // 2] = R + p
    return a


def _check_premise(levels, mix):
    if mix == "shallow":
        assert max(levels) <= 15 and len(set(levels)) == len(levels), levels  # distinct: some shards get zeroed planes
    elif mix == "one_deep":
        assert levels[-1] > 15 and max(levels[:-1]) <= 15, levels
    else:
        assert min(levels) > 15, levels


def _bits_equal(got, want):
    return torch.equal(got.view(torch.int32), torch.as_tensor(want).to("cuda").view(torch.int32))


# ------------------------------------------------------------------ all-gather decode through the wrapper
class _Job:
    """The torch.distributed surface sharded_geodesic_features reads, for `world` ranks in host threads.  The process
    group argument is the rank itself; the two collectives meet at a barrier.  All ranks enqueue on the same default
    stream, so a clone enqueued before the barrier is ordered before every read after it."""

    def __init__(self, world):
        self.world = world
        self.barrier = threading.Barrier(world, timeout=120)
        self.planes, self.blocks = [0] * world, [None] * world

    def is_initialized(self):
        return True

    def get_world_size(self, group=None):
        return self.world

    def get_rank(self, group=None):
        return group

    def agree_num_planes(self, local_num_planes, group=None, device="cpu"):
        self.planes[group] = int(local_num_planes)
        self.barrier.wait()
        return max(self.planes)

    def gather_planes(self, local, group=None):
        self.blocks[group] = local.clone()
        self.barrier.wait()
        return torch.stack(self.blocks)


def _sharded_features(monkeypatch, engines, ei_d, a_d, x, outs):
    world = len(engines)
    job = _Job(world)
    monkeypatch.setattr(gpd, "dist", job)
    monkeypatch.setattr(gpd, "agree_num_planes", job.agree_num_planes)
    monkeypatch.setattr(gpd, "gather_planes", job.gather_planes)
    errors = []

    def rank(r):
        try:
            got = gpd.sharded_geodesic_features(engines[r], ei_d, a_d, x, outs[r], group=r)
            assert got is outs[r]
        except BaseException as e:  # noqa: BLE001 - re-raised below; the barrier releases the other ranks
            errors.append(e)
            job.barrier.abort()

    threads = [threading.Thread(target=rank, args=(r,)) for r in range(world)]
    [t.start() for t in threads]
    [t.join() for t in threads]
    if errors:
        raise errors[0]
    torch.cuda.synchronize()


@pytest.mark.parametrize("kr", [1, 3, 12, 24, 64, 65, 200, 256, 264, 520])
@pytest.mark.parametrize("world", [2, 3, 4, 8])
def test_gathered_decode_of_virtual_ranks(dev, graphs, monkeypatch, world, kr):
    """Per rank an engine of K/G lanes: the scalar decoder (K/G % 4 != 0 or x of 7 columns), the float4 one (12), the
    byte-lane one (K/G % 8 == 0); 1, 2 and 4 words per batch, up to 3 batches with a ragged last one.  The engines
    first run a 700-node path, so every plane past what a later shallow shard writes holds stale bits: the wrapper
    must zero them when another shard needs more planes."""
    ei, _, long_path = graphs
    ei_d = torch.as_tensor(ei).cuda()
    engines = [dev.GeodesicEngine(N, ei.shape[1], kr) for _ in range(world)]
    rng = np.random.default_rng(world * 1000 + kr)
    for eng in engines:
        eng.csr.build(torch.as_tensor(long_path).cuda())
        eng.bfs.run(torch.as_tensor(rng.integers(0, 700, kr)).cuda())
    # deep (>= 349 hops, whatever the anchors): every level array and the deep-hop planes now hold bits
    assert all(eng.bfs.stats()["max_level"] > 15 for eng in engines)
    xs = {f: torch.as_tensor(rng.standard_normal((N, f)).astype(np.float32)) for f in (7, 500)}
    for mix in MIXES:
        anchors = _mix_anchors(world, kr, mix, seed=kr + world)
        a_d = torch.as_tensor(anchors).cuda()
        block = _oracle(ei, anchors)
        for f in (None, 7, 500):
            x = None if f is None else xs[f]
            width = (f or 0) + world * kr
            outs = [torch.full((N, width), float("nan"), device="cuda") for _ in range(world)]
            _sharded_features(monkeypatch, engines, ei_d, a_d, None if x is None else x.cuda(), outs)
            _check_premise([eng.bfs.stats()["max_level"] for eng in engines], mix)
            want = torch.as_tensor(block if x is None else np.concatenate([x.numpy(), block], axis=1)).cuda()
            for r in range(world):
                assert _bits_equal(outs[r], want), (mix, f, r)


# ------------------------------------------------------------------ gp_decode_gathered at the ABI
def _shard_planes(dev, ei, anchors, world):
    """[G, rank_stride] int64 block of every shard's planes (zero past its own count), as the gather delivers it with
    a rank stride padded by 3 words; plus the agreed plane count and the layout."""
    kr = len(anchors) // world
    ei_d = torch.as_tensor(ei).cuda()
    metas, engines = [], []
    for r in range(world):
        eng = dev.GeodesicEngine(N, ei.shape[1], kr)
        eng.csr.build(ei_d)
        eng.bfs.run(torch.as_tensor(anchors[r * kr:(r + 1) * kr]).cuda())
        metas.append(eng.bfs.planes())
        engines.append(eng)
    p = max(m["num_planes"] for m in metas)
    stride = metas[0]["plane_stride_words"]
    rank_stride = p * stride + 3
    block = torch.zeros((world, rank_stride), dtype=torch.int64, device="cuda")
    for r, m in enumerate(metas):
        block[r, :m["num_planes"] * stride] = gpd._wrap_device_words(m["ptr"], m["num_planes"] * stride)
    torch.cuda.synchronize()
    return block, p, rank_stride, metas[0]


@pytest.mark.parametrize("kr,gap,pad,xoff,ldx,mix", [
    (12, 4, 8, 4, 32, "one_deep"),   # float4 decoder, 16-byte aligned x rows of a wider matrix
    (64, 4, 4, 0, 23, "shallow"),    # byte-lane decoder, x pitch not a multiple of 4
    (65, 3, 5, 2, 27, "one_deep"),   # scalar decoder
    (264, 8, 12, 1, 24, "all_deep"),  # byte-lane decoder, 2 batches, x rows start off 16 bytes
])
def test_decode_gathered_into_a_padded_output(dev, graphs, kr, gap, pad, xoff, ldx, mix):
    """Layouts sharded_geodesic_features never passes: the anchor block starts `gap` columns after x, rows are `pad`
    columns longer than the anchor block, x is a column slice of a wider matrix, shards are 3 words apart.  Columns
    outside x and the anchor block keep their NaN."""
    from graphpope_b200 import _lib
    ei = graphs[0]
    world, f = 3, 20
    anchors = _mix_anchors(world, kr, mix, seed=kr)
    block, p, rank_stride, meta = _shard_planes(dev, ei, anchors, world)
    assert p == (32 if mix != "shallow" else 16)
    xb = torch.randn(N, ldx, device="cuda")
    x = xb[:, xoff:xoff + f]
    k, col = world * kr, f + gap
    ld_out = col + k + pad
    out = torch.full((N, ld_out), float("nan"), device="cuda")
    lib = _lib.load()
    _lib.check(lib.gp_decode_gathered(dev._ptr(block), rank_stride, world, N, kr, p, meta["batches"],
                                      meta["words_per_batch"], meta["plane_stride_words"], dev._ptr(x), f, ldx,
                                      dev._ptr(out), ld_out, col, dev._stream()))
    torch.cuda.synchronize()
    assert torch.equal(out[:, :f], x)
    assert bool(out[:, f:col].isnan().all()) and bool(out[:, col + k:].isnan().all())
    assert _bits_equal(out[:, col:col + k].contiguous(), _oracle(ei, anchors))


def test_decode_gathered_argument_errors(dev):
    """Plane counts gp_msbfs_planes never reports, strides smaller than a plane or a shard, a negative column offset,
    an x pitch below its width and NULL buffers are refused before anything is launched.  The buffers are large
    enough (32 planes per rank and more) that a launch with any of these arguments would stay inside them."""
    from graphpope_b200 import _lib
    lib = _lib.load()
    n, kr, world, f = 100, 64, 3, 8  # one word per batch, one batch: a plane is n words
    ps = n
    buf = torch.zeros((world * 33 + 32) * ps, dtype=torch.int64, device="cuda")
    x = torch.zeros(n * f, device="cuda")
    ld_out = f + world * kr
    out_base = torch.zeros(8 + n * ld_out, device="cuda")
    out = out_base[8:]  # col_offset -1 of row 0 stays inside the allocation
    s = dev._stream()
    good = dict(g=buf, rs=16 * ps, p=16, ps=ps, x=x, ldx=f, out=out, coff=f)

    def call(**kw):
        a = dict(good, **kw)
        return lib.gp_decode_gathered(dev._ptr(a["g"]), a["rs"], world, n, kr, a["p"], 1, 1, a["ps"], dev._ptr(a["x"]),
                                      f, a["ldx"], dev._ptr(a["out"]), ld_out, a["coff"], s)

    bad = [
        dict(p=0, rs=0),
        dict(p=17, rs=17 * ps),
        dict(p=31, rs=31 * ps),
        dict(p=33, rs=33 * ps),
        dict(ps=ps - 1, rs=16 * (ps - 1)),  # plane stride below batches * words_per_batch * N
        dict(rs=16 * ps - 1),               # shards overlap
        dict(coff=-1),
        dict(ldx=f - 1),
        dict(g=None),
        dict(out=None),
    ]
    before = dev.launch_count()
    for kw in bad:
        assert call(**kw) == _lib.GP_ERR_INVALID, kw
    assert dev.launch_count() == before
    for kw in (dict(p=1, rs=ps), dict(), dict(p=32, rs=32 * ps)):
        assert call(**kw) == _lib.GP_OK, kw
    torch.cuda.synchronize()
    assert dev.launch_count() == before + 3


# ------------------------------------------------------------------ push exchange: the deep flag
@pytest.mark.parametrize("world", [1, 2, 3])
def test_push_exchange_deep_flag_is_per_step(dev, graphs, world):
    """Shard 0 is deep (> 15 hops) on the graph with the path and shallow without it.  Steps deep, shallow, deep, deep,
    shallow, shallow run on both slot parities; after each, item() on every rank is that step's flag, a shallow
    step's matrix equals the oracle, and on a deep step the shallow shards' columns and x do."""
    from graphpope_b200 import _lib
    lib = _lib.load()
    deep_ei, shallow_ei, _ = graphs
    per, f = 16, 12
    anchors = np.random.default_rng(world).integers(0, R, world * per)
    anchors[3] = N - 1  # the end of the path
    a_d = torch.as_tensor(anchors).cuda()
    x = torch.randn(N, f, device="cuda")
    engines = [dev.GeodesicEngine(N, deep_ei.shape[1], per) for _ in range(world)]
    xch = [gpd.PushExchange(engines[r], world=world, rank=r, grid_blocks=24) for r in range(world)]
    for r in range(world):
        for q in range(world):
            if q != r:
                xch[r].set_peer(q, xch[q].local_ptr())
    streams = [torch.cuda.Stream() for _ in range(world)]
    wants = {deep: np.concatenate([x.cpu().numpy(), _oracle(deep_ei if deep else shallow_ei, anchors)], axis=1)
             for deep in (True, False)}
    for step, deep in enumerate((True, False, True, True, False, False)):
        ei_d = torch.as_tensor(deep_ei if deep else shallow_ei).cuda()
        outs = [torch.full((N, f + world * per), float("nan"), device="cuda") for _ in range(world)]
        for r in range(world):
            engines[r].csr.build(ei_d)
            engines[r].bfs.run(a_d[r * per:(r + 1) * per].contiguous())
        levels = [eng.bfs.stats()["max_level"] for eng in engines]  # syncs: every shard is done before any exchange
        assert (levels[0] > 15) == deep and max(levels[1:], default=0) <= 15, levels
        for r in range(world):
            with torch.cuda.stream(streams[r]):
                _lib.check(lib.gp_exchange_run(xch[r]._h, c_void_p(x.data_ptr()), f, f, c_void_p(outs[r].data_ptr()),
                                               f + world * per, f, c_void_p(streams[r].cuda_stream)))
        torch.cuda.synchronize()
        keep = slice(0, None) if not deep else slice(f + per, None)
        for r in range(world):
            assert xch[r].item() == int(deep), (step, r)
            assert torch.equal(outs[r][:, :f], x), (step, r)
            assert _bits_equal(outs[r][:, keep].contiguous(), wants[deep][:, keep]), (step, r)
    for e in xch:
        e.close()


# ------------------------------------------------------------------ node-shared host matrix
@pytest.mark.parametrize("f", [0, 9])
@pytest.mark.parametrize("k,world", [(10, 4), (2, 3), (1, 2), (256, 8)])
def test_node_shared_matrix_from_virtual_ranks(dev, graphs, k, world, f):
    """sharded_embed_host_shared for ranks 0..G-1 in turn into one registered SharedHostMatrix, each rank with its own
    engine of max(1, ceil(K/G)) lanes (as utils.attach_distance_embedding sizes it): strided device-to-host copies
    into column offsets, ranks without anchors ((2, 3), (1, 2)), x split by rows.  The matrix equals the one-GPU
    host entry and the oracle bit for bit."""
    ei = torch.as_tensor(graphs[0])
    anchors = np.random.default_rng(k * 10 + f).integers(0, N, k)
    anchors[0] = N - 1  # the end of the path: one shard is deep
    x = torch.as_tensor(np.random.default_rng(f).standard_normal((N, f)).astype(np.float32)) if f else None
    want, _, _ = dev.geodesic_embed_host(ei, N, anchors, x)
    assert np.array_equal(want.numpy().view(np.uint32),
                          _oracle(graphs[0], anchors, None if x is None else x.numpy()).view(np.uint32))
    shared = gpd.SharedHostMatrix(N, f + k)
    try:
        shared.tensor.fill_(float("nan"))
        shared.barrier = lambda: None
        for r in range(world):
            shared.rank, shared.world = r, world
            eng = dev.GeodesicEngine(N, ei.size(1), max(1, -(-k // world)))
            out = gpd.sharded_embed_host_shared(eng, ei, anchors, x, shared, {})
            assert out is shared.tensor
            assert shared.shard == gpd.shard_bounds(k, world, r)
        assert torch.equal(shared.tensor.view(torch.int32), want.view(torch.int32))
    finally:
        shared.close()
