"""Drop-in mirror of the reference's ``utils.py`` embedding helpers, backed by the B200 library.

Same names, argument meaning, side effects and error behaviour as
JeroendenBoef/GraphPOPE ``utils.py`` (citations are file:line into the reference):

    sample_anchor_nodes                      utils.py:18-62
    shortest_path_length                     utils.py:64-81
    merge_dicts                              utils.py:83-90
    all_pairs_shortest_path_length_parallel  utils.py:92-114
    get_geodesic_distance_vector             utils.py:116-126
    concat_into_features                     utils.py:129-135
    attach_distance_embedding                utils.py:137-147
    attach_node2vec                          utils.py:149-180
    Graphpope                                utils.py:182-210

``main.py`` keeps ``from utils import Graphpope`` and its flags (``--embedding_space``,
``--sampling_method``, ``--num_anchor_nodes``, ``--distance_function``,
``--num_workers``, main.py:34-39) unchanged; ``num_workers`` is accepted and ignored —
the CPU process pool it sized (utils.py:98) is replaced by one multi-source BFS on the GPU.

What runs where
  * geodesic distances, 1/(d+1) normalisation, concat: device (libgraphpope_b200.so).
  * ``stochastic`` anchors: host numpy global RNG, exactly utils.py:22-24 (same seed, same anchors).
  * ``degree_centrality`` / ``pagerank`` / ``closeness_centrality`` / ``clustering_coefficient`` /
    ``betweenness_centrality`` anchors: device (degree array, float64 SpMV power iteration, MS-BFS from every
    node + bit-sliced column sums, directed triangle counting, Brandes with 32 sources per warp-wide batch;
    stable top-k).
  * KMeans centres of the node2vec branch: device (k-means++ + Lloyd, tensor-core assignment; statistical
    parity with scikit-learn, which the reference runs unseeded).
  * ``eigenvector_centrality`` anchors: device (float64 power iteration on ``A^T + I``; strong connectivity
    checked with two single-anchor MS-BFS sweeps, as networkx >= 3.2 refuses disconnected graphs).
    ``GRAPHPOPE_BETWEENNESS=networkx`` / ``GRAPHPOPE_EIGENVECTOR=networkx`` keep the reference's own calls.
Inside a ``torch.distributed`` job ``GRAPHPOPE_SHARED=1`` makes the ranks of a node share the geodesic work and
return ONE node-shared host matrix instead of computing a private copy each (main.py:88-98 runs this in every rank).
There is no CPU fallback for the device parts: without the CUDA library or a GPU these functions raise.
"""
from __future__ import annotations

import os
import os.path as osp

import numpy as np
import torch

from . import device as _dev
from . import _lib

# Opt-in symmetrisation (north_star wording); the default keeps the reference's DiGraph semantics
# (utils.py:121).  It is the identity on Flickr / PubMed / ogbn-products, whose edge_index is symmetric.
SYMMETRIZE = os.environ.get("GRAPHPOPE_SYMMETRIZE", "0") == "1"
VERBOSE = os.environ.get("GRAPHPOPE_QUIET", "0") != "1"


def _output_device() -> str:
    """``GRAPHPOPE_OUTPUT=cuda`` keeps the ``[N, F+K]`` matrix in HBM (SURVEY §8f rank 3: the trainer's
    ``x[n_id]`` gathers, main.py:120,177, then run on the device and the 91 MB device->host copy plus the
    host concat disappear).  ``GRAPHPOPE_OUTPUT=compact`` returns a :class:`device.FeatureStore` instead: x on the
    device plus the anchor block in ``1 + bit_length(max hop)`` bits per entry, whose ``store[n_id]`` gathers the
    trainer's rows without ever forming the dense matrix (geodesic space only; node2vec values have no compact form
    and behave as ``cuda``).  Default ``cpu`` = the reference's contract."""
    return os.environ.get("GRAPHPOPE_OUTPUT", "cpu")


def _shared_world():
    """``GRAPHPOPE_SHARED=1`` inside an initialised ``torch.distributed`` job with more than one rank: the ranks of
    the node share the work AND the result (SURVEY §8 f3).  The reference runs ``Graphpope`` in every DDP rank
    (main.py:88-98) and each ends up with its own copy of the same matrix; here rank r runs the MS-BFS for its
    ``K/G`` anchors only and all ranks return one page-locked ``[N, F+K]`` matrix in POSIX shared memory
    (``distributed.SharedHostMatrix``).  Needs identical anchors on every rank — true for every sampler under the
    reference's ``seed_everything`` (main.py:260)."""
    if os.environ.get("GRAPHPOPE_SHARED", "0") != "1":
        return None
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1):
        return None
    return dist


_shared_keepalive: list = []  # node-shared matrices handed out (their CUDA registration lives as long as the process)


def _cache_dir():
    """``GRAPHPOPE_CACHE_DIR`` extends the reference's in-process memo (utils.py:195-208) across runs
    (SURVEY §8f rank 4): the float32 ``[N, K]`` distance block is stored under a key derived from the
    graph, the anchors and the options.  Unset = no files are read or written."""
    return os.environ.get("GRAPHPOPE_CACHE_DIR") or None


def block_cache_key(edge_index, num_nodes, anchors, symmetrize=False) -> str:
    import hashlib

    h = hashlib.sha256()
    h.update(b"graphpope-geodesic-block-v1")
    h.update(np.int64([int(num_nodes), int(bool(symmetrize))]).tobytes())
    ei = torch.as_tensor(edge_index).to(device="cpu", dtype=torch.int64).contiguous()
    h.update(np.int64(list(ei.shape)).tobytes())
    h.update(ei.numpy().tobytes())
    h.update(np.ascontiguousarray(np.asarray(anchors, dtype=np.int64)).tobytes())
    return h.hexdigest()


def _cached_block(data):
    d = _cache_dir()
    if d is None:
        return None, None
    key = block_cache_key(_edge_index_of(data), data.num_nodes, data.anchor_nodes, SYMMETRIZE)
    path = osp.join(d, key + ".pt")
    if osp.exists(path):
        try:
            # weights_only: the cache directory may be shared between users / DDP ranks; never unpickle code
            blk = torch.load(path, map_location="cpu", weights_only=True)
        except Exception:
            return None, path  # unreadable or foreign file: a cache miss, recomputed and overwritten
        if (torch.is_tensor(blk) and tuple(blk.shape) == (int(data.num_nodes), len(data.anchor_nodes))
                and blk.dtype == torch.float32):
            return blk, path
    return None, path


def _store_block(path, block):
    if path is None:
        return
    os.makedirs(osp.dirname(path), exist_ok=True)
    tmp = path + ".tmp%d" % os.getpid()
    torch.save(block.detach().cpu().contiguous(), tmp)
    os.replace(tmp, path)  # atomic: DDP ranks may race to write the same key

# reached only through GRAPHPOPE_BETWEENNESS=networkx / GRAPHPOPE_EIGENVECTOR=networkx, or (clustering) for graphs whose
# node bitmaps do not fit in shared memory: the reference's own networkx call
_HOST_CENTRALITIES = ("betweenness_centrality", "eigenvector_centrality", "clustering_coefficient")

last_stats: dict = {}  # stats of the most recent MS-BFS (levels, edges examined, ...)


def _say(msg):
    if VERBOSE:
        print(msg)


def _edge_index_of(data) -> torch.Tensor:
    ei = data.edge_index
    if not torch.is_tensor(ei):
        ei = torch.as_tensor(np.asarray(ei))
    return ei.to(torch.int64)


def _to_networkx(data):
    """PyG ``to_networkx(data)`` defaults as called at utils.py:27,33,...: DiGraph, nodes 0..N-1."""
    import networkx as nx

    G = nx.DiGraph()
    G.add_nodes_from(range(int(data.num_nodes)))
    ei = _edge_index_of(data).cpu()
    G.add_edges_from(zip(ei[0].tolist(), ei[1].tolist()))
    return G


def _device_csr(data) -> _dev.DeviceCsr:
    _lib.require_cuda()  # no CPU fallback: fail loudly before touching torch.cuda
    ei = _edge_index_of(data).cuda(non_blocking=True)
    csr = _dev.DeviceCsr(int(data.num_nodes), ei.size(1), symmetrize=False)
    return csr.build(ei)


def sample_anchor_nodes(data, num_anchor_nodes, sampling_method):
    """utils.py:18-62.  ndarray for ``stochastic``, ``list[int]`` (ascending score) otherwise."""
    if sampling_method == 'stochastic':
        # host numpy global RNG, with replacement — identical stream to utils.py:23-24
        return np.random.choice(np.arange(data.num_nodes), num_anchor_nodes)

    if sampling_method == 'degree_centrality':
        csr = _device_csr(data)
        csr.info()  # surfaces a bad edge_index as an exception
        return _dev.topk_stable(csr.degree(), num_anchor_nodes).cpu().tolist()

    if sampling_method == 'pagerank':
        csr = _device_csr(data)
        score, _ = csr.pagerank()  # networkx pagerank_scipy defaults
        return _dev.topk_stable(score, num_anchor_nodes).cpu().tolist()

    if sampling_method == 'closeness_centrality':
        # every node as an anchor of the MS-BFS + bit-sliced column sums (gp_closeness.cu)
        csr = _device_csr(data)
        return _dev.topk_stable(csr.closeness(), num_anchor_nodes).cpu().tolist()

    if sampling_method == 'clustering_coefficient' and int(data.num_nodes) <= 800_000:
        # directed triangle counting against shared-memory node bitmaps (gp_closeness.cu); larger graphs
        # keep the networkx call below
        csr = _device_csr(data)
        return _dev.topk_stable(csr.clustering(), num_anchor_nodes).cpu().tolist()

    if sampling_method == 'betweenness_centrality' and os.environ.get("GRAPHPOPE_BETWEENNESS", "cuda") != "networkx":
        # Brandes, 32 sources per warp-wide batch, level-synchronous pull sweeps (gp_betweenness.cu); scores
        # within a few ulp of networkx (GRAPHPOPE_BETWEENNESS=networkx keeps the reference's call below)
        csr = _device_csr(data)
        return _dev.topk_stable(csr.betweenness(), num_anchor_nodes).cpu().tolist()

    if sampling_method == 'eigenvector_centrality' and os.environ.get("GRAPHPOPE_EIGENVECTOR", "cuda") != "networkx":
        # float64 power iteration on A^T + I (gp_sampler.cu); networkx hands the matrix to ARPACK, whose random
        # start makes even the reference reproducible only to ~1e-16 (GRAPHPOPE_EIGENVECTOR=networkx keeps its call)
        import networkx as nx

        n = int(data.num_nodes)
        if n == 0:
            raise nx.NetworkXPointlessConcept("cannot compute centrality for the null graph")
        ei = _edge_index_of(data)
        # The power iteration has a unique limit only on a strongly connected graph: node 0 must reach, and be
        # reached by, every node — two single-anchor sweeps of the MS-BFS.  Anything else is handed to the
        # reference's own networkx call below, which decides for the installed networkx (>= 3.2 raises
        # AmbiguousSolution, older versions return ARPACK's vector for such graphs).
        connected = True
        for e in (ei, ei.flip(0)):
            _, hops, _ = _dev.geodesic_embed_host(e.contiguous(), n, [0], None, False, want_hops=True)
            if bool((hops.numpy() == _lib.GP_UNREACHABLE_U16).any()):
                connected = False
                break
        if connected:
            try:
                score, _ = _device_csr(data).eigenvector()
                return _dev.topk_stable(score, num_anchor_nodes).cpu().tolist()
            except nx.PowerIterationFailedConvergence:
                pass  # tiny spectral gap (e.g. long paths): ARPACK below does not depend on it

    if sampling_method in _HOST_CENTRALITIES:
        # Not re-implemented (north_star): the reference's own networkx call, same top-k rule.
        import networkx as nx

        G = _to_networkx(data)
        score = {
            'betweenness_centrality': nx.betweenness_centrality,
            'eigenvector_centrality': nx.eigenvector_centrality_numpy,
            'clustering_coefficient': nx.clustering,
        }[sampling_method](G)
        ranked = sorted(score.items(), key=lambda item: item[1])  # stable, ascending
        return [k for k, _ in ranked][-num_anchor_nodes:]

    # the reference falls through every ``if`` and fails at ``return`` (utils.py:62)
    raise UnboundLocalError("cannot access local variable 'sampled_anchor_nodes' where it is not "
                            "associated with a value")


def _graph_to_edge_index(G):
    n = G.number_of_nodes()
    if n and (min(G.nodes) != 0 or max(G.nodes) != n - 1):
        raise ValueError("graph nodes must be labelled 0..N-1 (as to_networkx produces)")
    edges = np.asarray(list(G.edges()), dtype=np.int64).reshape(-1, 2)
    if not G.is_directed():
        edges = np.concatenate([edges, edges[:, ::-1]], axis=0)
    return torch.from_numpy(np.ascontiguousarray(edges.T)), n


def _hops_of_graph(G, anchor_nodes):
    """uint16 hop matrix [N, K] of a networkx graph (nodes 0..N-1) from one device MS-BFS."""
    ei, n = _graph_to_edge_index(G)
    anchors = [int(a) for a in anchor_nodes]
    _, hops, stats = _dev.geodesic_embed_host(ei, n, anchors, None, False, want_hops=True)
    last_stats.update(stats)
    return hops.numpy()


def _rows_as_reference_lists(h, nodes):
    """utils.py:69-78: per node a list of Python floats ``1/len(path)`` = ``1/(hops+1)`` and the *int* ``0``
    where there is no path (utils.py:76 appends a literal 0)."""
    out = {}
    for node in nodes:
        out[node] = [0 if d == _lib.GP_UNREACHABLE_U16 else 1 / (int(d) + 1) for d in h[node].tolist()]
    return out


def shortest_path_length(G, anchor_nodes, partition_length):
    """utils.py:64-81: ``{node: [1/len(path) per anchor]}`` with ``0`` where there is no path, keys in the
    order of ``partition_length``.

    ``G`` is the networkx graph ``to_networkx`` built; distances come from one device MS-BFS.
    Values are Python floats ``1/(d+1)`` and the int ``0``, exactly as the reference appends them.
    """
    return _rows_as_reference_lists(_hops_of_graph(G, anchor_nodes), partition_length)


def merge_dicts(dicts):
    """utils.py:83-90: later dicts win, insertion order of first appearance is kept."""
    merged = {}
    for part in dicts:
        merged.update(part)
    return merged


def all_pairs_shortest_path_length_parallel(G, anchor_nodes, num_workers):
    """utils.py:92-114.  ``num_workers`` sized a CPU pool there; one GPU sweep replaces the pool, but the node
    slices ``nodes[int(N/w*i):int(N/w*(i+1))]`` (utils.py:100, float arithmetic) and their ordered merge are
    kept, so the returned dict has the reference's keys in the reference's order."""
    nodes = list(G.nodes)
    h = _hops_of_graph(G, anchor_nodes)
    parts = [_rows_as_reference_lists(h, nodes[int(len(nodes) / num_workers * i):int(len(nodes) / num_workers * (i + 1))])
             for i in range(num_workers)]
    return merge_dicts(parts)


def get_geodesic_distance_vector(data, num_workers):
    """utils.py:116-126: float32 ``[N, K]`` of ``1/(hops(node -> anchor)+1)``, 0 when unreachable.

    Reads ``data.anchor_nodes``.  Always float32 (the reference yields int64 in the degenerate case
    where every entry is 0, SURVEY.md App. A #3).  Under ``GRAPHPOPE_OUTPUT=compact`` a
    :class:`device.FeatureStore` with F = 0 (no cache file is read or written).
    """
    if _output_device() == "compact":
        return _compact_features(data, None)
    blk, path = _cached_block(data)
    if blk is not None:
        return blk.cuda() if _output_device() == "cuda" else blk
    if _output_device() == "cuda":
        out = _device_features(data, None)
    else:
        out, _, stats = _dev.geodesic_embed_host(_edge_index_of(data), int(data.num_nodes), data.anchor_nodes,
                                                 None, SYMMETRIZE)
        last_stats.update(stats)
    _store_block(path, out)
    return out


def _device_features(data, x):
    """Device-resident result: edge_index (and x) go up once, the ``[N, F+K]`` matrix stays in HBM."""
    _lib.require_cuda()
    n = int(data.num_nodes)
    ei = _edge_index_of(data).cuda(non_blocking=True)
    anchors = torch.as_tensor(np.asarray(data.anchor_nodes, dtype=np.int64)).cuda(non_blocking=True)
    eng = _dev.GeodesicEngine(n, ei.size(1), max(1, anchors.numel()), SYMMETRIZE)
    x_d = None if x is None else x.to(device="cuda", dtype=torch.float32, non_blocking=True).contiguous()
    out = eng.run(ei, anchors, x_d)
    last_stats.update(eng.bfs.stats())  # syncs; surfaces index errors
    return out


def _compact_features(data, x):
    """``GRAPHPOPE_OUTPUT=compact``: the device-resident result as a :class:`device.FeatureStore` (x on the device,
    the anchor block packed); the dense ``[N, F+K]`` matrix is never formed.  With ``GRAPHPOPE_SHARED=1`` in a
    multi-rank job the ranks split the anchors: each runs the MS-BFS for its ``K/G`` of them, and every rank ends up
    holding the same whole store (``distributed.sharded_feature_store``)."""
    if x is not None and x.dtype != torch.float32:
        raise TypeError(f"GRAPHPOPE_OUTPUT=compact needs float32 data.x (got {x.dtype}): concat_into_features would "
                        "type-promote the anchor block")
    if _shared_world() is not None:
        from . import distributed as _gpd

        store = _gpd.sharded_feature_store(_edge_index_of(data), int(data.num_nodes), data.anchor_nodes, x,
                                           SYMMETRIZE)
    else:
        store = _dev.FeatureStore.build(_edge_index_of(data), int(data.num_nodes), data.anchor_nodes, x, SYMMETRIZE)
    last_stats.update(store.stats)
    return store


def concat_into_features(embedding_matrix, data):
    """utils.py:129-135: ``torch.cat((data.x, embedding), 1)``."""
    emb = torch.as_tensor(embedding_matrix)
    if emb.is_cuda and not data.x.is_cuda:
        return torch.cat((data.x.to(emb.device), emb), 1)  # GRAPHPOPE_OUTPUT=cuda: the result lives in HBM
    return torch.cat((data.x, emb.to(data.x.device)), 1)


def attach_distance_embedding(data, dataset, num_anchor_nodes, sampling_method, distance_function, num_workers):
    """utils.py:137-147.  Sets ``data.anchor_nodes``; returns a new CPU float32 ``[N, F + K]`` (a device tensor or a
    :class:`device.FeatureStore` under ``GRAPHPOPE_OUTPUT=cuda`` / ``compact``).

    Distance block and concat are one fused C-ABI call (the epilogue writes the ``[N, F+K]`` rows once).
    """
    _say('sampling anchor nodes...')
    data.anchor_nodes = sample_anchor_nodes(data=data, num_anchor_nodes=num_anchor_nodes,
                                            sampling_method=sampling_method)
    _say('deriving shortest paths to anchor nodes...')
    x = data.x
    if _output_device() == "compact":
        out = _compact_features(data, x)
        _say('feature matrix is blessed by the POPE!')
        return out
    if x.dtype != torch.float32 or _cache_dir() is not None:
        # torch.cat type-promotes; keep that behaviour by taking the generic route (also the cached one:
        # the cache holds the [N, K] block, not the concatenation)
        return concat_into_features(get_geodesic_distance_vector(data, num_workers), data)
    dist = _shared_world()
    if _output_device() == "cuda":
        out = _device_features(data, x)
    elif dist is not None:
        from . import distributed as _gpd

        _lib.require_cuda()
        n, k = int(data.num_nodes), len(data.anchor_nodes)
        ei = _edge_index_of(data).to("cpu").contiguous()
        xc = x.to("cpu").contiguous()
        eng = _dev.GeodesicEngine(n, ei.size(1), max(1, -(-k // dist.get_world_size())), SYMMETRIZE)
        shared = _gpd.SharedHostMatrix(n, xc.size(1) + k)
        out = _gpd.sharded_embed_host_shared(eng, ei, data.anchor_nodes, xc, shared, {})
        _shared_keepalive.append(shared)
        if k and shared.shard[1] > shared.shard[0]:
            last_stats.update(eng.bfs.stats())
    else:
        out, _, stats = _dev.geodesic_embed_host(_edge_index_of(data), int(data.num_nodes), data.anchor_nodes,
                                                 x, SYMMETRIZE)
        last_stats.update(stats)
    _say('feature matrix is blessed by the POPE!')
    return out


def node2vec_path(dataset):
    """Where utils.py:155 looks: ``<module dir>/data/<dataset>_node2vec.pt`` (override: GRAPHPOPE_DATA_DIR)."""
    base = os.environ.get("GRAPHPOPE_DATA_DIR") or osp.join(osp.dirname(osp.realpath(__file__)), 'data')
    return osp.join(base, f'{dataset}_node2vec.pt')


def attach_node2vec(data, dataset, num_anchor_nodes, sampling_method, distance_function, num_workers):
    """utils.py:149-180: pairwise distances to anchor embeddings, per-column min-max, concat."""
    _say('sampling anchor nodes...')
    table = torch.load(node2vec_path(dataset), map_location="cpu").detach()
    mode = _lib.CDIST_MODES[distance_function]  # KeyError on an unknown key, as utils.py:164
    if sampling_method == 'stochastic':
        anchor_nodes = sample_anchor_nodes(data, num_anchor_nodes, sampling_method='stochastic')
        anchor_emb = table[torch.as_tensor(np.asarray(anchor_nodes, dtype=np.int64))]
    else:
        # anything but 'stochastic' means KMeans centres (utils.py:168-170).  Lloyd + k-means++ run on the
        # device (tensor-core assignment); GRAPHPOPE_KMEANS=sklearn keeps the reference's scikit-learn call.
        # (tables wider than 128 columns keep scikit-learn for the clustering; the pairwise block below runs on the
        # device for any width)
        if os.environ.get("GRAPHPOPE_KMEANS", "device") == "sklearn" or table.size(1) > 128:
            from sklearn.cluster import KMeans

            kmeans = KMeans(n_clusters=num_anchor_nodes).fit(table.numpy())
            anchor_emb = torch.as_tensor(kmeans.cluster_centers_)
        else:
            anchor_emb, _, _ = _dev.kmeans(table, num_anchor_nodes)
        _say('K means cluster anchor nodes derived!')
    block = _dev.cdist_minmax(table, anchor_emb, mode, apply_minmax=True)
    out = concat_into_features(block if _output_device() in ("cuda", "compact") else block.cpu(), data)
    _say('feature matrix is blessed by the POPE')
    return out


def clear_cache():
    """Drop the process-global memo (extension; the reference has no way to reset it)."""
    globals().pop("cached_pope_embedding", None)


def Graphpope(data, dataset: str, embedding_space: str, sampling_method: str, num_anchor_nodes: int,
              distance_function=None, num_workers=4):
    """utils.py:182-210.  Dispatch on ``embedding_space`` in {'geodesic', 'node2vec'}.

    Keeps the reference's process-global memo: the first call computes, every later call returns
    the cached tensor whatever its arguments (utils.py:195-208).
    """
    global cached_pope_embedding
    pope_map = {
        'geodesic': attach_distance_embedding,
        'node2vec': attach_node2vec,
    }
    try:
        enhanced_features = cached_pope_embedding
    except NameError:
        pope = pope_map[embedding_space]  # KeyError on an unknown space, as utils.py:206
        enhanced_features = pope(data, dataset, num_anchor_nodes, sampling_method, distance_function,
                                 num_workers=num_workers)
        cached_pope_embedding = enhanced_features
    return enhanced_features
