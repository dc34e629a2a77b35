"""torchrun check of the compact store under DDP: every rank calls utils.Graphpope with GRAPHPOPE_OUTPUT=compact and
GRAPHPOPE_SHARED=1, so the ranks split the anchors and all-gather their shard stores.  Every rank's store must be
byte-identical to a one-GPU FeatureStore.build on that rank, and rank 0 checks to_dense() against the oracle, for a
stochastic and a device sampler and for fewer anchors than ranks.

    torchrun --nproc_per_node G tools/ddp_compact_check.py
"""
import os, sys
os.environ["GRAPHPOPE_OUTPUT"] = "compact"; os.environ["GRAPHPOPE_SHARED"] = "1"; os.environ["GRAPHPOPE_QUIET"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
from graphpope_b200 import device as dev, distributed as gpd, synth, utils
rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ok = True
for name, k, method in (("pubmed-shape", 256, "stochastic"), ("flickr-shape", 100, "degree_centrality"), ("pubmed-shape", 3, "stochastic")):
    sh = synth.SHAPES[name]; n = sh.num_nodes
    ei = synth.make_graph(sh)
    x = torch.randn(n, 20, generator=torch.Generator().manual_seed(5))
    class D: pass
    d = D(); d.num_nodes, d.edge_index, d.x = n, torch.as_tensor(ei), x
    np.random.seed(42); utils.clear_cache()
    store = utils.Graphpope(d, name, "geodesic", method, k, None, num_workers=6)
    one = dev.FeatureStore.build(ei, n, d.anchor_nodes, x)
    lo, hi = gpd.shard_bounds(k, world, rank)
    good = (isinstance(store, dev.FeatureStore) and tuple(store.shape) == (n, 20 + k)
            and torch.equal(store.raw.view(torch.int64), one.raw.view(torch.int64))
            and store.stats["max_level"] == one.stats["max_level"])
    print(f"[rank {rank}: {name} K={k} {method} G={world}] anchors [{lo}, {hi}), P={store.num_planes}, "
          f"raw == one-GPU store {good}", flush=True)
    if rank == 0:
        from oracle import cbfs, geodesic
        want = geodesic.concat_features(x.numpy(), cbfs.geodesic_features(ei, n, np.asarray(d.anchor_nodes)))
        same = bool(np.array_equal(store.to_dense().cpu().numpy().view(np.uint32), want.view(np.uint32)))
        print(f"[{name} K={k} {method} G={world}] to_dense() == oracle {same}", flush=True)
        good &= same
    ok &= good
    del store, one
t = torch.tensor([int(ok)], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0: print("DDP COMPACT CHECK", "PASSED" if int(t.item()) else "FAILED", flush=True)
dist.destroy_process_group()
sys.exit(0 if int(t.item()) else 1)
