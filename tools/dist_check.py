"""torchrun check of the anchor-sharded path on real GPUs: bit-equal to the oracle / to the 1-GPU result."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
from graphpope_b200 import device as dev, distributed as gpd, synth

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
ok = True
for name, k_total in (("pubmed-shape", 256), ("flickr-shape", 1024), ("flickr-shape", 64 * world)):
    sh = synth.SHAPES[name]; n, f = sh.num_nodes, 20
    ei = synth.make_graph(sh); anchors = synth.stochastic_anchors(n, k_total, 42)
    ei_d, a_d = torch.as_tensor(ei).cuda(), torch.as_tensor(anchors).cuda()
    x_d = torch.randn(n, f, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    eng = dev.GeodesicEngine(n, ei.shape[1], k_total // world)
    out = gpd.sharded_geodesic_features(eng, ei_d, a_d, x_d)
    torch.cuda.synchronize()
    # single-GPU result of the same call (each rank computes it itself) must be bit-identical
    eng1 = dev.GeodesicEngine(n, ei.shape[1], k_total)
    ref = eng1.run(ei_d, a_d, x_d)
    same = bool(torch.equal(out, ref))
    if rank == 0:
        from oracle import cbfs
        want = cbfs.geodesic_features(ei, n, anchors)
        same_oracle = bool(np.array_equal(out[:, f:].cpu().numpy().view(np.uint32), want.view(np.uint32)))
        print(f"[{name} K={k_total} G={world}] sharded == 1-GPU: {same}; == oracle: {same_oracle}", flush=True)
        ok &= same_oracle
    ok &= same
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3): gpd.sharded_geodesic_features(eng, ei_d, a_d, x_d, out)
    dist.barrier(); torch.cuda.synchronize(); ev0.record()
    for _ in range(10): gpd.sharded_geodesic_features(eng, ei_d, a_d, x_d, out)
    ev1.record(); torch.cuda.synchronize()
    if rank == 0: print(f"    sharded step (NCCL all-gather of masks) {ev0.elapsed_time(ev1) / 10:.3f} ms", flush=True)
    # peer-to-peer assembly: one kernel packs this rank's shard and bulk-copies the peers' packed rows over NVLink
    peer = gpd.PeerAssembly(eng)
    out2, deep = peer.run(ei_d, a_d, x_d)
    torch.cuda.synchronize()
    same_p2p = bool(torch.equal(out2, ref)) and int(deep.item()) == 0
    ok &= same_p2p
    for _ in range(3): peer.run(ei_d, a_d, x_d, out2)
    dist.barrier(); torch.cuda.synchronize(); ev0.record()
    for _ in range(10): peer.run(ei_d, a_d, x_d, out2)
    ev1.record(); torch.cuda.synchronize()
    if rank == 0: print(f"    p2p == 1-GPU: {same_p2p}; p2p step {ev0.elapsed_time(ev1) / 10:.3f} ms", flush=True)
    dist.barrier(); peer.close()
# BASELINE config C4: Flickr-shape, 1024 anchors from the degree / PageRank samplers (device), anchor-sharded
from graphpope_b200 import utils
sh = synth.SHAPES["flickr-shape"]; n = sh.num_nodes
ei = synth.make_graph(sh); ei_d = torch.as_tensor(ei).cuda()
class _D: pass
d = _D(); d.num_nodes, d.edge_index = n, torch.as_tensor(ei)
for method in ("degree_centrality", "pagerank"):
    anchors = np.asarray(utils.sample_anchor_nodes(d, 1024, method), dtype=np.int64)  # identical on every rank
    a_d = torch.as_tensor(anchors).cuda()
    eng = dev.GeodesicEngine(n, ei.shape[1], 1024 // world)
    peer = gpd.PeerAssembly(eng)
    out, deep = peer.run(ei_d, a_d, None)
    torch.cuda.synchronize()
    good = int(deep.item()) == 0
    if rank == 0:
        from oracle import cbfs, samplers
        want_anchors = (samplers.degree_centrality_anchors if method == "degree_centrality" else samplers.pagerank_anchors)(ei, n, 1024)
        same_list = anchors.tolist() == want_anchors
        want = cbfs.geodesic_features(ei, n, anchors)
        same = bool(np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32)))
        print(f"[C4 flickr-shape K=1024 {method} G={world}] anchor list == oracle: {same_list}; features == oracle: {same}", flush=True)
        good &= same_list and same
    ok &= good
    dist.barrier(); peer.close()
t = torch.tensor([int(ok)], device="cuda"); dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0: print("DIST CHECK", "PASSED" if int(t.item()) else "FAILED", flush=True)
dist.destroy_process_group()
sys.exit(0 if int(t.item()) else 1)
