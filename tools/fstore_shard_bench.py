"""Anchor-sharded compact store build (distributed.sharded_feature_store) at the world size it is launched with.

For the Flickr-shape (K = 256) and products-shape (K = 4096) graphs of bench.py (same generators, graph seeds and
anchor seed 42) every rank reports, per shape:
  * ms of each stage, run one after another with the product's own helpers, each ended by a device synchronise:
    csr + MS-BFS (with the stats read that the pack needs), plane agreement, pack (+ zero padding of a short shard),
    NCCL all-gather (includes waiting for the slowest rank), merge (gp_fstore_merge, also timed by CUDA events);
  * ms of the whole sharded_feature_store call, from a barrier to a device synchronise and a barrier;
  * ms of the one-GPU FeatureStore.build of all K anchors on the same GPU, and whether the stores are byte-equal;
  * peak device memory of the sharded and the one-GPU build, from torch.cuda.mem_get_info drops (the BFS workspace
    is allocated by the library, outside torch's allocator);
  * the merge's bytes (S*N*P*Ws*8 read + N*P*W*8 written) per second against a device-to-device copy measured in
    the same run.
Medians over --reps repetitions after one warm-up.  Rank 0 prints one JSON line (all ranks' numbers, the GPU name
and power limit read in the same run).

    torchrun --nproc_per_node G tools/fstore_shard_bench.py [--shapes flickr-shape,products-shape] [--reps 5]
             [--json PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

SHAPE_K = {"flickr-shape": 256, "products-shape": 4096}


def card_info() -> dict:
    info = {"torch_name": torch.cuda.get_device_name()}
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                            "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"not available: {e}"
    return info


def copy_peak_gbs(nbytes=2 << 30, reps=5) -> float:
    """Device-to-device copy (bytes read + written per second), best of `reps`."""
    a = torch.empty(nbytes // 4, dtype=torch.float32, device="cuda").fill_(1.0)
    b = torch.empty_like(a)
    best = 0.0
    for _ in range(reps + 1):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        b.copy_(a)
        e.record()
        e.synchronize()
        best = max(best, 2 * nbytes / (s.elapsed_time(e) * 1e-3) / 1e9)
    del a, b
    torch.cuda.empty_cache()
    return best


def free_bytes() -> int:
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info()[0]


def make_graph(shape):
    from graphpope_b200 import synth
    if shape.name == "products-shape":
        return synth.chung_lu_symmetric_torch(shape.num_nodes, shape.num_directed_edges, shape.pareto_alpha,
                                              shape.seed, "cuda")
    return torch.as_tensor(synth.make_graph(shape)).cuda()


def same_on_every_rank(t: torch.Tensor) -> bool:
    """The ranks generated the same graph: MIN == MAX of a wrapping int64 digest."""
    w = torch.arange(1, t.numel() + 1, device=t.device, dtype=torch.int64)
    h = (t.reshape(-1).to(torch.int64) * w).sum().reshape(1)
    lo, hi = h.clone(), h.clone()
    dist.all_reduce(lo, op=dist.ReduceOp.MIN)
    dist.all_reduce(hi, op=dist.ReduceOp.MAX)
    return bool(lo.item() == hi.item())


def staged(ei, n, anchors):
    """sharded_feature_store's steps one at a time (same helpers, same order).  Returns (store, ms per stage,
    merge kernel ms, lowest free device memory seen, bytes of the gathered shards)."""
    from graphpope_b200 import device as dev
    from graphpope_b200 import distributed as gpd

    world, rank = dist.get_world_size(), dist.get_rank()
    k = anchors.size
    ms, low = {}, [free_bytes()]
    clock = [time.perf_counter()]

    def lap(name):
        torch.cuda.synchronize()
        now = time.perf_counter()
        ms[name] = (now - clock[0]) * 1e3
        clock[0] = now
        low.append(torch.cuda.mem_get_info()[0])

    gpd.check_anchors_agree(anchors, device="cuda")
    lap("anchor_check")
    lo, hi = gpd.shard_bounds(k, world, rank)
    csr = bfs = None
    level = 0
    if hi > lo:
        csr = dev.DeviceCsr(n, ei.size(1)).build(ei)
        bfs = dev.MsBfs(csr, hi - lo).run(torch.from_numpy(anchors[lo:hi]).cuda())
        level = bfs.stats()["max_level"]
    lap("csr_msbfs")
    p, _, _ = gpd.agree_store_layout(1 + level.bit_length(), level, False, None, "cuda")
    lap("plane_agreement")
    shard = dev.FeatureStore(bfs, num_planes=p).raw if bfs is not None else None
    block = gpd.pad_shard_store(shard, n, p, gpd.shard_words(k, world), device="cuda")
    lap("pack")
    for h in (bfs, csr):
        if h is not None:
            h.close()
    del shard
    gathered = gpd.gather_planes(block)
    del block
    lap("all_gather")
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    store = dev.FeatureStore.from_shards(gathered, k)
    e.record()
    lap("merge")
    merge_kernel_ms = s.elapsed_time(e)
    del gathered
    return store, ms, merge_kernel_ms, min(low), gathered_bytes(world, store, k)


def gathered_bytes(world, store, k):
    from graphpope_b200 import distributed as gpd
    return world * store.num_nodes * store.num_planes * gpd.shard_words(k, world) * 8


def run_shape(name, reps, peak):
    from graphpope_b200 import device as dev
    from graphpope_b200 import distributed as gpd
    from graphpope_b200 import synth

    world = dist.get_world_size()
    shape = synth.SHAPES[name]
    n, k = shape.num_nodes, SHAPE_K[name]
    ei = make_graph(shape)
    same_graph = same_on_every_rank(ei)
    anchors = np.asarray(synth.stochastic_anchors(n, k, 42), dtype=np.int64)
    torch.cuda.empty_cache()

    stages, merge_ms, whole, peak_sharded = [], [], [], 0
    for i in range(reps + 1):
        dist.barrier()
        free0 = free_bytes()
        store, ms, mk, low, gbytes = staged(ei, n, anchors)
        if i:
            stages.append(ms)
            merge_ms.append(mk)
        peak_sharded = max(peak_sharded, free0 - low)
        raw_sharded = store.raw.clone() if i == reps else None
        del store
        torch.cuda.empty_cache()
    for i in range(reps + 1):
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        store = gpd.sharded_feature_store(ei, n, anchors)
        torch.cuda.synchronize()
        dist.barrier()
        if i:
            whole.append((time.perf_counter() - t0) * 1e3)
        del store
        torch.cuda.empty_cache()

    one_ms, peak_one = [], 0
    for i in range(reps + 1):
        free0 = free_bytes()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        csr = dev.DeviceCsr(n, ei.size(1)).build(ei)
        bfs = dev.MsBfs(csr, k).run(torch.from_numpy(anchors).cuda())
        one = dev.FeatureStore(bfs)
        torch.cuda.synchronize()
        low = torch.cuda.mem_get_info()[0]
        bfs.close()
        csr.close()
        torch.cuda.synchronize()
        if i:
            one_ms.append((time.perf_counter() - t0) * 1e3)
        peak_one = max(peak_one, free0 - low)
        if i < reps:
            del one
        torch.cuda.empty_cache()
    equal = bool(torch.equal(raw_sharded.view(torch.int64), one.raw.view(torch.int64)))
    p, w = one.num_planes, one.raw.size(2)
    med = {key: statistics.median(s[key] for s in stages) for key in stages[0]}
    merge_bytes = gbytes + n * p * w * 8
    mk = statistics.median(merge_ms)
    res = {"shape": name, "num_nodes": n, "num_directed_edges": int(ei.size(1)), "anchors": k,
           "anchors_this_rank": list(gpd.shard_bounds(k, world, dist.get_rank())), "num_planes": p,
           "store_bytes": one.nbytes, "gathered_bytes": gbytes, "same_graph_on_every_rank": same_graph,
           "sharded_equals_one_gpu": equal,
           "stage_ms_median": med, "whole_call_ms": {"median": statistics.median(whole), "min": min(whole),
                                                     "max": max(whole)},
           "one_gpu_build_ms": {"median": statistics.median(one_ms), "min": min(one_ms), "max": max(one_ms)},
           "peak_device_bytes": {"sharded": peak_sharded, "one_gpu": peak_one},
           "merge": {"kernel_ms_median": mk, "bytes": merge_bytes, "gbs": merge_bytes / (mk * 1e-3) / 1e9,
                     "frac_of_copy_peak": merge_bytes / (mk * 1e-3) / 1e9 / peak}}
    del one, raw_sharded, ei
    torch.cuda.empty_cache()
    return res, equal and same_graph


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--shapes", default="flickr-shape,products-shape")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--json", default=None, help="rank 0 also writes the JSON line to this file")
    args = ap.parse_args()
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = dist.get_rank(), dist.get_world_size()
    peak = copy_peak_gbs()
    mine = {"rank": rank, "card": card_info(), "copy_peak_gbs": peak, "shapes": []}
    ok = True
    for name in args.shapes.split(","):
        res, good = run_shape(name, args.reps, peak)
        mine["shapes"].append(res)
        ok &= good
        if rank == 0:
            print(f"{name} G={world}: whole {res['whole_call_ms']['median']:.2f} ms, one-GPU build "
                  f"{res['one_gpu_build_ms']['median']:.2f} ms, stages {res['stage_ms_median']}, equal={good}",
                  file=sys.stderr, flush=True)
    every = [None] * world
    dist.all_gather_object(every, mine)
    t = torch.tensor([int(ok)], device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    if rank == 0:
        line = {"tool": "tools/fstore_shard_bench.py", "world_size": world, "reps": args.reps,
                "timing": "wall clock with a device synchronise after each stage; medians over reps after 1 warm-up",
                "equal_everywhere": bool(t.item()), "ranks": every}
        text = json.dumps(line)
        print(text, flush=True)
        if args.json:
            os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
            with open(args.json, "w") as fh:
                fh.write(text + "\n")
    dist.destroy_process_group()
    sys.exit(0 if int(t.item()) else 1)


if __name__ == "__main__":
    main()
