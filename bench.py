#!/usr/bin/env python
"""bench.py — GraphPOPE geodesic embedding generation on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload flickr-shape]
                    [--no-cpu-baseline] [--no-secondary] [--dump-outputs DIR]

A *step* is one full pass of the hot path over one synthetic graph already resident in HBM:
device CSR build (dedup) -> multi-source BFS (persistent kernel) -> fused normalise + concat
epilogue writing the float32 [N, F+K] matrix.  Metric: anchor-BFS GTEPS = K*|E'|/t with |E'| the
de-duplicated directed edge count.  At N>1 the anchors are sharded (256 per GPU, weak scaling) and
the packed results exchanged over NVLink so every rank holds the full [N, F + 256*N] matrix.

Prints ONE JSON line (rank 0).  Besides the headline (BASELINE config C2) the line carries
  * `parity_checked`: after the timed loop (untimed) the device result is compared bit for bit with the C oracle
    on sampled columns of every rank's shard, x in columns [0, F), and a checksum of the whole matrix is compared
    across ranks; any mismatch makes the run exit non-zero;
  * `roofline.stages`: csr build / MS-BFS / epilogue device times taken INSIDE the timed step (event nodes of the
    replayed CUDA graph) against their algorithmic bytes;
  * `secondary`: the other BASELINE configs — C3 (node2vec pairwise block on the tensor cores), C4 (K = 1024 fixed,
    degree / PageRank anchors, strong-scaled over the N GPUs), C5 (ogbn-products-shaped graph, K = 4096 fixed,
    strong-scaled) — each checked against its oracle, and the cold one-shot cost of the drop-in call.
`--impl reference` times the reference algorithm (utils.py:64-114: N*K networkx shortest_path calls in a process
pool) restated in oracle/ on a bounded row sample.
`--dump-outputs DIR` writes the [N, F+K] float32 matrix of the last timed step to DIR/features.npy (a fixed row sample
when the whole matrix exceeds DUMP_BYTES).  Inputs are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np

METRIC = "anchor-BFS GTEPS (K*|E|/s), geodesic GraphPOPE embedding, Flickr-shape K=256 per GPU"
UNIT = "GTEPS"
K_PER_GPU = 256
DUMP_BYTES = 60_000_000  # --dump-outputs stays below 64 MB


def dump_rows(n, cols):
    """Rows of the [n, cols] float32 matrix that --dump-outputs writes: all of them when they fit in DUMP_BYTES, else
    a fixed sample (seed 0, ascending)."""
    rows = min(n, DUMP_BYTES // (4 * max(1, cols)))
    if rows == n:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, rows, replace=False))


def dump_outputs(out_d, directory):
    import torch
    idx = dump_rows(*out_d.shape)
    if idx.size < out_d.size(0):
        out_d = out_d[torch.as_tensor(idx, device=out_d.device)]
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "features.npy"), out_d.cpu().numpy())


# --------------------------------------------------------------------------- CPU reference legs
def _t0_worker(args):
    """One pool job of utils.py:99-100: shortest_path_length over a node slice."""
    ei, n, anchors, rows = args
    from oracle import geodesic
    G = geodesic.to_digraph(ei, n)
    t = time.perf_counter()
    geodesic.t0_rows(G, anchors, rows)
    return time.perf_counter() - t, len(rows)


_PER_ROW_SECONDS = {}


def time_reference_sample(ei, n, anchors, num_workers, budget_s, probe_rows=3):
    """Time the reference algorithm (oracle T0 = utils.py:64-81 restated) on a bounded row sample.

    Rows are independent, so the rate measured on the sample is the rate of the full graph.
    Returns (seconds the full graph would take at that rate, seconds of the timed sample, rows timed).
    """
    import multiprocessing as mp
    from oracle import geodesic

    anchors = [int(a) for a in anchors]
    if "per_row" not in _PER_ROW_SECONDS:  # sizes the sample; probed once per process
        G = geodesic.to_digraph(ei, n)
        rng = np.random.default_rng(0)
        probe = rng.integers(0, n, probe_rows).tolist()
        t = time.perf_counter()
        geodesic.t0_rows(G, anchors, probe)
        _PER_ROW_SECONDS["per_row"] = max((time.perf_counter() - t) / probe_rows, 1e-6)
        del G
    per_row = _PER_ROW_SECONDS["per_row"]
    rows_total = int(max(num_workers, min(n, budget_s * num_workers / per_row)))
    stride = max(1, n // rows_total)
    rows = np.arange(0, n, stride)[:rows_total]
    chunks = [c.tolist() for c in np.array_split(rows, num_workers) if len(c)]
    ctx = mp.get_context("fork")
    with ctx.Pool(processes=len(chunks)) as pool:
        res = pool.map(_t0_worker, [(ei, n, anchors, c) for c in chunks])
    # the slowest worker's busy time bounds the pool, as in the reference (ordered job.get(), utils.py:102-104)
    busy = max(r[0] for r in res)
    timed_rows = sum(r[1] for r in res)
    full = busy * (n / max(1, max(r[1] for r in res) * len(chunks)))
    return full, busy, timed_rows


def workload_name(shape, k):
    return (f"{shape.name} synthetic graph ({shape.num_nodes} nodes, {shape.num_directed_edges} directed edges), "
            f"geodesic, stochastic sampling (seed 42), {k} anchors per GPU, F={shape.num_features}")


def headline_config(shape, world, e_unique):
    """`config` of both arms: what is computed, not how."""
    return {"workload": workload_name(shape, K_PER_GPU), "total_anchors": K_PER_GPU * world,
            "dedup_edges": int(e_unique)}


def run_reference_arm(args, shape, ei, anchors, e_unique):
    """The reference's CPU implementation of the path (oracle T0 port: the reference is Python and cannot travel to
    the GPU box) on all host threads; every step is a bounded row sample, `value` is the rate it measured."""
    cores = min(os.cpu_count() or 1, 32)
    n = shape.num_nodes
    total_budget = float(os.environ.get("GP_BENCH_REF_BUDGET_S", "150"))  # tests shrink it; the default fills ~4 minutes
    per_step = max(2.0, total_budget / max(1, args.steps + args.warmup))
    rates, secs, rows = [], [], 0
    for i in range(args.warmup + args.steps):
        full, busy, rows = time_reference_sample(ei, n, anchors, cores, per_step * 0.6)
        if i >= args.warmup:
            rates.append(K_PER_GPU * e_unique / full / 1e9)
            secs.append(busy)
    value = float(np.mean(rates))
    # one step with the reference's default pool (num_workers=6, main.py:39), same sampling
    full6, _, rows6 = time_reference_sample(ei, n, anchors, 6, per_step * 0.6)
    from oracle import cbfs
    t = time.perf_counter()
    cbfs.bfs_hops(cbfs.InCsr(ei, n), anchors[:K_PER_GPU])
    fair = time.perf_counter() - t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean(secs)) * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": headline_config(shape, 1, e_unique),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"oracle T0 (utils.py:64-81 restated: N*K nx.shortest_path, mp pool of {cores}); "
                                   f"{rows} of {n} rows per step ({100.0 * rows / n:.1f} % of the workload); value = "
                                   f"the rate of the sample, ms_per_step = the sample's own time",
                         "full_graph_seconds_at_this_rate": K_PER_GPU * e_unique / value / 1e9,
                         "num_workers_6_gteps": K_PER_GPU * e_unique / full6 / 1e9,
                         "num_workers_6_note": f"reference default pool size (main.py:39), {rows6} rows sampled",
                         "fair_cpu_gteps": K_PER_GPU * e_unique / fair / 1e9,
                         "fair_cpu_note": f"oracle C tier: K single-source BFS over reversed edges, 1 thread, the FULL "
                                          f"workload in {fair:.2f} s (same output as the reference, bit for bit)"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            p = [x.strip() for x in s.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- algorithmic bytes (DESIGN.md §4)
def bytes_bfs(n, e, k_g):
    """SURVEY §8(d): B_bfs = W*(4(N+1) + 4E + 8E + 16N) + 2*N*K_g."""
    w = -(-k_g // 64)
    return w * (4 * (n + 1) + 12 * e + 16 * n) + 2 * n * k_g


def bytes_csr(n, e_in, e_out):
    """Counting sort by row + in-row sort: edge_index (int64 pairs) read by the count and the scatter pass, the
    column array written raw and rewritten sorted, row_start / deg / rank (4 B each) and one 16-byte work-list
    descriptor per row."""
    return 2 * 16 * e_in + 2 * 4 * e_out + 12 * n + 16 * n


def bytes_epilogue(n, k_total, f):
    """SURVEY §8(d): B_epi + B_cat = 2*N*K + 4*N*K + 8*N*F."""
    return 6 * n * k_total + 8 * n * f


# --------------------------------------------------------------------------- parity
def check_device_result(out_d, x_d, ei, n, f, anchors, world, rank, dist, cols_per_rank=32):
    """Untimed.  Rank 0: sampled columns of every rank's shard bit-equal to the C oracle, x in place.  All ranks:
    a checksum of the whole [N, F+K] matrix agrees.  Returns a dict (rank 0) or raises."""
    import torch

    k_total = len(anchors)
    sums = torch.zeros(2, dtype=torch.int64, device=out_d.device)
    chunk = max(1, (64 << 20) // max(1, out_d.size(1)))  # rows per pass: keeps the int64 temporaries near 0.5 GB
    for r0 in range(0, n, chunk):
        v = out_d[r0:r0 + chunk].view(torch.int32).to(torch.int64)
        w = (torch.arange(r0, min(n, r0 + chunk), device=out_d.device, dtype=torch.int64) % 65521 + 1).unsqueeze(1)
        sums[0] += v.sum()
        sums[1] += (v * w).sum()
        del v, w
    same = True
    if world > 1:
        hi, lo = sums.clone(), sums.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        same = bool(torch.equal(hi, lo))
    info = None
    ok = same
    if rank == 0:
        from oracle import cbfs
        per = k_total // world
        rng = np.random.default_rng(7)
        cols = np.concatenate([r * per + np.sort(rng.choice(per, min(cols_per_rank, per), replace=False))
                               for r in range(world)]) if world > 1 else np.arange(k_total)
        want = cbfs.normalise(cbfs.bfs_hops(cbfs.InCsr(ei, n), np.asarray(anchors)[cols]))
        got = out_d[:, f + torch.as_tensor(cols, device=out_d.device)].cpu().numpy()
        cols_ok = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
        x_ok = bool(torch.equal(out_d[:, :f], x_d)) if f else True
        ok = ok and cols_ok and x_ok
        info = {"oracle": "oracle/bfs_oracle.c (K single-source BFS over reversed edges + IEEE 1/(d+1))",
                "columns_checked": int(cols.size), "columns_bit_equal": cols_ok, "x_columns_equal": x_ok,
                "ranks_checksum_equal": same, "checksum": [int(s) for s in sums.tolist()]}
    flag = torch.tensor([int(ok)], device=out_d.device)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    return bool(flag.item()), info


# --------------------------------------------------------------------------- secondary configs
def secondary_c3(dev, synth, peak_gbs, peaks):
    """BASELINE config C3: Flickr-shaped node2vec block, 128-d table, 256 KMeans centres, three distance functions
    with and without the per-column MinMax, on the tensor cores (gp_cdist.cu).  Checked against fp32 torch."""
    import torch
    n, k, d = 89250, 256, 128
    emb = torch.as_tensor(synth.node2vec_table(n, d, 3)).cuda()
    t0 = time.perf_counter()
    centres, inertia, iters = dev.kmeans(emb, k, n_init=1, seed=0)
    torch.cuda.synchronize()
    kmeans_s = time.perf_counter() - t0
    rows = torch.as_tensor(synth.stochastic_anchors(n, k, 42)).cuda()
    out = torch.empty(n, k, device="cuda")
    byt = 4 * (n * d + k * d + n * k)  # SURVEY §8(d): 137.2 MB
    res = {"shape": f"{n} x {k} x {d}", "anchors": "device KMeans centres (k-means++ + Lloyd, 1 init)",
           "kmeans_seconds": kmeans_s, "kmeans_iterations": int(iters), "algorithmic_bytes": byt,
           "hbm_floor_us": byt / peak_gbs / 1e3, "modes": {}}
    en = emb / emb.norm(dim=1, keepdim=True)
    ok_all = True
    for mode in ("euclidean", "distance", "similarity"):
        for mm in (False, True):
            for _ in range(3):
                dev.cdist_minmax(emb, centres, mode, mm, out=out)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                dev.cdist_minmax(emb, centres, mode, mm, out=out)
            e1.record(); torch.cuda.synchronize()
            us = e0.elapsed_time(e1) / 20 * 1e3
            # comparator (north_star): torch fp32 — non-mm cdist for euclidean, normalised matmul for cosine
            if mode == "euclidean":
                ref = torch.cdist(emb, centres, compute_mode="donot_use_mm_for_euclid_dist")
                scale = float((2 * d) ** 0.5)
            else:
                cn = centres / centres.norm(dim=1, keepdim=True)
                sim = en @ cn.t()
                ref = sim if mode == "similarity" else (1.0 - sim).clamp_(0.0, 2.0)
                scale = 1.0
            if mm:
                lo, hi = ref.min(dim=0).values, ref.max(dim=0).values
                rng_ = torch.where(hi > lo, hi - lo, torch.ones_like(hi))
                ref = (ref - lo) / rng_
                scale = 2.0  # values in [0, 1]; the division by (max - min) amplifies the absolute error
            err = (out - ref).abs()
            ok = bool((err <= 1e-4 * ref.abs() + 1e-5 * scale).all())
            ok_all &= ok
            res["modes"][f"{mode}{'+minmax' if mm else ''}"] = {
                "us": us, "frac_of_hbm_floor": (byt / peak_gbs / 1e3) / us, "gbs": byt / us / 1e3,
                "tflops_bf16x3": 2 * n * k * d * 3 * (2 if mm else 1) / us / 1e6,
                "within_1e-4_of_torch_fp32": ok, "max_abs_err": float(err.max())}
    # stochastic-row anchors (utils.py:165-167): node == its own anchor must give (near) zero distance
    dev.cdist_minmax(emb, emb[rows].contiguous(), "euclidean", False, out=out)
    res["self_distance_max"] = float(out[rows, torch.arange(k, device="cuda")].max())
    res["tensor_pipe_note"] = ("5.85 GFLOP x3 (split bf16) per pass; at D = 128 the block is HBM-bound (42.6 flop/B), so "
                               "tensor-pipe utilisation is low by construction: %.1f %% of the measured %.0f TFLOP/s "
                               "bf16 peak at the fastest mode; ncu summary under profiles/" %
                               (100 * max(m["tflops_bf16x3"] for m in res["modes"].values()) /
                                float(peaks.get("bf16_tflops", 1664.7)), float(peaks.get("bf16_tflops", 1664.7))))
    # SURVEY §8(d)(iii): the reference's scikit-learn path (pairwise + MinMaxScaler, utils.py:174-176) on the host cores
    try:
        from oracle import node2vec as onv
        emb_h, c_h = emb.cpu().numpy(), centres.cpu().numpy()
        cpu = {}
        for mode in ("euclidean", "distance"):
            t0 = time.perf_counter()
            onv.node2vec_block(emb_h, c_h, mode)
            cpu[mode + "+minmax_ms"] = (time.perf_counter() - t0) * 1e3
        res["cpu_sklearn_path"] = dict(cpu, cores=os.cpu_count(), kind="port",
                                       note="oracle restatement of sklearn pairwise + MinMaxScaler on host arrays, "
                                            "whatever threads BLAS takes; a reported baseline, not the target")
    except Exception as e:  # noqa: BLE001
        res["cpu_sklearn_path"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    res["parity_checked"] = ok_all
    return res, ok_all


def sharded_device_step(dev, gpd, peer, engine, ei_d, a_d, x_d, out_d, world):
    if world == 1:
        engine.run(ei_d, a_d, x_d, out_d)
        return None
    return peer.run(ei_d, a_d, x_d, out_d)[1]


def timed_steps(fn, barrier, dist, world, reps, flush=None):
    """Device time per call: events around each call, L2 flushed in between (untimed), max over ranks."""
    import torch
    total = 0.0
    align = torch.zeros(1, device="cuda")
    for i in range(reps):
        if flush is not None:
            flush(i)
        if world > 1:  # device-side alignment of the ranks (see align_ranks in main)
            dist.all_reduce(align)
            torch.cuda._sleep(400_000)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        total += a.elapsed_time(b)
    t = torch.tensor([total / reps], device="cuda", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def secondary_c4(dev, gpd, synth, utils, ei, ei_d, shape, world, rank, dist, barrier, flush_l2, peak_gbs):
    """BASELINE config C4: Flickr-shaped geodesic, K = 1024 FIXED (strong scaling: 1024 / N anchors per GPU), anchors
    from the degree-centrality and PageRank samplers (device), sampled inside the end-to-end region."""
    import torch
    n, f, k = shape.num_nodes, shape.num_features, 1024
    if k % (8 * world):
        return {"skipped": f"K = {k} does not split into 8-column lanes over {world} ranks"}, True
    res = {"k_total": k, "anchors_per_gpu": k // world, "scaling": "strong", "samplers": {}}
    engine = dev.GeodesicEngine(n, ei.shape[1], k // world)
    peer = gpd.PeerAssembly(engine) if world > 1 else None
    x_d = torch.randn(n, f, device="cuda", generator=torch.Generator("cuda").manual_seed(4))
    out_d = torch.empty(n, f + k, device="cuda")

    class _D:
        pass

    data = _D()
    data.num_nodes, data.edge_index = n, torch.as_tensor(ei)
    ok_all = True
    e_unique = None
    for method in ("degree_centrality", "pagerank"):
        t0 = time.perf_counter()
        anchors = np.asarray(utils.sample_anchor_nodes(data, k, method), dtype=np.int64)  # identical on every rank
        torch.cuda.synchronize()
        sample_s = time.perf_counter() - t0
        a_d = torch.as_tensor(anchors).cuda()
        barrier()  # the samplers' first call differs by seconds between ranks; the exchange waits only so long for a peer
        for _ in range(3):
            sharded_device_step(dev, gpd, peer, engine, ei_d, a_d, x_d, out_d, world)
        barrier()
        ms = timed_steps(lambda: sharded_device_step(dev, gpd, peer, engine, ei_d, a_d, x_d, out_d, world),
                         barrier, dist, world, 10, flush_l2)
        e_unique = engine.csr.info()["num_edges"]
        ok, info = check_device_result(out_d, x_d, ei, n, f, anchors, world, rank, dist, cols_per_rank=max(4, 32 // world))
        ok_all &= ok
        if rank == 0:
            from oracle import samplers
            want = (samplers.degree_centrality_anchors if method == "degree_centrality"
                    else samplers.pagerank_anchors)(ei, n, k)
            list_ok = anchors.tolist() == want
            ok_all &= list_ok
            b = bytes_csr(n, ei.shape[1], e_unique) + bytes_bfs(n, e_unique, k // world) + bytes_epilogue(n, k, f)
            res["samplers"][method] = {
                "step_ms": ms, "gteps": k * e_unique / ms / 1e6, "sampler_seconds_first_call": sample_s,
                "anchor_list_equals_oracle": list_ok, "parity": info,
                "step_frac_of_hbm": b / (ms * 1e-3) / 1e9 / peak_gbs}
    flag = torch.tensor([int(ok_all)], device="cuda")
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        barrier(); peer.close()
    res["parity_checked"] = bool(flag.item())
    return res, bool(flag.item())


def secondary_c5(dev, gpd, synth, world, rank, local_rank, dist, barrier, peak_gbs):
    """BASELINE config C5: ogbn-products-shaped power-law graph (2.45 M nodes, 123.7 M directed edges), K = 4096
    FIXED, anchor-sharded over the N GPUs (at N = 1 all 4096 anchors run on one GPU), F = 100."""
    import torch
    shape = synth.PRODUCTS_SHAPE
    n, f, k = shape.num_nodes, shape.num_features, 4096
    t0 = time.perf_counter()
    # every rank draws the same graph on its own GPU (same seed, same generator, same device type); verified below
    ei_d = synth.chung_lu_symmetric_torch(n, shape.num_directed_edges, shape.pareto_alpha, shape.seed, "cuda")
    torch.cuda.synchronize()
    gen_s = time.perf_counter() - t0
    chk = torch.stack([ei_d[0].sum(), (ei_d[0] * (ei_d[1] % 1021 + 1)).sum()])
    if world > 1:
        hi, lo = chk.clone(), chk.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX); dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        if not bool(torch.equal(hi, lo)):
            dist.broadcast(ei_d, src=0)  # fall back to rank 0's draw
    anchors = synth.stochastic_anchors(n, k, 42)
    a_d = torch.as_tensor(anchors).cuda()
    engine = dev.GeodesicEngine(n, ei_d.size(1), k // world)
    engine.bfs.set_stage_events(True)  # stage clocks (12 us of event nodes in a step of tens of milliseconds)
    peer = gpd.PeerAssembly(engine) if world > 1 else None
    x_d = torch.zeros(n, f, device="cuda")  # SURVEY §8(d): x = zeros [N, 100] for C5
    out_d = torch.empty(n, f + k, device="cuda")
    barrier()
    for _ in range(2):
        sharded_device_step(dev, gpd, peer, engine, ei_d, a_d, x_d, out_d, world)
    barrier()
    ms = timed_steps(lambda: sharded_device_step(dev, gpd, peer, engine, ei_d, a_d, x_d, out_d, world),
                     barrier, dist, world, 3)
    stage = engine.bfs.pipeline_stage_ms()
    stats = engine.bfs.stats()
    e_unique = engine.csr.info()["num_edges"]
    # parity: a few columns of every rank's shard against the C oracle (rank 0), checksum across ranks
    ei = ei_d.cpu().numpy() if rank == 0 else None
    ok, info = check_device_result(out_d, x_d, ei, n, f, anchors, world, rank, dist, cols_per_rank=max(1, 4 // world)) \
        if world > 1 else check_c5_single(out_d, x_d, ei, n, f, anchors)
    res = None
    if rank == 0:
        b = bytes_csr(n, ei_d.size(1), e_unique) + bytes_bfs(n, e_unique, k // world) + bytes_epilogue(n, k, f)
        res = {"shape": f"{n} nodes, {ei_d.size(1)} directed edges (torch Chung-Lu draw, alpha {shape.pareto_alpha}, "
                        f"seed {shape.seed}), F = {f}", "k_total": k, "anchors_per_gpu": k // world,
               "scaling": "strong", "graph_generation_seconds": gen_s, "step_ms": ms,
               "gteps": k * e_unique / ms / 1e6, "dedup_edges": int(e_unique),
               "stage_ms_rank0": {"csr_build": stage[0], "msbfs_kernel": stage[1],
                                  "exchange_and_epilogue" if world > 1 else "epilogue": stage[2]},
               "max_hops": stats["max_level"], "step_frac_of_hbm": b / (ms * 1e-3) / 1e9 / peak_gbs,
               "parity": info, "parity_checked": ok}
    if world > 1:
        barrier(); peer.close()
    return res, ok


def check_c5_single(out_d, x_d, ei, n, f, anchors):
    """N = 1: three columns of the 4096 against the C oracle (a full-oracle run takes minutes at this size)."""
    import torch
    from oracle import cbfs
    cols = np.array([0, len(anchors) // 2 + 1, len(anchors) - 1])
    want = cbfs.normalise(cbfs.bfs_hops(cbfs.InCsr(ei, n), np.asarray(anchors)[cols]))
    got = out_d[:, f + torch.as_tensor(cols, device="cuda")].cpu().numpy()
    cols_ok = bool(np.array_equal(got.view(np.uint32), want.view(np.uint32)))
    x_ok = bool(torch.equal(out_d[:, :f], x_d))
    return cols_ok and x_ok, {"oracle": "oracle/bfs_oracle.c", "columns_checked": 3, "columns_bit_equal": cols_ok,
                              "x_columns_equal": x_ok}


COLD_SCRIPT = r"""
import sys, time, json
t0 = time.perf_counter()
import numpy as np, torch
sys.path.insert(0, %(root)r)
from graphpope_b200 import synth, utils
t_import = time.perf_counter() - t0
shape = synth.SHAPES["flickr-shape"]
n, f, k = shape.num_nodes, shape.num_features, 256
ei = synth.make_graph(shape)
class D: pass
d = D(); d.num_nodes, d.edge_index, d.x = n, torch.as_tensor(ei), torch.randn(n, f)   # pageable host tensors
utils.VERBOSE = False
np.random.seed(42)
t = time.perf_counter(); out = utils.Graphpope(d, "flickr", "geodesic", "stochastic", k, None, num_workers=6)
cold = time.perf_counter() - t                     # library load + CUDA context + allocations + the call itself
warm = []
for _ in range(5):
    utils.clear_cache(); np.random.seed(42)
    t = time.perf_counter(); out2 = utils.Graphpope(d, "flickr", "geodesic", "stochastic", k, None, num_workers=6)
    warm.append(time.perf_counter() - t)
assert torch.equal(out, out2) and tuple(out.shape) == (n, f + k) and not out.is_cuda
# what a fresh pageable [N, F+K] tensor costs by itself (allocation + first touch of 270 MB: the reference's
# torch.cat pays the same), and the same call into a tensor that already exists
touch = []
for _ in range(3):
    t = time.perf_counter(); z = torch.empty(n, f + k); z.zero_(); touch.append(time.perf_counter() - t); del z
from graphpope_b200 import device as dev
reuse = torch.empty(n, f + k); reuse.zero_()
np.random.seed(42); anchors = np.random.choice(np.arange(n), k)
into = []
for _ in range(5):
    t = time.perf_counter(); dev.geodesic_embed_host(d.edge_index, n, anchors, d.x, out=reuse); into.append(time.perf_counter() - t)
assert torch.equal(reuse, out)
print(json.dumps({"import_s": t_import, "cold_ms": cold * 1e3, "warm_pageable_ms": float(np.median(warm)) * 1e3,
                  "fresh_output_tensor_first_touch_ms": float(np.median(touch)) * 1e3,
                  "warm_pageable_into_existing_tensor_ms": float(np.median(into)) * 1e3,
                  "note": "cold = first utils.Graphpope call of a fresh process on pageable tensors: library load, CUDA "
                          "context, allocations, lazy module load and the call; warm = later calls, each returning a NEW "
                          "pageable tensor (allocation + first touch of its pages included, as in the reference's torch.cat)"}))
"""


def guarded(fn, *a):
    """A secondary line that dies (out of memory on a shared box, ...) must not take the headline line with it: the
    error is reported in its place and the line is marked unchecked."""
    try:
        return fn(*a)
    except Exception as e:  # noqa: BLE001
        import traceback
        traceback.print_exc()
        return {"error": f"{type(e).__name__}: {e}"[:400], "parity_checked": False}, False


def cold_call():
    """Fresh process: the first utils.Graphpope call on PAGEABLE tensors (what main.py:94-98 does once per process)."""
    try:
        p = subprocess.run([sys.executable, "-c", COLD_SCRIPT % {"root": ROOT}], capture_output=True, text=True,
                           timeout=300)
        last = [l for l in p.stdout.strip().splitlines() if l.startswith("{")]
        if p.returncode != 0 or not last:
            return {"error": (p.stderr or p.stdout)[-300:]}
        return json.loads(last[-1])
    except Exception as e:  # noqa: BLE001
        return {"error": repr(e)}


# --------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="flickr-shape")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--secondary", default="c3,c4,c5,cold", help="comma list of secondary lines to run")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the [N, F+K] matrix of the last timed step to DIR/features.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours: the reference arm times a row sample and keeps no output")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from graphpope_b200 import synth
    shape = synth.SHAPES[args.workload]

    if args.impl == "reference":
        if rank != 0:
            return
        ei = synth.make_graph(shape)
        anchors = synth.stochastic_anchors(shape.num_nodes, K_PER_GPU, 42)
        from oracle import geodesic
        e_unique = geodesic.dedup_edges(ei, shape.num_nodes)[0].size
        run_reference_arm(args, shape, ei, anchors, e_unique)
        return

    n, f = shape.num_nodes, shape.num_features
    k_total = K_PER_GPU * world
    ei = synth.make_graph(shape)
    anchors = synth.stochastic_anchors(n, k_total, 42)  # identical on every rank (same seed)

    # ---- CPU baseline first (before CUDA is initialised: the pool forks), rank 0 at N=1 only
    cpu_baseline = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        from oracle import cbfs, geodesic
        e_unique_cpu = geodesic.dedup_edges(ei, n)[0].size
        workers = 6  # reference default, main.py:39
        full, busy, rows = time_reference_sample(ei, n, anchors[:K_PER_GPU], workers, budget_s=15.0)
        t = time.perf_counter()
        cbfs.bfs_hops(cbfs.InCsr(ei, n), anchors[:K_PER_GPU])
        fair = time.perf_counter() - t
        cpu_baseline = {
            "value": K_PER_GPU * e_unique_cpu / full / 1e9, "unit": UNIT, "cores": workers, "kind": "port",
            "sample": f"oracle T0 (utils.py:64-81 restated: N*K nx.shortest_path calls, mp pool of {workers} = reference "
                      f"default num_workers); {rows} of {n} rows timed in {busy:.1f} s; the full graph would take "
                      f"{full:.0f} s at this rate",
            "fair_cpu_gteps": K_PER_GPU * e_unique_cpu / fair / 1e9,
            "fair_cpu_note": f"oracle C tier (K single-source BFS, 1 thread, full workload) {fair:.2f} s",
            "host_cpus": os.cpu_count(),
        }

    import torch
    import torch.distributed as dist
    from graphpope_b200 import device as dev
    from graphpope_b200 import distributed as gpd
    from graphpope_b200 import utils

    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ei_d = torch.as_tensor(ei).cuda()
    a_d = torch.as_tensor(anchors).cuda()
    x_d = torch.randn(n, f, device="cuda", generator=torch.Generator("cuda").manual_seed(1))
    out_d = torch.empty(n, f + k_total, device="cuda")
    engine = dev.GeodesicEngine(n, ei.shape[1], K_PER_GPU)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    flush_r = torch.zeros(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")

    def flush_l2(i):
        """Untimed, between steps: write 256 MiB (evicts every line of the previous step from the 126 MB L2),
        then read a second 256 MiB buffer so the L2 is left full of CLEAN foreign lines — after the write alone
        it is full of dirty ones, whose write-back would be charged to the next timed step."""
        flush.fill_(float(i))
        return flush_r.sum()

    peer = gpd.PeerAssembly(engine) if world > 1 else None
    deep_flags = []

    def step():
        flag = sharded_device_step(dev, gpd, peer, engine, ei_d, a_d, x_d, out_d, world)
        if flag is not None:
            deep_flags.append(flag)

    # clocks are sampled from before the warm-up to the end of the e2e loop (the device-timed region
    # alone lasts a few milliseconds, shorter than one nvidia-smi sampling period)
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    for _ in range(args.warmup):
        step()
    barrier()
    e_unique = engine.csr.info()["num_edges"]
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stops = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    stage_ms, bfs_dev_ms = [], []
    launches0 = dev.launch_count()
    align_t = torch.zeros(1, device="cuda")

    def align_ranks():
        """Untimed alignment of the ranks on the device: a tiny all-reduce the host does not wait for ends at the same
        moment on every GPU, and a ~0.2 ms device-side spin after it gives every host time to queue the step behind
        it.  (dist.barrier() blocks the host, whose launch jitter afterwards — tens of microseconds — shows up inside
        the step as waiting for the last rank's flag; so does a host that queues its graph launch later than the
        all-reduce takes.)"""
        if world > 1:
            dist.all_reduce(align_t)
            torch.cuda._sleep(400_000)

    barrier()
    for i in range(args.steps):
        # untimed: flush the L2, then align the ranks ON THE DEVICE (align_ranks above)
        flush_l2(i)  # untimed: evict the previous step's lines from the 126 MB L2
        align_ranks()
        starts[i].record()
        step()
        stops[i].record()
        bfs_dev_ms.append(engine.bfs.kernel_device_ms())  # the kernel's own %globaltimer stamps (syncs)
    barrier()
    launches = dev.launch_count() - launches0
    if peer is not None and hasattr(peer, "trace"):
        tr = peer.trace()
        print(f"rank {rank} exchange kernel phases (us from its start): {tr}", file=sys.stderr, flush=True)
    if peer is not None and peer.trace_events and rank == 0:
        peer.trace_events = peer.trace_events[-args.steps:]
        print("peer step phases (median ms): csr+bfs+pack %.4f, flag all-reduce %.4f, peer decode %.4f"
              % tuple(peer.trace_summary()), file=sys.stderr, flush=True)
    if world > 1 and int(deep_flags[-1].item()) != 0:
        raise RuntimeError("a shard had hops > 15: the packed exchange is invalid for this graph; use "
                           "distributed.sharded_geodesic_features (all-gather path)")
    step_ms = [s.elapsed_time(e) for s, e in zip(starts, stops)]
    total_ms = float(sum(step_ms))
    stats = engine.bfs.stats()

    if world > 1:
        t = torch.tensor([total_ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    ms_per_step = total_ms / args.steps
    value = k_total * e_unique / (ms_per_step * 1e-3) / 1e9

    # ---- parity of what the timed loop produced (untimed)
    parity_ok, parity_info = check_device_result(out_d, x_d, ei, n, f, anchors, world, rank, dist)
    if args.dump_outputs and rank == 0:  # every rank holds the whole matrix (checksums compared above)
        dump_outputs(out_d, args.dump_outputs)

    # ---- stage times: a second pass over the same step with CUDA-event nodes inside the replayed graph (csr build |
    # MS-BFS kernel | epilogue).  An event-record node costs ~4 us of the step, so the timed loop above runs without
    # them (it reads the MS-BFS kernel's own device-clock stamps instead); this pass is not part of `value`.
    engine.bfs.set_stage_events(True)
    for _ in range(3):
        step()
    barrier()
    ev_pass_ms = []
    for i in range(args.steps):
        flush_l2(i)
        align_ranks()
        a_ev, b_ev = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a_ev.record(); step(); b_ev.record()
        stage_ms.append(engine.bfs.pipeline_stage_ms())
        ev_pass_ms.append(a_ev.elapsed_time(b_ev))
    barrier()
    engine.bfs.set_stage_events(False)
    stage_ok, _ = check_device_result(out_d, x_d, ei, n, f, anchors, world, rank, dist)
    parity_ok = parity_ok and stage_ok

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))

    # ---- e2e: the public host-buffer API, H2D + D2H inside the timed region
    ei_h = torch.as_tensor(ei).pin_memory()
    x_h = torch.randn(n, f, generator=torch.Generator().manual_seed(2)).pin_memory()  # identical on every rank, as data.x is
    lo, hi = gpd.shard_bounds(k_total, world, rank)
    e2e_staging = {}
    if world == 1:
        out_h = torch.empty(n, f + k_total).pin_memory()
        shared = None
    else:
        shared = gpd.SharedHostMatrix(n, f + k_total)  # one page-locked [N, F+K] matrix per node, mapped by every rank
        out_h = shared.tensor

    def e2e_step():
        if world == 1:
            dev.geodesic_embed_host(ei_h, n, anchors, x_h, out=out_h)
        else:
            gpd.sharded_embed_host_shared(engine, ei_h, anchors, x_h, shared, e2e_staging)

    for _ in range(3):
        e2e_step()
    barrier()
    e2e_steps = args.steps
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    barrier()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        t = torch.tensor([e2e_s], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = k_total * e_unique / e2e_s / 1e9
    # e2e parity: the host matrix every rank holds == [x | device result of the timed loop]
    e2e_ok = bool(torch.equal(out_h[:, f:], out_d[:, f:].cpu())) and bool(torch.equal(out_h[:, :f], x_h))
    flag = torch.tensor([int(e2e_ok)], device="cuda")
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    e2e_ok = bool(flag.item())
    clock_info = clocks.stop() if rank == 0 else None

    # ---- secondary configs (untimed for the headline; each carries its own timing and parity)
    secondary, sec_ok = {}, True
    want = set() if args.no_secondary else {s.strip() for s in args.secondary.split(",") if s.strip()}
    if "c3" in want and world == 1:
        secondary["C3_node2vec_block"], ok = guarded(secondary_c3, dev, synth, peak, peaks)
        sec_ok &= ok
    if "c4" in want:
        res, ok = guarded(secondary_c4, dev, gpd, synth, utils, ei, ei_d, shape, world, rank, dist, barrier, flush_l2, peak)
        secondary["C4_flickr_k1024_centrality_anchors"] = res
        sec_ok &= ok
    if "cold" in want and world == 1 and rank == 0:
        secondary["cold_one_shot_call"] = cold_call()
    if "c5" in want:
        del flush, flush_r, out_d, x_d
        torch.cuda.empty_cache()
        res, ok = guarded(secondary_c5, dev, gpd, synth, world, rank, local_rank, dist, barrier, peak)
        secondary["C5_products_k4096"] = res
        sec_ok &= ok

    if rank == 0:
        w_words = stats["lane_words"]
        b_bfs = bytes_bfs(n, e_unique, K_PER_GPU)
        b_csr = bytes_csr(n, ei.shape[1], e_unique)
        b_epi = bytes_epilogue(n, k_total, f)
        st = np.asarray(stage_ms)  # [steps, 3] csr, bfs kernel, epilogue — from the event pass
        csr_ms, bfs_avg_ms, epi_ms = [float(v) for v in st.mean(axis=0)]
        ev_step_ms = float(np.mean(ev_pass_ms))
        if world > 1 and not hasattr(peer, "trace"):  # pull path: the graph ends at the pack, exchange + decode follow it
            epi_ms = max(ev_step_ms - csr_ms - bfs_avg_ms, 1e-6)
        achieved = b_bfs / (bfs_avg_ms * 1e-3) / 1e9
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "msbfs_traffic.json")))
            traffic, traffic_src = tj["dram_bytes_per_launch"], "profiles/msbfs_traffic.json: " + tj.get("source", "ncu --set full capture")
        except Exception:
            pass

        def entry(ms, b):
            return {"ms": ms, "algorithmic_bytes": int(b), "achieved": b / (ms * 1e-3) / 1e9, "frac": b / (ms * 1e-3) / 1e9 / peak}

        cap = None
        if world > 1:
            # output replicated on every GPU: per-GPU epilogue bytes grow with N while csr + bfs do not
            t1 = 0.16 + bytes_epilogue(n, K_PER_GPU, f) / peak / 1e6
            tn = 0.16 + b_epi / peak / 1e6
            cap = {"weak_scaling_efficiency_cap": t1 / tn,
                   "note": "every GPU writes the whole [N, F + 256*N] matrix, so even an epilogue at the copy peak caps "
                           "v_N / (N*v_1) at (0.16 ms + B_epi(1)/peak) / (0.16 ms + B_epi(N)/peak)"}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic",
            "config": headline_config(shape, world, e_unique),
            "details": {"parallelism": f"anchor-shard x{world}",
                        "step_ms_rank0": {"min": float(np.min(step_ms)), "median": float(np.median(step_ms)),
                                          "max": float(np.max(step_ms))},
                        "l2": "between steps (untimed): 256 MiB buffer written, then a second 256 MiB buffer read, so the "
                              "L2 holds neither the previous step's lines nor dirty lines to write back",
                        "step": "csr build + ms-bfs + fused normalise/concat epilogue" +
                                (" + packed exchange over NVLink" if world > 1 else "")},
            "parity_checked": bool(parity_ok and e2e_ok and sec_ok),
            "parity": dict(parity_info or {}, e2e_host_matrix_equals_device_result=e2e_ok),
            "roofline": {"bound": "hbm", "kernel": "msbfs_kernel", "achieved": achieved, "peak": peak,
                         "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured)" if peaks else "fallback 6650",
                         "algorithmic_bytes": b_bfs, "kernel_ms": bfs_avg_ms,
                         "kernel_ms_device_clock_in_timed_loop": float(np.mean(bfs_dev_ms)),
                         "kernel_share_of_step": float(np.mean(bfs_dev_ms)) / ms_per_step,
                         "timing_note": "kernel_ms and `stages` = CUDA events recorded as nodes of the replayed graph in a "
                                        "second pass of the same step (rank 0); each event node costs ~4 us, so the timed loop "
                                        "runs without them and reads the kernel's own %globaltimer stamps (entry -> end of the "
                                        "last level; excludes the cooperative launch and the exit)",
                         "stages": {"csr_build": entry(csr_ms, b_csr), "msbfs_kernel": entry(bfs_avg_ms, b_bfs),
                                    ("exchange_and_epilogue" if world > 1 else "epilogue"): entry(epi_ms, b_epi),
                                    "step": entry(ms_per_step, b_csr + b_bfs + b_epi),
                                    "step_with_event_nodes_ms": ev_step_ms,
                                    "note": "stage times: event nodes inside the replayed CUDA graph, second pass (rank 0); "
                                            "`step` = the timed loop; bytes per DESIGN.md §4"}},
            "bfs": {"levels": stats["levels_run"], "max_level": stats["max_level"],
                    "pull_levels": stats["pull_levels"], "push_levels": stats["push_levels"],
                    "edges_examined_per_WE": stats["edges_examined"] / max(1, w_words * e_unique),
                    "grid_blocks": stats["grid_blocks"]},
            "e2e": {"value": e2e_value, "unit": UNIT, "ms": e2e_s * 1e3,
                    "h2d_bytes_per_step": int(ei_h.numel() * 8 + (hi - lo) * 8),
                    "d2h_bytes_per_step": int(n * (hi - lo) * 4) if world > 1 else int(n * k_total * 4),
                    "api": ("graphpope_b200.device.geodesic_embed_host (gp_geodesic_embed_host), pinned host buffers; x is "
                            "concatenated on the host" if world == 1 else
                            "graphpope_b200.distributed.sharded_embed_host_shared: one page-locked [N, F+K] matrix per "
                            "node in POSIX shared memory; each rank DMAs its own [N, K/G] block into it and copies N/G "
                            "rows of x; bytes are per rank")},
            "gpu_launches": int(launches),
            "clocks": clock_info,
        }
        if cap:
            line["scaling_cap"] = cap
        if secondary:
            line["secondary"] = secondary
        if cpu_baseline:
            line["cpu_baseline"] = cpu_baseline
        print(json.dumps(line), flush=True)
    ok = parity_ok and e2e_ok and sec_ok
    if world > 1:
        if shared is not None:
            shared.close()
        dist.destroy_process_group()
    if not ok:
        sys.exit(3)


if __name__ == "__main__":
    main()
