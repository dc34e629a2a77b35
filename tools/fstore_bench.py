"""Compact feature store against the dense [N, F+K] matrix on one GPU.

For the Flickr-shape (K = 256, F = 500) and products-shape (K = 4096, F = 100) workloads of bench.py (same synth
generators, graph seeds and anchor seed 42) it reports:
  * per shape: P, store bytes against dense bytes, the torch.cuda.mem_get_info drop that each build leaves behind
    (dense: GeodesicEngine.run's matrix; compact: FeatureStore's packed records), and the pack kernel's time;
  * per batch size B (a seeded prefix of a random permutation of the nodes: 1550 = main.py's batch size, 16384,
    65536, N): min / median / max device ms of FeatureStore.gather and of dense.index_select(0, n_id, out=...),
    the bytes each must move, GB/s and the fraction of the copy peak bench.py uses.  Every call is preceded,
    untimed, by a 256 MiB write and a 256 MiB read (as bench.py does), so the 126 MB L2 does not serve the store.
Gathered rows are compared bit for bit with index_select for every B; a mismatch exits non-zero.

    python tools/fstore_bench.py [--shapes flickr-shape,products-shape] [--reps 50] [--warmup 5] [--json PATH]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SHAPE_K = {"flickr-shape": 256, "products-shape": 4096}


def card_info() -> dict:
    info = {"torch_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                           capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"not available: {e}"
    return info


def copy_peak_gbs() -> tuple[float, str]:
    """The copy peak bench.py divides by: MEASURED_PEAKS.json hbm_gbs when present, else 6650 GB/s."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path)).get("hbm_gbs", 6650.0)), "MEASURED_PEAKS.json hbm_gbs"
    return 6650.0, "fallback 6650 (bench.py)"


def make_graph(shape):
    from graphpope_b200 import synth
    if shape.name == "products-shape":
        return synth.chung_lu_symmetric_torch(shape.num_nodes, shape.num_directed_edges, shape.pareto_alpha,
                                              shape.seed, "cuda")
    return torch.as_tensor(synth.make_graph(shape)).cuda()


def free_bytes() -> int:
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return torch.cuda.mem_get_info()[0]


def stats_ms(v):
    v = sorted(v)
    return {"min": v[0], "median": float(np.median(v)), "max": v[-1]}


def run_shape(name, reps, warmup, peak, flush_l2):
    from graphpope_b200 import _lib, synth
    from graphpope_b200 import device as dev

    shape = synth.SHAPES[name]
    n, f, k = shape.num_nodes, shape.num_features, SHAPE_K[name]
    ei_d = make_graph(shape)
    a_d = torch.as_tensor(synth.stochastic_anchors(n, k, 42)).cuda()
    x_d = torch.randn(n, f, device="cuda", generator=torch.Generator("cuda").manual_seed(1))

    # dense build: the matrix GeodesicEngine.run leaves behind (engine workspace freed)
    free0 = free_bytes()
    eng = dev.GeodesicEngine(n, ei_d.size(1), k)
    dense = eng.run(ei_d, a_d, x_d)
    max_level = eng.bfs.stats()["max_level"]
    eng.bfs.close()
    eng.csr.close()
    del eng
    dense_drop = free0 - free_bytes()

    # compact build: csr + MS-BFS + pack, workspace freed (FeatureStore.build), with the pack kernel timed in between
    free1 = free_bytes()
    csr = dev.DeviceCsr(n, ei_d.size(1)).build(ei_d)
    bfs = dev.MsBfs(csr, k).run(a_d)
    store = dev.FeatureStore(bfs, x_d)
    lib, stream = _lib.load(), dev._stream()
    pack_ms = []
    for _ in range(3):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        _lib.check(lib.gp_fstore_pack(bfs._h, dev._ptr(store.raw), store.num_planes, stream))
        e.record()
        e.synchronize()
        pack_ms.append(s.elapsed_time(e))
    bfs.close()
    csr.close()
    del bfs, csr
    compact_drop = free1 - free_bytes()
    p, w = store.num_planes, store.raw.size(2)

    res = {"shape": name, "num_nodes": n, "num_directed_edges": int(ei_d.size(1)), "anchors": k, "features": f,
           "max_hops": max_level, "num_planes": p, "words_per_plane": w,
           "store_bytes": store.nbytes, "dense_bytes": n * (f + k) * 4, "x_bytes": n * f * 4,
           "store_over_dense": store.nbytes / (n * (f + k) * 4),
           "mem_get_info_drop_bytes": {"dense_build": dense_drop, "compact_build": compact_drop},
           "pack_ms": stats_ms(pack_ms),
           "pack_ms_note": "CUDA events around gp_fstore_pack, which also syncs the stream twice (max-hop read and "
                           "the end of the pack); 3 calls",
           "batches": []}
    del ei_d
    ok = True
    perm = torch.randperm(n, generator=torch.Generator().manual_seed(0))
    for b in (1550, 16384, 65536, n):
        n_id = perm[:b].cuda()
        out_c = torch.empty(b, f + k, device="cuda")
        out_d = torch.empty(b, f + k, device="cuda")
        gather = lambda: store.gather(n_id, out=out_c)  # noqa: E731
        select = lambda: torch.index_select(dense, 0, n_id, out=out_d)  # noqa: E731
        for _ in range(warmup):
            gather()
            select()
        times = {"gather": [], "index_select": []}
        for i in range(reps):
            for key, fn in (("gather", gather), ("index_select", select)):  # alternated, L2 scrubbed before each
                flush_l2(i)
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                fn()
                e.record()
                e.synchronize()
                times[key].append(s.elapsed_time(e))
        equal = bool(torch.equal(out_c.view(torch.int32), out_d.view(torch.int32)))
        store.check()
        ok &= equal
        # algorithmic bytes: ids + x rows + packed records + output rows  /  ids + dense rows read + written
        byt = {"gather": b * (8 + 4 * f + p * w * 8 + 4 * (f + k)), "index_select": b * (8 + 8 * (f + k))}
        row = {"B": b, "bit_equal": equal}
        for key in ("gather", "index_select"):
            st = stats_ms(times[key])
            gbs = byt[key] / (st["median"] * 1e-3) / 1e9
            row[key] = {"ms": st, "bytes": byt[key], "gbs": gbs, "frac_of_copy_peak": gbs / peak}
        row["gather_over_index_select_median"] = row["gather"]["ms"]["median"] / row["index_select"]["ms"]["median"]
        res["batches"].append(row)
        print(f"{name} B={b}: gather {row['gather']['ms']['median']:.4f} ms, index_select "
              f"{row['index_select']['ms']['median']:.4f} ms, bit_equal={equal}", file=sys.stderr, flush=True)
        del out_c, out_d
    del dense, store
    return res, ok


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--shapes", default="flickr-shape,products-shape")
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--json", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if args.reps < 50:
        ap.error("--reps must be at least 50")
    from graphpope_b200 import _lib
    _lib.require_cuda()
    torch.cuda.set_device(0)
    peak, peak_source = copy_peak_gbs()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")
    flush_r = torch.zeros(256 * 1024 * 1024 // 4, dtype=torch.float32, device="cuda")

    def flush_l2(i):
        flush.fill_(float(i))
        return flush_r.sum()

    line = {"tool": "tools/fstore_bench.py", "card": card_info(), "copy_peak_gbs": peak, "peak_source": peak_source,
            "reps": args.reps, "warmup": args.warmup,
            "timing": "CUDA events around each call; 256 MiB written + 256 MiB read untimed before every call",
            "shapes": []}
    ok = True
    for name in args.shapes.split(","):
        res, good = run_shape(name, args.reps, args.warmup, peak, flush_l2)
        line["shapes"].append(res)
        ok &= good
    line["bit_equal"] = ok
    text = json.dumps(line)
    print(text, flush=True)
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as fh:
            fh.write(text + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
