"""Per-level phase timing of the persistent MS-BFS kernel (GP_BFS_TRACE=1): where the critical path is."""
import os, sys, ctypes
os.environ["GP_BFS_TRACE"] = "1"
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from graphpope_b200 import device as dev, synth, _lib

shape = synth.SHAPES[sys.argv[1] if len(sys.argv) > 1 else "flickr-shape"]
K = int(sys.argv[2]) if len(sys.argv) > 2 else 256
n = shape.num_nodes
ei = synth.make_graph(shape); anchors = synth.stochastic_anchors(n, K, 42)
ei_d = torch.as_tensor(ei).cuda(); a_d = torch.as_tensor(anchors).cuda()
eng = dev.GeodesicEngine(n, ei.shape[1], K); eng.bfs.set_stage_events(True)
out = torch.empty(n, K, device="cuda")
fused = os.environ.get("GP_TRACE_FUSED", "1") != "0"  # trace the fused pipeline (csr build + MS-BFS), else the MS-BFS alone
run = (lambda: eng.run(ei_d, a_d, None, out)) if fused else (lambda: eng.bfs.run(a_d))
eng.csr.build(ei_d)
for _ in range(3): run()
torch.cuda.synchronize()
ms = []
for _ in range(10):
    run(); ms.append(eng.bfs.kernel_ms())
print("env", {k: v for k, v in os.environ.items() if k.startswith("GP_")}, "kernel ms: min %.4f med %.4f" % (min(ms), np.median(ms)), eng.bfs.stats())
lib = _lib.load()
cap = 32 * 160 * 4 * 32 * 4
buf = np.zeros(cap, dtype=np.uint64); lv = ctypes.c_int32(); wp = ctypes.c_int32()
_lib.check(lib.gp_msbfs_trace(eng.bfs._h, buf.ctypes.data, cap, ctypes.byref(lv), ctypes.byref(wp)))
L, W = lv.value, wp.value
full = buf[: 32 * W * 4].reshape(32, W, 4).astype(np.int64)
t = full[:L]
if L < 32:
    pro = full[31]  # prologue stamps: kernel entry, seeds + class tables, tile cache, first grid barrier
    d = pro - pro[:, :1]
    print("prologue cycles (median over warps): seeds+tables %d, tile cache %d, first barrier %d; entry -> level 1 sweep start %d" % (
        np.median(d[:, 1]), np.median(d[:, 2] - d[:, 1]), np.median(d[:, 3] - d[:, 2]), np.median(t[0, :, 0] - pro[:, 0])))
    last = t[L - 1]
    print("kernel entry -> last sweep end (max over warps, same-SM clocks): %d cycles" % int((last[:, 3] - pro[:, 0]).max()))
wpc = W // eng.bfs.stats()['grid_blocks']  # warps per CTA
print("levels", L, "warps", W)
print("lvl | sweep cycles: max over warps | p50 | p90 | min | argmax warp")
for l in range(L):
    d = t[l]
    tot = d[:, 3] - d[:, 0]
    print("%3d | %7d | %7d | %7d | %7d | warp %d (cta %d)" % (l + 1, tot.max(), np.median(tot), np.percentile(tot, 90), tot.min(), tot.argmax(), tot.argmax() // wpc))
for l in range(L - 1):
    end = t[l, :, 3].reshape(-1, wpc).max(axis=1); start = t[l + 1, :, 0].reshape(-1, wpc).min(axis=1)
    w = start - end
    print("barrier after lvl %d: min wait %d  median %d  max %d cycles" % (l + 1, w.min(), np.median(w), w.max()))
