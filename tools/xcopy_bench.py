"""Bulk-copy-engine x copy (gp_xcopy.cu, gp_concat_x) against torch's strided copy_ at the Flickr shape."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from ctypes import c_void_p
from graphpope_b200 import synth, _lib
lib = _lib.load()
sh = synth.SHAPES["flickr-shape"]; n, f, k = sh.num_nodes, sh.num_features, 256
x = torch.randn(n, f, device="cuda"); out = torch.empty(n, f + k, device="cuda")
flush = torch.empty(64 * 1024 * 1024, device="cuda")
def timed(fn, reps=20):
    ms = []
    for i in range(reps):
        flush.fill_(float(i)); s = flush[:1024].sum()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize(); ms.append(a.elapsed_time(b))
    return float(np.median(ms)), float(np.min(ms))
st = lambda: c_void_p(torch.cuda.current_stream().cuda_stream)
cp = lambda: _lib.check(lib.gp_concat_x(c_void_p(x.data_ptr()), n, f, f, c_void_p(out.data_ptr()), f + k, st()))
for _ in range(3): cp()
med, mn = timed(cp)
print(f"gp_concat_x {med*1e3:.1f} us median ({mn*1e3:.1f} min) = {8*n*f/med/1e6:.0f} GB/s", flush=True)
med, mn = timed(lambda: out[:, :f].copy_(x))
print(f"torch strided copy_ {med*1e3:.1f} us = {8*n*f/med/1e6:.0f} GB/s", flush=True)
