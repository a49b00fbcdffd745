#!/usr/bin/env python3
"""Time series of one graph's frame stream (eps = 0.49, 16384 frames on 1024 lanes): duration of the sampled iteration launches in
buckets of the iteration index -- shows what the tail of the stream (no frames left to hand out) costs."""
import argparse, ctypes, json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import fl_scaling_sc_ldpc_b200 as eng
from fl_scaling_sc_ldpc_b200 import _lib

ap = argparse.ArgumentParser()
ap.add_argument("--eps", type=float, default=0.49)
ap.add_argument("--n-words", type=int, default=16)
ap.add_argument("--frames", type=int, default=16384)
ap.add_argument("--every", type=int, default=3)
ap.add_argument("--buckets", type=int, default=40)
a = ap.parse_args()
ens = eng.Ensemble(4, 8, 50, 10000)
lanes = 64 * a.n_words
fb = eng.FrameBatch(ens, 1, lanes, a.n_words).generate_graphs(11)
lib = _lib.lib()
eng.decode_bp_stream(fb, lanes, a.eps, 12, collect=False); torch.cuda.synchronize()
t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
t0.record(); r = eng.decode_bp_stream(fb, a.frames, a.eps, 12); t1.record(); torch.cuda.synchronize()
wall_plain = t0.elapsed_time(t1)
_lib.check(lib.scldpc_profile_begin(a.every, 8000))
t0.record(); r = eng.decode_bp_stream(fb, a.frames, a.eps, 12); t1.record(); torch.cuda.synchronize()
cap = 8000; ns = ctypes.c_int(0); idx = (ctypes.c_int * cap)(); cn = (ctypes.c_float * cap)(); vn = (ctypes.c_float * cap)()
_lib.check(lib.scldpc_profile_end(ctypes.byref(ns), idx, cn, vn, cap))
n = ns.value
idx = np.array(idx[:n]); us = np.array(cn[:n]) * 1e3
fi = int(r.iters.astype(np.int64).sum())
print(json.dumps(dict(eps=a.eps, frames=a.frames, launched=r.iters_launched, wall_ms_unsampled=wall_plain, wall_ms_sampled=t0.elapsed_time(t1),
                      sum_sampled_kernel_ms_scaled=float(us.sum() * a.every / 1e3), lane_util=fi / (r.iters_launched * lanes),
                      mean_iters=fi / a.frames)))
step = max(1, r.iters_launched // a.buckets)
for lo in range(0, r.iters_launched, step):
    m = (idx >= lo) & (idx < lo + step)
    if m.any():
        print(f"iter {lo:6d}-{lo + step:6d}  launches sampled {m.sum():5d}  avg {us[m].mean():7.1f} us  p50 {np.median(us[m]):7.1f} us  share of kernel time {us[m].sum() / us.sum():.3f}")
