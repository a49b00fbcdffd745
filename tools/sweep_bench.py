#!/usr/bin/env python3
"""Kernel micro-benchmark: times the CN / VN sweeps of capped full-BP runs (every frame still active, so each launch
processes all frames) with the library's CUDA-event sampler and prints achieved algorithmic GB/s per sweep.

    python tools/sweep_bench.py [--n-words 8] [--graphs 4] [--iters 40] [--eps 0.48] [--traj] [--window W]
"""
import argparse
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

import fl_scaling_sc_ldpc_b200 as eng
from fl_scaling_sc_ldpc_b200 import _lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n-words", type=int, default=8)
    ap.add_argument("--graphs", type=int, default=4)
    ap.add_argument("--iters", type=int, default=40)
    ap.add_argument("--eps", type=float, default=0.48)
    ap.add_argument("--L", type=int, default=50)
    ap.add_argument("--M", type=int, default=10000)
    ap.add_argument("--traj", action="store_true")
    ap.add_argument("--reps", type=int, default=3)
    a = ap.parse_args()
    ens = eng.Ensemble(4, 8, a.L, a.M)
    F = 64 * a.n_words
    fb = eng.FrameBatch(ens, a.graphs, F, a.n_words).generate_graphs(1).generate_erasures(a.eps, 2)
    lib = _lib.lib()
    for _ in range(2):
        eng.decode_bp_full(fb, a.iters, True, trajectory=a.traj, max_rows=a.iters, collect=False)
    torch.cuda.synchronize()
    _lib.check(lib.scldpc_profile_begin(1, 4096))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(a.reps):
        res = eng.decode_bp_full(fb, a.iters, True, trajectory=a.traj, max_rows=a.iters, collect=False)
    ev1.record()
    torch.cuda.synchronize()
    cap = 4096
    ns = ctypes.c_int(0)
    idx = (ctypes.c_int * cap)(); cn = (ctypes.c_float * cap)(); vn = (ctypes.c_float * cap)()
    _lib.check(lib.scldpc_profile_end(ctypes.byref(ns), idx, cn, vn, cap))
    its = res[0][0][:, :F].cpu().numpy() if isinstance(res, tuple) else None
    cn_ms = np.array(cn[:ns.value]); vn_ms = np.array(vn[:ns.value]); it = np.array(idx[:ns.value])
    keep = it >= 2
    frames = a.graphs * F
    cn_bytes = frames * 2 * ens.E / 8
    vn_bytes = frames * (2 * ens.E + ens.n) / 8
    out = dict(n_words=a.n_words, graphs=a.graphs, frames=frames, traj=a.traj,
               min_iters=int(res[0][0][:, :F].min().item()),
               cn_us=float(np.median(cn_ms[keep]) * 1e3), vn_us=float(np.median(vn_ms[keep]) * 1e3),
               cn_GBs=float(cn_bytes / np.median(cn_ms[keep]) / 1e6), vn_GBs=float(vn_bytes / np.median(vn_ms[keep]) / 1e6),
               both_GBs=float((cn_bytes + vn_bytes) / (np.median(cn_ms[keep]) + np.median(vn_ms[keep])) / 1e6),
               wall_ms_per_iter=float(ev0.elapsed_time(ev1) / a.reps / a.iters))
    out["wall_GBs"] = float((cn_bytes + vn_bytes) / out["wall_ms_per_iter"] / 1e6)
    st = (ctypes.c_longlong * 2)()
    flags = _lib.F_TERMINATED | (_lib.F_TRAJECTORY if a.traj else 0)
    _lib.check(lib.scldpc_bp_sweep_stats(ctypes.byref(fb.dims), flags, ctypes.c_void_p(fb.workspace(flags).data_ptr()), st))
    launched = res[3]
    out["swept_frac_cn"] = st[0] / max(1, a.graphs * launched * (a.L + 3))
    out["swept_frac_vn"] = st[1] / max(1, a.graphs * launched * a.L)
    out["launched"] = launched
    print(json.dumps(out))


if __name__ == "__main__":
    main()
