#!/usr/bin/env python3
"""Error rates at several iteration caps from one decode: what the checkpointed frame stream costs.

At the benchmark geometry ((4,8) L=50, M=10000, eps 0.46/0.47/0.48/0.49, one graph each, 16384 frames per graph on 1024
lanes) three configurations are timed in one process, alternating, with CUDA events around each call:
  (a) one stream with checkpoints at the caps 175, 200, 250, 300, 350   (decode_bp_stream(..., caps=...))
  (b) one capped stream at 350                                        (decode_bp_stream(..., max_it=350))
  (c) the five capped streams one after the other
and (a)'s per-frame results are checked against (c)'s.  Lane-iterations: "useful" is the sum of the frames' iterations
(under each cap for (c)); "launched" is iterations launched x lanes x graphs, an upper bound (a graph whose stream has
ended takes no further sweeps), so launched / useful shows the idle lanes, among them the lanes paused at a checkpoint.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import fl_scaling_sc_ldpc_b200 as eng  # noqa: E402

STATS = ("residual", "blocks_err", "erasures_exp", "blocks_err_exp")


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power = q.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def timed(fn):
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0.record()
    r = fn()
    t1.record()
    torch.cuda.synchronize()
    return r, t0.elapsed_time(t1) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=10000)
    ap.add_argument("--frames", type=int, default=16384, help="frames per graph")
    ap.add_argument("--lanes", type=int, default=1024)
    ap.add_argument("--caps", default="175,200,250,300,350")
    ap.add_argument("--reps", type=int, default=2, help="timed rounds of (a), (b), (c)")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    caps = [int(c) for c in a.caps.split(",")]
    eps = [0.46, 0.47, 0.48, 0.49]
    ens = eng.Ensemble(4, 8, 50, a.M)
    fb = eng.FrameBatch(ens, len(eps), a.lanes).generate_graphs(11)
    B, G, seed = a.frames, len(eps), 12
    run_a = lambda: eng.decode_bp_stream(fb, B, eps, seed, caps=caps)
    run_b = lambda: eng.decode_bp_stream(fb, B, eps, seed, max_it=caps[-1])
    run_c = lambda: [eng.decode_bp_stream(fb, B, eps, seed, max_it=T) for T in caps]
    # warm-up of every shape the timed window uses (a short stream of each kind)
    eng.decode_bp_stream(fb, a.lanes, eps, seed, caps=caps)
    eng.decode_bp_stream(fb, a.lanes, eps, seed, max_it=caps[-1])
    torch.cuda.synchronize()
    times = {"a": [], "b": [], "c": []}
    for _ in range(a.reps):
        ra, t = timed(run_a); times["a"].append(t)
        rb, t = timed(run_b); times["b"].append(t)
        rc, t = timed(run_c); times["c"].append(t)
    # (a) against (c), frame for frame; (b) is (c)'s last stream
    same = True
    for k, (T, r) in enumerate(zip(caps, rc)):
        same &= bool((np.minimum(ra.iters, T) == r.iters).all())
        for key in STATS:
            same &= bool((getattr(ra, key)[k] == getattr(r, key)).all())
    same &= bool((rb.iters == rc[-1].iters).all())
    frames = B * G
    useful_a = int(ra.iters.astype(np.int64).sum())
    useful_b = int(rb.iters.astype(np.int64).sum())
    useful_c = sum(int(r.iters.astype(np.int64).sum()) for r in rc)
    launched = {"a": ra.iters_launched * a.lanes * G, "b": rb.iters_launched * a.lanes * G,
                "c": sum(r.iters_launched for r in rc) * a.lanes * G}
    best = {k: min(v) for k, v in times.items()}
    name, power = gpu_info()
    res = dict(
        gpu=name, power_limit=power, geometry=dict(dv=4, dc=8, L=50, M=a.M, eps=eps, frames_per_graph=B, lanes=a.lanes), caps=caps,
        seconds=times, best_seconds=best,
        frames_per_s={k: frames / v for k, v in best.items()},
        # (c) decodes every frame once per cap: its rate counts each frame once, like (a)'s
        ratio_a_over_c=best["a"] / best["c"], ratio_a_over_b=best["a"] / best["b"],
        lane_iterations=dict(useful=dict(a=useful_a, b=useful_b, c=useful_c), launched_upper_bound=launched,
                             launched_over_useful={k: launched[k] / u for k, u in (("a", useful_a), ("b", useful_b), ("c", useful_c))}),
        a_equals_c=same, when=time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime()))
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt + "\n")
    return 0 if same else 1


if __name__ == "__main__":
    sys.exit(main())
