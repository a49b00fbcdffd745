#!/usr/bin/env python3
"""simulate_sc_ldpc (ber_sim) frames/s on the synchronous path against frame streams with stopping-set records.

At (4,8) L=50 M=10000, terminated and bounded, eps 0.46 / 0.47 / 0.48 / 0.49, --frames frames per eps with no early stop
(max_fuckups out of reach), four variants are timed, each call between device synchronisations:
  (a) synchronous, 128 frames per graph (the default)      (b) synchronous, 1024 frames per graph
  (c) frame streams, 1024 frames per graph                 (d) frame streams, 16384 frames per graph on 1024 lanes
plus (b), (c) and (d) once for an unbounded, non-terminated code (the unscanned-head variant of the sweep).  (b) and (c)
decode the same channel realisations: the tool checks that their 13-tuples are equal and, outside the timed calls, that
their per-frame records are equal.  The GPU name and power limit are read in the same run (nvidia-smi --query-gpu).
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
from fl_scaling_sc_ldpc_b200 import peeling_decoding as pdx  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True, timeout=60)
    name, power = (q.stdout.strip().split(", ") + ["unknown", "unknown"])[:2]
    return name, power


def run(e, L, M, term, bounded, n, fpg, gpb, seed, force_sync=False):
    """one timed simulate_sc_ldpc call; force_sync: the synchronous path even at >= 1024 frames per graph"""
    factory = None
    if force_sync:
        def factory(ens, G, f, gid0):                   # what the synchronous default draws
            fb = eng.FrameBatch(ens, G, f).generate_graphs(seed, first_graph_id=gid0)
            return fb.generate_erasures(e, seed + 1, first_graph_id=gid0)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = pdx.simulate_sc_ldpc(e, 4, 8, L, M, term, False, bounded, False, n, 10 ** 9, [], seed=seed, frames_per_graph=fpg,
                               graphs_per_batch=gpb, progress=False, _batch_factory=factory)
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def records(e, L_user, M, term, bounded, n, fpg, gpb, seed, stream):
    """per-frame records of all frames, drawn as simulate_sc_ldpc draws them (untimed)"""
    head, head_sched = (0, 0) if bounded else (20, 10)
    tail = 0 if term else 20
    L = L_user + head + tail
    ens = eng.Ensemble(4, 8, L, M)
    num_positions = L + 3 if term else L
    counted = pdx.counted_positions(4, L, num_positions, head, tail)
    unscanned = head_sched * ens.cns_pos
    out = []
    for gid0 in range(0, n // fpg, gpb):
        G = min(gpb, n // fpg - gid0)
        if stream:
            fb = eng.FrameBatch(ens, G, 1024).generate_graphs(seed, first_graph_id=gid0)
            r = eng.decode_bp_stream(fb, fpg, e, seed + 1, first_graph_id=gid0, is_term=term, stopping_sets=counted,
                                     unscanned_head_cns=unscanned)
            out.append(r.records.reshape(-1, 4))
        else:
            fb = eng.FrameBatch(ens, G, fpg).generate_graphs(seed, first_graph_id=gid0).generate_erasures(e, seed + 1, first_graph_id=gid0)
            r = eng.decode_bp_full(fb, eng.UNLIMITED, is_term=term, unscanned_head_cns=unscanned)
            out.append(pdx.stopping_set_records(fb, r.erased_words, counted)[:, :fpg].reshape(-1, 4))
        del fb
    return np.concatenate(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--M", type=int, default=10000)
    ap.add_argument("--L", type=int, default=50)
    ap.add_argument("--frames", type=int, default=16384, help="frames per eps (a multiple of 16384)")
    ap.add_argument("--eps", default="0.46,0.47,0.48,0.49")
    ap.add_argument("--head-eps", type=float, default=0.40, help="eps of the unbounded, non-terminated case")
    ap.add_argument("--seed", type=int, default=2024)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    name, power = gpu_info()
    n = a.frames
    variants = {"a_sync_128": (128, 8, True), "b_sync_1024": (1024, 8, True), "c_stream_1024": (1024, 8, False),
                "d_stream_16384": (16384, 1, False)}
    # warm-up: every path once at a small size (module loading, first-launch costs)
    for fpg, gpb, sync in variants.values():
        run(0.47, 12, 64, True, True, 2 * min(fpg, 1024), min(fpg, 1024), 2, 7, force_sync=sync)
    rows = []
    cases = [(float(e), True, True) for e in a.eps.split(",")] + [(a.head_eps, False, False)]
    for e, term, bounded in cases:
        row = {"eps": e, "terminated": term, "bounded": bounded, "frames": n}
        outs = {}
        for key, (fpg, gpb, sync) in variants.items():
            if not bounded and key == "a_sync_128":
                continue
            out, t = run(e, a.L, a.M, term, bounded, n, fpg, gpb, a.seed, force_sync=sync)
            outs[key] = out
            row[key] = {"seconds": round(t, 3), "frames_per_s": round(n / t, 1), "FER": out[0], "FER_exp": out[1]}
            print(e, term, bounded, key, row[key], flush=True)
        same = all((np.asarray(outs["b_sync_1024"][i]) == np.asarray(outs["c_stream_1024"][i])).all() for i in range(13))
        rb = records(e, a.L, a.M, term, bounded, n, 1024, 8, a.seed, stream=False)
        rc = records(e, a.L, a.M, term, bounded, n, 1024, 8, a.seed, stream=True)
        row["b_c_13_tuple_equal"] = bool(same)
        row["b_c_records_equal"] = bool(rb.shape == rc.shape and (rb == rc).all())
        row["c_over_b"] = round(row["b_sync_1024"]["seconds"] / row["c_stream_1024"]["seconds"], 3)
        print(e, "b == c:", row["b_c_13_tuple_equal"], row["b_c_records_equal"], "speed-up c/b", row["c_over_b"], flush=True)
        assert row["b_c_13_tuple_equal"] and row["b_c_records_equal"], row
        rows.append(row)
    res = {"gpu": name, "power_limit": power, "code": f"(4,8) L={a.L} M={a.M}", "rows": rows,
           "note": "frames/s of one simulate_sc_ldpc call per variant and eps, host clock between device synchronisations, "
                   "no early stop; graph generation is inside the timed call on every path"}
    print(json.dumps(res))
    if a.out:
        with open(a.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
