#!/usr/bin/env python3
"""Generates tests/golden/full_size_golden.npz: what the reference decoders return on the full-size cases of
tests/test_full_size_ref_gpu.py.  Needs a CUDA device (the graphs and channel realisations are drawn there, as in the
test).  The decoders are the compiled reference (oracle/_ref, tests/ref_pool.py) where it is built, else the oracle port;
`source` in the file records which.

    python tests/golden/make_full_size_golden.py [OUT]
"""
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import oracle  # noqa: E402
from tests import ref_pool  # noqa: E402
from tests import test_full_size_ref_gpu as T  # noqa: E402


def _port(job):
    """one ref_pool job decoded by the oracle port, returned in ref_pool's form (rows with the iteration column)"""
    kind, dv, dc, L, defM, vn_cn, chan, prm = job
    g = oracle.Graph(vn_cn, L, defM * dc // dv, defM, dv, dc)
    ch = chan.astype(np.int32)
    if kind == "sw":
        o = oracle.decode_bp_sw(g, ch, prm["W"], prm["max_it"], prm.get("init_it", 0), 1, 1)
    else:
        o = oracle.decode_bp(g, ch, prm["max_it"], prm.get("is_term", 1), max_rows=prm["max_it"] if prm.get("want_rows") else 1)
        o["rows"] = np.column_stack([np.arange(len(o["rows"])), o["rows"]]) if prm.get("want_rows") else None
    o["erased"] = np.packbits(o["erased"])
    return o


def main(out):
    gpu, inp = T.run_gpu()
    ens, vn, DV, DC, M = inp["ens"], inp["vn"], T.DV, T.DC, T.M
    jobs, z = [], {}
    z["stream_frames"] = np.asarray(T.stream_picks(gpu["stream"]), np.int32)
    z["capstream_frames"] = np.asarray(T.CAPSTREAM_FRAMES, np.int32)
    for name, cap in (("stream", 10 ** 9), ("capstream", 175)):
        for g, f in z[name + "_frames"]:
            ch = T._frame_channel(ens, T.EPS[g], T.SEED + 1, int(g), int(f))
            jobs.append(("bp", DV, DC, 50, M // 2, vn[g], ch, dict(max_it=cap, is_term=1)))
    z["traj_cases"] = np.asarray([(cap, t, f) for cap, t, fs in T.TRAJ_RUNS for f in fs], np.int32)
    for cap, t, f in z["traj_cases"]:
        jobs.append(("bp", DV, DC, 50, M // 2, vn[2], inp["cht"][f], dict(max_it=int(cap), is_term=int(t), want_rows=True)))
    z["sw_cases"] = np.asarray([(W, f) for W, _ in T.SW_RUNS for f in (0, 127)], np.int32)
    for W, f in z["sw_cases"]:
        jobs.append(("sw", DV, DC, 100, M // 2, gpu["vnw"], inp[("chw", W)][f], dict(W=int(W), max_it=8, init_it=60)))

    if ref_pool.available("traj", DV, DC, 50, M // 2) and ref_pool.available("sw", DV, DC, 100, M // 2):
        source, res = "compiled reference (oracle/_ref)", ref_pool.run(jobs)
    else:
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
            source, res = "oracle port (oracle/scldpc_oracle.c)", list(ex.map(_port, jobs))
    ns, nc, nt = len(z["stream_frames"]), len(z["capstream_frames"]), len(z["traj_cases"])
    bp = [[int(o[k]) for k in T.KEYS] for o in res[:ns + nc + nt]]
    z["stream_expect"] = np.asarray(bp[:ns], np.int64)
    z["capstream_expect"] = np.asarray(bp[ns:ns + nc], np.int64)
    z["traj_expect"] = np.asarray(bp[ns + nc:], np.int64)
    for i, o in enumerate(res[ns + nc:ns + nc + nt]):
        z[f"traj_rows{i}"] = np.asarray(o["rows"][:, 1:4], np.int32)
        z[f"traj_erased{i}"] = o["erased"]
    sw = res[ns + nc + nt:]
    z["sw_expect"] = np.asarray([[int(o[k]) for k in T.SW_KEYS] for o in sw], np.int64)
    for i, o in enumerate(sw):
        z[f"sw_erased{i}"] = o["erased"]
    z["source"] = np.asarray(source)
    np.savez_compressed(out, **z)
    print(f"{out}: {len(jobs)} cases from the {source}, {os.path.getsize(out)} bytes")


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden", "full_size_golden.npz"))
