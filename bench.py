#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path: full BP over the BEC, (4,8) SC-LDPC, L=50, M=10000.

    python bench.py --gpus N --steps K --warmup W            our arm (one rank per GPU under torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...   the reference's CPU decoder on the host cores
    python bench.py ... --dump-outputs DIR                    also writes the per-frame results of the last timed step (the
                                                              inputs are a function of the arguments: two builds compare
                                                              output for output)

Headline (BASELINE config 2).  A *step* draws 4 NEW graph realisations (one per eps of the 0.46..0.49 sweep) on the device
-- scldpc_graph_generate + scldpc_graph_build_tables run INSIDE the timed region -- and decodes --frames-per-graph
(default 16384) fresh channel realisations on each with full BP, unlimited iterations, until every frame has stalled or
finished.  1024 bit-sliced lanes per graph; a lane whose frame has stopped is re-armed with the graph's next channel
realisation (scldpc_bp_stream), so a graph is reused for frames_per_graph frames (the reference draws a graph per frame,
BP_FULL.c:2122; the reuse is stated in `config` and the workload "bp_full_fpg1024" reports the same step at 1024 frames
per graph).  Graph ids are global and never repeat: every step, warm-up included, decodes new realisations.
Throughput counts USEFUL work only: edge-updates = sum over frames of (iterations that frame executed) * 2E, the same
formula as for the CPU (SURVEY.md section 8d); iterations a finished frame rides along for do not count.

value    : the step above, everything on the device; --pipeline batches (default 2) are in flight at a time, each on its own
           host thread and CUDA stream, so the tail of one batch's frame streams runs behind the next batch (`sequential` in the
           line: the same steps one batch after the other).
e2e      : the same step through the host-buffer C-ABI call scldpc_stream_host: graph tables start in pinned HOST memory
           (a different set every step), per-frame results end in host memory; H2D / D2H inside the timed region.
roofline : one flooding iteration of the stream decoder (ns_iter_kernel, bp_node_kernels.cu): algorithmic bytes
           B_alg = (4E+n)/8 per useful frame-iteration (the message formulation's figure, SURVEY 8d) over the CUDA-event
           time of sampled launches (in the sequential segment, where a launch's elapsed time is its own), against
           MEASURED_PEAKS.json's HBM copy bandwidth; ncu's DRAM
           bytes and the node-state minimum are reported beside it.
workloads: (N = 1 only) the other BASELINE configs, each timed on the device with its own roofline and CPU baseline:
           turnover at 1024 frames per graph, message-passing sweeps, peeling trajectories (config 1), capped BP with
           trajectory rows (config 3), sliding window L=100 (config 4).
cpu_baseline : the unmodified reference decodeBP (oracle/_ref, compiled from /root/reference) on the host cores.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

DV, DC, L, M = 4, 8, 50, 10000
EPS_SWEEP = [0.46, 0.47, 0.48, 0.49]
N_WORDS = 16
E_EDGES = L * M * DV
N_VNS = L * M
N_CNS = (L + DV - 1) * (M * DV // DC)
B_ALG = (4 * E_EDGES + N_VNS) / 8.0          # bytes per frame-iteration, message formulation (SURVEY 8d)
FRAMES_PER_STREAM = 16384
CAP_LO = 2   # reference arm: iterations of the shorter of the two capped runs
METRIC = "edge-updates/s (frames/s alongside), (4,8) SC-LDPC L=50 M=10000 BEC BP"


def workload_name(fpg: int) -> str:
    return (f"full BP unlimited iterations, (4,8) SC-LDPC terminated L=50 M=10000, BEC eps sweep {{0.46,0.47,0.48,0.49}}: "
            f"4 new graphs x {fpg} frames per graph per step")


def make_config(args) -> dict:
    """The `config` object of the JSON line -- the same function (hence the same object) for both arms."""
    stream_mode = args.mode == "stream"
    lanes = 64 * N_WORDS
    B = args.frames_per_graph if stream_mode else lanes
    G = len(EPS_SWEEP) * args.graphs_per_eps
    messages = os.environ.get("SCLDPC_STREAM_NODE" if stream_mode else "SCLDPC_FULL_NODE", "1") == "0"
    # decoder state per batch: two planes of n x lanes bits, index tables, resolution lists, or the two message arrays
    n_bits = L * M * lanes * G
    state_mb = round(((2 * n_bits / 8) + (8 * E_EDGES + 4 * N_CNS * DC) * G * (0 if messages else 1) + (4 * E_EDGES * lanes / 8 * G if messages else 0)) / 2 ** 20)
    return {"workload": workload_name(B), "frames_per_graph": B, "graphs_per_step_per_gpu": G,
            "frames_per_step_per_gpu": G * B, "lanes_per_graph": lanes, "n_words": N_WORDS, "mode": args.mode,
            "sweeps": "message passing" if messages else "node-state",
            "graph_turnover": "new graphs every step, generated and indexed on the device inside the timed region; no "
                              "(graph, frame) realisation is decoded twice",
            "l2": f"inputs larger than L2 (126 MB): about {state_mb} MB of decoder state per batch, rewritten every step",
            "batches_in_flight": (max(1, getattr(args, "pipeline", 1)) if stream_mode else 1),
            "seed": args.seed}


# ------------------------------------------------------------------------------------------------------------------
# reference arm: the reference's own decoders on the host cores
# ------------------------------------------------------------------------------------------------------------------
def _ref_worker(args):
    """One frame on one core: generate_code + channel_doped, then decodeBP twice on the same frame, capped at CAP_LO
    and at CAP_LO+cap flooding iterations.  The difference of the two times is the cost of `cap` iterations of the
    reference's sweeps over the full-size frame; the common part (message initialisation) is subtracted out.  The
    post-decoding expurgation scan -- quadratic in the erasures a capped run leaves behind, negligible for a
    converged frame -- is skipped by passing decodeBP's L argument (used only as that scan's range) as 0.  Uses BP_TRAJ.c's
    decodeBP (same loops as BP_FULL.c's plus one fprintf per iteration) so that the number of executed iterations is known."""
    seed, eps, cap = args
    from oracle import ref_driver as rd
    r = rd.get("traj", DV, DC, L, M * DV // DC)
    r.srandom(seed)
    r.reset_perm()
    r.generate_code()
    r.channel_doped(eps)
    t0 = time.perf_counter()
    a = r.decode_bp(CAP_LO, 1, exp_positions=0)
    t1 = time.perf_counter()
    b = r.decode_bp(CAP_LO + cap, 1, exp_positions=0)
    t2 = time.perf_counter()
    return len(b["rows"]) - len(a["rows"]), (t2 - t1) - (t1 - t0)


def _port_worker(args):
    """Fallback when oracle/_ref is absent: the oracle port (same algorithm, table-driven reverse-edge lookup), timed like
    _ref_worker, expurgation scan skipped too."""
    seed, eps, cap = args
    import oracle
    oracle.srandom(seed)
    g, _ = oracle.generate_code(L, M, M * DV // DC, DV, DC)
    ch = oracle.channel_doped(g.n, eps, M)
    t0 = time.perf_counter()
    a = oracle.decode_bp(g, ch, CAP_LO, 1, max_rows=1, exp_positions=0)
    t1 = time.perf_counter()
    b = oracle.decode_bp(g, ch, CAP_LO + cap, 1, max_rows=1, exp_positions=0)
    t2 = time.perf_counter()
    return b["iters"] - a["iters"], (t2 - t1) - (t1 - t0)


def _ref_window_worker(args):
    """decodeBP_SW of the unmodified BP_SW.c (square window) on one full-size frame of config 4; eps low enough for the
    window decoder to succeed, so the expurgation scan has nothing to do.  Returns (edge updates, seconds)."""
    seed, eps, W, cap, init = args
    from oracle import ref_driver as rd
    Lw = 100
    r = rd.get("sw", DV, DC, Lw, M * DV // DC)
    r.srandom(seed)
    r.reset_perm()
    r.generate_code()
    r.channel_doped(eps)
    t0 = time.perf_counter()
    r.decode_bp_sw(W, cap, init)
    dt = time.perf_counter() - t0
    # executed iterations are not returned by the reference: count the work of a run that uses every allowed iteration,
    # which is an UPPER bound of what it executed (favours the CPU)
    its = init + (Lw - 1) * cap
    return its * 2 * W * M * DV, dt


def _peel_port_worker(args):
    """config 1 on one core: the oracle port of simulate_peeling_decoder_ldpc's frame loop (PD.py:740-785)"""
    seed, Mp, nfr = args
    import numpy as np
    import oracle
    l, r, Lp, e = 4, 8, 50, 0.48
    cns = Mp * l // r
    total_size = cns * Lp
    steps = int(Mp * Lp * (e + 0.1))
    oracle.srandom(seed)
    g, _ = oracle.generate_code(Lp, Mp, cns, l, r)
    rng = np.random.default_rng(seed)
    t = 0.0
    for _ in range(nfr):
        er = (rng.random(Lp * Mp) <= e).astype(np.uint8)
        picks = rng.integers(0, 2 ** 32, steps, dtype=np.uint32)
        t0 = time.perf_counter()
        oracle.peel_trajectory(g.vn_cn, er, total_size, g.nk, steps, picks)
        t += time.perf_counter() - t0
    return nfr * steps, t


def _preload_reference_libraries():
    """dlopen the compiled reference in THIS process before the workers fork, so the process that prints the line is the
    one that has oracle/_ref/*.so mapped (the driver records which shared objects a bench process loaded)."""
    from oracle import ref_driver as rd
    loaded = []
    for variant, Lr in (("traj", L), ("sw", 100)):
        if rd.available(variant, DV, DC, Lr, M * DV // DC):
            try:
                rd.get(variant, DV, DC, Lr, M * DV // DC)
                loaded.append(os.path.basename(rd.build_ref.so_name(variant, DV, DC, Lr, M * DV // DC)))
            except Exception:
                pass
    return loaded


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import multiprocessing as mp
    from oracle import ref_driver as rd
    cores = os.cpu_count() or 1
    loaded = _preload_reference_libraries()
    have_ref = rd.available("traj", DV, DC, L, M * DV // DC)
    worker, kind = (_ref_worker, "reference") if have_ref else (_port_worker, "port")
    cap = args.sample_iters
    ctx = mp.get_context("fork")
    per_step = []
    side = {}
    with ctx.Pool(cores) as pool:
        for s in range(args.warmup + args.steps):
            jobs = [(1000003 * (s + 1) + i, EPS_SWEEP[i % len(EPS_SWEEP)], cap) for i in range(cores)]
            t0 = time.perf_counter()
            res = pool.map(worker, jobs)
            wall = time.perf_counter() - t0
            decode_wall = max(dt for _, dt in res)
            if s >= args.warmup:
                per_step.append((sum(it for it, _ in res), decode_wall, wall))
        if args.side_baselines:
            # bounded samples for the side workloads of the default run (reported inside their workload entries)
            if rd.available("sw", DV, DC, 100, M * DV // DC):
                res = pool.map(_ref_window_worker, [(77 + i, 0.40, 5, 8, 60) for i in range(cores)])
                side["window_W5"] = {"value": sum(w for w, _ in res) / max(dt for _, dt in res), "unit": "edge-updates/s (upper bound)",
                                     "cores": cores, "kind": "reference",
                                     "sample": f"{cores} processes x 1 frame, unmodified decodeBP_SW (BP_SW.c:628), L=100 M=10000 W=5, 8 iterations "
                                               "per window / 60 for the first, eps=0.40; work counted as if every allowed iteration ran",
                                     "frames_per_s": cores / max(dt for _, dt in res)}
            for Mp, nfr in ((1000, 8), (10000, 1)):
                res = pool.map(_peel_port_worker, [(5 + i, Mp, nfr) for i in range(cores)])
                wall = max(dt for _, dt in res)
                side[f"peeling_M{Mp}"] = {"value": sum(s_ for s_, _ in res) / wall, "unit": "peel-steps/s", "cores": cores, "kind": "port",
                                          "frames_per_s": cores * nfr / wall,
                                          "sample": f"{cores} processes x {nfr} frame(s), oracle port (C) of simulate_peeling_decoder_ldpc's frame loop "
                                                    f"(PD.py:740-785), L=50 M={Mp} eps=0.48 non-terminated; the reference itself is Python: "
                                                    "1.37 s/frame at M=1000 on one core (SURVEY section 6), ~58-72 s/frame at M=10000 (NB:705, NB:825)"}
    iters = sum(p[0] for p in per_step)
    t = sum(p[1] for p in per_step)
    eu = iters * 2.0 * E_EDGES / t
    sample = (f"{cores} processes x 1 full-size frame per step; per frame the unmodified decodeBP runs capped at {CAP_LO} and at "
              f"{CAP_LO}+{cap} flooding iterations and the time difference is charged to the {cap} extra iterations "
              f"(every iteration of the reference sweeps all nodes, so cost per iteration is constant; graph/channel "
              f"generation is not timed and the expurgation scan is skipped via decodeBP's L argument)")
    line = {
        "impl": "reference", "metric": METRIC, "value": eu, "unit": "edge-updates/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / max(1, len(per_step)),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32 (0/1 messages)",
        "data": "synthetic", "config": make_config(args),
        "frame_iterations_per_s": iters / t, "frames_per_s_at_348_iterations": iters / t / 348.0,
        "reference_libraries_loaded": loaded,
        "cpu_baseline": {"value": eu, "unit": "edge-updates/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": eu, "unit": "edge-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    if side:
        line["side_baselines"] = side
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.path = tempfile.mktemp(suffix=".clocks.csv")
        self.proc = None
        self.t_begin = self.t_end = None
        # Started BEFORE the warm-up steps (nvidia-smi takes a few hundred ms to initialise NVML, during which host-blocking
        # CUDA calls stall); mark() brackets the timed region and only its samples are reported.  One sample per second: every NVML query takes a driver lock that host-blocking CUDA calls of the timed region
        # (the table builder's error-flag read-back) queue behind -- at 10 Hz that cost 50 ms per generated graph
        period = os.environ.get("SCLDPC_BENCH_CLOCK_MS", "1000")
        if period == "0":
            return
        try:
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", period,
                                          "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def mark(self, begin: bool):
        import datetime
        if begin:
            self.t_begin = datetime.datetime.now()
        else:
            self.t_end = datetime.datetime.now()

    def stop(self) -> dict:
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.f.close()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in open(self.path):
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 9:
                continue
            if self.t_begin is not None and self.t_end is not None:
                try:
                    ts = datetime.datetime.strptime(p[0], "%Y/%m/%d %H:%M:%S.%f")
                    if not (self.t_begin <= ts <= self.t_end + datetime.timedelta(seconds=1)):
                        continue
                except ValueError:
                    pass
            try:
                sm.append(float(p[1])); mx.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        try:
            os.unlink(self.path)
        except OSError:
            pass
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=max(mx), samples=len(sm))
        out["reasons"] = sorted(reasons)
        return out


def _peaks():
    try:
        pk = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pk = {}
    if "hbm_gbs" in pk:
        return float(pk["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback 6650 GB/s (B200_PROFILING.md)"


def _traffic():
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        return {}


class SweepProfile:
    """CUDA-event samples of the sweeps of every `every`-th iteration (scldpc_profile_begin / _end)."""

    def __init__(self, lib, check, every=13, cap=16384):
        self.lib, self.check, self.cap = lib, check, cap
        check(lib.scldpc_profile_begin(every, cap))

    def end(self):
        import numpy as np
        ns = ctypes.c_int(0)
        it = (ctypes.c_int * self.cap)()
        a = (ctypes.c_float * self.cap)()
        b = (ctypes.c_float * self.cap)()
        self.check(self.lib.scldpc_profile_end(ctypes.byref(ns), it, a, b, self.cap))
        n = ns.value
        return np.asarray(a[:n], dtype=np.float64), np.asarray(b[:n], dtype=np.float64)


# ------------------------------------------------------------------------------------------------------------------
# side workloads (N = 1): the other BASELINE configs, device-timed
# ------------------------------------------------------------------------------------------------------------------
def side_workloads(args, dev, side_cpu):
    import numpy as np
    import torch

    import fl_scaling_sc_ldpc_b200 as eng
    from fl_scaling_sc_ldpc_b200 import _lib
    from fl_scaling_sc_ldpc_b200 import peeling_decoding as pdx

    lib = _lib.lib()
    peak, peak_src = _peaks()
    tj = _traffic()
    out = {}
    want = set(args.workloads.split(",")) if args.workloads not in ("all", "") else None

    def timed(fn, steps, warm=1):
        for i in range(warm):
            fn(-1 - i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        lib.scldpc_launch_count(1)
        e0.record()
        acc = [fn(i) for i in range(steps)]
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e-3, acc, int(lib.scldpc_launch_count(1))

    ens = eng.Ensemble(DV, DC, L, M)
    eps4 = EPS_SWEEP

    # ---- turnover: a new graph for every 1024 frames, generation inside the timed region
    if want is None or "bp_full_fpg1024" in want:
        cfgs = {}
        for nw, G in ((16, 4), (4, 16)):
            lanes = 64 * nw
            fb = eng.FrameBatch(ens, G, lanes, nw, device=dev)
            eps = [e for e in eps4 for _ in range(G // 4)]
            tg = []

            def step(i, fb=fb, eps=eps, G=G, tg=tg):
                gid = (1 << 20) + (i + 8) * G
                g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                g0.record()
                fb.generate_graphs(seed=args.seed, first_graph_id=gid)
                g1.record()
                res, _ = eng.decode_bp_stream(fb, 1024, eps, args.seed + 1, first_graph_id=gid, collect=False)
                tg.append((g0, g1))
                return res
            steps = 8 if nw == 16 else 2
            dt, acc, launches = timed(step, steps)
            its = sum(int(r[0].sum().item()) for r in acc)
            nfail = sum(int((r[1] > 0).sum().item()) for r in acc)
            frames = steps * G * 1024
            g_ms = sum(a.elapsed_time(b) for a, b in tg[1:]) / (steps * G)      # tg[0] is the warm-up step
            cfgs[f"n_words={nw}"] = {"value": its * 2.0 * E_EDGES / dt, "unit": "edge-updates/s", "frames_per_s": frames / dt,
                                     "graphs_per_step": G, "lanes_per_graph": lanes, "frames_per_graph": 1024, "steps": steps,
                                     "ms_per_step": 1e3 * dt / steps, "ms_per_generated_graph": g_ms,
                                     "graph_generation_share": g_ms * G * steps / (1e3 * dt),
                                     "frame_error_rate": nfail / frames, "gpu_launches": launches}
            del fb, acc
            torch.cuda.empty_cache()
        # the one-frame-per-lane layout with two batches in flight (as in the headline): all of a 1024-frame stream is tail, so
        # the next batch's graphs fill the machine while the stalled frames of this one finish
        import threading
        Pp, G, nw, steps = 2, 4, 16, 8
        fbs = [eng.FrameBatch(ens, G, 64 * nw, nw, device=dev) for _ in range(Pp)]
        sts = [torch.cuda.Stream(device=dev) for _ in range(Pp)]
        accs, nl, errs = [[] for _ in range(Pp)], [0] * Pp, []

        def pstep(i, t):
            gid = (2 << 20) + (i + 8) * G
            fbs[t].generate_graphs(seed=args.seed, first_graph_id=gid)
            res, _ = eng.decode_bp_stream(fbs[t], 1024, eps4, args.seed + 1, first_graph_id=gid, collect=False)
            return res

        def pworker(t, first, count, keep):
            try:
                torch.cuda.set_device(dev)
                with torch.cuda.stream(sts[t]):
                    lib.scldpc_launch_count(1)
                    for i in range(first + t, first + count, Pp):
                        r = pstep(i, t)
                        if keep:
                            accs[t].append(r)
                    sts[t].synchronize()
                    nl[t] = int(lib.scldpc_launch_count(1))
            except Exception as e:  # pragma: no cover
                errs.append(e)

        def prun(first, count, keep):
            th = [threading.Thread(target=pworker, args=(t, first, count, keep)) for t in range(Pp)]
            for x in th:
                x.start()
            for x in th:
                x.join()
            if errs:
                raise errs[0]

        prun(-Pp, Pp, False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        prun(0, steps, True)
        torch.cuda.synchronize()
        e1.record()
        torch.cuda.synchronize()
        dt = e0.elapsed_time(e1) * 1e-3
        rs = [r for a_ in accs for r in a_]
        its = sum(int(r[0].sum().item()) for r in rs)
        nfail = sum(int((r[1] > 0).sum().item()) for r in rs)
        frames = steps * G * 1024
        cfgs["n_words=16, two batches in flight"] = {"value": its * 2.0 * E_EDGES / dt, "unit": "edge-updates/s", "frames_per_s": frames / dt,
                                                    "graphs_per_step": G, "lanes_per_graph": 64 * nw, "frames_per_graph": 1024, "steps": steps,
                                                    "ms_per_step": 1e3 * dt / steps, "frame_error_rate": nfail / frames, "gpu_launches": sum(nl)}
        del fbs, accs, rs
        torch.cuda.empty_cache()
        best = max(cfgs, key=lambda k: cfgs[k]["value"])
        out["bp_full_fpg1024"] = dict(cfgs[best], layout=best, layouts=cfgs,
                                      note="scldpc_graph_generate + scldpc_graph_build_tables + fresh frame ids inside the timed region; every "
                                           "graph decodes exactly 1024 frames (the reference draws a graph per frame, BP_FULL.c:2117-2143); "
                                           "n_words=16: one frame per lane, n_words=4: 256 lanes per graph recycled four times")

    # ---- message-passing sweeps (the implementation of record): the formulation that really moves B_alg through HBM
    if want is None or "bp_full_messages" in want:
        fb = eng.FrameBatch(ens, 4, 1024, 16, device=dev)
        fb.generate_graphs(seed=args.seed, first_graph_id=3 << 20)
        Bm = 4096

        def step(i):
            res, launched = eng.decode_bp_stream(fb, Bm, eps4, args.seed + 1, first_graph_id=(3 << 20) + 4 * (i + 2), collect=False, messages=True)
            return int(res[0].sum().item()), int(launched)
        step(-1)
        prof = SweepProfile(lib, _lib.check)
        dt, acc, launches = timed(step, 2, warm=0)
        cn_ms, vn_ms = prof.end()
        its = sum(a for a, _ in acc)
        fi_per_launch = its / max(1, sum(b for _, b in acc))
        cn_b, vn_b = fi_per_launch * 2 * E_EDGES / 8.0, fi_per_launch * (2 * E_EDGES + N_VNS) / 8.0
        ach = (cn_b + vn_b) / ((cn_ms.mean() + vn_ms.mean()) * 1e-3) / 1e9
        out["bp_full_messages"] = {
            "value": its * 2.0 * E_EDGES / dt, "unit": "edge-updates/s", "frames_per_s": 2 * 4 * Bm / dt, "frames_per_graph": Bm,
            "ms_per_step": 1e3 * dt / 2, "gpu_launches": launches,
            "roofline": {"bound": "hbm", "kernel": "bp_cn_wave_kernel<8,false> + bp_vn_stream_kernel<4> (one flooding iteration)",
                         "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                         "traffic": (tj.get("vn_sweep_dram_bytes_per_launch", 0) + tj.get("cn_sweep_dram_bytes_per_launch", 0)) or None,
                         "avg_launch_ms": [float(cn_ms.mean()), float(vn_ms.mean())], "launches_sampled": int(len(cn_ms)),
                         "frame_iterations_per_launch": fi_per_launch,
                         "cn_sweep": {"achieved": cn_b / (cn_ms.mean() * 1e-3) / 1e9, "frac": cn_b / (cn_ms.mean() * 1e-3) / 1e9 / peak},
                         "vn_sweep": {"achieved": vn_b / (vn_ms.mean() * 1e-3) / 1e9, "frac": vn_b / (vn_ms.mean() * 1e-3) / 1e9 / peak},
                         "algorithmic_bytes": "(4E+n)/8 B per useful frame-iteration: 2E/8 CN sweep + (2E+n)/8 VN sweep"}}
        del fb
        torch.cuda.empty_cache()

    # ---- config 3: iteration-limited BP with per-iteration trajectory rows
    if want is None or "bp_capped_175_traj" in want:
        cap = 175
        fb = eng.FrameBatch(ens, 4, 1024, 16, device=dev)
        fb.generate_graphs(seed=args.seed, first_graph_id=5 << 20)

        def step(i):
            fb.generate_erasures(eps4, args.seed + 1, first_graph_id=(5 << 20) + 4 * (i + 2))
            res, erased, rows, launched = eng.decode_bp_full(fb, cap, True, trajectory=True, max_rows=cap, collect=False)
            return int(res[0].sum().item()), int(launched), int(rows[:, :, :, 1].sum().item())
        step(-1)
        prof = SweepProfile(lib, _lib.check, every=7)
        dt, acc, launches = timed(step, 2, warm=0)
        cn_ms, vn_ms = prof.end()
        its = sum(a[0] for a in acc)
        fi_per_launch = its / max(1, sum(a[1] for a in acc))
        ach = fi_per_launch * B_ALG / ((cn_ms.mean() + vn_ms.mean()) * 1e-3) / 1e9
        out["bp_capped_175_traj"] = {
            "value": its * 2.0 * E_EDGES / dt, "unit": "edge-updates/s", "frames_per_s": 2 * 4 * 1024 / dt, "ms_per_step": 1e3 * dt / 2,
            "cap": cap, "trajectory_rows_per_step": 4 * 1024 * cap, "gpu_launches": launches,
            "note": "channel generation, decode with (deg_1_iter, dVNs, first erased position) rows for every iteration, 4 graphs x 1024 frames",
            "sweeps": "message passing" if os.environ.get("SCLDPC_FULL_NODE", "1") == "0" else "node-state",
            "roofline": {"bound": "hbm", "kernel": ("bp_cn_wave_kernel<8,true> + bp_vn_wave_kernel<4,true>" if os.environ.get("SCLDPC_FULL_NODE", "1") == "0"
                                                   else "bpw_iter_kernel<4,8,false,true>") + " (one flooding iteration with the trajectory counters)",
                         "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src, "traffic": None,
                         "avg_launch_ms": [float(cn_ms.mean()), float(vn_ms.mean())], "launches_sampled": int(len(cn_ms)),
                         "frame_iterations_per_launch": fi_per_launch, "algorithmic_bytes": "(4E+n)/8 B per useful frame-iteration"}}
        del fb
        torch.cuda.empty_cache()

    # ---- config 4: sliding window, L = 100, non-terminated (derived mode)
    if want is None or "window_L100" in want:
        ensw = eng.Ensemble(DV, DC, 100, M)
        GW = 8                                                   # W = 3 sweeps 3 CN positions per iteration: 4 graphs do not fill the GPU
        fb = eng.FrameBatch(ensw, GW, 1024, 16, device=dev)
        fb.generate_graphs(seed=args.seed, first_graph_id=7 << 20)
        wl = {}
        for W, e in ((3, 0.30), (5, 0.40), (10, 0.45)):
            def step(i, W=W, e=e):
                fb.generate_erasures(e, args.seed + 1, first_graph_id=(7 << 20) + GW * (i + 2))
                res, erased, rows, _ = eng.decode_bp_window(fb, W, 8, 60, square=True, is_term=False, collect=False)
                return res
            step(-1)
            prof = SweepProfile(lib, _lib.check, every=11)
            dt, acc, launches = timed(step, 2, warm=0)
            cn_ms, vn_ms = prof.end()
            # useful work: the per-lane edge-update counters of a collecting call on the last step's realisations
            r = eng.decode_bp_window(fb, W, 8, 60, square=True, is_term=False)
            work = 2 * r.edge_updates
            ach = work * (B_ALG / (2 * E_EDGES)) / dt / 1e9
            wl[f"W={W}"] = {"value": work / dt, "unit": "edge-updates/s", "frames_per_s": 2 * GW * 1024 / dt, "ms_per_step": 1e3 * dt / 2,
                            "eps": e, "frame_error_rate": float((r.residual > 0).mean()),
                            "undecoded_vn_fraction": float(r.residual.mean()) / (100 * M),     # non-terminated: the last positions stay erased
                            "gpu_launches": launches,
                            "roofline": {"bound": "hbm", "kernel": "bpw_cn_copy_kernel<4,8,false> + bpw_vn_copy_kernel (window iterations)",
                                         "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "peak_source": peak_src,
                                         "traffic": (tj.get("window_node", {}) or {}).get(f"W{W}_dram_bytes_per_launch"),
                                         "avg_launch_ms": [float(cn_ms.mean()), float(vn_ms.mean())] if len(cn_ms) else None,
                                         "launches_sampled": int(len(cn_ms)),
                                         "algorithmic_bytes": "0.2656 B per useful edge update (= (4E+n)/8 per frame-iteration of the window's "
                                                              "edges, message formulation); the node-state sweeps move less, so frac can exceed 1"}}
        out["window_L100"] = {"config": "(4,8) SC-LDPC non-terminated (derived mode) L=100 M=10000, square window, 8 iterations per window, "
                                        f"60 for the first; {GW} graphs x 1024 frames per step, channel generation inside the timed region",
                              "windows": wl, "cpu_baseline": (side_cpu or {}).get("window_W5")}
        del fb
        torch.cuda.empty_cache()

    # ---- config 1: peeling trajectories
    if want is None or "peeling" in want:
        for Mp, G, F in ((1000, 16, 1024), (10000, 8, 1024)):
            l, r, Lp, e = 4, 8, 50, 0.48
            ensp = eng.Ensemble(l, r, Lp, Mp)
            cns, num_positions, total_size, steps = pdx._peel_geometry(e, l, r, Lp, Mp, False)
            fb = eng.FrameBatch(ensp, G, F, device=dev)

            def step(i, fb=fb, ensp=ensp, total_size=total_size, steps=steps, G=G, F=F):
                gid = (9 << 20) + (i + 2) * G
                fb.generate_graphs(args.seed, first_graph_id=gid)
                fb.generate_erasures(e, args.seed + 1, first_graph_id=gid)
                r1, rec, ner = pdx.peel_batch(ensp, fb, total_size, steps, args.seed + 2, gid * F)
                return int(rec.sum().item())
            dt, acc, launches = timed(step, 2)
            frames = 2 * G * F
            psteps = frames * steps
            out[f"peeling_M{Mp}"] = {"value": psteps / dt, "unit": "peel-steps/s", "frames_per_s": frames / dt, "ms_per_step": 1e3 * dt / 2,
                                     "config": f"peeling decoding trajectories, (4,8) SC-LDPC L=50 M={Mp} non-terminated eps=0.48, "
                                               f"{G} new graphs x {F} frames per step, r1 int32[{steps + 1}] per frame materialised in HBM",
                                     "recovered_vns_per_frame": sum(acc) / frames, "gpu_launches": launches,
                                     "roofline": {"bound": "hbm", "kernel": "peel_trajectory_kernel (one warp per frame; latency-bound chain of dependent steps)",
                                                  "achieved": psteps * 36.0 / dt / 1e9, "peak": peak, "unit": "GB/s", "frac": psteps * 36.0 / dt / 1e9 / peak,
                                                  "peak_source": peak_src, "traffic": None,
                                                  "algorithmic_bytes": "36 B per peel step (16 B adjacency + 4 x 4 B degree updates + 4 B r1), SURVEY 8d"},
                                     "cpu_baseline": (side_cpu or {}).get(f"peeling_M{Mp}")}
            del fb
            torch.cuda.empty_cache()
    return out


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    cpu_baseline = side_cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # timed before CUDA is initialised in this process (the workers fork)
        try:
            cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "2", "--warmup", "0",
                   "--sample-iters", str(args.sample_iters)]
            if args.workloads != "none":
                cmd.append("--side-baselines")
            p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
            ref_line = json.loads(p.stdout.strip().splitlines()[-1])
            cpu_baseline = ref_line["cpu_baseline"]
            side_cpu = ref_line.get("side_baselines")
        except Exception as e:  # pragma: no cover
            cpu_baseline = {"value": None, "unit": "edge-updates/s", "cores": os.cpu_count(), "kind": "reference",
                            "sample": f"failed: {e!r}"}

    import numpy as np
    import torch
    import torch.distributed as dist

    import fl_scaling_sc_ldpc_b200 as eng
    from fl_scaling_sc_ldpc_b200 import _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = _lib.lib()
    ens = eng.Ensemble(DV, DC, L, M)
    stream_mode = args.mode == "stream"
    lanes = 64 * N_WORDS                                         # bit-sliced lanes per graph
    B = args.frames_per_graph if stream_mode else lanes         # frames decoded per graph and step
    G = len(EPS_SWEEP) * args.graphs_per_eps
    eps = [e for e in EPS_SWEEP for _ in range(args.graphs_per_eps)]
    eps_arr = np.asarray(eps, np.float64)
    messages = os.environ.get("SCLDPC_STREAM_NODE" if stream_mode else "SCLDPC_FULL_NODE", "1") == "0"
    sflag = _lib.F_MESSAGES if messages else 0

    # graph ids are global and never reused: step s of rank r decodes graphs [(s*world + r)*G, +G) -- warm-up steps first --
    # so the realisations (and therefore the results) do not depend on how many GPUs share the job
    def gid_of(step_index):
        return (step_index * world + rank) * G

    # Batches in flight: P host threads, each with its own CUDA stream, device buffers and scldpc_bp_stream calls, take the steps
    # in turn -- the tail of one batch's frame streams (no frames left to hand out: ~1500 short launches) runs behind the next
    # batch instead of in front of it.  Same work and same realisations as one batch after the other (`sequential` in the line).
    import threading
    P = max(1, args.pipeline) if stream_mode else 1
    fbs = [eng.FrameBatch(ens, G, lanes, N_WORDS, device=dev) for _ in range(P)]
    fb = fbs[0]
    cuda_streams = [torch.cuda.Stream(device=dev) for _ in range(P)]
    counters_t = [torch.zeros(4, dtype=torch.int64, device=dev) for _ in range(P)]   # frame-iterations, frames, frame errors, bit errors
    iters_launched = [0]                                       # iterations launched by this rank in the timed region
    graph_events = []
    lock = threading.Lock()
    last_timed = args.warmup + args.steps - 1
    last_res = []                                              # per-frame results of the last timed step (--dump-outputs)

    def step(s, acc=True, t=0):
        fbt = fbs[t]
        gid = gid_of(s)
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        fbt.generate_graphs(seed=args.seed, first_graph_id=gid)        # scldpc_graph_generate + scldpc_graph_build_tables
        g1.record()
        if stream_mode:
            res, launched = eng.decode_bp_stream(fbt, B, eps, args.seed + 1, first_graph_id=gid, harvest_every=args.harvest_every, collect=False)
            it, resid = res[0].to(torch.int64), res[1].to(torch.int64)
        else:
            fbt.generate_erasures(eps, seed=args.seed + 1, first_graph_id=gid)
            res, erased, rows, launched = eng.decode_bp_full(fbt, eng.UNLIMITED, True, collect=False)
            it, resid = res[0, :, :lanes].to(torch.int64), res[1, :, :lanes].to(torch.int64)
        if s == last_timed:
            last_res.append(res[:5])                           # a fresh tensor per call: nothing overwrites it later
        if acc:
            with lock:
                graph_events.append((g0, g1))
                iters_launched[0] += int(launched)
            counters_t[t].add_(torch.stack([it.sum(), torch.tensor(it.numel(), device=dev), (resid > 0).sum(), resid.sum()]))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(first, count, acc, pipes, sample_every=0):
        """steps first .. first+count-1 with `pipes` batches in flight; returns (device ms, launches, sampled sweep times)"""
        out = {"launches": 0, "prof": (np.zeros(0), np.zeros(0)), "err": None}
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

        def worker(t):
            try:
                torch.cuda.set_device(local_rank)
                with torch.cuda.stream(cuda_streams[t]):
                    lib.scldpc_launch_count(1)                 # the launch counter and the sampler are per host thread
                    prof = SweepProfile(lib, _lib.check, every=sample_every) if (sample_every and t == 0) else None
                    for i in range(t, count, pipes):
                        step(first + i, acc, t)
                    cuda_streams[t].synchronize()
                    n = int(lib.scldpc_launch_count(1))
                    pr = prof.end() if prof is not None else None
                with lock:
                    out["launches"] += n
                    if pr is not None:
                        out["prof"] = pr
            except Exception as e:  # pragma: no cover
                out["err"] = e

        barrier()
        ev0.record()
        if pipes == 1:
            lib.scldpc_launch_count(1)
            prof = SweepProfile(lib, _lib.check, every=sample_every) if sample_every else None
            for i in range(count):
                step(first + i, acc, 0)
            ev1.record()
            torch.cuda.synchronize()
            out["launches"] = int(lib.scldpc_launch_count(1))
            if prof is not None:
                out["prof"] = prof.end()
        else:
            th = [threading.Thread(target=worker, args=(t,)) for t in range(pipes)]
            for x in th:
                x.start()
            for x in th:
                x.join()
            if out["err"] is not None:
                raise out["err"]
            torch.cuda.synchronize()
            ev1.record()
            torch.cuda.synchronize()
        return ev0.elapsed_time(ev1), out["launches"], out["prof"]

    clocks = ClockSampler(local_rank)
    run_steps(0, args.warmup, False, P)
    barrier()

    # ---- timed region: K steps ------------------------------------------------------------------------------------
    barrier()
    clocks.mark(True)
    # sampling every 29th iteration: co-prime with the harvest periods in use; a sampled launch is not a programmatic dependent
    ms_local, launches, (cn_ms, vn_ms) = run_steps(args.warmup, args.steps, True, P, sample_every=29 if P == 1 else 0)
    barrier()
    clocks.mark(False)
    clk = clocks.stop()
    graph_ms = sum(a.elapsed_time(b) for a, b in graph_events)
    counters = torch.stack(counters_t).sum(0)

    local_frame_iters = int(counters[0].item())
    # The same steps one batch after the other (a few of them): the comparison figure for the batches in flight, and the segment
    # in which the iteration launches are sampled for the roofline -- with two batches in flight the kernels of the two streams
    # interleave, and the elapsed time of a launch is not its own.
    sequential = None
    roof_fi, roof_il = local_frame_iters, iters_launched[0]
    if P > 1:
        n_seq = min(args.steps, 4)
        il0 = iters_launched[0]
        seq_ms, _, (cn_ms, vn_ms) = run_steps(args.warmup + 2 * args.steps + 4, n_seq, True, 1, sample_every=29)
        seq_fi = int(torch.stack(counters_t).sum(0)[0].item()) - local_frame_iters
        roof_fi, roof_il = seq_fi, iters_launched[0] - il0
        sq = torch.tensor([seq_ms, float(seq_fi)], dtype=torch.float64, device=dev)
        if world > 1:
            mx = sq[:1].clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = sq[1:].clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
            sq = torch.cat([mx, sm])
        sequential = {"value": float(sq[1].item()) * 2.0 * E_EDGES / (float(sq[0].item()) * 1e-3), "unit": "edge-updates/s", "steps": n_seq,
                      "what": "the same step, one batch after the other on one stream (no batches in flight); the roofline's launch "
                              "durations are sampled here"}
    tmax = torch.tensor([ms_local], dtype=torch.float64, device=dev)
    tot = counters.clone()
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)      # the only collective of the job: final counters over NVLink
    ms = float(tmax.item())
    frame_iters, frames, ferr, berr = (int(x) for x in tot.tolist())
    value = frame_iters * 2.0 * E_EDGES / (ms * 1e-3)

    # ---- roofline of the dominant kernel ---------------------------------------------------------------------------
    roof = kernels = None
    if rank == 0 and len(cn_ms) > 0:
        peak, peak_src = _peaks()
        tj = _traffic()
        n_s = len(cn_ms)
        cn_avg, vn_avg = float(cn_ms.mean()) * 1e-3, float(vn_ms.mean()) * 1e-3
        fi_per_launch = roof_fi / max(1, roof_il)
        pct = lambda a, q: float(np.percentile(a, q))
        if not messages:
            # Node-state sweeps.  SURVEY 8(d): the denominator of record stays the message formulation's B_alg = (4E+n)/8 B per
            # frame-iteration; the DRAM bytes ncu measured and the node-state minimum (2n+nk)/8 are reported next to it, so a
            # fraction above 1 is explained, not hidden.
            if stream_mode:
                kname, tn = "ns_iter_kernel<4,8,false>", tj.get("node_state_r2", {})
                kwhat = "one flooding iteration = one launch: replay of the previous iteration's resolution lists + CN sweep + lane retirement"
            else:
                kname, tn = "bpw_iter_kernel<4,8,false,false>", {}
                kwhat = "one flooding iteration"
            it_t = cn_avg + vn_avg
            ach = fi_per_launch * B_ALG / it_t / 1e9
            traffic = tn.get("iteration_dram_bytes_per_launch")
            roof = {"bound": "hbm", "kernel": kname, "kernel_does": kwhat, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                    "traffic": traffic, "traffic_note": tn.get("note"), "peak_source": peak_src, "launches_sampled": n_s,
                    "sampled_in": "the timed region" if P == 1 else "the sequential segment that follows the timed region (see `sequential`)",
                    "avg_launch_ms": 1e3 * it_t, "p10_p50_p90_ms": [pct(cn_ms + vn_ms, 10), pct(cn_ms + vn_ms, 50), pct(cn_ms + vn_ms, 90)],
                    "frame_iterations_per_launch": fi_per_launch,
                    "algorithmic_bytes": "(4E+n)/8 B = 1.0625 MB per useful frame-iteration (message formulation, SURVEY 8d: the denominator of record)",
                    "node_state_min_bytes_per_launch": fi_per_launch * (2 * N_VNS + N_CNS) / 8.0,
                    "dram_frac_of_peak_one_graph": tn.get("dram_frac_of_peak"),
                    "explanation": "the node-state sweep keeps 1 bit per VN and frame instead of 2 bits per edge, and its gathers are served "
                                   "by L2 (a band of dv positions); HBM traffic per iteration is a fraction of B_alg, so frac > 1 is expected. "
                                   "The kernel is bound by L2 latency and instruction issue (profiles/README.md)",
                    "l2": {"bytes_per_launch": tn.get("l2_read_bytes_per_launch"), "note": tn.get("l2_note")}}
            kernels = {kname: {"avg_launch_ms": 1e3 * it_t, "share_of_iteration": 1.0 if stream_mode else None,
                               "dram_bytes_per_launch": traffic}}
        else:
            vn_b = fi_per_launch * (2 * E_EDGES + N_VNS) / 8.0
            cn_b = fi_per_launch * (2 * E_EDGES) / 8.0
            ach = vn_b / vn_avg / 1e9
            roof = {"bound": "hbm", "kernel": "bp_vn_stream_kernel<4>" if stream_mode else "bp_vn_wave_kernel<4,false>", "achieved": ach,
                    "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": tj.get("vn_sweep_dram_bytes_per_launch"), "peak_source": peak_src,
                    "launches_sampled": n_s, "avg_launch_ms": 1e3 * vn_avg, "frame_iterations_per_launch": fi_per_launch,
                    "algorithmic_bytes": "(2E+n)/8 B per useful frame-iteration (reads E c2v bits + n channel bits, writes E v2c bits)"}
            kernels = {"bp_cn_wave_kernel<8,false>": {"achieved": cn_b / cn_avg / 1e9, "frac": cn_b / cn_avg / 1e9 / peak, "unit": "GB/s",
                                                      "avg_launch_ms": 1e3 * cn_avg}}

    # ---- e2e: host buffers through the C ABI ---------------------------------------------------------------------
    # graph tables of every e2e step are drawn beforehand (on the device, copied to pinned host memory: untimed) -- each
    # step uploads a set it has not seen, decodes fresh frame ids and downloads the per-frame results
    dims = fb.dims
    nw_e2e = min(2, args.warmup)
    n_e2e = args.steps + nw_e2e
    e2e_base = args.warmup + args.steps
    h_vn = []
    for j in range(n_e2e):
        fb.generate_graphs(seed=args.seed, first_graph_id=gid_of(e2e_base + j))
        h_vn.append(fb.vn_cn.cpu().pin_memory())
    if stream_mode:
        outs_t = [[torch.zeros((G, B), dtype=torch.int32).pin_memory() for _ in range(5)] for _ in range(P)]
        outs = outs_t[0]
        cfgs = [_lib.StreamCfg(B, args.harvest_every, _lib.F_TERMINATED | sflag, 0, 0, eps_arr.ctypes.data_as(ctypes.c_void_p).value, None, None, None,
                               args.seed + 1, gid_of(e2e_base + j), 0) for j in range(n_e2e)]
        h2d = int(h_vn[0].numel() * 4)
        d2h = int(5 * G * B * 4)
        api = "scldpc_stream_host (graph tables in pinned host memory, a new set every step; channel realisations drawn on the device)"

        def e2e_step(j, t=0):
            _lib.check(lib.scldpc_stream_host(ctypes.byref(dims), ctypes.c_void_p(h_vn[j].data_ptr()), ctypes.byref(cfgs[j]),
                                              *[ctypes.c_void_p(o.data_ptr()) for o in outs_t[t]], None))
            return int(outs_t[t][0].sum().item())
    else:
        h_ch = []
        for j in range(n_e2e):
            fb.generate_erasures(eps, seed=args.seed + 1, first_graph_id=gid_of(e2e_base + j))
            h_ch.append(fb.chan.cpu().pin_memory())
        outs = [torch.zeros((G, lanes), dtype=torch.int32).pin_memory() for _ in range(5)]
        flags = _lib.F_TERMINATED | _lib.F_CHAN_PACKED | sflag
        h2d = int(h_vn[0].numel() * 4 + h_ch[0].numel() * 8)
        d2h = int(6 * G * lanes * 4)
        api = "scldpc_decode_host (graph tables + bit-sliced channel words in pinned host memory)"

        def e2e_step(j, t=0):
            _lib.check(lib.scldpc_decode_host(ctypes.byref(dims), ctypes.c_void_p(h_vn[j].data_ptr()),
                                              ctypes.c_void_p(h_ch[j].data_ptr()), 0, 0, 0, flags,
                                              *[ctypes.c_void_p(o.data_ptr()) for o in outs], None, None, None, 0))
            return int(outs[0].sum().item())

    # warm-up and timed calls of a batch slot run on the same host thread: the library gives every calling thread its own stream
    # (and the memory pool hands a thread's freed buffers back to it without a detour)
    e_parts = [0] * P
    gate0, gate1 = threading.Barrier(P + 1), threading.Barrier(P + 1)

    e_err = []

    def e2e_worker(t):
        try:
            torch.cuda.set_device(local_rank)
            for j in range(t, max(nw_e2e, P if nw_e2e else 0), P):
                e2e_step(j % max(1, nw_e2e), t)      # untimed
            gate0.wait()
            gate1.wait()
            for j in range(t, args.steps, P):
                e_parts[t] += e2e_step(nw_e2e + j, t)    # the call returns after its D2H copy has completed
        except threading.BrokenBarrierError:         # another slot failed
            pass
        except Exception as e:  # pragma: no cover
            e_err.append(e)
            gate0.abort()
            gate1.abort()

    th = [threading.Thread(target=e2e_worker, args=(t,)) for t in range(P)]
    for x in th:
        x.start()
    try:
        gate0.wait()                                 # every slot has warmed up
        barrier()
        t0 = time.perf_counter()
        gate1.wait()
    except threading.BrokenBarrierError:
        t0 = time.perf_counter()
    for x in th:
        x.join()
    if e_err:
        raise e_err[0]
    e_iters = sum(e_parts)
    torch.cuda.synchronize()
    e_dt = time.perf_counter() - t0
    et = torch.tensor([e_dt], dtype=torch.float64, device=dev)
    ei = torch.tensor([e_iters], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(et, op=dist.ReduceOp.MAX)
        dist.all_reduce(ei, op=dist.ReduceOp.SUM)
    e2e = {"value": float(ei.item()) * 2.0 * E_EDGES / float(et.item()), "unit": "edge-updates/s",
           "frames_per_s": world * args.steps * G * B / float(et.item()),
           "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "api": api}
    need = lib.scldpc_bp_stream_workspace_bytes(ctypes.byref(dims), sflag) if stream_mode else fb.workspace(_lib.F_TERMINATED | sflag).numel()
    del fb, fbs, h_vn
    torch.cuda.empty_cache()

    workloads = None
    if rank == 0 and world == 1 and args.workloads != "none":
        try:
            workloads = side_workloads(args, dev, side_cpu)
        except Exception as e:  # pragma: no cover  (a side workload must never take the headline line down)
            workloads = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "edge-updates/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64 (64 bit-sliced frames per word)", "data": "synthetic",
            "config": make_config(args),
            "frames_per_s": frames / (ms * 1e-3),
            "frame_iterations_per_s": frame_iters / (ms * 1e-3),
            "mean_iterations_per_frame": frame_iters / max(1, frames),
            "frame_error_rate": ferr / max(1, frames), "bit_error_rate": berr / max(1, frames) / N_VNS,
            "graph_generation": {"ms_per_generated_graph": graph_ms / max(1, args.steps * G), "share_of_step": graph_ms / max(1e-9, ms_local),
                                 "what": "scldpc_graph_generate (Philox keys + bitonic sort per CN position) + scldpc_graph_build_tables, rank 0"},
            "gpu_launches": int(launches), "clocks": clk, "e2e": e2e, "sequential": sequential, "roofline": roof, "kernels": kernels,
            "cpu_baseline": cpu_baseline, "workloads": workloads,
        }
        print(json.dumps(line))
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_res[0])
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_NAMES = ("iters", "residual", "blocks_err", "erasures_exp", "blocks_err_exp")
DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir: str, res) -> None:
    """Per-frame results of one step (int32 [5][graphs][frames], DUMP_NAMES) -> out_dir/<name>.npy, float64 [graphs][frames].
    Above DUMP_LIMIT bytes in all, every array keeps the same seeded sample of frame ids, listed in frame_ids.npy."""
    import numpy as np
    r = res.cpu().numpy().astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    k = DUMP_LIMIT // (8 * (r.shape[0] * r.shape[1] + 1))
    if r.shape[2] > k:
        ids = np.sort(np.random.default_rng(0).choice(r.shape[2], k, replace=False))
        r = r[:, :, ids]
        np.save(os.path.join(out_dir, "frame_ids.npy"), ids.astype(np.float64))
    for name, a in zip(DUMP_NAMES, r):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def main():
    global N_WORDS
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--seed", type=int, default=0x5C1D9C)
    ap.add_argument("--graphs-per-eps", type=int, default=1)
    ap.add_argument("--sample-iters", type=int, default=10, help="reference arm: flooding iterations per sampled frame")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--side-baselines", action="store_true", help="reference arm: also time the CPU samples of the side workloads")
    ap.add_argument("--workloads", default="all", help="side workloads at N=1: all | none | comma list of bp_full_fpg1024,"
                                                       "bp_full_messages,bp_capped_175_traj,window_L100,peeling")
    ap.add_argument("--n-words", type=int, default=N_WORDS, help="64-bit lane words per node (lanes per graph / 64)")
    ap.add_argument("--mode", default="stream", choices=["stream", "batch"],
                    help="stream: lane recycling over --frames-per-graph frames per graph; batch: one frame per lane")
    ap.add_argument("--frames-per-graph", type=int, default=FRAMES_PER_STREAM)
    ap.add_argument("--pipeline", type=int, default=2, help="stream mode: batches in flight (host threads x CUDA streams); 1 = one batch after the other")
    ap.add_argument("--harvest-every", type=int, default=0, help="stream mode: iterations between harvests (0: adaptive)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the per-frame results of the last timed step as DIR/<name>.npy "
                                                          "(float64 [graphs][frames]; rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    N_WORDS = args.n_words
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
