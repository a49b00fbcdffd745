"""Drop-ins for the three reference executables (``simulators_sc_ldpc/bp_decoding/CMakeLists.txt:8-10``):

    bp_lim_iter INDEX W NUM_DOPED MAX_IT [DOPED...]            full BP, iteration-limited      (BP_FULL.c main_terminated :2057)
                [--caps T1,T2,...]                              ... and at several caps from one decode (one file per cap)
    sw_lim_iter INDEX W NUM_DOPED MAX_IT INIT_IT [DOPED...]    sliding window (square window)  (BP_SW.c :2072)
    bp_traj     INDEX W NUM_DOPED MAX_IT IS_TERM [DOPED...]    full BP trajectories            (BP_TRAJ.c :2068)

Same positional arguments, same output file names and row formats (SURVEY.md App. B).  What the reference fixes at
compile time (``#define Def_dv/Def_dc/Def_L/Def_M/Def_epsIni/Def_epsDelta/Def_NUM_POINTS/...``, BP_FULL.c:22-67) are
run-time options here, defaulting to the reference's values.  The reference reads the doped positions starting at
argv[4], i.e. overlapping MAX_IT (BP_FULL.c:2083-2091); ``--compat-argv`` reproduces that, the default reads them after
the documented arguments.

Frames are decoded in batches on the GPU and accounted in frame order, so the early stop (``frame_err >=
numero_frame_err``, willIstop BP_FULL.c:440) ends a point at the same frame as the sequential reference would.
"""
from __future__ import annotations

import argparse
import sys

import numpy as np

from . import engine

DEFAULTS = {
    "bp_lim_iter": dict(M=500, eps_ini=0.48, eps_delta=0.00125, points=26, min_frame_err=1000, max_frames=1000),
    "sw_lim_iter": dict(M=500, eps_ini=0.475, eps_delta=0.00125, points=18, min_frame_err=1000, max_frames=1000),
    "bp_traj": dict(M=2500, eps_ini=0.46, eps_delta=0.005, points=1, min_frame_err=500, max_frames=500),
}
HEADER = "p BER FER BLER BER_EXP FER_EXP BLER_EXP n L f users_err frame_err block_err users_err_exp frame_err_exp block_err_exp\n"


def result_row(eps, n, L, f, c):
    """``risultati`` row (BP_FULL.c:499-515)."""
    return "%f %e %e %e %e %e %e %d %d %d %d %d %d %d %d %d\n" % (
        eps, c["users_err"] / n / f, c["frame_err"] / f, c["block_err"] / L / f, c["users_err_exp"] / n / f,
        c["frame_err_exp"] / f, c["block_err_exp"] / L / f, n, L, f, c["users_err"], c["frame_err"], c["block_err"],
        c["users_err_exp"], c["frame_err_exp"], c["block_err_exp"])


def account(counters, residual, blocks_err, erasures_exp, blocks_err_exp, erasures_p1=0):
    """``plr_computation`` (BP_FULL.c:1503-1520) for one frame."""
    if residual > 0:
        counters["users_err"] += int(residual)
        counters["frame_err"] += 1
        counters["block_err"] += int(blocks_err)
    if erasures_exp > 0:
        counters["users_err_exp"] += int(erasures_exp)
        counters["frame_err_exp"] += 1
        counters["block_err_exp"] += int(blocks_err_exp)
    if erasures_p1 > 0:
        counters["frame_errP1"] += 1


def new_counters():
    return dict(users_err=0, frame_err=0, block_err=0, users_err_exp=0, frame_err_exp=0, block_err_exp=0, frame_errP1=0)


def parse_caps(max_it: int, caps_arg: str) -> list[int]:
    """``bp_lim_iter --caps``: MAX_IT together with the listed caps, each through max(1, .) like MAX_IT itself, sorted and
    deduplicated."""
    vals = [max_it] + [int(x) for x in caps_arg.split(",") if x.strip()]
    return sorted({max(1, v) for v in vals})


def replay_caps(records, max_frames: int, min_frame_err: int, state=None):
    """Per-cap ``plr_computation`` / ``willIstop`` over one round of frames of a shared checkpointed stream.

    ``records``: int array [N][K][4], per frame in global frame order and per cap (ascending) the residual, blocks_err,
    erasures_exp and blocks_err_exp.  Every cap accounts frames in order until its own ``frame_err >= min_frame_err``
    or ``max_frames``, exactly as a separate run at that cap would over the same frames.  ``state``: the result of the
    previous round of the same point (None for the first); returns the updated list of K dicts with ``counters``,
    ``frames`` and ``stopped``."""
    rec = np.asarray(records)
    K = rec.shape[1]
    if state is None:
        state = [dict(counters=new_counters(), frames=0, stopped=False) for _ in range(K)]
    for k in range(K):
        s = state[k]
        c = s["counters"]
        for i in range(rec.shape[0]):
            if s["frames"] >= max_frames or s["stopped"]:
                break
            account(c, rec[i, k, 0], rec[i, k, 1], rec[i, k, 2], rec[i, k, 3])
            s["frames"] += 1
            if c["frame_err"] >= min_frame_err:
                s["stopped"] = True
    return state


def trajectory_text(rows: np.ndarray, iters: int) -> str:
    """decodeBP's per-frame text (BP_TRAJ.c:988,1051,1145): ``iter\\tdeg1\\tdVNs\\tfirst_pos`` lines + a blank line."""
    out = []
    for t in range(iters):
        out.append("%d\t%d\t%d\t%d\n" % (t, rows[t, 0], rows[t, 1], rows[t, 2]))
    out.append("\n")
    return "".join(out)


def _parser(prog):
    d = DEFAULTS[prog]
    ap = argparse.ArgumentParser(prog=prog)
    ap.add_argument("index", type=int)
    ap.add_argument("W", type=int)
    ap.add_argument("num_doped", type=int)
    ap.add_argument("max_it", type=int)
    if prog == "sw_lim_iter":
        ap.add_argument("init_it", type=int)
    if prog == "bp_traj":
        ap.add_argument("is_term", type=int)
    ap.add_argument("doped", type=int, nargs="*")
    ap.add_argument("--dv", type=int, default=4)
    ap.add_argument("--dc", type=int, default=8)
    ap.add_argument("--L", type=int, default=50)
    ap.add_argument("--M", type=int, default=d["M"], help="Def_M: CNs per position (VNs per position = Def_M*dc/dv)")
    ap.add_argument("--eps-ini", type=float, default=d["eps_ini"])
    ap.add_argument("--eps-delta", type=float, default=d["eps_delta"])
    ap.add_argument("--points", type=int, default=d["points"])
    ap.add_argument("--min-frame-err", type=int, default=d["min_frame_err"])
    ap.add_argument("--max-frames", type=int, default=d["max_frames"])
    ap.add_argument("--seed", type=int, default=None)
    # The reference draws a new code for every frame (BP_FULL.c:2122); bit-slicing needs 64 frames per code.  The default is
    # that minimum, so a point of max_frames frames averages over max_frames/64 code realisations; more frames per graph
    # decode faster but correlate the frames of a graph (same estimator, larger variance) -- the value in use is reported on
    # stderr with the number of graphs behind every point.
    ap.add_argument("--frames-per-graph", type=int, default=64)
    ap.add_argument("--graphs-per-batch", type=int, default=16)
    ap.add_argument("--stream", choices=["auto", "on", "off"], default="auto",
                    help="bp_lim_iter: decode each graph's frames as a stream with lane recycling (auto: from 1024 frames per graph)")
    if prog == "bp_lim_iter":
        ap.add_argument("--caps", default=None, metavar="T1,T2,...",
                        help="error rates at several iteration limits from one decode: the caps are MAX_IT and these values (each "
                             "max(1, .)), and every cap gets the file, name and rows a run with that MAX_IT writes, with its own "
                             "early stop and counters.  Always on the stream path (--stream off is an error).  The frames are "
                             "decoded once up to the largest cap.  A frame in error at a cap is in error at every smaller cap, so "
                             "the largest cap stops last and the points advance as in a separate run at the largest cap: its file "
                             "is byte-identical to that run's; every cap's first point is, and so is every point when no cap "
                             "stops early.  For later points a smaller cap's rows come from the frames the shared run drew, "
                             "which differ from the ones a separate run at that cap would draw")
    if prog == "bp_traj":
        ap.add_argument("--moments-file", default=None,
                        help="also accumulate the per-iteration moments of the rows on the device (engine.MOMENT_NAMES) and pickle "
                             "{eps: int64[max_it][8]} here; with --no-text the text rows are not written (large frame counts). "
                             "Moments cover whole batches: the 'frames' column says how many frames went in")
        ap.add_argument("--no-text", action="store_true")
    ap.add_argument("--compat-argv", action="store_true", help="read doped positions from argv[4] on like the reference")
    ap.add_argument("--outdir", default=".")
    return ap


def run(prog: str, argv=None) -> int:
    import os
    import time
    a = _parser(prog).parse_args(argv)
    if a.compat_argv:
        # the C programs read doped_positions[i] = atoi(argv[4 + i]) (BP_FULL.c:2083-2091): argv[4] is MAX_IT, then whatever
        # follows it.  Taken from the parsed namespace, so option values can never be mistaken for positionals.
        tail = [a.max_it] + ([a.init_it] if prog == "sw_lim_iter" else []) + ([a.is_term] if prog == "bp_traj" else []) + list(a.doped)
        if len(tail) < a.num_doped:
            raise SystemExit(f"{prog}: --compat-argv needs {a.num_doped} values from MAX_IT on")
        doped = [int(x) for x in tail[: a.num_doped]]
    else:
        doped = list(a.doped)[: a.num_doped]
    from . import dist as D
    rank, world = D.init_from_env()
    # srandom(tv_usec), BP_FULL.c:2059-2062.  Under torchrun every rank must draw from the same stream: rank 0's seed.
    seed = a.seed if a.seed is not None else D.broadcast_int(int(time.time() * 1e6) & 0x7FFFFFFF)
    vns_pos = a.M * a.dc // a.dv
    ens = engine.Ensemble(a.dv, a.dc, a.L, vns_pos)
    max_it = max(1, a.max_it)                                          # do { } while (iter < MaxNumIt) runs at least once
    init_it = getattr(a, "init_it", 0) or a.max_it                     # BP_SW.c:2099-2102
    fpg, G = a.frames_per_graph, a.graphs_per_batch
    nw = engine.words_for(fpg)
    if prog == "sw_lim_iter":
        name = "SC_LDPC_%d_%d_L%d_M%d_BP_SW%d_%dit_%dinit_Random_BLER_%d.dat" % (a.dv, a.dc, a.L, a.M, a.W, a.max_it, init_it, a.index)
    else:
        name = "SC_LDPC_%d_%d_L%d_M%d_BP_SW%d_%dit_Random_BLER_%d.dat" % (a.dv, a.dc, a.L, a.M, a.W, a.max_it, a.index)
    graph_id = 0
    moments_all = {}
    sw = prog == "sw_lim_iter"
    use_stream = prog == "bp_lim_iter" and (a.stream == "on" or (a.stream == "auto" and fpg >= 1024))
    caps = None
    if getattr(a, "caps", None) is not None:
        if a.stream == "off":
            raise SystemExit(f"{prog}: --caps decodes on the stream path; it cannot be combined with --stream off")
        caps = parse_caps(a.max_it, a.caps)
        if len(caps) > engine._lib.MAX_CAPS:
            raise SystemExit(f"{prog}: at most {engine._lib.MAX_CAPS} caps")
        use_stream = True
        # a run with MAX_IT = T writes "%dit" with T as given; the cap MAX_IT itself keeps that name
        cap_names = {c: name.replace("_%dit_" % a.max_it, "_%dit_" % (a.max_it if c == max_it else c)) for c in caps}
    for sim in range(a.points):
        eps = a.eps_ini - sim * a.eps_delta                            # inizio_sim, BP_FULL.c:300
        c = new_counters()
        f = 0
        traj_f = None
        mom = None
        want_mom = prog == "bp_traj" and a.moments_file is not None
        if prog == "bp_traj" and rank == 0 and not a.no_text:
            tname = "trajectories_%.4f_%s_SC_LDPC_%d_%d_L%d_M%d_BP_Full_%dit_Random_BLER_%d.dat" % (
                eps, "terminated" if a.is_term else "truncated", a.dv, a.dc, a.L, a.M, a.max_it, a.index)
            traj_f = open(os.path.join(a.outdir, tname), "w")
        stop = False
        # One round = world_size batches of G graphs (rank r decodes the r-th; graph and frame ids are global).  The
        # per-frame results are all-gathered and every rank replays plr_computation / willIstop over them in frame order,
        # so the files are the same for any number of GPUs.
        rnd = 0
        cap_state = None
        while f < a.max_frames and not stop:
            gid = graph_id + (rnd * world + rank) * G
            rnd += 1
            if use_stream:
                # same graphs and channel realisations as below (frame f of graph g is the same Philox draw), decoded on at
                # most 1024 lanes per graph: a lane whose frame has stopped or hit the cap takes the graph's next frame
                lanes = min(fpg, 1024)
                fb = engine.FrameBatch(ens, G, lanes, engine.words_for(lanes))
                fb.generate_graphs(seed, first_graph_id=gid)
                if caps is not None:
                    # one record of 1 + 4K integers per frame: iterations under the largest cap, then the statistics per cap
                    r = engine.decode_bp_stream(fb, fpg, eps, seed + 1, first_graph_id=gid, is_term=True, doping_points=doped, caps=caps)
                    K = len(caps)
                    st = np.stack([r.residual, r.blocks_err, r.erasures_exp, r.blocks_err_exp], axis=-1)      # [K][G][B][4]
                    rec = np.concatenate([r.iters.reshape(-1, 1), st.transpose(1, 2, 0, 3).reshape(-1, 4 * K)], axis=1).astype(np.int64)
                    rec = D.allgather_rows(rec).reshape(-1, 1 + 4 * K)
                    cap_state = replay_caps(rec[:, 1:].reshape(-1, K, 4), a.max_frames, a.min_frame_err, cap_state)
                    f, stop = cap_state[-1]["frames"], cap_state[-1]["stopped"]        # the largest cap stops last
                    c = cap_state[-1]["counters"]
                    continue
                r = engine.decode_bp_stream(fb, fpg, eps, seed + 1, first_graph_id=gid, is_term=True, doping_points=doped, max_it=max_it)
                rec = np.stack([r.residual, r.blocks_err, r.erasures_exp, r.blocks_err_exp, np.zeros_like(r.residual), r.iters],
                               axis=-1).astype(np.int64)
                rec = D.allgather_rows(rec).reshape(-1, 6)
                for k in range(len(rec)):
                    if f >= a.max_frames or stop:
                        break
                    account(c, rec[k, 0], rec[k, 1], rec[k, 2], rec[k, 3], rec[k, 4])
                    f += 1
                    if c["frame_err"] >= a.min_frame_err:
                        stop = True
                continue
            fb = engine.FrameBatch(ens, G, fpg, nw)
            fb.generate_graphs(seed, first_graph_id=gid)
            fb.generate_erasures(eps, seed + 1, first_graph_id=gid, doping_points=doped)
            if sw:
                r = engine.decode_bp_window(fb, a.W, max_it, max(1, init_it), square=True, is_term=True)
            elif prog == "bp_traj" and want_mom:
                res_d, erased_d, rows_d, launched = engine.decode_bp_full(fb, max_it, is_term=bool(a.is_term), trajectory=True,
                                                                          max_rows=max_it, collect=False)
                mom = engine.trajectory_moments(fb, res_d[0], rows_d, mom)
                if a.no_text:                                          # nothing but the counters leaves the device
                    rr = res_d.cpu().numpy()[:, :, :fpg]
                    r = engine.BpResult(rr[0], rr[1], rr[2], rr[3], rr[4], rr[5], erased_d, None, n_frames=fpg)
                else:
                    r = engine._collect(fb, res_d, erased_d, rows_d)
            elif prog == "bp_traj":
                r = engine.decode_bp_full(fb, max_it, is_term=bool(a.is_term), trajectory=True, max_rows=max_it)
            else:
                r = engine.decode_bp_full(fb, max_it, is_term=True)
            rec = np.stack([r.residual, r.blocks_err, r.erasures_exp, r.blocks_err_exp,
                            r.erasures_p1 if sw else np.zeros_like(r.residual), r.iters], axis=-1).astype(np.int64)
            rec = D.allgather_rows(rec).reshape(-1, 6)                 # [world*G*fpg], global frame order
            rows = D.allgather_rows(r.rows).reshape((-1,) + r.rows.shape[2:]) if (prog == "bp_traj" and r.rows is not None) else None
            for k in range(len(rec)):
                if f >= a.max_frames or stop:
                    break
                if traj_f is not None:
                    traj_f.write(trajectory_text(rows[k], int(rec[k, 5])))
                account(c, rec[k, 0], rec[k, 1], rec[k, 2], rec[k, 3], rec[k, 4])
                f += 1
                if c["frame_err"] >= a.min_frame_err:                  # willIstop, BP_FULL.c:440-451
                    stop = True
        n_graphs_point = (f + fpg - 1) // fpg
        graph_id += (f + G * fpg - 1) // (G * fpg) * G                 # the batches a single process would have drawn
        if traj_f is not None:
            traj_f.close()
        if want_mom:
            import pickle
            m = D.allreduce_counters(mom.cpu().numpy() if mom is not None else np.zeros((max_it, len(engine.MOMENT_NAMES)), np.int64),
                                     device=D._comm_device() if world > 1 else None)
            moments_all[float("%.6f" % eps)] = m
            if rank == 0:
                with open(os.path.join(a.outdir, a.moments_file), "wb") as mf:
                    pickle.dump({"names": engine.MOMENT_NAMES, "moments": moments_all}, mf)
        if rank == 0:
            print("%s: eps=%f frames=%d frames_per_graph=%d graphs=%d frame_err=%d (the reference draws one graph per frame)"
                  % (prog, eps, f, fpg, n_graphs_point, c["frame_err"]), file=sys.stderr)
        if rank == 0 and caps is not None:
            for cap, s in zip(caps, cap_state):
                with open(os.path.join(a.outdir, cap_names[cap]), "w" if sim == 0 else "a") as out:
                    if sim == 0:
                        out.write(HEADER)
                    out.write(result_row(eps, ens.n, a.L, s["frames"], s["counters"]))
            continue
        # BP_TRAJ.c's main_terminated only writes the trajectories file (its risultati call is commented out, :2176)
        if rank == 0 and prog != "bp_traj":
            with open(os.path.join(a.outdir, name), "w" if sim == 0 else "a") as out:
                if sim == 0:
                    out.write(HEADER)
                out.write(result_row(eps, ens.n, a.L, f, c))
    return 0


def bp_lim_iter(argv=None):
    return run("bp_lim_iter", argv)


def sw_lim_iter(argv=None):
    return run("sw_lim_iter", argv)


def bp_traj(argv=None):
    return run("bp_traj", argv)


if __name__ == "__main__":
    prog = sys.argv[1] if len(sys.argv) > 1 else ""
    if prog not in DEFAULTS:
        sys.exit("usage: python -m fl_scaling_sc_ldpc_b200.bp_cli {bp_lim_iter|sw_lim_iter|bp_traj} ARGS...")
    sys.exit(run(prog, sys.argv[2:]))
