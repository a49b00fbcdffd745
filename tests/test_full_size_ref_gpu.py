"""The BENCHMARKED shapes against the reference decoders at full size.

bench.py decodes G=4 graphs (eps 0.46..0.49) x 16384 frames on 1024 bit-sliced lanes (n_words=16), M=10000, with the
node-state stream kernels.  This module runs exactly that step (same seed, graph ids and frame ids as the bench's first
resident batch) and checks a sample of frame ids spread over lanes and harvests -- including frames that stall at
eps=0.49 -- against what decodeBP (BP_TRAJ.c:901-1151) returns for the same graph and channel realisation: iterations,
residual, blocks, expurgated counts.  The same for BASELINE config 3 (capped runs with every trajectory row, capped
streams) and config 4 (decodeBP_SW of BP_SW.c:628-912 at L=100, M=10000, W in {3,10}, 8 iterations per window, 60 for the
first), plus the derived non-terminated window mode and a wider sample of the bench step against the oracle port.

The expected values of the reference decoders are stored in tests/golden/full_size_golden.npz, written by
tests/golden/make_full_size_golden.py from the compiled reference (oracle/_ref) where it is built and from the oracle port
otherwise; the port is pinned to the compiled reference bit for bit by the golden vectors of test_oracle_golden.py, and
the file's `source` says which of the two produced it.  Since the device draws the graphs and channel realisations, the
stored values also pin the generators."""
import os

import numpy as np
import pytest

import fl_scaling_sc_ldpc_b200 as eng
import oracle

pytestmark = pytest.mark.gpu
DV, DC, M = 4, 8, 10000
SEED = 0x5C1D9C                      # bench.py's default
EPS = [0.46, 0.47, 0.48, 0.49]
KEYS = ("iters", "residual", "blocks_err", "erasures_exp", "blocks_err_exp")
SW_KEYS = ("residual", "erasures_p1", "blocks_err", "erasures_exp", "blocks_err_exp")
CAPSTREAM_FRAMES = ((1, 3), (2, 1500))
TRAJ_RUNS = ((175, 1, (0, 100)), (1000, 1, (64,)), (175, 0, (9,)))     # (cap, is_term, frames), graph of eps = 0.48
SW_RUNS = ((10, 0.45), (3, 0.36))                                     # (W, eps), frames 0 and 127
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "full_size_golden.npz")


def _frame_channel(ens, eps, seed, gid, frame):
    """the channel realisation of frame id `frame` of graph stream `gid` -- what the stream kernels draw in place"""
    fb = eng.FrameBatch(ens, 1, 4, 2)
    fb.generate_erasures(eps, seed, first_graph_id=gid, first_frame=frame & ~3)
    return fb.erasures_host()[0][frame & 3]


def stream_picks(s):
    """frame ids of the bench step to check: three per graph of eps 0.46..0.48, and at eps 0.49 the two shortest stalled
    and the two shortest decoded frames"""
    picks = [(g, f) for g in range(3) for f in (5, 1030 + g, 16000 + 7 * g)]
    fails = np.flatnonzero(s.residual[3] > 0)
    oks = np.flatnonzero(s.residual[3] == 0)
    assert len(fails) >= 2 and len(oks) >= 2
    picks += [(3, int(f)) for f in fails[np.argsort(s.iters[3][fails], kind="stable")[:2]]]
    picks += [(3, int(f)) for f in oks[np.argsort(s.iters[3][oks], kind="stable")[:2]]]
    return picks


def run_gpu():
    """GPU side of every case.  Returns (results by case, inputs): the inputs hold the ensembles, graphs and channel
    realisations the cases decoded, from which make_full_size_golden.py computes the expected values."""
    gpu, inp = {}, {}

    # ---- A: the bench step (stream, node-state kernels, unlimited iterations); C: capped stream, cap 175 ----
    ens = eng.Ensemble(DV, DC, 50, M)
    fbg = eng.FrameBatch(ens, 4, 1024, 16).generate_graphs(seed=SEED, first_graph_id=0)
    gpu["stream"] = eng.decode_bp_stream(fbg, 16384, EPS, SEED + 1, first_graph_id=0)
    gpu["capstream"] = eng.decode_bp_stream(fbg, 2048, EPS, SEED + 1, first_graph_id=0, max_it=175)
    inp["ens"], inp["vn"] = ens, fbg.vn_cn.cpu().numpy()

    # ---- B: capped runs with trajectory rows (config 3), graph of eps = 0.48 ----
    fbt = eng.FrameBatch(ens, 1, 128, 2)
    fbt.vn_cn.copy_(fbg.vn_cn[2:3]); fbt._build_tables()
    fbt.generate_erasures(0.48, SEED + 1, first_graph_id=2, first_frame=0)
    inp["cht"] = fbt.erasures_host()[0]
    for cap, is_term, _ in TRAJ_RUNS:
        gpu[("traj", cap, is_term)] = eng.decode_bp_full(fbt, cap, bool(is_term), trajectory=True, max_rows=cap)
    del fbt, fbg

    # ---- D: window decoder (config 4), L = 100 ----
    ensw = eng.Ensemble(DV, DC, 100, M)
    fbw = eng.FrameBatch(ensw, 1, 128, 2).generate_graphs(seed=SEED, first_graph_id=100)
    gpu["vnw"] = fbw.vn_cn.cpu().numpy()[0]
    for W, e in SW_RUNS:
        fbw.generate_erasures(e, SEED + 2, first_graph_id=100)
        chw = fbw.erasures_host()[0]
        inp[("chw", W)] = chw.copy()
        gpu[("sw", W)] = eng.decode_bp_window(fbw, W, 8, 60, square=True, is_term=True)
        gpu[("sw_nt", W)] = (eng.decode_bp_window(fbw, W, 8, 60, square=True, is_term=False), chw.copy())
    return gpu, inp


@pytest.fixture(scope="module")
def cases():
    gpu, _ = run_gpu()
    return gpu, np.load(GOLDEN)


def test_bench_step_matches_compiled_reference(cases):
    gpu, z = cases
    s = gpu["stream"]
    assert stream_picks(s) == [tuple(int(x) for x in p) for p in z["stream_frames"]]
    for (g, f), want in zip(z["stream_frames"], z["stream_expect"]):
        got = tuple(int(getattr(s, k)[g, f]) for k in KEYS)
        assert got == tuple(int(x) for x in want), (g, f, got)
    assert len(z["stream_frames"]) == 13
    # at least two of them are frames that stalled
    assert (z["stream_expect"][:, 1] > 0).sum() >= 2


def test_capped_stream_matches_compiled_reference(cases):
    gpu, z = cases
    s = gpu["capstream"]
    assert [tuple(int(x) for x in p) for p in z["capstream_frames"]] == list(CAPSTREAM_FRAMES)
    for (g, f), want in zip(z["capstream_frames"], z["capstream_expect"]):
        got = tuple(int(getattr(s, k)[g, f]) for k in KEYS)
        assert got == tuple(int(x) for x in want), (g, f, got)
        assert want[0] == 175 and want[1] > 0          # the cap binds at this size


def test_capped_trajectories_match_compiled_reference(cases):
    gpu, z = cases
    n_ens = 50 * M
    assert [tuple(int(x) for x in c) for c in z["traj_cases"]] == [(cap, t, f) for cap, t, fs in TRAJ_RUNS for f in fs]
    for i, (cap, is_term, f) in enumerate(z["traj_cases"]):
        r = gpu[("traj", cap, is_term)]
        want = [int(x) for x in z["traj_expect"][i]]
        k = int(r.iters[0, f])
        assert [k] + [int(getattr(r, key)[0, f]) for key in KEYS[1:]] == want, (cap, is_term, f)
        rows = z[f"traj_rows{i}"]
        assert len(rows) == k
        assert (r.rows[0, f, :k] == rows).all(), (cap, is_term, f)      # deg_1_iter, dVNs, first erased position: every row
        assert (np.packbits(r.erased()[0, f]) == z[f"traj_erased{i}"]).all(), (cap, is_term, f)
        assert rows[:, 1].sum() == n_ens - want[1]


def test_window_decoder_matches_compiled_reference(cases):
    gpu, z = cases
    assert [tuple(int(x) for x in c) for c in z["sw_cases"]] == [(W, f) for W, _ in SW_RUNS for f in (0, 127)]
    for i, (W, f) in enumerate(z["sw_cases"]):
        r = gpu[("sw", W)]
        got = tuple(int(getattr(r, k)[0, f]) for k in SW_KEYS)
        assert got == tuple(int(x) for x in z["sw_expect"][i]), (W, f, got)
        assert (np.packbits(r.erased()[0, f]) == z[f"sw_erased{i}"]).all(), (W, f)


def test_window_decoder_non_terminated_matches_oracle_port(cases):
    """the derived non-terminated mode (SURVEY 8a-B2: CN window clipped at L*cns_pos) has no compiled counterpart"""
    gpu, _ = cases
    ensw = eng.Ensemble(DV, DC, 100, M)
    g = oracle.Graph(gpu["vnw"], 100, M, ensw.cns_pos, DV, DC)
    for W in (10, 3):
        r, chw = gpu[("sw_nt", W)]
        er = r.erased()[0]
        for f in (1, 126):
            o = oracle.decode_bp_sw(g, chw[f].astype(np.int32), W, 8, 60, 1, 0)
            got = (int(r.residual[0, f]), int(r.erasures_p1[0, f]), int(r.blocks_err[0, f]), int(r.iters[0, f]))
            assert got == (o["residual"], o["erasures_p1"], o["blocks_err"], int(o["win_iters"].sum())), (W, f, got)
            assert (er[f] == o["erased"]).all()


def test_bench_step_sample_matches_oracle_port(cases):
    """a wider sample of the same step against the (much faster) oracle port: 12 frame ids per graph over all harvests"""
    gpu, _ = cases
    s = gpu["stream"]
    ens = eng.Ensemble(DV, DC, 50, M)
    fbg = eng.FrameBatch(ens, 4, 4, 2).generate_graphs(seed=SEED, first_graph_id=0)
    vn = fbg.vn_cn.cpu().numpy()
    rng = np.random.default_rng(3)
    jobs = []
    for g in range(4):
        gg = oracle.Graph(vn[g], 50, M, ens.cns_pos, DV, DC)
        for f in sorted(rng.choice(16384, 6 if g == 3 else 4, replace=False)):
            jobs.append((g, int(f), gg, _frame_channel(ens, EPS[g], SEED + 1, g, int(f)).astype(np.int32)))
    # the oracle port runs outside the GIL (ctypes): a thread per host core
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 1)) as ex:
        outs = list(ex.map(lambda j: oracle.decode_bp(j[2], j[3], 10 ** 9, 1, max_rows=1), jobs))
    for (g, f, _, _), o in zip(jobs, outs):
        got = tuple(int(getattr(s, k)[g, f]) for k in KEYS)
        assert got == tuple(int(o[k]) for k in KEYS), (g, f, got)
