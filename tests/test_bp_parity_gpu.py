"""GPU parity tests: the CUDA decoders (through the C ABI) against the CPU oracle and the committed golden vectors,
bit-exact on every output the reference produces: iterations executed, NumErasures, VNerased, block / expurgated
statistics and the per-iteration trajectory rows."""
import numpy as np
import pytest

import fl_scaling_sc_ldpc_b200 as eng
from tests import util

pytestmark = pytest.mark.gpu

KEYS = ("iters", "residual", "blocks_err", "erasures_exp", "blocks_err_exp")


def make_batch(dv, dc, L, M, graphs, chan, n_words=None):
    ens = eng.Ensemble(dv, dc, L, M)
    G, F, _ = chan.shape
    fb = eng.FrameBatch(ens, G, F, n_words)
    fb.set_graphs(np.stack([g.vn_cn for g in graphs]))
    fb.set_erasures(chan)
    return fb


def check_bp(res, ref, rows=False):
    for k in KEYS:
        assert (getattr(res, k) == ref[k]).all(), (k, getattr(res, k), ref[k])
    assert (res.erased() == ref["erased"]).all()
    if rows:
        G, F = ref["iters"].shape
        for g in range(G):
            for f in range(F):
                k = min(ref["iters"][g, f], res.rows.shape[2])
                assert (res.rows[g, f, :k] == ref["rows"][g, f, :k]).all(), (g, f)


@pytest.fixture(params=["node_state", "wave", "sweep_all"])
def sweep_mode(request, monkeypatch):
    """full BP in node-state form (default for runs without a trajectory), with message passing and wave tracking (only
    positions whose inputs changed are swept), and with message passing over every position in every iteration, like the
    reference; all must be bit-identical to the oracle.  Trajectory runs always pass messages."""
    monkeypatch.setenv("SCLDPC_FULL_NODE", "1" if request.param == "node_state" else "0")
    if request.param == "sweep_all":
        monkeypatch.setenv("SCLDPC_NO_WAVE", "1")
    else:
        monkeypatch.delenv("SCLDPC_NO_WAVE", raising=False)
    return request.param


@pytest.mark.parametrize("dv,dc,L,M", [(4, 8, 10, 50), (3, 6, 10, 48), (5, 10, 12, 40), (4, 8, 6, 16), (4, 8, 20, 128)])
def test_full_bp_matches_oracle(dv, dc, L, M, sweep_mode):
    eps = [0.30, 0.42, 0.46, 0.50, 0.56] if dv != 3 else [0.3, 0.38, 0.42, 0.47]
    graphs, chan, _ = util.random_case(dv, dc, L, M, G=2, F=70, eps_list=eps, seed=1000 + L + M, doped_every=9)
    fb = make_batch(dv, dc, L, M, graphs, chan)
    for is_term in (True, False):
        for cap in (0, 7, 1):
            ref = util.oracle_bp(graphs, chan, cap, int(is_term), max_rows=64)
            res = eng.decode_bp_full(fb, cap, is_term)
            check_bp(res, ref)
            rest = eng.decode_bp_full(fb, cap, is_term, trajectory=True, max_rows=64)
            check_bp(rest, ref, rows=True)


def test_full_bp_long_chain_wave_tracking():
    """a long chain at small M: the decoding wave leaves most positions idle for most iterations"""
    dv, dc, L, M = 4, 8, 60, 64
    graphs, chan, _ = util.random_case(dv, dc, L, M, G=2, F=130, eps_list=[0.40, 0.44, 0.47], seed=909)
    fb = make_batch(dv, dc, L, M, graphs, chan)
    for is_term in (True, False):
        ref = util.oracle_bp(graphs, chan, 0, int(is_term), max_rows=400)
        res = eng.decode_bp_full(fb, 0, is_term, trajectory=True, max_rows=400)
        check_bp(res, ref, rows=True)
        check_bp(eng.decode_bp_full(fb, 0, is_term), ref)
        check_bp(eng.decode_bp_full(fb, 25, is_term), util.oracle_bp(graphs, chan, 25, int(is_term), max_rows=1))


def test_full_bp_lane_words_and_ragged_frames():
    """every supported lane-word count, frame counts that do not fill the last word, and zero frames"""
    dv, dc, L, M = 4, 8, 8, 32
    for n_words, F in ((2, 1), (2, 128), (4, 130), (8, 300), (16, 700)):
        graphs, chan, _ = util.random_case(dv, dc, L, M, G=1, F=F, eps_list=[0.44, 0.5], seed=77 + F)
        fb = make_batch(dv, dc, L, M, graphs, chan, n_words)
        ref = util.oracle_bp(graphs, chan, 0, 1, max_rows=48)
        check_bp(eng.decode_bp_full(fb, 0, True, trajectory=True, max_rows=48), ref, rows=True)
    fb = eng.FrameBatch(eng.Ensemble(dv, dc, L, M), 1, 0, 2)
    fb.set_graphs(graphs[0].vn_cn[None])
    r = eng.decode_bp_full(fb, 0, True)
    assert r.iters.shape == (1, 0)


def test_full_bp_extreme_channels():
    """all-known, all-erased and single-erasure patterns"""
    dv, dc, L, M = 4, 8, 6, 16
    graphs, chan, _ = util.random_case(dv, dc, L, M, G=1, F=5, eps_list=[0.4], seed=5)
    chan[0, 0] = 0
    chan[0, 1] = 1
    chan[0, 2] = 0; chan[0, 2, 17] = 1
    chan[0, 3] = 1; chan[0, 3, : M] = 0
    fb = make_batch(dv, dc, L, M, graphs, chan)
    for is_term in (True, False):
        ref = util.oracle_bp(graphs, chan, 0, int(is_term), max_rows=32)
        check_bp(eng.decode_bp_full(fb, 0, is_term, trajectory=True, max_rows=32), ref, rows=True)


@pytest.fixture(params=["node_state", "two_launches"])
def window_mode(request, monkeypatch):
    """the window decoder in node-state form and with message-passing sweeps (two launches per iteration).  The node-state
    form takes resolution lists iff 2(W+dv-1) >= L and copies the VN window otherwise, so the windows below run both
    variants: the copy at W=2 for (3,6) L=10 and at W=2, 3 for (4,8) L=14, the lists everywhere else"""
    monkeypatch.setenv("SCLDPC_WINDOW_NODE", "1" if request.param == "node_state" else "0")
    return request.param


@pytest.mark.parametrize("dv,dc,L,M", [(4, 8, 10, 50), (3, 6, 10, 48), (4, 8, 14, 64)])
def test_window_bp_matches_oracle(dv, dc, L, M, window_mode):
    eps = [0.35, 0.44, 0.47, 0.52] if dv != 3 else [0.3, 0.38, 0.42]
    graphs, chan, _ = util.random_case(dv, dc, L, M, G=2, F=40, eps_list=eps, seed=2000 + L + M, doped_every=7)
    fb = make_batch(dv, dc, L, M, graphs, chan)
    for square in (True, False):
        for is_term in (True, False):
            for (W, cap, init) in ((3, 0, 0), (4, 4, 12), (5, 2, 0), (2, 1, 1), (L + 4, 3, 0)):
                ref = util.oracle_sw(graphs, chan, W, cap, init if square else 0, int(square), int(is_term))
                res = eng.decode_bp_window(fb, W, cap, init if square else 0, square, is_term)
                for k in KEYS + ("erasures_p1",):
                    assert (getattr(res, k) == ref[k]).all(), (square, is_term, W, cap, init, k)
                assert (res.erased() == ref["erased"]).all()


@pytest.mark.parametrize("path", util.golden_files(), ids=lambda p: p.split("bp_golden_")[-1])
def test_against_golden_vectors(path):
    """outputs of the compiled reference itself (tests/golden/make_golden.py)"""
    z, d = util.load_golden(path)
    ens = eng.Ensemble(d["dv"], d["dc"], d["L"], d["vns_pos"])
    fb = eng.FrameBatch(ens, d["G"], d["F"]).set_graphs(z["vn_cn"]).set_erasures(z["chan"])
    for is_term in (1, 0):
        for cap in (100000, 5, 1):
            key = f"bp_t{is_term}_c{cap}"
            r = eng.decode_bp_full(fb, cap, bool(is_term), trajectory=True, max_rows=64)
            st = z[key + "_stats"]
            got = np.stack([r.iters, r.residual, r.blocks_err, r.erasures_exp, r.blocks_err_exp], axis=-1)
            assert (got == st).all(), key
            assert (r.erased() == util.unpack_erased(z[key + "_erased"], d["n"])).all(), key
            for g in range(d["G"]):
                for f in range(d["F"]):
                    k = min(64, st[g, f, 0])
                    assert (r.rows[g, f, :k] == z[key + "_rows"][g, f, :k]).all(), key
    for (W, cap, init) in ((3, 100000, 0), (4, 4, 12), (5, 2, 0), (2, 1, 1)):
        for square in (1, 0):
            key = f"sw_s{square}_W{W}_c{cap}_i{init}"
            r = eng.decode_bp_window(fb, W, cap, init if square else 0, bool(square), True)
            got = np.stack([r.residual, r.erasures_p1, r.blocks_err, r.erasures_exp, r.blocks_err_exp], axis=-1)
            assert (got == z[key + "_stats"]).all(), key
            assert (r.erased() == util.unpack_erased(z[key + "_erased"], d["n"])).all(), key


def test_host_buffer_entry_point():
    """scldpc_decode_host: host graph + host erasure bytes in, per-frame results out"""
    dv, dc, L, M = 4, 8, 10, 50
    graphs, chan, _ = util.random_case(dv, dc, L, M, G=2, F=33, eps_list=[0.4, 0.47, 0.53], seed=31)
    vn_cn = np.stack([g.vn_cn for g in graphs])
    ens = eng.Ensemble(dv, dc, L, M)
    ref = util.oracle_bp(graphs, chan, 0, 1, max_rows=40)
    o = eng.decode_host(ens, vn_cn, chan, trajectory=True, max_rows=40, want_erased=True)
    for k in KEYS:
        assert (o[k] == ref[k]).all(), k
    assert (o["erased"] == ref["erased"]).all()
    for g in range(2):
        for f in range(33):
            k = min(40, ref["iters"][g, f])
            assert (o["rows"][g, f, :k] == ref["rows"][g, f, :k]).all()
    ref = util.oracle_sw(graphs, chan, 4, 3, 10, 1, 1)
    o = eng.decode_host(ens, vn_cn, chan, W=4, max_it=3, init_it=10, want_erased=True)
    for k in KEYS + ("erasures_p1",):
        assert (o[k] == ref[k]).all(), k
    assert (o["erased"] == ref["erased"]).all()


def test_malformed_graph_is_rejected():
    ens = eng.Ensemble(4, 8, 6, 16)
    fb = eng.FrameBatch(ens, 1, 4)
    bad = np.zeros((1, ens.n, 4), np.int32)          # every edge on CN 0
    with pytest.raises(eng.ScldpcError):
        fb.set_graphs(bad)


def test_trajectory_moments_on_the_device():
    """scldpc_bp_trajectory_moments: per-iteration counts / sums of the rows, accumulated over two batches on the device,
    against NumPy on the collected rows (the notebook's reductions of bp_traj files, NB cells 40-42)"""
    ens = eng.Ensemble(4, 8, 12, 48)
    cap = 40
    acc, ref = None, np.zeros((cap, 8), np.int64)
    for b, nf in enumerate((100, 128)):
        fb = eng.FrameBatch(ens, 2, nf).generate_graphs(5, first_graph_id=2 * b).generate_erasures([0.44, 0.49], 6, first_graph_id=2 * b)
        res, erased, rows, _ = eng.decode_bp_full(fb, cap, True, trajectory=True, max_rows=cap, collect=False)
        acc = eng.engine.trajectory_moments(fb, res[0], rows, acc)
        r = eng.engine._collect(fb, res, erased, rows)
        for t in range(cap):
            live = r.iters > t
            d1, dv, fp = (r.rows[:, :, t, k].astype(np.int64) for k in range(3))
            ref[t] += [live.sum(), (live & (dv != 0)).sum(), dv[live].sum(), (dv[live] ** 2).sum(), d1[live].sum(), (d1[live] ** 2).sum(),
                       fp[live].sum(), (dv[live] * d1[live]).sum()]
            assert not r.rows[:, :, t][~live].any()                   # rows of stopped frames are the zero padding
    assert (acc.cpu().numpy() == ref).all()
    assert ref[0, 0] == 2 * 228 and ref[-1, 0] < ref[0, 0]


def test_stream_ordered_table_build_reports_validity_without_a_sync():
    """scldpc_graph_build_tables_async: generated graphs are valid (flag 0) and decode like the checked build; a malformed
    injected graph leaves the reference's two failure modes in the flag instead of raising"""
    ens = eng.Ensemble(4, 8, 10, 32)
    fb = eng.FrameBatch(ens, 2, 64).generate_graphs(3).generate_erasures(0.45, 4)
    assert fb.graph_error() == 0
    a = eng.decode_bp_full(fb, 0, True)
    fb._build_tables(check=True)
    b = eng.decode_bp_full(fb, 0, True)
    assert (a.iters == b.iters).all() and (a.residual == b.residual).all()
    good = fb.vn_cn.clone()
    fb.vn_cn[1, 5, 2] = ens.nk + 7                    # CN index out of range
    fb._build_tables(check=False)
    assert fb.graph_error() == 1
    fb.vn_cn.copy_(good)
    fb.vn_cn[0, :9, 0] = fb.vn_cn[0, 0, 0]           # nine edges on one CN
    fb._build_tables(check=False)
    assert fb.graph_error() == 2
    with pytest.raises(eng.ScldpcError):
        fb._build_tables(check=True)
