"""Frame streams with stopping-set records (scldpc_bp_stream_stopping_sets) and simulate_sc_ldpc / ber_sim on them.

Every frame's iterations and record (num_lost, big component?, VNs in big components, positions they touch) must equal what
the synchronous path gives for the same frame: decode_bp_full(unscanned_head_cns=...) + stopping_set_records on the same
graphs, with the channels generate_erasures(first_frame=...) draws, in chunks of at most 1024 frames."""
import numpy as np
import pytest

import fl_scaling_sc_ldpc_b200 as eng
import oracle
from fl_scaling_sc_ldpc_b200 import peeling_decoding as pdx
from tests import util

pytestmark = pytest.mark.gpu


def sync_frames(fbg, graphs, B, eps, seed, gid0, is_term, counted, unscanned, doping_points=(), frames=None, chunk=1024):
    """iters [len(graphs)][B] and records [len(graphs)][B][4] of the synchronous path for the graphs `graphs` of fbg (chunks
    starting at `frames`, default all); frames not decoded are -1"""
    G = len(graphs)
    eps_all = np.full(fbg.n_graphs, float(eps)) if np.ndim(eps) == 0 else np.asarray(eps, np.float64)
    iters = np.full((G, B), -1, np.int64)
    recs = np.full((G, B, 4), -1, np.int64)
    starts = range(0, B, chunk) if frames is None else frames
    for f0 in starts:
        nf = min(chunk, B - f0)
        fb = eng.FrameBatch(fbg.ens, G, nf)
        fb.vn_cn.copy_(fbg.vn_cn[list(graphs)])
        fb._build_tables()
        for i, g in enumerate(graphs):            # graph g keeps its own channel stream (first_graph_id + g)
            one = eng.FrameBatch(fbg.ens, 1, nf)
            one.generate_erasures(float(eps_all[g]), seed, first_graph_id=gid0 + g, doping_points=doping_points, first_frame=f0)
            fb.chan[i].copy_(one.chan[0])
        res = eng.decode_bp_full(fb, eng.UNLIMITED, is_term=is_term, unscanned_head_cns=unscanned)
        iters[:, f0:f0 + nf] = res.iters
        recs[:, f0:f0 + nf] = pdx.stopping_set_records(fb, res.erased_words, counted)[:, :nf]
    return iters, recs


def stream(fbg, B, eps, seed, gid0, is_term, counted, unscanned, **kw):
    r = eng.decode_bp_stream(fbg, B, eps, seed, first_graph_id=gid0, is_term=is_term, stopping_sets=counted,
                             unscanned_head_cns=unscanned, **kw)
    assert isinstance(r, eng.StreamStoppingSetResult)
    assert r.iters.shape == (fbg.n_graphs, B) and r.records.shape == (fbg.n_graphs, B, 4)
    return r


# (dv, dc, L, M, graph ensemble, terminated, unscanned head in positions, doping, counted-position mask, eps of the two graphs:
# below and above the threshold -- the coupled one for terminated chains, the uncoupled one otherwise)
CASES = [
    (4, 8, 14, 48, {}, True, 0, (), "all", [0.44, 0.53]),                               # bounded, terminated
    (4, 8, 14, 48, {}, False, 3, (), "stripes", [0.33, 0.45]),                          # unbounded, non-terminated
    (3, 6, 14, 48, {"tail_biting": True}, False, 0, (), "stripes", [0.36, 0.48]),      # tail-biting
    (5, 10, 12, 40, {"protograph": True}, True, 2, [6], "all", [0.44, 0.53]),          # protograph ensemble, hard doping, unbounded
    (3, 9, 14, 36, {}, True, 3, {4: 0.5}, "stripes", [0.24, 0.34]),                    # soft doping, unbounded
]


def _counted(kind, L):
    return np.ones(L, bool) if kind == "all" else (np.arange(L) % 3 != 1)


@pytest.mark.parametrize("case", range(len(CASES)))
@pytest.mark.parametrize("lanes,B", [(64, 500), (192, 700), (1024, 2100)])
def test_stream_records_equal_synchronous(case, lanes, B):
    dv, dc, L, M, gen, term, head, doping, kind, eps = CASES[case]
    ens = eng.Ensemble(dv, dc, L, M)
    fbg = eng.FrameBatch(ens, 2, lanes).generate_graphs(31 + case, first_graph_id=5, **gen)
    counted = _counted(kind, L)
    unscanned = head * ens.cns_pos
    it, rec = sync_frames(fbg, (0, 1), B, eps, 9, 5, term, counted, unscanned, doping_points=doping)
    fails = rec[:, :, 0] > 0
    assert 0 < fails.mean() < 1 and fails[0].mean() < fails[1].mean(), fails.mean(axis=1)
    for H in (0, 1, 7, 64):
        r = stream(fbg, B, eps, 9, 5, term, counted, unscanned, doping_points=doping, harvest_every=H)
        assert (r.iters == it).all(), (case, H, np.argwhere(r.iters != it)[:5])
        assert (r.records == rec).all(), (case, H, np.argwhere((r.records != rec).any(-1))[:5])


def _components(lost, vn_cn):
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    k = len(lost)
    cns = vn_cn[lost]
    u, inv = np.unique(cns.reshape(-1), return_inverse=True)
    rows = np.repeat(np.arange(k), cns.shape[1])
    a = coo_matrix((np.ones(rows.size, np.int8), (rows, k + inv.reshape(-1))), shape=(k + len(u), k + len(u)))
    return connected_components(a, directed=False)[1][:k]


def account_lost(lost, vn_cn, M):
    """PD.py:668-691 for one frame, with SciPy components"""
    if len(lost) == 0:
        return (0, 0, 0, 0)
    lab = _components(lost, vn_cn)
    big = np.isin(lab, np.flatnonzero(np.bincount(lab) > 2))
    return (len(lost), int(big.any()), int(big.sum()), len(np.unique(lost[big] // M)))


def test_stream_records_against_the_oracle():
    """a short unbounded, non-terminated stream: every frame's record from the oracle's peeling fixed point"""
    dv, dc, L, M = 4, 8, 16, 40
    ens = eng.Ensemble(dv, dc, L, M)
    cns = ens.cns_pos
    head = 3 * cns
    fbg = eng.FrameBatch(ens, 1, 128).generate_graphs(71, first_graph_id=2)
    counted = np.arange(L) % 4 == 1                          # cuts residuals into components of one, two and more VNs
    B = 600
    r = stream(fbg, B, 0.38, 73, 2, False, counted, head, harvest_every=5)
    ch = np.concatenate([eng.FrameBatch(ens, 1, 200).generate_erasures(0.38, 73, first_graph_id=2, first_frame=f0).erasures_host()[0]
                         for f0 in range(0, B, 200)])
    vn = fbg.vn_cn[0].cpu().numpy().astype(np.int64)
    cvn = np.repeat(counted, M)
    sizes = set()
    for f in range(B):
        fp = oracle.peel_fixed_point(vn, ch[f], ens.nk, head, cns * L)
        want = account_lost(np.flatnonzero(fp.astype(bool) & cvn), vn, M)
        assert tuple(int(x) for x in r.records[0, f]) == want, (f, r.records[0, f], want)
        sizes.add((want[0] > 0) + (want[1] > 0))
    assert 0 in sizes and len(sizes) > 1                      # frames that succeed and frames that fail


def test_stream_records_with_lane_compaction():
    """an unbounded stream whose tail compacts its lanes: the head plane moves with the frames"""
    ens = eng.Ensemble(4, 8, 16, 64)
    fbg = eng.FrameBatch(ens, 2, 512).generate_graphs(47, first_graph_id=3)
    eps, counted, unscanned = [0.46, 0.49], np.ones(16, bool), 3 * ens.cns_pos
    r = stream(fbg, 3000, eps, 5, 3, True, counted, unscanned, harvest_every=4)
    n_cmp, moved = util.stream_compactions(fbg)
    assert n_cmp >= 1 and moved >= n_cmp, (n_cmp, moved)
    it, rec = sync_frames(fbg, (0, 1), 3000, eps, 5, 3, True, counted, unscanned)
    assert (r.iters == it).all() and (r.records == rec).all()


def test_stream_records_full_size():
    """(4,8) L=50 M=10000, eps 0.46-0.49, 16384 frames per graph on 1024 lanes, bounded and terminated: every frame of graph 0
    and the first and last 1024 frames of the other three against the synchronous decoder"""
    ens = eng.Ensemble(4, 8, 50, 10000)
    eps, B = [0.46, 0.47, 0.48, 0.49], 16384
    fbg = eng.FrameBatch(ens, 4, 1024).generate_graphs(61, first_graph_id=7)
    counted = np.ones(50, bool)
    r = stream(fbg, B, eps, 63, 7, True, counted, 0)
    it, rec = sync_frames(fbg, (0,), B, eps, 63, 7, True, counted, 0)
    assert (r.iters[0] == it[0]).all() and (r.records[0] == rec[0]).all()
    it, rec = sync_frames(fbg, (1, 2, 3), B, eps, 63, 7, True, counted, 0, frames=(0, B - 1024))
    for f0 in (0, B - 1024):
        sl = slice(f0, f0 + 1024)
        assert (r.iters[1:, sl] == it[:, sl]).all() and (r.records[1:, sl] == rec[:, sl]).all(), f0
    fer = (r.records[:, :, 0] > 0).mean(axis=1)
    assert fer[0] < fer[3] and fer[3] > 0.01, fer


# ---- simulate_sc_ldpc on frame streams --------------------------------------------------------------------------------
def _sync_records_fn(e, l, r, L_user, M, term, bounded, seed):
    """_records_fn for simulate_sc_ldpc: the records of the synchronous path, drawn as the default path draws them"""
    head, head_sched = (0, 0) if bounded else (20, 10)
    tail = 0 if term else 20
    L_eff = L_user + head + tail
    ens = eng.Ensemble(l, r, L_eff, M)
    num_positions = L_eff + l - 1 if term else L_eff
    counted = pdx.counted_positions(l, L_eff, num_positions, head, tail)

    def fn(G, fpg, gid0):
        fbg = eng.FrameBatch(ens, G, 64).generate_graphs(seed, first_graph_id=gid0)
        _, rec = sync_frames(fbg, range(G), fpg, e, seed + 1, gid0, term, counted, head_sched * ens.cns_pos)
        return rec.reshape(G * fpg, 4)
    return fn


@pytest.mark.parametrize("fpg,term,bounded", [(2048, True, True), (4096, False, False)])
def test_simulate_sc_ldpc_on_streams_equals_synchronous_records(fpg, term, bounded):
    l, r, L, M, e, seed = 4, 8, 12, 48, (0.48 if bounded else 0.45), 211
    n = 3 * fpg                                                # one and a half rounds of two graphs
    kw = dict(seed=seed, frames_per_graph=fpg, graphs_per_batch=2, progress=False)
    fn = _sync_records_fn(e, l, r, L, M, term, bounded, seed)
    full = pdx.simulate_sc_ldpc(e, l, r, L, M, term, False, bounded, False, n, 10 ** 9, [], **kw)
    want = pdx.simulate_sc_ldpc(e, l, r, L, M, term, False, bounded, False, n, 10 ** 9, [], _records_fn=fn, **kw)
    assert full[5] == n and 0 < full[0] < 1

    def same(a, b):
        return all((np.asarray(a[i]) == np.asarray(b[i])).all() for i in range(13))
    assert same(full, want), (full, want)
    cut = max(1, int(full[0] * n * 0.3))                       # the max_fuckups cut falls inside the first round
    a = pdx.simulate_sc_ldpc(e, l, r, L, M, term, False, bounded, False, n, cut, [], **kw)
    b = pdx.simulate_sc_ldpc(e, l, r, L, M, term, False, bounded, False, n, cut, [], _records_fn=fn, **kw)
    assert a[5] < 2 * fpg and same(a, b), (a, b)


def test_simulate_sc_ldpc_at_1024_frames_per_graph_equals_the_synchronous_path():
    l, r, L, M, e, seed = 4, 8, 12, 48, 0.48, 307

    def factory(ens, G, fpg, gid0):                           # what the synchronous default draws
        fb = eng.FrameBatch(ens, G, fpg).generate_graphs(seed, first_graph_id=gid0)
        return fb.generate_erasures(e, seed + 1, first_graph_id=gid0)
    kw = dict(seed=seed, frames_per_graph=1024, graphs_per_batch=2, progress=False)
    for bounded in (True, False):
        a = pdx.simulate_sc_ldpc(e, l, r, L, M, True, False, bounded, False, 5000, 10 ** 9, [], **kw)
        b = pdx.simulate_sc_ldpc(e, l, r, L, M, True, False, bounded, False, 5000, 10 ** 9, [], _batch_factory=factory, **kw)
        assert all((np.asarray(a[i]) == np.asarray(b[i])).all() for i in range(13)), (bounded, a, b)


def test_ber_sim_two_ranks_write_the_file_of_one_process(tmp_path):
    import os
    import socket
    import subprocess
    import sys
    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    driver = os.path.join(root, "tests", "ss_multi_rank_driver.py")
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    if torch.cuda.device_count() < 2:
        env["SCLDPC_DIST_BACKEND"] = "gloo"
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    text = {}
    for nproc in (1, 2):
        out = tmp_path / str(nproc)
        out.mkdir()
        cmd = [sys.executable, driver, str(out)] if nproc == 1 else \
            [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
             "--master-port", str(port), driver, str(out)]
        r = subprocess.run(cmd, cwd=str(out), env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
        text[nproc] = open(out / "ber.txt", "rb").read()
    assert text[1] == text[2] and len(text[1].splitlines()) == 3


# ---- bad arguments ---------------------------------------------------------------------------------------------------
def test_bad_arguments_are_rejected():
    import ctypes
    from fl_scaling_sc_ldpc_b200 import _lib
    ens = eng.Ensemble(4, 8, 12, 48)
    fbg = eng.FrameBatch(ens, 1, 64).generate_graphs(3, first_graph_id=3)
    counted = np.ones(12, bool)
    with pytest.raises(ValueError):
        eng.decode_bp_stream(fbg, 100, 0.47, 1, stopping_sets=counted, caps=[3, 9])
    with pytest.raises(ValueError):
        eng.decode_bp_stream(fbg, 100, 0.47, 1, stopping_sets=counted, max_it=9)
    with pytest.raises(eng.ScldpcError):                      # messages
        eng.decode_bp_stream(fbg, 100, 0.47, 1, stopping_sets=counted, messages=True)
    for is_term, bad in ((True, -1), (True, (12 + 3) * ens.cns_pos + 1), (False, 12 * ens.cns_pos + 1)):
        with pytest.raises(eng.ScldpcError):
            eng.decode_bp_stream(fbg, 100, 0.47, 1, is_term=is_term, stopping_sets=counted, unscanned_head_cns=bad)
    for is_term, ok in ((True, (12 + 3) * ens.cns_pos), (False, 12 * ens.cns_pos)):   # the whole swept range is fine
        eng.decode_bp_stream(fbg, 100, 0.47, 1, is_term=is_term, stopping_sets=counted, unscanned_head_cns=ok)
    # the C ABI itself: cfg->max_it != 0 and NULL outputs
    L = _lib.lib()
    eps = np.full(1, 0.47)
    a0 = np.zeros(1, np.int32)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p).value
    import torch
    need = L.scldpc_bp_stream_stopping_sets_workspace_bytes(ctypes.byref(fbg.dims))
    assert need > L.scldpc_bp_stream_workspace_bytes(ctypes.byref(fbg.dims), 0)
    torch_ws = torch.empty(need, dtype=torch.uint8, device=fbg.device)
    ws = ctypes.c_void_p(torch_ws.data_ptr())
    iters = torch.zeros((1, 100), dtype=torch.int32, device=fbg.device)
    recs = torch.zeros((1, 100, 4), dtype=torch.int32, device=fbg.device)
    good = _lib.StreamSsOut(iters.data_ptr(), recs.data_ptr())
    cp = np.ones(12, np.uint8)

    def call(max_it=0, out=good):
        cfg = _lib.StreamCfg(100, 0, 1, 0, 0, ptr(eps), ptr(a0), ptr(a0), ptr(a0), 1, 0, max_it)
        return L.scldpc_bp_stream_stopping_sets(ctypes.byref(fbg.dims), ctypes.byref(fbg.cbatch), ctypes.byref(cfg),
                                                cp.ctypes.data_as(ctypes.c_void_p), 0, ctypes.byref(out) if out is not None else None,
                                                ws, ctypes.c_size_t(need), None, eng.engine._stream())
    assert call() == 0
    assert call(max_it=9) == -1 and b"max_it" in L.scldpc_last_error()
    assert call(out=None) == -1
    assert call(out=_lib.StreamSsOut(iters.data_ptr(), None)) == -1
    assert call(out=_lib.StreamSsOut(None, recs.data_ptr())) == -1
    torch.cuda.synchronize()
