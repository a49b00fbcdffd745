"""Frame streams with checkpoints (scldpc_bp_stream_caps): slot k of one decode up to the largest cap must equal a capped
stream at caps[k], frame for frame, in all five outputs (the iteration count as min(iters, caps[k]))."""
import numpy as np
import pytest

import fl_scaling_sc_ldpc_b200 as eng
import oracle
from tests import util

pytestmark = pytest.mark.gpu
STATS = ("residual", "blocks_err", "erasures_exp", "blocks_err_exp")
CAP_LISTS = ([1, 2, 9, 40], [3, 7, 0], [5], [400, 800])


def assert_caps_equal_capped(fbg, B, eps, seed, caps, r=None, **kw):
    """one checkpointed stream (r, if the caller has decoded it already) against one capped stream per cap; returns it"""
    if r is None:
        r = eng.decode_bp_stream(fbg, B, eps, seed, first_graph_id=3, caps=caps, **kw)
    assert isinstance(r, eng.StreamCapsResult) and r.caps == tuple(caps)
    assert r.iters.shape == (fbg.n_graphs, B) and r.residual.shape == (len(caps), fbg.n_graphs, B)
    for k, T in enumerate(caps):
        ref = eng.decode_bp_stream(fbg, B, eps, seed, first_graph_id=3, max_it=max(0, T), **kw)
        its = np.minimum(r.iters, T) if T > 0 else r.iters
        assert (its == ref.iters).all(), (caps, T, "iters", kw)
        for key in STATS:
            assert (getattr(r, key)[k] == getattr(ref, key)).all(), (caps, T, key, kw)
    return r


@pytest.mark.parametrize("dv,dc,L,M", [(4, 8, 12, 48), (3, 6, 12, 48)])
@pytest.mark.parametrize("lanes,B", [(64, 700), (192, 500), (1024, 2500)])
def test_caps_equal_capped_streams(dv, dc, L, M, lanes, B):
    """both sides of the threshold (one graph each), terminated and truncated, fixed and adaptive harvest periods"""
    ens = eng.Ensemble(dv, dc, L, M)
    fbg = eng.FrameBatch(ens, 2, lanes).generate_graphs(17, first_graph_id=3)
    eps = [0.92 * dv / dc, 1.04 * dv / dc]
    paused = False
    for is_term in (True, False):
        for H in (0, 1, 5, 16):
            for caps in CAP_LISTS:
                r = assert_caps_equal_capped(fbg, B, eps, 5, caps, is_term=is_term, harvest_every=H)
                paused |= bool((r.iters > caps[0]).any()) and len(caps) > 1
    assert paused                                           # some frames ran past a checkpoint


def test_single_cap_is_the_plain_capped_stream():
    ens = eng.Ensemble(4, 8, 12, 48)
    fbg = eng.FrameBatch(ens, 2, 128).generate_graphs(3, first_graph_id=3)
    for T in (1, 6, 30):
        r = eng.decode_bp_stream(fbg, 400, [0.47, 0.5], 9, first_graph_id=3, caps=[T])
        s = eng.decode_bp_stream(fbg, 400, [0.47, 0.5], 9, first_graph_id=3, max_it=T)
        assert (r.iters == s.iters).all()
        for key in STATS:
            assert (getattr(r, key)[0] == getattr(s, key)).all(), (T, key)
    r = eng.decode_bp_stream(fbg, 400, [0.47, 0.5], 9, first_graph_id=3, caps=[0])
    s = eng.decode_bp_stream(fbg, 400, [0.47, 0.5], 9, first_graph_id=3)
    for key in ("iters",) + STATS:
        assert (np.asarray(getattr(r, key)).reshape(getattr(s, key).shape) == getattr(s, key)).all(), key


def test_caps_with_doping_and_exp_all():
    ens = eng.Ensemble(4, 8, 12, 48)
    fbg = eng.FrameBatch(ens, 2, 192).generate_graphs(23, first_graph_id=3)
    eps = [0.47, 0.53]
    for kw in (dict(doping_points=[5]), dict(doping_points={2: 0.5}), dict(exp_all=True), dict(exp_all=True, is_term=False)):
        for caps in ([1, 2, 9, 40], [3, 7, 0]):
            assert_caps_equal_capped(fbg, 600, eps, 11, caps, harvest_every=5, **kw)


def test_caps_against_the_oracle():
    """a few frames per graph compared directly with decodeBP at every cap, on the graph and channel pulled from the device"""
    ens = eng.Ensemble(4, 8, 10, 40)
    G, F = 2, 96
    fbg = eng.FrameBatch(ens, G, F).generate_graphs(29, first_graph_id=3)
    eps = [0.47, 0.52]
    caps = [1, 4, 13, 0]
    r = eng.decode_bp_stream(fbg, F, eps, 31, first_graph_id=3, caps=caps, harvest_every=3)
    fb = eng.FrameBatch(ens, G, F)
    fb.vn_cn.copy_(fbg.vn_cn); fb._build_tables()
    fb.generate_erasures(eps, 31, first_graph_id=3)
    chan = fb.erasures_host()
    vn = fbg.vn_cn.cpu().numpy()
    checked = 0
    for g in range(G):
        gr = oracle.Graph(vn[g], ens.L, ens.M, ens.cns_pos, ens.dv, ens.dc)
        for f in range(0, F, 3):
            for k, T in enumerate(caps):
                o = oracle.decode_bp(gr, chan[g, f].astype(np.int32), T if T > 0 else 10 ** 9, 1)
                assert (min(r.iters[g, f], T) if T > 0 else r.iters[g, f]) == o["iters"], (g, f, T)
                for key in STATS:
                    assert getattr(r, key)[k, g, f] == o[key], (g, f, T, key)
                checked += 1
    assert checked == G * 32 * len(caps)


def test_caps_full_size_with_lane_compaction():
    """(4,8) L=50 M=10000, eps = 0.49: 1024 lanes and 2048 frames, so the tail of the stream compacts lanes that have been
    paused; caps [100, 175, 350, unlimited] against capped streams"""
    ens = eng.Ensemble(4, 8, 50, 10000)
    fbg = eng.FrameBatch(ens, 1, 1024).generate_graphs(41, first_graph_id=3)
    r = assert_caps_equal_capped(fbg, 2048, 0.49, 43, [100, 175, 350, 0])
    assert (r.iters > 350).any() and (r.residual[0] > r.residual[2]).any()


def test_caps_with_lane_compaction_equal_capped_streams():
    """512 lanes in the tail of 3000 frames per graph: the checkpointed stream compacts its lanes"""
    ens = eng.Ensemble(4, 8, 16, 64)
    fbg = eng.FrameBatch(ens, 2, 512).generate_graphs(47, first_graph_id=3)
    eps, caps = [0.48, 0.5], [2, 20, 60, 0]
    r = eng.decode_bp_stream(fbg, 3000, eps, 5, first_graph_id=3, caps=caps, harvest_every=4)
    n_cmp, moved = util.stream_compactions(fbg)          # before the capped streams reuse the workspace
    assert n_cmp >= 1 and moved >= n_cmp, (n_cmp, moved)
    assert_caps_equal_capped(fbg, 3000, eps, 5, caps, r=r, harvest_every=4)


def test_bad_caps_are_rejected():
    ens = eng.Ensemble(4, 8, 12, 48)
    fbg = eng.FrameBatch(ens, 1, 64).generate_graphs(3, first_graph_id=3)
    for caps in ([9, 3], [3, 3], [0, 5], [-1, 4], list(range(1, 18)), []):
        with pytest.raises(eng.ScldpcError):
            eng.decode_bp_stream(fbg, 100, 0.47, 1, caps=caps)
    with pytest.raises(eng.ScldpcError):
        eng.decode_bp_stream(fbg, 100, 0.47, 1, caps=[3, 9], max_it=9)
    with pytest.raises(eng.ScldpcError):
        eng.decode_bp_stream(fbg, 100, 0.47, 1, caps=[3, 9], messages=True)
    r = eng.decode_bp_stream(fbg, 100, 0.47, 1, caps=list(range(1, 17)))       # 16 caps are fine
    assert r.residual.shape == (16, 1, 100)


# ---- bp_lim_iter --caps ----------------------------------------------------------------------------------------------
def _bp_lim_iter(out, max_it, extra):
    import os
    from fl_scaling_sc_ldpc_b200 import bp_cli
    os.makedirs(out, exist_ok=True)
    bp_cli.run("bp_lim_iter", ["3", "0", "0", str(max_it), "--L", "12", "--M", "24", "--outdir", str(out), "--seed", "9",
                               "--frames-per-graph", "300", "--graphs-per-batch", "2", "--stream", "on"] + extra)
    return {n: open(os.path.join(out, n)).read() for n in os.listdir(out)}


def test_cli_caps_files_equal_separate_runs_without_early_stops(tmp_path):
    extra = ["--points", "2", "--eps-ini", "0.48", "--eps-delta", "0.03", "--min-frame-err", "1000000", "--max-frames", "1500"]
    shared = _bp_lim_iter(tmp_path / "caps", 4, extra + ["--caps", "30,2,9,4"])
    assert len(shared) == 4
    for T in (2, 4, 9, 30):
        (name, text), = _bp_lim_iter(tmp_path / f"sep{T}", T, extra).items()
        assert "_%dit_" % T in name and shared[name] == text, T
    rows = [shared[n].splitlines()[1].split() for n in sorted(shared, key=lambda n: int(n.split("it_")[0].rsplit("_", 1)[1]))]
    assert [int(r[11]) for r in rows] == sorted((int(r[11]) for r in rows), reverse=True)   # frame errors fall with the cap


def test_cli_caps_with_early_stops(tmp_path):
    """every cap stops at its own frame: the first point of every file and every point of the largest cap's file are
    those of separate runs"""
    extra = ["--points", "3", "--eps-ini", "0.47", "--eps-delta", "0.02", "--min-frame-err", "40", "--max-frames", "3000"]
    caps = (3, 6, 12, 60)
    shared = _bp_lim_iter(tmp_path / "caps", 60, extra + ["--caps", "3,6,12"])
    frames = set()
    for T in caps:
        (name, text), = _bp_lim_iter(tmp_path / f"sep{T}", T, extra).items()
        a, b = shared[name].splitlines(), text.splitlines()
        assert len(a) == len(b) == 4
        assert a[:2] == b[:2], T
        if T == caps[-1]:
            assert a == b
        frames.add(int(a[1].split()[9]))
    assert len(frames) > 1                                  # the caps did stop at different frames


def test_cli_caps_two_ranks_write_the_files_of_one_process(tmp_path):
    import os
    import socket
    import subprocess
    import sys
    import torch
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    driver = os.path.join(root, "tests", "caps_multi_rank_driver.py")
    env = dict(os.environ, PYTHONPATH=root + os.pathsep + os.environ.get("PYTHONPATH", ""))
    if torch.cuda.device_count() < 2:
        env["SCLDPC_DIST_BACKEND"] = "gloo"
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    files = {}
    for nproc in (1, 2):
        out = tmp_path / str(nproc)
        out.mkdir()
        cmd = [sys.executable, driver, str(out)] if nproc == 1 else \
            [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
             "--master-port", str(port), driver, str(out)]
        r = subprocess.run(cmd, cwd=str(out), env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
        files[nproc] = {n: open(out / n, "rb").read() for n in os.listdir(out)}
    assert len(files[1]) == 3 and files[1] == files[2]
