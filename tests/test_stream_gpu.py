"""Frame streams (lane recycling): every frame id must decode exactly as in a synchronous batch of the same channel
realisations -- iterations, residual, block and expurgated statistics -- whatever lane it happened to land in."""
import numpy as np
import pytest

import fl_scaling_sc_ldpc_b200 as eng
from tests import util

pytestmark = pytest.mark.gpu
KEYS = ("iters", "residual", "blocks_err", "erasures_exp", "blocks_err_exp")


@pytest.fixture(autouse=True, params=["node_state", "messages"])
def stream_kernels(request, monkeypatch):
    """both stream implementations: the node-state sweeps (bp_node_kernels.cu, default) and the message-passing sweeps"""
    monkeypatch.setenv("SCLDPC_STREAM_NODE", "1" if request.param == "node_state" else "0")
    return request.param


def sync_reference(fb_graphs, ens, B, eps, seed, is_term, doping=(), max_it=0):
    """frames 0..B-1 decoded 128 at a time with the synchronous message-passing decoder on the same graphs"""
    import os
    old = os.environ.get("SCLDPC_FULL_NODE")
    os.environ["SCLDPC_FULL_NODE"] = "0"
    try:
        return _sync_reference(fb_graphs, ens, B, eps, seed, is_term, doping, max_it)
    finally:
        if old is None:
            del os.environ["SCLDPC_FULL_NODE"]
        else:
            os.environ["SCLDPC_FULL_NODE"] = old


def _sync_reference(fb_graphs, ens, B, eps, seed, is_term, doping=(), max_it=0):
    G = fb_graphs.n_graphs
    out = {k: np.zeros((G, B), np.int32) for k in KEYS}
    for f0 in range(0, B, 128):
        k = min(128, B - f0)
        fb = eng.FrameBatch(ens, G, k, 2)
        fb.vn_cn.copy_(fb_graphs.vn_cn); fb._build_tables()
        fb.generate_erasures(eps, seed, first_graph_id=3, doping_points=doping, first_frame=f0)
        r = eng.decode_bp_full(fb, max_it, is_term)
        for key in KEYS:
            out[key][:, f0:f0 + k] = getattr(r, key)
    return out


@pytest.mark.parametrize("L,M,lanes,B,eps", [(10, 50, 128, 700, [0.44, 0.50]), (16, 64, 100, 333, [0.47, 0.41]), (8, 32, 256, 256, [0.5, 0.3]),
                                               (6, 16, 64, 150, [1.0, 0.0]), (12, 40, 512, 1500, [0.46, 0.52]),
                                               (12, 40, 1024, 3000, [0.46, 0.50])])
def test_stream_equals_synchronous_batches(L, M, lanes, B, eps):
    ens = eng.Ensemble(4, 8, L, M)
    fbg = eng.FrameBatch(ens, 2, lanes).generate_graphs(21, first_graph_id=3)
    for is_term in (True, False):
        ref = sync_reference(fbg, ens, B, eps, 55, is_term)
        for H in (1, 7, 16):
            s = eng.decode_bp_stream(fbg, B, eps, 55, first_graph_id=3, is_term=is_term, harvest_every=H)
            for key in KEYS:
                assert (getattr(s, key) == ref[key]).all(), (is_term, H, key)
            assert s.iters_launched >= ref["iters"].max()


def test_stream_with_doping_and_other_degrees():
    ens = eng.Ensemble(3, 6, 12, 48)
    fbg = eng.FrameBatch(ens, 1, 128).generate_graphs(5, first_graph_id=3)
    ref = sync_reference(fbg, ens, 400, 0.42, 9, True, doping=[5])
    s = eng.decode_bp_stream(fbg, 400, 0.42, 9, first_graph_id=3, doping_points=[5])
    for key in KEYS:
        assert (getattr(s, key) == ref[key]).all(), key
    ref = sync_reference(fbg, ens, 130, 0.45, 9, True, doping={2: 0.5})
    s = eng.decode_bp_stream(fbg, 130, 0.45, 9, first_graph_id=3, doping_points={2: 0.5})
    for key in KEYS:
        assert (getattr(s, key) == ref[key]).all(), key


@pytest.mark.parametrize("dv,dc,L,M", [(4, 12, 9, 48), (5, 10, 8, 40), (3, 9, 10, 36)])
def test_stream_every_instantiated_degree(dv, dc, L, M):
    """the degree pairs the kernels are instantiated for, terminated and truncated, 192 lanes / 500 frames"""
    ens = eng.Ensemble(dv, dc, L, M)
    fbg = eng.FrameBatch(ens, 2, 192).generate_graphs(13, first_graph_id=3)
    eps = [0.9 * dv / dc, 1.15 * dv / dc]
    for is_term in (True, False):
        ref = sync_reference(fbg, ens, 500, eps, 21, is_term)
        s = eng.decode_bp_stream(fbg, 500, eps, 21, first_graph_id=3, is_term=is_term)
        for key in KEYS:
            assert (getattr(s, key) == ref[key]).all(), (is_term, key)


@pytest.mark.parametrize("cap", [1, 2, 9, 40])
def test_capped_stream_equals_capped_synchronous_batches(cap, stream_kernels):
    """lane recycling with an iteration cap per frame (do {} while (iter < MaxNumIt), BP_FULL.c:1066): frames that hit the
    cap keep the erased set of that iteration while they wait for the harvest"""
    ens = eng.Ensemble(4, 8, 12, 48)
    fbg = eng.FrameBatch(ens, 2, 192).generate_graphs(17, first_graph_id=3)
    eps = [0.46, 0.51]
    if stream_kernels == "messages":
        with pytest.raises(eng.ScldpcError):
            eng.decode_bp_stream(fbg, 64, eps, 5, first_graph_id=3, max_it=cap)
        return
    for is_term in (True, False):
        ref = sync_reference(fbg, ens, 600, eps, 5, is_term, max_it=cap)
        for H in (0, 1, 5):
            s = eng.decode_bp_stream(fbg, 600, eps, 5, first_graph_id=3, is_term=is_term, harvest_every=H, max_it=cap)
            for key in KEYS:
                assert (getattr(s, key) == ref[key]).all(), (is_term, H, key)
        assert ref["iters"].max() <= cap


def test_stream_full_size_sample():
    """(4,8), L=50, M=10000, eps=0.47: a 256-lane stream of 384 frames against synchronous decoding of the same frames"""
    ens = eng.Ensemble(4, 8, 50, 10000)
    fbg = eng.FrameBatch(ens, 1, 256, 4).generate_graphs(77, first_graph_id=3)
    s = eng.decode_bp_stream(fbg, 384, 0.47, 78, first_graph_id=3)
    out = {k: [] for k in KEYS}
    for f0 in (0, 128, 256):
        fb = eng.FrameBatch(ens, 1, 128, 2)
        fb.vn_cn.copy_(fbg.vn_cn); fb._build_tables()
        fb.generate_erasures(0.47, 78, first_graph_id=3, first_frame=f0)
        r = eng.decode_bp_full(fb, 0, True)
        for k in KEYS:
            out[k].append(getattr(r, k))
    for k in KEYS:
        assert (getattr(s, k) == np.concatenate(out[k], axis=1)).all(), k


def test_stream_matches_oracle_directly():
    """stream results against the CPU oracle (decodeBP restatement) on the very channel realisations the stream draws"""
    import oracle
    dv, dc, L, M, G, B = 4, 8, 14, 40, 2, 260
    ens = eng.Ensemble(dv, dc, L, M)
    fbg = eng.FrameBatch(ens, G, 128).generate_graphs(31, first_graph_id=3)
    eps = [0.45, 0.50]
    vn = fbg.vn_cn.cpu().numpy()
    for is_term in (True, False):
        s = eng.decode_bp_stream(fbg, B, eps, 77, first_graph_id=3, is_term=is_term)
        for f0 in range(0, B, 128):
            k = min(128, B - f0)
            fb = eng.FrameBatch(ens, G, k, 2)
            fb.vn_cn.copy_(fbg.vn_cn); fb._build_tables()
            fb.generate_erasures(eps, 77, first_graph_id=3, first_frame=f0)
            ch = fb.erasures_host()
            for g in range(G):
                gg = oracle.Graph(vn[g], L, M, ens.cns_pos, dv, dc)
                for f in range(0, k, 3):
                    o = oracle.decode_bp(gg, ch[g, f].astype(np.int32), 10 ** 9, int(is_term))
                    got = (s.iters[g, f0 + f], s.residual[g, f0 + f], s.blocks_err[g, f0 + f], s.erasures_exp[g, f0 + f], s.blocks_err_exp[g, f0 + f])
                    assert got == (o["iters"], o["residual"], o["blocks_err"], o["erasures_exp"], o["blocks_err_exp"]), (is_term, g, f0 + f)


@pytest.mark.parametrize("cap", [1, 7])
def test_resolution_list_overflow_falls_back_to_a_full_pass(cap, monkeypatch, stream_kernels):
    """per-warp resolution lists hold 1024 entries per iteration; a region that overflows flags the iteration and the next
    launch catches up with a pass over the plane.  SCLDPC_LIST_CAP forces that path on small graphs, for the stream kernel
    and for the list variant of the window / synchronous full-BP kernels"""
    if stream_kernels == "messages":
        pytest.skip("message-passing sweeps keep no lists")
    ens = eng.Ensemble(4, 8, 12, 48)
    fbg = eng.FrameBatch(ens, 2, 320).generate_graphs(29, first_graph_id=3)
    eps = [0.45, 0.50]
    ref = sync_reference(fbg, ens, 700, eps, 6, True)
    monkeypatch.setenv("SCLDPC_LIST_CAP", str(cap))
    for H in (1, 9):
        s = eng.decode_bp_stream(fbg, 700, eps, 6, first_graph_id=3, harvest_every=H)
        for key in KEYS:
            assert (getattr(s, key) == ref[key]).all(), (H, key)
    sc = eng.decode_bp_stream(fbg, 300, eps, 6, first_graph_id=3, max_it=5)
    monkeypatch.delenv("SCLDPC_LIST_CAP")
    sc_ref = eng.decode_bp_stream(fbg, 300, eps, 6, first_graph_id=3, max_it=5)
    for key in KEYS:
        assert (getattr(sc, key) == getattr(sc_ref, key)).all(), key
    # synchronous full BP and a long window (list variant) with overflowing regions
    fb = eng.FrameBatch(ens, 2, 128)
    fb.vn_cn.copy_(fbg.vn_cn); fb._build_tables()
    fb.generate_erasures(eps, 6, first_graph_id=3)
    a = eng.decode_bp_full(fb, 0, True)
    w = eng.decode_bp_window(fb, 9, 4, 10)
    monkeypatch.setenv("SCLDPC_LIST_CAP", str(cap))
    b = eng.decode_bp_full(fb, 0, True)
    w2 = eng.decode_bp_window(fb, 9, 4, 10)
    for key in KEYS:
        assert (getattr(a, key) == getattr(b, key)).all() and (getattr(w, key) == getattr(w2, key)).all(), key
    assert bool((a.erased_words == b.erased_words).all()) and bool((w.erased_words == w2.erased_words).all())


@pytest.mark.parametrize("lanes,B,cap", [(1024, 1300, 0), (512, 512, 0), (256, 700, 9), (1024, 1024, 0)])
def test_lane_compaction_in_the_tail_changes_nothing(lanes, B, cap, stream_kernels):
    """Once a graph has handed out its last frame the live frames move into the lowest 128-lane chunks (ns_compact_*): the
    per-frame results must not depend on it, and it must really happen (several times: 8 -> 4 -> 2 -> 1 chunks)"""
    if stream_kernels == "messages":
        pytest.skip("the message-passing streams do not compact")
    ens = eng.Ensemble(4, 8, 14, 48)
    fbg = eng.FrameBatch(ens, 3, lanes).generate_graphs(41, first_graph_id=3)
    eps = [0.44, 0.49, 0.52]                                     # the last one stalls: long-lived frames spread over all chunks
    ref = sync_reference(fbg, ens, B, eps, 9, True, max_it=cap)
    for H in (1, 4, 0):
        b = eng.decode_bp_stream(fbg, B, eps, 9, first_graph_id=3, harvest_every=H, max_it=cap)
        n_cmp, moved = util.stream_compactions(fbg)
        for key in KEYS:
            assert (getattr(b, key) == ref[key]).all(), (H, key)
        if H == 1 and cap == 0:                                  # every iteration is a chance to compact
            assert n_cmp >= 3 and moved >= n_cmp, (n_cmp, moved)


def test_many_graphs_finishing_at_different_times():
    """40 graphs with channels from easy to hopeless: graphs finish at very different times, the grids of the stream kernels
    shrink to the list of graphs still decoding (more than one ballot word of graphs)"""
    G = 40
    ens = eng.Ensemble(4, 8, 10, 32)
    fbg = eng.FrameBatch(ens, G, 64).generate_graphs(51, first_graph_id=3)
    eps = [0.30 + 0.24 * (g % 7) / 6 for g in range(G)]
    ref = sync_reference(fbg, ens, 150, eps, 13, True)
    for H in (1, 0):
        s = eng.decode_bp_stream(fbg, 150, eps, 13, first_graph_id=3, harvest_every=H)
        for key in KEYS:
            assert (getattr(s, key) == ref[key]).all(), (H, key)
