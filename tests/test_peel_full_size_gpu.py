"""The peeling decoder (peel_kernels.cu) and the stopping-set bookkeeping (ss_kernels.cu) at the sizes bench.py runs,
against the CPU oracle, value for value.

Paths that only these sizes reach, and where each is checked:
  * frames handed out by the work-stealing counter once every warp has had its first frame (G*F above the number of
    CN-state slots of the launch): test_bench_step_config_1, test_M10000_config_1_geometry, test_forced_work_stealing
  * lanes above 127 (n_words = 16) and frame ids >= 2^32 (the high word of the Philox counter): test_bench_step_config_1
  * the degree-one bitmap in shared memory (M = 1000 non-terminated) and in global memory, unforced (M = 1000 terminated,
    M = 10^4): test_M1000_full_length, test_M10000_*
  * more than one level-2 count per lane (more than 2^20 CNs), including a partly filled last lane: test_l2q_*
  * trajectory ends: stalls, the tail fill, num_steps not a multiple of 4, num_steps = 0: test_step_counts
  * stopping sets with n_words 2, 8 and 16 and the unscanned head of unbounded runs: test_stopping_sets_M1000
The oracle is oracle.peel_trajectory_fast (a Fenwick tree over the degree-one CNs, pinned to the scanning
oracle.peel_trajectory by tests/test_peel_oracle_cpu.py); the scanning one is a second witness on a few M = 1000 frames."""
import ctypes
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
import torch

import fl_scaling_sc_ldpc_b200 as eng
import oracle
from fl_scaling_sc_ldpc_b200 import _lib
from fl_scaling_sc_ldpc_b200 import peeling_decoding as pdx

pytestmark = pytest.mark.gpu
DV, DC, L = 4, 8, 50
SEED = 0x5C1D9C                     # bench.py's default --seed


def _pool_map(fn, jobs):
    # the oracle runs outside the GIL (ctypes): a thread per host core
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        return list(ex.map(fn, jobs))


def _free():
    torch.cuda.synchronize()
    torch.cuda.empty_cache()


def _state_words(n_cn_all, total_size):
    """u64 words of CN state per slot, and whether the degree-one bitmap lives in global memory: the bitmap plus its two
    count levels take 4 B per 32 / 1024 / 32768 CNs, and above 3400 B per warp the bitmap moves behind the CN state"""
    w = (total_size + 31) // 32
    a = (w + 31) // 32
    b = (a + 31) // 32
    big = 4 * (w + a + b) > 3400
    return n_cn_all + ((w + 1) // 2 if big else 0), big


def _slots(fb, total_size):
    """CN-state slots (= warps, = frames decoded concurrently) of a launch over fb, from the workspace size"""
    need = _lib.lib().scldpc_peel_workspace_bytes(ctypes.byref(fb.dims), fb.ens.nk, total_size)
    assert need > 0, _lib.lib().scldpc_last_error().decode()
    sw, _ = _state_words(fb.ens.nk, total_size)
    assert (need // 8 - 1) % sw == 0, (need, sw)
    return (need // 8 - 1) // sw


def _lane_erasures(fb, g, f):
    """channel realisation of lane f of graph g, read straight from the bit-sliced words"""
    return ((fb.chan[g, :, f >> 6] >> (f & 63)) & 1).to(torch.uint8).cpu().numpy()


def _popcounts(fb):
    """erased VNs per frame, int64 [G][F]"""
    sh = torch.arange(64, device=fb.device)
    out = torch.zeros((fb.n_graphs, 64 * fb.n_words), dtype=torch.int64, device=fb.device)
    for g in range(fb.n_graphs):
        for w in range(fb.n_words):
            out[g, 64 * w:64 * (w + 1)] = ((fb.chan[g, :, w].unsqueeze(-1) >> sh) & 1).sum(0)
    return out[:, : fb.n_frames].cpu().numpy()


def _check_frames(fb, total_size, steps, seed, first_frame, r1, rec, ner, frames, slow=()):
    """r1 row, recovered and n_erased of every (g, f) in frames against the fast oracle (and the scanning one for the
    frames in slow); r1/rec/ner are the device tensors of peel_batch"""
    vn = {g: fb.vn_cn[g].cpu().numpy() for g in sorted({g for g, _ in frames})}
    F, nk = fb.n_frames, fb.ens.nk
    jobs = []
    for g, f in frames:
        er = _lane_erasures(fb, g, f)
        jobs.append((g, f, vn[g], er, pdx.philox_picks(seed, first_frame + g * F + f, steps)))
    outs = _pool_map(lambda j: oracle.peel_trajectory_fast(j[2], j[3], total_size, nk, steps, j[4]), jobs)
    gi = torch.tensor([g for g, _ in frames], device=r1.device)
    fi = torch.tensor([f for _, f in frames], device=r1.device)
    rows = r1[gi, fi].cpu().numpy()
    rec_h, ner_h = rec.cpu().numpy(), ner.cpu().numpy()
    for k, ((g, f, _, er, _), (o_r1, o_rec)) in enumerate(zip(jobs, outs)):
        assert (rows[k] == o_r1).all(), (g, f, int(np.flatnonzero(rows[k] != o_r1)[0]))
        assert rec_h[g, f] == o_rec and ner_h[g, f] == er.sum(), (g, f, rec_h[g, f], o_rec, ner_h[g, f], er.sum())
    if slow:
        sj = [j for j in jobs if (j[0], j[1]) in set(slow)]
        assert len(sj) == len(slow)
        souts = _pool_map(lambda j: oracle.peel_trajectory(j[2], j[3], total_size, nk, steps, j[4]), sj)
        for j, (o_r1, o_rec) in zip(sj, souts):
            k = frames.index((j[0], j[1]))
            assert (rows[k] == o_r1).all() and rec_h[j[0], j[1]] == o_rec, (j[0], j[1])
    return rows, outs


# ---------------------------------------------------------------------------------------------------------------------
# peeling trajectories
# ---------------------------------------------------------------------------------------------------------------------
def test_bench_step_config_1():
    """exactly bench.py's peeling_M1000 call (first timed step): 16 new graphs x 1024 frames, seeds --seed + 0/1/2"""
    M, e, G, F = 1000, 0.48, 16, 1024
    ens = eng.Ensemble(DV, DC, L, M)
    _, _, total_size, steps = pdx._peel_geometry(e, DV, DC, L, M, False)
    fb = eng.FrameBatch(ens, G, F)
    assert fb.n_words == 16
    gid = (9 << 20) + 2 * G
    fb.generate_graphs(SEED, first_graph_id=gid)
    fb.generate_erasures(e, SEED + 1, first_graph_id=gid)
    first = gid * F
    assert first >= 1 << 32                                       # the Philox counter's high word is nonzero
    slots = _slots(fb, total_size)
    assert G * F > slots                                          # frames beyond the first wave come from the counter
    assert not _state_words(ens.nk, total_size)[1]                # bitmap in shared memory
    r1, rec, ner = pdx.peel_batch(ens, fb, total_size, steps, SEED + 2, first)
    frames = [(g, f) for g in (0, 6, 11) for f in (0, 63, 64, 127, 128, 1023)]
    frames += [(G - 1, f) for f in range(F - 5, F)]                # the last graph's last frames
    late = [slots, slots + 1, slots + 37, (slots + G * F) // 2, G * F - 100, G * F - 7]
    frames += [(fr // F, fr % F) for fr in late]
    rng = np.random.default_rng(1)
    frames += [(int(g), int(f)) for g, f in zip(rng.integers(0, G, 8), rng.integers(128, F, 8))]
    frames = list(dict.fromkeys(frames))
    assert sum(g * F + f >= slots for g, f in frames) >= 10
    assert sum(f >= 128 for _, f in frames) >= 10
    _check_frames(fb, total_size, steps, SEED + 2, first, r1, rec, ner, frames, slow=[(0, 1023), (G - 1, F - 1), (slots // F, slots % F)])
    # every frame: n_erased is the channel's popcount, and what peeling leaves is the residual of truncated BP
    rec_h, ner_h = rec.cpu().numpy(), ner.cpu().numpy()
    assert (ner_h == _popcounts(fb)).all()
    bp = eng.decode_bp_full(fb, eng.UNLIMITED, is_term=False)
    assert (ner_h - rec_h == bp.residual).all()
    del r1, rec, ner, fb, bp
    _free()


class _Run:
    """one peel_batch over freshly generated graphs and channels; picks from seed + 2, frame ids from first_frame"""

    def __init__(self, M, term, eps, G, F, n_words, seed, first_frame=0):
        self.ens = eng.Ensemble(DV, DC, L, M)
        self.term, self.seed, self.first = term, seed + 2, first_frame
        _, _, self.total_size, self.steps = pdx._peel_geometry(max(np.atleast_1d(eps)), DV, DC, L, M, term)
        self.fb = eng.FrameBatch(self.ens, G, F, n_words).generate_graphs(seed).generate_erasures(eps, seed + 1)
        self.r1, self.rec, self.ner = pdx.peel_batch(self.ens, self.fb, self.total_size, self.steps, self.seed, first_frame)

    def check(self, frames, slow=()):
        return _check_frames(self.fb, self.total_size, self.steps, self.seed, self.first, self.r1, self.rec, self.ner, frames, slow)


def test_M10000_config_1_geometry():
    """bench.py's peeling_M10000 shape: non-terminated, eps = 0.48, n_words = 16, more frames than slots, full 290000
    steps (frames here peel through most of the chain: ~229 000 recovered VNs on average)"""
    M, e, F = 10000, 0.48, 1024
    ens = eng.Ensemble(DV, DC, L, M)
    _, _, total_size, steps = pdx._peel_geometry(e, DV, DC, L, M, False)
    assert steps == 290000 and _state_words(ens.nk, total_size)[1]          # bitmap in global memory
    probe = eng.FrameBatch(ens, 1, 1, 2)
    probe.dims.n_graphs, probe.dims.n_frames, probe.dims.n_words = 64, F, 16
    G = _slots(probe, total_size) // F + 1                                  # just enough graphs to exceed the slots
    del probe
    fb = eng.FrameBatch(ens, G, F).generate_graphs(SEED, first_graph_id=(9 << 20) + 100)
    fb.generate_erasures(e, SEED + 1, first_graph_id=(9 << 20) + 100)
    slots = _slots(fb, total_size)
    assert G * F > slots and fb.n_words == 16
    first = ((9 << 20) + 100) * F
    r1, rec, ner = pdx.peel_batch(ens, fb, total_size, steps, SEED + 2, first)
    frames = [(0, 0), (0, 1023), (1, 200), (G // 2, 700), (slots // F, slots % F), ((slots + 5) // F, (slots + 5) % F),
              (G - 1, 1000), (G - 1, F - 1)]
    _, outs = _check_frames(fb, total_size, steps, SEED + 2, first, r1, rec, ner, frames)
    assert max(o[1] for o in outs) > 100000                                  # long trajectories, not only early stalls
    assert (ner.cpu().numpy() == _popcounts(fb)).all()
    del r1, rec, ner, fb
    _free()


def test_M10000_terminated_peels_to_the_end():
    """terminated, eps = 0.45: frames peel every erased VN, so the global-bitmap path runs through whole trajectories"""
    run = _Run(10000, True, 0.45, 1, 128, 2, 61)
    assert _state_words(run.ens.nk, run.total_size)[1]
    frames = [(0, 0), (0, 63), (0, 64), (0, 127)]
    _, outs = run.check(frames)
    ner_h = run.ner.cpu().numpy()
    assert all(o[1] == ner_h[g, f] for (g, f), o in zip(frames, outs))       # finished
    del run
    _free()


@pytest.fixture(scope="module")
def m1000_terminated():
    """M = 1000 terminated (26 500 CNs: the bitmap just does not fit shared memory), full length, eps per graph from
    early stalls to full decoding"""
    run = _Run(1000, True, [0.44, 0.47, 0.49, 0.51], 4, 256, 4, 71, first_frame=(5 << 32) + 8)
    yield run
    del run
    _free()


def _check_all(run):
    """every frame of the run, two of them also against the scanning oracle; frames that peel to the end of the chain
    (terminated: every erased VN; non-terminated: up to the truncated tail) and frames that stall before a quarter of
    their erasures must both be there"""
    G, F = run.fb.n_graphs, run.fb.n_frames
    frames = [(g, f) for g in range(G) for f in range(F)]
    _, outs = run.check(frames, slow=[(0, 0), (G - 1, F - 1)])
    ner_h = run.ner.cpu().numpy()
    if run.term:
        assert any(o[1] == ner_h[g, f] for (g, f), o in zip(frames, outs))
    else:
        assert any(o[1] >= 0.9 * ner_h[g, f] for (g, f), o in zip(frames, outs))
    assert any(o[1] < ner_h[g, f] // 4 for (g, f), o in zip(frames, outs))


def test_M1000_terminated_full_length(m1000_terminated):
    run = m1000_terminated
    assert run.total_size == 26500 and _state_words(run.ens.nk, run.total_size)[1]
    _check_all(run)


def test_M1000_non_terminated_full_length():
    run = _Run(1000, False, [0.40, 0.45, 0.47, 0.49], 4, 256, 4, 81)
    assert run.total_size == 25000 and not _state_words(run.ens.nk, run.total_size)[1]
    _check_all(run)
    del run
    _free()


def test_variance_on_real_trajectories(m1000_terminated):
    """calc_nu_chunk_device on the M = 1000 terminated trajectories, two chunks, against the NumPy restatement of
    calc_nu_chunk / calc_var_chunk, bit for bit; theory = the mean r1"""
    r1 = m1000_terminated.r1
    r1 = r1.reshape(-1, r1.shape[-1])
    r1_h = r1.cpu().numpy().astype(np.int64)
    theory = r1_h.mean(axis=0)
    assert (theory > 0).any()
    M = 1000
    cut = 397
    ssq, cnt = pdx.calc_nu_chunk_device([r1[:cut], r1[cut:]], theory, M)
    crop = np.max(np.where(theory > 0)) + 1
    th = theory[theory > 0] / M
    S = len(th)
    assert crop == S

    def chunk(a):
        c = a[:, :S] / M - th
        c[a[:, :S] == 0] = np.nan
        return np.nansum(c ** 2, axis=0), np.sum(a[:, :S] != 0, axis=0)
    a, b = chunk(r1_h[:cut]), chunk(r1_h[cut:])
    assert np.array_equal(cnt, a[1] + b[1])
    assert np.array_equal(ssq, a[0] + b[0])


@pytest.mark.parametrize("slots_env,expect", [("2", 2), ("3", 4)])
def test_forced_work_stealing(monkeypatch, slots_env, expect):
    """two (three, rounded up to whole blocks: four) warps decode 600 frames: a warp's CN state, bitmap and counts must
    be fully reset between frames"""
    monkeypatch.setenv("SCLDPC_PEEL_SLOTS", slots_env)
    ens = eng.Ensemble(DV, DC, 20, 200)
    G, F, e = 3, 200, [0.40, 0.47, 0.52]
    _, _, total_size, steps = pdx._peel_geometry(0.52, DV, DC, 20, 200, True)
    fb = eng.FrameBatch(ens, G, F, 4).generate_graphs(91).generate_erasures(e, 92)
    assert _slots(fb, total_size) == expect
    r1, rec, ner = pdx.peel_batch(ens, fb, total_size, steps, 93, 1 << 33)
    frames = [(g, f) for g in range(G) for f in range(F)]
    _, outs = _check_frames(fb, total_size, steps, 93, 1 << 33, r1, rec, ner, frames)
    ner_h = ner.cpu().numpy()
    assert any(o[1] == ner_h[g, f] for (g, f), o in zip(frames, outs))
    assert any(o[1] < ner_h[g, f] for (g, f), o in zip(frames, outs))


@pytest.mark.parametrize("steps", [0, 1, 3, 4, 5])
def test_step_counts(steps):
    """r1 has steps + 1 entries, recovered counts the steps taken, and nothing is written past the last row"""
    lib = _lib.lib()
    ens = eng.Ensemble(DV, DC, 12, 64)
    G, F = 2, 70
    fb = eng.FrameBatch(ens, G, F, 2).generate_graphs(101).generate_erasures([0.003, 0.45], 102)
    total_size = ens.nk
    need = lib.scldpc_peel_workspace_bytes(ctypes.byref(fb.dims), ens.nk, total_size)
    ws = torch.empty(need, dtype=torch.uint8, device=fb.device)
    row = steps + 1
    guard = 4096
    r1 = torch.full((G * F * row + guard,), -7, dtype=torch.int32, device=fb.device)
    rec = torch.full((G * F + guard,), -7, dtype=torch.int32, device=fb.device)
    ner = torch.full((G * F + guard,), -7, dtype=torch.int32, device=fb.device)
    first = (1 << 32) - 3
    _lib.check(lib.scldpc_peel_trajectories(
        ctypes.byref(fb.dims), ctypes.c_void_p(fb.vn_cn.data_ptr()), ctypes.c_void_p(fb.chan.data_ptr()), ens.nk, total_size, steps,
        ctypes.c_uint64(104), ctypes.c_uint64(first), ctypes.c_void_p(r1.data_ptr()), ctypes.c_void_p(rec.data_ptr()),
        ctypes.c_void_p(ner.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ctypes.c_size_t(need), eng.engine._stream()))
    r1_h, rec_h, ner_h = r1.cpu().numpy(), rec.cpu().numpy(), ner.cpu().numpy()
    assert (r1_h[G * F * row:] == -7).all() and (rec_h[G * F:] == -7).all() and (ner_h[G * F:] == -7).all()
    er = fb.erasures_host()
    vn = fb.vn_cn.cpu().numpy()
    for g in range(G):
        for f in range(F):
            fr = g * F + f
            o_r1, o_rec = oracle.peel_trajectory_fast(vn[g], er[g, f], total_size, ens.nk, steps, pdx.philox_picks(104, first + fr, steps))
            assert (r1_h[fr * row:(fr + 1) * row] == o_r1).all(), (g, f)
            assert rec_h[fr] == o_rec <= steps and ner_h[fr] == er[g, f].sum(), (g, f)
    assert steps < 3 or (rec_h[:F] < steps).any()                 # eps = 0.003: frames that run out of degree-one CNs early


def test_size_limit_is_a_clean_error():
    """more than 2^23 CNs would need a fourth level of counts: the workspace query refuses, nothing is launched"""
    ens = eng.Ensemble(DV, DC, L, 400000)
    fb = eng.FrameBatch(ens, 1, 1, 2)
    lib = _lib.lib()
    assert lib.scldpc_peel_workspace_bytes(ctypes.byref(fb.dims), ens.nk, 1 << 23) > 0
    assert lib.scldpc_peel_workspace_bytes(ctypes.byref(fb.dims), ens.nk, (1 << 23) + 1) == 0
    _, _, total_size, steps = pdx._peel_geometry(0.48, DV, DC, L, 400000, False)
    assert total_size > 1 << 23
    launches = lib.scldpc_launch_count(0)
    with pytest.raises(_lib.ScldpcError, match="too large"):
        pdx.peel_batch(ens, fb, total_size, steps, 1, 0)
    assert lib.scldpc_launch_count(0) == launches
    del fb
    _free()


def test_l2q_M1e5_doped_to_the_end():
    """config 5 at M = 10^5 (2.5 M CNs, 77 level-2 counts: three per lane), doped {24, 25}, two frames over all
    2 900 000 steps"""
    M, e = 100000, 0.48
    ens = eng.Ensemble(DV, DC, L, M)
    _, _, total_size, steps = pdx._peel_geometry(e, DV, DC, L, M, False)
    assert steps == 2900000 and (total_size + 32767) // 32768 == 77
    fb = eng.FrameBatch(ens, 1, 2, 2).generate_graphs(515).generate_erasures(e, 516, doping_points=[24, 25])
    r1, rec, ner = pdx.peel_batch(ens, fb, total_size, steps, 517, 3 << 32)
    _, outs = _check_frames(fb, total_size, steps, 517, 3 << 32, r1, rec, ner, [(0, 0), (0, 1)])
    assert max(o[1] for o in outs) > 100000
    del r1, rec, ner, fb
    _free()


def test_l2q_partly_filled_last_lane():
    """M = 42 000 non-terminated: 1 050 000 CNs, 33 level-2 counts, two per lane: lanes 0-16 in use, lane 16 with one"""
    M, e = 42000, 0.45
    ens = eng.Ensemble(DV, DC, L, M)
    _, _, total_size, steps = pdx._peel_geometry(e, DV, DC, L, M, False)
    n_l2 = (total_size + 32767) // 32768
    assert total_size == 1050000 and n_l2 == 33 and (n_l2 + 31) // 32 == 2
    fb = eng.FrameBatch(ens, 1, 4, 2).generate_graphs(121).generate_erasures(e, 122)
    for f in range(2):                                        # the last level-2 count is in play from the start
        er = _lane_erasures(fb, 0, f).astype(bool)
        deg = np.bincount(fb.vn_cn[0].cpu().numpy()[er].reshape(-1), minlength=ens.nk)
        assert (deg[32 * 32768:total_size] == 1).sum() > 0
    r1, rec, ner = pdx.peel_batch(ens, fb, total_size, steps, 123, 0)
    _, outs = _check_frames(fb, total_size, steps, 123, 0, r1, rec, ner, [(0, 0), (0, 1), (0, 3)])
    assert max(o[1] for o in outs) > 100000
    del r1, rec, ner, fb
    _free()


# ---------------------------------------------------------------------------------------------------------------------
# stopping-set bookkeeping of simulate_sc_ldpc (PD.py:591-701)
# ---------------------------------------------------------------------------------------------------------------------
def _counted_vns(l, L_eff, num_positions, head, tail, M):
    """PD.py:661-666: VN position q is counted when one of its slots q..q+l-1 lies in [head, num_positions - tail) and
    all of them lie below num_positions"""
    ok = np.zeros(L_eff, bool)
    for q in range(L_eff):
        slots = range(q, q + l)
        ok[q] = any(head <= s < num_positions - tail for s in slots) and all(s < num_positions for s in slots)
    return ok, np.repeat(ok, M)


def _components(lost, vn_cn):
    """connected components of the lost VNs (two of them are connected when they share a CN): a label per lost VN"""
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    k = len(lost)
    cns = vn_cn[lost]
    u, inv = np.unique(cns.reshape(-1), return_inverse=True)
    rows = np.repeat(np.arange(k), cns.shape[1])
    a = coo_matrix((np.ones(rows.size, np.int8), (rows, k + inv.reshape(-1))), shape=(k + len(u), k + len(u)))
    _, lab = connected_components(a, directed=False)
    return lab[:k]


def _record(lost, vn_cn, M):
    """PD.py:668-691 per frame: (lost VNs, any component of more than two, VNs in those, positions they touch)"""
    if len(lost) == 0:
        return (0, 0, 0, 0), []
    lab = _components(lost, vn_cn)
    sizes = np.bincount(lab)
    sizes = sizes[sizes > 0]
    big = np.isin(lab, np.flatnonzero(np.bincount(lab) > 2))
    return (len(lost), int(big.any()), int(big.sum()), len(np.unique(lost[big] // M))), sizes.tolist()


SS_CASES = [  # (is_terminated, is_bounded, eps, frames_per_graph); eps of the unbounded runs from a short trial: ~35 % / ~80 % FER
    (True, True, 0.45, 128),
    (True, True, 0.48, 512),
    (True, False, 0.47, 1024),
    (False, False, 0.39, 512),
]


@pytest.mark.parametrize("term,bounded,eps,fpg", SS_CASES)
def test_stopping_sets_M1000(term, bounded, eps, fpg):
    l, r, M = DV, DC, 1000
    head, head_sched = (0, 0) if bounded else (20, 10)
    tail = 0 if term else 20
    L_eff = L + head + tail
    cns = M * l // r
    num_positions = L_eff + l - 1 if term else L_eff
    total_size = cns * num_positions
    nk = cns * (L_eff + l - 1)
    counted_pos, counted_vn = _counted_vns(l, L_eff, num_positions, head, tail, M)
    seed = 1300 + 7 * fpg + int(term) + 2 * int(bounded)
    made = []

    def factory(ens, G, fpg_, gid0):
        assert fpg_ == fpg and ens.L == L_eff
        fb = eng.FrameBatch(ens, G, fpg).generate_graphs(seed, first_graph_id=gid0).generate_erasures(eps, seed + 1, first_graph_id=gid0)
        made.append(fb)
        return fb

    n_graphs = 2 if fpg < 1024 else 1
    out = pdx.simulate_sc_ldpc(eps, l, r, L, M, term, False, bounded, False, n_graphs * fpg, 10 ** 9, [], frames_per_graph=fpg,
                               graphs_per_batch=1, progress=False, _batch_factory=factory)
    assert len(made) == n_graphs and made[0].n_words == eng.engine.words_for(fpg)
    # what the GPU left in the same batches, frame by frame, against the oracle's fixed point and the restated bookkeeping
    stripes = np.arange(L_eff) % 4 == 1                          # a second mask that cuts every residual into small pieces
    recs, classes, striped_classes = [], set(), set()
    for fb in made:
        res = eng.decode_bp_full(fb, eng.UNLIMITED, is_term=term, unscanned_head_cns=head_sched * cns)
        got = pdx.stopping_set_records(fb, res.erased_words, counted_pos)
        got_s = pdx.stopping_set_records(fb, res.erased_words, stripes)
        assert (got[:, fpg:] == 0).all()
        erased = res.erased()[0]
        ch = fb.erasures_host()[0]
        vn = fb.vn_cn[0].cpu().numpy().astype(np.int64)

        def frame(f):
            fp = oracle.peel_fixed_point(vn, ch[f], nk, head_sched * cns, total_size)
            lost = np.flatnonzero(fp.astype(bool) & counted_vn)
            lost_s = np.flatnonzero(fp.astype(bool) & np.repeat(stripes, M))
            return fp, _record(lost, vn, M), _record(lost_s, vn, M) if f % 4 == 0 else None
        for f, (fp, (rec, sizes), striped) in enumerate(_pool_map(frame, range(fpg))):
            assert (erased[f] == fp).all(), f
            assert tuple(int(x) for x in got[0, f]) == rec, (f, got[0, f], rec)
            classes |= {min(s, 3) for s in sizes}
            if striped is not None:
                rec_s, sizes_s = striped
                assert tuple(int(x) for x in got_s[0, f]) == rec_s, (f, got_s[0, f], rec_s)
                striped_classes |= {min(s, 3) for s in sizes_s}
            recs.append(rec)
    # the 13-tuple against the sequential accounting of those records (no early stop: max_fuckups is out of reach)
    n = len(recs)
    gen, blocks = n * L * M, n * L
    fails = [x for x in recs if x[0] >= 1]
    n_big, lost, lost_exp, blocks_exp = (sum(x[1] for x in fails), sum(x[0] for x in fails), sum(x[2] for x in fails),
                                         sum(x[3] for x in fails))
    want = (len(fails) / n, n_big / n, lost / gen, lost_exp / gen, n_big, n, lost_exp, gen, None, None, blocks_exp, blocks, blocks_exp / blocks)
    assert [out[i] for i in range(13) if i not in (8, 9)] == [want[i] for i in range(13) if i not in (8, 9)]
    assert not out[8].any() and not out[9].any()
    if eps >= 0.47 or not term:
        assert 0 < len(fails) < n and 3 in classes              # failed frames and components of more than two VNs
        assert striped_classes == {1, 2, 3}                     # components of one, two and more VNs all occurred
    del fb, res
    made.clear()
    _free()
