"""Drop-in for the SC-LDPC part of the reference's ``simulators_sc_ldpc/peeling_decoding/peeling_decoding.py`` (PD.py).

Same call signatures, same return values and file formats; the per-frame hot loops run on the GPU:

* ``simulate_peeling_decoder_ldpc`` (PD.py:705-789)  random-order peeling with the degree-one trajectory ``r1``
  -> ``csrc/peel_kernels.cu`` (one warp per frame, rank/select over a shared-memory bitmap).
* ``simulate_sc_ldpc`` (PD.py:591-701)  peeling to the fixed point (``sic_round`` scan) -> the residual of unlimited
  flooding BP (``csrc/bp_wave_kernels.cu``); lost-VN bookkeeping and stopping-set expurgation (PD.py:659-691,
  ``extract_stopping_sets`` PD.py:1077) on the residual sets of the failed frames.
* ``main_simulate_variance`` (PD.py:1264-1294), ``main_simulate_sc_ldpc`` (PD.py:1327-1353): same argv, same outputs.

Terminology follows the reference (written for coded slotted ALOHA): user = VN, slot = CN, g / e = erasure
probability, "fuckup" = frame error.  M is the number of VNs per position.

Differences, all additive: randomness comes from counter-based Philox streams (``set_seed``) instead of NumPy's /
``random``'s global state, so a run does not depend on how frames are batched or split over GPUs; keyword-only
arguments (``seed``, ``frames_per_graph``, ``first_frame``) were added.  Both ensembles are available (``is_protograph``);
the two protograph combinations that are broken upstream (soft doping, tail-biting) raise.
"""
from __future__ import annotations

import ctypes
import os
import pickle
import sys

import numpy as np
import torch

from . import _lib, engine

_state = {"seed": 0x5C1D9C}


def set_seed(seed: int):
    _state["seed"] = int(seed)


try:                                   # progress reporting like the reference (tqdm.trange + set_description)
    from tqdm import trange as _trange
except Exception:                      # pragma: no cover
    _trange = None


class _Progress:
    def __init__(self, total, enable=True):
        self.bar = _trange(total) if (_trange is not None and enable and sys.stderr.isatty()) else None

    def update(self, n, desc=None):
        if self.bar is not None:
            self.bar.update(n)
            if desc:
                self.bar.set_description(desc)

    def close(self):
        if self.bar is not None:
            self.bar.close()


def _check_ensemble(is_protograph, doping_points=(), is_tail_biting=False):
    """The reference's protograph path has two upstream defects that are not reproduced: soft doping raises a NameError
    (PD.py:227, undefined ``position``) and tail-biting takes CN indices modulo L instead of modulo L*cns (PD.py:205)."""
    if is_protograph and (isinstance(doping_points, dict) and len(doping_points) > 0):
        raise NotImplementedError("soft doping of the protograph ensemble is broken upstream (PD.py:227)")
    if is_protograph and is_tail_biting:
        raise NotImplementedError("tail-biting protograph ensemble is broken upstream (PD.py:205)")


def _doping_count(doping_points):
    return len(doping_points)


# ---------------------------------------------------------------------------------------------------------------------
# peeling trajectories
# ---------------------------------------------------------------------------------------------------------------------
def peel_batch(ens: engine.Ensemble, fb: engine.FrameBatch, total_size: int, num_steps: int, seed: int, first_frame: int,
               want_r1: bool = True):
    """One kernel launch over a resident batch.  Returns (r1 int32 tensor [G][F][num_steps+1] or None, recovered,
    n_erased as int32 tensors [G][F])."""
    lib = _lib.lib()
    G, F = fb.n_graphs, fb.n_frames
    n_cn_all = ens.nk
    need = lib.scldpc_peel_workspace_bytes(ctypes.byref(fb.dims), n_cn_all, total_size)
    if need == 0:
        raise _lib.ScldpcError(lib.scldpc_last_error().decode())
    ws = torch.empty(need, dtype=torch.uint8, device=fb.device)
    r1 = torch.empty((G, F, num_steps + 1), dtype=torch.int32, device=fb.device) if want_r1 else None
    rec = torch.zeros((G, F), dtype=torch.int32, device=fb.device)
    ner = torch.zeros((G, F), dtype=torch.int32, device=fb.device)
    _lib.check(lib.scldpc_peel_trajectories(
        ctypes.byref(fb.dims), ctypes.c_void_p(fb.vn_cn.data_ptr()), ctypes.c_void_p(fb.chan.data_ptr()), n_cn_all,
        int(total_size), int(num_steps), ctypes.c_uint64(seed), ctypes.c_uint64(first_frame),
        ctypes.c_void_p(r1.data_ptr()) if r1 is not None else None, ctypes.c_void_p(rec.data_ptr()),
        ctypes.c_void_p(ner.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ctypes.c_size_t(need), engine._stream()))
    return r1, rec, ner


def philox_picks(seed: int, frame_id: int, n: int) -> np.ndarray:
    """The 32-bit draws behind the picks of one frame (to feed the reference / the oracle the same pick sequence)."""
    out = np.zeros(max(1, n), np.uint32)
    _lib.lib().scldpc_philox_picks(ctypes.c_uint64(seed), ctypes.c_uint64(frame_id), int(n), out.ctypes.data_as(ctypes.c_void_p))
    return out[:n]


def _peel_geometry(e, l_deg, r_deg, L, M, is_terminated):
    cns_per_pos = int(l_deg / r_deg * M)
    num_positions = L + l_deg - 1 if is_terminated else L
    total_size = cns_per_pos * num_positions
    num_pd_steps = int(M * num_positions * (e + 0.1))          # float truncation as in PD.py:721
    return cns_per_pos, num_positions, total_size, num_pd_steps


def simulate_peeling_decoder_ldpc(e, l_deg, r_deg, L, M, is_terminated, is_protograph, num_repeats=None, doping_points=[],
                                  *, seed=None, frames_per_graph=1, first_frame=0, max_batch_frames=None, device_r1=False,
                                  _local=False):
    """PD.py:705-789.  Returns ``(None, r1, plrs)``: ``r1`` int64 [num_repeats][num_pd_steps+1] with the number of
    degree-one CNs after every peeling step, ``plrs`` float64 [num_repeats] the fraction of VNs left erased.

    The reference draws a new code per frame; ``frames_per_graph`` (default 1) keeps that."""
    _check_ensemble(is_protograph, doping_points)
    if not num_repeats:
        num_repeats = 100
    from . import dist as D
    rank, world = D.world()
    if world > 1 and not _local:
        # every rank peels a contiguous range of the frames (frame ids are global) and the results are all-gathered
        q = (num_repeats + world - 1) // world
        fpg_ = max(1, int(frames_per_graph))
        q = (q + fpg_ - 1) // fpg_ * fpg_                              # whole graphs per rank: frame F is (graph F // fpg, lane F % fpg)
        lo, hi = min(rank * q, num_repeats), min((rank + 1) * q, num_repeats)
        cols = _peel_geometry(e, l_deg, r_deg, L, M, is_terminated)[3] + 1
        if hi > lo:
            _, r1_l, plrs_l = simulate_peeling_decoder_ldpc(e, l_deg, r_deg, L, M, is_terminated, is_protograph, hi - lo, doping_points,
                                                            seed=seed, frames_per_graph=frames_per_graph, first_frame=first_frame + lo,
                                                            max_batch_frames=max_batch_frames, device_r1=True, _local=True)
            r1_l = torch.cat(r1_l, dim=0)
        else:
            r1_l, plrs_l = torch.zeros((0, cols), dtype=torch.int32, device=engine._device()), np.zeros(0)
        pad = torch.zeros((q, cols), dtype=torch.int32, device=r1_l.device)
        pad[: hi - lo] = r1_l
        pl = np.zeros(q)
        pl[: hi - lo] = plrs_l
        r1_all = D.allgather_tensor(pad)                                 # [world][q][cols]
        plrs = D.allgather_rows(pl).reshape(-1)
        r1_all = r1_all.reshape(world * q, cols)[:num_repeats]         # rank r filled rows [r*q, r*q + its count): contiguous
        plrs = plrs[:num_repeats]
        if device_r1:
            return None, [r1_all], plrs
        return None, r1_all.cpu().numpy().astype("int"), plrs
    seed = _state["seed"] if seed is None else seed
    cns_per_pos, num_positions, total_size, num_pd_steps = _peel_geometry(e, l_deg, r_deg, L, M, is_terminated)
    ens = engine.Ensemble(l_deg, r_deg, L, M)
    total_generated = (L - _doping_count(doping_points)) * M
    r1 = np.zeros((num_repeats, num_pd_steps + 1), dtype="int")
    plrs = np.zeros(num_repeats)
    fpg = int(frames_per_graph)
    if max_batch_frames is None:       # keep the r1 buffer of a batch around 2 GiB
        max_batch_frames = max(fpg, min(4096, (2 << 30) // (4 * (num_pd_steps + 1))))
    graphs_per_batch = max(1, max_batch_frames // fpg)
    done = 0
    prog = _Progress(num_repeats)
    r1_dev = []
    while done < num_repeats:
        left = num_repeats - done
        G = min(graphs_per_batch, (left + fpg - 1) // fpg)
        gid0 = (first_frame + done) // fpg
        fb = engine.FrameBatch(ens, G, fpg, 2)
        fb.generate_graphs(seed, first_graph_id=gid0, protograph=bool(is_protograph))
        fb.generate_erasures(e, seed + 1, first_graph_id=gid0, doping_points=doping_points)
        r1_t, rec, ner = peel_batch(ens, fb, total_size, num_pd_steps, seed + 2, first_frame + done)
        k = min(left, G * fpg)
        if device_r1:
            r1_dev.append(r1_t.reshape(G * fpg, -1)[:k])
        else:
            r1[done:done + k] = r1_t.reshape(G * fpg, -1)[:k].cpu().numpy()
        lost = (ner - rec).reshape(-1)[:k].cpu().numpy()
        plrs[done:done + k] = lost / total_generated
        done += k
        prog.update(k)
    prog.close()
    if device_r1:
        return None, r1_dev, plrs
    return None, r1, plrs


# ---------------------------------------------------------------------------------------------------------------------
# error rates by peeling to the fixed point
# ---------------------------------------------------------------------------------------------------------------------
def extract_stopping_sets(lost_vns: np.ndarray, transmissions: np.ndarray):
    """Connected components of the residual graph of the lost VNs (PD.py:1077-1095): two lost VNs are connected when
    they share a CN.  Returns a list of index arrays into ``lost_vns``."""
    k = len(lost_vns)
    if k == 0:
        return []
    from scipy.sparse import coo_matrix
    from scipy.sparse.csgraph import connected_components
    tr = transmissions[lost_vns]                                   # [k][l]
    cns, inv = np.unique(tr.reshape(-1), return_inverse=True)
    rows = np.repeat(np.arange(k), tr.shape[1])
    b = coo_matrix((np.ones(rows.size, np.int8), (rows, inv.reshape(-1))), shape=(k, len(cns))).tocsr()
    ncomp, lab = connected_components(b @ b.T, directed=False)
    order = np.argsort(lab, kind="stable")
    bounds = np.searchsorted(lab[order], np.arange(ncomp + 1))
    return [order[bounds[i]:bounds[i + 1]] for i in range(ncomp)]


def account_lost(lost: np.ndarray, transmissions: np.ndarray, M: int):
    """Bookkeeping of one frame's lost VNs (PD.py:668-691): returns (num_lost, has_big_stopping_set,
    num_lost_expurgated, number_of_positions_with_an_expurgated_loss)."""
    ssets = extract_stopping_sets(lost, transmissions)
    big = [s for s in ssets if len(s) > 2]
    lost_exp = set()
    for s in big:
        lost_exp |= {int(v) // M for v in lost[s]}              # int(birthday / cns_per_pos) = VN position
    return len(lost), int(len(big) > 0), sum(len(s) for s in big), len(lost_exp)


def stopping_set_records(fb, erased_words, counted) -> np.ndarray:
    """``scldpc_bp_stopping_sets``: int32 [G][64*n_words][4] = (num_lost, has a stopping set of more than two VNs, VNs in
    such sets, VN positions they touch) per frame -- what ``account_lost`` returns, for every frame of the batch at once."""
    out = torch.empty((fb.n_graphs, 64 * fb.n_words, 4), dtype=torch.int32, device=fb.device)
    cp = np.ascontiguousarray(np.asarray(counted, dtype=np.uint8))
    assert cp.shape == (fb.ens.L,)
    _lib.check(_lib.lib().scldpc_bp_stopping_sets(ctypes.byref(fb.dims), ctypes.byref(fb.cbatch), ctypes.c_void_p(erased_words.data_ptr()),
                                                 cp.ctypes.data_as(ctypes.c_void_p), ctypes.c_void_p(out.data_ptr()), engine._stream()))
    return out.cpu().numpy()


def counted_positions(l, L, num_positions, ignored_head, ignored_tail, is_tail_biting=False) -> np.ndarray:
    """VN positions whose VNs can be "lost" (PD.py:661-666): at least one slot in the counted range
    [ignored_head, num_positions - ignored_tail) and every slot below total_size."""
    q = np.arange(L)
    cpos = q[:, None] + np.arange(l)[None, :]
    if is_tail_biting:
        cpos = cpos % L
    return ((cpos >= ignored_head) & (cpos < num_positions - ignored_tail)).any(axis=1) & (cpos < num_positions).all(axis=1)


# simulate_sc_ldpc decodes on frame streams from this many frames per graph on (the rule of bp_lim_iter --stream auto)
STREAM_MIN_FRAMES_PER_GRAPH = 1024


def simulate_sc_ldpc(e, l, r, L, M, is_terminated, is_protograph, is_bounded, is_tail_biting, num_repeats=int(1e5),
                     max_fuckups=2000, doping_points=[], *, seed=None, frames_per_graph=128, graphs_per_batch=8, first_frame=0,
                     progress=True, _batch_factory=None, _records_fn=None):
    """PD.py:591-701.  Returns the reference's 13-tuple
    ``(FER, FER_exp, PLR, PLR_exp, n_frames_failed_exp, n_frames, n_vn_failed_exp, n_vn_generated, failures, gens,
    n_blocks_failed_exp, n_blocks_generated, BLER_exp)``.

    The in-order ``sic_round`` scan (PD.py:656-657) reaches the peeling fixed point, which is the residual of unlimited
    flooding BP; that is what runs on the GPU.  Frames are decoded in batches and then accounted in frame order, so
    the ``max_fuckups`` early stop (PD.py:698) cuts at the same frame as a sequential run would.

    From ``STREAM_MIN_FRAMES_PER_GRAPH`` frames per graph on, each graph's frames are decoded as a frame stream on at most
    1024 lanes (``decode_bp_stream(..., stopping_sets=...)``): a lane whose frame has stopped takes the graph's next frame, so
    no frame waits for the slowest of its word, and any number of frames per graph works.  Frame f of graph g is the same
    channel realisation on both paths, so the records and the 13-tuple do not depend on the path."""
    _check_ensemble(is_protograph, doping_points, is_tail_biting)
    seed = _state["seed"] if seed is None else seed
    is_soft = isinstance(doping_points, dict)
    ignored_head = 0 if is_bounded else 20                      # PD.py:604-606
    ignored_head_schedule = 0 if is_bounded else 10
    ignored_tail = 0 if is_terminated else 20
    L = L + ignored_head + ignored_tail
    cns_per_pos = int(l / r * M)
    num_positions = L + l - 1 if is_terminated else L
    total_size = cns_per_pos * num_positions
    num_doping_points = len(doping_points)
    failures = np.zeros(num_repeats)
    gens = np.zeros(num_repeats)
    if is_soft:
        curr_generated = (L - ignored_head - ignored_tail) * M - sum(int(a * M) for a in doping_points.values())
    else:
        curr_generated = (L - num_doping_points - ignored_head - ignored_tail) * M
    blocks_per_frame = L - num_doping_points - ignored_head - ignored_tail

    ens = engine.Ensemble(l, r, L, M)
    fpg = int(frames_per_graph)
    use_stream = fpg >= STREAM_MIN_FRAMES_PER_GRAPH and _batch_factory is None and _records_fn is None
    counted = counted_positions(l, L, num_positions, ignored_head, ignored_tail, bool(is_tail_biting))

    from . import dist as D
    rank, world = D.world()
    num_fuckups = num_fuckups_truncated = 0
    total_generated = total_failed = total_failed_expurgated = 0
    total_blocks_generated = total_blocks_failed_exp = 0
    o = -1
    prog = _Progress(num_repeats, progress and rank == 0)
    stop = False
    unscanned = ignored_head_schedule * cns_per_pos

    def decode_records(G, gid0):
        """decodes G graphs x fpg frames; one row (num_lost, big, lost_exp, blocks_exp) per frame, in frame order"""
        rec = np.zeros((G * fpg, 4), np.int64)
        if G == 0:
            return rec
        if _records_fn is not None:                                      # CPU tests of the round / gather / replay logic
            return np.asarray(_records_fn(G, fpg, gid0), np.int64).reshape(G * fpg, 4)
        # non-terminated: the decoder never uses CNs >= total_size (truncated BP, BP_TRAJ.c:944-948 semantics).
        # unbounded: slots below ignored_head_schedule*cns_per_pos are never scanned (PD.py:656), they only decode
        # when a removal leaves them with one user -- scldpc_bp_full's unscanned_head_cns
        is_term = bool(is_terminated) and not is_tail_biting
        if use_stream:                                                   # the stream draws the channels of its frames itself
            fb = engine.FrameBatch(ens, G, min(fpg, 1024))
            fb.generate_graphs(seed, first_graph_id=gid0, tail_biting=bool(is_tail_biting), protograph=bool(is_protograph))
            res = engine.decode_bp_stream(fb, fpg, e, seed + 1, first_graph_id=gid0, is_term=is_term, doping_points=doping_points,
                                          stopping_sets=counted, unscanned_head_cns=unscanned)
            return res.records.reshape(G * fpg, 4).astype(np.int64)
        if _batch_factory is not None:                                   # tests inject codes and erasure masks here
            fb = _batch_factory(ens, G, fpg, gid0)
        else:
            fb = engine.FrameBatch(ens, G, fpg, engine.words_for(fpg))
            fb.generate_graphs(seed, first_graph_id=gid0, tail_biting=bool(is_tail_biting), protograph=bool(is_protograph))
            fb.generate_erasures(e, seed + 1, first_graph_id=gid0, doping_points=doping_points)
        res = engine.decode_bp_full(fb, engine.UNLIMITED, is_term=is_term, unscanned_head_cns=unscanned)
        # stopping sets of the lost VNs (PD.py:668-691) on the device: one record per frame, one copy per batch
        return stopping_set_records(fb, res.erased_words, counted)[:, :fpg].reshape(G * fpg, 4).astype(np.int64)

    # Frames are decoded in rounds of world_size x graphs_per_batch graphs (rank r takes the r-th batch of the round; graph
    # ids are global), the per-frame records are all-gathered, and every rank then walks the frames in global order with
    # the reference's sequential bookkeeping -- so the result, including the max_fuckups cut (PD.py:698), is the same for
    # any number of GPUs.
    while o + 1 < num_repeats and not stop:
        left = num_repeats - (o + 1)
        graphs_left = (left + fpg - 1) // fpg
        gid_round = (first_frame + o + 1) // fpg
        G_r = max(0, min(graphs_per_batch, graphs_left - rank * graphs_per_batch))
        rec = decode_records(G_r, gid_round + rank * graphs_per_batch)
        pad = np.full((graphs_per_batch * fpg, 4), -1, np.int64)
        pad[: len(rec)] = rec
        allrec = D.allgather_rows(pad).reshape(-1, 4)
        for row in allrec:
            if row[0] < 0:
                continue
            if o + 1 >= num_repeats:
                stop = True
                break
            o += 1
            total_generated += curr_generated
            total_blocks_generated += blocks_per_frame
            if row[0] >= 1:
                num_fuckups += 1
                total_failed += int(row[0])
                num_fuckups_truncated += int(row[1])
                total_failed_expurgated += int(row[2])
                total_blocks_failed_exp += int(row[3])
            if num_fuckups >= max_fuckups:
                stop = True
                break
        prog.update(min(left, world * graphs_per_batch * fpg), "FER: %.5f (%.5f); PLR: %.5f (%.5f); BLER: %.5f" % (
            num_fuckups / (o + 1), num_fuckups_truncated / (o + 1), total_failed / max(1, total_generated),
            total_failed_expurgated / max(1, total_generated), total_blocks_failed_exp / max(1, total_blocks_generated)))
    prog.close()
    total_plr = total_failed / total_generated
    total_plr_expurgated = total_failed_expurgated / total_generated
    total_bler_expurgated = total_blocks_failed_exp / total_blocks_generated
    return (num_fuckups / (o + 1), num_fuckups_truncated / (o + 1), total_plr, total_plr_expurgated, num_fuckups_truncated, o + 1,
            total_failed_expurgated, total_generated, failures, gens, total_blocks_failed_exp, total_blocks_generated,
            total_bler_expurgated)


# ---------------------------------------------------------------------------------------------------------------------
# variance estimation (PD.py:1264-1294 + est_scaling_params.calc_nu_chunk / calc_var_chunk)
# ---------------------------------------------------------------------------------------------------------------------
def calc_nu_chunk_device(r1_chunks, r1s_theory: np.ndarray, M):
    """``calc_nu_chunk`` (EST.py:90-94) + ``calc_var_chunk`` (EST.py:131-138) on the device.  ``r1_chunks``: list of int32
    device tensors [frames][num_steps+1] in frame order.  Returns (ssquares float64[S], counts int64[S])."""
    lib = _lib.lib()
    r1s_theory = np.asarray(r1s_theory, dtype=np.float64)
    crop = int(np.max(np.where(r1s_theory > 0))) + 1               # r1s_chunk[:, :max(where(theory > 0)) + 1]
    th = r1s_theory[r1s_theory > 0]                                # r1s_theory[r1s_theory > 0]
    crop = min(crop, r1s_theory.shape[0])
    S = min(crop, len(th))                                         # numpy broadcasting needs equal lengths; the
    if crop != len(th):                                            # reference relies on theory being positive up to crop
        raise ValueError("r1s_theory has zeros below its last positive entry; the reference's broadcast would fail")
    dev = r1_chunks[0].device
    th_d = torch.as_tensor(th, device=dev)
    ssq = torch.zeros(S, dtype=torch.float64, device=dev)
    cnt = torch.zeros(S, dtype=torch.int64, device=dev)
    for r1 in r1_chunks:
        if r1.shape[1] < S:
            raise ValueError("trajectories shorter than the theory curve")
        r1 = r1.contiguous()
        _lib.check(lib.scldpc_peel_variance_accumulate(ctypes.c_void_p(r1.data_ptr()), int(r1.shape[0]), int(r1.shape[1]),
                                                       ctypes.c_void_p(th_d.data_ptr()), S, ctypes.c_double(float(M)),
                                                       ctypes.c_void_p(ssq.data_ptr()), ctypes.c_void_p(cnt.data_ptr()),
                                                       engine._stream()))
    return ssq.cpu().numpy(), cnt.cpu().numpy()


def main_simulate_variance(argv=None):
    """argv: fname l r L M e T|N P|U num_runs num_runs_batch ftheory  (PD.py:1265-1275) -> pickle (ssquares, counts)."""
    argv = sys.argv if argv is None else argv
    fname = argv[1]
    l = int(argv[2]); r = int(argv[3]); L = int(argv[4]); M = int(argv[5]); e = float(argv[6])
    is_terminated = True if argv[7] == 'T' else False
    is_protograph = True if argv[8] == 'P' else False
    num_runs = int(argv[9]); num_runs_batch = int(argv[10]); ftheory = argv[11]
    with open(ftheory, 'rb') as f:
        r1s_theory = pickle.load(f)[0]
    from . import dist as D
    rank, _world = D.init_from_env()          # under torchrun the frames of every chunk are split over the GPUs
    isfirst = True
    ssquares, counts = None, None
    num_rounds = int(num_runs / num_runs_batch)
    for i in range(num_rounds):
        _, r1_dev, _ = simulate_peeling_decoder_ldpc(e, l, r, L, M, is_terminated, is_protograph, num_runs_batch,
                                                     first_frame=i * num_runs_batch, device_r1=True)
        ssquares_chunk, counts_chunk = calc_nu_chunk_device(r1_dev, r1s_theory, M)
        ssquares = ssquares_chunk if isfirst else ssquares + ssquares_chunk
        counts = counts_chunk if isfirst else counts + counts_chunk
        isfirst = False
    if rank == 0:
        with open(fname, 'wb') as f:
            pickle.dump((ssquares, counts), f)
    return ssquares, counts


def parse_sc_ldpc_options(extra):
    """Optional trailing arguments of ``main_simulate_sc_ldpc`` after the 13 positional ones of PD.py:1328-1340:
    ``--frames-per-graph N`` (default 128) and ``--graphs-per-batch G`` (default 8).  Returns (frames_per_graph,
    graphs_per_batch)."""
    import argparse
    ap = argparse.ArgumentParser(prog="ber_sim", description="options after the 13 positional arguments")
    ap.add_argument("--frames-per-graph", type=int, default=128,
                    help="frames decoded per graph realisation (from %d on: frame streams, any number)" % STREAM_MIN_FRAMES_PER_GRAPH)
    ap.add_argument("--graphs-per-batch", type=int, default=8, help="graphs decoded at once per GPU")
    a = ap.parse_args(list(extra))
    if a.frames_per_graph < 1 or a.graphs_per_batch < 1:
        ap.error("--frames-per-graph and --graphs-per-batch must be >= 1")
    return a.frames_per_graph, a.graphs_per_batch


def main_simulate_sc_ldpc(argv=None):
    """argv: fname l r L M "es" T|N P|U B|U TB|NTB num_repeats max_fuckups "doping"  (PD.py:1328-1340), optionally followed
    by ``--frames-per-graph N`` and ``--graphs-per-batch G`` (``parse_sc_ldpc_options``)."""
    argv = sys.argv if argv is None else argv
    fpg, gpb = parse_sc_ldpc_options(argv[14:])
    fname = argv[1]
    l = int(argv[2]); r = int(argv[3]); L = int(argv[4]); M = int(argv[5])
    es = eval(argv[6])
    is_terminated = True if argv[7] == 'T' else False
    is_protograph = True if argv[8] == 'P' else False
    is_bounded = True if argv[9] == 'B' else False
    is_tail_biting = True if argv[10] == 'TB' else False
    num_repeats = int(argv[11]); max_fuckups = int(argv[12])
    doping_points = eval(argv[13])
    L += len(doping_points)                                         # PD.py:1343
    hdr = (f"# SC-LDPC ({l},{r},L={L},M={M}) terminated:{is_terminated}, proto:{is_protograph}, bounded:{is_bounded}, "
           f"tail biting:{is_tail_biting}. num_repeats={num_repeats}, max_fuckups={max_fuckups}, doping_points={doping_points}.")
    from . import dist as D
    rank, _world = D.init_from_env()          # under torchrun every round of batches is spread over the GPUs
    with open(fname if rank == 0 else os.devnull, 'wt') as f:
        if rank == 0:
            print(hdr)
        print(hdr, file=f)
        f.flush()
        for e in es:
            ber, ber_truncated, plr, plr_exp, fbl, tbl, fbit, tgen, _flrs, _gens, fblocks, tblocks, bler = simulate_sc_ldpc(
                e, l, r, L, M, is_terminated, is_protograph, is_bounded, is_tail_biting, num_repeats, max_fuckups, doping_points,
                frames_per_graph=fpg, graphs_per_batch=gpb)
            print(e, ber, ber_truncated, plr, plr_exp, fbl, tbl, fbit, tgen, fblocks, tblocks, bler, file=f)
            if rank == 0:
                print(e, ber, ber_truncated, plr, plr_exp, fbl, tbl, fbit, tgen, fblocks, tblocks, bler)
            f.flush()
            sys.stdout.flush()
