"""Device-side containers and decoder calls.  PyTorch owns every device buffer (``torch.empty(..., device="cuda")``);
all arithmetic happens in the hand-written kernels of ``libscldpc.so`` reached through ctypes.

Vocabulary follows the reference: a *frame* is one (code, channel realisation) pair, a *position* one of the L
spatial positions of the coupled chain, M the number of VNs per position (``PD.py`` / paper convention; the C files'
``Def_M`` is the number of CNs per position).  A *batch* holds ``n_graphs`` graph realisations, each decoded for
``n_frames`` frames at once (bit-sliced, 64 frames per lane word).
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
import os

from ._lib import F_EXP_ALL, F_MESSAGES, F_NO_WAVE, F_SQUARE, F_TERMINATED, F_TRAJECTORY

UNLIMITED = 0  # max_it value meaning "until every frame has stalled or finished"


def _sweep_flags(env_name: str, messages: bool | None) -> int:
    """Implementation selector -> C-ABI flag.  ``messages=None`` takes the default from the environment variable (0 selects
    the message-passing sweeps); the library itself never reads the environment for this, so a workspace-size query and a
    decoder call always agree."""
    if messages is None:
        messages = os.environ.get(env_name, "1") == "0"
    return F_MESSAGES if messages else 0


@dataclass(frozen=True)
class Ensemble:
    """(dv, dc)-regular SC-LDPC ensemble: L positions, M VNs and M*dv/dc CNs per position."""
    dv: int
    dc: int
    L: int
    M: int

    def __post_init__(self):
        if (self.M * self.dv) % self.dc:
            raise ValueError("M*dv must be a multiple of dc")

    @property
    def cns_pos(self) -> int:
        return self.M * self.dv // self.dc

    @property
    def n(self) -> int:
        return self.L * self.M

    @property
    def nk(self) -> int:
        return (self.L + self.dv - 1) * self.cns_pos

    @property
    def E(self) -> int:
        return self.n * self.dv


def words_for(n_frames: int) -> int:
    """Smallest supported number of lane words (2, 4, 8, 16) that holds n_frames frames."""
    for w in (2, 4, 8, 16):
        if n_frames <= 64 * w:
            return w
    raise ValueError("at most 1024 frames per graph")


def _doping(doping_points, M: int):
    """(hard positions, soft positions, soft counts) of ``doping_points``: a list of positions (hard doping) or a dict
    {position: alpha} (soft doping: the first int(alpha*M) VNs of the position are known, PD.py:175-183)."""
    if isinstance(doping_points, dict):
        return [], [int(p) for p in doping_points], [int(a * M) for a in doping_points.values()]
    return [int(p) for p in doping_points], [], []


def _device(device=None) -> torch.device:
    if not torch.cuda.is_available():
        raise _lib.ScldpcError("no CUDA device: fl_scaling_sc_ldpc_b200 has no CPU fallback")
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


def _stream() -> ctypes.c_void_p:
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


class FrameBatch:
    """n_graphs graph realisations x n_frames channel realisations, resident in HBM."""

    def __init__(self, ens: Ensemble, n_graphs: int, n_frames: int, n_words: int | None = None, device=None):
        self.ens = ens
        self.n_graphs = int(n_graphs)
        self.n_frames = int(n_frames)
        self.n_words = int(n_words or words_for(n_frames))
        self.device = _device(device)
        self.dims = _lib.Dims(ens.dv, ens.dc, ens.L, ens.M, ens.cns_pos, self.n_graphs, self.n_words, self.n_frames)
        G, W = self.n_graphs, self.n_words
        dev = self.device
        self.vn_cn = torch.empty((G, ens.n, ens.dv), dtype=torch.int32, device=dev)
        self.vn_slot = torch.empty((G, ens.n, ens.dv), dtype=torch.int32, device=dev)
        self.cn_edge = torch.empty((G, ens.nk, ens.dc), dtype=torch.int32, device=dev)
        self.chan = torch.zeros((G, ens.n, W), dtype=torch.int64, device=dev)
        self._scratch = torch.empty((G, ens.nk), dtype=torch.int32, device=dev)
        self._graph_err = torch.zeros(1, dtype=torch.int32, device=dev)
        self._keys = None
        self._ws = None
        self.cbatch = _lib.Batch(self.vn_cn.data_ptr(), self.vn_slot.data_ptr(), self.cn_edge.data_ptr(), self.chan.data_ptr())

    # ---- graphs ------------------------------------------------------------------------------------------
    def set_graphs(self, vn_cn) -> "FrameBatch":
        """Inject graphs: int array [n_graphs][n][dv] of CN indices (``VNdegree[v][1+i]`` / ``transmissions``)."""
        t = torch.as_tensor(np.ascontiguousarray(vn_cn, dtype=np.int32)).reshape(self.n_graphs, self.ens.n, self.ens.dv)
        self.vn_cn.copy_(t, non_blocking=False)
        self._build_tables()
        return self

    def generate_graphs(self, seed: int, first_graph_id: int = 0, tail_biting: bool = False, protograph: bool = False,
                        first_position: int = 0) -> "FrameBatch":
        """Draw graphs on the device: the semi-structured ensemble (``generate_code`` BP_FULL.c:1656 / ``SC.gen_slots``
        SC.py:53), its tail-biting variant, or the protograph-based ensemble (``sc_ldpc_protograph.py``).
        ``first_position`` > 0: the batch is a piece of a longer chain starting at that absolute position (streams).
        Absolute CN positions are 32-bit Philox counter words, so ``first_position + L + dv - 1 <= 2**32``; a piece
        beyond that raises ``ValueError`` rather than reusing the permutations of position 0 onwards."""
        if first_position < 0 or first_position + self.ens.L + self.ens.dv - 1 > 1 << 32:
            raise ValueError(f"first_position {first_position} + L + dv - 1 exceeds 2**32 CN positions")
        L = _lib.lib()
        if first_position:
            if tail_biting or protograph:
                raise ValueError("chain pieces exist for the semi-structured ensemble only")
            nbytes = L.scldpc_graph_generate_scratch_bytes(ctypes.byref(self.dims), 0)
            if self._keys is None or self._keys.numel() * 8 < nbytes:
                self._keys = torch.empty((nbytes + 7) // 8, dtype=torch.int64, device=self.device)
            _lib.check(L.scldpc_graph_generate_at(ctypes.byref(self.dims), ctypes.c_void_p(self.vn_cn.data_ptr()),
                                                  ctypes.c_void_p(self._keys.data_ptr()), ctypes.c_uint64(seed),
                                                  ctypes.c_uint64(first_graph_id), ctypes.c_uint32(first_position), _stream()))
            self._build_tables(check=False)
            return self
        ensemble = 2 if protograph else int(bool(tail_biting))
        tail_biting = ensemble
        nbytes = L.scldpc_graph_generate_scratch_bytes(ctypes.byref(self.dims), int(tail_biting))
        if self._keys is None or self._keys.numel() * 8 < nbytes:
            self._keys = torch.empty((nbytes + 7) // 8, dtype=torch.int64, device=self.device)
        _lib.check(L.scldpc_graph_generate(ctypes.byref(self.dims), ctypes.c_void_p(self.vn_cn.data_ptr()),
                                           ctypes.c_void_p(self._keys.data_ptr()), ctypes.c_uint64(seed),
                                           ctypes.c_uint64(first_graph_id), int(tail_biting), _stream()))
        self._build_tables(check=False)
        return self

    def _build_tables(self, check: bool = True):
        """vn_slot / cn_edge from vn_cn.  ``check=False`` (graphs drawn by the library: valid by construction) stays
        stream-ordered -- no host synchronisation, so a loop that redraws its graphs every batch never stalls the device;
        the validity flag stays in ``self._graph_err`` (``graph_error()`` reads it)."""
        if check:
            _lib.check(_lib.lib().scldpc_graph_build_tables(ctypes.byref(self.dims), ctypes.byref(self.cbatch),
                                                            ctypes.c_void_p(self._scratch.data_ptr()), _stream()))
        else:
            _lib.check(_lib.lib().scldpc_graph_build_tables_async(ctypes.byref(self.dims), ctypes.byref(self.cbatch),
                                                                  ctypes.c_void_p(self._scratch.data_ptr()),
                                                                  ctypes.c_void_p(self._graph_err.data_ptr()), _stream()))

    def graph_error(self) -> int:
        """validity flag of the last stream-ordered table build: 0 fine, 1 CN index out of range, 2 CN degree > dc"""
        return int(self._graph_err.item())

    # ---- channel -----------------------------------------------------------------------------------------
    def set_erasures(self, erased) -> "FrameBatch":
        """Inject channel realisations: bool/uint8 array [n_graphs][n_frames][n], 1 = erased (``LLRsChannel``)."""
        e = np.ascontiguousarray(erased, dtype=np.uint8).reshape(self.n_graphs, self.n_frames, self.ens.n)
        _lib.check(_lib.lib().scldpc_channel_pack_host(ctypes.byref(self.dims), e.ctypes.data_as(ctypes.c_void_p),
                                                       ctypes.c_void_p(self.chan.data_ptr()), _stream()))
        return self

    def generate_erasures(self, eps, seed: int, first_graph_id: int = 0, doping_points=(), first_frame: int = 0,
                          first_vn: int = 0) -> "FrameBatch":
        """BEC(eps) realisations on the device; ``eps`` is a float or one value per graph of the batch.
        ``doping_points``: list of positions (hard doping) or dict {position: alpha} (soft doping: the first
        int(alpha*M) VNs are known, PD.py:175-183).  Lane f holds frame ``first_frame + f`` of the graph's channel
        stream (``first_frame`` a multiple of 4).  ``first_vn`` > 0: the batch is a piece of a longer chain whose first VN
        has that absolute index (hard doping only; positions are local to the piece).
        VN and frame ids are 32-bit Philox counter words: ``first_vn + n <= 2**32`` and
        ``first_frame + 64 * n_words <= 2**32`` (every lane, used or not, has its frame id), else ``ValueError`` -- ids
        past 2**32 would wrap and repeat earlier realisations."""
        if first_vn < 0 or first_vn + self.ens.n > 1 << 32:
            raise ValueError(f"first_vn {first_vn} + n ({self.ens.n}) exceeds 2**32 VN ids")
        if first_frame < 0 or first_frame + 64 * self.n_words > 1 << 32:
            raise ValueError(f"first_frame {first_frame} + 64 * n_words ({64 * self.n_words}) exceeds 2**32 frame ids")
        if first_vn:
            if isinstance(doping_points, dict) or np.ndim(eps) != 0:
                raise ValueError("chain pieces take one eps and hard doping only")
            hard = [int(p) for p in doping_points]
            a = (ctypes.c_int32 * max(1, len(hard)))(*hard)
            _lib.check(_lib.lib().scldpc_channel_generate_at(
                ctypes.byref(self.dims), ctypes.c_void_p(self.chan.data_ptr()), ctypes.c_double(float(eps)), a, len(hard),
                ctypes.c_uint64(seed), ctypes.c_uint64(first_graph_id), ctypes.c_uint32(first_frame), ctypes.c_uint32(first_vn), _stream()))
            return self
        hard, soft_p, soft_c = _doping(doping_points, self.ens.M)
        arr = lambda xs: (ctypes.c_int32 * max(1, len(xs)))(*xs)
        L = _lib.lib()
        if np.ndim(eps) == 0:
            calls = [(self.dims, self.chan.data_ptr(), float(eps), first_graph_id)]
        else:
            if len(eps) != self.n_graphs:
                raise ValueError("need one eps per graph")
            e, d = self.ens, self.dims
            calls = [(_lib.Dims(e.dv, e.dc, e.L, e.M, e.cns_pos, 1, d.n_words, d.n_frames), self.chan[g].data_ptr(),
                      float(eps[g]), first_graph_id + g) for g in range(self.n_graphs)]
        for dims, ptr, ep, gid in calls:
            _lib.check(L.scldpc_channel_generate(
                ctypes.byref(dims), ctypes.c_void_p(ptr), ctypes.c_double(ep), arr(hard), len(hard),
                arr(soft_p), arr(soft_c), len(soft_p), ctypes.c_uint64(seed), ctypes.c_uint64(gid), ctypes.c_uint32(first_frame),
                _stream()))
        return self

    def erasures_host(self) -> np.ndarray:
        """Channel realisations as uint8 [n_graphs][n_frames][n]."""
        return unpack_lanes(self.chan, self.n_frames)

    # ---- workspace ---------------------------------------------------------------------------------------
    def workspace(self, flags: int) -> torch.Tensor:
        return self._workspace_bytes(_lib.lib().scldpc_bp_workspace_bytes(ctypes.byref(self.dims), flags))

    def _workspace_bytes(self, need: int) -> torch.Tensor:
        """The workspace grown to ``need`` bytes, the result of a size query (0: the query failed)."""
        if need == 0:
            raise _lib.ScldpcError(_lib.lib().scldpc_last_error().decode())
        if self._ws is None or self._ws.numel() < need:
            self._ws = None
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        return self._ws


def unpack_lanes(words: torch.Tensor, n_frames: int) -> np.ndarray:
    """int64 [G][n][W] bit-sliced words -> uint8 [G][n_frames][n]."""
    w = words.cpu().numpy().view(np.uint64)
    G, n, W = w.shape
    bits = np.unpackbits(w.view(np.uint8).reshape(G, n, W * 8), axis=2, bitorder="little")  # [G][n][64W]
    return np.ascontiguousarray(bits[:, :, :n_frames].transpose(0, 2, 1))


@dataclass
class BpResult:
    """Per-frame outputs of a decoder call; arrays are [n_graphs][n_frames] unless noted."""
    iters: np.ndarray            # iterations executed (window decoder: summed over windows)
    residual: np.ndarray         # NumErasures (return value of decodeBP / decodeBP_SW)
    blocks_err: np.ndarray       # *num_blocks_err
    erasures_exp: np.ndarray     # *num_erasures_exp
    blocks_err_exp: np.ndarray   # *num_blocks_err_exp
    erasures_p1: np.ndarray      # *NumErasuresP1 (window decoder)
    erased_words: torch.Tensor   # int64 [G][n][W] VNerased, bit-sliced, on the device
    rows: np.ndarray | None      # [G][n_frames][max_rows][3] (deg_1_iter, dVNs, first erased position) or None
    iters_launched: int = 0
    edge_updates: int = 0        # useful directed-edge message updates (sum over frames of iterations * edges swept)
    n_frames: int = 0

    def erased(self) -> np.ndarray:
        """VNerased as uint8 [G][n_frames][n]."""
        return unpack_lanes(self.erased_words, self.n_frames)


def _alloc_out(fb: FrameBatch, max_rows: int):
    G, lanes = fb.n_graphs, 64 * fb.n_words
    res = torch.zeros((6, G, lanes), dtype=torch.int32, device=fb.device)
    erased = torch.empty((G, fb.ens.n, fb.n_words), dtype=torch.int64, device=fb.device)
    rows = torch.zeros((G, max_rows, lanes, 3), dtype=torch.int32, device=fb.device) if max_rows else None
    out = _lib.BpOut(res[0].data_ptr(), res[1].data_ptr(), res[2].data_ptr(), res[3].data_ptr(), res[4].data_ptr(),
                     res[5].data_ptr(), erased.data_ptr(), rows.data_ptr() if rows is not None else None, max_rows)
    return res, erased, rows, out


def _collect(fb: FrameBatch, res, erased, rows, **kw) -> BpResult:
    F = fb.n_frames
    r = res.cpu().numpy()[:, :, :F]
    rr = None
    if rows is not None:
        rr = np.ascontiguousarray(rows.cpu().numpy()[:, :, :F, :].transpose(0, 2, 1, 3))
    return BpResult(iters=r[0], residual=r[1], blocks_err=r[2], erasures_exp=r[3], blocks_err_exp=r[4], erasures_p1=r[5],
                    erased_words=erased, rows=rr, n_frames=F, **kw)


def decode_bp_full(fb: FrameBatch, max_it: int = UNLIMITED, is_term: bool = True, trajectory: bool = False,
                   max_rows: int | None = None, collect: bool = True, unscanned_head_cns: int = 0,
                   messages: bool | None = None):
    """Full flooding BP -- ``decodeBP`` (BP_FULL.c:900, BP_TRAJ.c:901).  ``max_it`` is the reference's ``MaxNumIt``
    (values <= 0 run until every frame has stalled or finished; note the reference's do-while executes at least one
    iteration, which callers reproduce by passing max(1, MaxNumIt)).  ``unscanned_head_cns``: CNs below this index are
    never scanned (``simulate_sc_ldpc`` with ``is_bounded=False``, PD.py:604-605,656).  ``messages``: pass explicit messages
    instead of the node-state sweeps (default from ``SCLDPC_FULL_NODE``; trajectories always pass messages)."""
    flags = (F_TERMINATED if is_term else 0) | (F_TRAJECTORY if trajectory else 0) | _sweep_flags("SCLDPC_FULL_NODE", messages)
    if os.environ.get("SCLDPC_NO_WAVE", "0") == "1":
        flags |= F_NO_WAVE
    if trajectory and not max_rows:
        if max_it <= 0:
            raise ValueError("trajectory mode needs max_rows when max_it is unlimited")
        max_rows = max_it
    res, erased, rows, out = _alloc_out(fb, max_rows if trajectory else 0)
    ws = fb.workspace(flags)
    launched = ctypes.c_int(0)
    _lib.check(_lib.lib().scldpc_bp_full(ctypes.byref(fb.dims), ctypes.byref(fb.cbatch), int(max_it), flags, int(unscanned_head_cns), ctypes.byref(out),
                                         ctypes.c_void_p(ws.data_ptr()), ctypes.c_size_t(ws.numel()), ctypes.byref(launched),
                                         _stream()))
    if not collect:
        return res, erased, rows, launched.value
    r = _collect(fb, res, erased, rows, iters_launched=launched.value)
    r.edge_updates = int(r.iters.astype(np.int64).sum()) * 2 * fb.ens.E
    return r


MOMENT_NAMES = ("frames", "frames_dvn_nonzero", "sum_dvn", "sum_dvn2", "sum_deg1", "sum_deg1_2", "sum_first_pos", "sum_dvn_deg1")


def trajectory_moments(fb: FrameBatch, iters_dev: torch.Tensor, rows_dev: torch.Tensor, acc: torch.Tensor | None = None) -> torch.Tensor:
    """Adds the per-iteration moments of a trajectory decode (``decode_bp_full(..., trajectory=True, collect=False)``:
    ``iters_dev = res[0]``, ``rows_dev = rows``) to ``acc`` int64 [max_rows][8] on the device (``MOMENT_NAMES``) --
    ``scldpc_bp_trajectory_moments``; what the notebook computes from bp_traj's text rows (NB cells 40-42), without the
    rows ever leaving the device."""
    max_rows = int(rows_dev.shape[1])
    if acc is None:
        acc = torch.zeros((max_rows, len(MOMENT_NAMES)), dtype=torch.int64, device=fb.device)
    assert acc.shape == (max_rows, len(MOMENT_NAMES)) and acc.is_contiguous()
    _lib.check(_lib.lib().scldpc_bp_trajectory_moments(ctypes.byref(fb.dims), ctypes.c_void_p(rows_dev.data_ptr()),
                                                      ctypes.c_void_p(iters_dev.data_ptr()), max_rows, ctypes.c_void_p(acc.data_ptr()), _stream()))
    return acc


def position_counts(fb: FrameBatch, flags: int):
    """Per-position erased-VN counts and accepted size-two stopping sets of the last decode on ``fb``:
    two int32 arrays [n_graphs][L][n_frames]."""
    G, Lp, lanes = fb.n_graphs, fb.ens.L, 64 * fb.n_words
    cnt = torch.empty((G, Lp, lanes), dtype=torch.int32, device=fb.device)
    pairs = torch.empty((G, Lp, lanes), dtype=torch.int32, device=fb.device)
    _lib.check(_lib.lib().scldpc_bp_position_counts(ctypes.byref(fb.dims), flags, ctypes.c_void_p(fb.workspace(flags).data_ptr()),
                                                    ctypes.c_void_p(cnt.data_ptr()), ctypes.c_void_p(pairs.data_ptr()), _stream()))
    return cnt[:, :, :fb.n_frames].cpu().numpy(), pairs[:, :, :fb.n_frames].cpu().numpy()


def decode_bp_window(fb: FrameBatch, W: int, max_it: int, init_it: int = 0, square: bool = True, is_term: bool = True,
                     collect: bool = True, messages: bool | None = None):
    """Sliding-window BP -- ``decodeBP_SW`` (square window BP_SW.c:628, classical window BP_FULL.c:627)."""
    flags = (F_TERMINATED if is_term else 0) | (F_SQUARE if square else 0) | F_EXP_ALL | _sweep_flags("SCLDPC_WINDOW_NODE", messages)
    res, erased, rows, out = _alloc_out(fb, 0)
    ws = fb.workspace(flags)
    work = ctypes.c_int64(0)
    _lib.check(_lib.lib().scldpc_bp_window(ctypes.byref(fb.dims), ctypes.byref(fb.cbatch), int(W), int(max_it), int(init_it),
                                           flags, ctypes.byref(out), ctypes.c_void_p(ws.data_ptr()), ctypes.c_size_t(ws.numel()),
                                           ctypes.byref(work) if collect else None, _stream()))
    if not collect:
        return res, erased, rows, 0
    return _collect(fb, res, erased, rows, edge_updates=work.value)


def decode_bp_window_range(fb: FrameBatch, W: int, max_it: int, first_window: int, n_windows: int, erased: torch.Tensor,
                           pending: torch.Tensor, resume: bool, init_it: int = 0, square: bool = False, is_term: bool = True):
    """Windows [first_window, first_window + n_windows) of ``decode_bp_window`` with the decoder state owned by the caller
    (``scldpc_bp_window_range``): ``erased`` (what the CNs see; ends as the decisions) and ``pending`` (what every VN has been
    told so far), int64 [G][n][W] each.  ``resume=False`` initialises them from ``fb.chan``.  Returns the per-frame result
    tensor int32 [6][G][lanes] (device); per-position counts through ``position_counts``."""
    flags = (F_TERMINATED if is_term else 0) | (F_SQUARE if square else 0) | F_EXP_ALL
    G, lanes = fb.n_graphs, 64 * fb.n_words
    res = torch.zeros((6, G, lanes), dtype=torch.int32, device=fb.device)
    assert erased.shape == pending.shape == (G, fb.ens.n, fb.n_words) and erased.is_contiguous() and pending.is_contiguous()
    out = _lib.BpOut(res[0].data_ptr(), res[1].data_ptr(), res[2].data_ptr(), res[3].data_ptr(), res[4].data_ptr(),
                     res[5].data_ptr(), erased.data_ptr(), None, 0)
    ws = fb.workspace(flags)
    _lib.check(_lib.lib().scldpc_bp_window_range(ctypes.byref(fb.dims), ctypes.byref(fb.cbatch), int(W), int(max_it), int(init_it), flags,
                                                 int(first_window), int(n_windows), ctypes.c_void_p(pending.data_ptr()), int(bool(resume)),
                                                 ctypes.byref(out), ctypes.c_void_p(ws.data_ptr()), ctypes.c_size_t(ws.numel()), None, _stream()))
    return res


@dataclass
class StreamResult:
    """Per-frame outputs of ``decode_bp_stream``; arrays are [n_graphs][frames_per_graph], indexed by frame id."""
    iters: np.ndarray
    residual: np.ndarray
    blocks_err: np.ndarray
    erasures_exp: np.ndarray
    blocks_err_exp: np.ndarray
    iters_launched: int = 0
    edge_updates: int = 0


@dataclass
class StreamCapsResult:
    """Per-frame outputs of ``decode_bp_stream(..., caps=...)``: ``iters`` [n_graphs][frames_per_graph] under the largest cap
    (under cap ``caps[k]`` a frame takes ``min(iters, caps[k])`` iterations), the statistics [K][n_graphs][frames_per_graph],
    slot k being what ``decode_bp_stream(..., max_it=caps[k])`` returns."""
    caps: tuple
    iters: np.ndarray
    residual: np.ndarray
    blocks_err: np.ndarray
    erasures_exp: np.ndarray
    blocks_err_exp: np.ndarray
    iters_launched: int = 0
    edge_updates: int = 0


@dataclass
class StreamStoppingSetResult:
    """Per-frame outputs of ``decode_bp_stream(..., stopping_sets=counted)``, indexed by frame id: ``iters``
    [n_graphs][frames_per_graph] of unlimited BP and ``records`` [n_graphs][frames_per_graph][4] = (num_lost, has a stopping
    set of more than two VNs, VNs in such sets, VN positions they touch) -- what ``stopping_set_records`` gives for the
    frame after ``decode_bp_full`` with the same ``unscanned_head_cns``."""
    iters: np.ndarray
    records: np.ndarray
    iters_launched: int = 0
    edge_updates: int = 0


def decode_bp_stream(fb: FrameBatch, frames_per_graph: int, eps, seed: int, first_graph_id: int = 0, is_term: bool = True,
                     doping_points=(), harvest_every: int = 0, exp_all: bool = False, collect: bool = True, max_it: int = 0,
                     messages: bool | None = None, caps=None, stopping_sets=None, unscanned_head_cns: int = 0):
    """Full BP (unlimited, or at most ``max_it`` iterations per frame) over a stream of ``frames_per_graph`` frames per
    graph with lane recycling (``scldpc_bp_stream``).  Frame f of graph g is the channel realisation ``generate_erasures(..., first_frame=...)``
    puts in lane f - first_frame; the graphs are the ones resident in ``fb`` (``fb.n_frames`` lanes are used).

    ``caps``: strictly ascending iteration caps (at most 16, each >= 1; the last may be <= 0, unlimited) in place of
    ``max_it``.  One decode up to the largest cap gives the results of every cap (``scldpc_bp_stream_caps``): a
    ``StreamCapsResult``, or with ``collect=False`` the device tensors (iters [G][B], statistics [4][K][G][B]) and the
    iterations launched.

    ``stopping_sets``: the counted positions (bool [L], ``counted_positions``) -- the stream records every frame's stopping
    sets in place of the size-two expurgation (``scldpc_bp_stream_stopping_sets``, unlimited BP only), with the unscanned
    head of ``simulate_sc_ldpc(is_bounded=False)`` below ``unscanned_head_cns``: a ``StreamStoppingSetResult``, or with
    ``collect=False`` the device tensors (iters [G][B], records [G][B][4]) and the iterations launched."""
    if stopping_sets is not None and (caps is not None or max_it):
        raise ValueError("stopping_sets needs unlimited BP: it cannot be combined with caps or max_it")
    if stopping_sets is None and unscanned_head_cns:
        raise ValueError("unscanned_head_cns applies to stopping_sets streams only")
    L = _lib.lib()
    G, B, dev = fb.n_graphs, int(frames_per_graph), fb.device
    eps_arr = np.full(G, float(eps)) if np.ndim(eps) == 0 else np.asarray(eps, np.float64)
    assert eps_arr.shape == (G,)
    arr = lambda xs: np.asarray(xs or [0], np.int32)
    hard, soft_p, soft_c = _doping(doping_points, fb.ens.M)
    a_h, a_sp, a_sc = arr(hard), arr(soft_p), arr(soft_c)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p).value
    flags = (F_TERMINATED if is_term else 0) | (F_EXP_ALL if exp_all else 0) | _sweep_flags("SCLDPC_STREAM_NODE", messages)
    # with caps, max_it goes through unchanged so that the library rejects a combination with caps
    cfg = _lib.StreamCfg(B, int(harvest_every), flags, len(hard), len(soft_p), ptr(eps_arr), ptr(a_h), ptr(a_sp), ptr(a_sc),
                         int(seed), int(first_graph_id), int(max_it) if caps is not None else max(0, int(max_it)))
    dims = ctypes.byref(fb.dims)
    if caps is not None:                       # scldpc_bp_stream_caps (the library validates the list)
        caps_arr = np.ascontiguousarray([int(c) for c in caps], np.int32)
        iters = torch.zeros((G, B), dtype=torch.int32, device=dev)
        stats = torch.zeros((4, max(len(caps_arr), 1), G, B), dtype=torch.int32, device=dev)
        outs = (iters, stats)
        call, need = L.scldpc_bp_stream_caps, L.scldpc_bp_stream_caps_workspace_bytes(dims)
        args = (caps_arr.ctypes.data_as(ctypes.c_void_p), len(caps_arr),
                ctypes.byref(_lib.StreamCapsOut(iters.data_ptr(), *[stats[i].data_ptr() for i in range(4)])))
    elif stopping_sets is not None:            # scldpc_bp_stream_stopping_sets
        cp = np.ascontiguousarray(np.asarray(stopping_sets, dtype=np.uint8))
        if cp.shape != (fb.ens.L,):
            raise ValueError("stopping_sets needs one counted flag per position")
        iters = torch.zeros((G, B), dtype=torch.int32, device=dev)
        records = torch.zeros((G, B, 4), dtype=torch.int32, device=dev)
        outs = (iters, records)
        call, need = L.scldpc_bp_stream_stopping_sets, L.scldpc_bp_stream_stopping_sets_workspace_bytes(dims)
        args = (cp.ctypes.data_as(ctypes.c_void_p), int(unscanned_head_cns),
                ctypes.byref(_lib.StreamSsOut(iters.data_ptr(), records.data_ptr())))
    else:                                      # scldpc_bp_stream: [5][G][B], iters first
        res = torch.zeros((5, G, B), dtype=torch.int32, device=dev)
        outs = (res,)
        call, need = L.scldpc_bp_stream, L.scldpc_bp_stream_workspace_bytes(dims, flags)
        args = (ctypes.byref(_lib.StreamOut(*[res[i].data_ptr() for i in range(5)])),)
    ws = fb._workspace_bytes(need)
    launched = ctypes.c_longlong(0)
    _lib.check(call(dims, ctypes.byref(fb.cbatch), ctypes.byref(cfg), *args, ctypes.c_void_p(ws.data_ptr()),
                    ctypes.c_size_t(ws.numel()), ctypes.byref(launched), _stream()))
    if not collect:
        return (*outs, launched.value)
    host = [t.cpu().numpy() for t in outs]
    kw = lambda it: dict(iters_launched=launched.value, edge_updates=int(it.astype(np.int64).sum()) * 2 * fb.ens.E)
    if caps is not None:
        it, st = host
        return StreamCapsResult(tuple(int(c) for c in caps_arr), it, *st, **kw(it))
    if stopping_sets is not None:
        it, rec = host
        return StreamStoppingSetResult(it, rec, **kw(it))
    (r,) = host
    return StreamResult(*r, **kw(r[0]))


def decode_host(ens: Ensemble, vn_cn: np.ndarray, erased: np.ndarray, W: int = 0, max_it: int = UNLIMITED, init_it: int = 0,
                is_term: bool = True, square: bool = True, trajectory: bool = False, max_rows: int = 0,
                want_erased: bool = False) -> dict:
    """One call with HOST buffers through ``scldpc_decode_host`` -- the drop-in for the reference's per-frame
    ``generate_code`` + ``channel_doped`` + ``decodeBP``/``decodeBP_SW`` sequence (BP_FULL.c:2122-2133).
    vn_cn: int32 [G][n][dv]; erased: uint8 [G][F][n]."""
    vn_cn = np.ascontiguousarray(vn_cn, np.int32)
    erased = np.ascontiguousarray(erased, np.uint8)
    G, F = erased.shape[0], erased.shape[1]
    dims = _lib.Dims(ens.dv, ens.dc, ens.L, ens.M, ens.cns_pos, G, words_for(F), F)
    flags = (F_TERMINATED if is_term else 0)
    if W > 0:
        flags |= (F_SQUARE if square else 0) | F_EXP_ALL
    if trajectory:
        flags |= F_TRAJECTORY
    o = {k: np.zeros((G, F), np.int32) for k in ("iters", "residual", "blocks_err", "erasures_exp", "blocks_err_exp", "erasures_p1")}
    vn_er = np.zeros((G, F, ens.n), np.uint8) if want_erased else None
    rows = np.zeros((G, F, max_rows, 3), np.int32) if trajectory else None
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p) if a is not None else None
    _lib.check(_lib.lib().scldpc_decode_host(ctypes.byref(dims), p(vn_cn), p(erased), int(W), int(max_it), int(init_it), flags,
                                             p(o["iters"]), p(o["residual"]), p(o["blocks_err"]), p(o["erasures_exp"]),
                                             p(o["blocks_err_exp"]), p(o["erasures_p1"]), p(vn_er), p(rows), int(max_rows)))
    o["erased"] = vn_er
    o["rows"] = rows
    return o
