"""CPU oracle for the SC-LDPC BEC decoders -- TEST INFRASTRUCTURE ONLY.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s ``cpu_baseline`` / ``--impl reference`` legs may
import this package, and only as the checker or the CPU baseline -- never as the thing measured or shipped.
The product package ``fl_scaling_sc_ldpc_b200`` must not (and does not) import it.

Contents
--------
* ``scldpc_oracle.c``  plain-C restatement of the reference algorithms (each function cites file:line),
                       loaded here through ctypes (``libscldpc_oracle.so``, built by ``oracle/Makefile``).
* ``build_ref.py`` / ``ref_driver.py``  the UNMODIFIED reference C files compiled in place from
                       ``/root/reference`` into ``oracle/_ref/*.so`` and driven through ctypes.
* ``peeling_ref.py``   imports the reference's own ``peeling_decoding.py`` (in this container only) with the
                       inputs injected, to pin the peeling restatements and generate ``tests/golden``.

Parity status: pinned against the compiled reference (see the header of ``scldpc_oracle.c``).
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(HERE, "libscldpc_oracle.so")
_lib = None

_i32p = np.ctypeslib.ndpointer(dtype=np.int32, flags="C_CONTIGUOUS")
_u8p = np.ctypeslib.ndpointer(dtype=np.uint8, flags="C_CONTIGUOUS")


def build(force: bool = False) -> str:
    src = os.path.join(HERE, "scldpc_oracle.c")
    if force or not os.path.isfile(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-s", "-C", HERE, "libscldpc_oracle.so"], check=True)
    return _LIB_PATH


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.orc_decode_bp.restype = ctypes.c_int
        _lib.orc_decode_bp_sw.restype = ctypes.c_int
        _lib.orc_build_cn.restype = ctypes.c_int
        _lib.orc_peel_trajectory.restype = ctypes.c_int
        _lib.orc_peel_trajectory_fast.restype = ctypes.c_int
        _lib.orc_is_position_doped_streaming.restype = ctypes.c_int
    return _lib


_libc = ctypes.CDLL(None)


def srandom(seed: int):
    _libc.srandom(ctypes.c_uint(seed))


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


class Graph:
    """VN->CN table plus the CN-side tables in the reference's order (``orc_build_cn``)."""

    def __init__(self, vn_cn: np.ndarray, L: int, vns_pos: int, cns_pos: int, dv: int, dc: int, nk: int | None = None):
        self.L, self.vns_pos, self.cns_pos, self.dv, self.dc = L, vns_pos, cns_pos, dv, dc
        self.n = L * vns_pos
        self.nk = (L + dv - 1) * cns_pos if nk is None else nk
        self.vn_cn = np.ascontiguousarray(vn_cn, dtype=np.int32).reshape(self.n, dv)
        self.cn_deg = np.zeros(self.nk, np.int32)
        self.cn_vn = np.zeros((self.nk, dc), np.int32)
        self.cn_ei = np.zeros((self.nk, dc), np.int32)
        self.vn_slot = np.zeros((self.n, dv), np.int32)
        rc = lib().orc_build_cn(self.n, self.nk, dv, dc, _ptr(self.vn_cn), _ptr(self.cn_deg), _ptr(self.cn_vn),
                                _ptr(self.cn_ei), _ptr(self.vn_slot))
        if rc != 0:
            raise ValueError("invalid graph (CN index out of range or CN degree > dc)")


def generate_code(L: int, vns_pos: int, cns_pos: int, dv: int, dc: int, perm_code: np.ndarray | None = None):
    """``orc_generate_code``; returns (Graph, perm_code).  Seed glibc with ``srandom`` first."""
    if perm_code is None:
        perm_code = np.arange(cns_pos * dc, dtype=np.int32)
    vn_cn = np.zeros((L * vns_pos, dv), np.int32)
    lib().orc_generate_code(L, vns_pos, cns_pos, dv, dc, _ptr(perm_code), _ptr(vn_cn))
    return Graph(vn_cn, L, vns_pos, cns_pos, dv, dc), perm_code


def channel_doped(n: int, eps: float, vns_pos: int, doped=()) -> np.ndarray:
    chan = np.zeros(n, np.int32)
    d = np.asarray(list(doped) or [0], np.int32)
    lib().orc_channel_doped(n, ctypes.c_double(eps), vns_pos, len(doped), _ptr(d), _ptr(chan))
    return chan


def is_position_doped_streaming(pos: int, doped) -> bool:
    d = np.asarray(list(doped) or [0], np.int32)
    return bool(lib().orc_is_position_doped_streaming(pos, len(doped), _ptr(d)))


def decode_bp(g: Graph, chan: np.ndarray, max_it: int, is_term: int = 1, max_rows: int | None = None,
              want_msgs: bool = False, exp_positions: int | None = None) -> dict:
    """``orc_decode_bp`` (reference ``decodeBP``).  ``exp_positions`` is the ``L`` argument, which a terminated decode
    uses only as the range of its post-decoding expurgation scan; 0 skips that scan, as ``ref_driver``'s does."""
    chan = np.ascontiguousarray(chan, np.int32)
    Larg = g.L if exp_positions is None else exp_positions
    assert is_term or Larg == g.L
    erased = np.zeros(g.n, np.uint8)
    max_rows = max(1, max_it) if max_rows is None else max_rows
    rows = np.zeros((max_rows, 3), np.int32)
    it, nb, ne, nbe = (ctypes.c_int(0) for _ in range(4))
    lji = np.zeros((g.n, g.dv), np.int32) if want_msgs else None
    lij = np.zeros((g.n, g.dv), np.int32) if want_msgs else None
    res = lib().orc_decode_bp(g.n, g.nk, Larg, g.vns_pos, g.cns_pos, g.dv, g.dc, _ptr(g.vn_cn), _ptr(g.cn_deg),
                              _ptr(g.cn_vn), _ptr(g.cn_ei), _ptr(g.vn_slot), _ptr(chan), max_it, is_term,
                              _ptr(erased), ctypes.byref(it), ctypes.byref(nb), ctypes.byref(ne), ctypes.byref(nbe),
                              _ptr(rows), max_rows, _ptr(lji), _ptr(lij))
    return dict(residual=int(res), iters=it.value, blocks_err=nb.value, erasures_exp=ne.value,
                blocks_err_exp=nbe.value, erased=erased, rows=rows[: min(it.value, max_rows)].copy(),
                v2c=lji, c2v=lij)


def decode_bp_sw(g: Graph, chan: np.ndarray, W: int, max_it: int, init_it: int = 0, square: int = 1,
                 is_term: int = 1, want_msgs: bool = False) -> dict:
    """``orc_decode_bp_sw`` (reference ``decodeBP_SW``).  ``init_it == 0`` means ``max_it`` (BP_SW.c:2099-2102)."""
    chan = np.ascontiguousarray(chan, np.int32)
    if init_it == 0:
        init_it = max_it
    erased = np.zeros(g.n, np.uint8)
    nwin = g.L if square else g.L + g.dv - 1
    win_iters = np.zeros(nwin, np.int32)
    p1, nb, ne, nbe = (ctypes.c_int(0) for _ in range(4))
    lji = np.zeros((g.n, g.dv), np.int32) if want_msgs else None
    lij = np.zeros((g.n, g.dv), np.int32) if want_msgs else None
    res = lib().orc_decode_bp_sw(g.n, g.nk, g.L, W, g.vns_pos, g.cns_pos, g.dv, g.dc, _ptr(g.vn_cn), _ptr(g.cn_deg),
                                 _ptr(g.cn_vn), _ptr(g.cn_ei), _ptr(g.vn_slot), _ptr(chan), max_it, init_it, square,
                                 is_term, _ptr(erased), ctypes.byref(p1), ctypes.byref(nb), ctypes.byref(ne),
                                 ctypes.byref(nbe), _ptr(win_iters), _ptr(lji), _ptr(lij))
    return dict(residual=int(res), erasures_p1=p1.value, blocks_err=nb.value, erasures_exp=ne.value,
                blocks_err_exp=nbe.value, erased=erased, win_iters=win_iters, v2c=lji, c2v=lij)


def position_counts(g: Graph, erased: np.ndarray):
    """``orc_position_counts``: per position (erased VNs, expurgated erased VNs as in ``get_deg_two_ss``)."""
    erased = np.ascontiguousarray(erased, np.uint8)
    plain = np.zeros(g.L, np.int32)
    ex = np.zeros(g.L, np.int32)
    lib().orc_position_counts(g.n, g.nk, g.L, g.vns_pos, g.dv, g.dc, _ptr(g.vn_cn), _ptr(g.cn_deg), _ptr(g.cn_vn), _ptr(erased),
                              _ptr(plain), _ptr(ex))
    return plain, ex


def stream_counters(plain: np.ndarray, ex: np.ndarray, n_steps: int, dv: int):
    """main_streaming's running counters (BP_FULL.c:2015-2031, decodeBP_SW_circular :1483-1497) after each of n_steps
    decode steps, from per-position counts: step `pos` decides absolute position pos-dv+1 and expurgates pos-2*dv+1.
    Returns int64 [n_steps][4] = (NumErasuresPos of the step, num_blocks_err, num_erasures_exp, num_blocks_err_exp)."""
    out = np.zeros((n_steps, 4), np.int64)
    nb = ne = nbe = 0
    for pos in range(n_steps):
        q = pos - dv + 1
        er = int(plain[q]) if q >= 0 else 0
        nb += er > 0
        q2 = pos - 2 * dv + 1
        if q2 >= 0 and ex[q2] > 0:
            ne += int(ex[q2]); nbe += 1
        out[pos] = (er, nb, ne, nbe)
    return out


def peel_trajectory(vn_cn: np.ndarray, erased: np.ndarray, total_size: int, n_cn_all: int, num_steps: int,
                    picks: np.ndarray):
    """``orc_peel_trajectory`` (PD.py:705-789 with an injected pick sequence).  Returns (r1, recovered)."""
    vn_cn = np.ascontiguousarray(vn_cn, np.int32)
    erased = np.ascontiguousarray(erased, np.uint8)
    picks = np.ascontiguousarray(picks, np.uint32)
    assert picks.size >= num_steps
    r1 = np.zeros(num_steps + 1, np.int64)
    rec = lib().orc_peel_trajectory(vn_cn.shape[0], vn_cn.shape[1], total_size, n_cn_all, _ptr(vn_cn), _ptr(erased),
                                    num_steps, _ptr(picks), _ptr(r1))
    return r1, int(rec)


def peel_trajectory_fast(vn_cn: np.ndarray, erased: np.ndarray, total_size: int, n_cn_all: int, num_steps: int,
                         picks: np.ndarray):
    """``orc_peel_trajectory_fast``: what ``peel_trajectory`` returns, in O(log #CN) per step (a Fenwick tree over the
    degree-one CNs) instead of a scan -- full-length trajectories at M >= 10^4."""
    vn_cn = np.ascontiguousarray(vn_cn, np.int32)
    erased = np.ascontiguousarray(erased, np.uint8)
    picks = np.ascontiguousarray(picks, np.uint32)
    assert picks.size >= num_steps
    r1 = np.zeros(num_steps + 1, np.int64)
    rec = lib().orc_peel_trajectory_fast(vn_cn.shape[0], vn_cn.shape[1], total_size, n_cn_all, _ptr(vn_cn), _ptr(erased),
                                         num_steps, _ptr(picks), _ptr(r1))
    return r1, int(rec)


def peel_fixed_point(vn_cn: np.ndarray, erased: np.ndarray, n_cn_all: int, scan_lo: int, cn_hi: int) -> np.ndarray:
    vn_cn = np.ascontiguousarray(vn_cn, np.int32)
    erased = np.ascontiguousarray(erased, np.uint8)
    lost = np.zeros(vn_cn.shape[0], np.uint8)
    lib().orc_peel_fixed_point(vn_cn.shape[0], vn_cn.shape[1], n_cn_all, scan_lo, cn_hi, _ptr(vn_cn), _ptr(erased),
                               _ptr(lost))
    return lost
