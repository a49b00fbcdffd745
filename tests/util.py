"""Shared helpers of the test-suite (the oracle is imported here, in tests/, only)."""
import glob
import os

import numpy as np

import oracle

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
M32 = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """Philox-4x32-10 (Salmon et al., SC'11; Random123), restated from the paper's round function.  The counter words are
    ints or NumPy integer arrays (broadcast together, computed as uint64), the key words ints; returns the four output
    words, ints or uint64 arrays."""
    c0, c1, c2, c3 = (x.astype(np.uint64) if isinstance(x, np.ndarray) else x for x in ctr)
    k0, k1 = key
    for _ in range(10):
        p0, p1 = 0xD2511F53 * c0, 0xCD9E8D57 * c2
        c0, c1, c2, c3 = (p1 >> 32) ^ c1 ^ k0, p1 & M32, (p0 >> 32) ^ c3 ^ k1, p0 & M32
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return [c0, c1, c2, c3]


def golden_files():
    return sorted(glob.glob(os.path.join(GOLDEN_DIR, "bp_golden_*.npz")))


def load_golden(path):
    z = np.load(path)
    dv, dc, L, vns_pos, cns_pos, G, F = (int(x) for x in z["dims"])
    return z, dict(dv=dv, dc=dc, L=L, vns_pos=vns_pos, cns_pos=cns_pos, G=G, F=F, n=L * vns_pos)


def unpack_erased(packed, n):
    return np.unpackbits(packed, axis=-1)[..., :n]


def random_case(dv, dc, L, M, G, F, eps_list, seed, doped_every=0):
    """G graphs from the reference ensemble (oracle.generate_code, glibc random()) and F channel realisations each."""
    cns_pos = M * dv // dc
    oracle.srandom(seed)
    rng = np.random.default_rng(seed)
    graphs, perm = [], None
    for _ in range(G):
        g, perm = oracle.generate_code(L, M, cns_pos, dv, dc, perm)
        graphs.append(g)
    n = L * M
    chan = np.zeros((G, F, n), np.uint8)
    eps = np.zeros((G, F))
    for g in range(G):
        for f in range(F):
            e = eps_list[(g * F + f) % len(eps_list)]
            eps[g, f] = e
            chan[g, f] = rng.random(n) < e
            if doped_every and f % doped_every == doped_every - 1:
                p = int(rng.integers(0, L))
                chan[g, f, p * M:(p + 1) * M] = 0
    return graphs, chan, eps


def oracle_bp(graphs, chan, max_it, is_term, max_rows):
    G, F, n = chan.shape
    out = dict(iters=np.zeros((G, F), np.int32), residual=np.zeros((G, F), np.int32), blocks_err=np.zeros((G, F), np.int32),
               erasures_exp=np.zeros((G, F), np.int32), blocks_err_exp=np.zeros((G, F), np.int32),
               erased=np.zeros((G, F, n), np.uint8), rows=np.zeros((G, F, max_rows, 3), np.int32))
    cap = max_it if max_it > 0 else 10 ** 9
    for g in range(G):
        for f in range(F):
            o = oracle.decode_bp(graphs[g], chan[g, f].astype(np.int32), cap, is_term, max_rows=max_rows)
            for k in ("iters", "residual", "blocks_err", "erasures_exp", "blocks_err_exp"):
                out[k][g, f] = o[k]
            out["erased"][g, f] = o["erased"]
            r = o["rows"]
            out["rows"][g, f, :len(r)] = r
    return out


def oracle_sw(graphs, chan, W, max_it, init_it, square, is_term):
    G, F, n = chan.shape
    out = dict(iters=np.zeros((G, F), np.int32), residual=np.zeros((G, F), np.int32), blocks_err=np.zeros((G, F), np.int32),
               erasures_exp=np.zeros((G, F), np.int32), blocks_err_exp=np.zeros((G, F), np.int32),
               erasures_p1=np.zeros((G, F), np.int32), erased=np.zeros((G, F, n), np.uint8))
    cap = max_it if max_it > 0 else 10 ** 9
    for g in range(G):
        for f in range(F):
            o = oracle.decode_bp_sw(graphs[g], chan[g, f].astype(np.int32), W, cap, init_it, square, is_term)
            for k in ("residual", "blocks_err", "erasures_exp", "blocks_err_exp", "erasures_p1"):
                out[k][g, f] = o[k]
            out["iters"][g, f] = o["win_iters"].sum()
            out["erased"][g, f] = o["erased"]
    return out


def stream_compactions(fb):
    """(compactions, frames moved) of the last node-state stream call on fb's workspace (scldpc_bp_sweep_stats)"""
    import ctypes
    from fl_scaling_sc_ldpc_b200 import _lib
    st = (ctypes.c_longlong * 2)()
    _lib.check(_lib.lib().scldpc_bp_sweep_stats(ctypes.byref(fb.dims), 32, ctypes.c_void_p(fb._ws.data_ptr()), st))   # SCLDPC_F_STREAM
    return int(st[0]), int(st[1])
