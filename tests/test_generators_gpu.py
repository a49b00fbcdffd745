"""The on-device generators (scldpc_graph_generate(_at), scldpc_channel_generate(_at)) against a NumPy restatement of their
Philox draws, bit for bit.

Every decoder test compares two decoders on the same graph and the same erasures, so a generator that is subtly wrong (a
sort that no longer sorts, a counter word that repeats) passes all of them while biasing every error rate.  The
restatements below follow the documented construction, not the kernels:

* graphs: CN position pos (absolute) of graph id gid draws one Philox call per socket pair q, counter (q, pos, gid.lo,
  gid.hi), key (seed.lo ^ 'grap', seed.hi); socket s = 2q+h gets the key (44 high bits of r[2h]:r[2h+1]) << 20 | s, and
  perm = argsort(keys).  VN t of position p, edge i, takes socket dv*t+i of CN position cp = p+i (mod L tail-biting)
  and goes to CN cp*cns_pos + perm_cp[dv*t+i] // dc (orc_generate_code).  The protograph ensemble sorts one segment of
  S = cns_pos keys per (position, portion, edge type), numbered in that order;
* channels: frame f of VN v is erased iff philox((first_vn+v, (first_frame+f) >> 2, gid.lo, gid.hi),
  (seed.lo ^ 'chan', seed.hi))[f & 3] < floor(eps * 2^32), unless doping makes v known.

The comparisons cover whole vn_cn tensors and raw channel words (unused lanes and words included), with both buffers
filled with ones before the call so that a word the kernel does not write shows up."""
import ctypes
import math

import numpy as np
import pytest

import fl_scaling_sc_ldpc_b200 as eng
from fl_scaling_sc_ldpc_b200 import _lib, streaming
from fl_scaling_sc_ldpc_b200 import sc_ldpc as scx, sc_ldpc_protograph as spx
from tests.util import M32, philox4x32_10

gpu = pytest.mark.gpu
TAG_GRAPH, TAG_CHAN = 0x67726170, 0x6368616E
U32 = 1 << 32


# ---- restatements ---------------------------------------------------------------------------------------------------
def socket_perms(seed, gid, counters, S):
    """[len(counters)][S]: perm[j][r] = the socket carried by the r-th smallest of the S keys of the segment whose
    position counter word is counters[j]"""
    q = np.arange((S + 1) // 2, dtype=np.uint64)[None, :]
    pos = np.asarray(counters, np.uint64)[:, None]
    r = philox4x32_10((q, pos, gid & M32, gid >> 32), ((seed & M32) ^ TAG_GRAPH, seed >> 32))
    rnd = np.stack([((r[0] << 32) | r[1]) >> 20, ((r[2] << 32) | r[3]) >> 20], axis=-1).reshape(len(counters), -1)[:, :S]
    return np.argsort((rnd << 20) | np.arange(S, dtype=np.uint64), axis=1)


def semi_structured(dv, dc, L, M, seed, gid, first_position=0, tail_biting=False):
    """vn_cn [L*M][dv] of the semi-structured ensemble (tail-biting: L CN positions, cp mod L; else L+dv-1)"""
    cns = M * dv // dc
    perm = socket_perms(seed, gid, first_position + np.arange(L if tail_biting else L + dv - 1), cns * dc)
    p, t, i = np.ogrid[:L, :M, :dv]
    cp = (p + i) % L if tail_biting else p + i
    return (cp * cns + perm[cp, dv * t + i] // dc).reshape(L * M, dv)


def protograph(dv, dc, L, M, seed, gid):
    """vn_cn [L*M][dv] of the protograph-based ensemble: edge i of VN t of portion q of position p goes to CN perm[t] of
    position p+i, one permutation of the cns_pos CNs per (p, q, i)"""
    cns = M * dv // dc
    P = M // cns
    perm = socket_perms(seed, gid, np.arange(L * P * dv), cns).reshape(L, P, dv, cns)
    p, q, t, i = np.ogrid[:L, :P, :cns, :dv]
    return ((p + i) * cns + perm[p, q, i, t]).reshape(L * M, dv)


def graphs(fn, G, gid, dv, dc, L, M, seed, **kw):
    """[G][L*M][dv]: graph g of a batch is graph id gid + g"""
    return np.stack([fn(dv, dc, L, M, seed, gid + g, **kw) for g in range(G)])


def known_counts(L, M, hard=(), soft=None):
    """known leading VNs per position: hard doping all M, soft clamp(int(alpha*M), 0, M), the larger of the two"""
    k = np.zeros(L, np.int64)
    for p in hard:
        k[p] = M
    for p, a in (soft or {}).items():
        k[p] = max(k[p], min(max(int(a * M), 0), M))
    return k


def threshold(eps):
    return 0 if eps <= 0 else (U32 if eps >= 1 else int(eps * U32))


def channel(n, n_frames, n_words, eps, seed, gid, first_frame=0, first_vn=0, known=None, M=1):
    """raw bit-sliced words uint64 [n][n_words]: bit b of word w is frame 64w+b; lanes >= n_frames are 0"""
    thr = threshold(eps)
    key = ((seed & M32) ^ TAG_CHAN, seed >> 32)
    v = first_vn + np.arange(n, dtype=np.uint64)
    words = np.zeros((n, n_words), np.uint64)
    for b in range((n_frames + 3) // 4):
        r = philox4x32_10((v, (first_frame >> 2) + b, gid & M32, gid >> 32), key)
        for h in range(min(4, n_frames - 4 * b)):
            f = 4 * b + h
            words[:, f >> 6] |= (r[h] < thr).astype(np.uint64) << np.uint64(f & 63)
    if known is not None:
        words[(np.arange(n) % M) < np.repeat(known, M)] = 0
    return words


def channels(G, gid, eps, n, n_frames, n_words, seed, **kw):
    """[G][n][n_words]: graph g of a batch is graph id gid + g; eps a float or one per graph"""
    eps = eps if np.ndim(eps) else [eps] * G
    return np.stack([channel(n, n_frames, n_words, eps[g], seed, gid + g, **kw) for g in range(G)])


# ---- the device side ------------------------------------------------------------------------------------------------
def drawn_graphs(ens, G, seed, gid=0, **kw):
    fb = eng.FrameBatch(ens, G, 0, 2)
    fb.vn_cn.fill_(-1)
    fb.generate_graphs(seed, first_graph_id=gid, **kw)
    out = fb.vn_cn.cpu().numpy()
    assert fb.graph_error() == 0
    return out


def drawn_channel(fb, *args, **kw):
    fb.chan.fill_(-1)
    fb.generate_erasures(*args, **kw)
    return fb.chan.cpu().numpy().view(np.uint64)


def assert_same(got, want, what):
    assert got.shape == want.shape, (what, got.shape, want.shape)
    bad = np.argwhere(got != want)
    assert len(bad) == 0, f"{what}: {len(bad)} of {got.size} entries differ, first at {bad[:4].tolist()}"


# ---- CPU: the restatement itself is a valid ensemble ------------------------------------------------------------------
def test_restatement_is_a_valid_code(oracle_mod):
    """every CN position's sockets are a permutation (interior CNs have degree dc), tail-biting CNs all have degree dc,
    and every protograph (position, portion, edge type) column is a permutation of the position's CNs"""
    dv, dc, L, M = 4, 8, 7, 48
    cns = M * dv // dc
    vn = semi_structured(dv, dc, L, M, 5, 1)
    oracle_mod.Graph(vn, L, M, cns, dv, dc)
    deg = np.bincount(vn.ravel(), minlength=(L + dv - 1) * cns)
    assert (deg[(dv - 1) * cns: L * cns] == dc).all() and deg.max() == dc
    assert ((vn // cns) == np.arange(L).repeat(M)[:, None] + np.arange(dv)).all()
    tb = semi_structured(dv, dc, L, M, 5, 1, tail_biting=True)
    assert (np.bincount(tb.ravel(), minlength=L * cns) == dc).all()
    pg = protograph(dv, dc, L, M, 5, 1).reshape(L, M // cns, cns, dv)
    for p in range(L):
        for i in range(dv):
            assert (np.sort(pg[p, :, :, i], axis=1) == (p + i) * cns + np.arange(cns)).all()
    # the permutations change with every counter word
    a = socket_perms(7, 3, [0, 1], 64)
    assert not (a[0] == a[1]).all()
    assert not (a == socket_perms(7, 3 + U32, [0, 1], 64)).all() and not (a == socket_perms(7 + U32, 3, [0, 1], 64)).all()


# ---- graphs -----------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dv,dc,L,M,G", [
    (4, 8, 6, 1000, 2),       # 4000 sockets, Spad = 4096 = SORT_TILE: the largest single-tile sort
    (4, 8, 5, 1026, 2),       # 4104 sockets: one key over a tile, about half of the 8192 slots are padding
    (4, 8, 50, 10000, 1),     # the benchmark's graphs: 40000 sockets in 65536 slots, 16 tiles
    (4, 8, 2, 100000, 1),     # 2^19 slots: the global passes loop over the 64-block grid
    (3, 6, 5, 100, 2), (3, 6, 4, 3000, 1),
    (5, 10, 6, 100, 2), (5, 10, 3, 2000, 1),
    (3, 9, 5, 99, 2), (3, 9, 3, 3000, 1),
    (4, 12, 6, 99, 2), (4, 12, 3, 3000, 1),
])
def test_semi_structured_graphs_match_restatement(dv, dc, L, M, G):
    ens = eng.Ensemble(dv, dc, L, M)
    got = drawn_graphs(ens, G, 91, 12)
    assert_same(got, graphs(semi_structured, G, 12, dv, dc, L, M, 91), f"({dv},{dc}) L={L} M={M}")


@gpu
def test_key_layout_limit():
    """the key holds the socket index in 20 bits: cns_pos*dc = 2^20 is drawn and restated, 2^20 + 8 is refused"""
    ens = eng.Ensemble(4, 8, 1, 262144)
    assert ens.cns_pos * 8 == 1 << 20
    assert_same(drawn_graphs(ens, 1, 3, 0), semi_structured(4, 8, 1, 262144, 3, 0)[None], "2^20 sockets")
    with pytest.raises(eng.ScldpcError):
        drawn_graphs(eng.Ensemble(4, 8, 1, 262146), 1, 3, 0)


@gpu
@pytest.mark.parametrize("dv,dc,L,M,G", [(4, 8, 6, 48, 3), (3, 6, 5, 40, 2), (4, 8, 50, 10000, 1)])
def test_tail_biting_graphs_match_restatement(dv, dc, L, M, G):
    got = drawn_graphs(eng.Ensemble(dv, dc, L, M), G, 23, 4, tail_biting=True)
    assert_same(got, graphs(semi_structured, G, 4, dv, dc, L, M, 23, tail_biting=True), f"tail-biting M={M}")


@gpu
@pytest.mark.parametrize("dv,dc,L,M,G", [
    (4, 8, 10, 10000, 1),     # 5000 CNs per segment: a two-tile sort
    (4, 8, 6, 2, 3),          # cns_pos = 1: Spad = 2
    (4, 8, 6, 6, 3),          # cns_pos = 3
    (3, 9, 4, 300, 2),
])
def test_protograph_graphs_match_restatement(dv, dc, L, M, G):
    got = drawn_graphs(eng.Ensemble(dv, dc, L, M), G, 31, 8, protograph=True)
    assert_same(got, graphs(protograph, G, 8, dv, dc, L, M, 31), f"protograph M={M}")


@gpu
def test_high_counter_words():
    """graph ids and seeds past 2^32 reach the high counter / key words; G > 1 advances the graph id per graph"""
    dv, dc, L, M, G = 4, 8, 6, 1026, 3
    ens = eng.Ensemble(dv, dc, L, M)
    for seed, gid in ((0x1234_5678_9ABC_DEF0, 5), (77, (3 << 32) + 5), (U32 + 9, U32 - 2)):
        assert_same(drawn_graphs(ens, G, seed, gid), graphs(semi_structured, G, gid, dv, dc, L, M, seed), f"graph {seed:#x} {gid:#x}")
        fb = eng.FrameBatch(ens, G, 100)
        got = drawn_channel(fb, 0.47, seed, first_graph_id=gid, first_frame=64)
        assert_same(got, channels(G, gid, 0.47, ens.n, 100, 2, seed, first_frame=64), f"channel {seed:#x} {gid:#x}")


@gpu
def test_ensemble_drop_ins():
    """sc_ldpc.set_seed then gen_slots draw graph ids 0, 1, 2 of the seed's stream; the tail-biting and protograph drop-ins
    take the next ids"""
    seed = 0xC0FFEE
    scx.set_seed(seed)
    for gid in range(3):
        tr = scx.gen_slots(4, 8, 5, 64)
        assert tr.dtype == np.int64
        assert_same(tr, semi_structured(4, 8, 5, 64, seed, gid), f"gen_slots #{gid}")
    assert_same(scx.gen_slots_tail_biting(3, 6, 5, 40), semi_structured(3, 6, 5, 40, seed, 3, tail_biting=True), "tail-biting")
    assert_same(spx.gen_slots_from_position(4, 8, 48), protograph(4, 8, 1, 48, seed, 4), "gen_slots_from_position")


# ---- chain pieces -----------------------------------------------------------------------------------------------------
@gpu
def test_chain_pieces_regenerate_the_full_chain():
    """streaming.ChainPieces draws the piece at absolute position A as the columns of one 40-position chain: the graph
    is full[A*M:(A+Lloc)*M] - A*cns_pos, the channel the full chain's VN columns; doping is periodic in absolute
    positions and passed to the generator as local ones"""
    dv, dc, M, Lfull, G, F, seed, gid = 4, 8, 1026, 40, 2, 100, 4242, 6
    doped = [3, 7]                                  # period 8: absolute positions 3 and 7 mod 8
    cp = streaming.ChainPieces(dv, dc, M, 3, 0.46, doped, G, F, seed, first_graph_id=gid, piece=4)
    Lloc, cns = cp.Lloc, cp.ens.cns_pos
    full = eng.FrameBatch(eng.Ensemble(dv, dc, Lfull, M), G, F)
    full.generate_graphs(seed, first_graph_id=gid)
    full.generate_erasures(0.46, seed + 1, first_graph_id=gid,
                           doping_points=[p for p in range(Lfull) if streaming.is_position_doped_streaming(p, doped)])
    fvn, fch = full.vn_cn.cpu().numpy(), full.chan.cpu().numpy().view(np.uint64)
    assert_same(fvn, graphs(semi_structured, G, gid, dv, dc, Lfull, M, seed), "full chain")
    for A in (0, 1, 17):
        assert A + Lloc <= Lfull
        cp.A = A
        cp.fb.vn_cn.fill_(-1)
        cp.fb.chan.fill_(-1)
        cp._load()
        vn, ch = cp.fb.vn_cn.cpu().numpy(), cp.fb.chan.cpu().numpy().view(np.uint64)
        assert_same(vn, fvn[:, A * M:(A + Lloc) * M] - A * cns, f"piece graph A={A}")
        assert_same(ch, fch[:, A * M:(A + Lloc) * M], f"piece channel A={A}")
        assert_same(vn, graphs(semi_structured, G, gid, dv, dc, Lloc, M, seed, first_position=A), f"restated graph A={A}")
        local = [j for j in range(Lloc) if streaming.is_position_doped_streaming(A + j, doped)]
        assert local and ch[:, local[0] * M:(local[0] + 1) * M].max() == 0
        want = channels(G, gid, 0.46, Lloc * M, F, 2, seed + 1, first_vn=A * M, known=known_counts(Lloc, M, local), M=M)
        assert_same(ch, want, f"restated channel A={A}")


@gpu
def test_counter_bounds(oracle_mod):
    """VN ids, frame ids and CN positions are 32-bit counter words: the largest accepted first_vn, first_frame and
    first_position draw the restated realisations and decode like the oracle; one more raises ValueError before any
    device work, where the counters used to wrap silently onto earlier realisations"""
    dv, dc, L, M, G, F, seed, gid = 4, 8, 6, 40, 2, 1024, 515, 9
    ens = eng.Ensemble(dv, dc, L, M)
    n, cns = ens.n, ens.cns_pos
    fb = eng.FrameBatch(ens, G, F)
    assert fb.n_words == 16
    top_vn, top_frame, top_pos = U32 - n, U32 - 64 * 16, U32 - (L + dv - 1)
    fb.vn_cn.fill_(-1)
    fb.generate_graphs(seed, first_graph_id=gid, first_position=top_pos)
    assert_same(fb.vn_cn.cpu().numpy(), graphs(semi_structured, G, gid, dv, dc, L, M, seed, first_position=top_pos), "top position")
    got = drawn_channel(fb, 0.45, seed + 1, first_graph_id=gid, first_frame=top_frame, first_vn=top_vn, doping_points=[2])
    want = channels(G, gid, 0.45, n, F, 16, seed + 1, first_frame=top_frame, first_vn=top_vn, known=known_counts(L, M, [2]), M=M)
    assert_same(got, want, "top VN and frame ids")
    res = eng.decode_bp_full(fb, 0, True)
    er, vn = fb.erasures_host(), fb.vn_cn.cpu().numpy()
    for g in range(G):
        gr = oracle_mod.Graph(vn[g], L, M, cns, dv, dc)
        for f in (0, 511, 1023):
            o = oracle_mod.decode_bp(gr, er[g, f].astype(np.int32), 10 ** 9, 1)
            assert (o["iters"], o["residual"]) == (res.iters[g, f], res.residual[g, f]), (g, f)
    fb.chan.fill_(-1)
    fb.vn_cn.fill_(-1)
    for kw in (dict(first_vn=top_vn + 1), dict(first_vn=-M), dict(first_frame=top_frame + 4), dict(first_frame=-4),
               dict(first_vn=top_vn + 1, first_frame=top_frame)):
        with pytest.raises(ValueError):
            fb.generate_erasures(0.45, seed + 1, first_graph_id=gid, **kw)
    for ff in (top_frame + 4, -4):
        with pytest.raises(ValueError):
            fb.generate_erasures([0.4] * G, seed + 1, first_graph_id=gid, first_frame=ff)
    for pos in (top_pos + 1, U32, -1):
        with pytest.raises(ValueError):
            fb.generate_graphs(seed, first_graph_id=gid, first_position=pos)
    assert (fb.chan.cpu().numpy() == -1).all() and (fb.vn_cn.cpu().numpy() == -1).all()      # no kernel ran
    # a narrower batch has a larger largest first_frame: every lane of its n_words has a frame id
    fb2 = eng.FrameBatch(ens, 1, 100, 2)
    assert_same(drawn_channel(fb2, 0.5, 3, first_frame=U32 - 128), channels(1, 0, 0.5, n, 100, 2, 3, first_frame=U32 - 128), "W=2 top")
    with pytest.raises(ValueError):
        fb2.generate_erasures(0.5, 3, first_frame=U32 - 124)
    # ChainPieces checks through the same calls: the largest piece start whose VN ids fit draws the restatement
    cp = streaming.ChainPieces(dv, dc, M, 3, 0.45, [], 1, 64, seed, first_graph_id=gid, piece=4)
    cp.A = U32 // M - cp.Lloc
    cp._load()
    want = channels(1, gid, 0.45, cp.ens.n, 64, 2, seed + 1, first_vn=cp.A * M)
    assert_same(cp.fb.chan.cpu().numpy().view(np.uint64), want, "top piece")
    cp.A += 1
    with pytest.raises(ValueError):
        cp._load()


# ---- channels ---------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("eps", [0.0, 2.0 ** -32, 0.4625, 0.5, 1 - 2.0 ** -32, 1.0])
def test_channel_thresholds(eps):
    """thr = floor(eps*2^32), 0 at eps = 0 and 2^32 at eps = 1; lanes 100..255 stay 0 even when every draw erases"""
    ens = eng.Ensemble(4, 8, 5, 200)
    fb = eng.FrameBatch(ens, 2, 100, 4)
    got = drawn_channel(fb, eps, 61, first_graph_id=3)
    assert_same(got, channels(2, 3, eps, ens.n, 100, 4, 61), f"eps={eps!r}")
    if eps == 1.0:
        assert (got[..., 0] == np.uint64(2 ** 64 - 1)).all() and (got[..., 1] == (1 << 36) - 1).all() and not got[..., 2:].any()


@gpu
def test_channel_threshold_is_strict_at_a_drawn_value():
    """erased iff draw < thr: with eps = d / 2^32 for a draw d of the stream (exact in double), that draw's bit is
    clear, and set at eps = (d+1) / 2^32"""
    ens = eng.Ensemble(4, 8, 3, 64)
    seed, gid = 101, 2
    fb = eng.FrameBatch(ens, 1, 64, 2)
    d = philox4x32_10((5, 0, gid, 0), ((seed & M32) ^ TAG_CHAN, 0))      # frames 0..3 of VN 5
    for h in range(4):
        for bump, erased in ((0, 0), (1, 1)):
            eps = (d[h] + bump) / U32
            assert threshold(eps) == d[h] + bump
            got = drawn_channel(fb, eps, seed, first_graph_id=gid)
            assert int(got[0, 5, 0] >> np.uint64(h)) & 1 == erased, (h, d[h], bump)
            assert_same(got, channels(1, gid, eps, ens.n, 64, 2, seed), f"eps = ({d[h]} + {bump}) / 2^32")


@gpu
@pytest.mark.parametrize("n_frames,n_words", [(1, 16), (63, 2), (64, 4), (65, 2), (100, 8), (1024, 16)])
def test_channel_frames_and_words(n_frames, n_words):
    """bit f of the lanes is frame f for f < n_frames and 0 beyond, in every word the batch has"""
    ens = eng.Ensemble(3, 6, 4, 300)
    fb = eng.FrameBatch(ens, 2, n_frames, n_words)
    got = drawn_channel(fb, 0.5, 17, first_graph_id=40)
    assert_same(got, channels(2, 40, 0.5, ens.n, n_frames, n_words, 17), f"{n_frames} frames in {n_words} words")
    lanes = np.unpackbits(got.view(np.uint8).reshape(2, ens.n, -1), axis=2, bitorder="little")
    assert not lanes[:, :, n_frames:].any() and lanes[:, :, :n_frames].any()


@gpu
@pytest.mark.parametrize("first_frame", [4, 1020, U32 - 1024])
def test_channel_first_frame(first_frame):
    """lane f holds frame first_frame + f: the batch equals the restatement and the matching lanes of a batch from frame 0"""
    ens = eng.Ensemble(4, 8, 4, 100)
    fb = eng.FrameBatch(ens, 2, 1000, 16)
    got = drawn_channel(fb, 0.42, 7, first_graph_id=11, first_frame=first_frame)
    assert_same(got, channels(2, 11, 0.42, ens.n, 1000, 16, 7, first_frame=first_frame), f"first_frame={first_frame}")
    if first_frame < 1000:
        a = fb.erasures_host()
        b = eng.FrameBatch(ens, 2, 1000, 16).generate_erasures(0.42, 7, first_graph_id=11).erasures_host()
        assert (a[:, :1000 - first_frame] == b[:, first_frame:]).all()


@gpu
def test_channel_per_graph_eps_and_doping():
    """one eps per graph (graph g at id first_graph_id + g); hard doping zeroes whole positions, soft doping the first
    clamp(int(alpha*M), 0, M) VNs of a position"""
    dv, dc, L, M, G, F = 4, 8, 8, 250, 3, 200
    ens = eng.Ensemble(dv, dc, L, M)
    fb = eng.FrameBatch(ens, G, F)
    eps = [0.1, 0.5, 0.9]
    for doping in ([], [0, 5, 7], {1: 0.25, 2: 1.5, 3: -0.5, 4: 0.999, 6: 1.0}):
        hard = [] if isinstance(doping, dict) else doping
        soft = doping if isinstance(doping, dict) else None
        got = drawn_channel(fb, eps, 29, first_graph_id=U32 - 1, doping_points=doping, first_frame=8)
        want = channels(G, U32 - 1, eps, ens.n, F, fb.n_words, 29, first_frame=8, known=known_counts(L, M, hard, soft), M=M)
        assert_same(got, want, f"doping {doping}")
    assert known_counts(L, M, [], {1: 0.25, 2: 1.5, 3: -0.5, 4: 0.999}).tolist() == [0, 62, 250, 0, 249, 0, 0, 0]


@gpu
def test_channel_hard_and_soft_doping_of_one_position():
    """through the C ABI a position can be both hard- and soft-doped: the larger count wins"""
    dv, dc, L, M, F = 4, 8, 5, 120, 64
    ens = eng.Ensemble(dv, dc, L, M)
    fb = eng.FrameBatch(ens, 1, F)
    fb.chan.fill_(-1)
    arr = lambda xs: (ctypes.c_int32 * len(xs))(*xs)
    _lib.check(_lib.lib().scldpc_channel_generate(
        ctypes.byref(fb.dims), ctypes.c_void_p(fb.chan.data_ptr()), ctypes.c_double(0.6), arr([1, 3]), 2,
        arr([1, 2, 4]), arr([30, 45, 500]), 3, ctypes.c_uint64(5), ctypes.c_uint64(0), ctypes.c_uint32(0), eng.engine._stream()))
    known = np.array([0, M, 45, M, M])
    assert_same(fb.chan.cpu().numpy().view(np.uint64), channels(1, 0, 0.6, ens.n, F, 2, 5, known=known, M=M), "hard + soft")


@gpu
def test_channel_rejects_bad_arguments():
    ens = eng.Ensemble(4, 8, 5, 40)
    fb = eng.FrameBatch(ens, 2, 64)
    for kw in (dict(first_frame=2), dict(first_frame=6), dict(doping_points=[5]), dict(doping_points=[-1]),
               dict(doping_points={5: 0.5}), dict(doping_points={-1: 0.5}), dict(first_vn=40, doping_points=[5])):
        with pytest.raises(eng.ScldpcError):
            fb.generate_erasures(0.4, 1, **kw)
    for eps in (-0.1, 1.0 + 1e-9, 2.0, math.nan, [0.4, math.nan], [0.4, -1.0]):
        with pytest.raises(eng.ScldpcError):
            fb.generate_erasures(eps, 1)
    with pytest.raises(eng.ScldpcError):
        fb.generate_erasures(math.nan, 1, first_vn=40)


@gpu
def test_benchmark_channel():
    """(4,8) L=50 M=10000, 4 graphs x 100 frames at eps 0.46-0.49, as bench.py draws them"""
    ens = eng.Ensemble(4, 8, 50, 10000)
    fb = eng.FrameBatch(ens, 4, 100)
    eps = [0.46, 0.47, 0.48, 0.49]
    got = drawn_channel(fb, eps, 0x5C1D9C + 1, first_graph_id=(5 << 20) + 8)
    assert_same(got, channels(4, (5 << 20) + 8, eps, ens.n, 100, 2, 0x5C1D9C + 1), "benchmark channel")


# ---- no repeated realisations (independent of the restatement) ---------------------------------------------------------
@gpu
def test_no_repeated_erasure_patterns():
    """at eps 0.5 a frame's pattern over n = 256 VNs is a function of (graph id, frame id, first VN): drawn again from
    another frame block it is the same pattern, and no two different triples share one -- across graph ids on both
    sides of 2^32, overlapping frame blocks (first_frame 0, 4, 64, 2^31) and chain pieces (first_vn 0, M, 17M).  A
    counter layout in which two of these share a counter repeats patterns, whatever the restatement says."""
    ens = eng.Ensemble(4, 8, 4, 64)
    fb = eng.FrameBatch(ens, 3, 64)
    pats = {}
    for gid in (0, U32 - 1):
        for ff in (0, 4, 64, 1 << 31):
            for A in (0, 1, 17):
                er = drawn_channel(fb, 0.5, 99, first_graph_id=gid, first_frame=ff, first_vn=A * 64)
                lanes = np.unpackbits(er.view(np.uint8).reshape(3, ens.n, -1), axis=2, bitorder="little")
                for g in range(3):
                    for f in range(64):
                        key, p = (gid + g, ff + f, A * 64), np.packbits(lanes[g, :, f]).tobytes()
                        assert pats.setdefault(key, p) == p, f"frame {key} drawn twice with different patterns"
    assert len(pats) == 2 * 3 * 3 * (128 + 64)                             # frames 0-127 and 2^31 + 0-63
    assert len(set(pats.values())) == len(pats), f"{len(pats) - len(set(pats.values()))} repeated erasure patterns"


@gpu
def test_no_repeated_socket_permutations():
    """every (graph id, absolute CN position) has its own socket -> CN map: drawn again in another piece it is the same
    map, and no two different (graph id, position) pairs share one"""
    dv, dc, M = 4, 8, 64
    cns = M * dv // dc
    maps = {}
    for gid, G in ((0, 3), (U32 - 1, 2)):
        for A, L in ((0, 24), (1, 12), (17, 9)):
            vn = drawn_graphs(eng.Ensemble(dv, dc, L, M), G, 55, gid, first_position=A).reshape(G, L, M, dv)
            for g in range(G):
                for cp in range(dv - 1, L):            # positions every edge type reaches
                    m = np.stack([vn[g, cp - i, :, i] - cp * cns for i in range(dv)], axis=1).reshape(-1)   # socket dv*t+i
                    assert m.min() >= 0 and m.max() < cns and (np.bincount(m, minlength=cns) == dc).all()
                    key = (gid + g, A + cp)
                    if key in maps:
                        assert (maps[key] == m).all(), key
                    maps[key] = m
    assert len(maps) > 100
    assert len({m.tobytes() for m in maps.values()}) == len(maps), "two (graph, position) pairs share a socket permutation"
