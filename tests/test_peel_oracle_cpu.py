"""CPU tests of the checkers behind tests/test_peel_full_size_gpu.py: the O(log n)-per-step peeling oracle
(orc_peel_trajectory_fast) against the scanning one that the reference's goldens pin, and the Philox draws that feed both
the kernel and the oracles against the published philox4x32_10 known answers."""
import os
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import oracle
from fl_scaling_sc_ldpc_b200 import peeling_decoding as pdx
from tests.util import M32, philox4x32_10

Z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "peel_golden.npz"))
PEEL_SEED = 777


def _pool_map(fn, jobs):
    # the oracle runs outside the GIL (ctypes): a thread per host core
    with ThreadPoolExecutor(max_workers=max(1, min(len(jobs), os.cpu_count() or 1))) as ex:
        return list(ex.map(fn, jobs))


@pytest.mark.parametrize("name", ["t0", "t1", "t2", "t3"])
def test_fast_oracle_matches_slow_oracle_on_reference_goldens(name):
    """the goldens hold the reference's r1; test_peel_golden.py pins the scanning oracle to them"""
    e, l, r, L, M, term = (Z[name + "_params"][i] for i in range(6))
    l, r, L, M = int(l), int(r), int(L), int(M)
    cns, num_positions, total_size, steps = pdx._peel_geometry(float(e), l, r, L, M, bool(term))
    for f in range(Z[name + "_tr"].shape[0]):
        er = np.unpackbits(Z[name + "_er"][f])[: L * M]
        args = (Z[name + "_tr"][f], er, total_size, cns * (L + l - 1), steps, Z[name + "_picks"][f])
        fast = oracle.peel_trajectory_fast(*args)
        slow = oracle.peel_trajectory(*args)
        assert (fast[0] == slow[0]).all() and fast[1] == slow[1], (name, f)
        assert (fast[0] == Z[name + "_r1"][f]).all()


@pytest.mark.parametrize("term", [False, True])
def test_fast_oracle_matches_slow_oracle_at_M_1000(term):
    """(4,8) L=50 M=1000 (BASELINE config 1), full num_pd_steps: frames that stall early, late and finish"""
    l, r, L, M = 4, 8, 50, 1000
    cns = M * l // r
    oracle.srandom(4242 + term)
    rng = np.random.default_rng(17 + term)
    jobs, perm = [], None
    for e in (0.40, 0.45, 0.48):
        g, perm = oracle.generate_code(L, M, cns, l, r, perm)
        _, _, total_size, steps = pdx._peel_geometry(e, l, r, L, M, term)
        for _ in range(2):
            er = (rng.random(L * M) < e).astype(np.uint8)
            picks = rng.integers(0, 1 << 32, steps, dtype=np.uint64).astype(np.uint32)
            jobs.append((g.vn_cn, er, total_size, g.nk, steps, picks))
    fast = _pool_map(lambda j: oracle.peel_trajectory_fast(*j), jobs)
    slow = _pool_map(lambda j: oracle.peel_trajectory(*j), jobs)
    ends = set()
    for j, a, b in zip(jobs, fast, slow):
        assert (a[0] == b[0]).all() and a[1] == b[1]
        ends.add("finished" if a[1] == j[1].sum() else ("stalled early" if a[1] < j[1].sum() // 2 else "stalled late"))
    assert len(ends) >= 2, ends


def test_fast_oracle_edge_cases():
    """num_steps of 0 and not a multiple of 4, no erasure at all, and a trajectory that runs out of degree-one CNs
    before num_steps (the rest of r1 repeats the last value)"""
    l, r, L, M = 4, 8, 8, 32
    oracle.srandom(5)
    g, _ = oracle.generate_code(L, M, M * l // r, l, r)
    rng = np.random.default_rng(5)
    total_size = (L + l - 1) * M * l // r
    for steps in (0, 1, 3, 5, 500):
        for er in (np.zeros(L * M, np.uint8), (rng.random(L * M) < 0.3).astype(np.uint8), np.ones(L * M, np.uint8)):
            picks = rng.integers(0, 1 << 32, steps, dtype=np.uint64).astype(np.uint32)
            a = oracle.peel_trajectory_fast(g.vn_cn, er, total_size, g.nk, steps, picks)
            b = oracle.peel_trajectory(g.vn_cn, er, total_size, g.nk, steps, picks)
            assert len(a[0]) == steps + 1 and (a[0] == b[0]).all() and a[1] == b[1]


def picks_restated(seed, frame_id, n):
    """draw s of a frame = philox4x32_10(counter = (s // 4, 0, frame_id.lo, frame_id.hi), key = (seed.lo ^ 'peel',
    seed.hi))[s % 4]"""
    key = ((seed & M32) ^ 0x7065656C, seed >> 32)
    out = []
    for b in range((n + 3) // 4):
        out += philox4x32_10((b, 0, frame_id & M32, frame_id >> 32), key)
    return np.array(out[:n], np.uint32)


def test_philox_restatement_reproduces_random123_known_answers():
    kat = [((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
           ((M32,) * 4, (M32, M32), (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
           ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
            (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1))]
    for ctr, key, want in kat:
        assert philox4x32_10(ctr, key) == list(want)
    # the vectorised form (uint64 arrays, as the generator restatements in test_generators_gpu.py use it) gives the same
    # words element by element, with the counters mixed with ints and broadcast
    c0 = np.array([kat[0][0][0], kat[1][0][0], kat[2][0][0]] * 2, np.int64)
    for j, (ctr, key, want) in enumerate(kat):
        out = philox4x32_10((c0,) + ctr[1:], key)
        assert all(o.dtype == np.uint64 and o.shape == (6,) for o in out)
        assert [int(o[j]) for o in out] == list(want) and [int(o[j + 3]) for o in out] == list(want)
        arr = philox4x32_10(tuple(np.full((2, 3), c, np.uint64) for c in ctr), key)
        assert all((o == w).all() for o, w in zip(arr, want))


def test_philox_picks_known_answer():
    """seed 0x7065656C cancels the key whitening: frame 0's first block is the all-zero known answer"""
    assert pdx.philox_picks(0x7065656C, 0, 4).tolist() == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]


@pytest.mark.parametrize("seed,frame_id", [
    (0, 0), (0x5C1D9C + 2, 0), (0x5C1D9C + 2, ((9 << 20) + 32) * 1024 + 1023),     # bench.py's peeling frame ids are >= 2^32
    ((1 << 32) + 5, 7), (0xDEADBEEFCAFEF00D, (1 << 63) + 12345), (3, (1 << 32) - 1), (3, 1 << 32)])
@pytest.mark.parametrize("n", [1, 3, 4, 5, 13, 64])
def test_philox_picks_match_restatement(seed, frame_id, n):
    assert (pdx.philox_picks(seed, frame_id, n) == picks_restated(seed, frame_id, n)).all()
    assert len(pdx.philox_picks(seed, frame_id, n)) == n
