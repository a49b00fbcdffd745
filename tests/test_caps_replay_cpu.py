"""bp_lim_iter --caps without a GPU: the cap list and the per-cap replay of plr_computation / willIstop over the records of
one shared checkpointed stream."""
import numpy as np
import pytest

from fl_scaling_sc_ldpc_b200 import bp_cli


def synthetic_records(N, caps, seed):
    """[N][K][4] records with nested frame errors: the residual never grows with the cap"""
    rng = np.random.default_rng(seed)
    K = len(caps)
    res = np.zeros((N, K), np.int64)
    res[:, 0] = rng.integers(0, 40, N) * (rng.random(N) < 0.6)
    for k in range(1, K):
        res[:, k] = np.where(rng.random(N) < 0.5, 0, res[:, k - 1] - rng.integers(0, 5, N)).clip(0)
    blocks = np.where(res > 0, 1 + res // 7, 0)
    e_exp = np.where(rng.random((N, K)) < 0.3, 0, res)
    b_exp = np.where(e_exp > 0, blocks, 0)
    return np.stack([res, blocks, e_exp, b_exp], axis=-1)


def sequential(rec_k, max_frames, min_frame_err):
    """what a separate run at one cap accounts: frames in order until frame_err >= min_frame_err or max_frames"""
    c, f = bp_cli.new_counters(), 0
    for row in rec_k:
        if f >= max_frames:
            break
        bp_cli.account(c, *row)
        f += 1
        if c["frame_err"] >= min_frame_err:
            break
    return c, f


@pytest.mark.parametrize("min_frame_err,max_frames", [(30, 10 ** 6), (10 ** 6, 700), (45, 300), (1, 50)])
@pytest.mark.parametrize("chunks", [1, 3])
def test_every_cap_cuts_at_its_own_frame(min_frame_err, max_frames, chunks):
    caps = [175, 200, 250, 300, 350]
    rec = synthetic_records(1000, caps, 7)
    state = None
    for part in np.array_split(rec, chunks):              # rounds of one point: the state carries over
        state = bp_cli.replay_caps(part, max_frames, min_frame_err, state)
    cuts = []
    for k in range(len(caps)):
        c, f = sequential(rec[:, k], max_frames, min_frame_err)
        assert state[k]["counters"] == c and state[k]["frames"] == f, k
        assert state[k]["stopped"] == (c["frame_err"] >= min_frame_err)
        cuts.append(f)
    assert cuts == sorted(cuts)                           # nested errors: a larger cap never stops earlier
    if min_frame_err == 30:
        assert len(set(cuts)) > 1                         # the caps really stop at different frames


def test_parse_caps_adds_max_it_clamps_sorts_and_dedups():
    assert bp_cli.parse_caps(175, "350,200,250,300,200") == [175, 200, 250, 300, 350]
    assert bp_cli.parse_caps(0, "0,-3,7") == [1, 7]
    assert bp_cli.parse_caps(50, "") == [50]


def test_caps_cli_rejects_stream_off(tmp_path):
    with pytest.raises(SystemExit):
        bp_cli.run("bp_lim_iter", ["0", "0", "0", "10", "--caps", "20", "--stream", "off", "--outdir", str(tmp_path)])
    with pytest.raises(SystemExit):
        bp_cli.run("bp_lim_iter", ["0", "0", "0", "10", "--caps", ",".join(str(i) for i in range(20, 40)), "--outdir", str(tmp_path)])
