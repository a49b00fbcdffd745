"""Trailing options of main_simulate_sc_ldpc / ber_sim: --frames-per-graph and --graphs-per-batch after the 13 positional
arguments of PD.py:1328-1340 (CPU only: simulate_sc_ldpc is replaced by a recorder)."""
import numpy as np
import pytest

from fl_scaling_sc_ldpc_b200 import peeling_decoding as pdx

POSITIONAL = ["ber_sim", "OUT", "4", "8", "12", "48", "[0.47, 0.5]", "T", "U", "B", "NTB", "900", "40", "[]"]


@pytest.fixture
def calls(monkeypatch, tmp_path):
    seen = []

    def fake(e, l, r, L, M, is_terminated, is_protograph, is_bounded, is_tail_biting, num_repeats, max_fuckups, doping_points,
             **kw):
        seen.append(dict(e=e, L=L, M=M, num_repeats=num_repeats, max_fuckups=max_fuckups, **kw))
        return (0.5, 0.25, 0.1, 0.05, 1, 2, 3, 4, np.zeros(2), np.zeros(2), 5, 6, 0.7)
    monkeypatch.setattr(pdx, "simulate_sc_ldpc", fake)
    POSITIONAL[1] = str(tmp_path / "ber.txt")
    return seen


def test_positional_arguments_alone_keep_the_defaults(calls, tmp_path):
    pdx.main_simulate_sc_ldpc(list(POSITIONAL))
    assert [c["e"] for c in calls] == [0.47, 0.5]
    assert all(c["frames_per_graph"] == 128 and c["graphs_per_batch"] == 8 for c in calls)
    assert all(c["L"] == 12 and c["M"] == 48 and c["num_repeats"] == 900 and c["max_fuckups"] == 40 for c in calls)
    lines = open(tmp_path / "ber.txt").read().splitlines()
    assert len(lines) == 3 and lines[1].split()[0] == "0.47"


@pytest.mark.parametrize("extra,fpg,gpb", [
    (["--frames-per-graph", "16384"], 16384, 8),
    (["--graphs-per-batch", "2"], 128, 2),
    (["--graphs-per-batch", "3", "--frames-per-graph", "2048"], 2048, 3),
    (["--frames-per-graph=4096"], 4096, 8),
])
def test_trailing_options(calls, extra, fpg, gpb):
    pdx.main_simulate_sc_ldpc(list(POSITIONAL) + extra)
    assert len(calls) == 2 and all(c["frames_per_graph"] == fpg and c["graphs_per_batch"] == gpb for c in calls)


@pytest.mark.parametrize("extra", [["--frames-per-graph", "0"], ["--graphs-per-batch", "-1"], ["--frames-per-graph"],
                                   ["--unknown", "3"], ["17"]])
def test_bad_trailing_options_exit(calls, extra):
    with pytest.raises(SystemExit):
        pdx.main_simulate_sc_ldpc(list(POSITIONAL) + extra)
    assert calls == []


def test_parse_defaults():
    assert pdx.parse_sc_ldpc_options([]) == (128, 8)
