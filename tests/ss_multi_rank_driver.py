"""Body of the two-rank ber_sim test of tests/test_stream_stopping_sets_gpu.py: one run on frame streams, written to argv[1]."""
import os
import sys

from fl_scaling_sc_ldpc_b200 import dist as D, peeling_decoding as pdx

out = sys.argv[1]
D.init_from_env()
pdx.main_simulate_sc_ldpc(["ber_sim", os.path.join(out, "ber.txt"), "4", "8", "12", "48", "[0.47, 0.5]", "T", "U", "B", "NTB",
                           "9000", "1500", "[]", "--frames-per-graph", "2048", "--graphs-per-batch", "1"])
D.shutdown()
