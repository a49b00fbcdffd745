"""Body of the two-rank test of bp_lim_iter --caps (tests/test_stream_caps_gpu.py): writes the per-cap files into argv[1]."""
import sys

from fl_scaling_sc_ldpc_b200 import bp_cli, dist as D

out = sys.argv[1]
D.init_from_env()
bp_cli.run("bp_lim_iter", ["1", "0", "0", "40", "--caps", "4,12", "--L", "12", "--M", "32", "--outdir", out, "--seed", "5",
                           "--points", "2", "--eps-ini", "0.47", "--eps-delta", "0.03", "--frames-per-graph", "96",
                           "--graphs-per-batch", "2", "--min-frame-err", "25", "--max-frames", "600"])
D.shutdown()
