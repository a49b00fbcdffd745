"""ctypes binding of ``libscldpc.so`` (C ABI declared in ``include/scldpc.h``).

The library is built in-tree (``fl_scaling_sc_ldpc_b200/csrc/Makefile``).  There is no CPU fallback: if the shared
object is missing, or no CUDA device is visible, the compute entry points raise.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SCLDPC_LIB") or os.path.join(HERE, "libscldpc.so")   # SCLDPC_LIB: A/B builds when tuning
CSRC = os.path.join(HERE, "csrc")

# flags (include/scldpc.h)
F_TERMINATED = 1
F_TRAJECTORY = 2
F_SQUARE = 4
F_EXP_ALL = 8
F_CHAN_PACKED = 16
F_MESSAGES = 64
F_NO_WAVE = 128
F_NODE_TRAJ = 256

EXPORTS = [
    "scldpc_last_error", "scldpc_version", "scldpc_build_info", "scldpc_device_count", "scldpc_graph_build_tables", "scldpc_graph_build_tables_async", "scldpc_graph_generate",
    "scldpc_graph_generate_scratch_bytes", "scldpc_channel_generate", "scldpc_channel_pack_host",
    "scldpc_bp_workspace_bytes", "scldpc_bp_full", "scldpc_bp_window", "scldpc_bp_window_range", "scldpc_decode_host",
    "scldpc_graph_generate_at", "scldpc_channel_generate_at",
    "scldpc_bp_stream_workspace_bytes", "scldpc_bp_stream", "scldpc_bp_stream_caps_workspace_bytes", "scldpc_bp_stream_caps", "scldpc_bp_stream_stopping_sets_workspace_bytes", "scldpc_bp_stream_stopping_sets", "scldpc_stream_host", "scldpc_bp_position_counts", "scldpc_bp_stopping_sets", "scldpc_bp_trajectory_moments", "scldpc_pairwise_moments_accumulate", "scldpc_allreduce_counters",
    "scldpc_peel_workspace_bytes", "scldpc_peel_trajectories", "scldpc_peel_variance_accumulate", "scldpc_philox_picks",
    "scldpc_launch_count", "scldpc_profile_begin", "scldpc_profile_end", "scldpc_bp_sweep_stats",
]


class ScldpcError(RuntimeError):
    pass


class Dims(ctypes.Structure):
    _fields_ = [(k, ctypes.c_int32) for k in ("dv", "dc", "L", "vns_pos", "cns_pos", "n_graphs", "n_words", "n_frames")]


class Batch(ctypes.Structure):
    _fields_ = [("vn_cn_dev", ctypes.c_void_p), ("vn_slot_dev", ctypes.c_void_p), ("cn_edge_dev", ctypes.c_void_p),
                ("chan_dev", ctypes.c_void_p)]


class BpOut(ctypes.Structure):
    _fields_ = [("iters_dev", ctypes.c_void_p), ("residual_dev", ctypes.c_void_p), ("blocks_err_dev", ctypes.c_void_p),
                ("erasures_exp_dev", ctypes.c_void_p), ("blocks_err_exp_dev", ctypes.c_void_p),
                ("erasures_p1_dev", ctypes.c_void_p), ("erased_dev", ctypes.c_void_p), ("rows_dev", ctypes.c_void_p),
                ("max_rows", ctypes.c_int32)]


class StreamCfg(ctypes.Structure):
    _fields_ = [("frames_per_graph", ctypes.c_int32), ("harvest_every", ctypes.c_int32), ("flags", ctypes.c_uint32),
                ("n_doped", ctypes.c_int32), ("n_soft", ctypes.c_int32), ("eps_host", ctypes.c_void_p),
                ("doped_pos_host", ctypes.c_void_p), ("soft_pos_host", ctypes.c_void_p), ("soft_count_host", ctypes.c_void_p),
                ("seed", ctypes.c_uint64), ("first_graph_id", ctypes.c_uint64), ("max_it", ctypes.c_int32)]


class StreamOut(ctypes.Structure):
    _fields_ = [(k, ctypes.c_void_p) for k in ("iters_dev", "residual_dev", "blocks_err_dev", "erasures_exp_dev", "blocks_err_exp_dev")]


class StreamCapsOut(ctypes.Structure):
    _fields_ = [(k, ctypes.c_void_p) for k in ("iters_dev", "residual_dev", "blocks_err_dev", "erasures_exp_dev", "blocks_err_exp_dev")]


class StreamSsOut(ctypes.Structure):
    _fields_ = [("iters_dev", ctypes.c_void_p), ("records_dev", ctypes.c_void_p)]


MAX_CAPS = 16  # SCLDPC_MAX_CAPS

_lib = None


def source_hash() -> str:
    """hash of the sources on disk, as the Makefile computes it (``scldpc_build_info`` carries the one the .so was built from)"""
    return subprocess.run(["make", "-s", "-C", CSRC, "print-hash"], check=True, capture_output=True, text=True).stdout.strip()


def build(force: bool = False) -> str:
    """Compile libscldpc.so for sm_100a (nvcc cross-compiles without a GPU).  ``force``: ``make clean`` first, so every
    object is compiled from the sources on disk; a record of the build goes to ``build_record.json`` next to the library."""
    import json
    import time
    t0 = time.time()
    if force:
        subprocess.run(["make", "-s", "-C", CSRC, "clean"], check=True)
    subprocess.run(["make", "-s", "-C", CSRC, "-j8"], check=True)
    objs = sorted(f for f in os.listdir(CSRC) if f.endswith(".o"))
    rec = {"mode": "clean" if force else "incremental", "seconds": round(time.time() - t0, 1), "source_hash": source_hash(),
           "library": os.path.basename(LIB_PATH), "library_bytes": os.path.getsize(LIB_PATH),
           "objects": {o: {"bytes": os.path.getsize(os.path.join(CSRC, o)), "mtime": os.path.getmtime(os.path.join(CSRC, o))} for o in objs},
           "nvcc": subprocess.run(["nvcc", "--version"], capture_output=True, text=True).stdout.strip().splitlines()[-1],
           "when": time.strftime("%Y-%m-%dT%H:%M:%SZ", time.gmtime())}
    with open(os.path.join(HERE, "build_record.json"), "w") as f:
        json.dump(rec, f, indent=1)
    return LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise ScldpcError(f"{LIB_PATH} is missing -- run `python -c 'import __graft_entry__ as g; g.build()'` "
                              f"or `make -C {CSRC}`; there is no CPU fallback")
        L = ctypes.CDLL(LIB_PATH)
        L.scldpc_last_error.restype = ctypes.c_char_p
        L.scldpc_build_info.restype = ctypes.c_char_p
        L.scldpc_bp_workspace_bytes.restype = ctypes.c_size_t
        L.scldpc_bp_stream_workspace_bytes.restype = ctypes.c_size_t
        L.scldpc_bp_stream_caps_workspace_bytes.restype = ctypes.c_size_t
        L.scldpc_bp_stream_stopping_sets_workspace_bytes.restype = ctypes.c_size_t
        L.scldpc_graph_generate_scratch_bytes.restype = ctypes.c_size_t
        L.scldpc_launch_count.restype = ctypes.c_longlong
        L.scldpc_peel_workspace_bytes.restype = ctypes.c_size_t
        L.scldpc_philox_picks.restype = None
        _lib = L
    return _lib


def check(rc: int):
    if rc != 0:
        raise ScldpcError(f"libscldpc error {rc}: {lib().scldpc_last_error().decode()}")
