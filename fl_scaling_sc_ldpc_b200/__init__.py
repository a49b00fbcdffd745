"""fl_scaling_sc_ldpc_b200 -- B200-native Monte-Carlo decoding engine for SC-LDPC codes over the BEC.

Accelerates the ``simulators_sc_ldpc`` hot path of rsokolovskii/fl_scaling_sc_ldpc (full / iteration-limited BP,
sliding-window BP, peeling decoding with trajectories) behind the reference's Python call signatures and file
formats.  Hand-written sm_100a CUDA kernels in ``csrc/`` are reached through the C ABI of ``libscldpc.so``
(``include/scldpc.h``); PyTorch only owns device buffers.  There is no CPU fallback.
"""
from .engine import (UNLIMITED, BpResult, Ensemble, FrameBatch, StreamCapsResult, StreamResult,  # noqa: F401
                     StreamStoppingSetResult, decode_bp_full, decode_bp_stream, decode_bp_window, decode_host, unpack_lanes, words_for)
from ._lib import ScldpcError  # noqa: F401

__version__ = "0.1.0"
from . import engine  # noqa: F401,E402
