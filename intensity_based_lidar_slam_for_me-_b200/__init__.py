"""B200-native LOAM scan-to-map registration hot path (libilsm_cuda.so behind the C ABI of include/ilsm.h).

This package holds only what the path needs: csrc/ (hand-written sm_100a kernels + the C ABI), binding.py (ctypes
marshalling + host-side mirror of the reference call sites) and synth.py (seeded synthetic inputs).
"""
from . import _build, config, synth  # noqa: F401
from .sharding import allgather_topk, shard_range  # noqa: F401
from .binding import (Pc2Layout, pc2_layout_ouster, CubeMap, Slam, SlamStats, GroundExtractor, MapOptimization, CONVERGENCE, FAILURE, NO_CONVERGENCE, Context, IlsmError, IcpOpts, IcpResult, LocalMap, LoopClosure, LoopOpts, LoopResult, SlamLoopOpts, SlamLoopEvent, RegOpts, RegReport,  # noqa: F401
                      SolveSummary, ScanContextDb, default_opts, merge_topk, launch_count, live_bytes, live_handles, load_library, FACTOR_DTYPE)

__all__ = ["Context", "LocalMap", "RegOpts", "RegReport", "SolveSummary", "default_opts", "load_library", "ScanContextDb", "LoopClosure", "merge_topk", "CubeMap", "Slam", "SlamLoopOpts", "SlamLoopEvent", "GroundExtractor", "MapOptimization", "IlsmError",
           "synth", "CONVERGENCE", "NO_CONVERGENCE", "FAILURE", "FACTOR_DTYPE"]
