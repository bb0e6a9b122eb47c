"""grlbwt_b200 -- B200 (sm_100a) parse phase of grlBWT behind a C ABI, plus the host induction phase.

Python here is plumbing only (ctypes over include/grlgpu.h and include/grlbwt.h, used by the tests
and bench.py); the product is lib/libgrlgpu.so, lib/libgrlbwt.so and the lib/grlbwt CLI.
"""
from .api import (GrlGpu, GrlGpuError, Round, Stats, build_bwt, build_bwt_file, build_bwt_packed, build_bwt_to, invert_rl_bwt, parse_rl_bwt, lib_gpu, lib_host,  # noqa: F401
                  selftest_compact, selftest_induce, selftest_scan, selftest_sort, FLAG_SMALL_TABLE,
                  FLAG_FORCE_SLOW_SCAN, FLAG_KEEP_DICT, FLAG_FORCE_UNCACHED, FLAG_SMALL_PILOT, FLAG_FORCE_DOUBLING, FLAG_FORCE_WALK,
                  FLAG_FORCE_JUMP, LIB_DIR, Slice)
