"""rowbowt_b200 — B200 (sm_100a) implementation of rowbowt's batched RLBWT query path.

The product is `librowbowt_gpu.so` (C ABI in include/rowbowt_gpu.h, CUDA kernels in
csrc/) plus the host `rb_align` binary (csrc/rb_align_main.cpp).  This package is the
thin ctypes front end used by tests and bench.py; it has no compute of its own and no
CPU fallback — if the library is missing or there is no GPU, calls raise.
"""
from .binding import (  # noqa: F401
    RBG_COUNT, RBG_LOCATE, RBG_MARKERS, RBG_NARROW_LOCS, RBG_NARROW_RANGES, RBG_READ_DEAD, RBG_READ_EXOTIC, RBG_LOAD_SA, RBG_LOAD_MA,
    BuildStats, BwtStats, GpuIndex, MaStats, RbgError, SEED_DTYPE, StagedReads, build_bwt, build_bwt_text, build_index, build_marker_array,
    check_suffix_array,
    build_marker_array_arrays, lib,
    lib_path, result_checksum,
)
