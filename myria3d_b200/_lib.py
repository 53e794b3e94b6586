"""ctypes binding of ``libb200randla.so`` (C ABI declared in ``include/b200randla.h``).

There is NO CPU fallback: if the shared object is missing or a call fails the error is raised.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_void_p
from pathlib import Path

import torch  # noqa: F401  (loads the CUDA runtime the library links against)

LIB_PATH = Path(__file__).resolve().parent / "libb200randla.so"

_P = c_void_p
_SIGNATURES = {
    "b200_abi_version": (c_int, []),
    "b200_last_error": (c_char_p, []),
    "b200_launch_count": (c_int64, []),
    "b200_check_device": (c_int, []),
    "b200_set_option": (c_int, [c_char_p, c_int64]),
    "b200_get_option": (c_int64, [c_char_p]),
    "b200_knn": (c_int, [_P, _P, c_int64, _P, _P, c_int64, c_int32, c_int64, c_int32, c_int32, _P, _P, _P]),
    "b200_knn_grid_workspace_bytes": (c_int64, [c_int64, c_int32, c_int64]),
    "b200_knn_grid": (c_int, [_P, _P, c_int64, _P, _P, c_int64, c_int32, c_int64, c_int64, c_int32, c_int32, _P, _P, _P,
                              c_int64, _P]),
    "b200_adam_flat": (c_int, [_P, _P, _P, _P, c_int64, c_float, _P, c_float, c_float, c_float, _P, _P]),
    "b200_decimation_draw": (c_int, [_P, _P, c_int32, c_int64, ctypes.c_uint64, _P, ctypes.c_uint32, _P, _P]),
    "b200_counter_add": (c_int, [_P, c_int64, _P]),
    "b200_segmented_sort_pairs": (c_int, [_P, _P, _P, _P, _P, c_int32, c_int32, _P]),
    "b200_receptive_fields_per_axis": (c_int32, [c_float, c_float, c_float]),
    "b200_receptive_fields_count": (c_int, [_P, c_int64, c_float, c_float, c_float, c_float, c_float, _P, _P]),
    "b200_receptive_fields_fill": (c_int, [_P, c_int64, c_float, c_float, c_float, c_float, c_float, _P, _P, _P, _P, _P, _P, _P]),
    "b200_grid_sampling_sort": (c_int, [_P, c_int32, c_float, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "b200_grid_sampling_pool": (c_int, [_P, _P, _P, c_int32, c_int32, _P, _P, c_int32, _P, c_int32, _P, _P, _P, _P, _P]),
    "b200_random_permutation": (c_int, [c_int64, ctypes.c_uint64, _P, ctypes.c_uint32, _P, _P, _P, _P, _P, _P]),
    "b200_center_pos": (c_int, [_P, c_int32, _P]),
    "b200_batch_prep_stats_len": (c_int64, [c_int32]),
    "b200_batch_prep_compact": (c_int, [c_int32, _P, _P, c_int32, _P, _P, _P, c_int32, c_int64, _P, c_float, _P, _P, _P, _P, _P,
                                        _P, _P, _P]),
    "b200_batch_prep_voxelize": (c_int, [_P, _P, _P, _P, _P, c_int32, _P, _P, _P]),
    "b200_batch_prep_pool": (c_int, [_P, _P, _P, c_int32, c_int64, _P, _P, _P, c_int32, _P, c_int32, _P, _P, _P, _P]),
    "b200_batch_prep_budget_draw": (c_int, [_P, _P, c_int32, c_int64, ctypes.c_uint64, _P, _P, _P, _P, _P, _P]),
    "b200_batch_prep_finalize": (c_int, [c_int32, _P, _P, c_int32, _P, _P, c_int32, _P, _P, _P, c_int32, c_int32, c_float, c_float,
                                         c_float, ctypes.c_uint64, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "b200_tc_gemm_selftest": (c_int, [_P, _P, _P, c_int32, c_int32, c_int32, c_int32, _P, _P]),
    "b200_edge_moments": (c_int, [_P, _P, c_int64, c_int32, _P, _P]),
    "b200_lfa_fwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int64, c_int32, c_int32, _P]),
    "b200_lfa_bwd_workspace_bytes": (c_int64, [c_int64, c_int32, c_int32]),
    "b200_lfa_bwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, c_int32, c_int32, _P]),
    "b200_gather_rows": (c_int, [_P, _P, _P, c_int64, c_int32, _P]),
    "b200_scatter_rows_add": (c_int, [_P, _P, _P, c_int64, c_int32, _P]),
    "b200_stitch_segment_sum": (c_int, [_P, _P, _P, _P, c_int64, c_int32, c_int64, _P]),
    "b200_stitch_finalize": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, c_int32, _P]),
    "b200_knn_interp_fwd": (c_int, [_P, _P, _P, _P, c_int64, c_int32, c_int32, c_int32, c_int64, _P]),
    "b200_knn_interp_bwd": (c_int, [_P, c_int64, _P, _P, _P, c_int64, c_int32, c_int32, c_int32, _P]),
    "b200_linear_fwd": (c_int, [_P, c_int64, c_int32, _P, c_int64, c_int32, _P, _P, _P, c_int64, c_int32, _P, _P]),
    "b200_linear_bwd_input_workspace_bytes": (c_int64, [c_int64, c_int32, c_int32, c_int32]),
    "b200_linear_bwd_input": (c_int, [_P, _P, _P, c_int64, c_int32, _P, c_int64, c_int32, _P, c_int64, c_int64, c_int32, _P]),
    "b200_linear_bwd_weight_workspace_bytes": (c_int64, [c_int64, c_int32, c_int32, c_int32, c_int32]),
    "b200_linear_bwd_weight": (c_int, [_P, _P, c_int64, c_int32, _P, c_int64, c_int32, _P, _P, _P, c_int64, c_int64, c_int32, _P]),
    "b200_linear_fwd_num_stat_partials": (c_int64, [c_int64, c_int32, c_int32, c_int32]),
    "b200_bn_finalize": (c_int, [_P, c_int32, c_int64, _P, _P, _P, _P, _P, c_float, c_float, _P, _P, _P, _P, c_int32, _P]),
    "b200_encoder_fold_fwd": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_float, c_float, _P, _P, c_int32, _P]),
    "b200_encoder_fold_bwd": (c_int, [_P, _P, _P, _P, _P, _P, c_float, _P, _P, _P, _P, _P, _P, c_int32, c_int32, _P]),
    "b200_cross_entropy_fwd": (c_int, [_P, _P, _P, c_int64, c_int32, c_int64, _P, _P, _P, _P]),
    "b200_cross_entropy_bwd": (c_int, [_P, _P, _P, c_int64, c_int32, c_int64, _P, _P, _P, _P]),
    "b200_affine_act_fwd": (c_int, [_P, _P, _P, _P, _P, _P, c_float, _P, c_int64, c_int32, _P]),
    "b200_affine_act_bwd_reduce": (c_int, [_P, _P, c_float, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int32, _P]),
    "b200_affine_act_bwd": (c_int, [_P, _P, c_float, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64,
                                    c_int32, _P]),
    "b200_affine_act_bwd_apply": (
        c_int,
        [_P, _P, c_float, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int32, _P],
    ),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)
ABI_VERSION = 6

_lib = None

# Set to a KernelProfiler to time every library call with CUDA events (bench.py's roofline pass).
PROFILER = None


class KernelProfiler:
    """Collects (entry point, integer arguments, start event, end event) per library call."""

    def __init__(self):
        self.records = []

    def add(self, name, args, start, end):
        ints = tuple(a for a in args if isinstance(a, int))
        self.records.append((name, ints, start, end))

    def summary(self):
        """Synchronise and return ``[(name, ints, milliseconds), ...]``."""
        import torch

        torch.cuda.synchronize()
        return [(n, ints, s.elapsed_time(e)) for n, ints, s, e in self.records]



class B200Error(RuntimeError):
    """A libb200randla entry point returned a non-zero status."""


def load() -> ctypes.CDLL:
    """Load (once) and type the shared library.  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise B200Error(
            f"{LIB_PATH} is missing: build it with `python -m myria3d_b200.build` "
            "(there is no CPU or PyTorch fallback for the B200 hot path)"
        )
    lib = ctypes.CDLL(os.fspath(LIB_PATH))
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.b200_abi_version() != ABI_VERSION:
        raise B200Error(f"ABI mismatch: library {lib.b200_abi_version()} != binding {ABI_VERSION}")
    # A/B switches for scripts (bench.py, scripts/microbench.py): B200_OPTIONS="tma_rows=0,knn_points_per_cell=8" is applied
    # HERE, by the Python binding, through the public b200_set_option -- the library itself reads no environment.
    for item in filter(None, os.environ.get("B200_OPTIONS", "").split(",")):
        key, _, value = item.partition("=")
        if lib.b200_set_option(key.strip().encode(), int(value)) != 0:
            raise B200Error(f"B200_OPTIONS: {lib.b200_last_error().decode('utf-8', 'replace')}")
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().b200_last_error().decode("utf-8", "replace")
        if rc == 1:
            raise ValueError(f"{what}: {msg}")
        raise B200Error(f"{what}: {msg} (code {rc})")


def launch_count() -> int:
    return int(load().b200_launch_count())
