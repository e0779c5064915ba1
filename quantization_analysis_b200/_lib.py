"""ctypes binding of the C ABI in include/qa_b200.h (libqa_b200.so, built in-tree by csrc/build.sh).

There is no CPU fallback: if the library is missing or CUDA is unavailable every compute entry
point raises.  ``ensure_built()`` only compiles (nvcc cross-compiles without a GPU).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libqa_b200.so"
CSRC = _PKG / "csrc"

QA_DT_BF16, QA_DT_F32 = 0, 1
METRIC_CODE = {"pcc": 0, "mae": 1, "atol": 2}
NFMT, NSTAT = 4, 22
STATS_FAST, STATS_STRICT, STATS_FAST_APPROX_ABS = 0, 1, 2

EXPORTS = [
    "qa_version", "qa_last_error", "qa_quant_recon", "qa_quant_recon_cols", "qa_tile_stats", "qa_tile_scores_f32", "qa_tile_scores_pair_f32",
    "qa_numpy_permutation", "qa_numpy_integers", "qa_greedy_work_bytes", "qa_greedy_assign",
    "qa_threshold_assign", "qa_random_samples", "qa_apply_assignment", "qa_assignment_sums", "qa_assignment_sums_batch",
    "qa_f32_to_bf16_checked", "qa_scalar_proxy", "qa_fp8_block_dequant", "qa_greedy_par_work_bytes", "qa_greedy_assign_par", "qa_numpy_permutation_par", "qa_greedy_cluster_cap", "qa_greedy_assign_passes", "qa_greedy_init_sums_range", "qa_greedy_init_deltas", "qa_tile_stats_rows", "qa_greedy_init_bytes", "qa_perm_resolve", "qa_perm_resolve_chain", "qa_perm_apply", "qa_perm_apply_work_bytes", "qa_pair_sums", "qa_pair_sums_work_bytes",
    "qa_pairwise_plan_words", "qa_pairwise_plan_build", "qa_tensor_scores_work_bytes", "qa_tensor_scores_f32",
    "qa_tile_stats_f32", "qa_tile_stats_fp8", "qa_tile_stats_items", "qa_tile_stats_batch", "qa_greedy_init_deltas_batch",
    "qa_greedy_sweep_work_bytes", "qa_greedy_assign_sweep", "qa_transpose_2d",
]


class QaError(RuntimeError):
    pass


class BatchDesc(C.Structure):
    """qa_batch_desc of include/qa_b200.h (one tensor of a descriptor-array launch)."""
    _fields_ = [("x", C.c_void_p), ("table", C.c_void_p), ("init", C.c_void_p), ("rows", C.c_int64), ("cols", C.c_int64),
                ("ld", C.c_int64), ("item_begin", C.c_int64), ("block_begin", C.c_int64)]


def _sources_newer() -> bool:
    if not LIB_PATH.exists():
        return True
    t = LIB_PATH.stat().st_mtime
    srcs = list(CSRC.glob("*.cu")) + list(CSRC.glob("*.cuh")) + [_PKG.parent / "include" / "qa_b200.h"]
    return any(s.stat().st_mtime > t for s in srcs if s.exists())


def ensure_built(force: bool = False) -> Path:
    """Compile the CUDA library for sm_100a if it is missing or stale (needs nvcc)."""
    if force or _sources_newer():
        subprocess.run(["sh", str(CSRC / "build.sh")], check=True)
    return LIB_PATH


_lib = None


def lib():
    """The loaded library; raises QaError when it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise QaError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `sh quantization_analysis_b200/csrc/build.sh`. There is no CPU fallback.")
    L = C.CDLL(os.fspath(LIB_PATH))
    vp, i32, i64, u32, f64 = C.c_void_p, C.c_int, C.c_int64, C.c_uint32, C.c_double
    L.qa_version.restype = i32
    L.qa_last_error.restype = C.c_char_p
    L.qa_quant_recon.argtypes = [vp, i32, i64, i64, i64, u32, C.POINTER(vp), vp]
    L.qa_quant_recon_cols.argtypes = L.qa_quant_recon.argtypes
    L.qa_tile_stats.argtypes = [vp, i32, i64, i64, i64, i64, u32, i32, vp, vp]
    L.qa_tile_scores_f32.argtypes = [vp, i32, i64, i64, i64, u32, vp, vp]
    L.qa_tile_scores_pair_f32.argtypes = [vp, vp, i64, vp, vp]
    L.qa_numpy_permutation.argtypes = [vp, i64, vp, vp, vp]
    L.qa_numpy_integers.argtypes = [vp, i32, i64, vp, vp]
    L.qa_greedy_work_bytes.argtypes = [i64]
    L.qa_greedy_work_bytes.restype = i64
    L.qa_greedy_assign.argtypes = [vp, i64, f64, i32, f64, C.POINTER(C.c_int32), i32, vp, vp, vp, vp, vp, vp]
    L.qa_greedy_par_work_bytes.argtypes = [i64]
    L.qa_greedy_par_work_bytes.restype = i64
    L.qa_greedy_assign_par.argtypes = [vp, i64, f64, i32, f64, C.POINTER(C.c_int32), i32, vp, vp, vp, vp, vp, vp]
    L.qa_numpy_permutation_par.argtypes = [vp, i64, vp, vp, vp]
    L.qa_greedy_cluster_cap.argtypes = [i32]
    L.qa_pair_sums.argtypes = [vp, vp, i64, vp, vp, vp]
    L.qa_pair_sums_work_bytes.argtypes = []
    L.qa_pair_sums_work_bytes.restype = i64
    L.qa_perm_resolve.argtypes = [vp, i64, vp, vp, vp]
    L.qa_perm_resolve_chain.argtypes = [vp, i64, i32, C.c_uint32, vp, vp, vp]
    L.qa_perm_apply_work_bytes.argtypes = [i64]
    L.qa_perm_apply_work_bytes.restype = i64
    L.qa_perm_apply.argtypes = [vp, i64, vp, vp, vp, vp]
    L.qa_greedy_assign_passes.argtypes = [vp, i64, f64, i32, f64, C.POINTER(C.c_int32), i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, vp]
    L.qa_greedy_sweep_work_bytes.argtypes = [i64, i32]
    L.qa_greedy_sweep_work_bytes.restype = i64
    L.qa_greedy_assign_sweep.argtypes = [vp, i64, f64, i32, vp, i32, C.POINTER(C.c_int32), i32, vp, vp, vp, vp, vp, vp, vp, vp, i32, vp]
    L.qa_greedy_init_bytes.argtypes = [i64]
    L.qa_greedy_init_bytes.restype = i64
    L.qa_greedy_init_deltas.argtypes = [vp, i64, i32, C.POINTER(C.c_int32), i32, vp, vp]
    L.qa_greedy_init_sums_range.argtypes = [vp, i64, i32, C.POINTER(C.c_int32), i32, vp, i64, i64, vp]
    L.qa_tile_stats_rows.argtypes = [vp, i32, i64, i64, i64, u32, i32, vp, i64, i64, vp]
    L.qa_tile_stats_f32.argtypes = [vp, i64, i64, i64, u32, i32, vp, i64, i64, vp]
    L.qa_tile_stats_fp8.argtypes = [vp, vp, i64, i64, i64, i64, i64, u32, i32, vp, i64, i64, vp, vp]
    L.qa_tile_stats_items.argtypes = [i64, i64]
    L.qa_tile_stats_items.restype = i64
    L.qa_tile_stats_batch.argtypes = [vp, i32, i64, u32, i32, vp]
    L.qa_greedy_init_deltas_batch.argtypes = [vp, i32, i64, C.POINTER(C.c_int32), i32, vp]
    L.qa_threshold_assign.argtypes = [vp, i64, C.POINTER(C.c_int32), i32, i32, vp, i32, vp, vp, vp]
    L.qa_random_samples.argtypes = [vp, i64, f64, C.POINTER(C.c_int32), i32, i32, vp, vp, i32, vp, vp, vp]
    L.qa_apply_assignment.argtypes = [vp, i32, i64, i64, i64, vp, vp, vp]
    L.qa_assignment_sums.argtypes = [vp, i64, vp, i32, vp, vp]
    L.qa_assignment_sums_batch.argtypes = [vp, i64, vp, i32, vp, vp]
    L.qa_f32_to_bf16_checked.argtypes = [vp, i64, vp, vp, vp]
    L.qa_scalar_proxy.argtypes = [vp, i32, i64, i32, vp, vp]
    L.qa_fp8_block_dequant.argtypes = [vp, vp, i64, i64, i64, i64, vp, vp, vp, vp]
    L.qa_pairwise_plan_words.argtypes = [i64]
    L.qa_pairwise_plan_words.restype = i64
    L.qa_pairwise_plan_build.argtypes = [i64, vp]
    L.qa_tensor_scores_work_bytes.argtypes = [i64, i32]
    L.qa_tensor_scores_work_bytes.restype = i64
    L.qa_tensor_scores_f32.argtypes = [vp, i32, vp, i32, i64, i32, i64, vp, vp, vp, vp, vp]
    L.qa_transpose_2d.argtypes = [vp, i32, i64, i64, i64, vp, vp]
    for name in EXPORTS:
        fn = getattr(L, name)
        if name not in ("qa_last_error", "qa_greedy_work_bytes", "qa_greedy_par_work_bytes", "qa_greedy_init_bytes", "qa_perm_apply_work_bytes", "qa_version",
                        "qa_pair_sums_work_bytes", "qa_pairwise_plan_words", "qa_tensor_scores_work_bytes", "qa_tile_stats_items",
                        "qa_greedy_sweep_work_bytes"):
            fn.restype = i32
    _lib = L
    return L


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib().qa_last_error().decode("utf-8", "replace")
        raise QaError(f"{what} failed (rc={rc}): {msg}")


def int32_array(values):
    arr = (C.c_int32 * len(values))(*[int(v) for v in values])
    return arr
