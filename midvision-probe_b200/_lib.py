"""ctypes binding of libmvmatch.so (C ABI declared in include/mvmatch.h).

Only raw pointers, sizes and a CUDA stream handle cross this boundary.  There is no fallback:
if the library is missing the import of any compute entry point raises.
"""
import ctypes
import os
from ctypes import c_char_p, c_float, c_int, c_size_t, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
# MVMATCH_LIB_PATH: load another build of the same ABI (same-box A/B of kernel variants)
LIB_PATH = os.environ.get("MVMATCH_LIB_PATH") or os.path.join(HERE, "lib", "libmvmatch.so")

P = c_void_p  # every device / host pointer

# name -> (restype, argtypes); mirrors include/mvmatch.h one to one
PROTOTYPES = {
    "mv_version": (c_int, []),
    "mv_last_error": (c_char_p, []),
    "mv_device_info": (c_int, [c_int, P, P, P, P]),
    "mv_h2d_staged": (c_int, [P, P, c_size_t, P]),
    "mv_h2d_staged_threads": (c_int, []),
    "mv_chw_to_hwc": (c_int, [P, P, c_int, c_int, c_int, P, P]),
    "mv_feat_to_hwc_f32": (c_int, [P, c_int, c_int, c_int, c_int, P, P]),
    "mv_compact_valid": (c_int, [P, c_int, c_int, P, P, P]),
    "mv_geom_backproject": (c_int, [P, c_int, c_int, P, P, P]),
    "mv_geom_project_coords": (c_int, [P, P, P, c_int, P, c_int, c_int, c_int, c_int, P, P, P]),
    "mv_geom_grid_coords": (c_int, [P, P, P, c_int, c_int, c_int, c_int, c_int, P, P, P, P]),
    "mv_geom_keypoint_coords": (c_int, [P, c_int, c_int, c_float, c_int, c_int, P, P]),
    "mv_k1_sample_normalize": (c_int, [c_int, P, c_int, c_int, c_int, P, P, c_int, c_int, P, P, P, P, P]),
    "mv_k1_sample_f16c": (c_int, [c_int, P, c_int, c_int, c_int, P, P, c_int, c_int, c_int, P, P, P, P, c_int, P, P, P, P, P]),
    "mv_rows_dot": (c_int, [P, c_int, c_int, P, P, P]),
    "mv_k1_sample_tf32c": (c_int, [c_int, P, c_int, c_int, c_int, P, P, c_int, c_int, c_int, P, P, P, P, c_int, P, P, P]),
    "mv_rows_center": (c_int, [P, c_int, c_int, P, c_int, P, P, P]),
    "mv_k1_grid_supported": (c_int, [c_int, c_int, c_int, c_int, c_int]),
    "mv_rank_of_valid": (c_int, [P, P, c_int, P, c_int, P]),
    "mv_k1_grid_f16c": (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, c_int, P, P, P, c_int, P, P]),
    "mv_lr_unit_rows": (c_int, [P, c_int, c_int, P, P, P]),
    "mv_lr_gram_exact": (c_int, [P, P, c_int, c_int, c_int, c_int, P, c_int, P, P, P]),
    "mv_lr_build_query": (c_int, [c_int, P, P, c_int, c_int, c_int, P, P, P, c_int, c_int, c_int, P, c_int, c_int, P, P]),
    "mv_lr_build_target": (c_int, [c_int, P, P, c_int, c_int, c_int, P, P, P, c_int, c_int, P, c_int, c_int, P, P]),
    "mv_k3_ratio_mutual_lr": (c_int, [c_int, P, P, P, P, P, c_int, c_int, c_int, c_int, c_int, P, c_int, P, P, c_int, P, P, P, P]),
    "mv_k2_workspace_bytes": (c_size_t, [c_int, c_int]),
    "mv_k2_sim_top2": (c_int, [P, P, c_int, c_int, c_int, P, P, c_int, c_int, P, P, P, P, c_size_t, P]),
    "mv_k2_sim_top2_ld": (c_int, [P, c_int, P, c_int, c_int, c_int, c_int, P, P, c_int, c_int, P, P, P, P, c_size_t, P]),
    "mv_k2_affinity": (c_int, [P, c_int, P, c_int, c_int, c_int, c_int, P, P, c_int, c_int, P, c_int, P, P, P, P, c_size_t, P]),
    "mv_affinity_threshold": (c_int, [P, c_int, c_int, c_int, c_float, c_float, P, P, P]),
    "mv_cosine_2afc": (c_int, [P, P, P, c_int, c_int, P, P, P, P]),
    "mv_k2_set_streamk": (c_int, [c_int]),
    "mv_spair_set_heatmap_terms": (c_int, [c_int]),
    "mv_k2_profile_begin": (c_int, [c_int]),
    "mv_k2_profile_read": (c_int, [P, c_int]),
    "mv_k2_profile_dims": (c_int, [P, c_int]),
    "mv_k2_unpack_col": (c_int, [P, c_int, P, P, P]),
    "mv_k2_topk_workspace_bytes": (c_size_t, [c_int, c_int, c_int]),
    "mv_k2_sim_topk_ld": (c_int, [P, c_int, P, c_int, c_int, c_int, c_int, P, P, c_int, c_int, c_int, P, P, P, c_size_t, P]),
    "mv_knn_rerank": (c_int, [P, c_int, P, c_int, c_int, P, c_int, P, c_int, c_int, c_int, P, P, P]),
    "mv_k3_ratio_mutual": (c_int, [P, P, c_int, P, c_int, P, P, c_int, P, P, P, P]),
    "mv_k3_ratio_mutual_split": (c_int, [P, P, P, P, c_int, P, c_int, P, P, c_int, P, P, P, P]),
    "mv_k3_ratio_mutual_f16c": (c_int, [P, P, P, P, c_int, c_int, P, P, c_int, P, P, c_int, P, P, P, P]),
    "mv_k3_topk_matches": (c_int, [P, P, P, c_int, c_int, P, P, P, P, P]),
    "mv_k3_score": (c_int, [P, P, P, c_int, P, P, P, P, P, P, c_int, P, c_int, P, P, P, P, P, P]),
    "mv_gather_rows": (c_int, [P, c_int, P, P, c_int, P, P]),
    "mv_pack_matches": (c_int, [P, P, P, P, c_int, P, P, P, P, P, P, P, P]),
    "mv_argmax_rows": (c_int, [P, c_int, c_int, c_int, P, P]),
    "mv_k3_spair_errors": (c_int, [P, c_int, c_int, P, P, c_int, c_float, c_float, c_float, P, P, P, P, P, P, c_int, P]),
    "mv_spair_match_batch": (c_int, [P, c_int, c_int, c_int, c_int, P, P, c_int, c_int, P, c_float, c_float, P, P, P, P, P, P,
                                     c_int, P]),
    "mv_spair_match_batch_typed": (c_int, [P, c_int, c_int, c_int, c_int, c_int, P, P, c_int, c_int, P, c_float, c_float, P, P,
                                           P, P, P, P, c_int, P]),
}

# enums of include/mvmatch.h
MV_SAMPLE_BILINEAR_ZEROS = 0
MV_SAMPLE_BICUBIC_CLAMP = 1
MV_SAMPLE_ROWS = 2
MV_DTYPE_BF16 = 0
MV_DTYPE_TF32 = 1
MV_DTYPE_F16 = 2
MV_ROLE_QUERY, MV_ROLE_TARGET = 0, 1
MV_FEAT_F32, MV_FEAT_BF16, MV_FEAT_F16 = 0, 1, 2
MV_LR_MAX_SOURCE_PIXELS = 1024
MV_SIM_MASKED = -3.0e38
MV_MAX_THRESHOLDS = 16
MV_METRIC_L2SQ, MV_METRIC_COSINE = 0, 1

_lib = None

# kernels launched per entry point (for bench.py's gpu_launches claim); memsets are not counted
KERNELS_PER_CALL = {
    "mv_chw_to_hwc": 1, "mv_feat_to_hwc_f32": 1, "mv_compact_valid": 1, "mv_geom_backproject": 1, "mv_geom_project_coords": 1,
    "mv_geom_grid_coords": 1, "mv_geom_keypoint_coords": 1, "mv_k1_sample_normalize": 1, "mv_k1_sample_f16c": 1, "mv_k1_sample_tf32c": 1, "mv_rows_center": 2, "mv_rows_dot": 1, "mv_rank_of_valid": 1, "mv_k1_grid_f16c": 1, "mv_lr_unit_rows": 1, "mv_lr_gram_exact": 2, "mv_lr_build_query": 1, "mv_lr_build_target": 1, "mv_k3_ratio_mutual_lr": 1, "mv_k2_sim_top2": 2, "mv_k2_sim_top2_ld": 2, "mv_k2_affinity": 2, "mv_k2_sim_topk_ld": 2, "mv_knn_rerank": 1, "mv_affinity_threshold": 1, "mv_cosine_2afc": 1,
    "mv_k2_unpack_col": 1, "mv_k3_ratio_mutual": 1, "mv_k3_ratio_mutual_split": 1, "mv_k3_ratio_mutual_f16c": 1, "mv_k3_topk_matches": 1, "mv_k3_score": 1, "mv_gather_rows": 1,
    "mv_pack_matches": 1, "mv_argmax_rows": 1, "mv_k3_spair_errors": 1, "mv_spair_match_batch": 1, "mv_spair_match_batch_typed": 1,
}
LAUNCHES = {"count": 0}


class MvMatchError(RuntimeError):
    pass


def load(build_if_missing=True):
    """dlopen libmvmatch.so (building it first when nvcc is available and the file is absent)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise MvMatchError(f"{LIB_PATH} not found; run `python {HERE}/build.py`")
        from .build import build_lib

        build_lib()
    _default_stage_threads()
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError here = header / library mismatch: fail loudly
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _default_stage_threads():
    """One process per GPU shares the host cores with its siblings: unless the user chose, give the staging ring of
    mv_h2d_staged (csrc/stage.cu reads MVMATCH_STAGE_THREADS once) this rank's share of the cores -- measured at N = 8 on a
    32-core box: 8 threads per rank (64 in total) uploaded pageable pairs at 2400 pairs/s, a third of 8 x the single-GPU rate."""
    if "MVMATCH_STAGE_THREADS" in os.environ:
        return
    try:
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", "1"))
    except ValueError:
        local_world = 1
    if local_world > 1:
        cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 8)
        os.environ["MVMATCH_STAGE_THREADS"] = str(max(2, min(8, cores // local_world)))


def f16c_pitch(C):
    """row pitch (elements) of f16c rows of C channels: C + 8 augmentation columns rounded up to a 128-byte multiple."""
    return (C + 8 + 63) // 64 * 64


def tf32c_pitch(C):
    """row pitch (elements) of tf32c operand rows: C + 8 augmentation columns rounded up to a 128-byte multiple."""
    return (C + 8 + 31) // 32 * 32


def call(name, *args):
    """Invoke an int-returning entry point; raise MvMatchError with mv_last_error() on failure."""
    lib = load()
    rc = getattr(lib, name)(*args)
    LAUNCHES["count"] += KERNELS_PER_CALL.get(name, 0)
    if rc != 0:
        msg = lib.mv_last_error()
        raise MvMatchError(f"{name} failed with code {rc}: {msg.decode() if msg else ''}")


def ptr(t):
    """data pointer of a torch tensor (None -> NULL)."""
    return None if t is None else c_void_p(t.data_ptr())


def host_floats(values):
    """Small host float array (K, Rt, thresholds) as a ctypes buffer; keep a reference while in use."""
    vals = [float(v) for v in values]
    return (c_float * len(vals))(*vals)
