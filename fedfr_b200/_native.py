"""ctypes binding of ``libfedfr_b200.so`` (the C ABI declared in ``include/fedfr_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` (nvcc, sm_100a).  There is no fallback: if the
shared object is missing, importing this module raises; if there is no sm_100 GPU, every compute entry
returns an error which ``check`` turns into ``RuntimeError``.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libfedfr_b200.so")

PATH_TENSOR = 0
PATH_CHECK = 1
FEDAVG_F32 = 0
FEDAVG_I64 = 1
FEDAVG_KEEP_FIRST_TERM = 0x100

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build the CUDA extension first "
        "(python -c 'import __graft_entry__ as g; g.build()' from the repo root). fedfr_b200 has no CPU/PyTorch fallback.")

lib = C.CDLL(LIB_PATH)

_vp, _i64, _i32, _f32, _sz = C.c_void_p, C.c_int64, C.c_int, C.c_float, C.c_size_t

# name -> (restype, argtypes); must list every symbol include/fedfr_b200.h declares (tests check this)
SIGNATURES = {
    "pfc_version": (_i32, []),
    "pfc_last_error": (C.c_char_p, []),
    "pfc_query_device": (_i32, [_i32, C.POINTER(_i32), C.POINTER(_i32), C.POINTER(_i32)]),
    "pfc_normalize_rows": (_i32, [_vp, _vp, _i64, _i32, _vp, _vp, _vp, _vp]),
    "pfc_sgd_step": (_i32, [_vp, _vp, _vp, _vp, _i64, _i32, _f32, _f32, _f32, _f32, _i32, _vp, _vp, _vp]),
    "pfc_cast_rows_bf16": (_i32, [_vp, _i64, _i32, _vp, _vp]),
    "pfc_gather_rows2": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "pfc_scatter_rows2": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _vp, _vp]),
    "pfc_remap_labels": (_i32, [_vp, _i64, _i64, _i64, _vp, _vp]),
    "pfc_sample_workspace_bytes": (_sz, [_i64]),
    "pfc_sample_index": (_i32, [_vp, _i64, _vp, _i64, _i64, _vp, _vp, _vp, _sz, _vp]),
    "pfc_fwd_num_partials": (_i32, [_i64, _i64, _i32, _i32]),
    "pfc_fwd_stats": (_i32, [_vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _i32, _vp, _vp, _vp, _i32, _vp]),
    "pfc_normalize_fwd_stats": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _vp]),
    "pfc_merge_stats": (_i32, [_vp, _vp, _vp, _i32, _i64, _vp, _vp]),
    "pfc_finalize_stats": (_i32, [_vp, _i32, _i64, _vp, _vp, _vp, _vp]),
    "pfc_bwd_workspace_bytes": (_sz, [_i64, _i64, _i32, _i32]),
    "pfc_bwd": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _i32, _f32, _vp, _vp, _i32, _vp, _sz, _i32, _vp]),
    "pfc_prob_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "pfc_normalize_fwd_prob": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pfc_set_range_flag": (_i32, [_vp, _f32]),
    "pfc_bwd_prob_workspace_bytes": (_sz, [_i64, _i64, _i32]),
    "pfc_bwd_prob": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _i32, _f32, _vp, _vp, _i32, _vp, _sz, _vp, _sz, _vp]),
    "pfc_spreadout_num_partials": (_i32, [_i64, _i32]),
    "pfc_spreadout_workspace_bytes": (_sz, [_i64, _i32]),
    "pfc_spreadout": (_i32, [_vp, _i64, _i32, _f32, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pfc_cosface_dense": (_i32, [_vp, _vp, _i64, _i64, _f32, _f32, _vp, _vp]),
    "pfc_arcface_dense": (_i32, [_vp, _vp, _i64, _i64, _f32, _f32, _vp]),
    "pfc_bce_head_fwd": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pfc_bce_head_bwd": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _vp, _vp, _vp, _vp]),
    "pfc_bce_loss_fwd": (_i32, [_vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "pfc_bce_loss_bwd": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i32, _f32, _f32, _f32, _f32, _f32, _vp, _vp, _vp, _vp]),
    "pfc_similar_columns": (_i32, [_vp, _i64, _vp, _i64, _i32, _f32, _vp, _vp]),
    "pfc_roc_histogram": (_i32, [_vp, _vp, _i64, _vp, _vp, _i64, _i64, _i32, _vp, _vp]),
    "pfc_template_pool": (_i32, [_vp, _vp, _vp, _vp, _vp, _i64, _i32, _vp, _vp]),
    "pfc_pair_scores": (_i32, [_vp, _i64, _i32, _vp, _vp, _i64, _vp, _vp]),
    "pfc_tar_at_far_workspace_bytes": (_sz, [_i64]),
    "pfc_tar_at_far": (_i32, [_vp, _vp, _i64, _vp, _i32, _vp, _vp, _vp, _sz, _vp]),
    "pfc_roc_curve_workspace_bytes": (_sz, [_i64]),
    "pfc_roc_curve": (_i32, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pfc_kfold_workspace_bytes": (_sz, [_i64, _i32, _i64]),
    "pfc_kfold_accuracy": (_i32, [_vp, _vp, _vp, _i64, _i32, _vp, _i32, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "pfc_identify_workspace_bytes": (_sz, [_i64]),
    "pfc_identify": (_i32, [_vp, _i64, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "fedavg_table_bytes": (_sz, [_i32, _i32]),
    "fedavg_weighted_sum": (_i32, [_vp, _vp, _vp, _vp, _i32, _vp, _i32, _vp, _sz, _vp]),
    "fedavg_blend": (_i32, [_vp, _vp, _f32, _f32, _i64, _vp, _vp]),
}
for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args
# developer hooks (profiling / launch accounting / tuning), not part of the reference-facing header
lib.pfc_launch_count.restype = C.c_longlong
lib.pfc_launch_count.argtypes = []
lib.pfc_profile_enable.restype = _i32
lib.pfc_profile_enable.argtypes = [_i32]
lib.pfc_profile_collect.restype = _i32
lib.pfc_profile_collect.argtypes = [C.POINTER(C.c_float), C.POINTER(_i32)]
lib.pfc_set_clusters.restype = _i32
lib.pfc_set_clusters.argtypes = [_i32, _i32]
lib.pfc_set_logits_tile.restype = _i32
lib.pfc_set_logits_tile.argtypes = [_i32]
lib.pfc_set_prefetch.restype = _i32
lib.pfc_set_prefetch.argtypes = [_i32, _i32, _i32]
lib.pfc_set_fwd_overlap.restype = _i32
lib.pfc_set_fwd_overlap.argtypes = [_i32, _i32]
lib.pfc_set_pipeline.restype = _i32
lib.pfc_set_pipeline.argtypes = [_i32, _i32, _i32, _i32, _i32]
lib.pfc_set_prob_split.restype = _i32
lib.pfc_set_prob_split.argtypes = [_i32, _f32, _i32]
for _knob in ("pfc_set_nvtx", "pfc_set_dw4", "pfc_set_dx_pair", "pfc_set_graph", "pfc_set_chunk_mb", "pfc_set_logits_pair", "pfc_set_roc_mode"):
    getattr(lib, _knob).restype = _i32
    getattr(lib, _knob).argtypes = [_i32]


MARGIN_COSFACE, MARGIN_ARCFACE = 0, 1


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = lib.pfc_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"fedfr_b200::{what} failed (code {rc}): {msg}")


def ptr(t):
    """Device/host pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()
