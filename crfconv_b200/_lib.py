"""ctypes loader for the C-ABI CUDA library (include/crfconv_b200.h).  There is no CPU fallback: if the library is
missing, or a call returns a non-zero status, a RuntimeError is raised."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcrfconv_b200.so")

_lib = None

_vp, _i64, _sz, _f32, _int = C.c_void_p, C.c_int64, C.c_size_t, C.c_float, C.c_int

# name -> (restype, argtypes); mirrors include/crfconv_b200.h one to one (checked by tests/test_cabi.py)
SIGNATURES = {
    "crfconv_abi_version": (_int, []),
    "crfconv_status_string": (C.c_char_p, [_int]),
    "crfconv_knn_workspace_bytes": (_sz, [_i64, _i64, _i64, _i64]),
    "crfconv_knn_batch": (_int, [_vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp, _sz, _vp]),
    "crfconv_cpp_knn_batch": (_int, [_vp, _sz, _sz, _sz, _vp, _sz, _sz, _vp]),
    "crfconv_knn_distance_pick_workspace_bytes": (_sz, [_i64, _i64]),
    "crfconv_knn_batch_distance_pick": (_int, [_vp, _i64, _i64, _i64, _i64, C.c_uint32, _vp, _vp, _vp, _sz, _vp]),
    "crfconv_cpp_knn_batch_distance_pick": (_int, [_vp, _sz, _sz, _sz, _vp, _sz, _sz, _vp, C.c_uint32]),
    "crfconv_radius_batch": (_int, [_vp, _i64, _i64, _vp, _i64, _f32, _i64, _vp, _vp, _sz, _vp]),
    "crfconv_fps": (_int, [_vp, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "crfconv_edge_softmax_fwd": (_int, [_vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "crfconv_edge_softmax_bwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "crfconv_edge_gauss_fwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _vp]),
    "crfconv_edge_gauss_bwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _int, _vp]),
    "crfconv_spmm_fwd": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "crfconv_spmm_bwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _int, _vp]),
    "crfconv_grid_subsample_workspace_bytes": (_sz, [_i64, _i64, _i64]),
    "crfconv_grid_subsample": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _f32, _int, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "crfconv_grid_subsample_host": (_int, [_vp, _i64, _vp, _i64, _vp, _i64, _f32, _int, _vp, _vp, _vp, _vp]),
    "crfconv_set_fast_path": (_int, [_int]),
    "crfconv_linear_fwd": (_int, [_vp, _int, _vp, _vp, _f32, _vp, _i64, _i64, _vp, _int, _vp, _vp, _vp, _vp, _i64, _int, _int, _vp]),
    "crfconv_bn_finalize_fwd": (_int, [_vp, _i64, _vp, _vp, _f32, _f32, _int, _vp, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "crfconv_bn_act_fwd": (_int, [_vp, _vp, _vp, _vp, _f32, _vp, _i64, _int, _vp]),
    "crfconv_bn_bwd_reduce": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _i64, _int, _vp]),
    "crfconv_bn_finalize_bwd": (_int, [_vp, _i64, _vp, _vp, _vp, _vp, _int, _vp]),
    "crfconv_linear_bwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32,
                                  _vp, _int, _vp, _vp, _f32, _vp, _i64, _i64, _vp, _int, _vp, _vp, _int, _vp, _int, _vp, _vp, _vp, _i64,
                                  _i64, _int, _int, _vp]),
    "crfconv_linear_bwd_launches": (_int, []),
    "crfconv_grad_slots_reduce": (_int, [_vp, _vp, _i64, _i64, _vp]),
    "crfconv_relpos": (_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _vp]),
    "crfconv_pointconv_aggregate_fwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _int, _vp]),
    "crfconv_pointconv_aggregate_bwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _int, _vp]),
    "crfconv_gather_max_fwd": (_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _int, _vp]),
    "crfconv_gather_max_bwd": (_int, [_vp, _vp, _vp, _i64, _int, _vp]),
    "crfconv_lrelu_bwd": (_int, [_vp, _vp, _f32, _vp, _i64, _vp]),
    "crfconv_add_inplace": (_int, [_vp, _vp, _i64, _vp]),
    "crfconv_scatter_add_rows": (_int, [_vp, _vp, _vp, _i64, _i64, _i64, _int, _vp]),
    "crfconv_fused_max_parts": (_int, []),
    "crfconv_fused_part_floats": (_int, []),
    "crfconv_fused_counter_ints": (_int, []),
    "crfconv_out_bwd_part_floats": (_int, []),
    "crfconv_lin16_fwd": (_int, [_vp, _int, _vp, _vp, _vp, _f32, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    "crfconv_up16_fwd": (_int, [_vp, _vp, _int, _vp, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp]),
    "crfconv_linear_fwd_bn": (_int, [_vp, _int, _vp, _vp, _f32, _vp, _int, _vp, _vp, _vp, _i64, _int, _int, _vp, _vp, _vp, _vp, _vp, _f32, _f32,
                                     _vp, _vp, _vp, _vp, _vp]),
    "crfconv_bn_bwd_reduce_fin": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _f32, _vp, _i64, _int, _vp, _vp, _vp, _vp, _vp, _vp]),
    "crfconv_mid16_bwd": (_int, [_vp] * 7 + [_vp] * 5 + [_f32, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "crfconv_in16_dgrad": (_int, [_vp] * 8 + [_int, _vp, _int, _i64, _vp]),
    "crfconv_in16_wgrad": (_int, [_vp] * 8 + [_int, _vp, _i64, _i64, _vp]),
    "crfconv_out16_bwd": (_int, [_vp] * 6 + [_f32, _vp, _vp, _vp, _i64] + [_vp] * 10),
    "crfconv_crf_step_bwd_fused": (_int, [_vp] * 12 + [_int, _vp, _vp, _vp, _vp, _i64, _vp, _i64, _i64, _int, _int, _int] + [_vp] * 7),
    "crfconv_crf_upsample_bwd_fused": (_int, [_vp] * 7 + [_i64, _i64, _i64] + [_vp] * 7),
    "crfconv_crf_compat_fwd": (_int, [_vp, _vp, _vp, _vp, _int, _vp]),
    "crfconv_crf_compat_bwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    "crfconv_crf_upsample_fwd": (_int, [_vp, _vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _vp]),
    "crfconv_pcf_supported": (_int, [_int]),
    "crfconv_pcf_fwd_scratch_floats": (_int, [_int]),
    "crfconv_pcf_bwd_scratch_floats": (_int, [_int]),
    "crfconv_pcf_relpos_moments": (_int, [_vp] * 5 + [_i64, _i64, _i64, _int, _vp]),
    "crfconv_pcf_stats1": (_int, [_vp, _vp, _vp, _int, _vp]),
    "crfconv_pcf_fwd": (_int, [_vp] * 7 + [_f32] + [_vp] * 4 + [_i64, _i64, _i64, _int, _int, _vp]),
    "crfconv_pcf_out": (_int, [_vp] * 5 + [_i64, _int, _vp]),
    "crfconv_pcf_bwd1": (_int, [_vp] * 8 + [_f32] + [_vp] * 7 + [_i64, _i64, _i64, _int, _int, _vp]),
    "crfconv_pcf_bwd2": (_int, [_vp] * 8 + [_f32] + [_vp] * 9 + [_i64, _i64, _i64, _int, _int, _vp]),
    "crfconv_pcf_param_grads": (_int, [_vp] * 18 + [_int, _vp]),
    "crfconv_cross_entropy_fwd": (_int, [_vp, _vp, _vp, _i64, _int, _i64, _vp, _vp]),
    "crfconv_cross_entropy_bwd": (_int, [_vp, _vp, _vp, _i64, _int, _i64, _vp, _vp, _int, _vp, _vp]),
    "crfconv_crf_upsample_bwd": (_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _int, _vp]),
    "crfconv_crf_step_fwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _i64, _int, _int, _vp]),
    "crfconv_pack_index_host": (_int, [_vp, _i64, _int, _vp, _int]),
    "crfconv_unpack_index": (_int, [_vp, _i64, _int, _vp, _vp]),
    "crfconv_crf_step_bwd": (_int, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _int, _i64, _i64, _int, _int, _vp]),
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -m crfconv_b200.build` (or __graft_entry__.build()). "
                "crfconv_b200 has no CPU / PyTorch fallback path.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError here = header / library mismatch: fail loudly
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(status: int, what: str = ""):
    if status != 0:
        msg = lib().crfconv_status_string(int(status)).decode()
        raise RuntimeError(f"crfconv_b200 {what} failed: {msg} (status {status})")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
