"""ctypes binding of include/b200_ops.h (libb200ops.so) + thin torch-tensor helpers.

Fails loudly when the CUDA library is missing: there is no CPU fallback on the product path.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("B200_OPS_LIB") or os.path.join(_HERE, "libb200ops.so")   # the override exists for A/B builds of one kernel

F32, F16, Q4_0, Q8_0, Q4_K, Q5_K, Q6_K = 0, 1, 2, 8, 12, 13, 14
WEIGHT_TYPES = (Q4_0, Q8_0, Q4_K, Q5_K, Q6_K)

if not os.path.exists(LIB_PATH):
    raise ImportError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      "(nvcc, sm_100a). llama-box_b200 has no CPU fallback.")
lib = C.CDLL(LIB_PATH)

vp, i64, i32, f32 = C.c_void_p, C.c_int64, C.c_int, C.c_float


class RopeParams(C.Structure):
    _fields_ = [("n_dims", C.c_int32), ("mode", C.c_int32), ("n_ctx_orig", C.c_int32), ("_pad", C.c_int32),
                ("freq_base", f32), ("freq_scale", f32), ("ext_factor", f32), ("attn_factor", f32),
                ("beta_fast", f32), ("beta_slow", f32)]


class MmvDesc(C.Structure):
    _fields_ = [("W", vp), ("dst", vp), ("bias", vp), ("m", i64), ("type", C.c_int32), ("_pad", C.c_int32)]


class MmvLaunch(C.Structure):
    _fields_ = [("mats", MmvDesc * 4), ("residual", vp * 4), ("dst_col_stride", i64 * 4), ("n_mats", C.c_int32), ("swiglu", C.c_int32),
                ("k", i64), ("ncols", i64), ("act_source", C.c_int32), ("eps", f32), ("act_q8K", vp), ("act_q80", vp),
                ("x", vp), ("x_col_stride", i64), ("norm_w", vp), ("y_out", vp), ("k_valid", i64)]


# name -> (restype, argtypes); must list every symbol include/b200_ops.h declares
SIGNATURES = {
    "b200_abi_version": (i32, []),
    "b200_device_count": (i32, []),
    "b200_device_sm_count": (i32, [i32]),
    "b200_last_error": (C.c_char_p, []),
    "b200_kernel_launches": (i64, []),
    "b200_mmv_trace_dump": (i32, [vp, i32]),
    "b200_fa_trace_dump": (i32, [vp, i32]),
    "b200_block_elems": (i64, [i32]),
    "b200_block_bytes": (i64, [i32]),
    "b200_row_bytes": (i64, [i32, i64]),
    "b200_repack_rows": (i32, [i32, vp, i64, i64, vp]),
    "b200_padded_k": (i64, [i32, i64]),
    "b200_repack_rows_padded": (i32, [i32, vp, vp, i64, i64, i32, vp]),
    "b200_quantize_act2": (i32, [i32, vp, i64, vp, i64, i64, i64, vp]),
    "b200_unpack_rows": (i32, [i32, vp, i64, i64, vp]),
    "b200_type_is_repacked": (i32, [i32]),
    "b200_act_kind_for": (i32, [i32]),
    "b200_act_col_bytes": (i64, [i32, i64]),
    "b200_act_d_offset": (i64, [i32, i64]),
    "b200_act_bsum_offset": (i64, [i32, i64]),
    "b200_quantize_act": (i32, [i32, vp, i64, vp, i64, i64, vp]),
    "b200_rms_norm_quantize": (i32, [vp, vp, vp, vp, i32, vp, i32, i64, i64, f32, vp]),
    "b200_mul_mat_vec_q": (i32, [i32, vp, vp, vp, i64, vp, vp, i64, i64, i64, vp]),
    "b200_mul_mat_vec_q_multi": (i32, [C.POINTER(MmvDesc), i32, vp, vp, i64, i64, vp]),
    "b200_mul_mat_vec_q_launch": (i32, [C.POINTER(MmvLaunch), vp]),
    "b200_rope_kv_store2": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, i64, i64, i64, i64, i64, C.POINTER(RopeParams), vp]),
    "b200_mul_mat_vec_q_swiglu": (i32, [i32, vp, i32, vp, vp, vp, vp, i64, i64, i64, vp]),
    "b200_mul_mat_q_workspace": (i64, [i32, i64, i64, i64]),
    "b200_mul_mat_q": (i32, [i32, vp, vp, i64, vp, i64, i64, i64, i64, vp, vp]),
    "b200_mul_mat_q2": (i32, [i32, vp, vp, i64, vp, i64, i64, i64, i64, i64, vp, vp]),
    "b200_rms_norm": (i32, [vp, vp, vp, i64, i64, i64, i64, f32, vp]),
    "b200_rope": (i32, [vp, vp, vp, vp, i64, i64, i64, i64, i64, i64, i64, C.POINTER(RopeParams), vp]),
    "b200_set_rows": (i32, [vp, i64, vp, vp, i32, i64, i64, i64, vp]),
    "b200_rope_kv_store": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, i64, i64, i64, i64, C.POINTER(RopeParams), vp]),
    "b200_flash_attn_workspace": (i64, [i64, i64, i64, i64]),
    "b200_flash_attn_ext": (i32, [vp, i64, i64, vp, i64, i64, vp, i64, i64, vp, i64, vp, i32, i64, i64, i64, i64, i64, i64, f32, f32, f32, vp, vp]),
    "b200_rope_kv_flash_attn": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, i64, i64, i64, vp, vp, i64, i64, i64, i64, C.POINTER(RopeParams),
                                      f32, f32, f32, vp, vp]),
    "b200_rope_kv_flash_attn2": (i32, [vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i32, i64, i64, i64, i64, vp, vp, i64, i64, i64, i64, C.POINTER(RopeParams),
                                       f32, f32, f32, vp, vp, i32, vp]),
    "b200_add": (i32, [vp, vp, vp, i64, i64, i64, vp]),
    "b200_mul": (i32, [vp, vp, vp, i64, i64, i64, vp]),
    "b200_swiglu": (i32, [vp, vp, vp, i64, vp]),
    "b200_get_rows_f32": (i32, [vp, i64, vp, vp, i64, i64, vp]),
    "b200_cpy_f32_f16": (i32, [vp, vp, i64, vp]),
    "b200_argmax_f32": (i32, [vp, vp, i64, i64, vp]),
    "b200_wide_type_supported": (i32, [i32]),
    "b200_wide_shape_supported": (i32, [i32, i64]),
    "b200_wide_row_bytes": (i64, [i32, i64]),
    "b200_mul_mat_vec_wide": (i32, [i32, vp, vp, i64, vp, i64, vp, vp, i64, i64, i64, vp]),
    "b200_mul_mat_id": (i32, [i32, vp, i64, vp, i64, i64, i64, vp, i64, vp, i64, i64, i64, i64, i64, i64, i64, vp]),
    "b200_mul_mat_id_q_workspace": (i64, [i32, i64, i64, i64, i64, i64]),
    "b200_mul_mat_id_q": (i32, [i32, vp, i64, vp, i64, i64, i64, vp, i64, vp, i64, i64, i64, i64, i64, i64, i64, vp, vp]),
    "b200_get_rows_q": (i32, [i32, vp, i64, i64, vp, vp, i64, i64, i64, vp]),
    "b200_binary_strided": (i32, [i32, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "b200_soft_max_rows": (i32, [vp, i64, vp, i64, i64, i64, f32, vp]),
    "b200_argsort_rows": (i32, [vp, i64, vp, i64, i64, i64, i32, vp]),
    "b200_sum_rows": (i32, [vp, i64, vp, i64, i64, vp]),
    "b200_get_rows_f32_batched": (i32, [vp, i64, i64, i64, vp, i64, vp, i64, i64, i64, i64, i64, vp]),
    "b200_mul_mat_f32": (i32, [vp, i64, vp, i64, vp, i64, i64, i64, i64, vp]),
    "b200_unary": (i32, [i32, vp, vp, i64, f32, f32, vp]),
    "b200_mul_mat_f16": (i32, [vp, i64, i64, i64, vp, i64, i64, vp, i64, i64, i64, i64, i64, i64, vp]),
    "b200_soft_max_mask": (i32, [vp, vp, vp, i32, i64, i64, i64, i64, f32, f32, vp]),
    "b200_scatter_rows1": (i32, [vp, vp, vp, i32, i64, i64, vp]),
    "b200_set_rows_q4_0": (i32, [vp, i64, vp, vp, i64, i64, i64, vp]),
    "b200_flash_attn_any": (i32, [i32, vp, i64, i64, vp, i64, i64, vp, i64, i64, vp, i64, vp, i64, i64, i64, i64, i64, f32, f32, f32, vp]),
    "b200_flash_attn_q4_0": (i32, [vp, i64, i64, vp, i64, i64, vp, i64, i64, vp, i64, vp, i64, i64, i64, i64, i64, f32, f32, f32, vp]),
}
for _n, (_r, _a) in SIGNATURES.items():
    _f = getattr(lib, _n)
    _f.restype, _f.argtypes = _r, _a


class B200Error(RuntimeError):
    pass


def check(status):
    if status != 0:
        raise B200Error(f"b200 status {status}: {lib.b200_last_error().decode()}")


def p(t):
    """device pointer of a torch tensor (or None)"""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def row_bytes(t, k):
    return lib.b200_row_bytes(t, k)


def act_col_bytes(kind, k):
    return lib.b200_act_col_bytes(kind, k)
