"""ctypes binding of libdcae_b200.so (include/dcae_b200.h).  There is no CPU fallback: if the
library is missing or the device is not sm_100, every call raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdcae_b200.so")

OK = 0
MATH = {"fp32": 0, "tf32x3": 1, "tf32": 2, "f16x3": 3, "f16": 4}
GC_EVAL, GC_NOISE, GC_DECODE = 0, 1, 2
GC_LIK = {"fast": 0, "reference": 1}
OPT_LIK_MATH, OPT_WANT_SYMBOLS = 0, 1
ACT_NONE, ACT_GELU, ACT_HALF_TANH, ACT_RELU = 0, 1, 2, 3

c_f32p = C.c_void_p   # device pointers travel as integers
c_i32p = C.c_void_p


class Planes(C.Structure):
    _fields_ = [("hi", C.c_void_p), ("lo", C.c_void_p), ("ld", C.c_int64)]


class GcArgs(C.Structure):
    _fields_ = [
        ("y", c_f32p), ("y_ld", C.c_int64),
        ("mu", c_f32p), ("mu_ld", C.c_int64),
        ("scale", c_f32p), ("scale_ld", C.c_int64),
        ("noise", c_f32p), ("noise_ld", C.c_int64),
        ("sym_in", c_i32p), ("sym_in_ld", C.c_int64),
        ("scale_table", c_f32p), ("n_table", C.c_int32),
        ("scale_bound", C.c_float), ("lik_bound", C.c_float),
        ("mode", C.c_int32),
        ("rows", C.c_int64), ("inner", C.c_int64),
        ("y_hat", c_f32p), ("y_hat_ld", C.c_int64),
        ("y_hat16", Planes),
        ("lik", c_f32p), ("lik_ld", C.c_int64),
        ("sym", c_i32p), ("sym_ld", C.c_int64),
        ("idx", c_i32p), ("idx_ld", C.c_int64),
        ("log2_partials", c_f32p),
        ("lik_math", C.c_int32),
    ]


class GcBwdArgs(C.Structure):
    _fields_ = [
        ("y", c_f32p), ("y_ld", C.c_int64), ("mu", c_f32p), ("mu_ld", C.c_int64), ("scale", c_f32p), ("scale_ld", C.c_int64),
        ("noise", c_f32p), ("noise_ld", C.c_int64), ("grad_lik", c_f32p), ("grad_lik_ld", C.c_int64),
        ("scale_bound", C.c_float), ("lik_bound", C.c_float), ("mode", C.c_int32), ("rows", C.c_int64), ("inner", C.c_int64),
        ("grad_y", c_f32p), ("grad_y_ld", C.c_int64), ("grad_mu", c_f32p), ("grad_mu_ld", C.c_int64),
        ("grad_scale", c_f32p), ("grad_scale_ld", C.c_int64),
    ]


class EbArgs(C.Structure):
    _fields_ = [("z", c_f32p), ("noise", c_f32p), ("sym_in", c_i32p), ("params", c_f32p), ("medians", c_f32p),
                ("mode", C.c_int32), ("B", C.c_int32), ("C", C.c_int32), ("HW", C.c_int64), ("lik_bound", C.c_float),
                ("z_hat", c_f32p), ("lik", c_f32p), ("sym", c_i32p)]


class EbBwdArgs(C.Structure):
    _fields_ = [("z", c_f32p), ("noise", c_f32p), ("params", c_f32p), ("medians", c_f32p), ("grad_lik", c_f32p),
                ("mode", C.c_int32), ("B", C.c_int32), ("C", C.c_int32), ("HW", C.c_int64), ("lik_bound", C.c_float),
                ("grad_z", c_f32p), ("grad_params", c_f32p)]


class MsssimArgs(C.Structure):
    _fields_ = [("x", c_f32p), ("y", c_f32p), ("B", C.c_int32), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("data_range", C.c_float), ("scratch", C.c_void_p), ("scratch_bytes", C.c_size_t),
                ("ssim", c_f32p), ("cs", c_f32p)]


class MsssimBwdArgs(C.Structure):
    _fields_ = [("x", c_f32p), ("y", c_f32p), ("B", C.c_int32), ("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("data_range", C.c_float), ("scratch", C.c_void_p), ("scratch_bytes", C.c_size_t),
                ("grad_ssim", c_f32p), ("grad_cs", c_f32p), ("grad_x", c_f32p)]


class CoderTables(C.Structure):
    _fields_ = [("cdfs", C.c_void_p), ("cdf_stride", C.c_int32), ("cdf_sizes", C.c_void_p), ("offsets", C.c_void_p),
                ("n_cdfs", C.c_int32)]


class IlvEncArgs(C.Structure):
    _fields_ = [("symbols", c_i32p), ("indexes", c_i32p), ("B", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("lanes", C.c_int32), ("tables", CoderTables), ("scratch", C.c_void_p), ("scratch_bytes", C.c_size_t),
                ("sizes", C.c_void_p), ("out", C.c_void_p), ("out_capacity", C.c_int64), ("status", c_i32p)]


class IlvDecArgs(C.Structure):
    _fields_ = [("strings", C.c_void_p), ("bounds", C.c_void_p), ("indexes", c_i32p), ("slice", C.c_int32),
                ("B", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("tables", CoderTables), ("symbols", c_i32p),
                ("status", c_i32p)]


ILV_STATUS = {1: "malformed header", 2: "corrupt stream", 3: "index outside the coder tables", 4: "unusable coder table row"}


class Operand(C.Structure):
    _fields_ = [("base", c_f32p), ("ld", C.c_int64), ("col0", C.c_int32), ("k0", C.c_int32),
                ("col1", C.c_int32), ("k1", C.c_int32), ("taps", C.c_int32),
                ("B", C.c_int32), ("h", C.c_int32), ("w", C.c_int32),
                ("planes", C.c_void_p), ("planes_bytes", C.c_int64), ("src16", Planes)]


class Epilogue(C.Structure):
    _fields_ = [("bias", c_f32p), ("addend", c_f32p), ("addend_ld", C.c_int64),
                ("residual", c_f32p), ("residual_ld", C.c_int64), ("res_scale", c_f32p),
                ("act", C.c_int32), ("act_cols", C.c_int32), ("out", c_f32p), ("out_ld", C.c_int64), ("out16", Planes),
                ("out16_act", Planes), ("act2", C.c_int32)]


class Weight(C.Structure):
    _fields_ = [("w", c_f32p), ("w_hi", c_f32p), ("w_lo", c_f32p), ("N", C.c_int32), ("K", C.c_int32),
                ("w16_hi", C.c_void_p), ("w16_lo", C.c_void_p), ("K16", C.c_int32), ("descale", C.c_float)]


class DictKV(C.Structure):
    _fields_ = [("Kh", c_f32p), ("Vh", c_f32p), ("Kh_hi", c_f32p), ("Kh_lo", c_f32p),
                ("Vt_hi", c_f32p), ("Vt_lo", c_f32p), ("head_scale", c_f32p),
                ("K16_hi", C.c_void_p), ("K16_lo", C.c_void_p), ("Vt16_hi", C.c_void_p), ("Vt16_lo", C.c_void_p),
                ("k_descale", C.c_float), ("v_descale", C.c_float)]


class SliceWeights(C.Structure):
    _fields_ = [
        ("x_trans", Weight), ("x_trans_b", c_f32p),
        ("ln_scale_g", c_f32p), ("ln_scale_b", c_f32p),
        ("msa_s", Weight), ("msa_s_b", c_f32p),
        ("dense_in", Weight * 3), ("dense_in_b", c_f32p * 3),
        ("dense_dw", c_f32p * 3), ("dense_dw_b", c_f32p * 3),
        ("dense_out", Weight * 3), ("dense_out_b", c_f32p * 3),
        ("dense_proj", Weight), ("dense_proj_b", c_f32p),
        ("spatial_w7", c_f32p),
        ("res_scale_1", c_f32p), ("res_scale_2", c_f32p), ("res_scale_3", c_f32p),
        ("lnx_g", c_f32p), ("lnx_b", c_f32p),
        ("q_trans", Weight), ("q_trans_b", c_f32p),
        ("kv", DictKV),
        ("linear", Weight), ("linear_b", c_f32p),
        ("ln_mlp_g", c_f32p), ("ln_mlp_b", c_f32p),
        ("fc1", Weight), ("fc1_b", c_f32p),
        ("mlp_dw", c_f32p), ("mlp_dw_b", c_f32p),
        ("fc2", Weight), ("fc2_b", c_f32p),
        ("output_trans", Weight), ("output_trans_b", c_f32p),
        ("cc1", Weight), ("cc1_b", c_f32p),
        ("mean2", Weight), ("mean2_b", c_f32p),
        ("scale2", Weight), ("scale2_b", c_f32p),
        ("mean3", Weight), ("mean3_b", c_f32p),
        ("scale3", Weight), ("scale3_b", c_f32p),
        ("lrp1y", Weight), ("lrp1_b", c_f32p),
        ("lrp2", Weight), ("lrp2_b", c_f32p),
        ("lrp3", Weight), ("lrp3_b", c_f32p),
    ]


# name -> (restype, argtypes); every symbol include/dcae_b200.h declares
_P, _I32, _I64, _F = C.c_void_p, C.c_int32, C.c_int64, C.c_float
SIGNATURES = {
    "dcae_version": (C.c_int, []),
    "dcae_last_error": (C.c_char_p, []),
    "dcae_device_check": (C.c_int, []),
    "dcae_launch_count": (_I64, []),
    "dcae_profile_start": (C.c_int, []),
    "dcae_profile_stop": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_I64)]),
    "dcae_profile_dump": (C.c_int, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(_I64)]),
    "dcae_gc_fused": (C.c_int, [C.POINTER(GcArgs), _P]),
    "dcae_gc_backward": (C.c_int, [C.POINTER(GcBwdArgs), _P]),
    "dcae_eb_fused": (C.c_int, [C.POINTER(EbArgs), _P]),
    "dcae_eb_backward": (C.c_int, [C.POINTER(EbBwdArgs), _P]),
    "dcae_msssim_scratch_bytes": (C.c_size_t, [_I32, _I32, _I32, _I32]),
    "dcae_msssim_forward": (C.c_int, [C.POINTER(MsssimArgs), _P]),
    "dcae_msssim_backward": (C.c_int, [C.POINTER(MsssimBwdArgs), _P]),
    "dcae_gc_num_partials": (_I64, [_I64, _I64]),
    "dcae_reduce_partials": (C.c_int, [_P, _I64, _P, _P]),
    "dcae_op_gemm": (C.c_int, [C.POINTER(Operand), C.POINTER(Weight), C.POINTER(Epilogue), C.c_int, _P]),
    "dcae_split_tf32": (C.c_int, [_P, _P, _P, _I64, _P]),
    "dcae_split_f16_weight": (C.c_int, [_P, _I32, _I32, _I32, _F, _P, _P, _P]),
    "dcae_planes_bytes": (_I64, [_I64, _I32]),
    "dcae_op_layernorm": (C.c_int, [_P, _I64, _P, _P, _I32, _I64, _P, _I64, C.POINTER(Planes), _P]),
    "dcae_op_gelu": (C.c_int, [_P, _I64, _I32, _I64, _P, _I64, C.POINTER(Planes), _P]),
    "dcae_op_dwconv3x3": (C.c_int, [_P, _I64, _P, _P, _I32, _I32, _I32, _I32, _I32, _P, _I64, _P, _I64, C.POINTER(Planes), _P]),
    "dcae_op_spatial_gate": (C.c_int, [_P, _I64, _P, _I64, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _I64, _P]),
    "dcae_op_spatial_gate_ln": (C.c_int, [_P, _I64, _P, _I64, _P, _P, _I32, _I32, _I32, _I32, _P, _P, _I64, _P, _P, C.POINTER(Planes), _P]),
    "dcae_op_dict_attention": (C.c_int, [_P, _I64, C.POINTER(Planes), C.POINTER(DictKV), _I64, _P, _I64, C.POINTER(Planes), C.c_int, _P]),
    "dcae_op_window_attention": (C.c_int, [_P, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _I32, _I32, _I32, _P, _I64, C.POINTER(Planes), _P]),
    "dcae_window_attention_backward_scratch_bytes": (C.c_size_t, [_I32, _I32, _I32, _I32, _I32, _I32]),
    "dcae_op_window_attention_backward": (C.c_int, [_P, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _I32, _P, _I32, _I32, _I32, _P, _I64, _P, _I64,
                                                    _P, _P, C.c_size_t, _P]),
    "dcae_op_space_to_depth":(C.c_int, [_P, _I64, _I32, _I32, _I32, _I32, _I32, _P, _I64, C.POINTER(Planes), _P]),
    "dcae_op_depth_to_space": (C.c_int, [_P, _I64, _I32, _I32, _I32, _I32, _I32, _I32, _P, _I64, C.POINTER(Planes), _P]),
    "dcae_op_nchw_to_tokens": (C.c_int, [_P, _I32, _I32, _I64, _P, _I64, C.POINTER(Planes), _P]),
    "dcae_op_tokens_to_nchw": (C.c_int, [_P, _I64, _I32, _I32, _I64, _P, _P]),
    "dcae_op_tokens_to_nchw_i32": (C.c_int, [_P, _I64, _I32, _I32, _I64, _P, _P]),
    "dcae_op_nchw_to_tokens_i32": (C.c_int, [_P, _I32, _I32, _I64, _P, _I64, _P]),
    "dcae_ilv_encode_scratch_bytes": (C.c_size_t, [_I32, _I32, _I32, _I32]),
    "dcae_ilv_encode_max_bytes": (_I64, [_I32, _I32, _I32, _I32]),
    "dcae_ilv_encode": (C.c_int, [C.POINTER(IlvEncArgs), _P]),
    "dcae_ilv_decode": (C.c_int, [C.POINTER(IlvDecArgs), _P]),
    "dcae_slice_loop_workspace_bytes": (C.c_size_t, [_I32, _I32, _I32]),
    "dcae_slice_loop_create": (C.c_int, [C.POINTER(_P), _I32, _I32, _I32, C.POINTER(SliceWeights), _P, _I32, _P, C.c_size_t, C.c_int]),
    "dcae_slice_loop_check_f16_range": (C.c_int, [_P, _I32, C.POINTER(C.c_ulonglong)]),
    "dcae_count_f16_clamped": (C.c_int, [C.POINTER(Planes), _I64, _I32, _P, _P]),
    "dcae_slice_loop_destroy": (None, [_P]),
    "dcae_slice_loop_set_option": (C.c_int, [_P, _I32, _I32]),
    "dcae_slice_loop_load": (C.c_int, [_P, _P, _P, _P, _P]),
    "dcae_slice_loop_params": (C.c_int, [_P, _I32, _P]),
    "dcae_slice_loop_encode": (C.c_int, [_P, _I32, _I32, _P, _P]),
    "dcae_slice_loop_indexes": (C.c_int, [_P, _I32, _P, _P]),
    "dcae_slice_loop_decode": (C.c_int, [_P, _I32, _P, _P]),
    "dcae_slice_loop_store": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dcae_slice_loop_module_dca": (C.c_int, [_P, C.c_int32, _P, _P, _P]),
    "dcae_slice_loop_module_conv": (C.c_int, [_P, C.c_int32, C.c_int32, _P, _P, _P]),
    "dcae_pack_symbols": (C.c_int, [_P, _P, _I64, _P, _P, _P, _P]),
    "dcae_slice_loop_forward": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "dcae_slice_loop_tap": (C.c_int, [_P, C.c_char_p, C.POINTER(_P), C.POINTER(_I32), C.POINTER(_I64)]),
    "dcae_slice_loop_tap16": (C.c_int, [_P, C.c_char_p, C.POINTER(Planes), C.POINTER(_I32)]),
}

_lib = None


class DcaeError(RuntimeError):
    pass


def load() -> C.CDLL:
    """Load the shared library (once) and bind every declared symbol; raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DcaeError(f"{LIB_PATH} not found: run `python __graft_entry__.py` (build()) first; "
                        "dcae_b200 has no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != OK:
        msg = load().dcae_last_error().decode("utf-8", "replace")
        raise DcaeError(f"{what or 'libdcae_b200'} failed ({rc}): {msg}")


def ptr(t) -> int | None:
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def current_stream(device) -> int:
    import torch
    return torch.cuda.current_stream(device).cuda_stream
