"""ctypes binding of libmxq.so (C ABI: include/mxq.h).  There is no CPU or PyTorch fallback: if the
library is missing or cannot be loaded every op raises."""
from __future__ import annotations

import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmxq.so")

OK, ERR_INVALID, ERR_UNSUPPORTED_SHAPE, ERR_CUDA = 0, 1, 2, 3
HP_BF16, HP_F32 = 0, 1
FLAG_HW_EXACT = 1
FLAG_OPERAND_LAYOUT = 2
GEMM_B_STATIC, GEMM_WIDE_TILES, GEMM_NO_PDL, GEMM_NO_MXF4 = 1, 2, 4, 8
ABI_VERSION = 6
MAX_DIMS = 6

EXPORTS = ("mxq_quantize", "mxq_dequantize", "mxq_dequantize_strided", "mxq_gemm", "mxq_gemm_dequant", "mxq_gemm_bf16", "mxq_transcode_to_e4m3", "mxq_pack_operand", "mxq_unpack_operand",
           "mxq_softmax_quantize", "mxq_flash_attention", "mxq_silu_mul_quantize", "mxq_rmsnorm", "mxq_rope", "mxq_quantize_heads", "mxq_quantize_transposed", "mxq_rope_quantize_kv",
           "mxq_moe_route", "mxq_moe_gemm", "mxq_moe_combine", "mxq_last_error", "mxq_version", "mxq_arch")


class GemmArgs(ctypes.Structure):
    _fields_ = [
        ("a_codes", ctypes.c_void_p), ("sfa", ctypes.c_void_p), ("lda", ctypes.c_int64), ("ld_sfa", ctypes.c_int64),
        ("a_batch_stride", ctypes.c_int64), ("sfa_batch_stride", ctypes.c_int64),
        ("b_codes", ctypes.c_void_p), ("sfb", ctypes.c_void_p), ("ldb", ctypes.c_int64), ("ld_sfb", ctypes.c_int64),
        ("b_batch_stride", ctypes.c_int64), ("sfb_batch_stride", ctypes.c_int64),
        ("bias", ctypes.c_void_p),
        ("d", ctypes.c_void_p), ("ldd", ctypes.c_int64), ("d_batch_stride", ctypes.c_int64),
        ("batch", ctypes.c_int64), ("M", ctypes.c_int64), ("N", ctypes.c_int64), ("K", ctypes.c_int64),
        ("a_format", ctypes.c_int), ("b_format", ctypes.c_int),
        ("d_multicast", ctypes.c_void_p),
        ("x_bf16", ctypes.c_void_p), ("ldx", ctypes.c_int64), ("x_quant_flags", ctypes.c_int),
        ("flags", ctypes.c_uint), ("split_k", ctypes.c_int),
    ]


class Operand(ctypes.Structure):
    _fields_ = [
        ("codes", ctypes.c_void_p), ("scales", ctypes.c_void_p),
        ("row_stride", ctypes.c_int64), ("k_stride", ctypes.c_int64), ("batch_stride", ctypes.c_int64),
        ("srow_stride", ctypes.c_int64), ("sk_stride", ctypes.c_int64), ("sbatch_stride", ctypes.c_int64),
        ("elem", ctypes.c_int), ("block_size", ctypes.c_int), ("blocked_along_k", ctypes.c_int),
    ]


class GemmDequantArgs(ctypes.Structure):
    _fields_ = [
        ("a", Operand), ("b", Operand),
        ("bias", ctypes.c_void_p),
        ("d", ctypes.c_void_p), ("ldd", ctypes.c_int64), ("d_batch_stride", ctypes.c_int64),
        ("batch", ctypes.c_int64), ("M", ctypes.c_int64), ("N", ctypes.c_int64), ("K", ctypes.c_int64),
    ]


class SoftmaxArgs(ctypes.Structure):
    _fields_ = [
        ("scores", ctypes.c_void_p),
        ("batch", ctypes.c_int64), ("heads", ctypes.c_int64), ("q_len", ctypes.c_int64), ("kv_len", ctypes.c_int64),
        ("scaling", ctypes.c_float),
        ("mask", ctypes.c_void_p), ("mask_stride_b", ctypes.c_int64), ("mask_stride_h", ctypes.c_int64), ("mask_stride_q", ctypes.c_int64),
        ("causal", ctypes.c_int),
        ("elem", ctypes.c_int), ("flags", ctypes.c_uint),
        ("codes", ctypes.c_void_p), ("scales", ctypes.c_void_p),
    ]


class AttentionArgs(ctypes.Structure):
    _fields_ = [
        ("q_codes", ctypes.c_void_p), ("q_scales", ctypes.c_void_p), ("q_format", ctypes.c_int),
        ("k_codes", ctypes.c_void_p), ("k_scales", ctypes.c_void_p), ("k_format", ctypes.c_int),
        ("vt_codes", ctypes.c_void_p), ("vt_scales", ctypes.c_void_p), ("v_format", ctypes.c_int),
        ("batch", ctypes.c_int64), ("heads", ctypes.c_int64), ("kv_heads", ctypes.c_int64), ("q_len", ctypes.c_int64), ("kv_len", ctypes.c_int64),
        ("head_dim", ctypes.c_int),
        ("scaling", ctypes.c_float),
        ("mask", ctypes.c_void_p), ("mask_stride_b", ctypes.c_int64), ("mask_stride_h", ctypes.c_int64), ("mask_stride_q", ctypes.c_int64),
        ("causal", ctypes.c_int),
        ("p_elem", ctypes.c_int), ("flags", ctypes.c_uint),
        ("out", ctypes.c_void_p), ("out_batch_stride", ctypes.c_int64), ("out_head_stride", ctypes.c_int64), ("out_row_stride", ctypes.c_int64),
        ("p_codes", ctypes.c_void_p), ("p_scales", ctypes.c_void_p),
        ("kv_pitch", ctypes.c_int64),
    ]


class RmsNormArgs(ctypes.Structure):
    _fields_ = [
        ("x", ctypes.c_void_p), ("ldx", ctypes.c_int64),
        ("residual", ctypes.c_void_p), ("ld_res", ctypes.c_int64),
        ("residual_out", ctypes.c_void_p), ("ld_res_out", ctypes.c_int64),
        ("weight", ctypes.c_void_p), ("eps", ctypes.c_float),
        ("rows", ctypes.c_int64), ("hidden", ctypes.c_int64),
        ("y", ctypes.c_void_p), ("ldy", ctypes.c_int64),
        ("codes", ctypes.c_void_p), ("scales", ctypes.c_void_p), ("elem", ctypes.c_int), ("flags", ctypes.c_uint),
    ]


class RopeArgs(ctypes.Structure):
    _fields_ = [
        ("q", ctypes.c_void_p), ("q_tok_stride", ctypes.c_int64), ("q_batch_stride", ctypes.c_int64), ("q_heads", ctypes.c_int),
        ("k", ctypes.c_void_p), ("k_tok_stride", ctypes.c_int64), ("k_batch_stride", ctypes.c_int64), ("k_heads", ctypes.c_int),
        ("cos", ctypes.c_void_p), ("sin", ctypes.c_void_p), ("cs_tok_stride", ctypes.c_int64), ("cs_batch_stride", ctypes.c_int64),
        ("batch", ctypes.c_int64), ("tokens", ctypes.c_int64), ("head_dim", ctypes.c_int),
        ("q_out", ctypes.c_void_p), ("k_out", ctypes.c_void_p),
        ("q_out_batch_stride", ctypes.c_int64), ("q_out_head_stride", ctypes.c_int64), ("q_out_tok_stride", ctypes.c_int64),
        ("k_out_batch_stride", ctypes.c_int64), ("k_out_head_stride", ctypes.c_int64), ("k_out_tok_stride", ctypes.c_int64),
        ("v", ctypes.c_void_p), ("v_tok_stride", ctypes.c_int64), ("v_batch_stride", ctypes.c_int64),
        ("v_out", ctypes.c_void_p), ("v_out_batch_stride", ctypes.c_int64), ("v_out_head_stride", ctypes.c_int64), ("v_out_tok_stride", ctypes.c_int64),
    ]


class TransposedQuantArgs(ctypes.Structure):
    _fields_ = [
        ("x", ctypes.c_void_p), ("n0", ctypes.c_int64), ("n1", ctypes.c_int64), ("rows", ctypes.c_int64), ("cols", ctypes.c_int64),
        ("s0", ctypes.c_int64), ("s1", ctypes.c_int64), ("row_stride", ctypes.c_int64),
        ("elem", ctypes.c_int), ("flags", ctypes.c_uint),
        ("codes", ctypes.c_void_p), ("scales", ctypes.c_void_p),
    ]


class RopeQuantizeKVArgs(ctypes.Structure):
    _fields_ = [
        ("q", ctypes.c_void_p), ("q_tok_stride", ctypes.c_int64), ("q_batch_stride", ctypes.c_int64), ("q_heads", ctypes.c_int),
        ("k", ctypes.c_void_p), ("k_tok_stride", ctypes.c_int64), ("k_batch_stride", ctypes.c_int64),
        ("v", ctypes.c_void_p), ("v_tok_stride", ctypes.c_int64), ("v_batch_stride", ctypes.c_int64), ("kv_heads", ctypes.c_int),
        ("cos", ctypes.c_void_p), ("sin", ctypes.c_void_p), ("cs_tok_stride", ctypes.c_int64), ("cs_batch_stride", ctypes.c_int64),
        ("batch", ctypes.c_int64), ("tokens", ctypes.c_int64), ("head_dim", ctypes.c_int),
        ("q_elem", ctypes.c_int), ("k_elem", ctypes.c_int), ("v_elem", ctypes.c_int), ("flags", ctypes.c_uint),
        ("q_codes", ctypes.c_void_p), ("q_scales", ctypes.c_void_p),
        ("k_codes", ctypes.c_void_p), ("k_scales", ctypes.c_void_p),
        ("vt_codes", ctypes.c_void_p), ("vt_scales", ctypes.c_void_p),
        ("v_open", ctypes.c_void_p),
        ("capacity", ctypes.c_int64), ("position", ctypes.c_void_p),
    ]


class MoeRouteArgs(ctypes.Structure):
    _fields_ = [
        ("top_k_index", ctypes.c_void_p), ("tokens", ctypes.c_int64), ("top_k", ctypes.c_int), ("num_experts", ctypes.c_int),
        ("offsets", ctypes.c_void_p), ("row_of_slot", ctypes.c_void_p), ("token_of_row", ctypes.c_void_p),
        ("x", ctypes.c_void_p), ("ldx", ctypes.c_int64), ("hidden", ctypes.c_int64),
        ("elem", ctypes.c_int), ("flags", ctypes.c_uint),
        ("codes", ctypes.c_void_p), ("scales", ctypes.c_void_p),
    ]


class MoeGemmArgs(ctypes.Structure):
    _fields_ = [
        ("w_codes", ctypes.c_void_p), ("w_scales", ctypes.c_void_p), ("w_format", ctypes.c_int),
        ("x_codes", ctypes.c_void_p), ("x_scales", ctypes.c_void_p), ("x_format", ctypes.c_int),
        ("offsets", ctypes.c_void_p),
        ("d", ctypes.c_void_p),
        ("rows", ctypes.c_int64), ("num_experts", ctypes.c_int64), ("N", ctypes.c_int64), ("K", ctypes.c_int64),
    ]


class MoeCombineArgs(ctypes.Structure):
    _fields_ = [
        ("y", ctypes.c_void_p), ("top_k_index", ctypes.c_void_p), ("top_k_weights", ctypes.c_void_p), ("weights_dtype", ctypes.c_int),
        ("row_of_slot", ctypes.c_void_p),
        ("tokens", ctypes.c_int64), ("top_k", ctypes.c_int), ("num_experts", ctypes.c_int), ("hidden", ctypes.c_int64),
        ("out", ctypes.c_void_p),
    ]


_lib = None
_lock = threading.Lock()


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"torchmx_b200: {LIB_PATH} is missing. Build it with `python -m torchmx_b200.build` "
                "(needs nvcc; sm_100a). There is no CPU / PyTorch fallback for the MX kernels.")
        L = ctypes.CDLL(LIB_PATH)
        i64, i32, vp, u32 = ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_uint
        L.mxq_last_error.restype = ctypes.c_char_p
        L.mxq_last_error.argtypes = []
        L.mxq_version.restype = i32
        L.mxq_arch.restype = i32
        L.mxq_quantize.restype = i32
        L.mxq_quantize.argtypes = [vp, i32, i64, i32, i32, u32, vp, vp, i32, vp]
        L.mxq_dequantize.restype = i32
        L.mxq_dequantize.argtypes = [vp, vp, i64, i32, i32, i32, vp, i32, vp]
        L.mxq_dequantize_strided.restype = i32
        L.mxq_dequantize_strided.argtypes = [vp, vp, i32, ctypes.POINTER(i64), ctypes.POINTER(i64), ctypes.POINTER(i64),
                                             i32, i32, i32, i32, vp, i32, vp]
        L.mxq_gemm.restype = i32
        L.mxq_gemm.argtypes = [ctypes.POINTER(GemmArgs), i32, vp]
        L.mxq_gemm_dequant.restype = i32
        L.mxq_gemm_dequant.argtypes = [ctypes.POINTER(GemmDequantArgs), i32, vp]
        L.mxq_gemm_bf16.restype = i32
        L.mxq_gemm_bf16.argtypes = [vp, i64, i64, vp, i64, i64, vp, vp, i64, i64, i64, i64, i64, i64, i32, vp]
        L.mxq_transcode_to_e4m3.restype = i32
        L.mxq_transcode_to_e4m3.argtypes = [vp, i32, i64, vp, i32, vp]
        L.mxq_pack_operand.restype = i32
        L.mxq_pack_operand.argtypes = [vp, i32, i64, vp, i32, vp]
        L.mxq_unpack_operand.restype = i32
        L.mxq_unpack_operand.argtypes = [vp, i32, i64, vp, i32, vp]
        L.mxq_silu_mul_quantize.restype = i32
        L.mxq_silu_mul_quantize.argtypes = [vp, vp, i64, i64, i64, i64, i32, u32, vp, vp, i32, vp]
        L.mxq_softmax_quantize.restype = i32
        L.mxq_softmax_quantize.argtypes = [ctypes.POINTER(SoftmaxArgs), i32, vp]
        L.mxq_flash_attention.restype = i32
        L.mxq_flash_attention.argtypes = [ctypes.POINTER(AttentionArgs), i32, vp]
        L.mxq_rmsnorm.restype = i32
        L.mxq_rmsnorm.argtypes = [ctypes.POINTER(RmsNormArgs), i32, vp]
        L.mxq_quantize_heads.restype = i32
        L.mxq_quantize_heads.argtypes = [vp, i64, i64, i64, i64, i32, u32, vp, vp, i32, vp]
        L.mxq_rope.restype = i32
        L.mxq_rope.argtypes = [ctypes.POINTER(RopeArgs), i32, vp]
        L.mxq_quantize_transposed.restype = i32
        L.mxq_quantize_transposed.argtypes = [ctypes.POINTER(TransposedQuantArgs), i32, vp]
        L.mxq_rope_quantize_kv.restype = i32
        L.mxq_rope_quantize_kv.argtypes = [ctypes.POINTER(RopeQuantizeKVArgs), i32, vp]
        for name, args in (("mxq_moe_route", MoeRouteArgs), ("mxq_moe_gemm", MoeGemmArgs), ("mxq_moe_combine", MoeCombineArgs)):
            getattr(L, name).restype = i32
            getattr(L, name).argtypes = [ctypes.POINTER(args), i32, vp]
        if L.mxq_version() != ABI_VERSION:
            raise RuntimeError(f"torchmx_b200: libmxq.so has ABI v{L.mxq_version()}, this package needs v{ABI_VERSION}: rebuild with `python -m torchmx_b200.build --force`")
        if L.mxq_arch() != 1000:
            raise RuntimeError(f"torchmx_b200: libmxq.so was built for arch {L.mxq_arch()}, expected sm_100a")
        _lib = L
    return _lib


def check(rc: int, what: str) -> None:
    if rc != OK:
        raise RuntimeError(f"{what} failed (status {rc}): {lib().mxq_last_error().decode()}")


def launch(name: str, *args) -> bool:
    """`lib().<name>(*args)` for an entry the caller may decline: False when it refuses the shape (the caller then takes another
    path), True when it ran.  Any other failure raises through `check`."""
    rc = getattr(lib(), name)(*args)
    if rc == ERR_UNSUPPORTED_SHAPE:
        return False
    check(rc, name)
    return True


def i64_array(values):
    return (ctypes.c_int64 * len(values))(*[int(v) for v in values])
