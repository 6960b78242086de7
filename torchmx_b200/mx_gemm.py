"""Host side of the tensor-core MX matmul (K3): decides whether an (A, B) pair of MXTensors can run
on the tcgen05 block-scaled kernel, prepares the E4M3-container operand views and calls mxq_gemm.
Returns None when the pair does not qualify; ops.py then takes the dequantize path the reference
itself uses (torchmx/ops.py:29-41).

Qualifying pair (what every layer of the reference produces, torchmx/layers/mx_linear.py:61-95,
mx_llama_attention.py:195-243): both operands FP element types, block size 32 along the contraction
dim, no padding, K a multiple of 128, codes K-contiguous in memory.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional

import torch

from . import _C, dtypes
from .mx_tensor import MXTensor, _codes_like, _quant_flags, _stream_ptr

aten = torch.ops.aten

# developer switch: MXQ_DISABLE_TC=1 forces the dequantize path (used by parity tests)
_DISABLED = os.environ.get("MXQ_DISABLE_TC", "0") == "1"
_SHADOW_ATTR = "_mxq_e4m3_shadow"

# tensor_core: launches of the block-scaled tcgen05 kernels (K3a/b/c); dequant_gemm: launches of the fused dequantize + bf16
# tcgen05 kernel (K3d) for operands the block-scaled instruction cannot take; fallback: contractions that reached neither and
# ran as K2 + aten (torch.compile tracing, non-bf16 advertised dtypes); dequant_once_gemm: the dequant_gemm launches that
# dequantized each operand once first; fused_act_quant / packed_act_quant: the tensor_core launches whose bf16 activation was
# quantized inside the GEMM / written by K1 as the packed operand stream
stats = {"tensor_core": 0, "dequant_gemm": 0, "dequant_once_gemm": 0, "fallback": 0, "transcode": 0, "fused_allreduce": 0,
         "fused_act_quant": 0, "packed_act_quant": 0}

class FusedOutput:
    """Target of a fused GEMM + all-reduce launch, handed EXPLICITLY from RowParallelMXLinear.forward down to the launch (no
    module-level state: layers are driven from arbitrary threads, torchmx/examples/quantized_llama_chat.py:123-129): `view` is
    the [rows, features] output view of a symmetric buffer, `multicast_ptr` the NVLink multicast address of that view.  A
    tensor-core launch that can honour it writes nothing locally -- its epilogue adds the partial into every rank's buffer
    (mxq_gemm_args_t.d_multicast) -- and sets `taken`; otherwise `taken` stays False and the layer all-reduces with NCCL."""
    __slots__ = ("view", "multicast_ptr", "taken")

    def __init__(self, view, multicast_ptr: int):
        self.view, self.multicast_ptr, self.taken = view, multicast_ptr, False


# Dispatch overrides for tests (every value maps to a documented field of mxq_gemm_args_t, include/mxq.h): keep the CTA-pair
# tiles on small grids, pin the decode kernel's K split count, keep fp4 x fp4 on kind::mxf8f6f4, launch without PDL.
overrides = {"wide_tiles": False, "split_k": 0, "no_mxf4": False, "no_pdl": False}


def _flags(static_b: bool) -> int:
    return ((_C.GEMM_B_STATIC if static_b else 0) | (_C.GEMM_WIDE_TILES if overrides["wide_tiles"] else 0)
            | (_C.GEMM_NO_MXF4 if overrides["no_mxf4"] else 0) | (_C.GEMM_NO_PDL if overrides["no_pdl"] else 0))


def mark_static(w) -> None:
    """Declare an MXTensor long-lived (a layer's pre-quantized weight): nothing enqueued from now on writes its codes / scales,
    so -- once the kernels that produced them have finished -- the decode kernel may prefetch them before its predecessor in
    the stream is done (MXQ_GEMM_B_STATIC).  A CUDA event recorded here tells `_static_b` when that is the case.  `w` is an
    MXTensor (the mark goes on the long-lived tensor its views come from) or any object that owns operand buffers (a module)."""
    dev = w._data.device if isinstance(w, MXTensor) else next(iter(w.buffers())).device
    w = getattr(w, "_mxq_origin", w)
    if dev.type == "cuda" and not torch.cuda.is_current_stream_capturing():
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(dev))
        w.__dict__["_mxq_static"] = ev


def _static_b(b_origin) -> bool:
    st = b_origin.__dict__.get("_mxq_static")
    if st is None:
        return False
    if st is True:
        return True
    if torch.cuda.is_current_stream_capturing() or not st.query():  # producers still in flight: this launch waits for them
        return False
    b_origin.__dict__["_mxq_static"] = True
    return True


def set_enabled(flag: bool) -> None:
    global _DISABLED
    _DISABLED = not flag


# operand storage formats of mxq_gemm (include/mxq.h: MXQ_OPERAND_*)
FMT_E4M3_BYTES, FMT_E2M1_PACKED, FMT_E3M2_PACKED, FMT_E2M3_PACKED, FMT_E5M2_BYTES = 0, 1, 2, 3, 4
_PACKED_FORMAT = {"float4_e2m1": FMT_E2M1_PACKED, "float6_e3m2": FMT_E3M2_PACKED, "float6_e2m3": FMT_E2M3_PACKED}
_PACKED_BITS = {FMT_E2M1_PACKED: 4, FMT_E3M2_PACKED: 6, FMT_E2M3_PACKED: 6}
# MXQ_PACKED_OPERANDS=0 keeps every fp6 / fp4 operand in the one-byte E4M3 container (the first implementation)
_USE_PACKED = os.environ.get("MXQ_PACKED_OPERANDS", "1") != "0"


def set_packed_operands(flag: bool) -> None:
    global _USE_PACKED
    _USE_PACKED = bool(flag)


def _operand_rows(codes: torch.Tensor, elem: dtypes.DType, cache_on: Optional[MXTensor], packed: Optional[bool] = None):
    """codes: [..., rows, Kb] reference-layout element codes with unit stride along Kb -> (uint8 operand tensor, format).

    float8_e4m3 passes through untouched (a view).  fp4 / fp6 codes become the packed 4 / 6-bit streams the sm_100a TMA
    unit expands and kind::mxf8f6f4 consumes natively (`mxq_pack_operand`: a nibble swap / a 6-bit pack, exact), so they
    cost 0.5 / 0.75 B of HBM traffic per element; with MXQ_PACKED_OPERANDS=0 they are re-encoded exactly as E4M3 bytes
    instead (`mxq_transcode_to_e4m3`).  When `cache_on` is given (the long-lived MXTensor the operand is a view of, i.e. a
    layer's weight) the result is cached on that Python object, keyed by the view geometry, the format and the version
    counter of the codes, so a weight is converted once, not once per forward."""
    if elem == dtypes.float8_e4m3:
        return codes, FMT_E4M3_BYTES
    if elem == dtypes.float8_e5m2:  # labelled extension element type: one byte per element, native MMA format
        return codes, FMT_E5M2_BYTES
    fmt = _PACKED_FORMAT[elem.name] if (_USE_PACKED if packed is None else packed) else FMT_E4M3_BYTES
    key = None
    if cache_on is not None:
        key = (codes.data_ptr(), tuple(codes.shape), tuple(codes.stride()), cache_on._data._version, fmt)
        hit = cache_on.__dict__.get(_SHADOW_ATTR)
        if hit is not None and hit[0] == key:
            return hit[1], fmt
    stats["transcode"] += 1
    src = codes.contiguous()
    per = 2 if elem == dtypes.float4_e2m1 else 1
    n_elements = src.numel() * per
    if fmt == FMT_E4M3_BYTES:
        out = torch.empty(tuple(src.shape[:-1]) + (src.shape[-1] * per,), dtype=torch.uint8, device=src.device)
        rc = _C.lib().mxq_transcode_to_e4m3(src.data_ptr(), dtypes.ELEM_ID[elem.name], n_elements, out.data_ptr(), src.device.index,
                                            _stream_ptr(src))
        _C.check(rc, "mxq_transcode_to_e4m3")
    else:
        k = src.shape[-1] * per
        out = torch.empty(tuple(src.shape[:-1]) + (k * _PACKED_BITS[fmt] // 8,), dtype=torch.uint8, device=src.device)
        rc = _C.lib().mxq_pack_operand(src.data_ptr(), dtypes.ELEM_ID[elem.name], n_elements, out.data_ptr(), src.device.index, _stream_ptr(src))
        _C.check(rc, "mxq_pack_operand")
    # A shadow created while a CUDA graph is being captured lives in that graph's private memory pool (and its conversion
    # kernel in the graph): it must not outlive the graph through this cache.  Warm a model up once before capturing it --
    # the shadows then exist as ordinary tensors and the graph contains no conversion kernels.
    if cache_on is not None and not torch.cuda.is_current_stream_capturing():
        cache_on.__dict__[_SHADOW_ATTR] = (key, out)
    return out, fmt


def _rows_k(t: MXTensor, k_dim_from_end: int):
    """(codes, scales) viewed as [..., rows, K-ish] with K innermost, or None if K is not unit-stride."""
    d, s = t._data, t._scale_e8m0
    if k_dim_from_end == 2:  # operand given as [..., K, rows]
        d, s = d.transpose(-1, -2), s.transpose(-1, -2)
    if d.stride(-1) != 1 or s.stride(-1) != 1:
        return None
    return d, s


def _qualifies(t: MXTensor) -> bool:
    # (plain inner tensors only: while torch.compile / AOT autograd trace through the subclass the inner tensors are fake or
    # functional wrappers without storage -- the override then takes the dequantize path, whose custom op has a fake kernel)
    return (isinstance(t, MXTensor) and type(t._data) is torch.Tensor and type(t._scale_e8m0) is torch.Tensor and (t._elem_dtype in dtypes.SUPPORTED_FP_ELEM_DTYPES or t._elem_dtype == dtypes.float8_e5m2) and t._block_size == 32 and t._padding == 0
            and t._data.is_cuda and t._orig_dtype == torch.bfloat16)


def _launch(a_codes, sfa, b_codes, sfb, bias, batch, M, N, K, a_bs, sfa_bs, b_bs, sfb_bs, out, a_fmt=FMT_E4M3_BYTES, b_fmt=FMT_E4M3_BYTES,
            d_multicast: int = 0, x_hp: Optional[torch.Tensor] = None, x_flags: int = 0, static_b: bool = False) -> bool:
    g = _C.GemmArgs()
    g.a_format, g.b_format = a_fmt, b_fmt
    g.flags, g.split_k = _flags(static_b), overrides["split_k"]
    g.d_multicast = d_multicast or None
    if x_hp is not None:  # fused activation quantization: the kernel reads the bf16 activation itself
        g.x_bf16, g.ldx, g.x_quant_flags = x_hp.data_ptr(), x_hp.stride(-2), x_flags
    else:
        g.a_codes, g.sfa, g.lda, g.ld_sfa = a_codes.data_ptr(), sfa.data_ptr(), a_codes.stride(-2), sfa.stride(-2)
    g.a_batch_stride, g.sfa_batch_stride = a_bs, sfa_bs
    g.b_codes, g.sfb, g.ldb, g.ld_sfb = b_codes.data_ptr(), sfb.data_ptr(), b_codes.stride(-2), sfb.stride(-2)
    g.b_batch_stride, g.sfb_batch_stride = b_bs, sfb_bs
    g.bias = bias.data_ptr() if bias is not None else None
    g.d, g.ldd, g.d_batch_stride = out.data_ptr(), N, M * N
    g.batch, g.M, g.N, g.K = batch, M, N, K
    return _C.launch("mxq_gemm", ctypes.byref(g), out.device.index, _stream_ptr(out))


def try_tensor_core(aten_op, a: MXTensor, b: MXTensor, extra_front, extra_back, count_fallback: bool = True,
                    fused: Optional[FusedOutput] = None) -> Optional[torch.Tensor]:
    """-> the contraction on the block-scaled tensor-core kernels, or None when the operands do not qualify (`count_fallback` is
    kept for callers of the first round and ignored: `contract` does the counting)"""
    out = None
    if not _DISABLED and not torch.compiler.is_compiling() and _qualifies(a) and _qualifies(b):
        out = _dispatch(aten_op, a, b, extra_front, extra_back, fused)
    if out is not None:
        stats["tensor_core"] += 1
    return out


# ---- K3d: every other operand pair (fused dequantize + bf16 tcgen05 GEMM, csrc/mxq_gemm_dequant.cu) ---------------------
_DEQUANT_GEMM = os.environ.get("MXQ_DEQUANT_GEMM", "1") != "0"


def set_dequant_gemm(flag: bool) -> bool:
    """tests: switch K3d off so that the same call takes the reference's own recipe (K2 + aten matmul); returns the old value"""
    global _DEQUANT_GEMM
    prev, _DEQUANT_GEMM = _DEQUANT_GEMM, bool(flag)
    return prev


def _plain(t: MXTensor) -> bool:
    return (isinstance(t, MXTensor) and type(t._data) is torch.Tensor and type(t._scale_e8m0) is torch.Tensor and t._data.is_cuda
            and t._orig_dtype == torch.bfloat16 and t._elem_dtype.name in dtypes.ELEM_ID)


def _collapse_rows(t: torch.Tensor):
    """[..., K] -> row stride over all leading dims taken as ONE row index, or None when they do not collapse"""
    if t.dim() == 1:
        return 0
    ld = t.stride(-2)
    expect = ld * t.shape[-2]
    for size, stride in zip(reversed(t.shape[:-2]), reversed(t.stride()[:-2])):
        if size > 1 and stride != expect:
            return None
        expect *= size
    return ld


def _fill_operand(o: "_C.Operand", t: MXTensor, rows_dim: int, k_dim: int, batched: bool, collapse: bool):
    """-> the (codes, scales) tensors the descriptor points into (the caller keeps them alive across the launch call), or None"""
    d, s = t._data, t._scale_e8m0
    nd = d.dim()
    rows_dim, k_dim = rows_dim % nd, k_dim % nd
    if t._block_dim not in (rows_dim, k_dim):
        return None
    if collapse and nd > 2:  # aten.linear on [..., K]: all leading dims form the row index
        if k_dim != nd - 1:
            return None
        cr, sr = _collapse_rows(d), _collapse_rows(s)
        if cr is None or sr is None:  # (not produced by the layers: make the operand dense once)
            d, s = d.contiguous(), s.contiguous()
            cr, sr = d.stride(-2), s.stride(-2)
        o.row_stride, o.srow_stride = cr, sr
    else:
        o.row_stride, o.srow_stride = d.stride(rows_dim), s.stride(rows_dim)
    o.codes, o.scales = d.data_ptr(), s.data_ptr()
    o.k_stride, o.sk_stride = d.stride(k_dim), s.stride(k_dim)
    o.batch_stride, o.sbatch_stride = (d.stride(0), s.stride(0)) if batched else (0, 0)
    o.elem, o.block_size, o.blocked_along_k = dtypes.ELEM_ID[t._elem_dtype.name], t._block_size, 1 if t._block_dim == k_dim else 0
    return d, s


DIRECT_MIN_ROWS = int(os.environ.get("MXQ_DEQUANT_ONCE_MIN_ROWS", 512))  # M and N from which operands are dequantized once (see try_dequant_gemm)


def try_dequant_gemm(aten_op, a: MXTensor, b: MXTensor, extra_front, extra_back) -> Optional[torch.Tensor]:
    """The contraction of two MXTensors of ANY element type / block size / block orientation / padding / strides as one
    kernel (`mxq_gemm_dequant`): what the reference computes as dequantize + bf16 matmul (torchmx/ops.py:29-41, 60-68,
    99-119), without materialising the bf16 operands and without a library GEMM.  None when the call is not one of the four
    compute overrides on plain CUDA MXTensors that advertise bf16."""
    if not _DEQUANT_GEMM or torch.compiler.is_compiling() or not _plain(a) or not _plain(b) or a._data.device != b._data.device:
        return None
    bias = None
    if aten_op is aten.linear.default:
        bias = extra_back[0] if extra_back else None
        b_rows, b_k = -2, -1   # weight [N, K]
    elif aten_op is aten.addmm.default:
        bias = extra_front[0]
        b_rows, b_k = -1, -2   # mat2 [K, N]
    elif aten_op in (aten.mm.default, aten.bmm.default):
        b_rows, b_k = -1, -2
    else:
        return None
    batched = aten_op is aten.bmm.default
    if batched:
        if a.dim() != 3 or b.dim() != 3 or a.shape[0] != b.shape[0]:
            return None
    elif b.dim() != 2 or a.dim() < 1 or (aten_op is not aten.linear.default and a.dim() != 2):
        return None
    K = a.shape[-1]
    if K != b.shape[b_k]:
        return None
    N = b.shape[b_rows]
    lead = tuple(a.shape[:-1])
    M = 1
    for v in (lead[1:] if batched else lead):
        M *= v
    batch = a.shape[0] if batched else 1
    if bias is not None:
        if isinstance(bias, MXTensor) or bias.dim() != 1 or bias.shape[0] != N or not bias.is_cuda:
            return None
        if bias.dtype != torch.bfloat16 or not bias.is_contiguous():
            return None
    if M >= DIRECT_MIN_ROWS and N >= DIRECT_MIN_ROWS and K % 8 == 0 and a.dim() >= 2:
        # large outputs: the fused kernel dequantizes every operand element once per 128 x 128 output tile it touches (N / 128 resp.
        # M / 128 times); dequantizing each operand ONCE (K2, any layout / block size / padding) and running the same tensor-core
        # loop on the bf16 matrices is what the reference's recipe does, and is ~4x faster at 8192^3 -- still no library GEMM
        a_hp = a.to_dtype(torch.bfloat16).reshape(batch, M, K)
        b_hp = (b if b_k == -1 else b.transpose(-1, -2)).to_dtype(torch.bfloat16).reshape(batch, N, K)
        out = torch.empty(lead + (N,), dtype=torch.bfloat16, device=a._data.device)
        if _C.launch("mxq_gemm_bf16", a_hp.data_ptr(), K, M * K, b_hp.data_ptr(), K, N * K, bias.data_ptr() if bias is not None else None,
                     out.data_ptr(), N, M * N, batch, M, N, K, out.device.index, _stream_ptr(out)):
            stats["dequant_gemm"] += 1
            stats["dequant_once_gemm"] += 1
            return out
    g = _C.GemmDequantArgs()
    keep_a = _fill_operand(g.a, a, -2, -1, batched, collapse=aten_op is aten.linear.default)
    keep_b = _fill_operand(g.b, b, b_rows, b_k, batched, False)
    if keep_a is None or keep_b is None:
        return None
    if a.dim() == 1:
        g.a.row_stride = g.a.srow_stride = 0
    out = torch.empty(lead + (N,), dtype=torch.bfloat16, device=a._data.device)
    if out.numel() == 0:
        return out
    g.bias = bias.data_ptr() if bias is not None else None
    g.d, g.ldd, g.d_batch_stride = out.data_ptr(), N, M * N
    g.batch, g.M, g.N, g.K = batch, M, N, K
    if not _C.launch("mxq_gemm_dequant", ctypes.byref(g), out.device.index, _stream_ptr(out)):
        return None
    del keep_a, keep_b
    stats["dequant_gemm"] += 1
    return out


def contract(aten_op, a: MXTensor, b: MXTensor, extra_front=(), extra_back=(), fused: Optional[FusedOutput] = None,
             count_fallback: bool = True) -> Optional[torch.Tensor]:
    """the MX matmul of the four compute overrides on this library's kernels: block-scaled tensor cores when the operands
    qualify, the fused dequantize GEMM otherwise; None (counted as `fallback`) only when neither applies"""
    out = try_tensor_core(aten_op, a, b, extra_front, extra_back, fused=fused)
    if out is None:
        out = try_dequant_gemm(aten_op, a, b, extra_front, extra_back)
    if out is None and count_fallback:
        stats["fallback"] += 1
    return out


def _dispatch(aten_op, a, b, extra_front, extra_back, fused: Optional[FusedOutput] = None):
    bias = None
    if aten_op is aten.linear.default:
        bias = extra_back[0] if extra_back else None
        b_k_from_end = 1  # weight is [N, K]
    elif aten_op is aten.addmm.default:
        bias = extra_front[0]
        b_k_from_end = 2  # mat2 is [K, N]
    elif aten_op in (aten.mm.default, aten.bmm.default):
        b_k_from_end = 2
    else:
        return None
    nd_a = a._data.dim()
    if a._block_dim != nd_a - 1:
        return None
    if b._block_dim != b._data.dim() - b_k_from_end:
        return None
    ak = _rows_k(a, 1)
    bk = _rows_k(b, b_k_from_end)
    if ak is None or bk is None:
        return None
    (a_codes, sfa), (b_codes, sfb) = ak, bk
    K = a.shape[-1]
    if K % 128 != 0 or K != (b.shape[-1] if b_k_from_end == 1 else b.shape[-2]):
        return None
    N = b.shape[-2] if b_k_from_end == 1 else b.shape[-1]
    if bias is not None:
        if isinstance(bias, MXTensor) or bias.dtype != torch.bfloat16 or bias.dim() != 1 or bias.shape[0] != N or not bias.is_contiguous():
            return None

    batched = aten_op is aten.bmm.default
    if batched:
        if a._data.dim() != 3 or b._data.dim() != 3:
            return None
        batch, M = a.shape[0], a.shape[1]
        lead_shape = (batch, M)
    else:
        if b._data.dim() != 2:
            return None
        if nd_a > 2:  # aten.linear on [..., K]: rows must collapse into one strided dim
            if not (a._data.is_contiguous() and a._scale_e8m0.is_contiguous()):
                return None
            a_codes, sfa = a_codes.reshape(-1, a_codes.shape[-1]), sfa.reshape(-1, sfa.shape[-1])
        batch, M = 1, a_codes.shape[0]
        lead_shape = tuple(a.shape[:-1])

    # tensor-core operand forms (packed 4 / 6-bit streams or E4M3 bytes; a weight caches its shadow on the origin MXTensor)
    b_origin = getattr(b, "_mxq_origin", b)
    a_e, a_fmt = _operand_rows(a_codes, a._elem_dtype, None)
    b_e, b_fmt = _operand_rows(b_codes, b._elem_dtype, b_origin if not batched else None)
    if a_e.stride(-1) != 1 or b_e.stride(-1) != 1:
        return None
    if fused is not None and not batched and fused.view.shape == (M, N) and fused.view.is_contiguous():
        out, d_mc = fused.view, fused.multicast_ptr
    else:
        fused, d_mc = None, 0
        out = torch.empty(lead_shape + (N,), dtype=torch.bfloat16, device=a._data.device)
    if out.numel() == 0:
        return out
    if batched:
        strides = (a_e.stride(0), sfa.stride(0), b_e.stride(0), sfb.stride(0))
        if any(s <= 0 for s in strides):
            return None  # expanded (stride 0) batch: not expressible as a TMA stride
    else:
        strides = (0, 0, 0, 0)
    static_b = not batched and _static_b(b_origin)
    ok = _launch(a_e, sfa, b_e, sfb, bias, batch, M, N, K, *strides, out, a_fmt, b_fmt, d_mc, static_b=static_b)
    if ok and fused is not None:
        fused.taken = True
        stats["fused_allreduce"] += 1
        return out.view(lead_shape + (N,))
    if not ok and fused is not None:  # shape not supported with the fused epilogue: plain output, the layer all-reduces it
        out = torch.empty(lead_shape + (N,), dtype=torch.bfloat16, device=a._data.device)
        ok = _launch(a_e, sfa, b_e, sfb, bias, batch, M, N, K, *strides, out, a_fmt, b_fmt, 0, static_b=static_b)
    return out if ok else None


# MXQ_FUSED_ACT_QUANT=0 keeps the separate activation-quantize launch in MXInferenceLinear.forward
_FUSED_ACT = os.environ.get("MXQ_FUSED_ACT_QUANT", "1") != "0"
FUSED_ACT_MAX_ROWS = 64


def linear_fused_act_quant(x: torch.Tensor, w: MXTensor, bias, fused: Optional[FusedOutput] = None) -> Optional[torch.Tensor]:
    """MXInferenceLinear.forward for decode-sized activations in ONE launch: y = quantize_mx(x, float8_e4m3, 32) @ w^T (+ bias)
    with the quantization done inside the weight-streaming kernel (bit-identical to the two-launch path).  Returns None when
    the operands do not qualify; the caller then quantizes with K1 and goes through `try_tensor_core`."""
    if _DISABLED or not _FUSED_ACT or torch.compiler.is_compiling() or type(x) is not torch.Tensor or not x.is_cuda or x.dtype != torch.bfloat16 or not _qualifies(w):
        return None
    K = x.shape[-1]
    if w._data.dim() != 2 or w._block_dim != 1 or K % 128 != 0 or w.shape[-1] != K or not x.is_contiguous():
        return None
    rows = x.numel() // K
    if rows == 0 or rows > FUSED_ACT_MAX_ROWS:
        return None
    wk = _rows_k(w, 1)
    if wk is None:
        return None
    if bias is not None and (isinstance(bias, MXTensor) or bias.dtype != torch.bfloat16 or bias.dim() != 1 or not bias.is_contiguous()):
        return None
    w_origin = getattr(w, "_mxq_origin", w)
    b_e, b_fmt = _operand_rows(wk[0], w._elem_dtype, w_origin)
    N = w.shape[0]
    x2 = x.view(rows, K)
    if fused is not None and fused.view.shape == (rows, N) and fused.view.is_contiguous():
        out, d_mc = fused.view, fused.multicast_ptr
    else:
        fused, d_mc = None, 0
        out = torch.empty(tuple(x.shape[:-1]) + (N,), dtype=torch.bfloat16, device=x.device)
    ok = _launch(None, None, b_e, wk[1], bias, 1, rows, N, K, 0, 0, 0, 0, out, FMT_E4M3_BYTES, b_fmt, d_mc, x_hp=x2,
                 x_flags=_quant_flags(dtypes.float8_e4m3), static_b=_static_b(w_origin))
    if not ok:
        return None
    stats["tensor_core"] += 1
    stats["fused_act_quant"] += 1
    if fused is not None:
        fused.taken = True
        stats["fused_allreduce"] += 1
        return out.view(tuple(x.shape[:-1]) + (N,))
    return out


def linear_packed_act_quant(x: torch.Tensor, w: MXTensor, bias, act_elem: dtypes.DType,
                            fused: Optional[FusedOutput] = None) -> Optional[torch.Tensor]:
    """MXInferenceLinear.forward with a 4 / 6-bit ACTIVATION config (reference: torchmx/layers/mx_linear.py:63-94 with
    `activations_config` float6_* / float4_e2m1): K1 writes the packed tensor-core operand stream itself (MXQ_FLAG_OPERAND_LAYOUT)
    and the GEMM reads it -- two launches, where quantize -> mxq_pack_operand -> GEMM were three and the codes made one more round
    trip through HBM.  Same codes, same scales, same GEMM: bit-identical to the three-launch path.  None when the operands do
    not qualify (the caller takes that path)."""
    if (_DISABLED or not _USE_PACKED or torch.compiler.is_compiling() or type(x) is not torch.Tensor or not x.is_cuda or x.dtype != torch.bfloat16
            or act_elem.name not in _PACKED_FORMAT or not _qualifies(w)):
        return None
    K = x.shape[-1]
    if w._data.dim() != 2 or w._block_dim != 1 or K % 128 != 0 or w.shape[-1] != K or not x.is_contiguous() or x.data_ptr() % 32:
        return None
    rows = x.numel() // K
    if rows == 0:
        return None
    wk = _rows_k(w, 1)
    if wk is None:
        return None
    if bias is not None and (isinstance(bias, MXTensor) or bias.dtype != torch.bfloat16 or bias.dim() != 1 or not bias.is_contiguous()):
        return None
    a_fmt = _PACKED_FORMAT[act_elem.name]
    a_e = torch.empty((rows, K * _PACKED_BITS[a_fmt] // 8), dtype=torch.uint8, device=x.device)
    sfa = torch.empty((rows, K // 32), dtype=torch.uint8, device=x.device)
    if not _C.launch("mxq_quantize", x.data_ptr(), _C.HP_BF16, rows * (K // 32), 32, dtypes.ELEM_ID[act_elem.name],
                     _C.FLAG_OPERAND_LAYOUT | _quant_flags(act_elem), a_e.data_ptr(), sfa.data_ptr(), x.device.index, _stream_ptr(x)):
        return None
    w_origin = getattr(w, "_mxq_origin", w)
    b_e, b_fmt = _operand_rows(wk[0], w._elem_dtype, w_origin)
    N = w.shape[0]
    if fused is not None and fused.view.shape == (rows, N) and fused.view.is_contiguous():
        out, d_mc = fused.view, fused.multicast_ptr
    else:
        fused, d_mc = None, 0
        out = torch.empty(tuple(x.shape[:-1]) + (N,), dtype=torch.bfloat16, device=x.device)
    ok = _launch(a_e, sfa, b_e, wk[1], bias, 1, rows, N, K, 0, 0, 0, 0, out, a_fmt, b_fmt, d_mc, static_b=_static_b(w_origin))
    if not ok and fused is not None:
        fused, d_mc = None, 0
        out = torch.empty(tuple(x.shape[:-1]) + (N,), dtype=torch.bfloat16, device=x.device)
        ok = _launch(a_e, sfa, b_e, wk[1], bias, 1, rows, N, K, 0, 0, 0, 0, out, a_fmt, b_fmt, 0, static_b=_static_b(w_origin))
    if not ok:
        return None
    stats["tensor_core"] += 1
    stats["packed_act_quant"] += 1
    if fused is not None:
        fused.taken = True
        stats["fused_allreduce"] += 1
        return out.view(tuple(x.shape[:-1]) + (N,))
    return out


def pack_weight(w: MXTensor):
    """MXTensor weight [N, K] (blocks along K) -> (operand tensor, MXQ_OPERAND_* format) in the form the tensor-core kernels
    consume: the dense 4 / 6-bit stream for fp4 / fp6, the code bytes themselves for fp8.  None if the weight cannot run on
    the tensor-core path at all (a packed-only layer has no dequantize path to fall back to)."""
    if not _qualifies(w) or w._data.dim() != 2 or w._block_dim != 1 or w.shape[-1] % 128 != 0 or not w._data.is_contiguous():
        return None
    return _operand_rows(w._data, w._elem_dtype, None, packed=True)


def unpack_weight(packed: torch.Tensor, fmt: int, elem: dtypes.DType) -> torch.Tensor:
    """the inverse of `pack_weight`: reference-layout codes (MXTensor._data), bit-for-bit"""
    if fmt in (FMT_E4M3_BYTES, FMT_E5M2_BYTES):
        return packed.clone()
    bits = _PACKED_BITS[fmt]
    k = packed.shape[-1] * 8 // bits
    out = _codes_like(packed.shape[:-1], k, elem, packed.device)
    rc = _C.lib().mxq_unpack_operand(packed.data_ptr(), dtypes.ELEM_ID[elem.name], packed.numel() * 8 // bits, out.data_ptr(),
                                     packed.device.index, _stream_ptr(packed))
    _C.check(rc, "mxq_unpack_operand")
    return out


def linear_packed_weight(x, b_e: torch.Tensor, sfb: torch.Tensor, b_fmt: int, bias, act_elem: dtypes.DType, owner=None) -> torch.Tensor:
    """y = quantize_mx(x, act_elem, 32) @ W^T (+ bias) for a weight held only as its tensor-core operand (`pack_weight`).
    x: bf16 [..., K] or an MXTensor already quantized with the layer's activation config.  Decode-sized bf16 activations
    are quantized inside the GEMM; everything else goes K1 -> K3.  Raises if the launch is refused: there is no other path."""
    N, K = b_e.shape[0], sfb.shape[-1] * 32
    lead = tuple(x.shape[:-1])
    assert x.shape[-1] == K, f"activation has {x.shape[-1]} features, the weight {K}"
    if bias is not None:
        assert bias.dtype == torch.bfloat16 and bias.dim() == 1 and bias.shape[0] == N and bias.is_contiguous()
    rows = x.numel() // K if K else 0
    out = torch.empty(lead + (N,), dtype=torch.bfloat16, device=b_e.device)
    if rows == 0:
        return out
    static_b = owner is not None and _static_b(owner)
    if (not isinstance(x, MXTensor) and _FUSED_ACT and act_elem == dtypes.float8_e4m3 and rows <= FUSED_ACT_MAX_ROWS and x.is_contiguous()
            and x.dtype == torch.bfloat16):
        ok = _launch(None, None, b_e, sfb, bias, 1, rows, N, K, 0, 0, 0, 0, out, FMT_E4M3_BYTES, b_fmt, 0, x_hp=x.view(rows, K),
                     x_flags=_quant_flags(act_elem), static_b=static_b)
        if ok:
            stats["tensor_core"] += 1
            stats["fused_act_quant"] += 1
            return out
    if (not isinstance(x, MXTensor) and _USE_PACKED and act_elem.name in _PACKED_FORMAT and type(x) is torch.Tensor and x.dtype == torch.bfloat16
            and x.is_contiguous() and x.data_ptr() % 32 == 0):
        # 4 / 6-bit activation config: K1 writes the packed operand stream itself (see linear_packed_act_quant)
        a_fmt = _PACKED_FORMAT[act_elem.name]
        a_e = torch.empty((rows, K * _PACKED_BITS[a_fmt] // 8), dtype=torch.uint8, device=x.device)
        sfa = torch.empty((rows, K // 32), dtype=torch.uint8, device=x.device)
        if (_C.launch("mxq_quantize", x.data_ptr(), _C.HP_BF16, rows * (K // 32), 32, dtypes.ELEM_ID[act_elem.name],
                      _C.FLAG_OPERAND_LAYOUT | _quant_flags(act_elem), a_e.data_ptr(), sfa.data_ptr(), x.device.index, _stream_ptr(x))
                and _launch(a_e, sfa, b_e, sfb, bias, 1, rows, N, K, 0, 0, 0, 0, out, a_fmt, b_fmt, 0, static_b=static_b)):
            stats["tensor_core"] += 1
            stats["packed_act_quant"] += 1
            return out
    x_mx = x if isinstance(x, MXTensor) else MXTensor.to_mx(x, act_elem, 32)
    assert _qualifies(x_mx) and x_mx._block_dim == x_mx._data.dim() - 1 and x_mx._data.is_contiguous(), "activation cannot run on the tensor-core path"
    a_codes, sfa = x_mx._data.reshape(rows, -1), x_mx._scale_e8m0.reshape(rows, -1)
    a_e, a_fmt = _operand_rows(a_codes, x_mx._elem_dtype, None)
    if not _launch(a_e, sfa, b_e, sfb, bias, 1, rows, N, K, 0, 0, 0, 0, out, a_fmt, b_fmt, 0, static_b=static_b):
        raise RuntimeError(f"mxq_gemm refused [{rows}, {K}] x [{N}, {K}]^T for a packed-only weight: {_C.lib().mxq_last_error().decode()}")
    stats["tensor_core"] += 1
    return out
