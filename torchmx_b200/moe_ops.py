"""Host side of K6 (csrc/mxq_moe.cu, C entries `mxq_moe_route` / `mxq_moe_gemm` / `mxq_moe_combine`): the three launches of a
mixture-of-experts layer that are not K1b.  None of them reads a device value on the host, so a decode step built from them can
be captured in a CUDA graph.  There is no CPU path; a refused launch raises (the layer checks the shapes before it comes here).
"""
from __future__ import annotations

import ctypes
from typing import Optional

import torch

from . import _C, dtypes, mx_gemm
from .mx_tensor import MXTensor, _codes_like, _quant_flags, _stream_ptr

stats = {"grouped_experts": 0}


def route(top_k_index: torch.Tensor, num_experts: int, x: Optional[torch.Tensor] = None, elem: Optional[dtypes.DType] = None):
    """top_k_index int64 [T, k] -> (offsets int32 [E + 1], row_of_slot int32 [T * k], token_of_row int32 [T * k], codes, scales).

    The routed rows of expert e are offsets[e] .. offsets[e + 1] - 1, in (token, slot) order; slot (t, s) went to row
    row_of_slot[t * k + s] (-1 when its expert is outside [0, E)).  With `x` (bf16 [T, H]) routed row r of `codes` / `scales`
    ([T * k, H] reference-layout codes, [T * k, H / 32]) is quantize_mx(x[token_of_row[r]], elem, 32); otherwise both are None."""
    T, k = top_k_index.shape
    dev = top_k_index.device
    idx = top_k_index.contiguous()
    offsets = torch.empty(num_experts + 1, dtype=torch.int32, device=dev)
    row_of_slot = torch.empty(T * k, dtype=torch.int32, device=dev)
    token_of_row = torch.empty(T * k, dtype=torch.int32, device=dev)
    a = _C.MoeRouteArgs()
    a.top_k_index, a.tokens, a.top_k, a.num_experts = idx.data_ptr(), T, k, num_experts
    a.offsets, a.row_of_slot, a.token_of_row = offsets.data_ptr(), row_of_slot.data_ptr(), token_of_row.data_ptr()
    codes = scales = None
    if x is not None:
        H = x.shape[-1]
        codes = _codes_like((T * k,), H, elem, dev)
        scales = torch.empty((T * k, H // 32), dtype=torch.uint8, device=dev)
        a.x, a.ldx, a.hidden = x.data_ptr(), x.stride(0), H
        a.elem, a.flags = dtypes.ELEM_ID[elem.name], _quant_flags(elem)
        a.codes, a.scales = codes.data_ptr(), scales.data_ptr()
    _C.check(_C.lib().mxq_moe_route(ctypes.byref(a), dev.index, _stream_ptr(idx)), "mxq_moe_route")
    return offsets, row_of_slot, token_of_row, codes, scales


def grouped_linear(x_codes: torch.Tensor, x_scales: torch.Tensor, x_elem: dtypes.DType, w: MXTensor, offsets: torch.Tensor) -> torch.Tensor:
    """D [R, N] bf16 with D[r] = X[r] . W[e(r)]^T for the routed rows r < offsets[E] (rows past it are left unwritten).
    x_codes / x_scales: reference-layout codes [R, K] / scales [R, K / 32]; w: an MXTensor bank [E, N, K] blocked along K.
    fp6 / fp4 operands run as their packed tensor-core streams (mx_gemm._operand_rows; the bank's stream is cached on it)."""
    E, N, K = w.shape
    R = x_scales.shape[0]
    x_op, x_fmt = mx_gemm._operand_rows(x_codes, x_elem, None)
    w_op, w_fmt = mx_gemm._operand_rows(w._data.view(E * N, -1), w._elem_dtype, getattr(w, "_mxq_origin", w))
    d = torch.empty((R, N), dtype=torch.bfloat16, device=x_codes.device)
    g = _C.MoeGemmArgs()
    g.w_codes, g.w_scales, g.w_format = w_op.data_ptr(), w._scale_e8m0.data_ptr(), w_fmt
    g.x_codes, g.x_scales, g.x_format = x_op.data_ptr(), x_scales.data_ptr(), x_fmt
    g.offsets, g.d = offsets.data_ptr(), d.data_ptr()
    g.rows, g.num_experts, g.N, g.K = R, E, N, K
    _C.check(_C.lib().mxq_moe_gemm(ctypes.byref(g), d.device.index, _stream_ptr(d)), "mxq_moe_gemm")
    return d


def combine(y: torch.Tensor, top_k_index: torch.Tensor, top_k_weights: torch.Tensor, row_of_slot: torch.Tensor, num_experts: int) -> torch.Tensor:
    """out [T, H] bf16: the loop's index_add_ sequence over the routed rows `y` [R, H] -- per token, starting from +0, the
    contributions bf16(fp32(y) * w) added in bf16 in ascending expert order.  top_k_weights: fp32 or bf16 [T, k]."""
    T, k = top_k_index.shape
    H = y.shape[-1]
    out = torch.empty((T, H), dtype=torch.bfloat16, device=y.device)
    idx, wts = top_k_index.contiguous(), top_k_weights.contiguous()
    c = _C.MoeCombineArgs()
    c.y, c.top_k_index, c.top_k_weights = y.data_ptr(), idx.data_ptr(), wts.data_ptr()
    c.weights_dtype = _C.HP_BF16 if wts.dtype == torch.bfloat16 else _C.HP_F32
    c.row_of_slot = row_of_slot.data_ptr()
    c.tokens, c.top_k, c.num_experts, c.hidden = T, k, num_experts, H
    c.out = out.data_ptr()
    _C.check(_C.lib().mxq_moe_combine(ctypes.byref(c), out.device.index, _stream_ptr(out)), "mxq_moe_combine")
    return out
