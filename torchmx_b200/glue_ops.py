"""Host side of K5 (csrc/mxq_glue.cu, C entries `mxq_rmsnorm` / `mxq_rope`): the row-wise and elementwise steps between the MX
linears of a Llama / Qwen2 decoder layer, each as ONE launch.

* `rmsnorm(x, weight, eps, residual=None, to_mx=None)`: transformers' LlamaRMSNorm / Qwen2RMSNorm arithmetic (fp32 statistics,
  normalised row rounded to bf16 before the bf16 multiply by the weight), optionally preceded by the residual add of the decoder
  layer and optionally followed by the MX quantization every consumer of the norm output applies on entry
  (reference: torchmx/layers/mx_linear.py:63-66) -- the codes are bit-identical to `MXTensor.to_mx` of the bf16 norm output.
* `rope(q, k, cos, sin)`: `apply_rotary_pos_emb` of transformers (reference call site: torchmx/layers/mx_llama_attention.py:171-187)
  with every bf16 rounding of the eager chain reproduced, reading the projection outputs in place.
* `rope_quantize_kv(...)` (K5e, csrc/mxq_kv_cache.cu): rope, the append to an MX-quantized static KV cache and the quantization of
  Q in one launch (the cache itself: torchmx_b200/kv_cache.py).

Both return None when the operands do not qualify (the caller runs the module / the eager chain); there is no CPU path.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch

from . import _C, dtypes
from .mlp_ops import _rows_view
from .mx_tensor import MXTensor, _codes_like, _quant_flags, _stream_ptr

stats = {"rmsnorm": 0, "rmsnorm_to_mx": 0, "rope": 0, "quantize_heads": 0, "quantize_transposed": 0, "rope_quantize_kv": 0}
_ENABLED = os.environ.get("MXQ_FUSED_GLUE", "1") != "0"
MAX_HIDDEN = 16384


def set_fused_glue(on: bool) -> bool:
    global _ENABLED
    prev, _ENABLED = _ENABLED, bool(on)
    return prev


def _plain_bf16(t, dev=None) -> bool:
    return type(t) in (torch.Tensor, torch.nn.Parameter) and t.is_cuda and t.dtype == torch.bfloat16 and (dev is None or t.device == dev)


def rmsnorm(x: torch.Tensor, weight: torch.Tensor, eps: float, residual: Optional[torch.Tensor] = None,
            to_mx: Optional[dtypes.DType] = None, want_y: bool = True):
    """-> (y | None, MXTensor | None, h | None) or None when the kernel does not apply.

    h = x + residual (bf16, only when `residual` is given: the stream the decoder layer carries on), y = weight * norm(h) in bf16
    (only when `want_y`), MXTensor = to_mx(y, to_mx, 32) (only when `to_mx` is given)."""
    if not _ENABLED or not _plain_bf16(x) or not _plain_bf16(weight, x.device) or x.dim() < 1 or x.numel() == 0:
        return None
    hidden = x.shape[-1]
    if hidden % 32 or hidden > MAX_HIDDEN or weight.shape != (hidden,) or not weight.is_contiguous() or weight.data_ptr() % 16:
        return None
    ldx = _rows_view(x)
    if ldx is None or ldx % 8 or x.data_ptr() % 16 or not (want_y or to_mx is not None):
        return None
    a = _C.RmsNormArgs()
    a.x, a.ldx = x.data_ptr(), ldx
    h = None
    if residual is not None:
        if not _plain_bf16(residual, x.device) or residual.shape != x.shape:
            return None
        ldr = _rows_view(residual)
        if ldr is None or ldr % 8 or residual.data_ptr() % 16:
            return None
        h = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
        a.residual, a.ld_res, a.residual_out, a.ld_res_out = residual.data_ptr(), ldr, h.data_ptr(), hidden
    a.weight, a.eps = weight.data_ptr(), float(eps)
    a.rows, a.hidden = x.numel() // hidden, hidden
    y = mx = None
    if want_y:
        y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
        a.y, a.ldy = y.data_ptr(), hidden
    if to_mx is not None:
        lead = tuple(x.shape[:-1])
        codes = _codes_like(lead, hidden, to_mx, x.device)
        scales = torch.empty(lead + (hidden // 32,), dtype=torch.uint8, device=x.device)
        a.codes, a.scales, a.elem = codes.data_ptr(), scales.data_ptr(), dtypes.ELEM_ID[to_mx.name]
        a.flags = _quant_flags(to_mx)
    if not _C.launch("mxq_rmsnorm", a, x.device.index, _stream_ptr(x)):
        return None
    if to_mx is not None:
        mx = MXTensor(scales, codes, to_mx, 32, torch.bfloat16)
        stats["rmsnorm_to_mx"] += 1
    else:
        stats["rmsnorm"] += 1
    return y, mx, h


def _head_view(t: torch.Tensor, head_dim: int):
    """[batch, heads, tokens, head_dim] view of a projection output whose heads are contiguous inside a token row
    -> (batch stride, token stride) in elements, or None"""
    if t.dim() != 4 or t.shape[3] != head_dim or t.stride(3) != 1 or (t.shape[1] > 1 and t.stride(1) != head_dim):
        return None
    return (t.stride(0) if t.shape[0] > 1 else 0), (t.stride(2) if t.shape[2] > 1 else t.shape[1] * head_dim)


def _out_view(t: torch.Tensor, like: torch.Tensor):
    """a caller-provided output [batch, heads, tokens, head_dim] (e.g. a slice of a KV cache): its three leading strides, or None"""
    if not _plain_bf16(t, like.device) or t.shape != like.shape or t.stride(3) != 1 or t.data_ptr() % 16 or any(st % 8 for st in t.stride()[:3]):
        return None
    return t.stride(0), t.stride(1), t.stride(2)


def _set_rope_tables(a, cos: torch.Tensor, sin: torch.Tensor, b: int, t: int, d: int) -> bool:
    """Point the cos / sin fields of K5b's / K5e's arguments at the tables ([b | 1, t, d], the same strides, unit last stride;
    d > 1); False when they do not qualify."""
    if cos.shape != sin.shape or cos.dim() != 3 or cos.shape[0] not in (1, b) or cos.shape[1] != t or cos.shape[2] != d \
            or cos.stride() != sin.stride() or cos.stride(2) != 1:
        return False
    a.cos, a.sin = cos.data_ptr(), sin.data_ptr()
    a.cs_tok_stride = cos.stride(1) if t > 1 else d
    a.cs_batch_stride = cos.stride(0) if cos.shape[0] > 1 else 0
    return True


def rope(q: torch.Tensor, k: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, k_out: Optional[torch.Tensor] = None,
         v: Optional[torch.Tensor] = None, v_out: Optional[torch.Tensor] = None) -> Optional[Tuple[torch.Tensor, torch.Tensor]]:
    """q / k: [batch, heads, tokens, head_dim] (transposed views of the [batch, tokens, heads * head_dim] projection outputs);
    cos / sin: bf16 [batch | 1, tokens, head_dim] -> rotated (q, k), contiguous [batch, heads, tokens, head_dim].

    `k_out` (optional): where the rotated keys go instead of a fresh tensor -- any [batch, heads, tokens, head_dim] view with unit
    last stride, e.g. `key_cache[:, :, pos : pos + tokens]`, so the cache update needs no launch of its own.  `v` / `v_out`
    (optional, together): the value heads (k's geometry) are copied unrotated into `v_out` by the same launch."""
    if not _ENABLED or not _plain_bf16(q) or not _plain_bf16(k, q.device) or not _plain_bf16(cos, q.device) or not _plain_bf16(sin, q.device):
        return None
    if q.dim() != 4 or k.dim() != 4 or q.numel() == 0 or k.numel() == 0:
        return None
    b, hq, t, d = q.shape
    if k.shape[0] != b or k.shape[2] != t or k.shape[3] != d or d % 16:
        return None
    qv, kv = _head_view(q, d), _head_view(k, d)
    if qv is None or kv is None:
        return None
    a = _C.RopeArgs()
    if not _set_rope_tables(a, cos, sin, b, t, d):
        return None
    a.q, a.q_batch_stride, a.q_tok_stride, a.q_heads = q.data_ptr(), qv[0], qv[1], hq
    a.k, a.k_batch_stride, a.k_tok_stride, a.k_heads = k.data_ptr(), kv[0], kv[1], k.shape[1]
    a.batch, a.tokens, a.head_dim = b, t, d
    q_out = torch.empty((b, hq, t, d), dtype=torch.bfloat16, device=q.device)
    if k_out is None:
        k_out = torch.empty((b, k.shape[1], t, d), dtype=torch.bfloat16, device=q.device)
    else:
        ko = _out_view(k_out, k)
        if ko is None:
            return None
        a.k_out_batch_stride, a.k_out_head_stride, a.k_out_tok_stride = ko
    if (v is None) != (v_out is None):
        return None
    if v is not None:
        vv, vo = (_head_view(v, d) if _plain_bf16(v, q.device) and v.shape == k.shape else None), _out_view(v_out, k)
        if vv is None or vo is None:
            return None
        a.v, a.v_batch_stride, a.v_tok_stride = v.data_ptr(), vv[0], vv[1]
        a.v_out = v_out.data_ptr()
        a.v_out_batch_stride, a.v_out_head_stride, a.v_out_tok_stride = vo
    a.q_out, a.k_out = q_out.data_ptr(), k_out.data_ptr()
    if not _C.launch("mxq_rope", a, q.device.index, _stream_ptr(q)):
        return None
    stats["rope"] += 1
    return q_out, k_out


def quantize_heads(x: torch.Tensor, elem_dtype: dtypes.DType, block_size: int = 32) -> Optional[MXTensor]:
    """x: bf16 [batch, heads, tokens, head_dim] contiguous (an attention kernel's output) -> the MXTensor
    `MXTensor.to_mx(x.transpose(1, 2).reshape(batch, tokens, heads * head_dim), elem_dtype, 32)` without writing the transposed
    tensor (K5c); None when the kernel does not apply"""
    if not _ENABLED or block_size != 32 or not _plain_bf16(x) or x.dim() != 4 or not x.is_contiguous() or x.numel() == 0:
        return None
    b, h, t, d = x.shape
    if d % 32 or x.data_ptr() % 32:
        return None
    codes = _codes_like((b, t), h * d, elem_dtype, x.device)
    scales = torch.empty((b, t, h * d // 32), dtype=torch.uint8, device=x.device)
    if not _C.launch("mxq_quantize_heads", x.data_ptr(), b, h, t, d, dtypes.ELEM_ID[elem_dtype.name], _quant_flags(elem_dtype), codes.data_ptr(),
                     scales.data_ptr(), x.device.index, _stream_ptr(x)):
        return None
    stats["quantize_heads"] += 1
    return MXTensor(scales, codes, elem_dtype, 32, torch.bfloat16)


def quantize_transposed(x: torch.Tensor, elem_dtype: dtypes.DType, block_size: int = 32) -> Optional[MXTensor]:
    """x: bf16 [n0, n1, rows, cols] (any strides over the first three dims, cols contiguous: a value tensor or a slice of a value
    cache) -> the MXTensor `MXTensor.to_mx(x.transpose(-2, -1), elem_dtype, 32)` -- shape [n0, n1, cols, rows], blocks along the
    rows (key positions) -- without materialising the transposed bf16 tensor (K5d); None when the kernel does not apply"""
    if not _ENABLED or block_size != 32 or not _plain_bf16(x) or x.dim() != 4 or x.numel() == 0 or x.stride(3) != 1:
        return None
    n0, n1, rows, cols = x.shape
    if rows % 32 or cols % 8 or n0 * n1 > 65535 or x.data_ptr() % 16 or any(st % 8 for st in x.stride()[:3]):
        return None
    codes = _codes_like((n0, n1, cols), rows, elem_dtype, x.device)
    scales = torch.empty((n0, n1, cols, rows // 32), dtype=torch.uint8, device=x.device)
    a = _C.TransposedQuantArgs()
    a.x, a.n0, a.n1, a.rows, a.cols = x.data_ptr(), n0, n1, rows, cols
    a.s0, a.s1, a.row_stride = x.stride(0), x.stride(1), x.stride(2)
    a.elem = dtypes.ELEM_ID[elem_dtype.name]
    a.flags = _quant_flags(elem_dtype)
    a.codes, a.scales = codes.data_ptr(), scales.data_ptr()
    if not _C.launch("mxq_quantize_transposed", a, x.device.index, _stream_ptr(x)):
        return None
    stats["quantize_transposed"] += 1
    return MXTensor(scales, codes, elem_dtype, 32, torch.bfloat16)


def byte_operand_dtype(elem_dtype: dtypes.DType) -> dtypes.DType:
    """The element type whose one-byte codes hold `elem_dtype`'s values in the form K4b reads: e4m3 / e5m2 themselves, fp6 / fp4
    as their exact E4M3 re-encoding (every e3m2 / e2m3 / e2m1 value is an e4m3 value)"""
    return dtypes.float8_e5m2 if elem_dtype == dtypes.float8_e5m2 else dtypes.float8_e4m3


def rope_quantize_kv(q: torch.Tensor, k: torch.Tensor, v: torch.Tensor, cos: torch.Tensor, sin: torch.Tensor, position: torch.Tensor,
                     k_codes: torch.Tensor, k_scales: torch.Tensor, vt_codes: torch.Tensor, vt_scales: torch.Tensor, v_open: torch.Tensor,
                     elem_dtypes: Tuple[dtypes.DType, dtypes.DType, dtypes.DType]) -> Optional[MXTensor]:
    """K5e: rotary embedding of q / k, the append of the rotated keys and of v to an MX-quantized static KV cache at the device
    position `position` (int64, one element; read, not advanced), and the quantization of the rotated queries -- one launch.

    q / k / v: [batch, heads, tokens, 128] transposed views of the projection outputs (as for `rope`); cos / sin: bf16
    [batch | 1, tokens, 128].  The cache (uint8, contiguous, capacity C): k_codes [b, hk, C, 128], k_scales [b, hk, C, 4],
    vt_codes [b, hk, 128, C], vt_scales [b, hk, 128, C / 32], v_open bf16 [b, hk, 32, 128].  `elem_dtypes`: the element types of
    Q, K and V; codes are stored as `byte_operand_dtype` codes.  Returns Q as an MXTensor [b, hq, tokens, 128] of that storage
    type, or None when the kernel does not apply."""
    if not all(_plain_bf16(t, q.device) for t in (q, k, v, cos, sin)) or q.dim() != 4 or k.dim() != 4 or q.numel() == 0:
        return None
    if any(e == dtypes.int8 for e in elem_dtypes):
        return None
    b, hq, t, d = q.shape
    hk = k.shape[1]
    if d != 128 or k.shape != (b, hk, t, d) or v.shape != k.shape:
        return None
    qv, kv, vv = _head_view(q, d), _head_view(k, d), _head_view(v, d)
    if qv is None or kv is None or vv is None:
        return None
    C = k_codes.shape[2]
    want = ((k_codes, (b, hk, C, d)), (k_scales, (b, hk, C, d // 32)), (vt_codes, (b, hk, d, C)), (vt_scales, (b, hk, d, C // 32)))
    if any(x.dtype != torch.uint8 or x.device != q.device or tuple(x.shape) != shp or not x.is_contiguous() for x, shp in want):
        return None
    if v_open.dtype != torch.bfloat16 or v_open.shape != (b, hk, 32, d) or not v_open.is_contiguous() or v_open.device != q.device:
        return None
    if position.dtype != torch.int64 or position.numel() != 1 or position.device != q.device:
        return None
    a = _C.RopeQuantizeKVArgs()
    if not _set_rope_tables(a, cos, sin, b, t, d):
        return None
    a.q, a.q_batch_stride, a.q_tok_stride, a.q_heads = q.data_ptr(), qv[0], qv[1], hq
    a.k, a.k_batch_stride, a.k_tok_stride = k.data_ptr(), kv[0], kv[1]
    a.v, a.v_batch_stride, a.v_tok_stride, a.kv_heads = v.data_ptr(), vv[0], vv[1], hk
    a.batch, a.tokens, a.head_dim = b, t, d
    a.q_elem, a.k_elem, a.v_elem = (dtypes.ELEM_ID[e.name] for e in elem_dtypes)
    a.flags = _quant_flags(elem_dtypes[0]) | _quant_flags(elem_dtypes[1]) | _quant_flags(elem_dtypes[2])
    q_codes = torch.empty((b, hq, t, d), dtype=torch.uint8, device=q.device)
    q_scales = torch.empty((b, hq, t, d // 32), dtype=torch.uint8, device=q.device)
    a.q_codes, a.q_scales = q_codes.data_ptr(), q_scales.data_ptr()
    a.k_codes, a.k_scales, a.vt_codes, a.vt_scales = k_codes.data_ptr(), k_scales.data_ptr(), vt_codes.data_ptr(), vt_scales.data_ptr()
    a.v_open, a.capacity, a.position = v_open.data_ptr(), C, position.data_ptr()
    if not _C.launch("mxq_rope_quantize_kv", a, q.device.index, _stream_ptr(q)):
        return None
    stats["rope_quantize_kv"] += 1
    return MXTensor(q_scales, q_codes, byte_operand_dtype(elem_dtypes[0]), 32, torch.bfloat16)
