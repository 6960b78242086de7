"""Host side of the fused attention kernels: K4a (csrc/mxq_softmax.cu, C entry `mxq_softmax_quantize`: the chain between the two MX
matmuls) and K4b (csrc/mxq_flash_attention.cu, C entry `mxq_flash_attention`: both matmuls and the chain as one kernel).

`softmax_to_mx(scores, scaling, mask, causal, elem_dtype)` is the chain between the two MX matmuls of the reference's MX
attention block (torchmx/layers/mx_llama_attention.py:214-239: `/ sqrt(head_dim)`, `+ causal_mask`, fp32 softmax, `.to(bf16)`,
`MXTensor.to_mx(..., attention_weights_config)`) as one pass over the bf16 scores.  There is no CPU / PyTorch fallback: when the
shape does not qualify the function returns None and the caller runs the unfused chain of K1 + aten ops.
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from . import _C, dtypes
from .mx_tensor import MXTensor, _codes_like, _quant_flags, _require_cuda, _stream_ptr

stats = {"fused_softmax": 0, "unfused_softmax": 0, "flash_attention": 0}
_ENABLED = os.environ.get("MXQ_FUSED_SOFTMAX", "1") != "0"
_FLASH = os.environ.get("MXQ_FLASH_ATTENTION", "1") != "0"
MAX_KV = 32768
MAX_FLASH_KV = 131072  # the longest key axis K4b takes, masked or not (MXQ_FLASH_MAX_KV)


def set_fused_softmax(on: bool) -> bool:
    """Switch the fused kernel on / off (tests compare the two paths); returns the previous setting."""
    global _ENABLED
    prev, _ENABLED = _ENABLED, bool(on)
    return prev


def _set_mask(a, mask: Optional[torch.Tensor], b: int, h: int, q_len: int, kv_len: int, device) -> bool:
    """Point the mask fields of K4a's / K4b's arguments at `mask` (None, or additive bf16 on `device` broadcastable to
    [b, h, q_len, >= kv_len] with kv stride 1); False when the mask does not qualify."""
    if mask is None:
        return True
    if mask.dtype != torch.bfloat16 or mask.dim() != 4 or mask.device != device or mask.shape[-1] < kv_len or mask.shape[2] != q_len \
            or mask.shape[0] not in (1, b) or mask.shape[1] not in (1, h) or (kv_len > 1 and mask.stride(3) != 1):
        return False
    a.mask = mask.data_ptr()
    a.mask_stride_b = 0 if mask.shape[0] == 1 else mask.stride(0)
    a.mask_stride_h = 0 if mask.shape[1] == 1 else mask.stride(1)
    a.mask_stride_q = mask.stride(2)
    return True


def softmax_to_mx(scores: torch.Tensor, scaling: float, mask: Optional[torch.Tensor], causal: bool, elem_dtype: dtypes.DType,
                  block_size: int = 32) -> Optional[MXTensor]:
    """bf16 scores [batch, heads, q_len, kv_len] -> MXTensor of softmax(scores * scaling + mask) quantized along kv.

    mask: None or an additive bf16 tensor broadcastable to the scores ([b | 1, h | 1, q_len, >= kv_len], kv stride 1);
    causal: additionally hide kv index j > q + (kv_len - q_len).  Returns None when the kernel does not apply.
    """
    if not _ENABLED or block_size != 32 or scores.dim() != 4 or scores.dtype != torch.bfloat16 or not scores.is_contiguous():
        return None
    b, h, q_len, kv_len = scores.shape
    if kv_len % 32 or kv_len > MAX_KV or scores.numel() == 0 or scores.data_ptr() % 32:
        return None
    _require_cuda(scores, "softmax_to_mx")
    a = _C.SoftmaxArgs()
    if not _set_mask(a, mask, b, h, q_len, kv_len, scores.device):
        return None
    codes = _codes_like((b, h, q_len), kv_len, elem_dtype, scores.device)
    scales = torch.empty((b, h, q_len, kv_len // 32), dtype=torch.uint8, device=scores.device)
    a.scores = scores.data_ptr()
    a.batch, a.heads, a.q_len, a.kv_len = b, h, q_len, kv_len
    a.scaling = float(scaling)
    a.causal = 1 if causal else 0
    a.elem = dtypes.ELEM_ID[elem_dtype.name]
    a.flags = _quant_flags(elem_dtype)
    a.codes, a.scales = codes.data_ptr(), scales.data_ptr()
    if not _C.launch("mxq_softmax_quantize", a, scores.device.index, _stream_ptr(scores)):
        return None
    stats["fused_softmax"] += 1
    return MXTensor(scales, codes, elem_dtype, 32, scores.dtype)


def set_flash_attention(on: bool) -> bool:
    """Switch K4b on / off (tests compare it with the K3 -> K4a -> K3 chain); returns the previous setting."""
    global _FLASH
    prev, _FLASH = _FLASH, bool(on)
    return prev


CHAIN_DECODE_MAX_CTAS = 16


def chain_is_faster(batch: int, kv_heads: int, q_len: int, kv_len: int, masked: bool) -> bool:
    """True for a decode step the K3 -> K4a -> K3 chain serves faster than K4b (same results either way: K4a takes the row).

    K4b has no split over the key axis: a decode step is batch x kv_heads CTAs, each walking the whole key axis three times, and
    costs about the same at 8 CTAs as at 256 (one wave).  The chain's cost grows with the batch instead.  On one B200 (1000 W),
    Llama-3-8B heads (8 kv heads), unmasked, K4b against the chain at 2048 / 8192 / 32768 keys (profiles/r4_long_attention.json):
    batch 1 (8 CTAs) 88 / 334 / 1322 us against 56 / 171 / 634; batch 2 (16 CTAs) 88 / 334 / 1330 against 87 / 315 / 1180;
    batch 4 (32 CTAs) 92 / 347 / 1380 against 159 / 592 / 2293; batch 32 109 / 420 / 1632 against 1168 / 4517 / 18129.
    Rows K4b took before it handled long key axes (up to 1024 keys unmasked, 8192 masked) stay with K4b."""
    return (q_len == 1 and batch * kv_heads <= CHAIN_DECODE_MAX_CTAS and kv_len <= MAX_KV
            and kv_len > (8192 if masked else 1024))


def _byte_operand(t: MXTensor):
    """contiguous MXTensor blocked along its last dim -> (one-byte-per-element codes, MXQ_OPERAND_* format, scales) or None"""
    from . import mx_gemm
    if mx_gemm._DISABLED or torch.compiler.is_compiling() or not mx_gemm._qualifies(t) or t._block_dim != t._data.dim() - 1 or not t._data.is_contiguous() or not t._scale_e8m0.is_contiguous():
        return None
    codes, fmt = mx_gemm._operand_rows(t._data, t._elem_dtype, None, packed=False)  # e4m3 / e5m2 as they are, fp6 / fp4 as E4M3 bytes
    return codes, fmt, t._scale_e8m0


def flash_attention(q_mx: MXTensor, k_mx: MXTensor, vt_mx: MXTensor, scaling: float, mask: Optional[torch.Tensor], causal: bool,
                    p_elem_dtype: dtypes.DType, p_block_size: int = 32, return_probs: bool = False, kv_len: Optional[int] = None):
    """The reference's MX attention (torchmx/layers/mx_llama_attention.py:195-243) in one launch.

    q_mx [b, h, q, 128] and k_mx [b, h_kv, kv, 128] quantized along head_dim, vt_mx [b, h_kv, 128, kv] = V quantized along the
    key axis (the reference's quantize-the-transpose), all contiguous with block size 32; mask: None or additive bf16
    broadcastable to [b, h, q, kv].  Returns the attention output already in the [b, q, h, 128] layout the reference transposes
    to next (bf16) -- plus the MXTensor of P when `return_probs` -- or None when the kernel does not apply (the caller then
    runs the K3 -> K4a -> K3 chain).

    kv_len: None, or the number of keys that exist in K / Vt buffers of a capacity (a multiple of 128) -- a KV cache read in
    place.  Then kv_len may be anything from q_len to the capacity, mask (if any) covers >= kv_len keys, and the result is
    that of the call without kv_len on `ragged_operands(...)` (P then has n = ceil128(kv_len) keys)."""
    if not _FLASH or p_block_size != 32 or p_elem_dtype == dtypes.int8 or q_mx.dim() != 4 or k_mx.dim() != 4 or vt_mx.dim() != 4:
        return None
    b, h, q_len, d = q_mx.shape
    hk, pitch = k_mx.shape[1], k_mx.shape[2]
    ragged = kv_len is not None
    if not ragged:
        kv_len, n = pitch, pitch
        if pitch % 32:
            return None
    else:
        n = -(-kv_len // 128) * 128
        if pitch % 128 or kv_len > pitch:
            return None
    if d != 128 or k_mx.shape != (b, hk, pitch, d) or vt_mx.shape != (b, hk, d, pitch) or h % hk or kv_len < q_len or q_len == 0:
        return None
    if pitch > MAX_FLASH_KV:
        return None
    ops = [_byte_operand(t) for t in (q_mx, k_mx, vt_mx)]
    if any(o is None for o in ops):
        return None
    dev = q_mx._data.device
    a = _C.AttentionArgs()
    if not _set_mask(a, mask, b, h, q_len, kv_len, dev):
        return None
    (a.q_codes, a.q_format, a.q_scales), (a.k_codes, a.k_format, a.k_scales), (a.vt_codes, a.v_format, a.vt_scales) = \
        [(c.data_ptr(), f, s.data_ptr()) for c, f, s in ops]
    a.batch, a.heads, a.kv_heads, a.q_len, a.kv_len, a.head_dim = b, h, hk, q_len, kv_len, d
    a.scaling, a.causal = float(scaling), 1 if causal else 0
    a.kv_pitch = pitch if ragged else 0
    # One query position (decode) with grouped-query heads: the query heads that share a key / value head become the ROWS of one
    # query tile ([b, h, 1, d] is [b, h_kv, groups, d] in memory), so a CTA works on `groups` live rows instead of one and the grid
    # shrinks by that factor.  Same rows, same keys, same arithmetic per row; the mask row is shared by the group.
    grouped = q_len == 1 and h > hk and not causal and (mask is None or mask.shape[1] == 1) and (not ragged or kv_len >= h // hk)
    if grouped:
        a.heads, a.q_len, a.mask_stride_q = hk, h // hk, 0
    a.p_elem = dtypes.ELEM_ID[p_elem_dtype.name]
    a.flags = _quant_flags(p_elem_dtype)
    out = torch.empty((b, q_len, h, d), dtype=torch.bfloat16, device=dev)
    a.out, a.out_batch_stride, a.out_row_stride, a.out_head_stride = out.data_ptr(), out.stride(0), out.stride(1), out.stride(2)
    if grouped:  # element (batch, key head, group row g, channel) of the kernel's view is head (key head * groups + g) of the one token
        a.out_row_stride, a.out_head_stride = out.stride(2), (h // hk) * out.stride(2)
    probs = None
    if return_probs:
        p_codes = _codes_like((b, h, q_len), n, p_elem_dtype, dev)
        p_scales = torch.empty((b, h, q_len, n // 32), dtype=torch.uint8, device=dev)
        a.p_codes, a.p_scales = p_codes.data_ptr(), p_scales.data_ptr()
        probs = MXTensor(p_scales, p_codes, p_elem_dtype, 32, torch.bfloat16)
    if not _C.launch("mxq_flash_attention", a, dev.index, _stream_ptr(q_mx._data)):
        return None
    stats["flash_attention"] += 1
    return (out, probs) if return_probs else out


def ragged_operands(k_mx: MXTensor, vt_mx: MXTensor, kv_len: int, q_len: int, mask: Optional[torch.Tensor], causal: bool):
    """What `flash_attention(..., kv_len=kv_len)` computes, as operands of the call without kv_len (and of the K3 -> K4a -> K3
    chain): (K, Vt, mask') with n = ceil128(kv_len) keys.  K / Vt are contiguous copies of the first n keys of the capacity
    buffers with zero codes at positions >= kv_len, the neutral scale 127 on those keys and on the V blocks wholly past kv_len;
    mask' is the additive bf16 `mask` (or zeros) with -inf on every key >= kv_len and, when `causal`, on every key j > q +
    (kv_len - q_len) -- or None when there is no mask, causal is off and kv_len == n.  O(kv_len) copies."""
    n = -(-kv_len // 128) * 128
    k_codes, k_scales = k_mx._data[:, :, :n].clone(), k_mx._scale_e8m0[:, :, :n].clone()
    vt_codes, vt_scales = vt_mx._data[..., :n].clone(), vt_mx._scale_e8m0[..., :n // 32].clone()
    k_codes[:, :, kv_len:] = 0
    k_scales[:, :, kv_len:] = 127
    vt_codes[..., kv_len:] = 0
    vt_scales[..., -(-kv_len // 32):] = 127
    k_n = MXTensor(k_scales, k_codes, k_mx._elem_dtype, 32, k_mx._orig_dtype)
    vt_n = MXTensor(vt_scales, vt_codes, vt_mx._elem_dtype, 32, vt_mx._orig_dtype)
    if mask is None and not causal and kv_len == n:
        return k_n, vt_n, None
    dev = k_codes.device
    shape = (1, 1, q_len) if mask is None else (*mask.shape[:2], q_len)
    mask_n = torch.full((*shape, n), float("-inf"), dtype=torch.bfloat16, device=dev)
    mask_n[..., :kv_len] = 0 if mask is None else mask[..., :kv_len]
    if causal:
        hidden = torch.ones(q_len, n, dtype=torch.bool, device=dev).triu_(kv_len - q_len + 1)
        mask_n.masked_fill_(hidden, float("-inf"))
    return k_n, vt_n, mask_n
