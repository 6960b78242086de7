"""Host side of K1b (csrc/mxq_act_quant.cu, C entry `mxq_silu_mul_quantize`): `silu_mul_to_mx(gate, up, elem_dtype)` is
`MXTensor.to_mx(F.silu(gate) * up, elem_dtype, 32)` -- the gating of a Llama / Qwen2 MLP block and the activation quantization
on entry to its down projection (reference: torchmx/layers/mx_llama_attention.py:19-59, torchmx/layers/mx_linear.py:63-66) --
in one launch, bit-identical to the three-launch chain.  Returns None when the operands do not qualify (the caller then runs
the chain); there is no CPU path.
"""
from __future__ import annotations

import os
from typing import Optional

import torch

from . import _C, dtypes
from .mx_tensor import MXTensor, _codes_like, _quant_flags, _stream_ptr

stats = {"fused_silu_mul": 0}
_ENABLED = os.environ.get("MXQ_FUSED_SILU_MUL", "1") != "0"


def set_fused_silu_mul(on: bool) -> bool:
    global _ENABLED
    prev, _ENABLED = _ENABLED, bool(on)
    return prev


def _rows_view(t: torch.Tensor):
    """[..., cols] with unit column stride and ONE row stride over all leading dims (size-1 dims are free) -> row stride in
    elements, or None"""
    cols = t.shape[-1]
    if t.stride(-1) != 1 and cols > 1:
        return None
    ld, expect = None, None
    for size, stride in zip(reversed(t.shape[:-1]), reversed(t.stride()[:-1])):
        if size == 1:
            continue
        if ld is None:
            ld, expect = stride, stride * size
        elif stride != expect:
            return None
        else:
            expect *= size
    return cols if ld is None else ld


def silu_mul_to_mx(gate: torch.Tensor, up: torch.Tensor, elem_dtype: dtypes.DType, block_size: int = 32) -> Optional[MXTensor]:
    if (not _ENABLED or block_size != 32 or type(gate) is not torch.Tensor or type(up) is not torch.Tensor or not gate.is_cuda
            or gate.dtype != torch.bfloat16 or up.dtype != torch.bfloat16 or gate.shape != up.shape or gate.dim() < 1 or gate.device != up.device):
        return None
    cols = gate.shape[-1]
    if cols % 32 or gate.numel() == 0:
        return None
    ldg, ldu = _rows_view(gate), _rows_view(up)
    if ldg is None or ldu is None or ldg % 16 or ldu % 16 or gate.data_ptr() % 32 or up.data_ptr() % 32:
        return None
    rows = gate.numel() // cols
    lead = tuple(gate.shape[:-1])
    codes = _codes_like(lead, cols, elem_dtype, gate.device)
    scales = torch.empty(lead + (cols // 32,), dtype=torch.uint8, device=gate.device)
    if not _C.launch("mxq_silu_mul_quantize", gate.data_ptr(), up.data_ptr(), rows, cols, ldg, ldu, dtypes.ELEM_ID[elem_dtype.name],
                     _quant_flags(elem_dtype), codes.data_ptr(), scales.data_ptr(), gate.device.index, _stream_ptr(gate)):
        return None
    stats["fused_silu_mul"] += 1
    return MXTensor(scales, codes, elem_dtype, 32, gate.dtype)
