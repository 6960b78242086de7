"""PackedMXLinear: an MX inference linear whose weight exists ONLY as the dense tensor-core operand stream (SURVEY §8f-3).

The reference keeps one byte per fp6 code and the fp4 pairs in even-high order (torchmx/mx_tensor.py:495-520,
torchmx/utils.py:120-145); `MXInferenceLinear` keeps that layout (its `state_dict` is the reference's) and caches a packed
shadow for the kernels, so a resident fp6 weight costs 1 + 0.75 B per element.  This module drops the reference layout:
`weight_packed` ([N, K*bits/8] uint8: 0.75 B per fp6 element, 0.5 B per fp4 element) + `weight_scale` ([N, K/32] E8M0) are the
only copies in HBM and in the `state_dict`, and `to_mx_linear()` / `unpack_linear_` give the reference layout back bit-for-bit
(`mxq_unpack_operand`).  The forward pass is the one of `MXInferenceLinear` (K1 / fused quantization + K3) on the same operand
bytes, hence bit-identical outputs.  A packed layer has no dequantize fallback: weights that cannot run on the tensor-core
path (int8 elements, in_features % 128 != 0) are left as `MXInferenceLinear` by `pack_linear_`.
"""
from __future__ import annotations

import torch

from .. import dtypes, mx_gemm
from ..config import QLinearConfig
from ..mx_tensor import MXTensor
from .mx_linear import MXInferenceLinear


class PackedMXLinear(torch.nn.Module):
    def __init__(self, in_features: int, out_features: int, qconfig: QLinearConfig, operand_format: int, bias=None, device=None):
        super().__init__()
        self.in_features, self.out_features, self.qconfig, self.operand_format = in_features, out_features, qconfig, operand_format
        bits = mx_gemm._PACKED_BITS.get(operand_format, 8)
        self.register_buffer("weight_packed", torch.empty(out_features, in_features * bits // 8, dtype=torch.uint8, device=device))
        self.register_buffer("weight_scale", torch.empty(out_features, in_features // 32, dtype=torch.uint8, device=device))
        if bias is None:
            self.register_parameter("bias", None)
        else:
            self.bias = bias

    def extra_repr(self) -> str:
        return (f"in_features={self.in_features}, out_features={self.out_features}, bias={self.bias is not None}, "
                f"bytes_per_weight_element={self.weight_packed.shape[1] / self.in_features + 1 / 32:.3f}, qconfig={self.qconfig}")

    @classmethod
    @torch.no_grad()
    def from_mx_linear(cls, lin: MXInferenceLinear, keep_source: bool = False):
        """-> PackedMXLinear, or None when the weight cannot run on the tensor-core path.  Unless `keep_source`, the source
        module's reference-layout weight (and its cached shadow) is released."""
        w = lin.weight
        if not isinstance(w, MXTensor) or lin.qconfig.weights_config.block_size != 32:
            return None
        packed = mx_gemm.pack_weight(w)
        if packed is None:
            return None
        b_e, fmt = packed
        new = cls.__new__(cls)
        torch.nn.Module.__init__(new)
        new.in_features, new.out_features, new.qconfig, new.operand_format = lin.in_features, lin.out_features, lin.qconfig, fmt
        new.register_buffer("weight_packed", b_e if b_e.data_ptr() != w._data.data_ptr() or not keep_source else b_e.clone())
        new.register_buffer("weight_scale", w._scale_e8m0)
        if lin.bias is None:
            new.register_parameter("bias", None)
        else:
            new.bias = lin.bias
        if not keep_source:
            w.__dict__.pop(mx_gemm._SHADOW_ATTR, None)
            lin._parameters.pop("weight", None)
        mx_gemm.mark_static(new)
        return new

    @classmethod
    @torch.no_grad()
    def view_of(cls, stacked: "PackedMXLinear", row0: int, rows: int, bias=None) -> "PackedMXLinear":
        """a layer over rows [row0, row0 + rows) of `stacked`'s operand stream and scales (aliases, nothing is copied): the
        per-projection face of a stacked q/k/v or gate/up weight"""
        new = cls.__new__(cls)
        torch.nn.Module.__init__(new)
        new.in_features, new.out_features, new.qconfig, new.operand_format = stacked.in_features, rows, stacked.qconfig, stacked.operand_format
        new.register_buffer("weight_packed", stacked.weight_packed[row0:row0 + rows])
        new.register_buffer("weight_scale", stacked.weight_scale[row0:row0 + rows])
        if bias is None:
            new.register_parameter("bias", None)
        else:
            new.bias = bias
        mx_gemm.mark_static(new)
        return new

    @torch.no_grad()
    def weight_mx(self) -> MXTensor:
        """the weight in the reference layout (bit-identical to what `MXTensor.to_mx` produced before packing)"""
        elem = self.qconfig.weights_config.elem_dtype
        return MXTensor(self.weight_scale, mx_gemm.unpack_weight(self.weight_packed, self.operand_format, elem), elem, 32, torch.bfloat16)

    @torch.no_grad()
    def to_mx_linear(self) -> MXInferenceLinear:
        new = MXInferenceLinear.__new__(MXInferenceLinear)
        torch.nn.Module.__init__(new)
        new.in_features, new.out_features, new.qconfig = self.in_features, self.out_features, self.qconfig
        new.weight = torch.nn.Parameter(self.weight_mx(), requires_grad=False)
        if self.bias is None:
            new.register_parameter("bias", None)
        else:
            new.bias = self.bias
        return new

    def prepare_input(self, x):
        return MXInferenceLinear.prepare_input(self, x)

    @torch.no_grad()
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        ac = self.qconfig.activations_config
        assert ac.block_size == 32 and ac.elem_dtype in dtypes.SUPPORTED_FP_ELEM_DTYPES + (dtypes.float8_e5m2,), \
            "a packed-only weight needs an FP activation format with block size 32 (no dequantize fallback)"
        if isinstance(x, MXTensor):
            assert x._elem_dtype == ac.elem_dtype and x._block_size == ac.block_size, "activation was quantized with another config"
        return mx_gemm.linear_packed_weight(x, self.weight_packed, self.weight_scale, self.operand_format, self.bias, ac.elem_dtype, owner=self)
