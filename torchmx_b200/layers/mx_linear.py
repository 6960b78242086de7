"""MXInferenceLinear: nn.Linear whose weight is pre-quantized to MX and whose activation is
quantized on every forward (reference: /root/reference/torchmx/layers/mx_linear.py:8-95).

forward = K1 (activation quantize) -> MX matmul (aten.linear / addmm override -> K3 tensor-core
kernel, or the dequantize path when the operands do not qualify).
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from .. import mx_gemm
from ..config import QLinearConfig
from ..mx_tensor import MXTensor


class MXInferenceLinear(torch.nn.Linear):
    def extra_repr(self) -> str:
        return f"{super().extra_repr()}, qconfig={self.qconfig}"

    @classmethod
    @torch.no_grad()
    def from_float(cls, mod: torch.nn.Linear, qconfig: QLinearConfig) -> "MXInferenceLinear":
        """Swap-in constructor (reference: mx_linear.py:21-59): the module skeleton is built on the
        meta device, the weight is quantized once unless it lives on `meta` itself (accelerate
        offload), the bias object is shared with the source module."""
        # Same result as building `cls(in, out, bias=False)` on the meta device and swapping the weight in (the
        # reference's recipe), without running nn.Linear.__init__ / reset_parameters per layer: whole-model
        # quantization is host-bound otherwise (the quantize kernel of a 4096 x 14336 weight takes ~30 us).
        new = cls.__new__(cls)
        torch.nn.Module.__init__(new)
        new.in_features, new.out_features = mod.in_features, mod.out_features
        new.qconfig = qconfig
        w = mod.weight.data
        if w.device.type != "meta":
            wc = qconfig.weights_config
            new.weight = torch.nn.Parameter(MXTensor.to_mx(w, wc.elem_dtype, wc.block_size), requires_grad=False)
            mx_gemm.mark_static(new.weight)
        else:
            new.weight = torch.nn.Parameter(torch.empty(mod.out_features, mod.in_features, device="meta", dtype=w.dtype), requires_grad=False)
        if mod.bias is None:
            new.register_parameter("bias", None)
        else:
            new.bias = mod.bias
        return new

    def _weight_mx(self) -> MXTensor:
        if isinstance(self.weight, MXTensor):  # (a Parameter made from an MXTensor IS that subclass; `.data` would dispatch a detach)
            return self.weight
        w = self.weight.data
        # weights that were on `meta` at conversion time arrive high-precision (often fp32) at call time
        # (reference: mx_linear.py:68-92): quantize on the fly, leave self.weight untouched
        wc = self.qconfig.weights_config
        return MXTensor.to_mx(w.to(torch.bfloat16), wc.elem_dtype, wc.block_size)

    def prepare_input(self, x: torch.Tensor):
        """Quantize an activation that SEVERAL layers with this layer's activation config will consume (q/k/v, gate/up): the
        reference quantizes it once per layer (mx_linear.py:63-66); a block that owns its projections can quantize it once
        and hand the MXTensor to each of them.  Decode-sized inputs are returned as they are -- for those every layer fuses
        the quantization into its GEMM, which is cheaper than a separate launch."""
        ac = self.qconfig.activations_config
        rows = x.numel() // x.shape[-1] if x.dim() else 0
        if isinstance(x, MXTensor) or (mx_gemm._FUSED_ACT and ac.elem_dtype_name == "float8_e4m3" and ac.block_size == 32
                                        and rows <= mx_gemm.FUSED_ACT_MAX_ROWS):
            return x
        return MXTensor.to_mx(x, ac.elem_dtype, ac.block_size)

    @torch.no_grad()
    def forward(self, x: torch.Tensor, _fused=None) -> torch.Tensor:
        """`_fused` (mx_gemm.FusedOutput, internal): set by RowParallelMXLinear -- the launch may add its result into that
        symmetric buffer instead of returning a local tensor."""
        ac = self.qconfig.activations_config
        bias = self.bias
        if torch.compiler.is_compiling():
            # under torch.compile the layer is what the reference's is (mx_linear.py:61-95): quantize, then the aten.linear
            # override on two MXTensors -- ops the tracer knows (custom ops with fake kernels); the direct launches below
            # are host code it cannot see through
            if not isinstance(self.weight, MXTensor) and bias is not None:
                bias = bias.to(torch.bfloat16)
            x_mx = x if isinstance(x, MXTensor) else MXTensor.to_mx(x, ac.elem_dtype, ac.block_size)
            return F.linear(x_mx, self._weight_mx(), bias)
        if isinstance(x, MXTensor):  # already quantized by the owning block (prepare_input)
            assert x._elem_dtype == ac.elem_dtype and x._block_size == ac.block_size, "activation was quantized with another config"
            if not isinstance(self.weight, MXTensor) and bias is not None:
                bias = bias.to(torch.bfloat16)
            w_mx = self._weight_mx()
            out = mx_gemm.contract(torch.ops.aten.linear.default, x, w_mx, (), (bias,), fused=_fused, count_fallback=False)
            return out if out is not None else F.linear(x, w_mx, bias)
        if not isinstance(self.weight, MXTensor) and bias is not None:
            bias = bias.to(torch.bfloat16)
        w_mx = self._weight_mx()
        if ac.elem_dtype_name == "float8_e4m3" and ac.block_size == 32:
            # decode-sized activations: quantization fused into the weight-streaming GEMM (one launch, no code round trip)
            out = mx_gemm.linear_fused_act_quant(x, w_mx, bias, fused=_fused)
            if out is not None:
                return out
        elif ac.block_size == 32 and ac.elem_dtype_name in ("float6_e3m2", "float6_e2m3", "float4_e2m1"):
            # 4 / 6-bit activations: K1 writes the packed operand stream the GEMM reads (no mxq_pack_operand launch in between)
            out = mx_gemm.linear_packed_act_quant(x, w_mx, bias, ac.elem_dtype, fused=_fused)
            if out is not None:
                return out
        x_mx = MXTensor.to_mx(x, ac.elem_dtype, ac.block_size)
        # F.linear(x_mx, w_mx, bias) reaches the same kernel through the dispatcher (aten.t + aten.mm / addmm on MXTensor
        # views, ~50 us of host time per layer); hand the operands to the tensor-core path directly when they qualify
        out = mx_gemm.contract(torch.ops.aten.linear.default, x_mx, w_mx, (), (bias,), fused=_fused, count_fallback=False)
        if out is not None:
            return out
        return F.linear(x_mx, w_mx, bias)
