"""MXInferenceExperts: an MX-quantized mixture-of-experts expert bank.

transformers (5.x) stores the experts of Mixtral, Qwen2-MoE, Qwen3-MoE and OLMoE as two 3-D parameters, gate_up_proj [E, 2I, H]
and down_proj [E, H, I], with SiLU gating and no bias; the reference's quantize_llm_ (written for transformers 4.44, where these were
per-expert nn.Linear modules) quantized all of them.  This module is that quantization for the fused banks.  Its result is defined
as transformers' expert loop (MixtralExperts.forward) with every F.linear an MX matmul: the weight quantized along its contraction
dim with `weights_config`, the activation rows with `activations_config`.

forward takes the grouped path -- K6 route, one grouped GEMM for gate_up, K1b, one grouped GEMM for down, K6 combine
(moe_ops.py, csrc/mxq_moe.cu) -- whenever the kernels cover the configuration; it never reads a device value on the host, so a
decode step can be captured in a CUDA graph.  Everything else runs the loop path: the loop itself on MXTensor operands through the
MX matmul override, which is also the reference the tests compare the grouped path with.
"""
from __future__ import annotations

import os

import torch
import torch.nn.functional as F

from .. import mlp_ops, moe_ops
from ..config import QLinearConfig
from ..mx_tensor import MXTensor

# MXQ_MOE_GROUPED=0 runs every bank on the loop path (the tests' reference for the grouped path)
_GROUPED = os.environ.get("MXQ_MOE_GROUPED", "1") != "0"
_GROUPED_ELEMS = ("float8_e4m3", "float8_e5m2", "float6_e3m2", "float6_e2m3", "float4_e2m1")


def set_grouped(flag: bool) -> bool:
    """switch the grouped path on or off; returns the old value"""
    global _GROUPED
    prev, _GROUPED = _GROUPED, bool(flag)
    return prev


def _bank_classes() -> tuple:
    """the transformers expert banks quantize_llm_ swaps (all four share MixtralExperts' layout and forward)"""
    from transformers.models.mixtral.modeling_mixtral import MixtralExperts
    from transformers.models.olmoe.modeling_olmoe import OlmoeExperts
    from transformers.models.qwen2_moe.modeling_qwen2_moe import Qwen2MoeExperts
    from transformers.models.qwen3_moe.modeling_qwen3_moe import Qwen3MoeExperts
    return (MixtralExperts, Qwen2MoeExperts, Qwen3MoeExperts, OlmoeExperts)


def is_expert_bank(mod: torch.nn.Module) -> bool:
    """one of the four bank classes with the layout this module reproduces: 3-D gate_up_proj [E, 2I, H] / down_proj [E, H, I],
    SiLU gating, no bias, not transposed"""
    from transformers.activations import SiLUActivation
    if type(mod) not in _bank_classes():
        return False
    gu, dn = getattr(mod, "gate_up_proj", None), getattr(mod, "down_proj", None)
    if not isinstance(gu, torch.Tensor) or not isinstance(dn, torch.Tensor) or gu.dim() != 3 or dn.dim() != 3:
        return False
    E, two_i, H = gu.shape
    return (two_i % 2 == 0 and tuple(dn.shape) == (E, H, two_i // 2) and isinstance(getattr(mod, "act_fn", None), (torch.nn.SiLU, SiLUActivation))
            and not getattr(mod, "has_bias", False) and not getattr(mod, "is_transposed", False) and getattr(mod, "has_gate", True))


def _expert(w: MXTensor, e: int) -> MXTensor:
    """expert e of an MXTensor bank [E, rows, K] as a 2-D MXTensor weight"""
    return MXTensor(w._scale_e8m0[e], w._data[e], w._elem_dtype, w._block_size, w._orig_dtype)


class MXInferenceExperts(torch.nn.Module):
    def extra_repr(self) -> str:
        return f"num_experts={self.num_experts}, hidden_dim={self.hidden_dim}, intermediate_dim={self.intermediate_dim}, qconfig={self.qconfig}"

    @classmethod
    @torch.no_grad()
    def from_float(cls, bank: torch.nn.Module, qconfig: QLinearConfig) -> "MXInferenceExperts":
        """Swap-in constructor: both banks quantized once along their contraction dim (gate_up along H, down along I), unless
        they live on `meta` (then they stay meta and are quantized at call time, as MXInferenceLinear does)."""
        assert is_expert_bank(bank), f"{type(bank).__name__} is not an expert bank of the supported layout"
        new = cls.__new__(cls)
        torch.nn.Module.__init__(new)
        new.num_experts, new.intermediate_dim, new.hidden_dim = bank.gate_up_proj.shape[0], bank.gate_up_proj.shape[1] // 2, bank.gate_up_proj.shape[2]
        new.qconfig = qconfig
        wc = qconfig.weights_config
        for name in ("gate_up_proj", "down_proj"):
            w = getattr(bank, name).data
            if w.device.type != "meta":
                setattr(new, name, torch.nn.Parameter(MXTensor.to_mx(w, wc.elem_dtype, wc.block_size), requires_grad=False))
            else:
                setattr(new, name, torch.nn.Parameter(torch.empty(w.shape, device="meta", dtype=w.dtype), requires_grad=False))
        return new

    def _bank(self, name: str) -> MXTensor:
        w = getattr(self, name)
        if isinstance(w, MXTensor):
            return w
        wc = self.qconfig.weights_config  # banks that were on `meta` at conversion time: quantize on the fly
        return MXTensor.to_mx(w.data.to(torch.bfloat16), wc.elem_dtype, wc.block_size)

    def _grouped_ok(self, x: torch.Tensor, top_k_index: torch.Tensor, top_k_weights: torch.Tensor) -> bool:
        wc, ac = self.qconfig.weights_config, self.qconfig.activations_config
        return (_GROUPED and not torch.compiler.is_compiling() and wc.block_size == 32 and ac.block_size == 32
                and wc.elem_dtype_name in _GROUPED_ELEMS and ac.elem_dtype_name in _GROUPED_ELEMS
                and self.hidden_dim % 128 == 0 and self.intermediate_dim % 128 == 0 and self.num_experts <= 256
                and type(x) is torch.Tensor and x.is_cuda and x.dtype == torch.bfloat16 and x.dim() == 2 and x.shape[0] <= 16384
                and top_k_index.dtype == torch.int64 and top_k_index.dim() == 2 and top_k_index.shape[0] == x.shape[0]
                and top_k_index.shape[1] <= 8 and top_k_index.is_cuda
                and top_k_weights.dtype in (torch.float32, torch.bfloat16) and top_k_weights.shape == top_k_index.shape)

    @torch.no_grad()
    def forward(self, hidden_states: torch.Tensor, top_k_index: torch.Tensor, top_k_weights: torch.Tensor) -> torch.Tensor:
        if hidden_states.shape[0] == 0:
            return torch.zeros_like(hidden_states)
        if self._grouped_ok(hidden_states, top_k_index, top_k_weights):
            return self._grouped(hidden_states.contiguous(), top_k_index, top_k_weights)
        return self._loop(hidden_states, top_k_index, top_k_weights)

    def _grouped(self, x: torch.Tensor, top_k_index: torch.Tensor, top_k_weights: torch.Tensor) -> torch.Tensor:
        act = self.qconfig.activations_config.elem_dtype
        E, I = self.num_experts, self.intermediate_dim
        offsets, row_of_slot, _, codes, scales = moe_ops.route(top_k_index, E, x, act)
        gu = moe_ops.grouped_linear(codes, scales, act, self._bank("gate_up_proj"), offsets)
        h = mlp_ops.silu_mul_to_mx(gu[:, :I], gu[:, I:], act)
        if h is None:  # K1b switched off: the chain it fuses
            h = MXTensor.to_mx(F.silu(gu[:, :I]) * gu[:, I:], act, 32)
        y = moe_ops.grouped_linear(h._data, h._scale_e8m0, act, self._bank("down_proj"), offsets)
        moe_ops.stats["grouped_experts"] += 1
        return moe_ops.combine(y, top_k_index, top_k_weights, row_of_slot, E)

    def _loop(self, hidden_states: torch.Tensor, top_k_index: torch.Tensor, top_k_weights: torch.Tensor) -> torch.Tensor:
        """transformers' MixtralExperts.forward with MX operands"""
        ac = self.qconfig.activations_config
        gate_up, down = self._bank("gate_up_proj"), self._bank("down_proj")
        final_hidden_states = torch.zeros_like(hidden_states)
        expert_mask = F.one_hot(top_k_index, num_classes=self.num_experts).permute(2, 1, 0)
        expert_hit = torch.greater(expert_mask.sum(dim=(-1, -2)), 0).nonzero()
        for expert_idx in expert_hit:
            e = int(expert_idx[0])
            top_k_pos, token_idx = torch.where(expert_mask[e])
            x = MXTensor.to_mx(hidden_states[token_idx], ac.elem_dtype, ac.block_size)
            gate, up = F.linear(x, _expert(gate_up, e)).chunk(2, dim=-1)
            h = MXTensor.to_mx(F.silu(gate) * up, ac.elem_dtype, ac.block_size)
            h = F.linear(h, _expert(down, e))
            h = h * top_k_weights[token_idx, top_k_pos, None]
            final_hidden_states.index_add_(0, token_idx, h.to(final_hidden_states.dtype))
        return final_hidden_states
