"""Model surgery: swap nn.Linear for MXInferenceLinear in place
(reference: /root/reference/torchmx/quant_api.py:161-215).

`quantize_llm_` (reference: quant_api.py:218-271) swaps the attention and MLP blocks of Llama / Qwen2 models for their MX
versions (`layers/mx_llama_attention.py`, written against the installed transformers' attention interface) and then every
remaining nn.Linear.  The torchao tensor-subclass inserter of the reference (quant_api.py:96-147) depends on torchao and is
not provided.
"""
from __future__ import annotations

from pprint import pformat
from typing import Callable, Optional

import torch

from .config import QAttentionConfig, QLinearConfig
from .layers.mx_linear import MXInferenceLinear
from .mx_tensor import small_scale_arena
from .utils import get_logger

logger = get_logger(__name__)


def _swap_children(model: torch.nn.Module, replacement_fn: Callable, filter_fn: Callable, on_visit: Optional[Callable] = None,
                   prefix: str = "") -> None:
    """Depth-first walk; a matching child is replaced and NOT descended into
    (reference: quant_api.py:161-185)."""
    for name, child in list(model.named_children()):
        fqn = f"{prefix}.{name}" if prefix else name
        if on_visit:
            on_visit(fqn)
        if filter_fn(child, fqn):
            setattr(model, name, replacement_fn(child))
        else:
            _swap_children(child, replacement_fn, filter_fn, on_visit, fqn)


def quantize_linear_(model: torch.nn.Module, qconfig: QLinearConfig, layer_filter: Optional[Callable[[str], bool]] = None) -> None:
    """Replace every module whose type is exactly `torch.nn.Linear` (lm_head included) with
    `MXInferenceLinear.from_float(mod, qconfig)`, in place (reference: quant_api.py:188-215).
    Mixture-of-experts banks stored as 3-D parameters are not nn.Linear; `quantize_llm_` quantizes those.

    `layer_filter(fqn) -> bool` is a B200-side extension used by the layer-sharded multi-GPU
    driver: only layers whose qualified name passes the filter are quantized by this rank.
    """
    logger.info("Quantizing the model by swapping nn.Linear with TorchMX's MXInferenceLinear")
    logger.warning("This method only replaces/quantizes the linear layers. Use this as an approximation as we do not "
                   "quantize QKV and other stuff. Use this only when a specific attention layer is not implemented.")
    logger.info(f"Quantizing Linear layers with config:\n{pformat(qconfig)}\n")
    try:
        from tqdm import tqdm
        bar = tqdm(desc="Quantizing linear layers in model...")
        on_visit = lambda fqn: bar.update(1)  # noqa: E731
    except Exception:  # tqdm is optional
        bar, on_visit = None, None
    with small_scale_arena():  # (sub-MiB scale tensors share large-pool chunks: no 2 MiB cudaMalloc per handful of layers)
        _swap_children(
            model,
            replacement_fn=lambda mod: MXInferenceLinear.from_float(mod, qconfig),
            filter_fn=lambda mod, fqn: type(mod) is torch.nn.Linear and (layer_filter is None or layer_filter(fqn)),
            on_visit=on_visit,
        )
    if bar is not None:
        bar.close()


class FusedRMSNorm(torch.nn.Module):
    """Drop-in for the transformers `LlamaRMSNorm` / `Qwen2RMSNorm` module: same parameters, ONE launch (K5a, `glue_ops.rmsnorm`:
    fp32 statistics, the module's bf16 roundings) instead of the six elementwise / reduction launches of the eager module.
    When the only consumers of the output are MX linears of one activation config (`to_mx`, set by `quantize_llm_` for the two
    norms of a decoder layer whose attention and MLP blocks are MX blocks) the same launch also quantizes: the module returns the
    MXTensor the layers would have produced from its bf16 output (`MXTensor.to_mx` of it, bit for bit) and the bf16 tensor is never
    written.  That holds at decode sizes too: a decode GEMM that quantizes its activation itself does so once per CTA (every CTA
    needs the whole activation), which caps it at ~6 T weight elements/s; fed codes it streams 4 / 6-bit weights 15-30 % faster
    (profiles/r2_decode_gemm_cold.txt).
    Not part of the reference; `quantize_llm_(..., fuse_rmsnorm=True)` opts in."""

    def __init__(self, weight: torch.nn.Parameter, eps: float, to_mx=None):
        super().__init__()
        self.weight, self.variance_epsilon, self.to_mx = weight, eps, to_mx

    def forward(self, hidden_states: torch.Tensor) -> torch.Tensor:
        from . import glue_ops
        if not torch.compiler.is_compiling():
            quant = self.to_mx is not None
            r = glue_ops.rmsnorm(hidden_states, self.weight, self.variance_epsilon, to_mx=self.to_mx if quant else None, want_y=not quant)
            if r is not None:
                return r[1] if quant else r[0]
        return torch.nn.functional.rms_norm(hidden_states, (hidden_states.shape[-1],), self.weight, self.variance_epsilon)

    def extra_repr(self) -> str:
        return f"{tuple(self.weight.shape)}, eps={self.variance_epsilon}" + (f", to_mx={self.to_mx.name}" if self.to_mx is not None else "")


def _fuse_norms_(model: torch.nn.Module) -> None:
    """every Llama / Qwen2 RMSNorm -> FusedRMSNorm; the two norms of a decoder layer whose consumers are MX blocks quantize too"""
    from .layers.mx_llama_attention import _MXAttentionMixin, _MXMLPMixin
    is_norm = lambda m: type(m).__name__ in ("LlamaRMSNorm", "Qwen2RMSNorm")  # noqa: E731

    def act_dtype(qc):
        ac = qc.activations_config
        return ac.elem_dtype if ac.block_size == 32 else None

    for layer in model.modules():
        for norm_name, consumer_name, mixin in (("input_layernorm", "self_attn", _MXAttentionMixin), ("post_attention_layernorm", "mlp", _MXMLPMixin)):
            norm, consumer = getattr(layer, norm_name, None), getattr(layer, consumer_name, None)
            if norm is None or not is_norm(norm) or not isinstance(consumer, mixin):
                continue
            qc = consumer.qconfig.projection_config if mixin is _MXAttentionMixin else consumer.qconfig
            setattr(layer, norm_name, FusedRMSNorm(norm.weight, norm.variance_epsilon, to_mx=act_dtype(qc)))
    _swap_children(model, replacement_fn=lambda mod: FusedRMSNorm(mod.weight, mod.variance_epsilon), filter_fn=lambda mod, fqn: is_norm(mod))


def quantize_llm_(model: torch.nn.Module, qattention_config: QAttentionConfig, qmlp_config: QLinearConfig, fuse_rmsnorm: bool = False) -> None:
    """Quantize an LLM in place: every Llama / Qwen2 attention block becomes its MX version with `qattention_config`
    (projections as MXInferenceLinear; Q / K / V / attention-weights quantization when all four configs are given), every
    MLP block its MX version with `qmlp_config`, every mixture-of-experts expert bank of transformers' Mixtral / Qwen2-MoE /
    Qwen3-MoE / OLMoE models (3-D gate_up_proj / down_proj parameters) an `MXInferenceExperts` with `qmlp_config`, and whatever
    nn.Linear is left (lm_head, shared experts) an MXInferenceLinear with `qmlp_config` (reference: quant_api.py:218-271; at the
    transformers version the reference targets the experts were per-expert nn.Linear modules).  The routers stay as they are."""
    from .layers.mx_experts import MXInferenceExperts, is_expert_bank
    from .layers.mx_llama_attention import ATTENTION_LAYERS, MLP_LAYERS
    logger.info("Quantizing the model by swapping the Attention and MLP layers")
    logger.info(f"Attention Layer Quantization config:\n{pformat(qattention_config)}\n")
    logger.info(f"MLP Layer Quantization config:\n{pformat(qmlp_config)}\n")
    table = dict(ATTENTION_LAYERS)
    table.update(MLP_LAYERS)

    def replace(mod):
        cls = table[type(mod)]
        return cls.from_float(mod, qattention_config if type(mod) in ATTENTION_LAYERS else qmlp_config)

    with small_scale_arena():
        _swap_children(model, replacement_fn=replace, filter_fn=lambda mod, fqn: type(mod) in table)
        _swap_children(model, replacement_fn=lambda mod: MXInferenceExperts.from_float(mod, qmlp_config), filter_fn=lambda mod, fqn: is_expert_bank(mod))
    quantize_linear_(model, qmlp_config)
    if fuse_rmsnorm:
        _fuse_norms_(model)


def pack_linear_(model: torch.nn.Module) -> int:
    """Drop the reference storage layout of every `MXInferenceLinear` weight that can run on the tensor cores: the layer becomes a
    `PackedMXLinear` whose only copy of the weight is the dense 4 / 6-bit operand stream (0.5 / 0.75 B per element + scales;
    SURVEY §8f-3).  Same outputs bit for bit, smaller HBM footprint and `state_dict`.  Returns the number of layers packed;
    layers that need the dequantize path (int8 elements, in_features % 128 != 0, meta weights) are left alone."""
    from .layers.mx_llama_attention import pack_stacked_
    from .layers.packed_linear import PackedMXLinear
    n = 0
    for blk in list(model.modules()):  # blocks that own stacked q/k/v or gate/up weights: pack the stacked stream, alias the parts
        if "_qkv" in blk.__dict__ or "_gate_up" in blk.__dict__:
            n += pack_stacked_(blk)

    def replace(mod):
        nonlocal n
        new = PackedMXLinear.from_mx_linear(mod)
        if new is None:
            return mod
        n += 1
        return new

    _swap_children(model, replacement_fn=replace, filter_fn=lambda mod, fqn: type(mod) is MXInferenceLinear)
    return n


def unpack_linear_(model: torch.nn.Module) -> int:
    """The inverse of `pack_linear_`: every `PackedMXLinear` becomes an `MXInferenceLinear` again whose MXTensor weight (and
    therefore `state_dict`) is bit-identical to the reference layout it was packed from."""
    from .layers.packed_linear import PackedMXLinear
    n = 0

    def replace(mod):
        nonlocal n
        n += 1
        return mod.to_mx_linear()

    _swap_children(model, replacement_fn=replace, filter_fn=lambda mod, fqn: type(mod) is PackedMXLinear)
    for blk in model.modules():  # stacked q/k/v / gate/up streams the blocks still hold: their parts are separate layers again
        for attr in ("_qkv", "_gate_up"):
            if type(blk.__dict__.get(attr)) is PackedMXLinear:
                object.__setattr__(blk, attr, None)
    return n
