"""MX inference versions of the Llama (and Qwen2) attention / MLP blocks for `quantize_llm_`
(reference: /root/reference/torchmx/layers/mx_llama_attention.py:19-262, mx_qwen2_attention.py), written against the
attention interface of the installed transformers (5.x: `forward(hidden_states, position_embeddings, attention_mask,
past_key_values, **kwargs) -> (attn_output, attn_weights)`), not the 4.44 internals the reference subclasses.

* the four projections (and the three MLP linears) become `MXInferenceLinear` (K1 + K3, or the fused decode kernel);
* with a full `QAttentionConfig` (query / key / value / attention-weights configs) the attention itself runs on MX operands
  exactly as the reference spells it out (:195-243): Q and K are quantized along head_dim, V along the key/value sequence
  (quantize the transpose, transpose back), scores = Q_mx @ K_mx^T * scaling (+ mask), softmax in fp32, P quantized along
  the key/value sequence, out = P_mx @ V_mx -- both contractions reach the tcgen05 block-scaled bmm when the blocked
  extents are multiples of 128 (otherwise the dequantize path, like the reference), and everything between them is one
  kernel (`attention_ops.softmax_to_mx`, K4a) when the key/value length is a multiple of 32;
* without it the module keeps the model's configured attention function (sdpa / flash / eager) on the rotated bf16 Q, K, V.
With HF's caches the KV cache stays in high precision (reference :186-187) and, with a full `QAttentionConfig`, the whole cache is
quantized again at every forward.  With an `MXStaticCache` (torchmx_b200/kv_cache.py) and a full `QAttentionConfig` the cache holds
the MX codes themselves: one launch (K5e) rotates, quantizes Q and appends only the new tokens' blocks, and the attention reads the
cache in place -- the same codes, so the same logits as with a bf16 StaticCache.  An `MXDynamicCache` works the same way with a
cache that grows with the sequence: the attention reads its first L positions in place, at any length L.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch
from torch import nn

from .. import attention_ops, glue_ops, mlp_ops, mx_gemm
from ..config import QAttentionConfig, QLinearConfig
from ..kv_cache import MXDynamicCache, MXStaticCache
from ..mx_tensor import MXTensor
from .mx_linear import MXInferenceLinear


# MXQ_FUSE_PROJECTIONS=0 keeps one launch per projection (q, k, v / gate, up) in the MX attention and MLP blocks
FUSE_PROJECTIONS = os.environ.get("MXQ_FUSE_PROJECTIONS", "1") != "0"


def _swap_linears(dst: nn.Module, src: nn.Module, names, qconfig: QLinearConfig) -> None:
    for n in names:
        setattr(dst, n, MXInferenceLinear.from_float(getattr(src, n), qconfig))


def _shell_like(cls, mod: nn.Module, skip=()) -> nn.Module:
    """An instance of `cls` that shares every attribute / submodule of `mod` except the ones in `skip` -- the same result as
    the reference's 'construct on meta, then overwrite the projections', without re-running the HF constructor."""
    new = cls.__new__(cls)
    nn.Module.__init__(new)
    for k, v in mod.__dict__.items():
        if k in ("_modules", "_parameters", "_buffers"):
            continue
        new.__dict__[k] = v
    for k, v in mod._parameters.items():
        new._parameters[k] = v
    for k, v in mod._buffers.items():
        new._buffers[k] = v
    for k, v in mod._modules.items():
        if k not in skip:
            new._modules[k] = v
    return new


def _fuse_linears(mods) -> Optional[MXInferenceLinear]:
    """Several MXInferenceLinear layers that read the SAME activation (q/k/v, gate/up) as one layer with their weights stacked
    along the output dim: one launch instead of len(mods), and under-filled projections (k / v: 1024 outputs) ride along with
    the large one.  The stacked codes / scales become the storage and each source layer's weight is re-pointed at its row slice
    of them, so nothing is held twice and every layer's `state_dict` entry is unchanged.  Output columns are computed exactly
    as by the separate layers (a row of the weight never meets another row).  None when the layers cannot be stacked."""
    ws = [m.weight for m in mods]
    w0 = ws[0]
    if not all(isinstance(w, MXTensor) and w._data.dim() == 2 and w._block_dim == 1 and w._padding == 0 and w._data.is_cuda
               and w._elem_dtype == w0._elem_dtype and w._block_size == w0._block_size and w.shape[1] == w0.shape[1]
               and w._data.is_contiguous() and w._scale_e8m0.is_contiguous() and w._data.device == w0._data.device for w in ws):
        return None
    if any(m.qconfig != mods[0].qconfig for m in mods) or len({m.bias is None for m in mods}) != 1:
        return None
    codes = torch.cat([w._data for w in ws], 0)
    scales = torch.cat([w._scale_e8m0 for w in ws], 0)
    fused = MXInferenceLinear.__new__(MXInferenceLinear)
    nn.Module.__init__(fused)
    fused.in_features, fused.out_features, fused.qconfig = mods[0].in_features, codes.shape[0], mods[0].qconfig
    fused.weight = nn.Parameter(MXTensor(scales, codes, w0._elem_dtype, w0._block_size, w0._orig_dtype), requires_grad=False)
    if mods[0].bias is None:
        fused.register_parameter("bias", None)
    else:
        if any(m.bias.dtype != torch.bfloat16 or m.bias.device != codes.device for m in mods):
            return None
        fused.bias = nn.Parameter(torch.cat([m.bias.data for m in mods], 0), requires_grad=False)
    row = 0
    for m, w in zip(mods, ws):  # re-point the source layers at their slice of the stacked storage (weights and biases alike)
        n = w.shape[0]
        m.weight = nn.Parameter(MXTensor(scales[row:row + n], codes[row:row + n], w._elem_dtype, w._block_size, w._orig_dtype), requires_grad=False)
        if fused.bias is not None:
            m.bias = nn.Parameter(fused.bias.data[row:row + n], requires_grad=False)
        mx_gemm.mark_static(m.weight)
        row += n
    mx_gemm.mark_static(fused.weight)
    fused._split = [w.shape[0] for w in ws]
    return fused


def _stacked_from_float(srcs, qconfig: QLinearConfig):
    """What `MXInferenceLinear.from_float` on every module of `srcs` followed by `_fuse_linears` gives -- (stacked layer, [per-module
    layers whose weights are row slices of its storage]) -- with every weight quantized STRAIGHT into its rows of the stacked codes /
    scales: no per-projection tensors, no concatenation (and, across the layers of a model, the stacked gate/up codes are exactly
    the size of a bf16 projection weight being released, so the caching allocator serves them without going to the driver).  Same
    kernel per projection, same bytes.  None when the modules do not qualify (the caller converts them one by one)."""
    from ..mx_tensor import _codes_like, _empty_scales, _quantize_into
    wc = qconfig.weights_config
    ws = [getattr(m, "weight", None) for m in srcs]
    w0 = ws[0]
    if not all(type(m) is nn.Linear and isinstance(w, torch.Tensor) and not isinstance(w, MXTensor) and w.is_cuda and w.dtype == torch.bfloat16 and w.dim() == 2
               and w.is_contiguous() and w.shape[1] == w0.shape[1] and w.device == w0.device for m, w in zip(srcs, ws)):
        return None
    K, bs, elem = w0.shape[1], wc.block_size, wc.elem_dtype
    if K % bs or (elem.name == "float4_e2m1" and K % 2) or len({m.bias is None for m in srcs}) != 1:
        return None
    if srcs[0].bias is not None and any(m.bias.dtype != torch.bfloat16 or m.bias.device != w0.device for m in srcs):
        return None
    rows = [w.shape[0] for w in ws]
    codes = _codes_like((sum(rows),), K, elem, w0.device)
    scales = _empty_scales((sum(rows), K // bs), w0.device)
    layers, row = [], 0
    bias_all = torch.cat([m.bias.data for m in srcs], 0) if srcs[0].bias is not None else None
    for m, w, n in zip(srcs, ws, rows):
        _quantize_into(w.data, elem, bs, codes[row:row + n], scales[row:row + n])
        lin = MXInferenceLinear.__new__(MXInferenceLinear)
        nn.Module.__init__(lin)
        lin.in_features, lin.out_features, lin.qconfig = m.in_features, m.out_features, qconfig
        lin.weight = nn.Parameter(MXTensor(scales[row:row + n], codes[row:row + n], elem, bs, torch.bfloat16), requires_grad=False)
        mx_gemm.mark_static(lin.weight)
        if bias_all is None:
            lin.register_parameter("bias", None)
        else:
            lin.bias = nn.Parameter(bias_all[row:row + n], requires_grad=False)
        layers.append(lin)
        row += n
    fused = MXInferenceLinear.__new__(MXInferenceLinear)
    nn.Module.__init__(fused)
    fused.in_features, fused.out_features, fused.qconfig = srcs[0].in_features, sum(rows), qconfig
    fused.weight = nn.Parameter(MXTensor(scales, codes, elem, bs, torch.bfloat16), requires_grad=False)
    mx_gemm.mark_static(fused.weight)
    if bias_all is None:
        fused.register_parameter("bias", None)
    else:
        fused.bias = nn.Parameter(bias_all, requires_grad=False)
    fused._split = rows
    return fused, layers


GROUPED_DECODE_SDPA = os.environ.get("MXQ_GROUPED_DECODE_SDPA", "1") != "0"  # decode under sdpa: no repeat_kv copies (see forward)
# q/k/v as ONE launch on the row-stacked weights at every size.  Round 1 stacked only decode-sized activations: the column slices
# of a stacked output made every following elementwise kernel and copy strided (prefill 27.1 -> 29.3 ms).  Since K5b (rotary)
# reads the projection outputs in place through their strides, stacking wins at prefill too: Llama-8B 22.4 -> 21.2 ms (with MX
# attention 25.1 -> 24.7 ms).  MXQ_STACKED_MAX_ROWS caps the activation rows it applies to.
STACKED_MAX_ROWS = int(os.environ.get("MXQ_STACKED_MAX_ROWS", 1 << 30))


# gate/up feed K1b, which reads the two column slices in place: no strided follow-up kernels, so the MLP stacks at every size
# (Llama-8B prefill 27.0 -> 26.4 ms)
MLP_STACKED_MAX_ROWS = int(os.environ.get("MXQ_MLP_STACKED_MAX_ROWS", 1 << 30))


def _weight_rows(m):
    """(device, address of row 0, row pitch in bytes, rows) of a layer's resident weight codes: the reference-layout codes of
    an MXInferenceLinear or the packed operand stream of a PackedMXLinear; None for anything else"""
    from .packed_linear import PackedMXLinear
    if type(m) is MXInferenceLinear and isinstance(getattr(m, "weight", None), MXTensor):
        d = m.weight._data
    elif type(m) is PackedMXLinear:
        d = m.weight_packed
    else:
        return None
    return d.device, d.data_ptr(), d.stride(0) * d.element_size(), d.shape[0]


def _fused_still_valid(fused, mods, x: torch.Tensor, max_rows: int = 0) -> bool:
    """the stacked layer is used for decode-sized activations, and only while the source layers still alias it (a later
    .to(device) / weight swap re-materialises them separately)"""
    if fused is None:
        return False
    fw = _weight_rows(fused)
    if fw is None or fw[0] != x.device or x.numel() > (max_rows or STACKED_MAX_ROWS) * x.shape[-1]:
        return False
    row = 0
    for m, n in zip(mods, fused._split):
        w = _weight_rows(m)  # (same class as the stacked layer: both reference layout, or both packed by pack_linear_)
        if w is None or type(m) is not type(fused) or w[1] != fw[1] + row * fw[2] or w[3] != n:
            return False
        if (m.bias is None) != (fused.bias is None) or (m.bias is not None and m.bias.data_ptr() != fused.bias.data_ptr() + row * fused.bias.element_size()):
            return False
        row += n
    return True


def pack_stacked_(block: nn.Module) -> int:
    """`pack_linear_` support: a block that owns a stacked projection (`_qkv` / `_gate_up`) gets the STACKED weight packed once
    and its per-projection layers replaced by PackedMXLinear views of row slices of that stream, so the dense 4 / 6-bit form is
    the only resident copy (no reference-layout codes left behind in the stacked layer).  Returns the number of layers packed."""
    from .packed_linear import PackedMXLinear
    n = 0
    for attr, names in (("_qkv", ("q_proj", "k_proj", "v_proj")), ("_gate_up", ("gate_proj", "up_proj"))):
        fused = block.__dict__.get(attr)
        if fused is None or type(fused) is not MXInferenceLinear or not all(hasattr(block, k) for k in names):
            continue
        mods = [getattr(block, k) for k in names]
        if not all(type(m) is MXInferenceLinear for m in mods) or not _fused_still_valid(fused, mods, fused.weight._data.new_empty(0, fused.in_features)):
            continue
        packed = PackedMXLinear.from_mx_linear(fused)
        if packed is None:
            continue
        packed._split = list(fused._split)
        row = 0
        for k, m, rows in zip(names, mods, packed._split):
            view = PackedMXLinear.view_of(packed, row, rows, None if m.bias is None else m.bias)
            m._parameters.pop("weight", None)
            setattr(block, k, view)
            row += rows
            n += 1
        object.__setattr__(block, attr, packed)
    return n


def _repeat_heads(t: MXTensor, n_rep: int) -> MXTensor:
    """`repeat_kv` (transformers) on an MXTensor [batch, kv_heads, rows, cols]: each head n_rep times, codes and scales copied"""
    if n_rep == 1:
        return t

    def rep(x):
        b, h, r, c = x.shape
        return x[:, :, None].expand(b, h, n_rep, r, c).reshape(b, h * n_rep, r, c)

    return MXTensor(rep(t._scale_e8m0), rep(t._data), t._elem_dtype, t._block_size, t._orig_dtype, t._padding, t._block_dim)


_mask_cache = (None, None)  # (weakref to the boolean mask tensor, its additive form): one conversion per forward, not per layer


_mask_cache_layer = None  # layer index of the block that filled the cache while a CUDA graph was being captured


def _additive_mask(mask: torch.Tensor, dtype: torch.dtype, layer_idx: Optional[int] = None) -> torch.Tensor:
    """One conversion per forward, not per layer.  Outside graph capture the entry is keyed by the mask object and its version.
    A tensor made WHILE a graph is captured lives in that graph's memory pool and must not be handed out after the capture: during
    capture an entry is therefore only reused by blocks with a HIGHER layer index than the one that made it (the later layers of
    the same forward pass); the first block of the next pass makes a new one."""
    global _mask_cache, _mask_cache_layer
    import weakref
    capturing = torch.cuda.is_current_stream_capturing()
    ref, add = _mask_cache
    if ref is not None and ref[0]() is mask and ref[1] == mask._version and add.dtype == dtype:
        if not capturing and _mask_cache_layer is None:
            return add
        if capturing and _mask_cache_layer is not None and layer_idx is not None and layer_idx > _mask_cache_layer:
            return add
    # finfo.min, not -inf (what transformers' eager mask and the reference's 4.44 causal mask use): a query row that may attend
    # to nothing -- left padding under the sdpa mask interface -- then softmaxes to a uniform row instead of NaN, and NaN would
    # spread to every token of the batch through the next layer's K / V
    add = torch.zeros_like(mask, dtype=dtype).masked_fill_(~mask, torch.finfo(dtype).min)
    if not capturing:
        _mask_cache, _mask_cache_layer = ((weakref.ref(mask), mask._version), add), None
    elif layer_idx is not None:
        _mask_cache, _mask_cache_layer = ((weakref.ref(mask), mask._version), add), layer_idx
    return add


class _MXMLPMixin:
    @classmethod
    @torch.no_grad()
    def from_float(cls, mod: nn.Module, qconfig: QLinearConfig):
        assert isinstance(mod, cls.__mro__[2]), f"mod must be an instance of {cls.__mro__[2].__name__}, but got {type(mod)}"
        new = _shell_like(cls, mod, skip=("gate_proj", "up_proj", "down_proj"))
        new.qconfig = qconfig
        stacked = _stacked_from_float([mod.gate_proj, mod.up_proj], qconfig) if FUSE_PROJECTIONS else None
        if stacked is not None:
            new.gate_proj, new.up_proj = stacked[1]
            _swap_linears(new, mod, ("down_proj",), qconfig)
            object.__setattr__(new, "_gate_up", stacked[0])
            return new
        _swap_linears(new, mod, ("gate_proj", "up_proj", "down_proj"), qconfig)
        object.__setattr__(new, "_gate_up", _fuse_linears([new.gate_proj, new.up_proj]) if FUSE_PROJECTIONS else None)
        return new

    def _gated(self, gate, up):
        """act_fn(gate) * up, handed to down_proj -- for SiLU as the already quantized MXTensor (K1b: gating + quantization in one
        launch, bit-identical to silu, mul and K1), otherwise as the bf16 product"""
        if type(self.act_fn).__name__ in ("SiLU", "SiLUActivation") and isinstance(self.down_proj, MXInferenceLinear):
            ac = self.down_proj.qconfig.activations_config
            h = mlp_ops.silu_mul_to_mx(gate, up, ac.elem_dtype, ac.block_size)
            if h is not None:
                return h
        return self.act_fn(gate) * up

    def forward(self, x):
        fused = self.__dict__.get("_gate_up")
        if _fused_still_valid(fused, (self.gate_proj, self.up_proj), x, MLP_STACKED_MAX_ROWS):
            gate, up = fused(x).split(fused._split, dim=-1)  # one launch for both projections
        else:
            x_in = self.gate_proj.prepare_input(x)  # gate and up read the same activation: quantize it once
            gate, up = self.gate_proj(x_in), self.up_proj(x_in)
        return self.down_proj(self._gated(gate, up))


class _MXAttentionMixin:
    @classmethod
    @torch.no_grad()
    def from_float(cls, mod: nn.Module, qconfig: QAttentionConfig):
        assert isinstance(mod, cls.__mro__[2]), f"mod must be an instance of {cls.__mro__[2].__name__}, but got {type(mod)}"
        new = _shell_like(cls, mod, skip=("q_proj", "k_proj", "v_proj", "o_proj"))
        new.qconfig = qconfig
        stacked = _stacked_from_float([mod.q_proj, mod.k_proj, mod.v_proj], qconfig.projection_config) if FUSE_PROJECTIONS else None
        if stacked is not None:
            new.q_proj, new.k_proj, new.v_proj = stacked[1]
            _swap_linears(new, mod, ("o_proj",), qconfig.projection_config)
            object.__setattr__(new, "_qkv", stacked[0])
            return new
        _swap_linears(new, mod, ("q_proj", "k_proj", "v_proj", "o_proj"), qconfig.projection_config)
        object.__setattr__(new, "_qkv", _fuse_linears([new.q_proj, new.k_proj, new.v_proj]) if FUSE_PROJECTIONS else None)
        return new

    def extra_repr(self) -> str:
        return ", ".join(s for s in (super().extra_repr(), f"qconfig={self.qconfig}") if s)

    def _mx_attention(self, query_states, key_states, value_states, attention_mask, scaling: float) -> torch.Tensor:
        """reference :195-243; inputs [bs, heads, len, head_dim] after rotary / cache update -> [bs, q_len, heads, head_dim]"""
        qc = self.qconfig
        dtype = query_states.dtype
        q_mx = MXTensor.to_mx(query_states.contiguous(), qc.query_config.elem_dtype, qc.query_config.block_size)
        k_one = MXTensor.to_mx(key_states.contiguous(), qc.key_config.elem_dtype, qc.key_config.block_size)
        # V is quantized along the sequence axis (reference :205-212: transpose, quantize, transpose back): K5d reads the
        # [bs, heads, kv, head_dim] tensor in place; the strided copy of the whole value cache it replaces was the largest
        # single launch of a decode step (38 us of a 230 us layer at batch 32)
        vt_one = glue_ops.quantize_transposed(value_states, qc.value_config.elem_dtype, qc.value_config.block_size)
        if vt_one is None:
            vt_one = MXTensor.to_mx(value_states.transpose(2, 3).contiguous(), qc.value_config.elem_dtype, qc.value_config.block_size)
        return self._mx_attend(q_mx, k_one, vt_one, attention_mask, scaling, dtype)

    def _mx_attend(self, q_mx: MXTensor, k_one: MXTensor, vt_one: MXTensor, attention_mask, scaling: float, dtype: torch.dtype,
                   kv_len: Optional[int] = None) -> torch.Tensor:
        """the attention on MX operands: q_mx [bs, heads, q_len, head_dim], k_one [bs, kv_heads, kv_len, head_dim] and vt_one
        [bs, kv_heads, head_dim, kv_len] (V quantized along the sequence) -> [bs, q_len, heads, head_dim].  With `kv_len`, k_one
        / vt_one are the buffers of an MXDynamicCache, of which the first kv_len positions exist."""
        qc = self.qconfig
        groups = self.num_key_value_groups
        pc = qc.attention_weights_config
        ragged = kv_len is not None
        q_len, kv_len = q_mx.shape[-2], (kv_len if ragged else k_one.shape[-2])
        mask, causal = None, False
        if attention_mask is not None:  # no matter the length, we just slice it (reference :218-220)
            mask = attention_mask[:, :, :, :kv_len]
            if mask.dtype == torch.bool:  # the sdpa mask interface hands out "may attend" booleans instead of an additive mask
                mask = _additive_mask(attention_mask, dtype, getattr(self, "layer_idx", None))[:, :, :, :kv_len]
        elif q_len > 1 and getattr(self, "is_causal", True):
            causal = True  # mask creation was skipped because the attention function is expected to apply is_causal itself
        dropout = self.training and getattr(self, "attention_dropout", 0.0)
        # a cache read in place walks n = ceil128(kv_len) keys, the tail past kv_len masked (attention_ops.ragged_operands)
        n = -(-kv_len // 128) * 128 if ragged else kv_len
        if not dropout and 32 == qc.query_config.block_size == qc.key_config.block_size == qc.value_config.block_size \
                and not attention_ops.chain_is_faster(q_mx.shape[0], k_one.shape[1], q_len, n, mask is not None or causal or n != kv_len):
            # K4b: both contractions, the softmax chain and the quantization of P as one kernel -- the scores and P never reach HBM;
            # key / value heads are read in place by the query heads that share them (no repeated copies)
            out = attention_ops.flash_attention(q_mx, k_one, vt_one, scaling, mask, causal, pc.elem_dtype, pc.block_size,
                                                kv_len=kv_len if ragged else None)
            if out is not None:
                return out
        if ragged:  # the same result from the chain, on copies of the first n positions with the tail and the causal rule in the mask
            k_n, vt_n, mask_n = attention_ops.ragged_operands(k_one, vt_one, kv_len, q_len, mask, causal)
            return self._mx_attend(q_mx, k_n, vt_n, mask_n, scaling, dtype)
        # The reference repeats K and V to the number of query heads and then quantizes (:189-213).  Every MX block lives inside
        # one head (K: along head_dim; V: along the sequence of one (head, channel) row), so quantizing the key/value heads once
        # and repeating the CODES is bit-identical -- a quarter of the quantization work and of the bytes copied under 4-way GQA.
        k_mx = _repeat_heads(k_one, groups)
        v_mx = _repeat_heads(vt_one, groups).transpose(2, 3)
        scores = torch.matmul(q_mx, k_mx.transpose(2, 3))
        # scale, mask, fp32 softmax, bf16 rounding and P quantization in one pass over the scores (K4a) ...
        p_mx = None if dropout else attention_ops.softmax_to_mx(scores, scaling, mask, causal, pc.elem_dtype, pc.block_size)
        if p_mx is None:  # ... or the chain as the reference spells it (:214-239)
            attention_ops.stats["unfused_softmax"] += 1
            attn_weights = scores * scaling
            if mask is not None:
                attn_weights = attn_weights + mask
            if causal:
                hidden = torch.ones(q_len, kv_len, dtype=torch.bool, device=scores.device).triu_(kv_len - q_len + 1)
                attn_weights = attn_weights.masked_fill(hidden, float("-inf"))
            attn_weights = nn.functional.softmax(attn_weights, dim=-1, dtype=torch.float32).to(dtype)
            if dropout:
                attn_weights = nn.functional.dropout(attn_weights, p=self.attention_dropout, training=True)
            p_mx = MXTensor.to_mx(attn_weights, pc.elem_dtype, pc.block_size)
        attn_output = torch.matmul(p_mx, v_mx)
        return attn_output.transpose(1, 2).contiguous()

    def forward(self, hidden_states: torch.Tensor, position_embeddings: Optional[Tuple[torch.Tensor, torch.Tensor]] = None,
                attention_mask: Optional[torch.Tensor] = None, past_key_values=None, **kwargs):
        mod_llama = self._hf_module()
        input_shape = hidden_states.shape[:-1]
        hidden_shape = (*input_shape, -1, self.head_dim)
        fused = self.__dict__.get("_qkv")
        if _fused_still_valid(fused, (self.q_proj, self.k_proj, self.v_proj), hidden_states):
            q, k, v = fused(hidden_states).split(fused._split, dim=-1)  # one launch for the three projections
        else:
            x_in = self.q_proj.prepare_input(hidden_states)  # one activation quantization for the three projections
            q, k, v = self.q_proj(x_in), self.k_proj(x_in), self.v_proj(x_in)
        query_states = q.view(hidden_shape).transpose(1, 2)
        key_states = k.view(hidden_shape).transpose(1, 2)
        value_states = v.view(hidden_shape).transpose(1, 2)
        cos, sin = position_embeddings
        if isinstance(past_key_values, (MXStaticCache, MXDynamicCache)) and self.qconfig.is_qkv_quantization_enabled:
            # the cache holds MX codes: rotary, the quantization of Q and the append of the new tokens' K / V blocks are one launch
            # (K5e), and the attention reads the cache in place (a dynamic cache: its first `length` positions)
            layer = past_key_values.layers[self.layer_idx]
            q_mx, k_mx, vt_mx = layer.mx_append(query_states, key_states, value_states, cos, sin, self.qconfig)
            kv_len = layer.length if isinstance(past_key_values, MXDynamicCache) else None
            attn_output = self._mx_attend(q_mx, k_mx, vt_mx, attention_mask, self.scaling, query_states.dtype, kv_len=kv_len)
            return self.o_proj(attn_output.reshape(*input_shape, -1).contiguous()), None
        rotated = glue_ops.rope(query_states, key_states, cos, sin)  # one launch, the eager chain's roundings (K5b)
        query_states, key_states = rotated if rotated is not None else mod_llama.apply_rotary_pos_emb(query_states, key_states, cos, sin)
        if past_key_values is not None:
            key_states, value_states = past_key_values.update(key_states, value_states, self.layer_idx)
        if self.qconfig.is_qkv_quantization_enabled:
            attn_output, attn_weights = self._mx_attention(query_states, key_states, value_states, attention_mask, self.scaling), None
        elif (GROUPED_DECODE_SDPA and query_states.shape[2] == 1 and getattr(self.config, "_attn_implementation", "eager") == "sdpa" and not self.training
              and self.num_key_value_groups > 1 and query_states.is_cuda and (attention_mask is None or attention_mask.dim() == 4)):
            # Decode with grouped-query heads under the sdpa configuration.  transformers repeats K and V to the number of query
            # heads whenever a mask is present (sdpa_attention_forward -> repeat_kv: two copies of the whole KV cache per layer and
            # step, 82 us of a 245 us Llama-3-8B decoder layer at batch 32).  With ONE query position the query heads that share
            # a key / value head can sit on the query-length axis instead -- the same dot products and the same softmax rows, and
            # nothing is copied: q [b, h, 1, d] viewed as [b, h_kv, groups, d], the mask broadcast over the group rows.
            b, h, _, d = query_states.shape
            hk = key_states.shape[1]
            mask = None if attention_mask is None else attention_mask[:, :, :, : key_states.shape[-2]]
            out = nn.functional.scaled_dot_product_attention(query_states.reshape(b, hk, h // hk, d), key_states, value_states, attn_mask=mask,
                                                             dropout_p=0.0, scale=self.scaling, is_causal=False)
            attn_output, attn_weights = out.reshape(b, 1, h, d), None
        elif (GROUPED_DECODE_SDPA and attention_mask is None and getattr(self.config, "_attn_implementation", "eager") == "sdpa" and not self.training
              and query_states.is_cuda and isinstance(self.o_proj, MXInferenceLinear) and self.o_proj.qconfig.activations_config.block_size == 32
              and self.head_dim % 32 == 0 and not torch.compiler.is_compiling()):
            # Prefill under sdpa without a mask tensor (transformers leaves the causal rule to the kernel): the same SDPA call, but
            # its [b, h, q, d] output is quantized for o_proj straight from that layout (K5c) instead of being transposed into a
            # contiguous [b, q, h * d] copy first (sdpa_attention_forward ends with .transpose(1, 2).contiguous()) and quantized
            # by o_proj on entry -- the codes are the same bit for bit
            causal = query_states.shape[2] > 1 and getattr(self, "is_causal", True)
            out = nn.functional.scaled_dot_product_attention(query_states, key_states, value_states, attn_mask=None, dropout_p=0.0, scale=self.scaling,
                                                             is_causal=causal, enable_gqa=self.num_key_value_groups > 1)
            x_mx = glue_ops.quantize_heads(out, self.o_proj.qconfig.activations_config.elem_dtype)
            if x_mx is not None:
                return self.o_proj(x_mx), None
            attn_output, attn_weights = out.transpose(1, 2), None
        else:
            fn = mod_llama.eager_attention_forward
            impl = getattr(self.config, "_attn_implementation", "eager")
            if impl != "eager":
                fn = mod_llama.ALL_ATTENTION_FUNCTIONS.get_interface(impl, fn) if hasattr(mod_llama.ALL_ATTENTION_FUNCTIONS, "get_interface") \
                    else mod_llama.ALL_ATTENTION_FUNCTIONS[impl]
            attn_output, attn_weights = fn(self, query_states, key_states, value_states, attention_mask,
                                           dropout=0.0 if not self.training else self.attention_dropout, scaling=self.scaling, **kwargs)
        attn_output = attn_output.reshape(*input_shape, -1).contiguous()
        return self.o_proj(attn_output), attn_weights


def _make_classes():
    from transformers.models.llama import modeling_llama as ml
    from transformers.models.qwen2 import modeling_qwen2 as mq

    class MXInferenceLlamaMLP(_MXMLPMixin, ml.LlamaMLP):
        """The MX inference version of LlamaMLP (reference: mx_llama_attention.py:19-59)."""

    class MXInferenceLlamaAttention(_MXAttentionMixin, ml.LlamaAttention):
        """The MX inference version of LlamaAttention (reference: mx_llama_attention.py:62-262)."""

        @staticmethod
        def _hf_module():
            return ml

    class MXInferenceQwen2MLP(_MXMLPMixin, mq.Qwen2MLP):
        """The MX inference version of Qwen2MLP (reference: mx_qwen2_attention.py)."""

    class MXInferenceQwen2Attention(_MXAttentionMixin, mq.Qwen2Attention):
        """The MX inference version of Qwen2Attention (reference: mx_qwen2_attention.py); sliding-window layers keep the
        model's configured attention function unless every layer uses full attention."""

        @staticmethod
        def _hf_module():
            return mq

    return ml, mq, MXInferenceLlamaMLP, MXInferenceLlamaAttention, MXInferenceQwen2MLP, MXInferenceQwen2Attention


_ml, _mq, MXInferenceLlamaMLP, MXInferenceLlamaAttention, MXInferenceQwen2MLP, MXInferenceQwen2Attention = _make_classes()
ATTENTION_LAYERS = {_ml.LlamaAttention: MXInferenceLlamaAttention, _mq.Qwen2Attention: MXInferenceQwen2Attention}
MLP_LAYERS = {_ml.LlamaMLP: MXInferenceLlamaMLP, _mq.Qwen2MLP: MXInferenceQwen2MLP}
