"""KV caches held as MX codes -- `MXStaticCache` (fixed capacity) and `MXDynamicCache` (grows with the sequence) -- for the MX
attention blocks of `quantize_llm_` with a full `QAttentionConfig` (query / key / value / attention-weights configs).

The MX attention block quantizes K along head_dim and V along the sequence axis (32 consecutive positions of one channel per
block) before both attention contractions.  With transformers' bf16 `StaticCache` it stores the rotated keys and the values in
bf16 and quantizes the WHOLE cache again at every forward, so a decode step's work grows with the capacity, not with the new
tokens.  Here the cache holds exactly the operands the attention kernel (K4b) consumes, and each forward computes only the
blocks its new tokens touch, in one launch with rotary and the quantization of Q (K5e, `glue_ops.rope_quantize_kv`):

* keys: codes [batch, kv_heads, C, 128] + scales [batch, kv_heads, C, 4] -- a key row's blocks depend on that row alone;
* values: codes [batch, kv_heads, 128, C] + scales [batch, kv_heads, 128, C / 32], blocked along the positions; only the block
  holding the current length (the *open* block) can still change, and a bf16 copy of it ([batch, kv_heads, 32, 128]) is enough
  to re-derive it exactly.

The codes are the ones the whole-cache quantization of a zero-initialised bf16 StaticCache gives, bit for bit, so a model's
logits are unchanged.  Codes are one byte per element in the form K4b reads: e4m3 / e5m2 as they are, fp6 / fp4 as their exact
E4M3 re-encoding (the tensors are typed float8_e4m3 -- same values).  Every float element type therefore costs 1 + 1/32 B per
element against the 2 B of bf16; int8 has no attention operand and is refused.

Usage: `model(..., past_key_values=MXStaticCache(model.config, max_cache_len=C), use_cache=True)` (or `generate(...,
past_key_values=...)`).  The layers subclass transformers' StaticLayer / StaticCache, so generate and the mask code see an
ordinary static cache; a layer that is not an MX attention block with Q / K / V quantization reaches `update` and raises.

`MXDynamicCache(model.config)` stores the same layout in buffers whose capacity grows geometrically (a multiple of 128, up to
attention_ops.MAX_FLASH_KV = 131072 positions).  It subclasses transformers' DynamicCache / DynamicLayer, so it works wherever
the default dynamic cache does (greedy and beam-search generate included).  The attention kernel reads it in place at whatever
length it has (`attention_ops.flash_attention(..., kv_len=L)`): no bf16 concatenation and no re-quantization of the cache per
step, and no key length the kernel declines.
"""
from __future__ import annotations

import torch
from transformers.cache_utils import DynamicCache, DynamicLayer, StaticCache, StaticLayer

from . import glue_ops, mx_gemm
from .attention_ops import MAX_FLASH_KV
from .dtypes import int8
from .mx_tensor import MXTensor

HEAD_DIM = 128      # the attention kernel's head_dim
MAX_CAPACITY = 8192  # the longest key axis the attention kernel takes with a mask


def _zero_block_scale(elem, device) -> int:
    """E8M0 scale the quantizer gives an all-zero block (its codes are all +0, byte 0, in every element type)"""
    return int(MXTensor.to_mx(torch.zeros(32, dtype=torch.bfloat16, device=device), elem, 32)._scale_e8m0.item())


def _check_config(name: str, text_config) -> None:
    head_dim = getattr(text_config, "head_dim", None) or text_config.hidden_size // text_config.num_attention_heads
    if head_dim != HEAD_DIM:
        raise ValueError(f"{name}: head_dim must be {HEAD_DIM} (the MX attention kernel's), got {head_dim}")


def _check_qconfig(name: str, qconfig, head_dim: int):
    """the element types of Q, K and V, or ValueError when the cache cannot hold them"""
    elems = (qconfig.query_config.elem_dtype, qconfig.key_config.elem_dtype, qconfig.value_config.elem_dtype)
    if any(e == int8 for e in elems):
        raise ValueError(f"{name}: int8 query / key / value configs have no one-byte attention operand")
    if any(c.block_size != 32 for c in (qconfig.query_config, qconfig.key_config, qconfig.value_config)):
        raise ValueError(f"{name}: query / key / value configs need block size 32")
    if head_dim != HEAD_DIM:
        raise ValueError(f"{name}: head_dim must be {HEAD_DIM}, got {head_dim}")
    return elems


def _clear_from(layer, n: int, length: int, name: str) -> None:
    """Make positions >= n of a layer holding `length` positions read as never written (the crop rule of both caches): n must
    be a multiple of 32 or lie in the open block, whose bf16 copy re-derives the codes of the positions below n."""
    if n % 32 and n // 32 != length // 32:
        raise ValueError(f"{name}.crop({n}): position {n} lies in a closed value block (the cache holds {length}); the bf16 values "
                         "that would re-derive it are no longer kept -- crop to a multiple of 32 or within the open block")
    layer.k_codes[:, :, n:].zero_()
    layer.k_scales[:, :, n:].fill_(layer._zero_scales[0])
    nb = n // 32
    layer.vt_codes[..., 32 * nb:].zero_()
    layer.vt_scales[..., nb:].fill_(layer._zero_scales[1])
    if n % 32:  # the open block keeps positions below n: re-derive its codes from the bf16 copy, K5d's arithmetic
        layer.v_open[:, :, n % 32:].zero_()
        v_elem = layer.elem_dtypes[2]
        vt = glue_ops.quantize_transposed(layer.v_open, v_elem)
        if vt is None:
            raise RuntimeError(f"{name}.crop: the transposed quantization kernel (K5d) does not take the open block")
        codes, _ = mx_gemm._operand_rows(vt._data, v_elem, None, packed=False)  # the cache's one-byte form
        layer.vt_codes[..., 32 * nb:32 * nb + 32].copy_(codes)
        layer.vt_scales[..., nb].copy_(vt._scale_e8m0[..., 0])
    else:
        layer.v_open.zero_()


def _append(layer, name: str, query_states, key_states, value_states, cos, sin, position):
    """K5e on a layer's buffers at the device position `position` (not advanced) -> Q as an MXTensor"""
    q_mx = glue_ops.rope_quantize_kv(query_states, key_states, value_states, cos, sin, position, layer.k_codes, layer.k_scales,
                                     layer.vt_codes, layer.vt_scales, layer.v_open, layer.elem_dtypes)
    if q_mx is None:
        raise RuntimeError(f"{name}: the rope + quantize kernel (K5e) does not take these operands (bf16 CUDA q / k / v with heads "
                           "contiguous inside a token row, 16-byte aligned, cos / sin [batch | 1, tokens, 128])")
    return q_mx


class MXStaticLayer(StaticLayer):
    """One layer of `MXStaticCache`: MX codes and scales of the keys and values, the bf16 open value block, and HF's device-side
    write position `cumulative_length`.  Buffers are allocated on the first append."""

    def __init__(self, max_cache_len: int):
        if max_cache_len <= 0 or max_cache_len % 32:
            raise ValueError(f"MXStaticCache: max_cache_len must be a positive multiple of 32 (V is blocked along 32 positions), got {max_cache_len}")
        if max_cache_len > MAX_CAPACITY:
            raise ValueError(f"MXStaticCache: max_cache_len {max_cache_len} exceeds {MAX_CAPACITY}, the longest masked key axis of the MX attention kernel")
        super().__init__(max_cache_len)

    def lazy_initialization(self, key_states, value_states):
        raise TypeError("MXStaticCache holds MX codes, not bf16 keys / values: only MX attention blocks with Q / K / V quantization "
                        "(quantize_llm_ with a full QAttentionConfig) can use it")

    def update(self, key_states, value_states, *args, **kwargs):
        self.lazy_initialization(key_states, value_states)

    def _mx_initialize(self, key_states: torch.Tensor, qconfig) -> None:
        b, hk, _, d = key_states.shape
        elems = _check_qconfig("MXStaticCache", qconfig, d)
        dev, C = key_states.device, self.max_cache_len
        self.dtype, self.device = torch.bfloat16, dev
        self.max_batch_size, self.num_heads, self.k_head_dim, self.v_head_dim = b, hk, d, d
        self.elem_dtypes = elems
        self._zero_scales = (_zero_block_scale(elems[1], dev), _zero_block_scale(elems[2], dev))
        self.k_codes = torch.zeros((b, hk, C, d), dtype=torch.uint8, device=dev)
        self.k_scales = torch.full((b, hk, C, d // 32), self._zero_scales[0], dtype=torch.uint8, device=dev)
        self.vt_codes = torch.zeros((b, hk, d, C), dtype=torch.uint8, device=dev)
        self.vt_scales = torch.full((b, hk, d, C // 32), self._zero_scales[1], dtype=torch.uint8, device=dev)
        self.v_open = torch.zeros((b, hk, 32, d), dtype=torch.bfloat16, device=dev)
        self.cumulative_length = self.cumulative_length.to(dev)
        # the operands K4b reads: views of the whole cache, typed by their one-byte storage
        self.k_mx = MXTensor(self.k_scales, self.k_codes, glue_ops.byte_operand_dtype(elems[1]), 32, torch.bfloat16)
        self.vt_mx = MXTensor(self.vt_scales, self.vt_codes, glue_ops.byte_operand_dtype(elems[2]), 32, torch.bfloat16)
        if not torch.compiler.is_compiling():
            for t in (self.k_codes, self.k_scales, self.vt_codes, self.vt_scales, self.v_open, self.cumulative_length):
                torch._dynamo.mark_static_address(t)
        self.is_initialized = True

    def mx_append(self, query_states, key_states, value_states, cos, sin, qconfig):
        """Rotary embedding of the new queries / keys, their keys and values appended at the current length, the length advanced:
        -> (Q, K, Vt) MXTensors, K / Vt views of the whole cache (what K4b takes)."""
        if not self.is_initialized:
            self._mx_initialize(key_states, qconfig)
        elif key_states.shape[:2] != (self.max_batch_size, self.num_heads):
            raise ValueError(f"MXStaticCache: batch / kv heads {tuple(key_states.shape[:2])} differ from the cache's {(self.max_batch_size, self.num_heads)}")
        q_mx = _append(self, "MXStaticCache", query_states, key_states, value_states, cos, sin, self.cumulative_length)
        self.cumulative_length.add_(key_states.shape[2])
        return q_mx, self.k_mx, self.vt_mx

    def reset(self) -> None:
        if self.is_initialized:
            self.k_codes.zero_()
            self.k_scales.fill_(self._zero_scales[0])
            self.vt_codes.zero_()
            self.vt_scales.fill_(self._zero_scales[1])
            self.v_open.zero_()
        self.cumulative_length.zero_()

    def crop(self, max_length: int) -> None:
        """Keep the first `max_length` positions (negative: drop that many) and clear the rest, as if they had never been
        written.  Supported when `max_length` is a multiple of 32 or lies in the open block (the block holding the current
        length), whose bf16 copy re-derives the codes; a cut into a closed V block raises ValueError."""
        if not self.is_initialized:
            return
        length = int(self.cumulative_length.item())
        n = length + max_length if max_length < 0 else max_length
        if n >= length:
            return
        if n < 0:
            raise ValueError(f"MXStaticCache.crop: cannot crop to {max_length} positions")
        _clear_from(self, n, length, "MXStaticCache")
        self.cumulative_length.fill_(n)


class MXStaticCache(StaticCache):
    """transformers' StaticCache with every layer an `MXStaticLayer`: keys and values stored as MX codes in the element types of
    each attention block's key / value configs.  Same constructor as StaticCache.  Refuses (ValueError) sliding-window or
    chunked layers, head_dim != 128, max_cache_len not a multiple of 32 or above 8192; int8 configs at the first forward."""

    def __init__(self, config, max_cache_len: int):
        super().__init__(config=config, max_cache_len=max_cache_len)
        if any(type(layer) is not StaticLayer for layer in self.layers):
            raise ValueError("MXStaticCache: only full-attention layers are supported (no sliding-window, chunked or linear-attention layers)")
        _check_config("MXStaticCache", config.get_text_config(decoder=True))
        self.layers = [MXStaticLayer(max_cache_len) for _ in self.layers]


def grown_capacity(capacity: int, needed: int, initial: int = 1024) -> int:
    """Capacity of an MXDynamicLayer that must hold `needed` positions and now holds `capacity` (0: not allocated yet): the
    first allocation is `needed` rounded up to a multiple of `initial`, later ones double until `needed` fits, capped at
    MAX_FLASH_KV.  ValueError past MAX_FLASH_KV positions."""
    if needed > MAX_FLASH_KV:
        raise ValueError(f"MXDynamicCache: {needed} positions exceed {MAX_FLASH_KV}, the longest key axis of the MX attention kernel")
    if needed <= capacity:
        return capacity
    if capacity == 0:
        return min(MAX_FLASH_KV, -(-max(needed, 1) // initial) * initial)
    while capacity < needed:
        capacity *= 2
    return min(MAX_FLASH_KV, capacity)


class MXDynamicLayer(DynamicLayer):
    """One layer of `MXDynamicCache`: the layout of `MXStaticLayer` (MX codes and scales of the keys and values, the bf16 open
    value block) in buffers of a capacity that grows with the sequence, the host-side length and the device write position K5e
    reads.  Positions at or past the length read as never written (zero codes, the zero block's scale).  Nothing here holds bf16
    keys or values: `update` and everything else that would need them raise."""

    def __init__(self, initial_capacity: int = 1024):
        if initial_capacity <= 0 or initial_capacity % 128 or initial_capacity > MAX_FLASH_KV:
            raise ValueError(f"MXDynamicCache: initial_capacity must be a positive multiple of 128 up to {MAX_FLASH_KV}, got {initial_capacity}")
        super().__init__()
        self.initial_capacity = initial_capacity
        self.capacity = 0
        self.length = 0

    def lazy_initialization(self, key_states, value_states):
        raise TypeError("MXDynamicCache holds MX codes, not bf16 keys / values: only MX attention blocks with Q / K / V quantization "
                        "(quantize_llm_ with a full QAttentionConfig) can use it")

    def update(self, key_states, value_states, *args, **kwargs):
        self.lazy_initialization(key_states, value_states)

    def offload(self):
        self.lazy_initialization(None, None)

    def prefetch(self):
        self.lazy_initialization(None, None)

    def get_seq_length(self) -> int:
        return self.length

    def get_mask_sizes(self, query_length: int) -> tuple[int, int]:
        return self.length + query_length, 0

    def _allocate(self, capacity: int) -> None:
        """buffers of `capacity` positions, every position unwritten except the first `length`, copied from the current ones"""
        b, hk, d, dev = self.max_batch_size, self.num_heads, HEAD_DIM, self.device
        k_codes = torch.zeros((b, hk, capacity, d), dtype=torch.uint8, device=dev)
        k_scales = torch.full((b, hk, capacity, d // 32), self._zero_scales[0], dtype=torch.uint8, device=dev)
        vt_codes = torch.zeros((b, hk, d, capacity), dtype=torch.uint8, device=dev)
        vt_scales = torch.full((b, hk, d, capacity // 32), self._zero_scales[1], dtype=torch.uint8, device=dev)
        if self.capacity:
            L, nb = self.length, -(-self.length // 32)  # (positions of the open block past L are unwritten in the old buffers too)
            k_codes[:, :, :L].copy_(self.k_codes[:, :, :L])
            k_scales[:, :, :L].copy_(self.k_scales[:, :, :L])
            vt_codes[..., :32 * nb].copy_(self.vt_codes[..., :32 * nb])
            vt_scales[..., :nb].copy_(self.vt_scales[..., :nb])
        self.k_codes, self.k_scales, self.vt_codes, self.vt_scales = k_codes, k_scales, vt_codes, vt_scales
        self.capacity = capacity
        self._make_views()

    def _make_views(self) -> None:
        # the operands K4b reads: the whole capacity, typed by the one-byte storage
        self.k_mx = MXTensor(self.k_scales, self.k_codes, glue_ops.byte_operand_dtype(self.elem_dtypes[1]), 32, torch.bfloat16)
        self.vt_mx = MXTensor(self.vt_scales, self.vt_codes, glue_ops.byte_operand_dtype(self.elem_dtypes[2]), 32, torch.bfloat16)

    def mx_append(self, query_states, key_states, value_states, cos, sin, qconfig):
        """Rotary embedding of the new queries / keys, their keys and values appended at the current length (the buffers grow
        first when they must), the length advanced -> (Q, K, Vt) MXTensors, K / Vt views of the whole capacity, of which the
        first `self.length` positions exist."""
        b, hk, t, d = key_states.shape
        if not self.is_initialized:
            self.elem_dtypes = _check_qconfig("MXDynamicCache", qconfig, d)
            self.dtype, self.device = torch.bfloat16, key_states.device
            self.max_batch_size, self.num_heads = b, hk
            self._zero_scales = (_zero_block_scale(self.elem_dtypes[1], self.device), _zero_block_scale(self.elem_dtypes[2], self.device))
            self.v_open = torch.zeros((b, hk, 32, d), dtype=torch.bfloat16, device=self.device)
            self.position = torch.zeros((), dtype=torch.int64, device=self.device)
            self.is_initialized = True
        elif (b, hk) != (self.max_batch_size, self.num_heads):
            raise ValueError(f"MXDynamicCache: batch / kv heads {(b, hk)} differ from the cache's {(self.max_batch_size, self.num_heads)}")
        capacity = grown_capacity(self.capacity, self.length + t, self.initial_capacity)
        if capacity != self.capacity:
            self._allocate(capacity)
        q_mx = _append(self, "MXDynamicCache", query_states, key_states, value_states, cos, sin, self.position)
        self.position.add_(t)
        self.length += t
        return q_mx, self.k_mx, self.vt_mx

    def reset(self) -> None:
        if self.is_initialized and self.capacity:
            _clear_from(self, 0, self.length, "MXDynamicCache")
            self.position.zero_()
        self.length = 0

    def crop(self, max_length: int) -> None:
        """Keep the first `max_length` positions (negative: drop that many), as `MXStaticLayer.crop` does: to a multiple of 32
        or within the open block; a cut into a closed V block raises ValueError.  The capacity stays."""
        n = self.length + max_length if max_length < 0 else max_length
        if n >= self.length:
            return
        if n < 0:
            raise ValueError(f"MXDynamicCache.crop: cannot crop to {max_length} positions")
        _clear_from(self, n, self.length, "MXDynamicCache")
        self.position.fill_(n)
        self.length = n

    def _index_batch(self, fn) -> None:
        """apply `fn` (an index operation on dim 0) to every per-sequence buffer"""
        if not self.is_initialized:
            return
        self.v_open = fn(self.v_open)
        if self.capacity:
            self.k_codes, self.k_scales, self.vt_codes, self.vt_scales = (fn(x) for x in (self.k_codes, self.k_scales, self.vt_codes, self.vt_scales))
            self._make_views()
        self.max_batch_size = self.v_open.shape[0]

    def batch_repeat_interleave(self, repeats: int) -> None:
        self._index_batch(lambda x: x.repeat_interleave(repeats, dim=0))

    def batch_select_indices(self, indices: torch.Tensor) -> None:
        self._index_batch(lambda x: x[indices].contiguous())

    def reorder_cache(self, beam_idx: torch.LongTensor) -> None:
        self._index_batch(lambda x: x.index_select(0, beam_idx.to(x.device)))


class MXDynamicCache(DynamicCache):
    """transformers' DynamicCache with every layer an `MXDynamicLayer`: keys and values stored as MX codes in the element types
    of each attention block's key / value configs, in buffers that grow with the sequence up to MAX_FLASH_KV positions.
    `initial_capacity` (a multiple of 128) is the granularity of the first allocation.  Refuses (ValueError) sliding-window,
    chunked or linear-attention layers and head_dim != 128; int8 configs and block sizes other than 32 at the first forward;
    an append past MAX_FLASH_KV positions."""

    def __init__(self, config, initial_capacity: int = 1024):
        super().__init__(config=config)
        if any(type(layer) is not DynamicLayer for layer in self.layers):
            raise ValueError("MXDynamicCache: only full-attention layers are supported (no sliding-window, chunked or linear-attention layers)")
        _check_config("MXDynamicCache", config.get_text_config(decoder=True))
        self.layers = [MXDynamicLayer(initial_capacity) for _ in self.layers]
