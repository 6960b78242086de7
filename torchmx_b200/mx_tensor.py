"""MXTensor and the two custom ops of the MX hot path, API-compatible with the reference's
`torchmx.mx_tensor` (/root/reference/torchmx/mx_tensor.py) but with the op bodies executed by
hand-written sm_100a CUDA (libmxq.so, C ABI in include/mxq.h) instead of chains of aten ops.

  torchmx::quantize_mx(Tensor data_hp, str elem_dtype_name, SymInt block_size) -> (Tensor, Tensor)
      reference: mx_tensor.py:36-96 (+ fake kernel :99-120)   -> mxq_quantize
  torchmx::dequantize_mx(Tensor data_lp, Tensor shared_exp_e8m0, str elem_dtype_name,
                         SymInt block_size, ScalarType target_dtype, SymInt block_dim) -> Tensor
      reference: mx_tensor.py:123-164 (+ fake kernel :167-193) -> mxq_dequantize[_strided]

Storage layout (user-visible and persisted through state_dict, so identical to the reference):
`_data` uint8 (int8 for the int8 element type), one byte per element, fp6 codes in bits [5:0],
fp4 two per byte with the even element in the high nibble; `_scale_e8m0` uint8 `[..., L/block]`.

There is no CPU implementation: tensors must live on a CUDA device, otherwise the ops raise.
"""
from __future__ import annotations

import contextlib
import math
import threading
from typing import Dict, Optional, Tuple

import torch
import torch.nn.functional as F

from . import _C, dtypes
from . import env_variables as env
from .utils import tensor_size_fp4x2_to_hp

_HP_ID = {torch.bfloat16: _C.HP_BF16, torch.float32: _C.HP_F32}


def _require_cuda(t: torch.Tensor, what: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"{what}: tensor is on '{t.device}'. torchmx_b200 runs the MX kernels on CUDA (sm_100a) only; "
            "there is no CPU fallback. Move the tensor to a B200 first.")


def _stream_ptr(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _quant_flags(elem: dtypes.DType) -> int:
    """MXQ_FLAG_HW_EXACT when the reference's hardware-exact quantization is on and `elem` is one of the four element types it
    applies to (mx_tensor.py:80-90), else 0.  `env` is read at call time: callers may flip it after import."""
    return _C.FLAG_HW_EXACT if env.MX_EXACT_QUANTIZATION == "True" and elem in dtypes.SUPPORTED_FP_ELEM_DTYPES else 0


def _codes_shape(lead, cols, elem: dtypes.DType) -> Tuple[tuple, torch.dtype]:
    """(shape, dtype) of the codes of `cols` elements per row, blocked along the last axis: fp4 packs two codes per byte, int8
    codes are int8, every other element type is one uint8 per element"""
    return tuple(lead) + (cols // 2 if elem == dtypes.float4_e2m1 else cols,), torch.int8 if elem == dtypes.int8 else torch.uint8


def _codes_like(lead, cols, elem: dtypes.DType, device) -> torch.Tensor:
    shape, dtype = _codes_shape(lead, cols, elem)
    return torch.empty(shape, dtype=dtype, device=device)


# ------------------------------------------------------------------------------------------------
# where the scale tensors of a whole-model quantization live
# ------------------------------------------------------------------------------------------------
# The E8M0 scales of most transformer weights are smaller than 1 MiB (q_proj of Llama-8B: 512 KiB, k_proj: 128 KiB), which is the
# caching allocator's SMALL pool: 2 MiB segments of their own, each a cudaMalloc -- and on a box with tens of GB mapped one such call
# was measured at 1-18 ms, 20+ of them per `quantize_linear_` (tools/quantize_linear_diag.py), while the memory of the bf16 weights
# being released sits unused in the large pool.  Inside `small_scale_arena()` scale tensors below 1 MiB are carved out of large-pool
# chunks instead (views, 256-byte aligned; a chunk lives as long as any scale in it).  Values and layouts are unchanged.
_arena_state = threading.local()


@contextlib.contextmanager
def small_scale_arena(chunk_bytes: int = 32 << 20):
    prev = getattr(_arena_state, "cur", None)
    _arena_state.cur = {"buf": None, "off": 0, "chunk": int(chunk_bytes)}
    try:
        yield
    finally:
        _arena_state.cur = prev


def _empty_scales(shape, device) -> torch.Tensor:
    n = math.prod(shape)
    a = getattr(_arena_state, "cur", None)
    if a is None or n == 0 or n >= (1 << 20) or (torch.device(device).type == "cuda" and torch.cuda.is_current_stream_capturing()):
        return torch.empty(shape, dtype=torch.uint8, device=device)
    need = (n + 255) & ~255
    if a["buf"] is None or a["buf"].device != device or a["off"] + need > a["buf"].numel():
        a["buf"], a["off"] = torch.empty(max(a["chunk"], need), dtype=torch.uint8, device=device), 0
    out = a["buf"][a["off"]:a["off"] + n].view(shape)
    a["off"] += need
    return out


# ------------------------------------------------------------------------------------------------
# custom ops
# ------------------------------------------------------------------------------------------------
def _quantize_mx_impl(data_hp: torch.Tensor, elem_dtype_name: str, block_size: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """High-precision tensor -> (E8M0 scales, element codes), blocks along the last dim.

    Same contract as the reference op (mx_tensor.py:36-96): returns the SCALE FIRST; `data_hp` must
    be bfloat16 with a last dim that is a multiple of `block_size`.  Supersets: a non-contiguous
    input is compacted first instead of asserting (mx_tensor.py:62), float32 input and the
    `float8_e5m2` element type are accepted as labelled extensions (parity unpinned).
    """
    assert elem_dtype_name in dtypes.STR_TO_ELEM_DTYPE, (
        f"Unsupported dtype {elem_dtype_name}. Supported: {dtypes.SUPPORTED_ELEM_DTYPES}")
    elem = dtypes.STR_TO_ELEM_DTYPE[elem_dtype_name]
    assert data_hp.dtype in _HP_ID, f"Only torch.bfloat16 input dtype is supported, got {data_hp.dtype}"
    assert block_size >= 1 and data_hp.dim() >= 1
    assert data_hp.shape[-1] % block_size == 0, "The last dimension of the input tensor must be a multiple of block_size"
    _require_cuda(data_hp, "torchmx::quantize_mx")
    x = data_hp.contiguous()
    shape = tuple(x.shape)
    n_blocks = x.numel() // block_size
    scales = _empty_scales(shape[:-1] + (shape[-1] // block_size,), x.device)
    assert elem != dtypes.float4_e2m1 or shape[-1] % 2 == 0  # pack_uint4's requirement (utils.py:143)
    codes = _codes_like(shape[:-1], shape[-1], elem, x.device)
    if n_blocks:
        rc = _C.lib().mxq_quantize(x.data_ptr(), _HP_ID[x.dtype], n_blocks, block_size, dtypes.ELEM_ID[elem.name], _quant_flags(elem),
                                   codes.data_ptr(), scales.data_ptr(), x.device.index, _stream_ptr(x))
        _C.check(rc, "torchmx::quantize_mx")
    return scales, codes


def _quantize_into(data_hp: torch.Tensor, elem: dtypes.DType, block_size: int, codes_out: torch.Tensor, scales_out: torch.Tensor) -> None:
    """`_quantize_mx_impl` writing into caller-provided CONTIGUOUS code / scale tensors (internal: a block that stacks several
    weights quantizes each of them straight into its rows of the stacked storage instead of quantizing and copying)."""
    assert data_hp.dtype in _HP_ID and data_hp.is_contiguous() and codes_out.is_contiguous() and scales_out.is_contiguous()
    assert data_hp.shape[-1] % block_size == 0 and scales_out.numel() * block_size == data_hp.numel()
    assert codes_out.numel() * (2 if elem == dtypes.float4_e2m1 else 1) == data_hp.numel() and codes_out.device == data_hp.device == scales_out.device
    _require_cuda(data_hp, "torchmx::quantize_mx")
    if data_hp.numel():
        rc = _C.lib().mxq_quantize(data_hp.data_ptr(), _HP_ID[data_hp.dtype], data_hp.numel() // block_size, block_size, dtypes.ELEM_ID[elem.name],
                                   _quant_flags(elem), codes_out.data_ptr(), scales_out.data_ptr(), data_hp.device.index, _stream_ptr(data_hp))
        _C.check(rc, "torchmx::quantize_mx")


@torch.library.custom_op("torchmx::quantize_mx", mutates_args=())
def quantize_mx(data_hp: torch.Tensor, elem_dtype_name: str, block_size: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """The registered op (schema and semantics of the reference's, mx_tensor.py:36-96); body = `_quantize_mx_impl`."""
    return _quantize_mx_impl(data_hp, elem_dtype_name, block_size)


@quantize_mx.register_fake
def _(data_hp: torch.Tensor, elem_dtype_name: str, block_size: int) -> Tuple[torch.Tensor, torch.Tensor]:
    shape = tuple(data_hp.shape)
    scales = data_hp.new_empty(shape[:-1] + (shape[-1] // block_size,), dtype=torch.uint8)
    codes_shape, codes_dtype = _codes_shape(shape[:-1], shape[-1], dtypes.STR_TO_ELEM_DTYPE[elem_dtype_name])
    return scales, data_hp.new_empty(codes_shape, dtype=codes_dtype)


def _collapse_around(t_sizes, t_strides, d):
    """[pre..., d, post...] of a C-contiguous tensor -> 3 dims (pre, d, post)."""
    pre = math.prod(t_sizes[:d])
    post = math.prod(t_sizes[d + 1:])
    return [pre, t_sizes[d], post], [t_sizes[d] * post, post, 1]


def _dequantize_mx_impl(data_lp: torch.Tensor, shared_exp_e8m0: torch.Tensor, elem_dtype_name: str, block_size: int,
                        target_dtype: torch.dtype, block_dim: int) -> torch.Tensor:
    """(codes, scales) -> high precision, contiguous in the logical shape.

    Same contract as the reference op (mx_tensor.py:123-164).  `data_lp` / `shared_exp_e8m0` may be
    arbitrary views (transposed, expanded, ...) whose blocked axis is `block_dim`; fp4 is packed
    along `block_dim`.  `target_dtype` must be bfloat16 or float32 (the two the reference documents,
    mx_tensor.py:467-470).
    """
    assert elem_dtype_name in dtypes.STR_TO_ELEM_DTYPE, f"unsupported dtype: {elem_dtype_name}"
    elem = dtypes.STR_TO_ELEM_DTYPE[elem_dtype_name]
    if target_dtype not in _HP_ID:
        raise NotImplementedError(f"torchmx::dequantize_mx: target dtype {target_dtype} (supported: bfloat16, float32)")
    assert data_lp.dtype in (torch.uint8, torch.int8), f"{data_lp.dtype} is unsupported"
    assert shared_exp_e8m0.dtype == torch.uint8
    _require_cuda(data_lp, "torchmx::dequantize_mx")
    nd = data_lp.dim()
    bd = block_dim if block_dim >= 0 else block_dim + nd
    assert 0 <= bd < nd and shared_exp_e8m0.dim() == nd
    sizes = list(data_lp.shape)
    if elem == dtypes.float4_e2m1:
        sizes[bd] *= 2
    assert shared_exp_e8m0.shape[bd] * block_size == sizes[bd], (
        f"scale shape {tuple(shared_exp_e8m0.shape)} does not cover data shape {tuple(sizes)} with block {block_size}")
    out = torch.empty(sizes, dtype=target_dtype, device=data_lp.device)
    if out.numel() == 0:
        return out
    L = _C.lib()
    eid, tid = dtypes.ELEM_ID[elem.name], _HP_ID[target_dtype]
    if bd == nd - 1 and data_lp.is_contiguous() and shared_exp_e8m0.is_contiguous():
        rc = L.mxq_dequantize(data_lp.data_ptr(), shared_exp_e8m0.data_ptr(), shared_exp_e8m0.numel(), block_size, eid, tid,
                              out.data_ptr(), data_lp.device.index, _stream_ptr(data_lp))
        _C.check(rc, "torchmx::dequantize_mx")
        return out
    cs, ss = list(data_lp.stride()), list(shared_exp_e8m0.stride())
    if nd > _C.MAX_DIMS:
        # plain layout copies (no MX arithmetic), then view as (pre, blocked, post)
        data_lp, shared_exp_e8m0 = data_lp.contiguous(), shared_exp_e8m0.contiguous()
        sizes3, cs = _collapse_around(list(data_lp.shape), None, bd)
        _, ss = _collapse_around(list(shared_exp_e8m0.shape), None, bd)
        sizes3[1] = sizes[bd]
        sizes, bd, nd = sizes3, 1, 3
    rc = L.mxq_dequantize_strided(data_lp.data_ptr(), shared_exp_e8m0.data_ptr(), nd, _C.i64_array(sizes), _C.i64_array(cs),
                                  _C.i64_array(ss), bd, block_size, eid, tid, out.data_ptr(), data_lp.device.index,
                                  _stream_ptr(data_lp))
    _C.check(rc, "torchmx::dequantize_mx")
    return out


@torch.library.custom_op("torchmx::dequantize_mx", mutates_args=())
def dequantize_mx(data_lp: torch.Tensor, shared_exp_e8m0: torch.Tensor, elem_dtype_name: str, block_size: int,
                  target_dtype: torch.dtype, block_dim: int) -> torch.Tensor:
    """The registered op (schema and semantics of the reference's, mx_tensor.py:123-164); body = `_dequantize_mx_impl`."""
    return _dequantize_mx_impl(data_lp, shared_exp_e8m0, elem_dtype_name, block_size, target_dtype, block_dim)


@dequantize_mx.register_fake
def _(data_lp: torch.Tensor, shared_exp_e8m0: torch.Tensor, elem_dtype_name: str, block_size: int,
      target_dtype: torch.dtype, block_dim: int) -> torch.Tensor:
    sizes = list(data_lp.shape)
    if elem_dtype_name == dtypes.float4_e2m1.name:
        sizes[block_dim] = sizes[block_dim] * 2
    return data_lp.new_empty(sizes, dtype=target_dtype)


# ------------------------------------------------------------------------------------------------
# autograd wrappers: padding / slicing around the ops, identity backward
# ------------------------------------------------------------------------------------------------
@torch._dynamo.allow_in_graph
class ToMXConstrFunc(torch.autograd.Function):
    """Differentiable cast to MX; backward is the identity (reference: mx_tensor.py:196-252)."""

    @staticmethod
    def forward(ctx, data_hp: torch.Tensor, elem_dtype: dtypes.DType, block_size: int, _op=None):
        last = data_hp.shape[-1]
        padding = -last % block_size
        if padding:
            assert block_size % 2 == 0, f"block_size must be even to support padding but got {block_size}"
            data_hp = F.pad(data_hp, (0, padding))  # zeros never raise a block's max exponent
        scale, codes = (_op or quantize_mx)(data_hp, elem_dtype.name, block_size)
        if padding:
            # fp4: an odd tail keeps its (zero) partner nibble -> ceil (mx_tensor.py:231-239)
            keep = math.ceil(last / 2) if elem_dtype == dtypes.float4_e2m1 else last
            codes = codes[..., :keep].contiguous()
        return MXTensor(scale, codes, elem_dtype, block_size, data_hp.dtype, padding)

    @staticmethod
    def backward(ctx, g):
        return g, None, None


@torch._dynamo.allow_in_graph
class FromMXConstrFunc(torch.autograd.Function):
    """Differentiable cast from MX; backward is the identity (reference: mx_tensor.py:255-331)."""

    @staticmethod
    def forward(ctx, tensor_lp: "MXTensor", target_dtype: torch.dtype, _op=None) -> torch.Tensor:
        if ctx is not None:
            ctx._padding = tensor_lp._padding
            ctx._elem_dtype = tensor_lp._elem_dtype
        codes, bd, padding = tensor_lp._data, tensor_lp._block_dim, tensor_lp._padding
        is_fp4 = tensor_lp._elem_dtype == dtypes.float4_e2m1
        logical = codes.shape[bd] * 2 - (padding % 2) if is_fp4 else codes.shape[bd]
        if padding:
            # re-create the zero codes that were sliced off so every block is complete (mx_tensor.py:296-305)
            pad_spec = [0] * (2 * codes.dim())
            pad_spec[2 * (codes.dim() - 1 - bd) + 1] = padding // 2 if is_fp4 else padding
            codes = F.pad(codes, pad_spec, mode="constant", value=0)
        out = (_op or dequantize_mx)(codes, tensor_lp._scale_e8m0, tensor_lp._elem_dtype.name, tensor_lp._block_size, target_dtype, bd)
        if padding:
            out = out.narrow(bd, 0, logical)
        return out.contiguous()

    @staticmethod
    def backward(ctx, g):
        if ctx._padding > 0 and ctx._elem_dtype == dtypes.float4_e2m1:
            raise ValueError("Padding is not supported in the backward pass for float4_e2m1")
        return g, None, None


@torch._dynamo.allow_in_graph
class NoopFwToMXBw(torch.autograd.Function):
    """Forward: identity.  Backward: quantize the gradient (reference: mx_tensor.py:334-354)."""

    @staticmethod
    def forward(ctx, x: torch.Tensor, elem_dtype: dtypes.DType, block_size: int):
        ctx.elem_dtype, ctx.block_size = elem_dtype, block_size
        return x

    @staticmethod
    def backward(ctx, g):
        scale, codes = quantize_mx(g, ctx.elem_dtype.name, ctx.block_size)
        return MXTensor(scale, codes, ctx.elem_dtype, ctx.block_size, g.dtype), None, None


# ------------------------------------------------------------------------------------------------
# the tensor subclass
# ------------------------------------------------------------------------------------------------
class MXTensor(torch.Tensor):
    """Wrapper subclass: outer shape / dtype are those of the high-precision tensor, storage is
    `_scale_e8m0` + `_data` (reference: mx_tensor.py:357-523; the reference derives from torchao's
    TorchAOBaseTensor only for the `implements` table, which is provided here directly)."""

    _ATEN_TABLE: Dict = {}

    @staticmethod
    def __new__(cls, scale_e8m0_bits: torch.Tensor, data_bits: torch.Tensor, elem_dtype: dtypes.DType, block_size: int,
                orig_dtype: torch.dtype, padding: int = 0, block_dim: Optional[int] = None):
        nd = data_bits.dim()
        block_dim = nd - 1 if block_dim is None else (block_dim if block_dim >= 0 else block_dim + nd)
        size = list(data_bits.size())
        if elem_dtype == dtypes.float4_e2m1:
            size = tensor_size_fp4x2_to_hp(size, block_dim)
            size[block_dim] -= padding % 2  # the partner nibble of an odd tail is padding, not data
        self = torch.Tensor._make_wrapper_subclass(cls, size, dtype=orig_dtype, device=data_bits.device)
        assert scale_e8m0_bits.dtype == torch.uint8, "unsupported"
        assert elem_dtype in dtypes.EXTENDED_ELEM_DTYPES, f"unsupported elem_dtype {elem_dtype}"
        assert data_bits.dtype in (torch.uint8, torch.int8), f"{data_bits.dtype} is unsupported"
        if not isinstance(data_bits, torch._subclasses.fake_tensor.FakeTensor):
            covered = list(scale_e8m0_bits.shape)
            covered[block_dim] = covered[block_dim] * block_size - padding
            assert math.prod(covered) == math.prod(size), f"{math.prod(covered)} != {math.prod(size)}"
        self._scale_e8m0 = scale_e8m0_bits
        self._data = data_bits
        self._elem_dtype = elem_dtype
        self._block_size = block_size
        self._orig_dtype = orig_dtype
        self._block_dim = block_dim
        self._padding = padding
        return self

    def __init__(self, *args, **kwargs):
        pass

    # --- aten override table (same decorator surface as TorchAOBaseTensor.implements) -----------
    @classmethod
    def implements(cls, aten_ops):
        if not isinstance(aten_ops, (list, tuple)):
            aten_ops = [aten_ops]

        def deco(fn):
            for op in aten_ops:
                cls._ATEN_TABLE[op] = fn
            return fn

        return deco

    @classmethod
    def __torch_dispatch__(cls, func, types, args=(), kwargs=None):
        handler = cls._ATEN_TABLE.get(func)
        if handler is None:
            raise NotImplementedError(f"{cls.__name__} dispatch: attempting to run unimplemented operator/function: {func}")
        return handler(func, types, args, {} if kwargs is None else kwargs)

    __torch_function__ = torch._C._disabled_torch_function_impl

    # --- user API -----------------------------------------------------------------------------
    def to_dtype(self, target_dtype: torch.dtype) -> torch.Tensor:
        """Dequantize to `target_dtype` (bfloat16 or float32); reference: mx_tensor.py:456-472."""
        if not torch.is_grad_enabled() and type(self._data) is torch.Tensor and self._data.is_cuda and not torch.compiler.is_compiling():
            return FromMXConstrFunc.forward(None, self, target_dtype, _op=_dequantize_mx_impl)  # inference fast path, see to_mx
        return FromMXConstrFunc.apply(self, target_dtype)

    @staticmethod
    @torch._dynamo.allow_in_graph
    def to_mx(data_hp: torch.Tensor, elem_dtype: dtypes.DType, block_size: int = 32) -> "MXTensor":
        """Quantize a bfloat16 tensor along its last dim; reference: mx_tensor.py:474-493."""
        if (not torch.is_grad_enabled() or not data_hp.requires_grad) and type(data_hp) is torch.Tensor and data_hp.is_cuda \
                and not torch.compiler.is_compiling():
            # inference fast path: same arithmetic, without the autograd.Function and the Python custom-op dispatcher
            # (~0.2 ms of host time per call -- per layer and forward in eager mode, per weight in quantize_linear_)
            return ToMXConstrFunc.forward(None, data_hp, elem_dtype, block_size, _op=_quantize_mx_impl)
        return ToMXConstrFunc.apply(data_hp, elem_dtype, block_size)

    def _quantization_type(self):
        return (f"shape={self.shape}, block_size={self._block_size}, device={self.device}, "
                f"elem_dtype={self._elem_dtype}, orig_dtype={self._orig_dtype}, ")

    def __repr__(self):
        s = f"MXTensor: _elem_dtype: {self._elem_dtype}, _scale_e8m0: {self._scale_e8m0}, _data: {self._data}"
        if type(self._data) is torch.Tensor and self._data.is_cuda:  # (not while tracing: fake / functional inner tensors)
            s += f", d_hp: {self.to_dtype(self._orig_dtype)}"
        if self._padding > 0:
            s += f", padding: {self._padding}"
        return s

    # --- subclass flattening (torch.compile, state_dict) --------------------------------------
    def __tensor_flatten__(self):
        meta = {"_elem_dtype": self._elem_dtype, "_block_size": self._block_size, "_orig_dtype": self._orig_dtype,
                "_block_dim": self._block_dim, "_padding": self._padding}
        return ["_scale_e8m0", "_data"], meta

    @staticmethod
    def __tensor_unflatten__(inner_tensors: Dict, metadata, outer_size, outer_stride):
        return MXTensor(inner_tensors["_scale_e8m0"], inner_tensors["_data"], metadata["_elem_dtype"], metadata["_block_size"],
                        metadata["_orig_dtype"], metadata["_padding"], metadata["_block_dim"])


# a state_dict holding MXTensor parameters loads with weights_only=True (reference: mx_tensor.py:526-528)
torch.serialization.add_safe_globals([MXTensor, dtypes.DType])
