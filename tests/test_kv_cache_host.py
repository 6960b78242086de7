"""CPU tier for the MX-quantized static KV cache: argument checks of the C entry `mxq_rope_quantize_kv` (K5e) and the
refusals `MXStaticCache` raises at construction -- none of them needs a GPU."""
import ctypes

import pytest


def _args():
    from torchmx_b200 import _C
    a = _C.RopeQuantizeKVArgs()
    p = 256  # (a non-null, aligned placeholder address: every check below fails before anything is dereferenced)
    a.q = a.k = a.v = a.cos = a.sin = a.q_codes = a.q_scales = a.k_codes = a.k_scales = a.vt_codes = a.vt_scales = a.v_open = a.position = p
    a.batch, a.tokens, a.q_heads, a.kv_heads, a.head_dim, a.capacity = 2, 5, 4, 2, 128, 64
    return a


def test_rope_quantize_kv_argument_validation_without_gpu():
    from torchmx_b200 import _C
    L = _C.lib()
    assert L.mxq_rope_quantize_kv(None, -1, None) == _C.ERR_INVALID and b"null args" in L.mxq_last_error()
    a = _args()
    a.k_elem = 4  # int8: K4b has no int8 operand
    assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_INVALID and b"element type 4" in L.mxq_last_error()
    a = _args()
    a.v_elem = 9
    assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_INVALID
    for cap in (0, 48, -32):
        a = _args()
        a.capacity = cap
        assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_INVALID and b"multiple of 32" in L.mxq_last_error()
    a = _args()
    a.tokens = 65  # more tokens than the cache holds
    assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_INVALID
    a = _args()
    a.batch = -1
    assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_INVALID and b"negative" in L.mxq_last_error()
    for field in ("q", "v", "cos", "vt_scales", "v_open", "position"):
        a = _args()
        setattr(a, field, None)
        assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_INVALID and b"null pointer" in L.mxq_last_error(), field
    a = _args()
    a.kv_heads = 0
    assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_INVALID and b"no heads" in L.mxq_last_error()
    a = _args()
    a.head_dim = 64
    assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.ERR_UNSUPPORTED_SHAPE and b"head_dim" in L.mxq_last_error()
    a = _args()
    a.tokens = 0  # nothing to append: a no-op, whatever the pointers
    a.q = None
    assert L.mxq_rope_quantize_kv(ctypes.byref(a), -1, None) == _C.OK


def _llama_config(**kw):
    from transformers import LlamaConfig
    base = dict(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, vocab_size=512,
                max_position_embeddings=512)
    base.update(kw)
    return LlamaConfig(**base)


def test_mx_static_cache_construction_and_refusals():
    from transformers.cache_utils import StaticCache
    from torchmx.kv_cache import MXStaticCache, MXStaticLayer
    cache = MXStaticCache(_llama_config(), max_cache_len=128)
    assert isinstance(cache, StaticCache) and len(cache.layers) == 2 and all(type(layer) is MXStaticLayer for layer in cache.layers)
    assert cache.get_seq_length() == 0 and cache.max_cache_len == 128 and cache.is_compileable
    assert cache.get_mask_sizes(1, 0) == (128, 0)  # what the mask code sees: an ordinary static cache of capacity 128
    with pytest.raises(ValueError, match="multiple of 32"):
        MXStaticCache(_llama_config(), max_cache_len=100)
    with pytest.raises(ValueError, match="8192"):
        MXStaticCache(_llama_config(), max_cache_len=8192 + 32)
    MXStaticCache(_llama_config(), max_cache_len=8192)
    with pytest.raises(ValueError, match="head_dim"):
        MXStaticCache(_llama_config(hidden_size=256), max_cache_len=64)  # head_dim 64
    with pytest.raises(ValueError, match="full-attention"):
        from transformers import Qwen2Config
        MXStaticCache(Qwen2Config(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
                                  vocab_size=512, use_sliding_window=True, sliding_window=64, max_window_layers=0), max_cache_len=128)
    with pytest.raises(TypeError, match="MX attention blocks"):  # a layer that is not an MX attention block with Q / K / V quantization
        cache.update(None, None, 0)
    cache.reset()
    cache.crop(0)  # (nothing written yet: no-ops)
