"""CPU tier for the MX-quantized dynamic KV cache: the refusals `MXDynamicCache` raises at construction, what it reports before the
first append, its capacity policy, and the checks the C entry `mxq_flash_attention` makes on `kv_pitch` before it selects a device
-- none of them needs a GPU."""
import ctypes

import pytest

from tests.test_kv_cache_host import _llama_config


def test_mx_dynamic_cache_construction_and_refusals():
    from transformers.cache_utils import DynamicCache, DynamicLayer
    from torchmx.kv_cache import MXDynamicCache, MXDynamicLayer
    cache = MXDynamicCache(_llama_config())
    assert isinstance(cache, DynamicCache) and len(cache.layers) == 2 and all(type(layer) is MXDynamicLayer for layer in cache.layers)
    assert all(isinstance(layer, DynamicLayer) for layer in cache.layers)
    # before the first append: an empty dynamic cache, as the mask code expects
    assert cache.get_seq_length() == 0 and cache.get_mask_sizes(7, 0) == (7, 0) and cache.get_mask_sizes(1, 1) == (1, 0)
    assert cache.layers[0].get_max_cache_shape() == -1
    with pytest.raises(ValueError, match="head_dim"):
        MXDynamicCache(_llama_config(hidden_size=256))  # head_dim 64
    with pytest.raises(ValueError, match="full-attention"):
        from transformers import Qwen2Config
        MXDynamicCache(Qwen2Config(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2,
                                   vocab_size=512, use_sliding_window=True, sliding_window=64, max_window_layers=0))
    for bad in (0, 100, 131072 + 128):
        with pytest.raises(ValueError, match="initial_capacity"):
            MXDynamicCache(_llama_config(), initial_capacity=bad)
    with pytest.raises(TypeError, match="MX attention blocks"):  # a layer that is not an MX attention block with Q / K / V quantization
        cache.update(None, None, 0)
    with pytest.raises(TypeError, match="not bf16 keys"):
        cache.layers[0].offload()
    cache.reset()
    cache.crop(0)  # (nothing written yet: no-ops)
    cache.reorder_cache(None)
    assert cache.get_seq_length() == 0


def test_mx_dynamic_cache_qconfig_refusals():
    from torchmx.config import MXConfig, QAttentionConfig, QLinearConfig
    from torchmx_b200.kv_cache import _check_qconfig
    lin = QLinearConfig(weights_config=MXConfig("float8_e4m3", 32), activations_config=MXConfig("float8_e4m3", 32))
    e = MXConfig("float8_e4m3", 32)

    def qc(**kw):
        cfgs = dict(query_config=e, key_config=e, value_config=e)
        cfgs.update(kw)
        return QAttentionConfig(projection_config=lin, attention_weights_config=e, **cfgs)

    with pytest.raises(ValueError, match="int8"):
        _check_qconfig("MXDynamicCache", qc(key_config=MXConfig("int8", 32)), 128)
    with pytest.raises(ValueError, match="block size 32"):
        _check_qconfig("MXDynamicCache", qc(value_config=MXConfig("float8_e4m3", 64)), 128)
    with pytest.raises(ValueError, match="head_dim"):
        _check_qconfig("MXDynamicCache", qc(), 64)
    assert len(_check_qconfig("MXDynamicCache", qc(), 128)) == 3


def test_mx_dynamic_cache_growth_policy():
    from torchmx_b200.attention_ops import MAX_FLASH_KV
    from torchmx_b200.kv_cache import grown_capacity
    assert grown_capacity(0, 1) == 1024 and grown_capacity(0, 1024) == 1024 and grown_capacity(0, 1025) == 2048
    assert grown_capacity(0, 77, initial=128) == 128 and grown_capacity(0, 129, initial=128) == 256
    assert grown_capacity(1024, 1024) == 1024 and grown_capacity(1024, 1025) == 2048 and grown_capacity(1024, 5000) == 8192
    assert grown_capacity(128, 129, initial=128) == 256
    assert grown_capacity(65536 + 1024, 65536 + 1025) == MAX_FLASH_KV  # doubling is capped
    assert grown_capacity(0, 100000) == 100352 and grown_capacity(0, MAX_FLASH_KV) == MAX_FLASH_KV
    for cap in (0, 1024, MAX_FLASH_KV):
        with pytest.raises(ValueError, match="131072"):
            grown_capacity(cap, MAX_FLASH_KV + 1)
    # every capacity is a multiple of 128 (the attention kernel's key pitch)
    cap = 0
    for need in range(1, 40000, 997):
        cap = grown_capacity(cap, need, initial=384)
        assert cap % 128 == 0 and cap >= need


def _attention_args(kv_len, kv_pitch, q_len=1):
    from torchmx_b200 import _C
    a = _C.AttentionArgs()
    p = 256  # (a non-null, aligned placeholder address: every check below fails before anything is dereferenced)
    a.q_codes = a.q_scales = a.k_codes = a.k_scales = a.vt_codes = a.vt_scales = a.out = p
    a.batch, a.heads, a.kv_heads, a.q_len, a.kv_len, a.head_dim, a.kv_pitch = 1, 4, 2, q_len, kv_len, 128, kv_pitch
    a.p_elem = 0
    return a


def test_flash_attention_kv_pitch_validation_without_gpu():
    from torchmx_b200 import _C
    L = _C.lib()
    for kv_len, pitch, q_len in ((300, 256, 1),      # pitch below kv_len
                                 (100, 200, 1),      # pitch not a multiple of 128
                                 (100, 131072 + 128, 1),  # above MXQ_FLASH_MAX_KV
                                 (5, 128, 6),        # more queries than keys
                                 (5, -128, 1)):
        a = _attention_args(kv_len, pitch, q_len)
        assert L.mxq_flash_attention(ctypes.byref(a), -1, None) == _C.ERR_INVALID, (kv_len, pitch, q_len)
        assert b"kv_pitch" in L.mxq_last_error()
