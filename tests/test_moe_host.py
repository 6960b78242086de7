"""CPU tier of the mixture-of-experts layer (K6): argument validation of the three C entries before any CUDA call, and the module
surgery of quantize_llm_ on MoE models built on the meta device."""
import ctypes
import os
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _route_args(**kw):
    from torchmx_b200 import _C
    a = _C.MoeRouteArgs()
    a.top_k_index, a.tokens, a.top_k, a.num_experts = 256, 4, 2, 8
    a.offsets, a.row_of_slot, a.token_of_row = 256, 512, 768
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def _gemm_args(**kw):
    from torchmx_b200 import _C
    g = _C.MoeGemmArgs()
    g.w_codes, g.w_scales, g.x_codes, g.x_scales, g.offsets, g.d = 256, 512, 768, 1024, 1280, 1536
    g.rows, g.num_experts, g.N, g.K = 8, 4, 256, 256
    for k, v in kw.items():
        setattr(g, k, v)
    return g


def _combine_args(**kw):
    from torchmx_b200 import _C
    c = _C.MoeCombineArgs()
    c.y, c.top_k_index, c.top_k_weights, c.row_of_slot, c.out = 256, 512, 768, 1024, 1280
    c.weights_dtype, c.tokens, c.top_k, c.num_experts, c.hidden = _C.HP_F32, 4, 2, 8, 128
    for k, v in kw.items():
        setattr(c, k, v)
    return c


@pytest.mark.parametrize("field, value, code, words", [
    ("top_k_index", None, "INVALID", b"top_k_index"), ("offsets", None, "INVALID", b"offsets"), ("row_of_slot", None, "INVALID", b"row_of_slot"),
    ("token_of_row", None, "INVALID", b"token_of_row"), ("top_k", 9, "INVALID", b"top_k"), ("top_k", 0, "INVALID", b"top_k"),
    ("num_experts", 257, "INVALID", b"num_experts"), ("tokens", 16385, "INVALID", b"tokens"),
])
def test_route_rejects(field, value, code, words):
    from torchmx_b200 import _C
    L = _C.lib()
    a = _route_args(**{field: value})
    assert L.mxq_moe_route(ctypes.byref(a), -1, None) == getattr(_C, "ERR_" + code)
    assert words in L.mxq_last_error()


def test_route_rejects_quantization_arguments():
    from torchmx_b200 import _C
    L = _C.lib()
    assert L.mxq_moe_route(None, -1, None) == _C.ERR_INVALID
    for missing, word in (("x", b"null x"), ("codes", b"null codes"), ("scales", b"null scales")):
        kw = dict(x=4096, codes=8192, scales=12288, hidden=256, ldx=256)
        kw[missing] = None
        assert L.mxq_moe_route(ctypes.byref(_route_args(**kw)), -1, None) == _C.ERR_INVALID and word in L.mxq_last_error()
    base = dict(x=4096, codes=8192, scales=12288, hidden=256, ldx=256)
    assert L.mxq_moe_route(ctypes.byref(_route_args(**dict(base, elem=9))), -1, None) == _C.ERR_INVALID and b"element type" in L.mxq_last_error()
    assert L.mxq_moe_route(ctypes.byref(_route_args(**dict(base, hidden=48, ldx=48))), -1, None) == _C.ERR_UNSUPPORTED_SHAPE and b"hidden" in L.mxq_last_error()
    assert L.mxq_moe_route(ctypes.byref(_route_args(**dict(base, x=4104))), -1, None) == _C.ERR_UNSUPPORTED_SHAPE and b"x is not" in L.mxq_last_error()
    assert L.mxq_moe_route(ctypes.byref(_route_args(**dict(base, codes=8200))), -1, None) == _C.ERR_UNSUPPORTED_SHAPE and b"codes" in L.mxq_last_error()
    assert L.mxq_moe_route(ctypes.byref(_route_args(**dict(base, tokens=0))), -1, None) == _C.OK  # empty batch: no launch


@pytest.mark.parametrize("field, value, code, words", [
    ("w_codes", None, "INVALID", b"w_codes"), ("w_scales", None, "INVALID", b"w_scales"), ("x_codes", None, "INVALID", b"x_codes"),
    ("x_scales", None, "INVALID", b"x_scales"), ("offsets", None, "INVALID", b"offsets"), ("d", None, "INVALID", b"null d"),
    ("num_experts", 257, "INVALID", b"num_experts"), ("num_experts", 0, "INVALID", b"num_experts"), ("w_format", 5, "INVALID", b"operand format"),
    ("K", 192, "UNSUPPORTED_SHAPE", b"K 192"), ("N", 200, "UNSUPPORTED_SHAPE", b"N 200"),
    ("w_codes", 272, "UNSUPPORTED_SHAPE", b"w_codes"), ("x_codes", 784, "UNSUPPORTED_SHAPE", b"x_codes"),
    ("w_scales", 520, "UNSUPPORTED_SHAPE", b"w_scales"), ("d", 1544, "UNSUPPORTED_SHAPE", b"d is not"),
])
def test_gemm_rejects(field, value, code, words):
    from torchmx_b200 import _C
    L = _C.lib()
    assert L.mxq_moe_gemm(ctypes.byref(_gemm_args(**{field: value})), -1, None) == getattr(_C, "ERR_" + code)
    assert words in L.mxq_last_error()


def test_gemm_and_combine_empty_problems_launch_nothing():
    from torchmx_b200 import _C
    L = _C.lib()
    assert L.mxq_moe_gemm(None, -1, None) == _C.ERR_INVALID
    assert L.mxq_moe_gemm(ctypes.byref(_gemm_args(rows=0)), -1, None) == _C.OK
    assert L.mxq_moe_combine(None, -1, None) == _C.ERR_INVALID
    assert L.mxq_moe_combine(ctypes.byref(_combine_args(tokens=0)), -1, None) == _C.OK


@pytest.mark.parametrize("field, value, code, words", [
    ("y", None, "INVALID", b"null y"), ("top_k_index", None, "INVALID", b"top_k_index"), ("top_k_weights", None, "INVALID", b"top_k_weights"),
    ("row_of_slot", None, "INVALID", b"row_of_slot"), ("out", None, "INVALID", b"null out"), ("top_k", 9, "INVALID", b"top_k"),
    ("num_experts", 300, "INVALID", b"num_experts"), ("weights_dtype", 7, "INVALID", b"weights_dtype"),
    ("hidden", 100, "UNSUPPORTED_SHAPE", b"hidden"), ("y", 264, "UNSUPPORTED_SHAPE", b"y is not"), ("out", 1288, "UNSUPPORTED_SHAPE", b"out is not"),
])
def test_combine_rejects(field, value, code, words):
    from torchmx_b200 import _C
    L = _C.lib()
    assert L.mxq_moe_combine(ctypes.byref(_combine_args(**{field: value})), -1, None) == getattr(_C, "ERR_" + code)
    assert words in L.mxq_last_error()


def _tiny_moe_models():
    from transformers import (MixtralConfig, MixtralForCausalLM, OlmoeConfig, OlmoeForCausalLM, Qwen2MoeConfig, Qwen2MoeForCausalLM,
                              Qwen3MoeConfig, Qwen3MoeForCausalLM)
    kw = dict(hidden_size=256, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, vocab_size=320)
    return (
        (MixtralForCausalLM, MixtralConfig(intermediate_size=384, num_local_experts=8, num_experts_per_tok=2, **kw)),
        (Qwen2MoeForCausalLM, Qwen2MoeConfig(moe_intermediate_size=128, shared_expert_intermediate_size=256, num_experts=8, num_experts_per_tok=2, **kw)),
        (Qwen3MoeForCausalLM, Qwen3MoeConfig(moe_intermediate_size=128, num_experts=16, num_experts_per_tok=4, head_dim=64, **kw)),
        (OlmoeForCausalLM, OlmoeConfig(intermediate_size=128, num_experts=8, num_experts_per_tok=2, **kw)),
    )


def test_quantize_llm_swaps_every_expert_bank_on_meta():
    """quantize_llm_ on tiny Mixtral / Qwen2-MoE / Qwen3-MoE / OLMoE models: exactly the expert banks become MXInferenceExperts
    (meta weights stay meta), the routers are untouched and no nn.Linear is left"""
    from torchmx_b200.config import MXConfig, QAttentionConfig, QLinearConfig
    from torchmx_b200.layers.mx_experts import MXInferenceExperts, _bank_classes
    from torchmx_b200.quant_api import quantize_llm_
    lin = QLinearConfig(weights_config=MXConfig("float4_e2m1", 32), activations_config=MXConfig("float8_e4m3", 32))
    for model_cls, cfg in _tiny_moe_models():
        with torch.device("meta"):
            m = model_cls(cfg)
        banks = [n for n, x in m.named_modules() if type(x) in _bank_classes()]
        routers = {n: type(x) for n, x in m.named_modules() if type(x).__name__.endswith("TopKRouter")}
        assert len(banks) == 2 and len(routers) == 2
        quantize_llm_(m, QAttentionConfig(projection_config=lin), lin)
        swapped = {n for n, x in m.named_modules() if type(x) is MXInferenceExperts}
        assert swapped == set(banks), (model_cls.__name__, swapped, banks)
        assert {n: type(x) for n, x in m.named_modules() if type(x).__name__.endswith("TopKRouter")} == routers
        assert not any(type(x) is torch.nn.Linear for x in m.modules())
        assert not any(type(x) in _bank_classes() for x in m.modules())
        for n in swapped:
            e = m.get_submodule(n)
            assert e.qconfig is lin and e.gate_up_proj.device.type == "meta"
            assert tuple(e.gate_up_proj.shape) == (e.num_experts, 2 * e.intermediate_dim, e.hidden_dim)
            assert tuple(e.down_proj.shape) == (e.num_experts, e.hidden_dim, e.intermediate_dim)
            assert set(e.state_dict()) == {"gate_up_proj", "down_proj"}


def test_only_the_supported_bank_layout_is_swapped():
    """a bank with a bias, a transposed layout or another activation is not the layout MXInferenceExperts reproduces"""
    from transformers import MixtralConfig
    from transformers.models.mixtral.modeling_mixtral import MixtralExperts
    from torchmx_b200.layers.mx_experts import is_expert_bank
    with torch.device("meta"):
        bank = MixtralExperts(MixtralConfig(hidden_size=128, intermediate_size=128, num_local_experts=4))
    assert is_expert_bank(bank)
    bank.has_bias = True
    assert not is_expert_bank(bank)
    bank.has_bias, bank.is_transposed = False, True
    assert not is_expert_bank(bank)
    bank.is_transposed, bank.act_fn = False, torch.nn.GELU()
    assert not is_expert_bank(bank)
    assert not is_expert_bank(torch.nn.Linear(4, 4, device="meta"))
