"""GPU tier: the MX-quantized static KV cache (torchmx_b200/kv_cache.py) and its one-launch append (K5e, `glue_ops.rope_quantize_kv`).

The cache must hold exactly what the MX attention block computes from a bf16 StaticCache: rotary (transformers'
apply_rotary_pos_emb), the bf16 cache write, then the whole-cache quantization -- K along head_dim (`MXTensor.to_mx`), V along
the positions (`quantize_transposed`) -- in the one-byte form the attention kernel reads (`attention_ops._byte_operand`).  So
every comparison here is bit for bit: buffers with `torch.equal`, logits with `torch.equal`."""
import types

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
D = 128

E4M3, E3M2, E2M3, E2M1, E5M2 = "float8_e4m3", "float6_e3m2", "float6_e2m3", "float4_e2m1", "float8_e5m2"
# (Q, K, V) element types: every float type in every role once
COMBOS = [(E4M3, E4M3, E4M3), (E3M2, E2M3, E2M1), (E5M2, E2M1, E3M2), (E2M1, E5M2, E2M3), (E2M3, E3M2, E5M2)]


def _sqnr(ref, x):
    return float(20 * torch.log10(ref.float().norm() / (ref.float() - x.float()).norm()))


def _qconfig(names):
    from torchmx_b200 import dtypes
    cfg = [types.SimpleNamespace(elem_dtype=dtypes.STR_TO_ELEM_DTYPE[n], block_size=32) for n in names]
    return types.SimpleNamespace(query_config=cfg[0], key_config=cfg[1], value_config=cfg[2])


class _Reference:
    """rope -> bf16 static cache (zero-initialised) -> whole-cache quantization, as the MX attention block does it with HF's cache"""

    def __init__(self, b, hk, C, names):
        from torchmx_b200 import dtypes
        self.keys = torch.zeros(b, hk, C, D, dtype=torch.bfloat16, device=DEV)
        self.values = torch.zeros_like(self.keys)
        self.elems = [dtypes.STR_TO_ELEM_DTYPE[n] for n in names]
        self.length = 0

    def append(self, q, k, v, cos, sin):
        from transformers.models.llama.modeling_llama import apply_rotary_pos_emb
        from torchmx_b200 import attention_ops, glue_ops
        from torchmx_b200.mx_tensor import MXTensor
        qr, kr = apply_rotary_pos_emb(q, k, cos, sin)
        t = k.shape[2]
        self.keys[:, :, self.length:self.length + t] = kr
        self.values[:, :, self.length:self.length + t] = v
        self.length += t
        prev = glue_ops.set_fused_glue(True)
        try:
            vt = glue_ops.quantize_transposed(self.values, self.elems[2])
        finally:
            glue_ops.set_fused_glue(prev)
        return [attention_ops._byte_operand(x) for x in (MXTensor.to_mx(qr.contiguous(), self.elems[0], 32), MXTensor.to_mx(self.keys, self.elems[1], 32), vt)]


def _qkv(b, t, hq, hk, gen, scale=2.0):
    """q / k / v as column slices of one stacked projection output [b, t, (hq + 2 hk) * 128], viewed [b, heads, t, 128]; cos / sin"""
    x = torch.randn(b, t, (hq + 2 * hk) * D, device=DEV, generator=gen).mul_(scale).to(torch.bfloat16)
    q, k, v = x.split([hq * D, hk * D, hk * D], -1)
    views = [y.view(b, t, -1, D).transpose(1, 2) for y in (q, k, v)]
    ang = torch.rand(1 if b == 1 else b, t, D // 2, device=DEV, generator=gen) * 6.3
    ang = torch.cat([ang, ang], -1)
    return (*views, ang.cos().to(torch.bfloat16), ang.sin().to(torch.bfloat16))


def _check(layer, ref, got_q, want):
    (qc, qf, qs), (kc, kf, ks), (vc, vf, vs) = want
    assert torch.equal(got_q._data, qc) and torch.equal(got_q._scale_e8m0, qs), "Q codes"
    assert torch.equal(layer.k_codes, kc) and torch.equal(layer.k_scales, ks), "K cache"
    assert torch.equal(layer.vt_codes, vc) and torch.equal(layer.vt_scales, vs), "V cache"
    blk = ref.length // 32 * 32
    open_want = torch.zeros_like(layer.v_open)
    n = min(ref.values.shape[2], blk + 32) - blk
    open_want[:, :, :n] = ref.values[:, :, blk:blk + n]
    assert torch.equal(layer.v_open.view(torch.int16), open_want.view(torch.int16)), "open block"  # (bits: NaN != NaN)
    assert int(layer.cumulative_length.item()) == ref.length


def _run_sequence(names, b, hq, hk, C, lengths, exact, monkeypatch, poison=None):
    from torchmx_b200 import env_variables as env
    from torchmx_b200 import glue_ops
    from torchmx_b200.kv_cache import MXStaticLayer
    monkeypatch.setattr(env, "MX_EXACT_QUANTIZATION", "True" if exact else "False")
    gen = torch.Generator(device=DEV).manual_seed(sum(lengths) + b)
    layer, ref, qcfg = MXStaticLayer(C), _Reference(b, hk, C, names), _qconfig(names)
    n0 = glue_ops.stats["rope_quantize_kv"]
    for i, t in enumerate(lengths):
        q, k, v, cos, sin = _qkv(b, t, hq, hk, gen)
        if poison is not None and i == poison[0]:
            v[0, 0, 0, 3], v[-1, -1, 0, 70] = poison[1], -poison[1]  # a NaN / Inf lands in the block that stays open
        got_q, k_mx, vt_mx = layer.mx_append(q, k, v, cos, sin, qcfg)
        assert k_mx._data is layer.k_codes and vt_mx._data is layer.vt_codes
        _check(layer, ref, got_q, ref.append(q, k, v, cos, sin))
    assert glue_ops.stats["rope_quantize_kv"] - n0 == len(lengths)  # one launch per append


@pytest.mark.parametrize("exact", [False, True])
@pytest.mark.parametrize("prefill", [1, 5, 32, 37, 300])
def test_prefill_then_decode_appends_bit_identical(prefill, exact, monkeypatch):
    """a prefill, then single-token appends across at least two V block boundaries; every float type as Q, K and V"""
    names = COMBOS[[1, 5, 32, 37, 300].index(prefill)]
    steps = 64 - prefill % 32 + 1
    _run_sequence(names, 1, 4, 2, 384, [prefill] + [1] * steps, exact, monkeypatch)


@pytest.mark.parametrize("start", [0, 7, 31, 32, 100])
@pytest.mark.parametrize("b,hq,hk", [(1, 4, 4), (3, 8, 2)])
def test_multi_token_appends_at_any_position(start, b, hq, hk, monkeypatch):
    """an append of 45 tokens starting at L (touching two or three V blocks), then one more token; batch 1 and 3, GQA"""
    names = COMBOS[start % 5]
    _run_sequence(names, b, hq, hk, 256, ([start] if start else []) + [45, 1], False, monkeypatch)


@pytest.mark.parametrize("bad", [float("nan"), float("inf")])
@pytest.mark.parametrize("exact", [False, True])
def test_nan_or_inf_inside_the_open_value_block(bad, exact, monkeypatch):
    """the open block is re-derived from its bf16 copy on every append, NaN / Inf included (NaN-scale block rules)"""
    _run_sequence((E4M3, E2M3, E3M2), 2, 4, 2, 128, [37, 1, 1, 5, 1], exact, monkeypatch, poison=(1, bad))
    _run_sequence((E4M3, E4M3, E2M1), 2, 4, 2, 128, [3, 1, 2], exact, monkeypatch, poison=(0, bad))


# ---- the model ----------------------------------------------------------------------------------------------------------------
def _model(names=(E4M3, E4M3, E4M3), impl="eager", qkv=True):
    import copy
    import torchmx  # noqa: F401
    from transformers import LlamaConfig, LlamaForCausalLM
    from torchmx.config import MXConfig, QAttentionConfig, QLinearConfig
    from torchmx.quant_api import quantize_llm_
    cfg = LlamaConfig(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, vocab_size=512,
                      max_position_embeddings=512)
    cfg._attn_implementation = impl
    torch.manual_seed(0)
    model = LlamaForCausalLM(cfg).to(DEV, torch.bfloat16).eval()
    qm = copy.deepcopy(model)
    lin = QLinearConfig(weights_config=MXConfig("float6_e3m2", 32), activations_config=MXConfig("float8_e4m3", 32))
    q, k, v = (MXConfig(n, 32) for n in names)
    qa = QAttentionConfig(projection_config=lin, query_config=q, key_config=k, value_config=v, attention_weights_config=MXConfig(E4M3, 32)) if qkv \
        else QAttentionConfig(projection_config=lin)
    quantize_llm_(qm, qa, lin)
    return qm, cfg


def _decode(qm, cache, ids, mask, prefill=37, steps=40):
    """prefill, then teacher-forced single-token steps: the logits of every forward"""
    out = [qm(input_ids=ids[:, :prefill], attention_mask=mask[:, :prefill], past_key_values=cache, use_cache=True).logits]
    for i in range(prefill, prefill + steps):
        out.append(qm(input_ids=ids[:, i:i + 1], attention_mask=mask[:, :i + 1], past_key_values=cache, use_cache=True).logits)
    return out


def _padded_batch(cfg, n=77):
    g = torch.Generator(device=DEV).manual_seed(3)
    ids = torch.randint(1, cfg.vocab_size, (3, n), device=DEV, generator=g)
    mask = torch.ones(3, n, dtype=torch.long, device=DEV)
    mask[1, :9] = 0
    mask[2, :21] = 0  # left padding
    return ids, mask


@pytest.mark.parametrize("impl", ["eager", "sdpa"])
@torch.no_grad()
def test_model_logits_and_generate_equal_the_bf16_static_cache(impl):
    from transformers.cache_utils import StaticCache
    from torchmx import attention_ops
    from torchmx.kv_cache import MXStaticCache
    qm, cfg = _model(impl=impl)
    ids, mask = _padded_batch(cfg)
    want = _decode(qm, StaticCache(config=qm.config, max_cache_len=128), ids, mask)
    n0 = attention_ops.stats["flash_attention"]
    got = _decode(qm, MXStaticCache(qm.config, max_cache_len=128), ids, mask)
    assert attention_ops.stats["flash_attention"] - n0 == 2 * 41  # one K4b launch per layer and forward
    for i, (a, b) in enumerate(zip(want, got)):
        assert torch.equal(a, b), f"forward {i}"
    # (disable_compile: generate would otherwise compile the decoding step of a static cache, which the ctypes launches do not trace)
    gen_kw = dict(input_ids=ids[:, :37], attention_mask=mask[:, :37], max_new_tokens=16, do_sample=False, min_new_tokens=16, disable_compile=True)
    ref = qm.generate(past_key_values=StaticCache(config=qm.config, max_cache_len=128), **gen_kw)
    out = qm.generate(past_key_values=MXStaticCache(qm.config, max_cache_len=128), **gen_kw)
    assert out.shape == (3, 37 + 16) and torch.equal(ref, out)


@torch.no_grad()
def test_decode_step_replayed_from_a_cuda_graph():
    """the write position lives on the device: a captured decode step replays at the advancing position, same logits as eager
    (sdpa: transformers' eager mask makes a host tensor on every forward, which a capture refuses)"""
    from torchmx.kv_cache import MXStaticCache
    qm, cfg = _model(impl="sdpa")
    ids, _ = _padded_batch(cfg)
    eager = MXStaticCache(qm.config, max_cache_len=128)
    qm(input_ids=ids[:, :37], past_key_values=eager, use_cache=True)
    want = [qm(input_ids=ids[:, i:i + 1], past_key_values=eager, use_cache=True).logits for i in range(37, 45)]
    cache = MXStaticCache(qm.config, max_cache_len=128)
    qm(input_ids=ids[:, :37], past_key_values=cache, use_cache=True)
    tok = ids[:, 37:38].clone()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for i in (37, 38):  # warm-up steps: real appends
            tok.copy_(ids[:, i:i + 1])
            assert torch.equal(qm(input_ids=tok, past_key_values=cache, use_cache=True).logits, want[i - 37])
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = qm(input_ids=tok, past_key_values=cache, use_cache=True).logits
    assert int(cache.layers[0].cumulative_length.item()) == 39  # (capture runs nothing)
    for i in range(39, 45):
        tok.copy_(ids[:, i:i + 1])
        g.replay()
        assert torch.equal(out, want[i - 37]), f"replayed step at position {i}"
    assert all(int(layer.cumulative_length.item()) == 45 for layer in cache.layers)


@pytest.mark.parametrize("names", [(E4M3, E4M3, E4M3), (E3M2, E2M1, E2M3)])
@torch.no_grad()
def test_chain_without_the_attention_kernel_matches_the_bf16_cache_chain(names):
    """K4b switched off: the K3 -> K4a -> K3 chain runs on the cache views.  e4m3: equal.  fp6 / fp4: the cache operands are typed
    float8_e4m3 (same values) while the bf16-cache chain contracts the fp6 / fp4 codes -- equal is not promised; SQNR > 40 dB"""
    from transformers.cache_utils import StaticCache
    from torchmx import attention_ops
    from torchmx.kv_cache import MXStaticCache
    qm, cfg = _model(names)
    ids, mask = _padded_batch(cfg)
    prev = attention_ops.set_flash_attention(False)
    try:
        n0 = attention_ops.stats["flash_attention"]
        want = _decode(qm, StaticCache(config=qm.config, max_cache_len=128), ids, mask, steps=6)
        got = _decode(qm, MXStaticCache(qm.config, max_cache_len=128), ids, mask, steps=6)
        assert attention_ops.stats["flash_attention"] == n0
    finally:
        attention_ops.set_flash_attention(prev)
    for a, b in zip(want, got):
        if names[0] == E4M3:
            assert torch.equal(a, b)
        else:
            assert torch.equal(a, b) or _sqnr(a, b) > 40, _sqnr(a, b)


@torch.no_grad()
def test_resident_bytes_after_prefill():
    """(1 + 1/32) B per key and value element plus the open blocks: at most 0.53 of the bf16 StaticCache of the same shape"""
    from torchmx.kv_cache import MXStaticCache
    qm, cfg = _model()
    ids, _ = _padded_batch(cfg)
    C, b, hk, layers = 2048, 3, 2, 2
    qm(input_ids=ids[:, :37], past_key_values=MXStaticCache(qm.config, max_cache_len=C), use_cache=True)  # warm-up: lazily made state
    torch.cuda.synchronize()
    m0 = torch.cuda.memory_allocated()
    cache = MXStaticCache(qm.config, max_cache_len=C)
    out = qm(input_ids=ids[:, :37], past_key_values=cache, use_cache=True)
    del out
    torch.cuda.synchronize()
    grown = torch.cuda.memory_allocated() - m0
    elems = layers * b * hk * C * D  # per K and per V
    bf16 = 2 * elems * 2
    bound = 2 * elems * (1 + 1 / 32) + layers * b * hk * 32 * D * 2
    assert grown <= bound + layers * 2 * 512, (grown, bound)  # (+ the two 8-byte positions, 512-byte allocator blocks)
    assert grown <= 0.53 * bf16, grown / bf16


@torch.no_grad()
def test_refusals():
    from torchmx.kv_cache import MXStaticCache
    qm, cfg = _model((E4M3, "int8", E4M3))
    ids, _ = _padded_batch(cfg)
    with pytest.raises(ValueError, match="int8"):
        qm(input_ids=ids[:, :5], past_key_values=MXStaticCache(qm.config, max_cache_len=64), use_cache=True)
    plain, _ = _model(qkv=False)
    with pytest.raises(TypeError, match="MX attention blocks"):
        plain(input_ids=ids[:, :5], past_key_values=MXStaticCache(plain.config, max_cache_len=64), use_cache=True)
    qm, _ = _model()
    cache = MXStaticCache(qm.config, max_cache_len=64)
    qm(input_ids=ids[:, :37], past_key_values=cache, use_cache=True)
    with pytest.raises(ValueError, match="closed value block"):
        cache.crop(20)
    assert int(cache.layers[0].cumulative_length.item()) == 37


@pytest.mark.parametrize("keep,junk", [(32, 20), (33, 4)])
@torch.no_grad()
def test_crop_then_append_equals_never_having_written(keep, junk):
    """crop(n), n a multiple of 32 or inside the open block: the cache is byte for byte the one that never held the cropped
    tokens, and appends continue identically"""
    from torchmx.kv_cache import MXStaticCache
    qm, cfg = _model((E3M2, E4M3, E2M1))
    ids, _ = _padded_batch(cfg)
    junk_ids = torch.flip(ids, [1])
    a, b = MXStaticCache(qm.config, max_cache_len=96), MXStaticCache(qm.config, max_cache_len=96)
    qm(input_ids=ids[:, :keep], past_key_values=a, use_cache=True)
    qm(input_ids=ids[:, :keep], past_key_values=b, use_cache=True)
    qm(input_ids=junk_ids[:, :junk], past_key_values=b, use_cache=True)
    b.crop(keep)
    la, lb = a.layers[0], b.layers[0]
    for name in ("k_codes", "k_scales", "vt_codes", "vt_scales", "v_open", "cumulative_length"):
        assert torch.equal(getattr(la, name), getattr(lb, name)), name
    out_a = qm(input_ids=ids[:, keep:keep + 13], past_key_values=a, use_cache=True).logits
    out_b = qm(input_ids=ids[:, keep:keep + 13], past_key_values=b, use_cache=True).logits
    assert torch.equal(out_a, out_b)
    for la, lb in zip(a.layers, b.layers):
        for name in ("k_codes", "k_scales", "vt_codes", "vt_scales", "v_open", "cumulative_length"):
            assert torch.equal(getattr(la, name), getattr(lb, name)), name
    b.reset()
    assert b.get_seq_length() == 0 and not b.layers[1].vt_codes.any() and not b.layers[1].v_open.any()
