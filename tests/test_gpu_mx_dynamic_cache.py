"""GPU tier: the MX-quantized dynamic KV cache (torchmx_b200/kv_cache.py: MXDynamicCache) and the mode of K4b that reads it in
place, `attention_ops.flash_attention(..., kv_len=L)` on buffers pitched for a capacity.

Kernel level, the bar is the definition of that mode: with n = ceil128(L), the result of the call without kv_len on contiguous copies
of the first n keys with the tail and the causal rule folded into the mask (`attention_ops.ragged_operands`).  Up to 32768 keys that
call is checked against the K3 -> K4a -> K3 chain on the same copies (P bit for bit, output up to the sign of a zero); beyond, P
against the PyTorch restatement of the chain in K4a's order and the output within the fp64 bound of
tests/test_gpu_flash_attention_long.py.  Model level, logits with the cache equal those of the chain fallback at every step."""
import pytest
import torch

from tests.test_gpu_attention import _chain as _softmax_chain
from tests.test_gpu_flash_attention import _chain, _inputs, _quantize, _same_up_to_zero_sign
from tests.util import assert_bits_equal, bits_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SCALING = 128 ** -0.5
FMIN = torch.finfo(torch.bfloat16).min


@pytest.fixture(scope="module", autouse=True)
def _release_cached_blocks():
    yield
    torch.cuda.empty_cache()


def _as_bytes(t):
    """an MXTensor in the one-byte storage the caches hold (fp6 / fp4 as their exact E4M3 re-encoding)"""
    from torchmx_b200 import glue_ops, mx_gemm
    from torchmx_b200.mx_tensor import MXTensor
    codes, _ = mx_gemm._operand_rows(t._data, t._elem_dtype, None, packed=False)
    return MXTensor(t._scale_e8m0, codes.contiguous(), glue_ops.byte_operand_dtype(t._elem_dtype), 32, torch.bfloat16)


def _buffers(b, h, hk, q_len, kv_len, pitch, seed, elems=("float8_e4m3",) * 3, junk=False):
    """Q and K / Vt buffers of capacity `pitch` whose first kv_len keys exist; the tail holds zero codes or, with `junk`, random
    bytes (0xFF scales included) everywhere the kernel must not read"""
    q, k, v = _inputs(b, h, hk, q_len, pitch, seed=seed)
    q_mx, k_mx, vt_mx = _quantize(q, k, v, *elems)
    k_mx, vt_mx = _as_bytes(k_mx), _as_bytes(vt_mx)
    nb = -(-kv_len // 32)
    if junk:
        g = torch.Generator(device=DEV).manual_seed(seed + 1)
        rnd = lambda x: x.copy_(torch.randint(0, 256, x.shape, device=DEV, dtype=torch.int32, generator=g).to(torch.uint8))  # noqa: E731
        rnd(k_mx._data[:, :, kv_len:].view(torch.uint8))
        rnd(k_mx._scale_e8m0[:, :, kv_len:])
        rnd(vt_mx._data[..., kv_len:].view(torch.uint8))
        rnd(vt_mx._scale_e8m0[..., nb:])
        k_mx._scale_e8m0[:, :, kv_len:kv_len + 3] = 0xFF
        vt_mx._scale_e8m0[..., nb:nb + 1] = 0xFF
    else:
        k_mx._data[:, :, kv_len:].view(torch.uint8).zero_()
        vt_mx._data[..., kv_len:].view(torch.uint8).zero_()
    return q_mx, k_mx, vt_mx


def _run(q_mx, k_mx, vt_mx, kv_len, mask, causal, p_dt):
    from torchmx_b200 import attention_ops
    before = attention_ops.stats["flash_attention"]
    res = attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, mask, causal, p_dt, 32, return_probs=True, kv_len=kv_len)
    assert res is not None and attention_ops.stats["flash_attention"] == before + 1
    return res


def _check(q_mx, k_mx, vt_mx, kv_len, mask, causal, p_dt):
    """flash_attention(kv_len=...) against the chain on ragged_operands(...)"""
    from torchmx_b200 import attention_ops
    from torchmx_b200.mx_tensor import MXTensor
    out, probs = _run(q_mx, k_mx, vt_mx, kv_len, mask, causal, p_dt)
    n = -(-kv_len // 128) * 128
    assert probs._scale_e8m0.shape[-1] == n // 32
    k_n, vt_n, mask_n = attention_ops.ragged_operands(k_mx, vt_mx, kv_len, q_mx.shape[2], mask, causal)
    if n <= attention_ops.MAX_KV:
        want, p_ref = _chain(q_mx, k_n, vt_n, SCALING, mask_n, False, p_dt)
        assert_bits_equal(bits_of(probs._scale_e8m0), bits_of(p_ref._scale_e8m0), "scales of P")
        assert_bits_equal(bits_of(probs._data), bits_of(p_ref._data), "codes of P")
        _same_up_to_zero_sign(out, want, "attention output")
        return out, probs
    from tests.test_gpu_flash_attention import _repeat
    groups = q_mx.shape[1] // k_n.shape[1]
    scores = torch.matmul(q_mx, _repeat(k_n, groups).transpose(2, 3))
    want = MXTensor.to_mx(_softmax_chain(scores, SCALING, mask_n, False, ordered=True), p_dt, 32)
    assert_bits_equal(bits_of(probs._scale_e8m0), bits_of(want._scale_e8m0), "scales of P")
    assert_bits_equal(bits_of(probs._data), bits_of(want._data), "codes of P")
    pd, vd = probs.to_dtype(torch.float32).double(), _repeat(vt_n, groups).to_dtype(torch.float32).double()
    ref, S = (pd @ vd.transpose(2, 3)).transpose(1, 2), (pd.abs() @ vd.abs().transpose(2, 3)).transpose(1, 2)
    bound = 2.0 ** -8 * ref.abs() + n / 32 * 2.0 ** -23 * S + 1e-30
    assert ((out.double() - ref).abs() / bound).max().item() <= 1.0
    return out, probs


def _left_pad(b, q_len, kv_len, step=7):
    m = torch.zeros(b, 1, q_len, kv_len, device=DEV, dtype=torch.bfloat16)
    for i in range(b):
        m[i, ..., :i * step] = FMIN
    if q_len > 1:
        m.masked_fill_(torch.ones(q_len, kv_len, dtype=torch.bool, device=DEV).triu_(kv_len - q_len + 1), FMIN)
    return m


CASES = [
    # b, h, hk, q_len, kv_len, pitch, masking
    (1, 2, 2, 1, 1, 128, "none"),
    (2, 8, 2, 1, 31, 1024, "none"),          # grouped decode view
    (2, 8, 2, 1, 33, 1024, "left_pad"),
    (1, 4, 1, 1, 127, 128, "none"),
    (2, 8, 2, 1, 129, 2048, "left_pad"),
    (3, 8, 2, 1, 1055, 2048, "none"),
    (1, 8, 2, 1, 8191, 8192, "left_pad"),
    (1, 8, 2, 1, 32769, 33792, "none"),      # n = 32896: beyond the chain
    (1, 2, 1, 3, 131071, 131072, "causal"),
    (1, 2, 2, 77, 77, 1024, "causal"),       # ragged causal prefill, one-tile variant
    (1, 2, 1, 1000, 1000, 1024, "causal"),   # ... two-tile variant
    (2, 2, 2, 200, 1000, 1024, "left_pad"),  # a chunked prefill behind a cached prefix, left padding
    (2, 4, 2, 40, 300, 384, "causal"),
    (1, 2, 2, 129, 129, 256, "causal"),
]


@pytest.mark.parametrize("b,h,hk,q_len,kv_len,pitch,masking", CASES)
def test_ragged_flash_attention_matches_its_definition(b, h, hk, q_len, kv_len, pitch, masking):
    import torchmx  # noqa: F401
    from torchmx_b200 import dtypes
    q_mx, k_mx, vt_mx = _buffers(b, h, hk, q_len, kv_len, pitch, seed=kv_len + q_len)
    mask = _left_pad(b, q_len, kv_len) if masking == "left_pad" else None
    _check(q_mx, k_mx, vt_mx, kv_len, mask, masking == "causal", dtypes.float8_e4m3)


@pytest.mark.parametrize("qd,kd,vd,pd", [("float6_e3m2", "float6_e2m3", "float4_e2m1", "float6_e3m2"), ("float4_e2m1", "float4_e2m1", "float6_e3m2", "float4_e2m1"),
                                        ("float8_e4m3", "float6_e3m2", "float8_e4m3", "float6_e2m3"), ("float8_e5m2", "float8_e4m3", "float8_e5m2", "float8_e5m2")])
@pytest.mark.parametrize("mode", ["False", "True"])
def test_ragged_flash_attention_every_element_type(qd, kd, vd, pd, mode, monkeypatch):
    import torchmx  # noqa: F401
    from torchmx_b200 import dtypes
    from torchmx_b200 import env_variables as env
    monkeypatch.setattr(env, "MX_EXACT_QUANTIZATION", mode)
    p_dt = dtypes.STR_TO_ELEM_DTYPE[pd]
    q_mx, k_mx, vt_mx = _buffers(1, 2, 1, 130, 1100, 1280, seed=5, elems=(qd, kd, vd))
    _check(q_mx, k_mx, vt_mx, 1100, None, True, p_dt)
    q_mx, k_mx, vt_mx = _buffers(2, 8, 2, 1, 601, 1024, seed=6, elems=(qd, kd, vd))
    _check(q_mx, k_mx, vt_mx, 601, _left_pad(2, 1, 601), False, p_dt)


def test_ragged_flash_attention_nan_and_saturated_rows():
    import torchmx  # noqa: F401
    from torchmx_b200 import dtypes
    from torchmx_b200.mx_tensor import MXTensor
    q, k, v = _inputs(1, 2, 2, 200, 1024, seed=3)
    q[0, 0, 5, 17] = float("nan")
    q[0, 1, 100] *= 64
    k[0, 1, 400] *= 64
    k[0, 0, 600:] = 0
    v[0, :, 600:] = 0
    q_mx, k_mx, vt_mx = _quantize(q, k, v, "float8_e4m3", "float8_e4m3", "float8_e4m3")
    out, _ = _check(q_mx, k_mx, vt_mx, 555, None, True, dtypes.float8_e4m3)
    assert bool(torch.isnan(out[0, 5, 0]).all())
    assert isinstance(q_mx, MXTensor)


@pytest.mark.parametrize("q_len,kv_len,masking", [(1, 1055, "left_pad"), (1, 200, "none"), (150, 977, "causal"), (64, 300, "left_pad")])
def test_ragged_flash_attention_never_reads_the_tail(q_len, kv_len, masking):
    """random bytes (0xFF scales included) in the K codes / scales and V codes past kv_len, and in the V scales of blocks wholly
    past it, change no bit of the output or of P"""
    import torchmx  # noqa: F401
    from torchmx_b200 import dtypes
    b, h, hk, pitch = 2, 8, 2, 2048
    mask = _left_pad(b, q_len, kv_len) if masking == "left_pad" else None
    clean = _run(*_buffers(b, h, hk, q_len, kv_len, pitch, seed=9), kv_len, mask, masking == "causal", dtypes.float8_e4m3)
    junk = _run(*_buffers(b, h, hk, q_len, kv_len, pitch, seed=9, junk=True), kv_len, mask, masking == "causal", dtypes.float8_e4m3)
    assert torch.equal(clean[0].view(torch.int16), junk[0].view(torch.int16))
    assert torch.equal(clean[1]._data, junk[1]._data) and torch.equal(clean[1]._scale_e8m0, junk[1]._scale_e8m0)


@pytest.mark.parametrize("q_len,masking", [(1, "none"), (1, "left_pad"), (256, "mask")])
def test_ragged_flash_attention_on_a_full_buffer_equals_the_plain_call(q_len, masking):
    import torchmx  # noqa: F401
    from torchmx_b200 import attention_ops, dtypes
    b, h, hk, kv = 2, 8, 2, 1024
    q_mx, k_mx, vt_mx = _buffers(b, h, hk, q_len, kv, kv, seed=11)
    mask = None
    if masking != "none":
        mask = _left_pad(b, q_len, kv)
    o1, p1 = attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, mask, False, dtypes.float8_e4m3, 32, return_probs=True)
    o2, p2 = _run(q_mx, k_mx, vt_mx, kv, mask, False, dtypes.float8_e4m3)
    assert torch.equal(o1.view(torch.int16), o2.view(torch.int16))
    assert torch.equal(p1._data, p2._data) and torch.equal(p1._scale_e8m0, p2._scale_e8m0)


def test_ragged_key_axis_without_a_pitch_is_still_declined():
    import torchmx  # noqa: F401
    from torchmx_b200 import attention_ops, dtypes
    q, k, v = _inputs(1, 4, 2, 1, 1000, seed=1)
    q_mx, k_mx, vt_mx = _quantize(q, k, v, "float8_e4m3", "float8_e4m3", "float8_e4m3")
    assert attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, None, False, dtypes.float8_e4m3, 32) is None


# ---------------------------------------------------------------- model level

def _model(impl, seed=0):
    from transformers import LlamaConfig, LlamaForCausalLM
    import torchmx  # noqa: F401
    from torchmx.config import MXConfig, QAttentionConfig, QLinearConfig
    from torchmx.quant_api import quantize_llm_
    cfg = LlamaConfig(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, vocab_size=512,
                      max_position_embeddings=4096)
    cfg._attn_implementation = impl
    torch.manual_seed(seed)
    model = LlamaForCausalLM(cfg).to(DEV, torch.bfloat16).eval()
    lin = QLinearConfig(weights_config=MXConfig("float8_e4m3", 32), activations_config=MXConfig("float8_e4m3", 32))
    e = MXConfig("float8_e4m3", 32)
    quantize_llm_(model, QAttentionConfig(projection_config=lin, query_config=e, key_config=e, value_config=e, attention_weights_config=e), lin)
    return model, cfg


def _check_cache_codes(mx_cache, bf16_cache):
    """the MX cache holds exactly to_mx(K) and K5d(V) of the bf16 cache's rotated keys and values -- in the first layer, whose
    keys and values do not depend on how the attention of the two runs was computed"""
    from torchmx_b200 import glue_ops, mx_gemm
    from torchmx_b200.mx_tensor import MXTensor
    from torchmx_b200.dtypes import float8_e4m3
    for mx_layer, layer in zip(mx_cache.layers[:1], bf16_cache.layers[:1]):
        L = mx_layer.length
        assert L == layer.keys.shape[2]
        n = -(-L // 32) * 32
        keys = torch.nn.functional.pad(layer.keys, (0, 0, 0, n - L))
        values = torch.nn.functional.pad(layer.values, (0, 0, 0, n - L))
        k = MXTensor.to_mx(keys.contiguous(), float8_e4m3, 32)
        vt = glue_ops.quantize_transposed(values, float8_e4m3)
        assert torch.equal(mx_layer.k_codes[:, :, :n], k._data.view(torch.uint8)) and torch.equal(mx_layer.k_scales[:, :, :n], k._scale_e8m0)
        codes, _ = mx_gemm._operand_rows(vt._data, float8_e4m3, None, packed=False)
        assert torch.equal(mx_layer.vt_codes[..., :n], codes.view(torch.uint8)) and torch.equal(mx_layer.vt_scales[..., :n // 32], vt._scale_e8m0)
        assert not mx_layer.k_codes[:, :, n:].any() and not mx_layer.vt_codes[..., n:].any()


def _steps(model, cfg, cache, ids, attn, chunks):
    out = []
    for lo, hi in chunks:
        with torch.no_grad():
            out.append(model(input_ids=ids[:, lo:hi], attention_mask=attn[:, :hi], past_key_values=cache, use_cache=True).logits)
    return out


@pytest.mark.parametrize("impl", ["eager", "sdpa"])
def test_mx_dynamic_cache_logits_equal_the_fallback_at_every_step(impl):
    """left-padded ragged prefill, 44 decode steps crossing 32 / 128 and a capacity growth (initial capacity 128), a multi-token
    append; the same logits with K4b reading the cache in place as with the chain on copies, whatever the initial capacity, and
    the cache's codes are those of the bf16 DynamicCache"""
    from transformers import DynamicCache
    from torchmx_b200 import attention_ops
    from torchmx_b200.kv_cache import MXDynamicCache
    model, cfg = _model(impl)
    b = 3
    ids = torch.randint(0, cfg.vocab_size, (b, 160), device=DEV)
    attn = torch.ones(b, 160, dtype=torch.long, device=DEV)
    attn[1, :5] = 0
    attn[2, :17] = 0
    chunks = [(0, 101)] + [(i, i + 1) for i in range(101, 145)] + [(145, 160)]
    cache = MXDynamicCache(cfg, initial_capacity=128)
    flash, bf16 = [], DynamicCache(config=cfg)
    for lo, hi in chunks:
        with torch.no_grad():
            flash.append(model(input_ids=ids[:, lo:hi], attention_mask=attn[:, :hi], past_key_values=cache, use_cache=True).logits)
            model(input_ids=ids[:, lo:hi], attention_mask=attn[:, :hi], past_key_values=bf16, use_cache=True)
        _check_cache_codes(cache, bf16)
    assert cache.layers[0].capacity == 256 and cache.get_seq_length() == 160
    prev = attention_ops.set_flash_attention(False)
    try:
        chain = _steps(model, cfg, MXDynamicCache(cfg, initial_capacity=128), ids, attn, chunks)
    finally:
        attention_ops.set_flash_attention(prev)
    other = _steps(model, cfg, MXDynamicCache(cfg), ids, attn, chunks)  # initial capacity 1024: no growth
    for a, c, o in zip(flash, chain, other):
        _same_up_to_zero_sign(a, c, "logits")
        _same_up_to_zero_sign(a, o, "logits")


def test_mx_dynamic_cache_aligned_forwards_equal_the_bf16_dynamic_cache():
    """when every forward's key length is a multiple of 128, the cache read in place is the quantization of the bf16 cache with
    nothing hidden: the logits equal those of the bf16 DynamicCache path"""
    from transformers import DynamicCache
    from torchmx_b200.kv_cache import MXDynamicCache
    model, cfg = _model("sdpa")
    ids = torch.randint(0, cfg.vocab_size, (2, 384), device=DEV)
    attn = torch.ones(2, 384, dtype=torch.long, device=DEV)
    chunks = [(0, 128), (128, 256), (256, 384)]
    a = _steps(model, cfg, MXDynamicCache(cfg, initial_capacity=128), ids, attn, chunks)
    c = _steps(model, cfg, DynamicCache(config=cfg), ids, attn, chunks)
    for x, y in zip(a, c):
        _same_up_to_zero_sign(x, y, "logits")


@pytest.mark.parametrize("num_beams", [1, 2])
def test_mx_dynamic_cache_generate(num_beams):
    from torchmx_b200 import attention_ops
    from torchmx_b200.kv_cache import MXDynamicCache
    model, cfg = _model("sdpa")
    ids = torch.randint(0, cfg.vocab_size, (2, 37), device=DEV)
    attn = torch.ones_like(ids)
    attn[1, :4] = 0
    kw = dict(attention_mask=attn, max_new_tokens=40, do_sample=False, num_beams=num_beams, pad_token_id=0)
    with torch.no_grad():
        got = model.generate(ids, past_key_values=MXDynamicCache(cfg, initial_capacity=128), **kw)
        prev = attention_ops.set_flash_attention(False)
        try:
            want = model.generate(ids, past_key_values=MXDynamicCache(cfg), **kw)
        finally:
            attention_ops.set_flash_attention(prev)
    assert torch.equal(got, want)


def test_mx_dynamic_cache_crop_reset_and_the_length_limit():
    from torchmx_b200.kv_cache import MXDynamicCache
    model, cfg = _model("sdpa")
    ids = torch.randint(0, cfg.vocab_size, (1, 80), device=DEV)
    cache = MXDynamicCache(cfg, initial_capacity=128)
    with torch.no_grad():
        model(input_ids=ids[:, :70], past_key_values=cache, use_cache=True)
        with pytest.raises(ValueError, match="closed value block"):
            cache.crop(50)
        cache.crop(64)
        assert cache.get_seq_length() == 64
        a = model(input_ids=ids[:, 64:80], past_key_values=cache, use_cache=True).logits
        fresh = MXDynamicCache(cfg)
        model(input_ids=ids[:, :64], past_key_values=fresh, use_cache=True)
        b = model(input_ids=ids[:, 64:80], past_key_values=fresh, use_cache=True).logits
        _same_up_to_zero_sign(a, b, "logits after crop")
        cache.reset()
        assert cache.get_seq_length() == 0 and not cache.layers[0].k_codes.any()
        layer = cache.layers[0]
        layer.length = 131072 - 2  # (only the length: an append past the kernel's longest key axis is refused before any work)
        with pytest.raises(ValueError, match="131072"):
            model(input_ids=ids[:, :3], past_key_values=cache, use_cache=True)
