"""GPU tier: K4b (csrc/mxq_flash_attention.cu) on long key axes -- rows whose block sums K4a adds as butterfly-reduced groups of 32
(sm::sum_layout 2: unmasked rows of more than 32 blocks, masked rows of more than 256) and rows of more than 64 key chunks (the
live-chunk table then holds slots of several chunks), up to attention_ops.MAX_FLASH_KV keys.

Up to 32768 keys the reference is the chain K3 bmm -> K4a -> K3 bmm (tests/test_gpu_flash_attention.py).  K4a refuses longer
rows, so beyond that P is compared with the PyTorch restatement of the chain in K4a's summation order (tests/test_gpu_attention.py),
and the output with the exact products of the kernel's own P, within an fp32 accumulation bound."""
import pytest
import torch

from tests.test_gpu_attention import _chain as _softmax_chain
from tests.test_gpu_flash_attention import _chain, _inputs, _quantize, _repeat, _same_up_to_zero_sign
from tests.util import assert_bits_equal, bits_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

SCALING = 128 ** -0.5
FMIN = torch.finfo(torch.bfloat16).min


@pytest.fixture(scope="module", autouse=True)
def _release_cached_blocks():
    """these tests allocate tens of GB (long score rows for the chain): hand the cached blocks back afterwards, so that later
    tests which measure allocated bytes see the allocator as the rest of the suite leaves it"""
    yield
    torch.cuda.empty_cache()


def _mask(b, q_len, kv_len, kind, seed=0):
    """additive bf16 masks: 'causal' (+ padded keys from kv_len - 70 when 'pad'), per-batch left padding for a decode row, or
    'scattered': everything hidden except a few chunks that differ between rows"""
    if kind in ("causal", "causal+pad"):
        m = torch.full((1, 1, q_len, kv_len), FMIN, device=DEV, dtype=torch.bfloat16).triu_(kv_len - q_len + 1)
        if kind == "causal+pad":
            m[..., kv_len - 70:] = FMIN
        return m
    if kind == "left_pad":
        m = torch.zeros(b, 1, q_len, kv_len, device=DEV, dtype=torch.bfloat16)
        for i in range(b):
            m[i, ..., :i * 3000] = FMIN
        return m
    assert kind == "scattered"
    g = torch.Generator(device="cpu").manual_seed(seed)
    m = torch.full((b, 1, q_len, kv_len), FMIN, device=DEV, dtype=torch.bfloat16)
    n_chunks = kv_len // 128
    for r in range(q_len):
        for c in torch.randint(0, n_chunks, (3,), generator=g).tolist():
            m[..., r, c * 128 + 17:c * 128 + 90] = 0
    return m


def _check_against_chain(b, h, hk, q_len, kv_len, mask, causal, seed):
    from torchmx_b200 import attention_ops, dtypes
    q, k, v = _inputs(b, h, hk, q_len, kv_len, seed=seed)
    q_mx, k_mx, vt_mx = _quantize(q, k, v, "float8_e4m3", "float8_e4m3", "float8_e4m3")
    before = attention_ops.stats["flash_attention"]
    res = attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, mask, causal, dtypes.float8_e4m3, 32, return_probs=True)
    assert res is not None and attention_ops.stats["flash_attention"] == before + 1
    out, probs = res
    want, p_ref = _chain(q_mx, k_mx, vt_mx, SCALING, mask, causal, dtypes.float8_e4m3)
    assert_bits_equal(bits_of(probs._scale_e8m0), bits_of(p_ref._scale_e8m0), "scales of P")
    assert_bits_equal(bits_of(probs._data), bits_of(p_ref._data), "codes of P")
    if kv_len % 128 == 0:
        _same_up_to_zero_sign(out, want, "attention output")
    else:  # the chain's P @ V goes through the dequantize GEMM: same products, another order (tests/test_gpu_flash_attention.py)
        pd, vd = p_ref.to_dtype(torch.float32).double(), _repeat(vt_mx, h // hk).to_dtype(torch.float32).double()
        ref, S = (pd @ vd.transpose(2, 3)).transpose(1, 2), (pd.abs() @ vd.abs().transpose(2, 3)).transpose(1, 2)
        for o in (out, want):
            assert int(((o.double() - ref).abs() > 2.0 ** -8 * ref.abs() + 2.0 ** -18 * S + 1e-30).sum()) == 0
    return out, probs


CASES = [
    # b, h, hk, q_len, kv_len, masking
    (2, 8, 2, 1, 1056, "none"),          # decode rows (grouped heads), 33 blocks: the first unmasked layout-2 length
    (1, 2, 2, 130, 1056, "none"),        # two query tiles
    (2, 8, 2, 1, 2048, "none"),
    (1, 2, 1, 130, 2048, "none"),
    (1, 8, 2, 1, 32768, "none"),         # 256 chunks: slots of 4 chunks
    (1, 2, 2, 130, 32768, "none"),
    (1, 2, 1, 8224, 8224, "causal"),     # implied-causal prefill, 257 blocks, ragged last chunk
    (1, 2, 1, 16384, 16384, "causal"),   # q_len == kv_len, 128 chunks: slots of 2
    (1, 2, 1, 2048, 12288, "causal+pad"),  # additive causal mask behind a cached prefix, padded keys at the end
    (4, 8, 2, 1, 32768, "left_pad"),     # a masked decode step against a 32768-key cache
    (1, 2, 2, 130, 32768, "scattered"),  # only a few chunks live: coarse slots that are partly live, two query tiles
    (1, 2, 2, 64, 32768, "scattered"),   # ... and the one-tile variant
]


@pytest.mark.parametrize("b,h,hk,q_len,kv_len,masking", CASES)
def test_long_flash_attention_matches_the_chain_bit_for_bit(b, h, hk, q_len, kv_len, masking):
    import torchmx  # noqa: F401
    mask = None if masking in ("none", "causal") else _mask(b, q_len, kv_len, masking, seed=kv_len)
    _check_against_chain(b, h, hk, q_len, kv_len, mask, masking == "causal", seed=q_len + kv_len)


@pytest.mark.parametrize("kv_len,masking", [(65536, "none"), (65536, "causal"), (131072, "none"), (131072, "mask")])
def test_flash_attention_beyond_the_softmax_kernel(kv_len, masking):
    """K4a refuses rows of more than 32768 keys: P against the restated chain in K4a's order, the output against the bmm of the
    kernel's own P"""
    import torchmx  # noqa: F401
    from torchmx_b200 import attention_ops, dtypes
    from torchmx_b200.mx_tensor import MXTensor
    q_len = 5
    q, k, v = _inputs(1, 1, 1, q_len, kv_len, seed=kv_len + len(masking))
    q_mx, k_mx, vt_mx = _quantize(q, k, v, "float8_e4m3", "float8_e4m3", "float8_e4m3")
    mask, causal = None, masking == "causal"
    if masking == "mask":
        g = torch.Generator(device=DEV).manual_seed(3)
        mask = torch.zeros(1, 1, q_len, kv_len, device=DEV, dtype=torch.bfloat16)
        mask.masked_fill_(torch.rand(1, 1, q_len, kv_len, device=DEV, generator=g) < 0.3, FMIN)
        mask[..., kv_len - 1000:] = FMIN  # padded keys
    res = attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, mask, causal, dtypes.float8_e4m3, 32, return_probs=True)
    assert res is not None
    out, probs = res
    scores = torch.matmul(q_mx, k_mx.transpose(2, 3))
    want = MXTensor.to_mx(_softmax_chain(scores, SCALING, mask, causal, ordered=True), dtypes.float8_e4m3, 32)
    assert_bits_equal(bits_of(probs._scale_e8m0), bits_of(want._scale_e8m0), "scales of P")
    assert_bits_equal(bits_of(probs._data), bits_of(want._data), "codes of P")
    # the bmm of the kernel's own P takes a few query rows over 65536+ keys in another accumulation order: both against the exact
    # products of the same codes.  Bound: the bf16 rounding of the output plus fp32 accumulation over kv_len / 32 MMA steps,
    # one rounding each (n u S; the 2^-18 S of tests/test_gpu_flash_attention.py is a typical, not a worst-case, error at this n)
    bmm = torch.matmul(probs, vt_mx.transpose(2, 3)).transpose(1, 2)
    pd, vd = probs.to_dtype(torch.float32).double(), vt_mx.to_dtype(torch.float32).double()
    ref, S = (pd @ vd.transpose(2, 3)).transpose(1, 2), (pd.abs() @ vd.abs().transpose(2, 3)).transpose(1, 2)
    bound = 2.0 ** -8 * ref.abs() + kv_len / 32 * 2.0 ** -23 * S + 1e-30
    for name, o in (("kernel", out), ("bmm", bmm)):
        excess = ((o.double() - ref).abs() / bound).max().item()
        assert excess <= 1.0, (name, excess)


@pytest.mark.parametrize("qd,kd,vd,pd", [("float6_e3m2", "float6_e2m3", "float4_e2m1", "float6_e3m2"), ("float4_e2m1", "float4_e2m1", "float6_e3m2", "float4_e2m1"),
                                        ("float8_e4m3", "float6_e3m2", "float8_e4m3", "float6_e2m3"), ("float8_e5m2", "float8_e4m3", "float8_e5m2", "float8_e5m2")])
@pytest.mark.parametrize("mode", ["False", "True"])
def test_long_flash_attention_every_element_type(qd, kd, vd, pd, mode, monkeypatch):
    import torchmx  # noqa: F401
    from torchmx_b200 import attention_ops, dtypes
    from torchmx_b200 import env_variables as env
    monkeypatch.setattr(env, "MX_EXACT_QUANTIZATION", mode)
    q, k, v = _inputs(1, 2, 1, 130, 9216, seed=7)  # causal, 288 blocks (layout 2), 72 chunks (slots of 2)
    q_mx, k_mx, vt_mx = _quantize(q, k, v, qd, kd, vd)
    p_dt = dtypes.STR_TO_ELEM_DTYPE[pd]
    out, probs = attention_ops.flash_attention(q_mx, k_mx, vt_mx, 0.09, None, True, p_dt, 32, return_probs=True)
    want, p_ref = _chain(q_mx, k_mx, vt_mx, 0.09, None, True, p_dt)
    assert_bits_equal(bits_of(probs._scale_e8m0), bits_of(p_ref._scale_e8m0), "scales of P")
    assert_bits_equal(bits_of(probs._data), bits_of(p_ref._data), "codes of P")
    _same_up_to_zero_sign(out, want, "attention output")


def test_long_flash_attention_nan_and_extreme_rows():
    import torchmx  # noqa: F401
    from torchmx_b200 import attention_ops, dtypes
    q, k, v = _inputs(1, 2, 2, 256, 8448, seed=3)
    q[0, 0, 5, 17] = float("nan")
    q[0, 1, 100] *= 64
    k[0, 1, 4000] *= 64
    q_mx, k_mx, vt_mx = _quantize(q, k, v, "float8_e4m3", "float8_e4m3", "float8_e4m3")
    out, probs = attention_ops.flash_attention(q_mx, k_mx, vt_mx, 0.09, None, True, dtypes.float8_e4m3, 32, return_probs=True)
    want, p_ref = _chain(q_mx, k_mx, vt_mx, 0.09, None, True, dtypes.float8_e4m3)
    assert_bits_equal(bits_of(probs._scale_e8m0), bits_of(p_ref._scale_e8m0), "scales of P")
    assert_bits_equal(bits_of(probs._data), bits_of(p_ref._data), "codes of P")
    assert bool(torch.isnan(out[0, 5, 0]).all()) and bool(torch.isnan(want[0, 5, 0]).all())
    _same_up_to_zero_sign(out, want, "attention output")


def test_long_flash_attention_declines_and_repeats():
    import torchmx  # noqa: F401
    from torchmx_b200 import attention_ops, dtypes
    q, k, v = _inputs(1, 4, 1, 1, attention_ops.MAX_FLASH_KV + 32, seed=2)
    q_mx, k_mx, vt_mx = _quantize(q, k, v, "float8_e4m3", "float8_e4m3", "float8_e4m3")
    assert attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, None, False, dtypes.float8_e4m3, 32) is None
    q, k, v = _inputs(1, 4, 1, 3, attention_ops.MAX_FLASH_KV, seed=2)
    q_mx, k_mx, vt_mx = _quantize(q, k, v, "float8_e4m3", "float8_e4m3", "float8_e4m3")
    mask = _mask(1, 3, attention_ops.MAX_FLASH_KV, "causal+pad")
    for m, causal in ((None, True), (mask, False)):
        o1, p1 = attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, m, causal, dtypes.float8_e4m3, 32, return_probs=True)
        o2, p2 = attention_ops.flash_attention(q_mx, k_mx, vt_mx, SCALING, m, causal, dtypes.float8_e4m3, 32, return_probs=True)
        assert torch.equal(o1.view(torch.int16), o2.view(torch.int16))
        assert torch.equal(p1._data, p2._data) and torch.equal(p1._scale_e8m0, p2._scale_e8m0)


def test_mx_attention_block_long_prefill_and_decode_use_the_flash_kernel():
    """a tiny quantize_llm_ Llama (head_dim 128, sdpa): an unpadded prefill of 8320 tokens (the implied-causal path) and a
    mask-free decode step against the DynamicCache are one K4b launch per layer each, and the logits equal the chain's.  (Batch 9
    x 2 kv heads: above attention_ops.CHAIN_DECODE_MAX_CTAS, where a decode step stays with K4b.)"""
    from transformers import DynamicCache, LlamaConfig, LlamaForCausalLM
    import torchmx  # noqa: F401
    from torchmx_b200 import attention_ops
    from torchmx.config import MXConfig, QAttentionConfig, QLinearConfig
    from torchmx.quant_api import quantize_llm_
    cfg = LlamaConfig(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=4, num_key_value_heads=2, vocab_size=512,
                      max_position_embeddings=16384)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    model = LlamaForCausalLM(cfg).to(DEV, torch.bfloat16).eval()
    lin = QLinearConfig(weights_config=MXConfig("float8_e4m3", 32), activations_config=MXConfig("float8_e4m3", 32))
    e = MXConfig("float8_e4m3", 32)
    quantize_llm_(model, QAttentionConfig(projection_config=lin, query_config=e, key_config=e, value_config=e, attention_weights_config=e), lin)
    ids = torch.randint(0, cfg.vocab_size, (9, 8320 + 127 + 1), device=DEV)

    def run():
        cache, logits, counts = DynamicCache(config=cfg), [], []
        # prefill (8320 = 65 chunks of 128 keys), 127 more tokens (a key axis the kernels do not take), one decode step at 8448 keys
        for lo, hi, checked in ((0, 8320, True), (8320, 8447, False), (8447, 8448, True)):
            before = dict(attention_ops.stats)
            with torch.no_grad():
                logits.append(model(input_ids=ids[:, lo:hi], past_key_values=cache, use_cache=True).logits)
            if checked:
                counts.append({key: attention_ops.stats[key] - before[key] for key in before})
        return logits, counts

    flash, counts = run()
    for c in counts:
        assert c == {"flash_attention": 2, "fused_softmax": 0, "unfused_softmax": 0}, c
    prev = attention_ops.set_flash_attention(False)
    try:
        chain, counts = run()
    finally:
        attention_ops.set_flash_attention(prev)
    assert all(c["flash_attention"] == 0 and c["fused_softmax"] == 2 for c in counts), counts
    for a, c in zip(flash, chain):
        _same_up_to_zero_sign(a, c, "logits")
