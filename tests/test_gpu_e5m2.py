"""GPU tier: every kernel that reads or writes float8_e5m2 against an independent reference of the same operation.

float8_e5m2 is a labelled extension element type with no reference output to match.  Each test here compares a kernel directly
with the C oracle (oracle/mx_oracle.c) or with the torch restatement of tests/test_e5m2_reference.py -- which are pinned to each
other on the CPU -- on the kernel's own inputs, never with K1.  So an error in the e5m2 arithmetic the kernels share (the scale
rule, the saturation, the NaN-block rule, the decode) cannot hide behind two kernels that agree with each other.

e5m2 has no hardware-exact variant.  The host passes MXQ_FLAG_HW_EXACT only for the reference's element types, so for e5m2
MX_EXACT_QUANTIZATION never reaches a kernel: one test checks that every e5m2 entry ignores it, and K1's tests set the
kernel-level flag directly through the C entry, where the bytes must not change either."""
import numpy as np
import pytest
import torch

from oracle import grids
from tests.test_e5m2_reference import _block_size_sample, _e5m2_dequantize_ref, _e5m2_quantize_ref, _fp32_sample
from tests.test_gpu_attention import _chain as _softmax_chain
from tests.util import MODES, assert_bits_equal, bf16_tensor, bits_of

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
E5M2 = "float8_e5m2"
FMIN = torch.finfo(torch.bfloat16).min


@pytest.fixture(scope="module", autouse=True)
def _release_cached_blocks():
    """the 16384^2 tensors and the full grids take several GB: hand the cached blocks back afterwards"""
    yield
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def e5m2():
    import torchmx  # noqa: F401
    from torchmx_b200 import _C, dtypes
    _C.lib()
    return dtypes.float8_e5m2


def _k1(x: torch.Tensor, bs: int, hw_exact: bool):
    """K1 through its C entry (mxq_quantize), with MXQ_FLAG_HW_EXACT set or not -> (scales, codes) numpy"""
    from torchmx_b200 import _C, dtypes
    from torchmx_b200.mx_tensor import _HP_ID, _stream_ptr
    n_blocks = x.numel() // bs
    scales = torch.empty(x.shape[:-1] + (x.shape[-1] // bs,), dtype=torch.uint8, device=DEV)
    codes = torch.empty(x.shape, dtype=torch.uint8, device=DEV)
    rc = _C.lib().mxq_quantize(x.data_ptr(), _HP_ID[x.dtype], n_blocks, bs, dtypes.ELEM_ID[E5M2], _C.FLAG_HW_EXACT if hw_exact else 0,
                               codes.data_ptr(), scales.data_ptr(), x.device.index, _stream_ptr(x))
    _C.check(rc, "mxq_quantize")
    torch.cuda.synchronize()
    return bits_of(scales), bits_of(codes)


def _misaligned(x: torch.Tensor) -> torch.Tensor:
    """a copy of x at a 2- / 4-byte offset from a 32-byte boundary: K1 takes its element-wise kernels"""
    pad = torch.empty(x.numel() + 8, dtype=x.dtype, device=DEV)
    mis = pad[1:1 + x.numel()].view(x.shape)
    mis.copy_(x)
    return mis


def _oracle_mx(oracle, x: torch.Tensor, bs: int = 32):
    """the oracle's (scales, codes) of a bf16 tensor, blocks along its last dim"""
    return oracle.quantize(bits_of(x.contiguous()), E5M2, bs, threads=8)


def _check_mx(got, want, what=""):
    """got: MXTensor, or (scales, codes) as tensors or numpy arrays; want: the oracle's (scales, codes)"""
    s, c = (got._scale_e8m0, got._data) if hasattr(got, "_data") else got
    s, c = (t if isinstance(t, np.ndarray) else bits_of(t) for t in (s, c))
    assert_bits_equal(s.reshape(want[0].shape), want[0], f"{what} scales")
    assert_bits_equal(c.reshape(want[1].shape), want[1], f"{what} codes")


# ---- K1: quantize -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("hw_exact", [False, True])
def test_quantize_exhaustive_grid(e5m2, oracle, hw_exact):
    """every bf16 bit pattern under every block exponent, Inf / NaN leads included (17.5 M elements), block 32"""
    grid = grids.quant_grid()
    scales, codes = _k1(bf16_tensor(grid, DEV), 32, hw_exact)
    o_scales, o_codes = oracle.quantize(grid, E5M2, 32, threads=8)
    assert_bits_equal(scales, o_scales, "scales vs oracle")
    assert_bits_equal(codes, o_codes, "codes vs oracle")


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("bs", [8, 16, 64, 128])
def test_quantize_vector_kernel_other_block_sizes(e5m2, oracle, bs, mode, monkeypatch):
    """block sizes 8 / 16 / 64 / 128: the vectorised kernel and, through a misaligned view, the element-wise kernels"""
    from torchmx_b200 import env_variables as env
    monkeypatch.setattr(env, "MX_EXACT_QUANTIZATION", MODES[mode])
    bits = _block_size_sample(bs)
    want = oracle.quantize(bits, E5M2, bs)
    x = bf16_tensor(bits, DEV)
    for name, src in (("vector", x), ("element-wise", _misaligned(x))):
        _check_mx(torch.ops.torchmx.quantize_mx(src, E5M2, bs), want, f"block {bs} {name}")
        _check_mx(_k1(src, bs, mode == "hw_exact"), want, f"block {bs} {name}, C entry")


@pytest.mark.parametrize("bs", [2, 4, 7])
def test_quantize_generic_block_sizes(e5m2, oracle, bs):
    """block sizes that are not a multiple of 8 run the generic kernel: the structured cases (normal, saturated and subnormal
    targets, bf16 subnormal inputs) where the grid has them, and random patterns with Inf / NaN blocks"""
    rng = np.random.default_rng(100 + bs)
    bits = rng.integers(0, 65536, size=(301, 12 * bs), dtype=np.uint16)
    bits[(bits & 0x7F80) == 0x7F80] &= 0x3FFF
    bits[4, 1], bits[9, bs + 1], bits[300, -1] = 0x7F80, 0xFF80, 0xFFC1
    inputs = [bits]
    case = grids.structured_cases().get(f"bs{bs}")
    if case is not None:
        inputs.append(case[0])
    for x in inputs:
        want = oracle.quantize(x, E5M2, bs)
        for hw_exact in (False, True):
            _check_mx(_k1(bf16_tensor(x, DEV), bs, hw_exact), want, f"block {bs} {x.shape}")
        assert_bits_equal(want[1], _e5m2_quantize_ref(x, bs)[1], "oracle vs torch restatement")


def test_quantize_shapes_and_tails(e5m2, oracle):
    """ragged sizes: block counts that are not multiples of the CTA / warp tile, 1 block, 3-D"""
    rng = np.random.default_rng(7)
    for shape in [(1, 32), (3, 32), (1, 64), (5, 96), (17, 2080), (2, 3, 160), (1000, 32), (257, 4128)]:
        bits = rng.integers(0, 65536, size=shape, dtype=np.uint16)
        bits[(bits & 0x7F80) == 0x7F80] &= 0x3FFF
        want = oracle.quantize(bits, E5M2, 32)
        for hw_exact in (False, True):
            _check_mx(_k1(bf16_tensor(bits, DEV), 32, hw_exact), want, f"{shape}")


def test_quantize_fp32_input_against_the_torch_restatement(e5m2):
    """float32 input (block-32 fast kernel and element-wise kernels) against torch's own float8_e5m2 cast"""
    x = _fp32_sample()
    want = _e5m2_quantize_ref(x, 32)
    xt = torch.from_numpy(x.copy()).to(DEV)
    for name, src in (("fast", xt), ("element-wise", _misaligned(xt))):
        _check_mx(torch.ops.torchmx.quantize_mx(src, E5M2, 32), want, name)


def test_full_size_sample_and_idempotence(e5m2, oracle):
    """16384 x 16384 bf16 with a per-row exponent spread: quantizing the dequantized tensor reproduces codes and scales, and a
    strided sample of rows equals the oracle bit for bit, dequantized values included"""
    from torchmx_b200.mx_tensor import MXTensor
    g = torch.Generator(device=DEV).manual_seed(0)
    x = torch.randn(16384, 16384, dtype=torch.bfloat16, device=DEV, generator=g)
    x *= torch.exp2(torch.randint(-40, 40, (16384, 1), device=DEV, generator=g).to(torch.float32)).to(torch.bfloat16)
    m = MXTensor.to_mx(x, e5m2, 32)
    y = m.to_dtype(torch.bfloat16)
    m2 = MXTensor.to_mx(y, e5m2, 32)
    assert torch.equal(m2._data, m._data) and torch.equal(m2._scale_e8m0, m._scale_e8m0)
    rows = torch.arange(0, 16384, 1031, device=DEV)
    s, c = _oracle_mx(oracle, x[rows])
    _check_mx((m._scale_e8m0[rows], m._data[rows]), (s, c), "sampled rows")
    assert_bits_equal(bits_of(y[rows]), oracle.dequantize(c, s, E5M2, 32, "bf16"), "dequantized rows")
    del y, m, m2, x


def test_hw_exact_flag_changes_nothing_in_nan_blocks(e5m2, oracle):
    """the hardware-exact NaN-block quirk of the reference's element types re-emits subnormal codes in a NaN-scale block; e5m2
    has no such variant: with or without the flag, every code of a NaN block is +0 (bf16 and fp32 sources)"""
    bits = grids.quant_grid(grids.LEADS[-4:])  # +Inf, -Inf, +NaN, -NaN leads: every block is a NaN block
    x = bf16_tensor(bits, DEV)
    for hw_exact in (False, True):
        for src in (x, x.float()):
            scales, codes = _k1(src, 32, hw_exact)
            assert (scales == 255).all() and not codes.any()


# ---- K2: dequantize -----------------------------------------------------------------------------------------------------------
def _dequant(codes, scales, bs, target, block_dim):
    td = torch.bfloat16 if target == "bf16" else torch.float32
    out = torch.ops.torchmx.dequantize_mx(codes, scales, E5M2, bs, td, block_dim)
    torch.cuda.synchronize()
    return bits_of(out)


@pytest.mark.parametrize("target", ["bf16", "f32"])
def test_dequantize_exhaustive_grid(e5m2, oracle, target):
    """every (code byte, scale) pair through the flat kernel, the +-Inf and NaN codes included"""
    codes, scales = grids.dequant_grid(E5M2)
    out = _dequant(torch.from_numpy(codes).to(DEV), torch.from_numpy(scales).to(DEV), 32, target, 1)
    want = oracle.dequantize(codes, scales, E5M2, 32, target, 1)
    want = want.view(np.uint32) if target == "f32" else want
    assert_bits_equal(out, want, "vs oracle")
    ref = _e5m2_dequantize_ref(codes, scales, 32, target)
    assert_bits_equal(out, ref.view(np.uint32) if target == "f32" else ref, "vs torch restatement")


@pytest.mark.parametrize("target", ["bf16", "f32"])
def test_dequantize_transposed_vector_kernel_every_scale(e5m2, oracle, target):
    """the vectorised transposing kernel (block 32, blocked axis physically innermost, logically second-to-last): every scale
    byte incl. 0, 254 and 255, every code byte, ragged logical columns, batches"""
    rng = np.random.default_rng(17)
    for shape, perm in (((257, 512), (1, 0)), ((3, 70, 256), (0, 2, 1))):
        codes = rng.integers(0, 256, size=shape, dtype=np.uint8)
        scales = rng.integers(0, 256, size=shape[:-1] + (shape[-1] // 32,), dtype=np.uint8)
        bd = perm.index(len(shape) - 1)
        out = _dequant(torch.from_numpy(codes).to(DEV).permute(perm), torch.from_numpy(scales).to(DEV).permute(perm), 32, target, bd)
        want = oracle.dequantize(np.transpose(codes, perm), np.transpose(scales, perm), E5M2, 32, target, bd)
        assert_bits_equal(out, want.view(np.uint32) if target == "f32" else want, f"{shape} perm {perm}")


@pytest.mark.parametrize("target", ["bf16", "f32"])
def test_dequantize_strided_views(e5m2, oracle, target):
    """block_dim != last, permuted views, odd block sizes (the strided and transposing kernels)"""
    rng = np.random.default_rng(3)
    for (shape, bs, perm) in [((6, 64), 32, (1, 0)), ((2, 3, 40, 64), 32, (0, 1, 3, 2)), ((4, 70, 96), 32, (0, 2, 1)),
                              ((5, 12), 4, (1, 0)), ((3, 8, 6), 6, (2, 0, 1)), ((130, 192), 32, (1, 0))]:
        codes = rng.integers(0, 256, size=shape, dtype=np.uint8)
        scales = rng.integers(100, 150, size=shape[:-1] + (shape[-1] // bs,), dtype=np.uint8)
        bd = perm.index(len(shape) - 1)
        c_t, s_t = torch.from_numpy(codes).to(DEV).permute(perm), torch.from_numpy(scales).to(DEV).permute(perm)
        td = torch.bfloat16 if target == "bf16" else torch.float32
        out = torch.ops.torchmx.dequantize_mx(c_t, s_t, E5M2, bs, td, bd)
        assert out.is_contiguous()
        want = oracle.dequantize(np.transpose(codes, perm), np.transpose(scales, perm), E5M2, bs, target, bd)
        assert_bits_equal(bits_of(out), want.view(np.uint32) if target == "f32" else want, f"{shape} perm {perm}")


# ---- fused producers ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rows,hidden", [(67, 4096), (1024, 3072)])
def test_rmsnorm_to_mx(e5m2, oracle, rows, hidden):
    """K5a: the codes of the kernel's own bf16 output y; an Inf input row makes NaN blocks, a huge weight Inf blocks"""
    from torchmx_b200 import glue_ops
    g = torch.Generator(device=DEV).manual_seed(3)
    x = torch.randn(rows, hidden, device=DEV, dtype=torch.bfloat16, generator=g)
    x *= torch.exp2(torch.randint(-30, 30, (rows, hidden // 32), device=DEV, generator=g).float()).repeat_interleave(32, -1).to(torch.bfloat16)
    x[5, 100] = float("inf")   # row statistic inf -> rsqrt 0 -> 0 * inf = NaN
    x[9, 7] = float("nan")
    w = torch.randn(hidden, device=DEV, dtype=torch.bfloat16, generator=g)
    w[200] = 3e38              # y overflows to +-Inf in that column wherever |norm(x)| > ~1.13
    res = torch.randn(rows, hidden, device=DEV, dtype=torch.bfloat16, generator=g)
    y, mx, _ = glue_ops.rmsnorm(x, w, 1e-6, residual=res, to_mx=e5m2)
    assert bool(torch.isinf(y).any()) and bool(torch.isnan(y).any())
    want = _oracle_mx(oracle, y)
    _check_mx(mx, want, "rmsnorm")
    assert (want[0] == 255).sum() > 2
    _, mx2, _ = glue_ops.rmsnorm(x, w, 1e-6, residual=res, to_mx=e5m2, want_y=False)
    _check_mx(mx2, want, "rmsnorm, codes only")


@pytest.mark.parametrize("shape", [(1, 32, 2048, 128), (32, 8, 1, 128), (2, 3, 77, 64), (1, 2, 5, 32)])
def test_quantize_heads(e5m2, oracle, shape):
    """K5c: the oracle on the transposed reshape [b, t, h * d]"""
    from torchmx_b200 import glue_ops
    b, h, t, d = shape
    g = torch.Generator(device=DEV).manual_seed(t)
    x = torch.randn(*shape, device=DEV, dtype=torch.bfloat16, generator=g)
    x *= torch.exp2(torch.randint(-20, 20, (b, h, t, d // 32), device=DEV, generator=g).float()).repeat_interleave(32, -1).to(torch.bfloat16)
    x[0, 0, 0, 3] = float("nan")
    x[-1, -1, -1, -1] = float("inf")
    got = glue_ops.quantize_heads(x, e5m2)
    assert got is not None
    _check_mx(got, _oracle_mx(oracle, x.transpose(1, 2).reshape(b, t, h * d)), f"{shape}")


@pytest.mark.parametrize("shape,cache_len", [((32, 8, 256, 128), 0), ((2, 3, 96, 64), 160), ((1, 2, 32, 40), 0), ((3, 1, 416, 72), 512)])
def test_quantize_transposed(e5m2, oracle, shape, cache_len):
    """K5d: V quantized along the sequence axis, also from a slice of a longer cache; the oracle on the transposed copy"""
    from torchmx_b200 import glue_ops
    b, h, kv, d = shape
    g = torch.Generator(device=DEV).manual_seed(kv + d)
    full = torch.randn(b, h, max(cache_len, kv), d, device=DEV, dtype=torch.bfloat16, generator=g)
    full *= torch.exp2(torch.randint(-20, 20, (b, h, full.shape[2] // 32, 1, d), device=DEV, generator=g).float()).expand(-1, -1, -1, 32, -1).reshape(full.shape).to(torch.bfloat16)
    x = full[:, :, :kv]
    x[0, 0, 3, 1] = float("nan")
    x[-1, -1, -1, -1] = float("-inf")
    x[0, -1, :32, 2] = 0
    got = glue_ops.quantize_transposed(x, e5m2)
    assert got is not None and got.shape == (b, h, d, kv)
    _check_mx(got, _oracle_mx(oracle, x.transpose(2, 3)), f"{shape} in {cache_len}")


@pytest.mark.parametrize("shape", [(1, 96), (3, 7, 96), (300, 1024), (2, 128, 14336)])
def test_silu_mul_to_mx(e5m2, oracle, shape):
    """K1b: the oracle on torch's bf16(bf16(silu(gate)) * up).  The first block holds the extreme gates, the last block a NaN
    gate and an Inf up element (NaN blocks); every shape keeps blocks in between that are finite, so the scale rule and the
    codes are checked too"""
    from torchmx_b200 import mlp_ops
    g = torch.Generator(device=DEV).manual_seed(11)
    gate = (torch.randn(*shape, device=DEV, generator=g) * 4).to(torch.bfloat16)
    up = (torch.randn(*shape, device=DEV, generator=g) * 2).to(torch.bfloat16)
    gate.view(-1)[:8] = torch.tensor([0.0, -0.0, 88.0, -88.0, -120.0, 3e38, -3e38, 1e-30], device=DEV).to(torch.bfloat16)
    gate.view(-1)[-5] = float("nan")
    up.view(-1)[-20] = float("inf")
    got = mlp_ops.silu_mul_to_mx(gate, up, e5m2, 32)
    assert got is not None
    want = _oracle_mx(oracle, torch.nn.functional.silu(gate) * up)
    _check_mx(got, want, f"{shape}")
    assert want[0].reshape(-1)[-1] == 255 and (want[0] != 255).sum() >= want[0].size - 2


def _softmax_scores(b, h, q, kv, mode, seed):
    """bf16 scores with a NaN and a +Inf score (NaN rows) and, for 'mask', an additive mask of 0 / finfo.min / -inf"""
    g = torch.Generator(device=DEV).manual_seed(seed)
    scores = (torch.randn(b, h, q, kv, device=DEV, generator=g) * 24).to(torch.bfloat16)
    scores[0, 0, 0, kv // 3] = float("nan")
    scores[-1, -1, -1, kv - 1] = float("inf")
    mask = None
    if mode == "mask":
        r = torch.rand(b, h, q, kv, device=DEV, generator=g)
        mask = torch.zeros(b, h, q, kv, device=DEV, dtype=torch.bfloat16)
        mask.masked_fill_(r < 0.3, FMIN)
        mask.masked_fill_(r > 0.8, float("-inf"))
        mask[..., 0] = 0
    return scores, mask


@pytest.mark.parametrize("shape,mode", [
    ((2, 3, 64, 32), "none"), ((1, 2, 40, 96), "causal"), ((2, 2, 17, 160), "mask"), ((1, 4, 128, 1024), "causal"),
    ((1, 2, 50, 1024), "none"), ((1, 1, 20, 2080), "none"), ((1, 1, 8, 4096), "mask"), ((1, 1, 9, 8192), "mask"),
    ((1, 1, 5, 8224), "causal"), ((1, 1, 4, 16384), "mask"), ((1, 1, 3, 32768), "none"),
])
def test_softmax_to_mx(e5m2, oracle, shape, mode):
    """K4a with P e5m2: the bf16 probabilities of the chain restated in K4a's summation order, quantized by the oracle.  No mask,
    implied causal and additive masks (finfo.min and -inf) cover the kernel's three thread layouts."""
    from torchmx_b200 import attention_ops
    scores, mask = _softmax_scores(*shape, mode, seed=sum(shape))
    causal = mode == "causal"
    got = attention_ops.softmax_to_mx(scores, 128 ** -0.5, mask, causal, e5m2, 32)
    assert got is not None
    want = _oracle_mx(oracle, _softmax_chain(scores, 128 ** -0.5, mask, causal, ordered=True))
    _check_mx(got, want, f"{shape} {mode}")
    assert want[0][0, 0, 0].tolist() == [255] * (shape[3] // 32)


def test_host_entries_ignore_the_quantization_mode(e5m2):
    """MX_EXACT_QUANTIZATION selects the reference's hardware-exact cast, which e5m2 does not have: every host entry that
    produces e5m2 codes returns the same bytes under both values (the other tests run under the default only)"""
    from tests.test_gpu_kv_cache import _qconfig, _qkv
    from torchmx_b200 import attention_ops, env_variables as env, glue_ops, mlp_ops
    from torchmx_b200.kv_cache import MXStaticLayer
    from torchmx_b200.mx_tensor import MXTensor
    g = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn(64, 4096, device=DEV, dtype=torch.bfloat16, generator=g)
    x[3, 7], x[9, 300] = float("nan"), float("inf")
    w = torch.randn(4096, device=DEV, dtype=torch.bfloat16, generator=g)
    heads = x.view(2, 4, 32, 1024)[..., :128].contiguous()
    scores, mask = _softmax_scores(1, 2, 40, 1024, "mask", seed=5)
    q, k, v, cos, sin = _qkv(2, 37, 4, 2, g)

    def static_cache():
        layer = MXStaticLayer(128)
        q_mx, _, _ = layer.mx_append(q, k, v, cos, sin, _qconfig((E5M2, E5M2, E5M2)))
        return [q_mx._data, q_mx._scale_e8m0, layer.k_codes, layer.k_scales, layer.vt_codes, layer.vt_scales]

    def bytes_of(t):
        return [t._data, t._scale_e8m0]

    calls = {
        "to_mx": lambda: bytes_of(MXTensor.to_mx(x, e5m2, 32)),
        "rmsnorm": lambda: bytes_of(glue_ops.rmsnorm(x, w, 1e-6, to_mx=e5m2)[1]),
        "quantize_heads": lambda: bytes_of(glue_ops.quantize_heads(heads, e5m2)),
        "quantize_transposed": lambda: bytes_of(glue_ops.quantize_transposed(heads, e5m2)),
        "silu_mul_to_mx": lambda: bytes_of(mlp_ops.silu_mul_to_mx(x, x.flip(0), e5m2, 32)),
        "softmax_to_mx": lambda: bytes_of(attention_ops.softmax_to_mx(scores, 0.09, mask, False, e5m2, 32)),
        "static cache append": static_cache,
    }
    prev = env.MX_EXACT_QUANTIZATION
    try:
        for name, call in calls.items():
            env.MX_EXACT_QUANTIZATION = "False"
            a = call()
            env.MX_EXACT_QUANTIZATION = "True"
            b = call()
            assert all(torch.equal(t, u) for t, u in zip(a, b)), name
    finally:
        env.MX_EXACT_QUANTIZATION = prev


# ---- K5e: the static KV cache's append --------------------------------------------------------------------------------------
class _CacheReference:
    """rope -> bf16 static cache (zero-initialised) -> whole-cache quantization by the oracle: K along head_dim, V along the
    positions, Q along head_dim"""

    def __init__(self, oracle, b, hk, C):
        self.oracle = oracle
        self.keys = torch.zeros(b, hk, C, 128, dtype=torch.bfloat16, device=DEV)
        self.values = torch.zeros_like(self.keys)
        self.length = 0

    def append(self, q, k, v, cos, sin):
        from transformers.models.llama.modeling_llama import apply_rotary_pos_emb
        qr, kr = apply_rotary_pos_emb(q, k, cos, sin)
        t = k.shape[2]
        self.keys[:, :, self.length:self.length + t] = kr
        self.values[:, :, self.length:self.length + t] = v
        self.length += t
        return _oracle_mx(self.oracle, qr), _oracle_mx(self.oracle, self.keys), _oracle_mx(self.oracle, self.values.transpose(2, 3))


@pytest.mark.parametrize("lengths", [[37] + [1] * 60, [7, 45, 1]], ids=["prefill_then_decode", "append_45_at_7"])
def test_static_cache_append(e5m2, oracle, lengths):
    """K5e with e5m2 Q, K and V: a prefill then single-token appends across two V block boundaries, and a 45-token append at
    position 7; a NaN query, an Inf key and a NaN / Inf value (which stays in the open block for several appends)"""
    from tests.test_gpu_kv_cache import _qconfig, _qkv
    from torchmx_b200.kv_cache import MXStaticLayer
    b, hq, hk, C = 2, 4, 2, 128
    gen = torch.Generator(device=DEV).manual_seed(len(lengths))
    layer, ref = MXStaticLayer(C), _CacheReference(oracle, b, hk, C)
    for i, t in enumerate(lengths):
        q, k, v, cos, sin = _qkv(b, t, hq, hk, gen)
        if i == 1:
            q[0, 1, 0, 5] = float("nan")
            k[-1, 0, -1, 100] = float("inf")
            v[0, 0, 0, 3], v[-1, -1, 0, 70] = float("nan"), float("-inf")
        got_q, k_mx, vt_mx = layer.mx_append(q, k, v, cos, sin, _qconfig((E5M2, E5M2, E5M2)))
        want_q, want_k, want_v = ref.append(q, k, v, cos, sin)
        _check_mx(got_q, want_q, f"append {i}: Q")
        _check_mx((layer.k_scales, layer.k_codes), want_k, f"append {i}: K cache")
        _check_mx((layer.vt_scales, layer.vt_codes), want_v, f"append {i}: V cache")
        if i == 1:
            assert (want_q[0] == 255).any() and (want_k[0] == 255).any() and (want_v[0] == 255).any()


# ---- K4b: the fused attention kernel ---------------------------------------------------------------------------------------
def _exact_operand(oracle, shape, elem, seed):
    """an MXTensor built by the oracle from bf16 values of magnitude in [1, 16) (random sign, some zeros): the products of two
    such dequantized e5m2 / e4m3 operands are multiples of 2^-6 below 2^8, so every partial sum of a 128-term dot product is
    exact in fp32 and the bf16 scores do not depend on the accumulation order"""
    from torchmx_b200 import dtypes
    from torchmx_b200.mx_tensor import MXTensor
    g = torch.Generator(device="cpu").manual_seed(seed)
    mag = torch.exp2(torch.rand(shape, generator=g) * 4)
    x = torch.where(torch.rand(shape, generator=g) < 0.5, -mag, mag)
    x = torch.where(torch.rand(shape, generator=g) < 0.05, 0.0, x).to(torch.bfloat16)
    s, c = oracle.quantize(bits_of(x), elem, 32, threads=8)
    t = MXTensor(torch.from_numpy(s).to(DEV), torch.from_numpy(c).to(DEV), dtypes.STR_TO_ELEM_DTYPE[elem], 32, torch.bfloat16)
    return t, oracle.bf16_bits_to_f32(oracle.dequantize(c, s, elem, 32, "bf16"))


def _attention_reference(oracle, q_deq, k_deq, vt_deq, scaling, mask, causal, p_elem, groups):
    """P (oracle codes of the restated K4a chain on the exact bf16 scores) and the fp64 attention output of the dequantized
    operands, with the magnitude sum S of its bound"""
    q64 = torch.from_numpy(q_deq).double()
    k64 = torch.from_numpy(k_deq).double().repeat_interleave(groups, 1)
    vt64 = torch.from_numpy(vt_deq).double().repeat_interleave(groups, 1)
    scores = (q64 @ k64.transpose(2, 3)).float().to(torch.bfloat16).to(DEV)
    p_bf16 = _softmax_chain(scores, scaling, mask, causal, ordered=True)
    p_s, p_c = oracle.quantize(bits_of(p_bf16), p_elem, 32, threads=8)
    p64 = torch.from_numpy(oracle.bf16_bits_to_f32(oracle.dequantize(p_c, p_s, p_elem, 32, "bf16"))).double()
    ref = (p64 @ vt64.transpose(2, 3)).transpose(1, 2)
    S = (p64.abs() @ vt64.abs().transpose(2, 3)).transpose(1, 2)
    return (p_s, p_c), ref, S


@pytest.mark.parametrize("b,h,hk,q_len,kv_len,masking,qkv,p", [
    (1, 2, 2, 96, 256, "causal", E5M2, E5M2),               # one query tile per (batch, head): the one-tile variant
    (1, 4, 2, 300, 384, "causal", E5M2, "float8_e4m3"),     # three query tiles: the two-tile variant, grouped-query heads
    (1, 2, 2, 130, 512, "mask", "float8_e4m3", E5M2),       # additive mask: the table variant
    (2, 2, 2, 200, 640, "mask", E5M2, E5M2),
    (1, 4, 2, 5, 300, "ragged", E5M2, E5M2),                # a ragged key axis read in place from a 384-key capacity
])
def test_flash_attention(e5m2, oracle, b, h, hk, q_len, kv_len, masking, qkv, p):
    """K4b with e5m2 operands and / or e5m2 P: P's codes and scales against the restated K4a chain quantized by the oracle, the
    output against the fp64 attention of the oracle-dequantized operands and P (bound: the bf16 rounding of the output plus fp32
    accumulation over n / 32 MMA steps)"""
    from torchmx_b200 import attention_ops, dtypes
    from torchmx_b200.mx_tensor import MXTensor
    scaling = 2.0 ** -8
    ragged = masking == "ragged"
    pitch = -(-kv_len // 128) * 128 if ragged else kv_len
    seed = q_len + kv_len
    q_mx, q_deq = _exact_operand(oracle, (b, h, q_len, 128), qkv, seed)
    k_mx, k_deq = _exact_operand(oracle, (b, hk, pitch, 128), qkv, seed + 1)
    vt_mx, vt_deq = _exact_operand(oracle, (b, hk, 128, pitch), qkv, seed + 2)
    mask, causal = None, masking in ("causal", "ragged")
    if masking == "mask":
        g = torch.Generator(device=DEV).manual_seed(seed)
        r = torch.rand(b, 1, q_len, kv_len, device=DEV, generator=g)
        mask = torch.zeros(b, 1, q_len, kv_len, device=DEV, dtype=torch.bfloat16)
        mask.masked_fill_(r < 0.3, FMIN)
        mask.masked_fill_(r > 0.9, float("-inf"))
        mask[..., kv_len - 70:] = FMIN
        mask[..., 0] = 0
    p_dt = dtypes.STR_TO_ELEM_DTYPE[p]
    before = attention_ops.stats["flash_attention"]
    res = attention_ops.flash_attention(q_mx, k_mx, vt_mx, scaling, mask, causal, p_dt, 32, return_probs=True, kv_len=kv_len if ragged else None)
    assert res is not None and attention_ops.stats["flash_attention"] == before + 1
    out, probs = res
    if ragged:  # the defined result: the call on contiguous copies of the first ceil128(kv_len) keys with the tail masked
        k_n, vt_n, mask = attention_ops.ragged_operands(k_mx, vt_mx, kv_len, q_len, None, causal)
        causal = False
        deq = lambda t: oracle.bf16_bits_to_f32(oracle.dequantize(bits_of(t._data), bits_of(t._scale_e8m0), qkv, 32, "bf16"))  # noqa: E731
        k_deq, vt_deq = deq(k_n), deq(vt_n)
    want_p, ref, S = _attention_reference(oracle, q_deq, k_deq, vt_deq, scaling, mask, causal, p, h // hk)
    _check_mx(probs, want_p, "P")
    n = probs.shape[-1]
    bound = 2.0 ** -8 * ref.abs() + n / 32 * 2.0 ** -23 * S + 1e-30
    excess = ((out.double().cpu() - ref).abs() / bound).max().item()
    assert excess <= 1.0, excess
    assert isinstance(probs, MXTensor) and not torch.isnan(out).any()


# ---- K3: the MX matmul end to end -------------------------------------------------------------------------------------------
GEMM_CASES = [
    (64, 1000, 512, E5M2, E5M2, 0, 32),                     # M <= 128, not batched: the skinny weight-streaming kernel (K3c)
    (17, 700, 1024, "float4_e2m1", E5M2, 0, 32),
    (300, 520, 640, E5M2, "float6_e3m2", 0, 32),            # M, N > 128: see GEMM_RULES
    (257, 300, 384, E5M2, E5M2, 0, 32),
    (96, 120, 256, "float4_e2m1", E5M2, 2, 32),             # N <= 128: the single-CTA kernel (K3a), batched
    (200, 64, 256, E5M2, "float6_e3m2", 3, 32),
    (100, 200, 256, E5M2, E5M2, 0, 16),                     # block 16: the fused dequantize GEMM (K3d)
]
# M, N > 128 runs the CTA-pair kernel (K3b) only when its 256 x 256 tiles fill more than a quarter of the SMs; these small shapes
# would otherwise take 128 x 128 tiles of the single-CTA kernel (K3a).  "pair" sets MXQ_GEMM_WIDE_TILES, which switches that rule
# off, so K3b runs them; "auto" keeps the rule and runs them on K3a.
GEMM_RULES = [(*c, rule) for c in GEMM_CASES for rule in (("auto", "pair") if c[0] > 128 and c[1] > 128 and c[6] == 32 else ("auto",))]


@pytest.mark.parametrize("M,N,K,ea,eb,batch,bs,rule", GEMM_RULES)
def test_mx_matmul_against_the_oracle_end_to_end(e5m2, oracle, monkeypatch, M, N, K, ea, eb, batch, bs, rule):
    """K1 on both operands, then the GEMM, against the oracle's quantize -> dequantize -> double-accumulated contraction of the same
    bf16 bits; tolerance: the bf16 rounding of the output plus the fp32 accumulation order"""
    from torchmx_b200 import dtypes, mx_gemm
    from torchmx_b200.mx_tensor import MXTensor
    monkeypatch.setitem(mx_gemm.overrides, "wide_tiles", rule == "pair")  # mxq_gemm_args_t.flags: MXQ_GEMM_WIDE_TILES
    g = torch.Generator(device=DEV).manual_seed(M + N + K)
    sa, sb = ((batch, M, K), (batch, N, K)) if batch else ((M, K), (N, K))
    x = torch.randn(*sa, device=DEV, dtype=torch.bfloat16, generator=g) * 2
    w = torch.randn(*sb, device=DEV, dtype=torch.bfloat16, generator=g)
    w *= torch.exp2(torch.randint(-6, 6, (*sb[:-1], K // bs), device=DEV, generator=g).float()).repeat_interleave(bs, -1).to(torch.bfloat16)
    A, B = MXTensor.to_mx(x, dtypes.STR_TO_ELEM_DTYPE[ea], bs), MXTensor.to_mx(w, dtypes.STR_TO_ELEM_DTYPE[eb], bs)
    before = dict(mx_gemm.stats)
    out = torch.bmm(A, B.transpose(1, 2)) if batch else torch.nn.functional.linear(A, B)
    assert mx_gemm.stats["tensor_core" if bs == 32 else "dequant_gemm"] == before["tensor_core" if bs == 32 else "dequant_gemm"] + 1
    assert mx_gemm.stats["fallback"] == before["fallback"]
    xs, ws = bits_of(x).reshape(-1, M, K), bits_of(w).reshape(-1, N, K)
    for i in range(max(batch, 1)):
        deq = []
        for t, el in ((xs[i], ea), (ws[i], eb)):
            scales, codes = oracle.quantize(t, el, bs)
            deq.append(oracle.dequantize(codes, scales, el, bs, target="bf16"))
        ref = oracle.gemm_nt(deq[0], deq[1]).astype(np.float64)
        S = np.abs(oracle.bf16_bits_to_f32(deq[0]).astype(np.float64)) @ np.abs(oracle.bf16_bits_to_f32(deq[1]).astype(np.float64)).T
        err = np.abs(out.reshape(-1, M, N)[i].double().cpu().numpy() - ref)
        tol = 2.0 ** -8 * np.abs(ref) + 2.0 ** -18 * S + 1e-30
        assert (err <= tol).all(), f"batch {i}: {int((err > tol).sum())} of {err.size} outside tolerance"
