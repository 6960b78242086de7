"""GPU tier (pytest -m gpu): the CUDA kernels, called through the torchmx operator surface and
therefore through the C ABI, against the CPU oracle on identical inputs and against the digests /
fixtures produced by the unmodified reference (tests/golden).  Bit-exact: every comparison is
integer equality on codes, scales and output bit patterns (NaN payloads canonicalised)."""
import numpy as np
import pytest
import torch

from oracle import grids
from tests.util import ELEMS, FP_ELEMS, MODES, assert_bits_equal, bf16_tensor, bits_of, canon_nan, sha

pytestmark = pytest.mark.gpu

DEV = "cuda:0"


@pytest.fixture(scope="module")
def mx():
    import torchmx  # the drop-in alias of torchmx_b200
    from torchmx_b200 import _C
    _C.lib()  # fail loudly if the CUDA library is missing
    return torchmx


def _quant(bits, elem, bs, mode):
    from torchmx import env_variables as env
    env.MX_EXACT_QUANTIZATION = MODES[mode]
    scale, codes = torch.ops.torchmx.quantize_mx(bf16_tensor(bits, DEV), elem, bs)
    torch.cuda.synchronize()
    return bits_of(scale), bits_of(codes)


def _dequant(codes, scales, elem, bs, target, block_dim):
    td = torch.bfloat16 if target == "bf16" else torch.float32
    out = torch.ops.torchmx.dequantize_mx(torch.from_numpy(np.ascontiguousarray(codes)).to(DEV), torch.from_numpy(scales).to(DEV), elem, bs, td,
                                          block_dim)
    torch.cuda.synchronize()
    return bits_of(out)


# ---- quantize ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("elem", ELEMS)
def test_quantize_exhaustive_grid(mx, oracle, digests, elem, mode):
    """every bf16 bit pattern under every block exponent (17.5 M elements), block 32"""
    grid = grids.quant_grid()
    assert sha(grid) == digests["quant_grid_input"]
    scales, codes = _quant(grid, elem, 32, mode)
    o_scales, o_codes = oracle.quantize(grid, elem, 32, hw_exact=(mode == "hw_exact"), threads=8)
    assert_bits_equal(scales, o_scales, "scales vs oracle")
    assert_bits_equal(codes, o_codes, "codes vs oracle")
    assert sha(scales) == digests[f"quant_grid/{elem}/{mode}/scales"], "scales vs reference digest"
    assert sha(codes) == digests[f"quant_grid/{elem}/{mode}/codes"], "codes vs reference digest"


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("elem", ELEMS)
def test_quantize_structured_block_sizes(mx, fixtures, elem, mode):
    """block sizes 2..16 (generic kernels) against the reference's outputs"""
    for name, (bits, bs) in grids.structured_cases().items():
        key = f"struct/{name}/{elem}/{mode}/codes"
        if key not in fixtures:
            continue
        scales, codes = _quant(bits, elem, bs, mode)
        assert_bits_equal(scales, fixtures[f"struct/{name}/{elem}/{mode}/scales"], f"{name} scales")
        assert_bits_equal(codes, fixtures[key], f"{name} codes")


@pytest.mark.parametrize("elem", ELEMS)
def test_quantize_shapes_and_tails(mx, oracle, elem):
    """ragged sizes: block counts that are not multiples of the CTA / warp tile, 1 block, 3-D"""
    rng = np.random.default_rng(7)
    for shape in [(1, 32), (3, 32), (1, 64), (5, 96), (17, 2080), (2, 3, 160), (1000, 32), (257, 4128)]:
        bits = rng.integers(0, 65536, size=shape, dtype=np.uint16)
        bits[(bits & 0x7F80) == 0x7F80] &= 0x3FFF  # keep most blocks finite
        scales, codes = _quant(bits, elem, 32, "simulated")
        o_scales, o_codes = oracle.quantize(bits, elem, 32)
        assert_bits_equal(scales, o_scales, f"{shape} scales")
        assert_bits_equal(codes, o_codes, f"{shape} codes")


def test_quantize_empty_and_noncontiguous(mx, oracle):
    from torchmx import dtypes
    from torchmx.mx_tensor import MXTensor
    x = torch.empty(0, 64, dtype=torch.bfloat16, device=DEV)
    m = MXTensor.to_mx(x, dtypes.float8_e4m3, 32)
    assert m._data.shape == (0, 64) and m._scale_e8m0.shape == (0, 2)
    assert m.to_dtype(torch.bfloat16).shape == (0, 64)
    # non-contiguous input: the reference asserts (mx_tensor.py:62); we accept and match contiguous()
    base = torch.randn(64, 130, dtype=torch.bfloat16, device=DEV)
    v = base[:, 1:129:2]
    m = MXTensor.to_mx(v, dtypes.float6_e3m2, 32)
    s, c = oracle.quantize(bits_of(v.contiguous()), "float6_e3m2", 32)
    assert_bits_equal(bits_of(m._scale_e8m0), s)
    assert_bits_equal(bits_of(m._data), c)


def test_cpu_tensor_raises(mx):
    from torchmx import dtypes
    from torchmx.mx_tensor import MXTensor
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        MXTensor.to_mx(torch.randn(4, 32, dtype=torch.bfloat16), dtypes.int8, 32)


# ---- dequantize ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("target", ["bf16", "f32"])
@pytest.mark.parametrize("elem", ELEMS)
def test_dequantize_exhaustive_grid(mx, oracle, digests, elem, target):
    """every (code byte, scale) pair, both targets"""
    codes, scales = grids.dequant_grid(elem)
    out = _dequant(codes, scales, elem, 32, target, 1)
    want = oracle.dequantize(codes, scales, elem, 32, target, 1)
    want = want.view(np.uint32) if target == "f32" else want
    assert_bits_equal(out, want, "vs oracle")
    assert sha(canon_nan(out)) == digests[f"dequant_grid/{elem}/{target}"], "vs reference digest"


@pytest.mark.parametrize("target", ["bf16", "f32"])
@pytest.mark.parametrize("elem", ELEMS)
def test_dequantize_strided_views(mx, oracle, elem, target):
    """block_dim != last, permuted / expanded views, odd block sizes (strided + transposing kernels)"""
    rng = np.random.default_rng(3)
    td = torch.bfloat16 if target == "bf16" else torch.float32
    for (shape, bs, perm) in [((6, 64), 32, (1, 0)), ((2, 3, 40, 64), 32, (0, 1, 3, 2)), ((4, 70, 96), 32, (0, 2, 1)),
                              ((5, 12), 4, (1, 0)), ((3, 8, 6), 6, (2, 0, 1)), ((130, 192), 32, (1, 0))]:
        L = shape[-1]
        per = 2 if elem == "float4_e2m1" else 1
        hi = 64 if elem.startswith("float6") else 256
        codes = rng.integers(0, hi, size=shape[:-1] + (L // per,), dtype=np.uint8)
        scales = rng.integers(100, 150, size=shape[:-1] + (L // bs,), dtype=np.uint8)
        if elem == "int8":
            codes = codes.view(np.int8)
        bd = perm.index(len(shape) - 1)
        c_t = torch.from_numpy(codes).to(DEV).permute(perm)
        s_t = torch.from_numpy(scales).to(DEV).permute(perm)
        out = torch.ops.torchmx.dequantize_mx(c_t, s_t, elem, bs, td, bd)
        assert out.is_contiguous()
        want = oracle.dequantize(np.transpose(codes, perm), np.transpose(scales, perm), elem, bs, target, bd)
        want = want.view(np.uint32) if target == "f32" else want
        assert_bits_equal(bits_of(out), want, f"{shape} perm {perm}")


@pytest.mark.parametrize("target", ["bf16", "f32"])
@pytest.mark.parametrize("elem", ELEMS)
def test_dequantize_transposed_vector_kernel_every_scale(mx, oracle, elem, target):
    """the vectorised transposing kernel (block 32, blocked axis physically innermost, logically second-to-last -- what aten.t of a
    quantized weight gives): every scale byte incl. 0, 254 and 255 (NaN), every code, ragged logical columns, batches"""
    rng = np.random.default_rng(17)
    td = torch.bfloat16 if target == "bf16" else torch.float32
    per = 2 if elem == "float4_e2m1" else 1
    hi = 64 if elem.startswith("float6") else 256
    for shape, perm in (((257, 512), (1, 0)), ((3, 70, 256), (0, 2, 1))):
        codes = rng.integers(0, hi, size=shape[:-1] + (shape[-1] // per,), dtype=np.uint8)
        scales = rng.integers(0, 256, size=shape[:-1] + (shape[-1] // 32,), dtype=np.uint8)
        if elem == "int8":
            codes = codes.view(np.int8)
        bd = perm.index(len(shape) - 1)
        out = torch.ops.torchmx.dequantize_mx(torch.from_numpy(codes).to(DEV).permute(perm), torch.from_numpy(scales).to(DEV).permute(perm), elem, 32, td, bd)
        want = oracle.dequantize(np.transpose(codes, perm), np.transpose(scales, perm), elem, 32, target, bd)
        want = want.view(np.uint32) if target == "f32" else want
        assert_bits_equal(bits_of(out), want, f"{shape} perm {perm}")


# ---- MXTensor level (user API) against reference fixtures --------------------------------------------------
@pytest.mark.parametrize("elem", ELEMS)
def test_readme_example(mx, fixtures, elem):
    """BASELINE config 1"""
    from torchmx import dtypes, env_variables as env
    from torchmx.mx_tensor import MXTensor
    x = bf16_tensor(fixtures["readme/x"], DEV)
    for mode in MODES:
        env.MX_EXACT_QUANTIZATION = MODES[mode]
        m = MXTensor.to_mx(x, dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[elem], 32)
        assert_bits_equal(bits_of(m._scale_e8m0), fixtures[f"readme/{elem}/{mode}/scales"])
        assert_bits_equal(bits_of(m._data), fixtures[f"readme/{elem}/{mode}/codes"])
        assert m.shape == x.shape and m.dtype == torch.bfloat16
    assert_bits_equal(bits_of(m.to_dtype(torch.bfloat16)), fixtures[f"readme/{elem}/bf16"])
    assert_bits_equal(bits_of(m.to_dtype(torch.float32)), fixtures[f"readme/{elem}/f32"])


@pytest.mark.parametrize("elem", ELEMS)
def test_special_values(mx, fixtures, elem):
    from torchmx import dtypes, env_variables as env
    from torchmx.mx_tensor import MXTensor
    x = bf16_tensor(fixtures["special/x"], DEV)
    for mode in MODES:
        env.MX_EXACT_QUANTIZATION = MODES[mode]
        m = MXTensor.to_mx(x, dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[elem], 4)
        assert_bits_equal(bits_of(m._scale_e8m0), fixtures[f"special/{elem}/{mode}/scales"])
        assert_bits_equal(bits_of(m._data), fixtures[f"special/{elem}/{mode}/codes"])
        assert torch.isnan(m.to_dtype(torch.bfloat16)).all()


@pytest.mark.parametrize("elem", ELEMS)
def test_padding(mx, fixtures, elem):
    """last dim not a multiple of the block (reference: mx_tensor.py:218-248, 288-321)"""
    from torchmx import dtypes
    from torchmx.mx_tensor import MXTensor
    keys = sorted({k.split("/")[1] for k in fixtures.files if k.startswith("pad/")})
    assert keys
    for key in keys:
        bs = int(key.split("_bs")[1])
        x = bf16_tensor(fixtures[f"pad/{key}/x"], DEV)
        m = MXTensor.to_mx(x, dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[elem], bs)
        assert m._padding == int(fixtures[f"pad/{key}/{elem}/padding"][0])
        assert list(m.shape) == list(fixtures[f"pad/{key}/{elem}/shape"])
        assert_bits_equal(bits_of(m._scale_e8m0), fixtures[f"pad/{key}/{elem}/scales"], key)
        assert_bits_equal(bits_of(m._data), fixtures[f"pad/{key}/{elem}/codes"], key)
        assert_bits_equal(bits_of(m.to_dtype(torch.bfloat16)), fixtures[f"pad/{key}/{elem}/bf16"], key)


@pytest.mark.parametrize("elem", ELEMS)
def test_layout_ops(mx, fixtures, elem):
    """t / transpose / view then to_dtype (reference: tests/test_mx_tensor.py:195-356)"""
    from torchmx import dtypes
    from torchmx.mx_tensor import MXTensor
    et = dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[elem]
    x = bf16_tensor(fixtures["layout/x"], DEV)
    m = MXTensor.to_mx(x, et, 32)
    assert_bits_equal(bits_of(m.transpose(2, 3).to_dtype(torch.bfloat16)), fixtures[f"layout/{elem}/transpose23_bf16"])
    assert_bits_equal(bits_of(m.transpose(2, 3).to_dtype(torch.float32)), fixtures[f"layout/{elem}/transpose23_f32"])
    m2 = MXTensor.to_mx(x[0, 0], et, 32)
    assert_bits_equal(bits_of(m2.t().to_dtype(torch.bfloat16)), fixtures[f"layout/{elem}/t_bf16"])
    assert_bits_equal(bits_of(m.view(24, 64, 96).to_dtype(torch.bfloat16)), fixtures[f"layout/{elem}/view_bf16"])
    # exact equivalences the reference asserts with atol = rtol = 0
    assert torch.equal(m.transpose(2, 3).to_dtype(torch.bfloat16), m.to_dtype(torch.bfloat16).transpose(2, 3))
    assert torch.equal(m2.t().t().to_dtype(torch.bfloat16), m2.to_dtype(torch.bfloat16))


# ---- BASELINE config 2 size: properties that do not need the oracle at full size ----------------------
@pytest.mark.parametrize("elem", ELEMS)
def test_full_size_properties(mx, oracle, elem):
    """16384 x 16384 bf16: (a) idempotence -- quantizing the dequantized tensor reproduces codes and
    scales exactly; (b) a strided sample of rows equals the oracle bit-for-bit; (c) dequantize(bf16)
    and dequantize(f32) agree after rounding."""
    from torchmx import dtypes
    from torchmx.mx_tensor import MXTensor
    et = dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[elem]
    g = torch.Generator(device=DEV).manual_seed(0)
    x = torch.randn(16384, 16384, dtype=torch.bfloat16, device=DEV, generator=g)
    x *= torch.exp2(torch.randint(-40, 40, (16384, 1), device=DEV, generator=g).to(torch.float32)).to(torch.bfloat16)
    m = MXTensor.to_mx(x, et, 32)
    y = m.to_dtype(torch.bfloat16)
    m2 = MXTensor.to_mx(y, et, 32)
    assert torch.equal(m2._data, m._data)
    # idempotence of the scale can legitimately fail only if a block's max rounds down a binade; RNE never does
    assert torch.equal(m2._scale_e8m0, m._scale_e8m0)
    rows = torch.arange(0, 16384, 1031, device=DEV)
    s, c = oracle.quantize(bits_of(x[rows]), elem, 32, threads=8)
    assert_bits_equal(bits_of(m._scale_e8m0[rows]), s)
    assert_bits_equal(bits_of(m._data[rows]), c)
    assert_bits_equal(bits_of(y[rows]), oracle.dequantize(c, s, elem, 32, "bf16"))
    y32 = m.to_dtype(torch.float32)
    assert torch.equal(y32.to(torch.bfloat16), y)
    del y32, y, m, m2, x
    torch.cuda.empty_cache()


def test_ops_are_cuda_graph_capturable_and_stream_correct():
    """quantize / dequantize / MX linear enqueue on the CURRENT stream and never synchronise: they can be captured into a
    CUDA graph (what an inference server does with a decode step) and replayed on new data with identical results."""
    import torchmx_b200  # noqa: F401
    from torchmx_b200 import dtypes
    from torchmx_b200.config import MXConfig, QLinearConfig
    from torchmx_b200.layers.mx_linear import MXInferenceLinear
    from torchmx_b200.mx_tensor import MXTensor
    dev = "cuda:0"
    torch.manual_seed(0)
    lin = torch.nn.Linear(512, 384, bias=True).to(dev, torch.bfloat16)
    layer = MXInferenceLinear.from_float(lin, QLinearConfig(weights_config=MXConfig("float6_e3m2", 32), activations_config=MXConfig("float8_e4m3", 32)))
    x = torch.randn(16, 512, device=dev, dtype=torch.bfloat16)
    xl = torch.randn(200, 512, device=dev, dtype=torch.bfloat16)

    def work():
        m = MXTensor.to_mx(x, dtypes.float4_e2m1, 32)
        return m.to_dtype(torch.bfloat16), layer(x), layer(xl)   # decode-sized (fused quantize) and prefill-sized linears

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        for _ in range(2):
            work()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(g):
        outs = work()
    for trial in range(2):
        x.copy_(torch.randn(16, 512, device=dev, dtype=torch.bfloat16))
        xl.copy_(torch.randn(200, 512, device=dev, dtype=torch.bfloat16))
        g.replay()
        torch.cuda.synchronize()
        with torch.no_grad():
            want = work()
        torch.cuda.synchronize()
        for a, b in zip(outs, want):
            assert torch.equal(a, b), trial


# ---- K1 variants added in round 2 ------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("elem", ELEMS)
@pytest.mark.parametrize("bs", [8, 16, 64, 128])
def test_quantize_vector_kernel_other_block_sizes(mx, oracle, elem, bs, mode):
    """block sizes 8 / 16 / 64 / 128 run the vectorised kernel with 1, 1, 2, 4 lanes per block (the reference accepts any block
    size, torchmx/mx_tensor.py:68-73): random bit patterns incl. Inf / NaN / subnormal blocks, bit-exact against the oracle, and
    identical to the element-wise kernels (reached through a misaligned view)"""
    rng = np.random.default_rng(bs)
    bits = rng.integers(0, 65536, size=(257, 8 * bs), dtype=np.uint16)
    bits[(bits & 0x7F80) == 0x7F80] &= 0x3FFF           # mostly finite ...
    bits[3, 5], bits[100, 2 * bs + 1], bits[256, 8 * bs - 1] = 0x7F80, 0xFF80, 0x7FC1   # ... with +Inf, -Inf, NaN blocks
    bits[7, :bs] &= 0x807F                              # a block of bf16 subnormals
    scales, codes = _quant(bits, elem, bs, mode)
    o_scales, o_codes = oracle.quantize(bits, elem, bs, hw_exact=(mode == "hw_exact"))
    assert_bits_equal(scales, o_scales, f"block {bs} scales")
    assert_bits_equal(codes, o_codes, f"block {bs} codes")
    from torchmx import env_variables as env
    env.MX_EXACT_QUANTIZATION = MODES[mode]
    pad = torch.empty(bits.size + 8, dtype=torch.bfloat16, device=DEV)
    mis = pad[1:1 + bits.size].view(bits.shape)  # 2-byte offset: not 32-byte aligned -> element-wise kernels
    mis.copy_(bf16_tensor(bits, DEV))
    s2, c2 = torch.ops.torchmx.quantize_mx(mis, elem, bs)
    assert_bits_equal(bits_of(s2), scales)
    assert_bits_equal(bits_of(c2), codes)


@pytest.mark.parametrize("elem", ELEMS + ["float8_e5m2"])
def test_quantize_fp32_input_fast_path(mx, oracle, elem):
    """float32 input (labelled extension, PARITY UNPINNED: the reference asserts bf16, torchmx/mx_tensor.py:59-61; its fp32
    exponent branch is mx_quantization_utils.py:532-540): the coalesced block-32 kernel against the oracle's restatement with the
    assert bypassed, and against the element-wise kernels on the same values"""
    rng = np.random.default_rng(11)
    u = rng.integers(0, 2 ** 32, size=(513, 256), dtype=np.uint32)
    nan_or_inf = (u & 0x7F800000) == 0x7F800000
    u[nan_or_inf] &= 0xBFFFFFFF                          # mostly finite, every exponent incl. fp32 subnormals
    u[2, 7], u[77, 33], u[512, 255] = 0x7F800000, 0xFF800000, 0x7FC00001
    x = u.view(np.float32)
    xt = torch.from_numpy(x.copy()).to(DEV)
    scale, codes = torch.ops.torchmx.quantize_mx(xt, elem, 32)
    pad = torch.empty(x.size + 8, dtype=torch.float32, device=DEV)
    mis = pad[1:1 + x.size].view(x.shape)
    mis.copy_(xt)
    s2, c2 = torch.ops.torchmx.quantize_mx(mis, elem, 32)
    assert_bits_equal(bits_of(s2), bits_of(scale), "fast vs element-wise scales")
    assert_bits_equal(bits_of(c2), bits_of(codes), "fast vs element-wise codes")
    o_scales, o_codes = oracle.quantize(x, elem, 32)
    assert_bits_equal(bits_of(scale), o_scales, "fp32 scales vs oracle")
    assert_bits_equal(bits_of(codes), o_codes, "fp32 codes vs oracle")
