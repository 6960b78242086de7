"""CPU tier: the C oracle's float8_e5m2 path against a restatement built on torch's own float8_e5m2 cast.

float8_e5m2 is a labelled extension element type: the reference has none, so there is no reference output to match.  What pins
it instead is two independent statements of the same arithmetic that must agree bit for bit:
* oracle/mx_oracle.c: shared exponent maxE - 15, fp32 x / 2^(s-127), clamp to +-57344, its own fp32 -> e5m2 RNE (`f32_to_e5m2`);
* `_e5m2_quantize_ref` / `_e5m2_dequantize_ref` below: the same scale rule, the division done exactly in fp64, the element cast
  done by torch (`.to(torch.float8_e5m2)`), the decode by reinterpreting the code byte as torch.float8_e5m2.
tests/test_gpu_e5m2.py then holds every kernel that reads or writes e5m2 to these two."""
import numpy as np
import pytest
import torch

from oracle import grids
from tests.util import MODES, assert_bits_equal

E5M2 = "float8_e5m2"
E5M2_MAX = 57344.0  # 1.75 * 2^15, the largest finite e5m2 value
E5M2_MAX_POW2 = 15  # exponent of the largest e5m2 binade: the shared scale is 2^(maxE - 15)


def _e5m2_quantize_ref(x: np.ndarray, block_size: int):
    """x: uint16 bf16 bit patterns or float32, blocks along the last axis -> (scales uint8 [..., L/bs], codes uint8 [..., L]).

    s = 255 if any exponent field of the block is 255 (Inf / NaN), else clamp(maxE - 15, 0, 254); a code is
    float8_e5m2(float32(clamp(x * 2^(127 - s), +-57344))) with the product exact in fp64; a block with s = 255 has all codes +0."""
    x = np.ascontiguousarray(x)
    assert x.dtype in (np.uint16, np.float32) and x.shape[-1] % block_size == 0
    if x.dtype == np.uint16:
        exp = (x.astype(np.int32) >> 7) & 0xFF
        val = torch.from_numpy(x.view(np.int16).copy()).view(torch.bfloat16).double()
    else:
        exp = (x.view(np.uint32) >> 23).astype(np.int32) & 0xFF
        val = torch.from_numpy(x.copy()).double()
    blocks = x.shape[:-1] + (x.shape[-1] // block_size, block_size)
    max_e = torch.from_numpy(exp.reshape(blocks)).amax(-1)
    s = torch.where(max_e == 255, 255, (max_e - E5M2_MAX_POW2).clamp(0, 254))
    y = val.reshape(blocks) * torch.exp2((127 - s).double()).unsqueeze(-1)
    y = y.clamp(-E5M2_MAX, E5M2_MAX)
    nan_block = (s == 255).unsqueeze(-1)
    y = torch.where(nan_block, 0.0, y)
    codes = y.to(torch.float32).to(torch.float8_e5m2).view(torch.uint8)
    return s.to(torch.uint8).numpy(), codes.reshape(x.shape).numpy()


def _e5m2_dequantize_ref(codes: np.ndarray, scales: np.ndarray, block_size: int, target: str) -> np.ndarray:
    """codes uint8 [..., L], scales uint8 [..., L/bs], blocks along the last axis -> bf16 bit patterns (uint16) or float32:
    the code's float8_e5m2 value times 2^(s-127) in fp64 (NaN for s = 255), then rounded to the target."""
    c = torch.from_numpy(np.ascontiguousarray(codes).view(np.uint8).copy()).view(torch.float8_e5m2).double()
    s = torch.from_numpy(np.ascontiguousarray(scales).astype(np.int64))
    sc = torch.where(s == 255, float("nan"), torch.exp2((s - 127).double())).repeat_interleave(block_size, -1)
    v = (c * sc).to(torch.float32)  # exact: at most 3 significant bits, fp32 subnormals reach 2^-149 (or +-Inf past 2^128)
    if target == "f32":
        return v.numpy().copy()
    assert target == "bf16"
    return v.to(torch.bfloat16).view(torch.int16).numpy().view(np.uint16).copy()


def _fp32_sample() -> np.ndarray:
    """float32 [513, 256]: random bit patterns with every exponent field (fp32 subnormals included) and +-Inf / NaN blocks"""
    rng = np.random.default_rng(11)
    u = rng.integers(0, 2 ** 32, size=(513, 256), dtype=np.uint32)
    nan_or_inf = (u & 0x7F800000) == 0x7F800000
    u[nan_or_inf] &= 0xBFFFFFFF                          # mostly finite, every exponent incl. fp32 subnormals
    u[2, 7], u[77, 33], u[512, 255] = 0x7F800000, 0xFF800000, 0x7FC00001
    return u.view(np.float32)


def _block_size_sample(bs: int) -> np.ndarray:
    """bf16 bits [257, 8 bs]: random patterns, mostly finite, with +Inf, -Inf and NaN blocks and a block of bf16 subnormals"""
    rng = np.random.default_rng(bs)
    bits = rng.integers(0, 65536, size=(257, 8 * bs), dtype=np.uint16)
    bits[(bits & 0x7F80) == 0x7F80] &= 0x3FFF
    bits[3, 5], bits[100, 2 * bs + 1], bits[256, 8 * bs - 1] = 0x7F80, 0xFF80, 0x7FC1
    bits[7, :bs] &= 0x807F
    return bits


@pytest.mark.parametrize("mode", list(MODES))
def test_quantize_grid_small(oracle, mode):
    """every bf16 pattern under a subsample of block exponents (incl. the extremes and Inf / NaN leads); e5m2 has no hardware-
    exact variant, so both values of MX_EXACT_QUANTIZATION give the same bytes"""
    grid = grids.quant_grid_small()
    scales, codes = oracle.quantize(grid, E5M2, 32, hw_exact=(mode == "hw_exact"), threads=4)
    r_scales, r_codes = _e5m2_quantize_ref(grid, 32)
    assert_bits_equal(scales, r_scales, "scales")
    assert_bits_equal(codes, r_codes, "codes")
    other = oracle.quantize(grid, E5M2, 32, hw_exact=(mode != "hw_exact"), threads=4)
    assert_bits_equal(other[0], scales, "scales under the other mode")
    assert_bits_equal(other[1], codes, "codes under the other mode")


def test_quantize_grid_small_covers_every_e5m2_code():
    """the grid reaches every finite code byte, the saturated +-57344 (0x7B / 0xFB) and both zeros, and no Inf / NaN code"""
    _, codes = _e5m2_quantize_ref(grids.quant_grid_small(), 32)
    seen = np.zeros(256, dtype=bool)
    seen[np.unique(codes)] = True
    finite = np.array([(c & 0x7F) < 0x7C for c in range(256)])
    assert seen[finite].all() and not seen[~finite].any()


def test_quantize_fp32_sample(oracle):
    x = _fp32_sample()
    scales, codes = oracle.quantize(x, E5M2, 32)
    r_scales, r_codes = _e5m2_quantize_ref(x, 32)
    assert_bits_equal(scales, r_scales, "fp32 scales")
    assert_bits_equal(codes, r_codes, "fp32 codes")
    assert (scales[2, 0], scales[77, 1], scales[512, 7]) == (255, 255, 255)
    assert (((x.view(np.uint32) >> 23) & 0xFF) == 0).any()  # fp32 subnormal elements


@pytest.mark.parametrize("bs", [8, 16, 64, 128])
def test_quantize_other_block_sizes(oracle, bs):
    bits = _block_size_sample(bs)
    for hw_exact in (False, True):
        scales, codes = oracle.quantize(bits, E5M2, bs, hw_exact=hw_exact)
        r_scales, r_codes = _e5m2_quantize_ref(bits, bs)
        assert_bits_equal(scales, r_scales, f"block {bs} scales")
        assert_bits_equal(codes, r_codes, f"block {bs} codes")


def test_saturation_and_scale_rule():
    """known answers: the largest binade keeps 1.0 / 1.25 / 1.5 / 1.75 and saturates 1.875 and 1.9921875 to 57344 (0x7B); the
    scale is maxE - 15 and clamps at 0; an Inf anywhere makes the block NaN (scale 255, codes +0)"""
    one = np.array([0x3F80, 0x3FA0, 0x3FC0, 0x3FE0, 0x3FF0, 0x3FFF, 0xBFF0, 0x0000], dtype=np.uint16)  # 1, 1.25 .. 1.99, -1.875, 0
    scales, codes = _e5m2_quantize_ref(one[None, :], 8)
    assert scales.tolist() == [[127 - 15]]
    assert codes.tolist() == [[0x78, 0x79, 0x7A, 0x7B, 0x7B, 0x7B, 0xFB, 0x00]]
    tiny = np.array([0x0001, 0x0080, 0x0000, 0x8001], dtype=np.uint16)  # 2^-133 (bf16 subnormal), 2^-126, 0, -2^-133: maxE 1
    scales, codes = _e5m2_quantize_ref(tiny[None, :], 4)
    assert scales.tolist() == [[0]] and codes.tolist() == [[0x24, 0x40, 0x00, 0xA4]]  # 2^-6, 2, 0, -2^-6 after the 2^127 scaling
    inf = np.array([0x3F80, 0x7F80, 0x4000, 0xC000], dtype=np.uint16)
    scales, codes = _e5m2_quantize_ref(inf[None, :], 4)
    assert scales.tolist() == [[255]] and codes.tolist() == [[0, 0, 0, 0]]


@pytest.mark.parametrize("target", ["bf16", "f32"])
def test_dequantize_grid(oracle, target):
    """every (code byte, scale) pair, the +-Inf codes 0x7C / 0xFC and the NaN codes 0x7D-0x7F / 0xFD-0xFF included (K1 never writes
    them, an MXTensor built by a user can hold them)"""
    codes, scales = grids.dequant_grid(E5M2)
    out = oracle.dequantize(codes, scales, E5M2, 32, target, 1)
    want = _e5m2_dequantize_ref(codes, scales, 32, target)
    if target == "f32":
        out, want = out.view(np.uint32), want.view(np.uint32)
    assert_bits_equal(out, want, f"dequantize -> {target}")
    v = want.view(np.float32) if target == "f32" else (want.astype(np.uint32) << 16).view(np.float32)
    inf_cols, nan_cols = [0x7C, 0xFC], [0x7D, 0x7E, 0x7F, 0xFD, 0xFE, 0xFF]
    assert np.isinf(v[:255, inf_cols]).all() and np.isnan(v[:, nan_cols]).all() and np.isnan(v[255]).all()
    assert np.signbit(v[:255, 0xFC]).all() and not np.signbit(v[:255, 0x7C]).any()
