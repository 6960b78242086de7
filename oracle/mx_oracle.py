"""ctypes/numpy front end of the CPU oracle (oracle/mx_oracle.c).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package (torchmx_b200/) never imports it.

The functions mirror the two reference custom ops:
  quantize   <-> torchmx::quantize_mx    (/root/reference/torchmx/mx_tensor.py:36-96)
  dequantize <-> torchmx::dequantize_mx  (/root/reference/torchmx/mx_tensor.py:123-164)
Arrays are numpy; bf16 travels as uint16 bit patterns.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
from typing import Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libmx_oracle.so")

ELEM_IDS = {
    "float8_e4m3": 0,
    "float6_e3m2": 1,
    "float6_e2m3": 2,
    "float4_e2m1": 3,
    "int8": 4,
    "float8_e5m2": 5,  # extension: pinned against torch's float8_e5m2 cast (tests/test_e5m2_reference.py)
}

_lib = None


def build(force: bool = False) -> str:
    """Compile oracle/mx_oracle.c -> oracle/libmx_oracle.so (gcc, seconds)."""
    src = os.path.join(_HERE, "mx_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", "libmx_oracle.so"])
    return _LIB_PATH


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        build()
        L = ctypes.CDLL(_LIB_PATH)
        L.mxo_quantize.restype = ctypes.c_int
        L.mxo_quantize.argtypes = [
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
            ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
        ]
        L.mxo_dequantize.restype = ctypes.c_int
        L.mxo_dequantize.argtypes = [
            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int,
            ctypes.c_int, ctypes.c_void_p,
        ]
        L.mxo_dequantize_mt.restype = ctypes.c_int
        L.mxo_dequantize_mt.argtypes = L.mxo_dequantize.argtypes + [ctypes.c_int]
        L.mxo_gemm_nt_bf16.restype = ctypes.c_int
        L.mxo_gemm_nt_bf16.argtypes = [
            ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, ctypes.c_void_p,
        ]
        _lib = L
    return _lib


def _ptr(a: np.ndarray) -> ctypes.c_void_p:
    return ctypes.c_void_p(a.ctypes.data)


def quantize(x: np.ndarray, elem: str, block_size: int, hw_exact: bool = False,
             threads: int = 1) -> Tuple[np.ndarray, np.ndarray]:
    """x: uint16 (bf16 bit patterns) or float32, blocks along the last axis.

    Returns (scales uint8 [..., L/bs], codes) exactly as the reference op does -- scale first
    (mx_tensor.py:96).  codes is uint8 [..., L] (int8 dtype for elem == 'int8'), or
    [..., L/2] for float4_e2m1 (even element in the high nibble, utils.py:145).
    """
    assert x.dtype in (np.uint16, np.float32), x.dtype
    x = np.ascontiguousarray(x)
    L = x.shape[-1]
    assert L % block_size == 0, "last dim must be a multiple of block_size (mx_tensor.py:68-70)"
    n_blocks = x.size // block_size
    e = ELEM_IDS[elem]
    scales = np.empty(x.shape[:-1] + (L // block_size,), dtype=np.uint8)
    if elem == "float4_e2m1":
        if block_size % 2 == 0:
            codes = np.empty(x.shape[:-1] + (L // 2,), dtype=np.uint8)
            rc = lib().mxo_quantize(_ptr(x), int(x.dtype == np.float32), n_blocks, block_size, e,
                                    int(hw_exact), _ptr(scales), _ptr(codes), threads)
            assert rc == 0, rc
            return scales, codes
        # odd block size: quantize as unpacked e2m1 via a 2x wider trick is not possible; do it
        # block by block through the even-size entry by duplicating the block (max unchanged).
        assert x.size % 2 == 0, "pack_uint4 needs an even number of elements (utils.py:143)"
        xb = x.reshape(n_blocks, block_size)
        dup = np.concatenate([xb, xb], axis=1)  # same max exponent -> same scale, same codes twice
        sc2 = np.empty((n_blocks,), dtype=np.uint8)
        c2 = np.empty((n_blocks, block_size), dtype=np.uint8)
        rc = lib().mxo_quantize(_ptr(np.ascontiguousarray(dup)), int(x.dtype == np.float32), n_blocks,
                                2 * block_size, e, int(hw_exact), _ptr(sc2), _ptr(c2), threads)
        assert rc == 0, rc
        nib = np.empty((n_blocks, 2 * block_size), dtype=np.uint8)
        nib[:, 0::2] = c2 >> 4
        nib[:, 1::2] = c2 & 0xF
        flat = nib[:, :block_size].reshape(-1)
        codes = ((flat[0::2] << 4) | flat[1::2]).astype(np.uint8).reshape(x.shape[:-1] + (L // 2,))
        return sc2.reshape(scales.shape), codes
    codes = np.empty(x.shape, dtype=np.uint8)
    rc = lib().mxo_quantize(_ptr(x), int(x.dtype == np.float32), n_blocks, block_size, e,
                            int(hw_exact), _ptr(scales), _ptr(codes), threads)
    assert rc == 0, rc
    if elem == "int8":
        codes = codes.view(np.int8)
    return scales, codes


def dequantize(codes: np.ndarray, scales: np.ndarray, elem: str, block_size: int,
               target: str = "bf16", block_dim: int = -1, threads: int = 1) -> np.ndarray:
    """Inverse op.  `codes` may be any (possibly permuted) view whose blocked axis is
    `block_dim`; the result is C-contiguous in the logical shape, as FromMXConstrFunc returns it
    (mx_tensor.py:323).  target 'bf16' -> uint16 bit patterns, 'f32' -> float32."""
    assert target in ("bf16", "f32")
    nd = codes.ndim
    bd = block_dim if block_dim >= 0 else block_dim + nd
    c = np.ascontiguousarray(np.moveaxis(codes.view(np.uint8), bd, -1))
    s = np.ascontiguousarray(np.moveaxis(scales, bd, -1))
    n_blocks = s.size
    per = 2 if elem == "float4_e2m1" else 1
    assert c.size * per == n_blocks * block_size, (c.shape, s.shape, block_size)
    out_shape = c.shape[:-1] + (c.shape[-1] * per,)
    out = np.empty(out_shape, dtype=np.float32 if target == "f32" else np.uint16)
    if elem == "float4_e2m1" and block_size % 2:
        nib = np.empty(c.size * 2, dtype=np.uint8)
        nib[0::2] = c.reshape(-1) >> 4
        nib[1::2] = c.reshape(-1) & 0xF
        # decode nibble by nibble through the int-free path: reuse e2m1 with block_size*2 by
        # duplicating nibbles is overkill; decode in numpy instead (16-entry table).
        lut = np.array([0, .5, 1, 1.5, 2, 3, 4, 6, -0.0, -.5, -1, -1.5, -2, -3, -4, -6], dtype=np.float32)
        v = lut[nib].reshape(n_blocks, block_size)
        sc = np.where(s.reshape(-1, 1) == 255, np.float32(np.nan),
                      np.ldexp(np.float32(1.0), s.reshape(-1, 1).astype(np.int32) - 127)).astype(np.float32)
        with np.errstate(invalid="ignore", over="ignore"):
            prod = (v * sc).astype(np.float32).reshape(out_shape)
        out = prod if target == "f32" else f32_to_bf16_bits(prod)
    else:
        rc = lib().mxo_dequantize_mt(_ptr(c), _ptr(s), n_blocks, block_size, ELEM_IDS[elem],
                                     int(target == "f32"), _ptr(out), threads)
        assert rc == 0, rc
    return np.ascontiguousarray(np.moveaxis(out, -1, bd))


def quantize_into(x: np.ndarray, elem: str, block_size: int, scales: np.ndarray, codes: np.ndarray,
                  hw_exact: bool = False, threads: int = 1) -> None:
    """allocation-free variant for timing (bench.py cpu_baseline): outputs are caller-provided."""
    assert x.flags.c_contiguous and scales.flags.c_contiguous and codes.flags.c_contiguous
    rc = lib().mxo_quantize(_ptr(x), int(x.dtype == np.float32), x.size // block_size, block_size, ELEM_IDS[elem],
                            int(hw_exact), _ptr(scales), _ptr(codes), threads)
    assert rc == 0, rc


def dequantize_into(codes: np.ndarray, scales: np.ndarray, elem: str, block_size: int, out: np.ndarray,
                    threads: int = 1) -> None:
    """allocation-free variant for timing: blocked axis last, everything contiguous."""
    assert codes.flags.c_contiguous and scales.flags.c_contiguous and out.flags.c_contiguous
    rc = lib().mxo_dequantize_mt(_ptr(codes), _ptr(scales), scales.size, block_size, ELEM_IDS[elem],
                                 int(out.dtype == np.float32), _ptr(out), threads)
    assert rc == 0, rc


def f32_to_bf16_bits(x: np.ndarray) -> np.ndarray:
    """fp32 -> bf16 bit patterns, round-to-nearest-even, NaN quieted (torch's .to(bfloat16))."""
    u = np.ascontiguousarray(x, dtype=np.float32).view(np.uint32)
    nan = (u & 0x7FFFFFFF) > 0x7F800000
    r = ((u + (0x7FFF + ((u >> 16) & 1))) >> 16).astype(np.uint16)
    return np.where(nan, ((u >> 16) | 0x40).astype(np.uint16), r)


def bf16_bits_to_f32(b: np.ndarray) -> np.ndarray:
    return (b.astype(np.uint32) << 16).view(np.float32)


def gemm_nt(a_bf16_bits: np.ndarray, b_bf16_bits: np.ndarray) -> np.ndarray:
    """out[m, n] = sum_k a[m, k] * b[n, k] with double accumulation (see mx_oracle.c)."""
    a = np.ascontiguousarray(a_bf16_bits, dtype=np.uint16)
    b = np.ascontiguousarray(b_bf16_bits, dtype=np.uint16)
    M, K = a.shape
    N, K2 = b.shape
    assert K == K2
    out = np.empty((M, N), dtype=np.float32)
    rc = lib().mxo_gemm_nt_bf16(_ptr(a), _ptr(b), M, N, K, _ptr(out))
    assert rc == 0
    return out
