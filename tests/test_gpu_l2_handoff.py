"""GPU tier: the block-32 quantize (K1) and dequantize (K2) kernels on both sides of their L2 size gate.

A K1 launch whose input + code bytes exceed the device's L2 loads the input of its last window of codes L2 evict-first; a K2
launch to bf16 whose code + output bytes exceed L2 walks its tiles back to front, with evict-first accesses over the first
window for 1-byte codes.  For bf16 both gates fall at the same element count.  Every element type is checked bit for bit against the CPU oracle (codes, scales, bf16 values)
just below and just above the gate, on a shape whose chunk count leaves a partial tile (the reversed walk processes it
first), and with MXQ_WAVES=1 (a capped grid: the reversed grid-stride mapping).  fp32 targets keep one kernel on both sides
of the gate; one shape above it checks them beside the bf16 values."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.util import assert_bits_equal, bits_of

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ELEMS = ["float8_e4m3", "float6_e3m2", "float6_e2m3", "float4_e2m1", "int8", "float8_e5m2"]
COLS = 16384


def _check(elem: str, target: str, rows: int, cols: int):
    """quantize a seeded [rows, cols] bf16 tensor, dequantize it to `target`; codes, scales and values against the oracle"""
    from oracle import mx_oracle
    from torchmx_b200 import dtypes
    from torchmx_b200.mx_tensor import MXTensor
    mx_oracle.lib()
    g = torch.Generator(device=DEV).manual_seed(rows * 7 + cols)
    x = torch.randn(rows, cols, dtype=torch.bfloat16, device=DEV, generator=g)
    x *= torch.exp2(torch.randint(-40, 40, (rows, 1), device=DEV, generator=g).to(torch.float32)).to(torch.bfloat16)
    m = MXTensor.to_mx(x, getattr(dtypes, elem), 32)
    y = m.to_dtype(torch.bfloat16 if target == "bf16" else torch.float32)
    torch.cuda.synchronize()
    s, c = mx_oracle.quantize(bits_of(x), elem, 32, threads=8)
    del x
    assert_bits_equal(bits_of(m._scale_e8m0), s, f"{elem} scales [{rows}, {cols}]")
    assert_bits_equal(bits_of(m._data), c, f"{elem} codes [{rows}, {cols}]")
    del m
    want = mx_oracle.dequantize(c, s, elem, 32, target, threads=8)
    assert_bits_equal(bits_of(y), want.view(np.uint32) if target == "f32" else want, f"{elem} -> {target} [{rows}, {cols}]")
    del y
    torch.cuda.empty_cache()


def _gate_rows(stream_bytes_per_block: int) -> int:
    """the most rows of COLS elements whose launch streams no more bytes than L2 holds (one more row crosses the gate)"""
    l2 = torch.cuda.get_device_properties(0).L2_cache_size
    return l2 // (COLS // 32 * stream_bytes_per_block)


@pytest.mark.parametrize("side", ["below", "above"])
@pytest.mark.parametrize("elem", ELEMS)
def test_both_sides_of_the_l2_gate(elem, side):
    """K1's gate (bf16 input + code bytes) and K2's (code + bf16 output bytes): the same bytes per block"""
    code_bytes = 16 if elem == "float4_e2m1" else 32
    rows = _gate_rows(code_bytes + 64) + (side == "above")
    _check(elem, "bf16", rows, COLS)


@pytest.mark.parametrize("target", ["bf16", "f32"])
@pytest.mark.parametrize("elem", ELEMS)
def test_reversed_walk_partial_tile(elem, target):
    """[8193, 16416]: 4,203,009 blocks, above the gate, no chunk count a multiple of the 256-thread tile; the hint window ends
    inside both kernels' range"""
    _check(elem, target, 8193, 16416)


def test_reversed_grid_stride_with_capped_grid():
    """MXQ_WAVES=1 (read once per process) caps both grids at 8 CTAs per SM, so the large launches stride over their tiles"""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "from tests.test_gpu_l2_handoff import ELEMS, _check\n"
            "for e in ELEMS:\n"
            "    _check(e, 'bf16', 8193, 16416)\n"
            "print('ok')\n") % ROOT
    args = [sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", code]
    r = subprocess.run(args, cwd=ROOT, env=dict(os.environ, MXQ_WAVES="1"), capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0 and r.stdout.strip().endswith("ok"), r.stdout[-2000:] + r.stderr[-4000:]
