"""GPU tier: the block-scaled MX GEMM kernels (K3a / K3b / K3c, DESIGN.md §K3) at their dispatch and tile edges.

Which kernel runs follows from `launch_gemm`: M <= 128 and not batched -> K3c (the decode kernel); M, N > 128 -> K3b, unless its
256 x 256 tiles would occupy at most a quarter of the SM pairs (MXQ_GEMM_WIDE_TILES keeps them); everything else -> K3a.  K3c
picks its variant from M (32 / 64 / 128 token columns) and from the grid: `ceil(N / 128) * splits <= sm_count` runs the deep
one-CTA-per-SM variants (two MMA issuers for M <= 64, a push reduction of the K splits), anything wider the 4-stage two-CTA-per-SM
variants (one issuer, a pull reduction).  The decode lm_head (N = 128256) runs the latter.

Reference and tolerance as in tests/test_gpu_gemm.py: `ref` is the fp64 contraction of the operands dequantized by K2
(`to_dtype(torch.float32)`, itself pinned to the CPU oracle; the small cases check that again here), plus bias, and
|out - ref| <= 2^-8 |ref| + 2^-18 * sum_k |a_k b_k|.  Two launches of the same kernel with the same K split must agree bit for
bit: K3c reduces its splits in a fixed order.
"""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
E4M3, FP6, FP4 = "float8_e4m3", "float6_e3m2", "float4_e2m1"


@pytest.fixture(scope="module")
def sm():
    import torchmx  # noqa: F401
    from torchmx_b200 import _C
    _C.lib()
    return torch.cuda.get_device_properties(0).multi_processor_count


def _et(name):
    from torchmx import dtypes
    return dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[name]


def _mx(t, elem):
    from torchmx.mx_tensor import MXTensor
    return MXTensor.to_mx(t, _et(elem), 32)


def _deq(t, oracle=None):
    """fp64 values of an MXTensor through K2; with `oracle`, K2's float32 values are also checked against the CPU oracle's"""
    d = t.to_dtype(torch.float32)
    if oracle is not None:
        want = oracle.dequantize(t._data.cpu().numpy().view(np.uint8), t._scale_e8m0.cpu().numpy(), t._elem_dtype.name, 32, target="f32")
        assert np.array_equal(d.cpu().numpy(), want), "K2 and the oracle dequantize differently"
    return d.double()


def _refs(ad, bd):
    return ad @ bd.transpose(-1, -2), ad.abs() @ bd.abs().transpose(-1, -2)


def _check(out, ref, S, bias=None, what=""):
    if bias is not None:
        ref, S = ref + bias.double(), S + bias.double().abs()
    assert out.shape == ref.shape, (what, tuple(out.shape), tuple(ref.shape))
    assert not torch.isnan(out).any(), f"{what}: NaN in the output"
    err = (out.double() - ref).abs()
    tol = 2.0 ** -8 * ref.abs() + 2.0 ** -18 * S + 1e-30
    bad = int((err > tol).sum())
    assert bad == 0, f"{what}: {bad}/{err.numel()} outside tolerance, worst err/S {(err / (S + 1e-30)).max().item():.3e}"


def _spread(t, g, spread):
    """multiply every 32-block by 2^e, e uniform in [-spread, spread): operands whose scale bytes differ block to block"""
    e = torch.randint(-spread, spread, (*t.shape[:-1], t.shape[-1] // 32), device=DEV, generator=g).float()
    return t * torch.exp2(e).repeat_interleave(32, -1).to(torch.bfloat16)


def _layer(N, K, wdt, g, spread=0):
    """MXInferenceLinear with a bf16 bias and an e4m3 activation config (decode-sized inputs quantized inside the GEMM)"""
    from torchmx.config import MXConfig, QLinearConfig
    from torchmx.layers.mx_linear import MXInferenceLinear
    lin = torch.nn.utils.skip_init(torch.nn.Linear, K, N, bias=True, device=DEV, dtype=torch.bfloat16)
    w = torch.randn(N, K, device=DEV, dtype=torch.bfloat16, generator=g)
    lin.weight.data.copy_(_spread(w, g, spread) if spread else w)
    lin.bias.data.copy_(torch.randn(N, device=DEV, dtype=torch.bfloat16, generator=g))
    del w
    return MXInferenceLinear.from_float(lin, QLinearConfig(weights_config=MXConfig(wdt, 32), activations_config=MXConfig(E4M3, 32)))


def _count(key="tensor_core"):
    from torchmx_b200 import mx_gemm
    return mx_gemm.stats.get(key, 0)


# ---- 1. K3c at N wider than one tile per SM: the 4-stage variants the decode lm_head runs --------------------------------------
_WIDE_CACHE = {}


def _wide(wdt, N):
    """(layer, bias, fp64 weight) for one (weight type, N); one entry at a time -- the fp64 copy of a 128256 x 4096 weight is 4 GB"""
    key = (wdt, N)
    if key not in _WIDE_CACHE:
        _WIDE_CACHE.clear()
        torch.cuda.empty_cache()
        layer = _layer(N, 4096, wdt, torch.Generator(device=DEV).manual_seed(N + len(wdt)))
        _WIDE_CACHE[key] = (layer, layer.bias, _deq(layer.weight), {})
    return _WIDE_CACHE[key]


@pytest.fixture(scope="module", autouse=True)
def _release_wide_weights():
    yield
    _WIDE_CACHE.clear()


def _wide_n(n, sm):
    return 128 * (sm + 1) + 40 if n == "sm+1" else n


@pytest.mark.parametrize("wdt,n,M", [(w, n, m) for w in (E4M3, FP6, FP4) for n in ("sm+1", 128256) for m in (1, 32, 33, 64, 65, 128)])
def test_decode_kernel_at_wide_n(sm, wdt, n, M):
    """F.linear on MXTensors and MXInferenceLinear on bf16 input (quantized inside the GEMM for M <= 64), bias on and off, against
    the fp64 contraction; the layer equals the F.linear result bit for bit.  N = 128256 x K = 4096 is Llama-3's lm_head."""
    N = _wide_n(n, sm)
    assert (N + 127) // 128 > sm, "expected the wide-grid variants"
    layer, bias, wd, extra = _wide(wdt, N)
    g = torch.Generator(device=DEV).manual_seed(M)
    x = torch.randn(M, 4096, device=DEV, dtype=torch.bfloat16, generator=g)
    X = _mx(x, E4M3)
    ref, S = _refs(_deq(X), wd)
    try:
        for b in (None, bias):
            t0, f0 = _count(), _count("fused_act_quant")
            y = F.linear(X, layer.weight, b)
            assert _count() == t0 + 1, "expected the tensor-core path"
            _check(y, ref, S, b, f"{M}x{N} {wdt} bias={b is not None}")
            layer.bias = b
            y2 = layer(x)
            assert _count() == t0 + 2 and _count("fused_act_quant") == f0 + (M <= 64)
            assert torch.equal(y2, y), "fused activation quantization differs from K1 + GEMM"
        if wdt == FP6 and N == 128256:
            # the same weight held only as its packed operand stream (PackedMXLinear): same kernel, same bytes
            from torchmx.layers.packed_linear import PackedMXLinear
            if "packed" not in extra:
                extra["packed"] = PackedMXLinear.from_mx_linear(layer, keep_source=True)
            t0, f0 = _count(), _count("fused_act_quant")
            assert torch.equal(extra["packed"](x), y)
            assert _count() == t0 + 1 and _count("fused_act_quant") == f0 + (M <= 64)
    finally:
        layer.bias = bias


@pytest.mark.parametrize("M", [1, 32, 33, 64])
@pytest.mark.parametrize("splits", [2, 3])
def test_decode_kernel_at_wide_n_with_forced_splits(sm, monkeypatch, M, splits):
    """K splits on the wide grid: the 4-stage variants reduce them by pulling the peers' partials through DSMEM (32 K blocks
    over 3 splits is uneven, and moves the scales to the LDG loader)"""
    from torchmx_b200 import mx_gemm
    monkeypatch.setitem(mx_gemm.overrides, "split_k", splits)
    N = _wide_n("sm+1", sm)
    layer, bias, wd, _ = _wide(FP6, N)
    g = torch.Generator(device=DEV).manual_seed(100 + M)
    x = torch.randn(M, 4096, device=DEV, dtype=torch.bfloat16, generator=g)
    X = _mx(x, E4M3)
    y = F.linear(X, layer.weight, bias)
    ref, S = _refs(_deq(X), wd)
    _check(y, ref, S, bias, f"{M}x{N} splits={splits}")
    assert torch.equal(F.linear(X, layer.weight, bias), y)
    f0 = _count("fused_act_quant")
    assert torch.equal(layer(x), y)
    assert _count("fused_act_quant") == f0 + 1


# ---- 2. K3c: one to five K blocks, one or two MMA issuers, tiles shorter than their 128 rows -----------------------------------
_EDGE_M = (1, 31, 32, 33, 63, 64, 65, 127, 128)
_EDGE_W = {8: E4M3, 120: FP6, 129: FP4, 1000: FP6}


def _dirty_tensor_memory(sm):
    """run the deep two-issuer variants (32 and 64 token columns) over every SM with two K blocks, so that their second
    accumulator holds partial sums when the next launch starts: an epilogue that read it after a one-K-block launch would add them"""
    g = torch.Generator(device=DEV).manual_seed(7)
    W = _mx(torch.randn(128 * sm, 256, device=DEV, dtype=torch.bfloat16, generator=g), E4M3)
    for m in (32, 64):
        F.linear(_mx(torch.randn(m, 256, device=DEV, dtype=torch.bfloat16, generator=g), E4M3), W)


@pytest.mark.parametrize("N", list(_EDGE_W))
@pytest.mark.parametrize("K", [128, 256, 384, 640])
def test_decode_kernel_k_block_and_issuer_edges(sm, oracle, K, N):
    """every token bucket edge (M = 31..33, 63..65, 127, 128) at one to five K blocks: plain, and with the activation quantized
    inside the GEMM (M <= 64) under both values of MX_EXACT_QUANTIZATION, bit-identical to K1 followed by the GEMM"""
    from torchmx import env_variables as env
    g = torch.Generator(device=DEV).manual_seed(K * 3 + N)
    layer = _layer(N, K, _EDGE_W[N], g, spread=6)
    wd = _deq(layer.weight, oracle)
    _dirty_tensor_memory(sm)
    for mode in ("False", "True"):
        env.MX_EXACT_QUANTIZATION = mode
        for M in _EDGE_M:
            x = _spread(torch.randn(M, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 8)
            X = _mx(x, E4M3)
            t0, f0 = _count(), _count("fused_act_quant")
            y = F.linear(X, layer.weight, layer.bias)
            assert _count() == t0 + 1
            ref, S = _refs(_deq(X, oracle if mode == "False" else None), wd)
            _check(y, ref, S, layer.bias, f"{M}x{N}x{K} hw_exact={mode}")
            if M <= 64:
                assert torch.equal(layer(x), y), f"{M}x{N}x{K} hw_exact={mode}: fused differs from K1 + GEMM"
                assert _count("fused_act_quant") == f0 + 1


# ---- 3. K3c: every split count the C ABI accepts, at every K-block count up to nine ---------------------------------------------
@pytest.mark.parametrize("splits", range(1, 9))
def test_decode_kernel_every_k_split(monkeypatch, splits):
    """split_k 1..8 at k_blocks 1..9 (clamped to k_blocks; uneven split points; LDG scale loading when the split points are not
    4-K-block aligned) on a deep grid (N = 200: two tiles): within the tolerance, and bit-identical when repeated"""
    from torchmx_b200 import mx_gemm
    monkeypatch.setitem(mx_gemm.overrides, "split_k", splits)
    N = 200
    for kb in range(1, 10):
        K = 128 * kb
        g = torch.Generator(device=DEV).manual_seed(kb * 10 + splits)
        W = _mx(_spread(torch.randn(N, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 4), FP6)
        bias = torch.randn(N, device=DEV, dtype=torch.bfloat16, generator=g)
        wd = _deq(W)
        for M in (1, 33, 64, 100):
            X = _mx(torch.randn(M, K, device=DEV, dtype=torch.bfloat16, generator=g), E4M3)
            t0 = _count()
            y = F.linear(X, W, bias)
            assert _count() == t0 + 1
            ref, S = _refs(_deq(X), wd)
            _check(y, ref, S, bias, f"{M}x{N}x{K} split_k={splits}")
            assert torch.equal(F.linear(X, W, bias), y), f"{M}x{N}x{K} split_k={splits}: not reproducible"


# ---- 4. K3b and K3a at ragged edges -------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [128, 256, 384])
@pytest.mark.parametrize("M", [129, 255, 256, 257])
def test_pair_kernel_edges(monkeypatch, oracle, M, K):
    """K3b (wide tiles kept): M, N in {129, 255, 256, 257}; K <= 256 runs the 3-stage operand ring"""
    from torchmx_b200 import mx_gemm
    monkeypatch.setitem(mx_gemm.overrides, "wide_tiles", True)
    g = torch.Generator(device=DEV).manual_seed(M * 5 + K)
    A = _mx(_spread(torch.randn(M, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), E4M3)
    ad = _deq(A, oracle)
    for N in (129, 255, 256, 257):
        wdt = FP6 if N < 256 else FP4
        W = _mx(_spread(torch.randn(N, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), wdt)
        bias = torch.randn(N, device=DEV, dtype=torch.bfloat16, generator=g) if N % 2 else None
        t0 = _count()
        y = F.linear(A, W, bias)
        assert _count() == t0 + 1
        ref, S = _refs(ad, _deq(W, oracle))
        _check(y, ref, S, bias, f"{M}x{N}x{K} {wdt}")


@pytest.mark.parametrize("M,N", [(300, 520), (257, 129), (129, 257)])
@pytest.mark.parametrize("K", [256, 384])
def test_pair_kernel_fp4_by_fp4(monkeypatch, oracle, M, N, K):
    """fp4 x fp4: kind::mxf4 on the dense 4-bit streams when K % 256 == 0, kind::mxf8f6f4 otherwise"""
    from torchmx_b200 import mx_gemm
    monkeypatch.setitem(mx_gemm.overrides, "wide_tiles", True)
    g = torch.Generator(device=DEV).manual_seed(M + N + K)
    A = _mx(_spread(torch.randn(M, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), FP4)
    W = _mx(_spread(torch.randn(N, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), FP4)
    bias = torch.randn(N, device=DEV, dtype=torch.bfloat16, generator=g)
    t0 = _count()
    y = F.linear(A, W, bias)
    assert _count() == t0 + 1
    ref, S = _refs(_deq(A, oracle), _deq(W, oracle))
    _check(y, ref, S, bias, f"fp4 {M}x{N}x{K}")


@pytest.mark.parametrize("N", [1, 7, 8, 127, 128])
@pytest.mark.parametrize("K", [256, 640])
def test_single_cta_kernel_narrow_n(oracle, N, K):
    """K3a (M > 128, N <= 128): output widths from one column to one full tile, bias on"""
    g = torch.Generator(device=DEV).manual_seed(N * 7 + K)
    A = _mx(_spread(torch.randn(300, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), E4M3)
    W = _mx(_spread(torch.randn(N, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), FP6)
    bias = torch.randn(N, device=DEV, dtype=torch.bfloat16, generator=g)
    t0 = _count()
    y = F.linear(A, W, bias)
    assert _count() == t0 + 1
    ref, S = _refs(_deq(A, oracle), _deq(W, oracle))
    _check(y, ref, S, bias, f"300x{N}x{K}")


@pytest.mark.parametrize("M", [1, 77, 128])
@pytest.mark.parametrize("N", [100, 200])
def test_single_cta_kernel_batched_short_m(oracle, M, N):
    """batched M <= 128 (never the decode kernel): K3a with 128- and 256-column tiles"""
    g = torch.Generator(device=DEV).manual_seed(M * 3 + N)
    A = _mx(torch.randn(3, M, 384, device=DEV, dtype=torch.bfloat16, generator=g), E4M3)
    B = _mx(_spread(torch.randn(3, N, 384, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), FP4)
    t0 = _count()
    y = torch.bmm(A, B.transpose(1, 2))
    assert _count() == t0 + 1
    ref, S = _refs(_deq(A, oracle), _deq(B, oracle))
    _check(y, ref, S, None, f"3x{M}x{N}x384")


# ---- 5. the C ABI with row pitches: nothing is written outside the output window, nothing read past the operands' extent -------
_SENTINEL = 0x7FA5  # a bf16 NaN bit pattern no kernel produces (they write the canonical NaN)


def _gemm(A, sfa, B, sfb, bias, d_ptr, *, M, N, K, batch, a_fmt, b_fmt, ldd, d_bs, flags, lda, ldb, ld_sfa, ld_sfb, a_bs, b_bs, sfa_bs, sfb_bs):
    from torchmx_b200 import _C
    from torchmx_b200.mx_tensor import _stream_ptr
    ga = _C.GemmArgs()
    ga.a_codes, ga.sfa, ga.lda, ga.ld_sfa, ga.a_batch_stride, ga.sfa_batch_stride = A.data_ptr(), sfa.data_ptr(), lda, ld_sfa, a_bs, sfa_bs
    ga.b_codes, ga.sfb, ga.ldb, ga.ld_sfb, ga.b_batch_stride, ga.sfb_batch_stride = B.data_ptr(), sfb.data_ptr(), ldb, ld_sfb, b_bs, sfb_bs
    ga.bias = bias.data_ptr() if bias is not None else None
    ga.d, ga.ldd, ga.d_batch_stride = d_ptr, ldd, d_bs
    ga.batch, ga.M, ga.N, ga.K = batch, M, N, K
    ga.a_format, ga.b_format, ga.flags = a_fmt, b_fmt, flags
    _C.check(_C.lib().mxq_gemm(ctypes.byref(ga), 0, _stream_ptr(A)), "mxq_gemm")


def _padded(t, extra_rows, extra_cols, fill):
    """t [batch, rows, cols] uint8 copied into the top-left corner of a [batch, rows + extra_rows, cols + extra_cols] buffer"""
    b, r, c = t.shape
    buf = fill((b, r + extra_rows, c + extra_cols))
    buf[:, :r, :c] = t
    return buf


_CANARY = [  # kernel, M, N, K, batch, weight type, flags
    ("K3c split 2", 33, 1000, 1024, 1, FP6, 0),
    ("K3c", 100, 1000, 512, 1, FP4, 0),
    ("K3a", 300, 520, 512, 1, FP6, 0),
    ("K3a", 300, 520, 512, 3, E4M3, 0),
    ("K3b", 300, 520, 512, 1, FP4, "wide"),
    ("K3b", 300, 520, 512, 3, FP6, "wide"),
]


@pytest.mark.parametrize("placement", ["aligned", "offset", "odd_ldd"])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("kernel,M,N,K,batch,wdt,flags", _CANARY)
def test_output_window_and_operand_padding(sm, kernel, M, N, K, batch, wdt, flags, bias, placement):
    """mxq_gemm with padded pitches equals the compact call bit for bit.  The output window (ldd = N + pad, batch stride past
    M * ldd) sits in a sentinel-filled buffer, 16-byte aligned with ldd % 8 == 0 (TMA store / 16- and 8-byte stores), one element
    off (scalar stores), or with an odd ldd: every element outside it keeps the sentinel.  The operands sit in buffers with 128
    junk code bytes past K in every row, four NaN scale bytes past K/32 (a pitch that is not a multiple of 16, which moves K3c to
    its LDG scale loader) and junk rows past M and N."""
    from torchmx_b200 import _C, mx_gemm
    g = torch.Generator(device=DEV).manual_seed(M + N + K + batch)
    A = _mx(torch.randn(batch, M, K, device=DEV, dtype=torch.bfloat16, generator=g), E4M3)
    W = _mx(_spread(torch.randn(batch, N, K, device=DEV, dtype=torch.bfloat16, generator=g), g, 6), wdt)
    a_e, a_fmt = mx_gemm._operand_rows(A._data, A._elem_dtype, None, packed=True)
    b_e, b_fmt = mx_gemm._operand_rows(W._data, W._elem_dtype, None, packed=True)
    sfa, sfb = A._scale_e8m0, W._scale_e8m0
    bias_t = torch.randn(N, device=DEV, dtype=torch.bfloat16, generator=g) if bias else None
    fl = _C.GEMM_WIDE_TILES if flags == "wide" else 0
    dims = dict(M=M, N=N, K=K, batch=batch, a_fmt=a_fmt, b_fmt=b_fmt, flags=fl)
    compact = torch.empty(batch, M, N, device=DEV, dtype=torch.bfloat16)
    _gemm(a_e, sfa, b_e, sfb, bias_t, compact.data_ptr(), ldd=N, d_bs=M * N, lda=a_e.shape[-1], ldb=b_e.shape[-1], ld_sfa=K // 32,
          ld_sfb=K // 32, a_bs=a_e[0].numel(), b_bs=b_e[0].numel(), sfa_bs=M * K // 32, sfb_bs=N * K // 32, **dims)
    ref, S = _refs(_deq(A), _deq(W))
    _check(compact, ref, S, bias_t, f"{kernel} compact")

    junk = lambda shape: torch.randint(0, 256, shape, device=DEV, dtype=torch.uint8, generator=g)
    nan = lambda shape: torch.full(shape, 0xFF, device=DEV, dtype=torch.uint8)
    pa, pb = _padded(a_e, 5, 128, junk), _padded(b_e, 7, 128, junk)
    psa, psb = _padded(sfa, 5, 4, nan), _padded(sfb, 7, 4, nan)
    ldd = -(-(N + 5) // 8) * 8 if placement != "odd_ldd" else (N + 5) | 1
    off = 1 if placement == "offset" else 0
    d_bs = M * ldd + (16 if placement != "odd_ldd" else 9)
    size = off + batch * d_bs + 64
    buf = torch.full((size,), _SENTINEL, device=DEV, dtype=torch.int16)
    _gemm(pa, psa, pb, psb, bias_t, buf.data_ptr() + 2 * off, ldd=ldd, d_bs=d_bs, lda=pa.shape[-1], ldb=pb.shape[-1], ld_sfa=psa.shape[-1],
          ld_sfb=psb.shape[-1], a_bs=pa[0].numel(), b_bs=pb[0].numel(), sfa_bs=psa[0].numel(), sfb_bs=psb[0].numel(), **dims)
    window = buf.as_strided((batch, M, N), (d_bs, ldd, 1), off)
    assert torch.equal(window, compact.view(torch.int16)), f"{kernel} {placement}: padded call differs from the compact one"
    outside = torch.ones(size, device=DEV, dtype=torch.bool)
    outside.as_strided((batch, M, N), (d_bs, ldd, 1), off).fill_(False)
    stray = int((buf[outside] != _SENTINEL).sum())
    assert stray == 0, f"{kernel} {placement}: {stray} elements written outside the output window"


# ---- 6. scale bytes over the whole E8M0 range ---------------------------------------------------------------------------------
def _range_operand(rows, K, elem, e, sign, g):
    """MXTensor straight from codes and scale bytes: random finite codes; block j of row r has scale byte 127 + sign * e_j,
    plus a per-row offset in [-3, 3] on the blocks that leave room for it"""
    from torchmx.mx_tensor import MXTensor
    if elem == E4M3:  # magnitudes 0..126: every code but the NaN pair 0x7F / 0xFF
        codes = torch.randint(0, 127, (rows, K), device=DEV, dtype=torch.uint8, generator=g) | (torch.randint(0, 2, (rows, K), device=DEV, dtype=torch.uint8, generator=g) << 7)
    elif elem == FP4:
        codes = torch.randint(0, 256, (rows, K // 2), device=DEV, dtype=torch.uint8, generator=g)
    else:
        codes = torch.randint(0, 64, (rows, K), device=DEV, dtype=torch.uint8, generator=g)
    jitter = torch.randint(-3, 4, (rows, 1), device=DEV, generator=g) * (e.abs() <= 120)
    scale = (127 + sign * e + jitter).to(torch.uint8)
    t = MXTensor(scale, codes, _et(elem), 32, torch.bfloat16)
    # fp64 values: the codes through K2 at unit scale, the scale applied in fp64 (2^127 times a large code overflows float32)
    unit = MXTensor(torch.full_like(scale, 127), codes, _et(elem), 32, torch.bfloat16).to_dtype(torch.float32).double()
    return t, unit * torch.exp2(scale.double() - 127).repeat_interleave(32, -1)


@pytest.mark.parametrize("kernel,M,N,adt,wdt", [(k, m, n, E4M3, w) for (k, m, n) in (("K3c", 33, 1000), ("K3a", 300, 100), ("K3b", 300, 520))
                                                for w in (E4M3, FP6, FP4)] + [("K3b", 300, 520, FP4, FP4)])
def test_scale_bytes_over_the_whole_range(monkeypatch, kernel, M, N, adt, wdt):
    """K = 8192 (256 scale blocks): A's scale byte of block j is 127 + e_j and B's 127 - e_j with e_j running over -127..127, so
    every product has a scale near 2^0 while bytes 0, 1, 253 and 254 reach the MMA; a misread byte is a huge error"""
    from torchmx_b200 import mx_gemm
    monkeypatch.setitem(mx_gemm.overrides, "wide_tiles", kernel == "K3b")
    K = 8192
    g = torch.Generator(device=DEV).manual_seed(M + N + len(wdt) + len(adt))
    e = torch.cat([torch.randperm(255, device=DEV, generator=g) - 127, torch.zeros(1, device=DEV, dtype=torch.int64)])
    A, ad = _range_operand(M, K, adt, e, 1, g)
    B, bd = _range_operand(N, K, wdt, e, -1, g)
    for t in (A, B):
        assert all(bool((t._scale_e8m0 == v).any()) for v in (0, 1, 253, 254))
    t0 = _count()
    y = F.linear(A, B)
    assert _count() == t0 + 1
    ref, S = _refs(ad, bd)
    _check(y, ref, S, None, f"{kernel} {adt}x{wdt}")
