"""Decode-sized MX linears with COLD weights: a CUDA graph cycles through enough distinct weight matrices (> 2 x L2) that every
launch streams its weights from HBM, like a real decoder stack.  Prints us per launch and GB/s of operand+output bytes."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torchmx_b200  # noqa
from torchmx_b200 import dtypes
from torchmx_b200.mx_tensor import MXTensor
wdt = getattr(dtypes, os.environ.get("GT_W", "float6_e3m2"))
FUSED = os.environ.get("GT_FUSED", "0") == "1"  # bf16 activation quantized inside the GEMM (what MXInferenceLinear does at decode sizes)
M = int(os.environ.get("GT_M", "32"))
for shape in os.environ.get("GT_SHAPES", "4096x4096,1024x4096,14336x4096,4096x14336").split(","):
    N, K = (int(v) for v in shape.split("x"))
    n_w = int(os.environ.get("GT_NW", "0")) or max(4, int(400e6 // (N * K)) + 1)  # GT_NW=1: the same (L2-resident) weight every launch
    xb = torch.randn(M, K, device="cuda", dtype=torch.bfloat16)
    X = MXTensor.to_mx(xb, dtypes.float8_e4m3, 32)
    from torchmx_b200 import mx_gemm
    run = (lambda W: mx_gemm.linear_fused_act_quant(xb, W, None)) if FUSED else (lambda W: torch.nn.functional.linear(X, W))
    Ws = [MXTensor.to_mx(torch.randn(N, K, device="cuda", dtype=torch.bfloat16), wdt, 32) for _ in range(n_w)]
    for W in Ws:
        mx_gemm.mark_static(W)
        run(W)
    torch.cuda.synchronize()
    g, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
    with torch.cuda.stream(st):
        with torch.cuda.graph(g, stream=st):
            for W in Ws:
                y = run(W)
    ts = []
    for r in range(4):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / n_w * 1e3)
    us = min(ts[1:])
    bits = {"float4_e2m1": 4, "float6_e3m2": 6, "float6_e2m3": 6, "float8_e4m3": 8}[wdt.name]
    if n_w == 1:  # one launch per replay would time the graph launch: replay a graph of 20 launches on the one weight
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(st):
            with torch.cuda.graph(g, stream=st):
                for _ in range(20):
                    y = run(Ws[0])
        ts = []
        for r in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / 20 * 1e3)
        us = min(ts[1:])
    by = N * K * (bits / 8 + 1 / 32) + M * K * (1 + 1 / 32) + M * N * 2
    print(f"M={M} N={N} K={K} W={wdt.name} fused_act_quant={FUSED} ({n_w} distinct weights): {us:.1f} us per launch, {by/us/1e3:.0f} GB/s of packed operand bytes, {N*K/us/1e6:.2f} T weight elements/s", flush=True)
