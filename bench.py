#!/usr/bin/env python
"""bench.py -- headline benchmark of the MX quantize / dequantize hot path on B200.

Workload (BASELINE.json configs[1]): quantize/dequantize sweep over a 16384 x 16384 bf16 tensor
for all element types (float8_e4m3, float6_e3m2, float6_e2m3, float4_e2m1, int8), block_size 32.
One "step" = MXTensor.to_mx followed by MXTensor.to_dtype(bfloat16) for each of the five element
types (10 kernel launches).  Metric: algorithmic GB/s = (2 + code + 1/32 bytes per element, once
for quantize and once for dequantize) / device time.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU): the tensors are independent, every rank runs the
same sweep on its own GPU (weak scaling, no data-path collective); time = max over ranks.
`--impl reference` times the CPU oracle (oracle/, the restatement of the reference's own CPU
path -- the Python reference itself cannot travel to the GPU box) with all host threads.
`--dump-outputs DIR` writes a fixed sample of what the last timed step computed (see dump_outputs),
so that two builds can be compared output for output on identical seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ELEMS = ["float8_e4m3", "float6_e3m2", "float6_e2m3", "float4_e2m1", "int8"]
ROWS = COLS = 16384
BLOCK = 32
METRIC = "to_mx/to_dtype GB/s (algorithmic bytes: quantize + dequantize->bf16, 16384x16384 bf16, all elem dtypes, block 32)"


def code_bytes(elem: str) -> float:
    return 0.5 if elem == "float4_e2m1" else 1.0


def algo_bytes(elem: str, n_elems: int) -> float:
    """bytes one quantize (or one dequantize->bf16) of n_elems must move: 2 B hp + code + 1/32 B scale"""
    return n_elems * (2.0 + code_bytes(elem) + 1.0 / BLOCK)


def step_bytes(n_elems: int) -> float:
    return sum(2.0 * algo_bytes(e, n_elems) for e in ELEMS)


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (copy, measured)"
    except Exception:
        return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def bind_to_gpu_numa_node(local_rank: int):
    """Run this process on the CPUs of the NUMA node its GPU hangs off (sysfs; best effort, None when unknown), so that with one rank
    per GPU the pinned host buffers of the e2e leg are first-touched next to their GPU.  On this pool's boxes it is a no-op: they
    expose ONE NUMA node (nvidia-smi topo: every GPU "NUMA affinity 0", numa_node = -1 in sysfs), and the e2e leg saturates at
    ~130 GB/s aggregate from 2 GPUs on (82 GB/s at 1): the host side of the copies, not the kernels, is the limit there."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bus = f"{getattr(pr, 'pci_domain_id', 0):04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"  # sysfs address of the GPU
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                lo, _, hi = part.partition("-")
                cpus.update(range(int(lo), int(hi or lo) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return None
        os.sched_setaffinity(0, allowed)
        return node
    except Exception:  # noqa: BLE001
        return None


def ncu_traffic(kernel_key: str):
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel_key)
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """samples SM clock + throttle reasons through NVML while the timed region runs"""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._halt = index, [], set(), None, threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------
_CPU_BUFS = {}


def cpu_port_throughput(rows: int, threads: int, repeats: int = 1):
    """GB/s of the CPU oracle (the port of the reference's CPU path) on `rows` x 16384 of the workload."""
    import numpy as np
    from oracle import mx_oracle as mxo
    mxo.lib()
    if rows not in _CPU_BUFS:
        rng = np.random.default_rng(0)
        _CPU_BUFS[rows] = (mxo.f32_to_bf16_bits(rng.standard_normal((rows, COLS), dtype=np.float32)),
                           np.zeros((rows, COLS), dtype=np.uint16), np.zeros((rows, COLS // BLOCK), dtype=np.uint8),
                           np.zeros((rows, COLS), dtype=np.uint8), np.zeros((rows, COLS // 2), dtype=np.uint8))
    x, out, scales, codes_full, codes_half = _CPU_BUFS[rows]
    n = x.size
    best = None
    for _ in range(repeats):
        t0 = time.perf_counter()
        for e in ELEMS:
            codes = codes_half if e == "float4_e2m1" else codes_full
            mxo.quantize_into(x, e, BLOCK, scales, codes, threads=threads)
            mxo.dequantize_into(codes, scales, e, BLOCK, out, threads=threads)
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return step_bytes(n) / best / 1e9, best


def run_reference(args):
    """--impl reference: the reference's CPU path (oracle port), all host threads, bounded sample."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    rows = 1024  # 1/16 of the workload per step: ~16.8 M elements x 5 dtypes x (quantize + dequantize)
    for _ in range(max(args.warmup, 1)):
        cpu_port_throughput(rows, threads)
    times = []
    for _ in range(args.steps):
        _, dt = cpu_port_throughput(rows, threads)
        times.append(dt)
    total = sum(times)
    value = step_bytes(rows * COLS) * args.steps / total / 1e9
    sample = f"{rows}x{COLS} bf16 rows of the 16384x16384 workload per step (1/16), all 5 elem dtypes, quantize+dequantize"
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(1e3 * total / args.steps, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8 codes / f32 scaling arithmetic", "data": "synthetic",
        "config": {"workload": "quantize/dequantize sweep 16384x16384 bf16, all elem dtypes, block 32 (BASELINE configs[1])",
                   "sample": sample},
        "cpu_baseline": {"value": round(value, 4), "unit": "GB/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def measured_tensor_peaks():
    """(nominal block-scaled fp8/fp6 dense peak, 2 x measured cuBLAS bf16 burst) in TFLOP/s"""
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return 4500.0, 2.0 * float(json.load(f)["bf16_tflops"]), "2 x MEASURED_PEAKS.json bf16_tflops (cuBLAS burst, measured)"
    except Exception:
        return 4500.0, 2.0 * 1590.0, "2 x fallback 1.59 PFLOP/s (B200_PROFILING.md)"


def mx_matmul_extras(dev):
    """Secondary numbers of the metric ("MX matmul TFLOP/s", BASELINE configs[2]): the 8192^3 fp8_e4m3 x fp6_e3m2 MX linear,
    the 4-D attention Q@K^T MX bmm and one decode-sized linear, each through the public op (F.linear / torch.matmul on
    MXTensors), replayed from a CUDA graph (10 launches) so host dispatch is not in the number; min / median of 5 replays."""
    import torch
    from torchmx_b200 import dtypes, mx_gemm
    from torchmx_b200.mx_tensor import MXTensor

    def timed(fn, n=10, rounds=5):
        fn()
        torch.cuda.synchronize()
        g, st = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.stream(st):
            with torch.cuda.graph(g, stream=st):
                for _ in range(n):
                    fn()
        ts = []
        for r in range(rounds + 1):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            if r:
                ts.append(e0.elapsed_time(e1) / n * 1e3)
        return min(ts), statistics.median(ts)

    out = {}
    gen = torch.Generator(device=dev).manual_seed(7)
    before = dict(mx_gemm.stats)
    # (1) 8192^3 linear
    M = N = K = 8192
    A = MXTensor.to_mx(torch.randn(M, K, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float8_e4m3, BLOCK)
    W = MXTensor.to_mx(torch.randn(N, K, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float6_e3m2, BLOCK)
    us_min, us_med = timed(lambda: torch.nn.functional.linear(A, W))
    nominal, meas2, src = measured_tensor_peaks()
    flops = 2.0 * M * N * K
    out["linear_8192x8192x8192_e4m3xe3m2"] = {
        "us": round(us_med, 1), "us_best": round(us_min, 1), "TFLOP/s": round(flops / us_med / 1e6, 1),
        "roofline": {"bound": "tensor", "kernel": "mx_gemm_pair_kernel (tcgen05 cta_group::2 kind::mxf8f6f4.block_scale)",
                     "achieved": round(flops / us_med / 1e6, 1), "peak": nominal, "unit": "TFLOP/s", "frac": round(flops / us_med / 1e6 / nominal, 4),
                     "peak_source": "nominal dense block-scaled fp8/fp6 (4.5 PFLOP/s)", "frac_of_2x_measured_bf16": round(flops / us_med / 1e6 / meas2, 4),
                     "peak_2x_measured_bf16": meas2, "peak_2x_source": src, "flop_per_launch": flops}}
    del A, W
    # (2) attention-shaped batched MX bmm: Q @ K^T, [1, 32, 2048, 128] x [1, 32, 2048, 128]^T -> bf16 [1, 32, 2048, 2048] (output-bound)
    Q = MXTensor.to_mx(torch.randn(1, 32, 2048, 128, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float8_e4m3, BLOCK)
    Kt = MXTensor.to_mx(torch.randn(1, 32, 2048, 128, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float6_e3m2, BLOCK)
    us_min, us_med = timed(lambda: torch.matmul(Q, Kt.transpose(2, 3)))
    qk_bytes = 32 * 2048 * 2048 * 2 + 2 * 32 * 2048 * 128 * (1 + 1 / 32)
    out["bmm_qk_1x32x2048x2048x128"] = {"us": round(us_med, 1), "us_best": round(us_min, 1), "GB/s": round(qk_bytes / us_med / 1e3, 1),
                                        "TFLOP/s": round(2.0 * 32 * 2048 * 2048 * 128 / us_med / 1e6, 1), "bound": "hbm (268 MB bf16 output)"}
    del Q, Kt
    # (3) decode-sized linear (batch 32 x Llama-3-8B gate_proj): weight streaming
    X = MXTensor.to_mx(torch.randn(32, 4096, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float8_e4m3, BLOCK)
    W = MXTensor.to_mx(torch.randn(14336, 4096, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float6_e3m2, BLOCK)
    us_min, us_med = timed(lambda: torch.nn.functional.linear(X, W))
    w_bytes = 14336 * 4096 * (1 + 1 / 32) + 32 * 4096 * (1 + 1 / 32) + 32 * 14336 * 2
    out["linear_32x14336x4096_decode"] = {"us": round(us_med, 1), "us_best": round(us_min, 1), "GB/s": round(w_bytes / us_med / 1e3, 1),
                                          "bound": "hbm (weight codes + scales read once)"}
    del X, W
    # (3b) the same on COLD weights: a CUDA graph cycles through > 2 x L2 of distinct weight matrices, so every launch streams its
    # weights from HBM like a decoder stack does (tools/decode_gemm_cold.py); packed bytes = what the kernel reads
    from torchmx_b200 import mx_gemm
    peak_gbs, _ = measured_peak_gbs()

    def cold(N, K, wname):
        wdt = getattr(dtypes, wname)
        n_w = max(4, int(400e6 // (N * K)) + 1)
        Xc = MXTensor.to_mx(torch.randn(32, K, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float8_e4m3, BLOCK)
        Ws = [MXTensor.to_mx(torch.randn(N, K, device=dev, dtype=torch.bfloat16, generator=gen), wdt, BLOCK) for _ in range(n_w)]
        for Wc in Ws:
            mx_gemm.mark_static(Wc)
            torch.nn.functional.linear(Xc, Wc)
        torch.cuda.synchronize()
        g, side = torch.cuda.CUDAGraph(), torch.cuda.Stream()
        with torch.cuda.stream(side):
            with torch.cuda.graph(g, stream=side):
                for Wc in Ws:
                    torch.nn.functional.linear(Xc, Wc)
        ts = []
        for _ in range(4):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) / n_w * 1e3)
        us = min(ts[1:])
        bits = {"float4_e2m1": 4, "float6_e3m2": 6, "float8_e4m3": 8}[wname]
        by = N * K * (bits / 8 + 1 / 32) + 32 * K * (1 + 1 / 32) + 32 * N * 2
        del g, Ws
        return {"us": round(us, 1), "GB/s_packed_bytes": round(by / us / 1e3, 1), "frac_of_hbm_peak": round(by / us / 1e3 / peak_gbs, 3),
                "T_weight_elements/s": round(N * K / us / 1e6, 2), "distinct_weights": n_w}

    out["decode_linear_cold_weights_M32"] = {f"{N}x{K}": {w: cold(N, K, w) for w in ("float8_e4m3", "float6_e3m2", "float4_e2m1")}
                                              for (N, K) in ((4096, 4096), (14336, 4096), (57344, 8192))}
    out["decode_linear_cold_weights_M32"]["bound"] = "hbm for one-byte codes; ~0.27 us per K block and SM whatever the element width for the packed formats (DESIGN.md K3c)"
    torch.cuda.empty_cache()
    # (4) the chain between the two attention matmuls as one kernel (K4a): scale + causal rule + softmax + to_mx(P, e4m3)
    from torchmx_b200 import attention_ops, mlp_ops
    scores = (torch.randn(1, 32, 2048, 2048, device=dev, generator=gen) * 11).to(torch.bfloat16)
    us_min, us_med = timed(lambda: attention_ops.softmax_to_mx(scores, 128 ** -0.5, None, True, dtypes.float8_e4m3, BLOCK))
    n_el = 32 * 2048 * 2048
    out["softmax_to_mx_1x32x2048x2048_causal"] = {"us": round(us_med, 1), "us_best": round(us_min, 1),
                                                  "GB/s_all_blocks": round(n_el * (3 + 1 / 32) / us_med / 1e3, 1),
                                                  "GB/s_moved": round(n_el * (1 + 1 + 1 / 32) / us_med / 1e3, 1),
                                                  "bound": "instruction issue (exact expf / divide per visible element), see DESIGN.md K4a"}
    del scores
    # (5) SwiGLU gating + quantization of down_proj's input (K1b) on a 2048-token Llama-3-8B MLP activation
    gate_up = torch.randn(2048, 2 * 14336, device=dev, dtype=torch.bfloat16, generator=gen)
    g_, u_ = gate_up.split([14336, 14336], dim=-1)
    us_min, us_med = timed(lambda: mlp_ops.silu_mul_to_mx(g_, u_, dtypes.float8_e4m3, BLOCK))
    out["silu_mul_to_mx_2048x14336"] = {"us": round(us_med, 1), "us_best": round(us_min, 1),
                                        "GB/s": round(2048 * 14336 * (5 + 1 / 32) / us_med / 1e3, 1), "bound": "hbm (2 + 2 + 1 + 1/32 B per element)"}
    del gate_up, g_, u_
    # (6) SURVEY 8(d) config 2 side conditions: the quantize / dequantize times must not depend on the value distribution
    # (plain N(0,1); per-block exponents spread over 2^+-40; every bf16 bit pattern incl. NaN / Inf / subnormals), plus the
    # fp32 dequantize target and the float8_e5m2 extension element type.  16384 x 16384, CUDA-graph replay of 4 launches.
    R = C = 16384
    n_el = R * C
    dist = {}
    x0 = torch.randn(R, C, device=dev, dtype=torch.bfloat16, generator=gen)
    variants = {"normal": lambda: x0,
                "wide_2^+-40_per_block": lambda: (x0.view(R, C // 32, 32) * torch.exp2(torch.randint(-40, 41, (R, C // 32, 1), device=dev, generator=gen).float()).to(torch.bfloat16)).view(R, C),
                "all_bf16_bit_patterns": lambda: torch.arange(n_el, device=dev, dtype=torch.int32).bitwise_and_(0xFFFF).to(torch.int16).view(torch.bfloat16).view(R, C)}
    for name, make in variants.items():
        x = make().contiguous()
        _, q_us = timed(lambda: MXTensor.to_mx(x, dtypes.float8_e4m3, BLOCK), n=4, rounds=3)
        m = MXTensor.to_mx(x, dtypes.float8_e4m3, BLOCK)
        _, d_us = timed(lambda: m.to_dtype(torch.bfloat16), n=4, rounds=3)
        dist[name] = {"to_mx_e4m3_us": round(q_us, 1), "to_dtype_bf16_us": round(d_us, 1), "GB/s": [round(n_el * (3 + 1 / 32) / q_us / 1e3, 1), round(n_el * (3 + 1 / 32) / d_us / 1e3, 1)]}
        del x, m
    out["value_distribution_independence_16384x16384"] = dist
    m8, m4 = MXTensor.to_mx(x0, dtypes.float8_e4m3, BLOCK), MXTensor.to_mx(x0, dtypes.float4_e2m1, BLOCK)
    _, us8 = timed(lambda: m8.to_dtype(torch.float32), n=4, rounds=3)
    _, us4 = timed(lambda: m4.to_dtype(torch.float32), n=4, rounds=3)
    out["to_dtype_fp32_16384x16384"] = {"float8_e4m3": {"us": round(us8, 1), "GB/s": round(n_el * (5 + 1 / 32) / us8 / 1e3, 1)},
                                        "float4_e2m1": {"us": round(us4, 1), "GB/s": round(n_el * (4.5 + 1 / 32) / us4 / 1e3, 1)}}
    # secondary K2 / K1 paths: the transposing dequantize (`MXTensor.t().to_dtype()`: blocked axis physically innermost, logically
    # second-to-last) and float32 input to `to_mx` (labelled extension)
    _, us8t = timed(lambda: m8.t().to_dtype(torch.bfloat16), n=4, rounds=3)
    _, us4t = timed(lambda: m4.t().to_dtype(torch.bfloat16), n=4, rounds=3)
    out["t_to_dtype_bf16_16384x16384"] = {"float8_e4m3": {"us": round(us8t, 1), "GB/s": round(n_el * (3 + 1 / 32) / us8t / 1e3, 1)},
                                          "float4_e2m1": {"us": round(us4t, 1), "GB/s": round(n_el * (2.5 + 1 / 32) / us4t / 1e3, 1)}}
    del m8, m4
    x32 = x0.float()
    _, us32 = timed(lambda: MXTensor.to_mx(x32, dtypes.float8_e4m3, BLOCK), n=4, rounds=3)
    out["to_mx_float32_input_extension_16384x16384"] = {"us": round(us32, 1), "GB/s": round(n_el * (5 + 1 / 32) / us32 / 1e3, 1), "parity": "unpinned (the reference asserts bf16 input)"}
    del x32
    _, us5 = timed(lambda: MXTensor.to_mx(x0, dtypes.float8_e5m2, BLOCK), n=4, rounds=3)
    out["to_mx_float8_e5m2_extension_16384x16384"] = {"us": round(us5, 1), "GB/s": round(n_el * (3 + 1 / 32) / us5 / 1e3, 1), "parity": "unpinned (element type absent from the reference)"}
    del x0
    # (7) fp4 x fp4 on kind::mxf4 (dense 4-bit operand streams, twice the rate of kind::mxf8f6f4) -- and the same operands on
    # kind::mxf8f6f4 beside it
    A4 = MXTensor.to_mx(torch.randn(M, K, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float4_e2m1, BLOCK)
    W4 = MXTensor.to_mx(torch.randn(N, K, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.float4_e2m1, BLOCK)
    us_min, us_med = timed(lambda: torch.nn.functional.linear(A4, W4))
    mx_gemm.overrides["no_mxf4"] = True
    try:
        _, us_f8 = timed(lambda: torch.nn.functional.linear(A4, W4))
    finally:
        mx_gemm.overrides["no_mxf4"] = False
    out["linear_8192x8192x8192_e2m1xe2m1_mxf4"] = {
        "us": round(us_med, 1), "us_best": round(us_min, 1), "TFLOP/s": round(flops / us_med / 1e6, 1), "same_operands_on_mxf8f6f4_us": round(us_f8, 1),
        "roofline": {"bound": "tensor", "kernel": "mx_gemm_pair_kernel<MXF4> (tcgen05 cta_group::2 kind::mxf4.block_scale.scale_vec::2X)",
                     "achieved": round(flops / us_med / 1e6, 1), "peak": 9000.0, "unit": "TFLOP/s", "frac": round(flops / us_med / 1e6 / 9000.0, 4),
                     "peak_source": "nominal dense fp4 (9 PFLOP/s)", "frac_of_4x_measured_bf16": round(flops / us_med / 1e6 / (2 * meas2), 4)}}
    del A4, W4
    # (8) operands the block-scaled MMA cannot take (int8 elements: the reference's chat example) -> K3d, dequantize fused into a
    # bf16 tcgen05 GEMM; beside it the recipe it replaces (two K2 launches + a cuBLAS bf16 GEMM)
    Mi, Ni, Ki = 2048, 4096, 4096
    Ai = MXTensor.to_mx(torch.randn(Mi, Ki, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.int8, BLOCK)
    Wi = MXTensor.to_mx(torch.randn(Ni, Ki, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.int8, BLOCK)
    d0, o0 = mx_gemm.stats["dequant_gemm"], mx_gemm.stats.get("dequant_once_gemm", 0)
    _, us_k3d = timed(lambda: torch.nn.functional.linear(Ai, Wi), n=4)
    used_k3d = mx_gemm.stats["dequant_gemm"] > d0
    once = mx_gemm.stats.get("dequant_once_gemm", 0) > o0
    Xi = MXTensor.to_mx(torch.randn(32, Ki, device=dev, dtype=torch.bfloat16, generator=gen), dtypes.int8, BLOCK)
    _, us_dec = timed(lambda: torch.nn.functional.linear(Xi, Wi), n=4)
    prev = mx_gemm.set_dequant_gemm(False)
    try:
        _, us_lib = timed(lambda: torch.nn.functional.linear(Ai, Wi), n=4)
    finally:
        mx_gemm.set_dequant_gemm(prev)
    fi = 2.0 * Mi * Ni * Ki
    out["linear_2048x4096x4096_int8_dequant_gemm"] = {
        "us": round(us_k3d, 1), "TFLOP/s": round(fi / us_k3d / 1e6, 1),
        "kernel_used": ("two K2 launches (each operand dequantized once) + mx_gemm_dequant_kernel in bf16-direct mode (tcgen05 kind::f16, operands by TMA)" if once
                        else "mx_gemm_dequant_kernel (K3d, dequantization fused)") if used_k3d else "fallback",
        "decode_32x4096x4096_fused_us": round(us_dec, 1),
        "k2_plus_cublas_bf16_us": round(us_lib, 1),
        "roofline": {"bound": "tensor", "achieved": round(fi / us_k3d / 1e6, 1), "peak": meas2 / 2, "unit": "TFLOP/s", "frac": round(fi / us_k3d / 1e6 / (meas2 / 2), 4),
                     "peak_source": "measured cuBLAS bf16 (kind::f16 operands)", "note": "large outputs: each operand dequantized once, then a single-CTA 128x128 bf16 tcgen05 GEMM (shared-memory-bandwidth bound at this tile size); small / decode outputs: dequantization fused into the GEMM, CUDA-core bound; see DESIGN.md K3d"}}
    del Ai, Wi, Xi
    # (9) MX attention as one kernel (K4b) vs the bmm -> K4a -> bmm chain: a Llama-3-8B layer at 2048 tokens (32 query / 8 key-value
    # heads, head_dim 128, e4m3 Q / K / V / P, causal)
    from torchmx_b200.layers.mx_llama_attention import _repeat_heads
    q = torch.randn(1, 32, 2048, 128, device=dev, dtype=torch.bfloat16, generator=gen)
    k = torch.randn(1, 8, 2048, 128, device=dev, dtype=torch.bfloat16, generator=gen)
    v = torch.randn(1, 8, 2048, 128, device=dev, dtype=torch.bfloat16, generator=gen)
    E8 = dtypes.float8_e4m3
    Qm, Km, Vt = MXTensor.to_mx(q, E8, BLOCK), MXTensor.to_mx(k, E8, BLOCK), MXTensor.to_mx(v.transpose(2, 3).contiguous(), E8, BLOCK)

    def chain():
        kk, vv = _repeat_heads(Km, 4), _repeat_heads(Vt, 4).transpose(2, 3)
        p_ = attention_ops.softmax_to_mx(torch.matmul(Qm, kk.transpose(2, 3)), 128 ** -0.5, None, True, E8, BLOCK)
        return torch.matmul(p_, vv).transpose(1, 2).contiguous()

    f0 = attention_ops.stats["flash_attention"]
    _, us_fa = timed(lambda: attention_ops.flash_attention(Qm, Km, Vt, 128 ** -0.5, None, True, E8, BLOCK))
    _, us_ch = timed(chain, n=4)
    io_bytes = (32 + 2 * 8) * 2048 * 128 * (1 + 1 / 32) + 32 * 2048 * 128 * 2
    out["mx_attention_1x32x2048x128_causal"] = {
        "flash_kernel_us": round(us_fa, 1), "bmm_softmax_bmm_chain_us": round(us_ch, 1), "kernel_used": attention_ops.stats["flash_attention"] > f0,
        "algorithmic_bytes": int(io_bytes), "chain_extra_hbm_bytes": int(32 * 2048 * 2048 * (2 + 2 + 2 * (1 + 1 / 32))),
        "bound": "instruction issue: three exact softmax passes over the visible scores (row max, row sum, P) -- the reference quantizes the NORMALISED probabilities"}
    del q, k, v, Qm, Km, Vt
    out["tensor_core_calls"] = mx_gemm.stats["tensor_core"] - before["tensor_core"]
    out["fallback_calls"] = mx_gemm.stats["fallback"] - before["fallback"]
    return out


def llama8b_extras():
    """BASELINE configs[3] ("MX-Llama tokens/s"): random-init HF Llama-3-8B, weights fp6_e3m2 / activations fp8_e4m3 through the
    public API -- `quantize_linear_` (the reference's call) and `quantize_llm_` (MX attention / MLP blocks) -- prefill of 2048
    tokens and decode at batch 32, CUDA events; each with its roofline: prefill against the block-scaled tensor peak
    (2 * weight elements * tokens flop), decode against streaming the weight codes + scales once per step."""
    import gc

    import torch
    from tools import llama_bench
    out = {}
    peak_hbm, _ = measured_peak_gbs()
    for key, kw in (("quantize_linear_", dict(llm_api=False)), ("quantize_llm_fused_norm", dict(llm_api=True, fuse_norm=True)),
                    ("quantize_llm_mx_attention_fused_norm", dict(llm_api=True, fuse_norm=True, mx_attention=True))):
        try:
            r = llama_bench.run_cfg(model="8b", steps=32, prefill_iters=3, **kw)
        except Exception as e:  # noqa: BLE001  (the headline line must still be printed)
            out[key] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
            continue
        w_el = r["weight_elements"]
        stream_bytes = w_el * (1 + 1 / 32)  # reference layout: one byte per fp6 code + one scale byte per 32
        pre_ms = r.get("prefill_graph_ms", r["prefill_eager_ms"])
        dec_ms = r.get("decode_graph_ms_per_step", r["decode_eager_ms_per_step"])
        out[key] = {
            "quantize": {"wall_s": round(r["quantize_wall_s"], 4), "gpu_ms": round(r["quantize_gpu_ms"], 2), "GB/s": round(r["quantize_GBps_gpu"], 1),
                         "algorithmic_bytes": w_el * (2 + 1 + 1 / 32), "frac_of_hbm_peak": round(r["quantize_GBps_gpu"] / peak_hbm, 4), "linears": r["linears"]},
            "prefill_2048": {"ms": round(pre_ms, 3), "tok/s": round(2048 / pre_ms * 1e3, 1), "eager_ms": round(r["prefill_eager_ms"], 3),
                             "flop": 2.0 * w_el * 2048, "TFLOP/s": round(2.0 * w_el * 2048 / pre_ms / 1e9, 1),
                             "frac_of_block_scaled_peak": round(2.0 * w_el * 2048 / pre_ms / 1e9 / 4500.0, 4)},
            "decode_batch32": {"ms_per_step": round(dec_ms, 3), "tok/s": round(32 / dec_ms * 1e3, 1), "eager_ms_per_step": round(r["decode_eager_ms_per_step"], 3),
                               "weight_stream_bytes": stream_bytes, "weight_stream_floor_ms": round(stream_bytes / peak_hbm / 1e6, 3),
                               "frac_of_weight_stream_roofline": round(stream_bytes / peak_hbm / 1e6 / dec_ms, 4)},
            "timing": "CUDA-graph replay of the whole forward (eager numbers beside it include Python dispatch)",
            "gemm_stats": r["gemm_stats"], "attention_stats": r.get("attention_stats"), "resident_GB": round(r["resident_after_run_GB"], 2),
        }
        gc.collect()
        torch.cuda.empty_cache()
    return out


def tp70b_extras(world, rank):
    """BASELINE configs[4]: Llama-3-70B shape, fp4_e2m1 weights / fp8_e4m3 activations.  (i) layer-sharded weight quantization
    (80 layers / N ranks, no collective), (ii) tensor-parallel MX-linear inference: column-parallel q/k/v/gate/up, row-parallel
    o/down with an all-reduce of the bf16 [tokens, 8192] partials -- NCCL, and fused into the GEMM epilogue (NVLink multicast)
    for decode.  Strong scaling: the same model on N GPUs; compare the lines of the N = 1, 2, 4, 8 runs."""
    import torch
    from tools import tp_llama_bench as tp
    out = {}
    try:
        out["tp_infer"] = tp.run_infer(tp.default_args(iters=3, also_fused=True), world, rank)
    except Exception as e:  # noqa: BLE001
        out["tp_infer"] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
    torch.cuda.empty_cache()
    try:
        out["layer_sharded_quantize"] = tp.run_quantize(tp.default_args(mode="quantize"), world, rank)
    except Exception as e:  # noqa: BLE001
        out["layer_sharded_quantize"] = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
    torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------
DUMP_ROWS = 64  # 64 of the 16384 rows: ~39 MB of float32 over the five element types (codes, scales, dequantized values)


def dump_outputs(outs, directory: str):
    """Write what the caller of the timed path received in one step -- per element type the MXTensor's codes (`_data`) and E8M0
    scales (`_scale_e8m0`) and the dequantized bf16 tensor -- restricted to the same DUMP_ROWS rows, picked with a fixed seed, as
    float32 `<elem>_{codes,scales,dequantized}.npy` (every value is exact in float32: byte codes, scale bytes, bf16)."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    rows = torch.randperm(ROWS, generator=torch.Generator().manual_seed(0))[:DUMP_ROWS].sort().values
    for elem, (m, y) in zip(ELEMS, outs):
        idx = rows.to(y.device)
        for name, t in (("codes", m._data), ("scales", m._scale_e8m0), ("dequantized", y)):
            np.save(os.path.join(directory, f"{elem}_{name}.npy"), t[idx].float().cpu().numpy())


def run_b200(args):
    import torch
    import torchmx_b200  # noqa: F401  registers the ops; raises if libmxq.so is missing
    from torchmx_b200 import _C, dtypes
    from torchmx_b200.mx_tensor import MXTensor
    _C.lib()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    n_elems = ROWS * COLS
    etypes = [dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[e] for e in ELEMS]
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    # three rotating 512 MiB inputs (each > 126 MB L2), N(0,1) with a per-row power-of-two spread
    xs = []
    for _ in range(3):
        x = torch.randn(ROWS, COLS, dtype=torch.bfloat16, device=dev, generator=g)
        x *= torch.exp2(torch.randint(-20, 20, (ROWS, 1), device=dev, generator=g).float()).to(torch.bfloat16)
        xs.append(x)

    def step(i, ev=None):
        x = xs[i % 3]
        outs = []
        for j, et in enumerate(etypes):
            if ev is not None:
                ev[j][0].record()
            m = MXTensor.to_mx(x, et, BLOCK)
            if ev is not None:
                ev[j][1].record()
            y = m.to_dtype(torch.bfloat16)
            if ev is not None:
                ev[j][2].record()
            outs.append((m, y))
        return outs

    # Warm-up keeps each step's results alive the way the timed loop does, so the caching allocator already holds every block
    # the timed loop asks for.
    for i in range(args.warmup):
        outs = step(i)
    # per-launch events (on the launching = current stream) for the roofline of the dominant kernel
    evs = [[[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in ELEMS] for _ in range(args.steps)]
    t_start, t_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    # A device-side wait (~10 ms, before the first timed event) lets the eager Python dispatch run ahead of the GPU, as it does in
    # steady state: the timed region is only steps x 1.2 ms long, and with 8 ranks sharing the host cores one descheduled process
    # otherwise shows up as a GPU idle gap in the max over ranks (seen once: 1.37 instead of 1.21 ms/step with identical kernel times).
    torch.cuda._sleep(20_000_000)
    t_start.record()
    for i in range(args.steps):
        outs = step(i, evs[i])
    t_end.record()
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        dump_outputs(outs, args.dump_outputs)
    del outs
    elapsed_ms = t_start.elapsed_time(t_end)
    if dist is not None:
        t = torch.tensor([elapsed_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    value = world * step_bytes(n_elems) * args.steps / (elapsed_ms * 1e-3) / 1e9

    # ---- per-kernel durations -> roofline of the kernel with the largest share of the step
    q_ms = {e: statistics.mean(evs[i][j][0].elapsed_time(evs[i][j][1]) for i in range(args.steps)) for j, e in enumerate(ELEMS)}
    d_ms = {e: statistics.mean(evs[i][j][1].elapsed_time(evs[i][j][2]) for i in range(args.steps)) for j, e in enumerate(ELEMS)}
    kernels = {}
    for e in ELEMS:
        kernels[f"quantize_b32_bf16_kernel<{e}>"] = {"ms": q_ms[e], "GB/s": algo_bytes(e, n_elems) / (q_ms[e] * 1e-3) / 1e9}
        kernels[f"dequantize_b32_kernel<{e},bf16>"] = {"ms": d_ms[e], "GB/s": algo_bytes(e, n_elems) / (d_ms[e] * 1e-3) / 1e9}
    families = {
        "dequantize_b32_kernel (1-byte codes -> bf16)": [f"dequantize_b32_kernel<{e},bf16>" for e in ELEMS if e != "float4_e2m1"],
        "quantize_b32_bf16_kernel (bf16 -> 1-byte codes)": [f"quantize_b32_bf16_kernel<{e}>" for e in ELEMS if e != "float4_e2m1"],
    }
    fam_ms = {k: sum(kernels[n]["ms"] for n in v) for k, v in families.items()}
    dom = max(fam_ms, key=fam_ms.get)
    dom_launch_ms = fam_ms[dom] / len(families[dom])
    peak, peak_src = measured_peak_gbs()
    achieved = algo_bytes("float8_e4m3", n_elems) / (dom_launch_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": dom, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "frac_of_8TBps": round(achieved / 8000.0, 4), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_bytes("float8_e4m3", n_elems), "avg_launch_us": round(dom_launch_ms * 1e3, 2),
                "traffic": ncu_traffic(dom), "traffic_source": "profiles/traffic.json (dram__bytes_read + dram__bytes_write of one ncu --set full capture; not re-measured in this run)",
                "share_of_step": round(fam_ms[dom] / (elapsed_ms / args.steps), 4)}

    # ---- end to end through the public API with HOST buffers (pinned), copies inside the timed region
    e2e_steps = max(1, min(args.steps, 5))
    numa = bind_to_gpu_numa_node(local)  # the pinned buffers below are first-touched on the GPU's own NUMA node (N > 1: no shared DRAM channel)
    xh = torch.empty(ROWS, COLS, dtype=torch.bfloat16).pin_memory()
    xh.copy_(xs[0])

    # Four streams, one per pipeline stage, chained by events, so that the PCIe link carries traffic in both directions all the
    # time: s0 H2D input + to_mx, s1 D2H codes + scales, s2 H2D the codes + scales that just reached the host + to_dtype, s3
    # D2H result.  Stage k of element type i waits for stage k-1 of element type i only, so the stages of consecutive element
    # types overlap.  Same bytes, same ops and the same host round trip per step as a single-stream version.
    st = [torch.cuda.Stream(dev) for _ in range(4)]
    chs = {et.name: (torch.empty(ROWS, COLS if code_bytes(et.name) == 1.0 else COLS // 2, dtype=torch.uint8).pin_memory(),
                     torch.empty(ROWS, COLS // BLOCK, dtype=torch.uint8).pin_memory()) for et in etypes}
    yhs = [torch.empty(ROWS, COLS, dtype=torch.bfloat16).pin_memory() for _ in range(2)]

    def e2e_run(n_steps):
        """n_steps passes over the host batch, pipelined: nothing waits between steps except where a pinned host buffer is reused
        (the download of a step's codes waits for the previous step's upload out of the same buffer), so step k + 1's uploads
        overlap step k's downloads and the link stays busy in both directions; ONE synchronize at the end."""
        h2d = d2h = 0
        for s_ in st:
            s_.wait_stream(torch.cuda.current_stream())
        keep = []
        reupload_done = {et.name: None for et in etypes}
        for step in range(n_steps):
            for i, et in enumerate(etypes):
                c_host, s_host = chs[et.name]
                with torch.cuda.stream(st[0]):
                    xd = xh.to(dev, non_blocking=True)                                   # H2D: the step's input
                    m = MXTensor.to_mx(xd, et, BLOCK)
                    e0 = torch.cuda.Event(); e0.record(st[0])
                with torch.cuda.stream(st[1]):
                    st[1].wait_event(e0)
                    if reupload_done[et.name] is not None:
                        st[1].wait_event(reupload_done[et.name])                        # the host buffer is free again
                    c_host.view(m._data.dtype).copy_(m._data, non_blocking=True)         # D2H: the quantized result
                    s_host.copy_(m._scale_e8m0, non_blocking=True)
                    e1 = torch.cuda.Event(); e1.record(st[1])
                with torch.cuda.stream(st[2]):
                    st[2].wait_event(e1)
                    cd = c_host.view(m._data.dtype).to(dev, non_blocking=True)           # H2D: codes + scales back in
                    sdv = s_host.to(dev, non_blocking=True)
                    e2u = torch.cuda.Event(); e2u.record(st[2])
                    reupload_done[et.name] = e2u
                    y = MXTensor(sdv, cd, et, BLOCK, torch.bfloat16).to_dtype(torch.bfloat16)
                    e2 = torch.cuda.Event(); e2.record(st[2])
                with torch.cuda.stream(st[3]):
                    st[3].wait_event(e2)
                    yh = yhs[i % 2]
                    yh.copy_(y, non_blocking=True)                                       # D2H: the dequantized result
                keep.append((xd, m, cd, sdv, y))  # alive until the final synchronize (no allocator reuse across streams)
                if step == 0:
                    h2d += xh.numel() * 2 + c_host.numel() + s_host.numel()
                    d2h += c_host.numel() + s_host.numel() + yh.numel() * 2
        for s_ in st:
            s_.synchronize()
        return h2d, d2h

    h2d = d2h = 0
    if args.skip_e2e:
        e2e_steps = 0
    else:
        e2e_run(e2e_steps)  # (the same number of steps as the timed run: every device block it needs is in the caching allocator afterwards)
    barrier()
    t0 = time.perf_counter()
    if e2e_steps:
        h2d, d2h = e2e_run(e2e_steps)
    barrier()
    e2e_s = max(time.perf_counter() - t0, 1e-9)
    if dist is not None:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_value = world * step_bytes(n_elems) * e2e_steps / e2e_s / 1e9 if e2e_steps else 0.0
    # what the link itself does: the same pinned buffers copied in both directions at once, nothing else running (rank 0's number
    # is reported; at N > 1 every rank copies at the same time, like in the e2e leg)
    link = None
    if e2e_steps:
        dbuf_in, dbuf_out = torch.empty_like(xh, device=dev), torch.empty_like(xh, device=dev)
        def duplex(reps):
            for _ in range(reps):
                with torch.cuda.stream(st[0]):
                    dbuf_in.copy_(xh, non_blocking=True)
                with torch.cuda.stream(st[1]):
                    yhs[0].copy_(dbuf_out, non_blocking=True)
            st[0].synchronize(); st[1].synchronize()
        duplex(1)
        barrier()
        t0 = time.perf_counter()
        duplex(6)
        link_s = time.perf_counter() - t0
        per_dir = 6 * xh.numel() * 2 / link_s / 1e9
        link = {"each_direction_when_both_GBps": round(per_dir, 1), "e2e_achieved_per_direction_GBps": round(h2d * e2e_steps / e2e_s / 1e9, 1),
                "frac": round((h2d * e2e_steps / e2e_s / 1e9) / per_dir, 3), "note": "512 MiB pinned copies, H2D and D2H at once, measured right after the e2e leg"}
        del dbuf_in, dbuf_out

    extras = llama = tp70b = None
    del xs, xh, yhs, chs
    torch.cuda.empty_cache()
    if rank == 0 and not args.skip_gemm and world == 1:  # single-GPU numbers; under torchrun the other ranks would only wait
        try:
            extras = mx_matmul_extras(dev)
        except Exception as e:  # noqa: BLE001  (secondary numbers must never cost the headline line)
            extras = {"error": f"{type(e).__name__}: {str(e)[:300]}"}
        torch.cuda.empty_cache()
    if not args.skip_llama:
        if world == 1:
            llama = llama8b_extras()
            import torch.distributed as dist1
            if not dist1.is_initialized():  # the tensor-parallel harness synchronises through a process group, also with one rank
                import socket
                sk = socket.socket(); sk.bind(("127.0.0.1", 0)); port = sk.getsockname()[1]; sk.close()
                dist1.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=0, world_size=1, device_id=dev)
        tp70b = tp70b_extras(world, rank)
    if rank == 0:
        cpu_threads = os.cpu_count() or 1
        cpu_rows = 2048
        cpu_value, cpu_dt = (None, None)
        if not args.skip_cpu:
            cpu_port_throughput(256, cpu_threads)  # warm the pages / thread pool
            cpu_value, cpu_dt = cpu_port_throughput(cpu_rows, cpu_threads, repeats=2)
        line = {
            "metric": METRIC, "value": round(value, 1), "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(elapsed_ms / args.steps, 4), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8 codes / f32 scaling arithmetic", "data": "synthetic",
            "config": {"workload": "quantize/dequantize sweep 16384x16384 bf16, all elem dtypes (fp8 e4m3, fp6 e3m2/e2m3, fp4 e2m1, int8), "
                                   "block 32 (BASELINE configs[1])",
                       "step": "to_mx + to_dtype(bf16) per elem dtype = 10 launches", "l2": "inputs (512 MiB, 3 rotating) larger than L2", "host_lead": "a ~10 ms device-side wait precedes the first timed event, so eager dispatch runs ahead of the GPU",
                       "parallelism": f"independent tensors per GPU x{world}, no collective"},
            "clocks": clocks,
            "e2e": {"value": round(e2e_value, 2), "unit": "GB/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": round(1e3 * e2e_s / max(e2e_steps, 1), 2), "pcie_link": link, "note": "pinned host buffers, every PCIe copy of every step inside the timed region; four pipelined streams (H2D / D2H overlap, full-duplex PCIe), steps pipelined behind each other, one synchronize at the end of the timed region",
                    "host_numa_node_of_rank0": numa},
            "gpu_launches": args.steps * 2 * len(ELEMS),
            "roofline": roofline,
            "cpu_baseline": None if cpu_value is None else {
                "value": round(cpu_value, 3), "unit": "GB/s", "cores": cpu_threads, "kind": "port",
                "sample": f"{cpu_rows}x{COLS} rows of the workload (1/8), all 5 elem dtypes, quantize+dequantize, best of 2, {cpu_dt:.2f} s",
                "python_reference_context": "the unmodified Python reference (torch CPU ops) measured 0.04-1.8 GB/s on 8 cores on this workload (BASELINE.md section 4); it cannot travel to the GPU box, the C port (validated against it bit for bit) is what is timed here"},
            "kernels": {k: {"us": round(v["ms"] * 1e3, 2), "GB/s": round(v["GB/s"], 1)} for k, v in kernels.items()},
            "mx_matmul": extras,
            "llama8b": llama,
            "tp70b": tp70b,
        }
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--skip-cpu", action="store_true", help="profiling runs only: skip the cpu_baseline leg")
    ap.add_argument("--skip-gemm", action="store_true", help="skip the secondary MX matmul numbers (rank 0, after the timed sweep)")
    ap.add_argument("--skip-llama", action="store_true", help="skip the MX-Llama extras (8B through the public API at N = 1, 70B tensor-parallel at every N)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write a fixed row sample of the last step's codes, scales and "
                                                          "dequantized tensors of every element type to DIR/<name>.npy (float32, rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
