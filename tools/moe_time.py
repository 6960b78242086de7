"""Time one mixture-of-experts layer (K6): transformers' bf16 experts (`eager` loop and `grouped_mm`), the MX loop path and the
MX grouped path, at Qwen3-30B-A3B shape (E 128, k 8, H 2048, I 768) and Mixtral-8x7B shape (E 8, k 2, H 4096, I 14336), for
decode (T = 1, 32) and prefill (T = 2048), fp4 / fp6 weights with e4m3 activations.

    python tools/moe_time.py [--out profiles/r6_moe_time.json] [--rounds 3] [--iters 20]

Each call is timed on its own with CUDA events; L2 is overwritten between calls (a 256 MB write outside the timed window), so the
hit experts' weights come from HBM every time.  Paths that can be captured (bf16 grouped_mm, MX grouped) are replayed from a CUDA
graph; the others (host synchronisation in the loop) run eagerly.  Rounds interleave the paths.  Reported per case: median
us per layer, and the weight bytes of the experts the batch hits over that time, beside the HBM rate a 2 GB device copy reaches
in the same run.  The card's name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SHAPES = {"qwen3_30b_a3b": dict(E=128, k=8, H=2048, I=768), "mixtral_8x7b": dict(E=8, k=2, H=4096, I=14336)}
BATCHES = (1, 32, 2048)
WEIGHTS = ("float4_e2m1", "float6_e2m3")
BITS = {"float4_e2m1": 4, "float6_e2m3": 6, "bf16": 16}


def _card():
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    except OSError:
        smi = ""
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi_name_power_limit": smi.splitlines()[0] if smi else "unavailable"}


def _hbm_rate(flush):
    src = torch.empty(2 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    times = []
    for _ in range(10):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        dst.copy_(src)
        b.record()
        torch.cuda.synchronize()
        times.append(a.elapsed_time(b) * 1e-3)
    del src, dst
    return 2 * (2 << 30) / min(times)


def _time(fn, flush, iters):
    out = []
    for _ in range(iters):
        flush.fill_(1)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        out.append(a.elapsed_time(b) * 1e3)
    return out


def _graphed(fn):
    """fn replayed from a CUDA graph, or None when it cannot be captured"""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    try:
        with torch.cuda.stream(s):
            for _ in range(2):
                fn()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            fn()
        return g.replay
    except Exception:  # (host synchronisation inside: not capturable)
        torch.cuda.synchronize()
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r6_moe_time.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "moe_time.py measures on the GPU"
    import torchmx  # noqa: F401
    from transformers import MixtralConfig
    from transformers.models.mixtral.modeling_mixtral import MixtralExperts
    from torchmx_b200.config import MXConfig, QLinearConfig
    from torchmx_b200.layers import mx_experts
    from torchmx_b200.layers.mx_experts import MXInferenceExperts

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    result = {"card": _card(), "hbm_copy_bytes_per_s": _hbm_rate(flush), "rounds": args.rounds, "iters_per_round": args.iters,
              "l2": "overwritten (256 MB write) before every timed call", "cases": []}
    for shape_name, s in SHAPES.items():
        E, k, H, I = s["E"], s["k"], s["H"], s["I"]
        cfg = MixtralConfig(hidden_size=H, intermediate_size=I, num_local_experts=E, num_experts_per_tok=k)
        torch.manual_seed(0)
        bank = MixtralExperts(cfg).to("cuda", torch.bfloat16)
        with torch.no_grad():
            bank.gate_up_proj.normal_(0, 0.02)
            bank.down_proj.normal_(0, 0.02)
        mods = {w: MXInferenceExperts.from_float(bank, QLinearConfig(MXConfig(w, 32), MXConfig("float8_e4m3", 32))) for w in WEIGHTS}
        for T in BATCHES:
            g = torch.Generator(device="cuda").manual_seed(T)
            x = torch.randn(T, H, device="cuda", generator=g).to(torch.bfloat16)
            logits = torch.randn(T, E, device="cuda", generator=g)
            w_top, idx = torch.topk(torch.softmax(logits, -1), k, dim=-1)
            hit = int(torch.unique(idx).numel())
            paths = {}

            def bf16(impl):
                def run():
                    cfg._experts_implementation = impl
                    with torch.no_grad():
                        return bank(x, idx, w_top)
                return run

            paths["bf16_eager"] = (bf16("eager"), False, "bf16")
            paths["bf16_grouped_mm"] = (bf16("grouped_mm"), True, "bf16")
            for w, m in mods.items():
                def loop(m=m):
                    prev = mx_experts.set_grouped(False)
                    try:
                        return m(x, idx, w_top)
                    finally:
                        mx_experts.set_grouped(prev)
                paths[f"mx_loop_{w}"] = (loop, False, w)
                paths[f"mx_grouped_{w}"] = ((lambda m=m: m(x, idx, w_top)), True, w)
            runners = {}
            for name, (fn, capture, _) in paths.items():
                fn()  # warm-up (operand shadows, algorithm choice)
                torch.cuda.synchronize()
                rep = _graphed(fn) if capture else None
                runners[name] = (rep or fn, rep is not None)
            times = {name: [] for name in paths}
            for _ in range(args.rounds):
                for name, (fn, _) in runners.items():
                    times[name].append(statistics.median(_time(fn, flush, args.iters)))
            for name, (_, _, wfmt) in paths.items():
                per_expert = 3 * H * I * BITS[wfmt] / 8 + (3 * H * I / 32 if wfmt != "bf16" else 0)
                us = statistics.median(times[name])
                case = dict(shape=shape_name, T=T, path=name, weights=wfmt, activations="float8_e4m3" if name.startswith("mx") else "bf16",
                            cuda_graph=runners[name][1], us_per_layer=us, us_per_round=times[name], experts_hit=hit,
                            hit_weight_bytes=per_expert * hit, hit_weight_bytes_per_s=per_expert * hit / (us * 1e-6))
                result["cases"].append(case)
                print(f"{shape_name:14s} T={T:5d} {name:28s} {'graph' if case['cuda_graph'] else 'eager'} {us:10.1f} us  "
                      f"{case['hit_weight_bytes_per_s'] / 1e12:6.2f} TB/s of hit weights", flush=True)
            del runners
        del bank, mods
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(f"card: {result['card']}  HBM copy: {result['hbm_copy_bytes_per_s'] / 1e12:.2f} TB/s -> {args.out}")


if __name__ == "__main__":
    main()
