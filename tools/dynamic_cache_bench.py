"""MX-attention decode of a Llama-3-8B-shaped model (random init, `--layers` layers; weights fp6_e3m2 / activations fp8_e4m3, e4m3
Q / K / V / P) with transformers' bf16 DynamicCache against MXDynamicCache, at batch 1 / 8 / 32 and contexts ctx + 17 (a key length
that is not a multiple of 32, as on 31 of 32 decode steps):
  * ms per decode step: `--steps` eager steps between CUDA events (a dynamic cache changes its host-side length every step, so
    it cannot be replayed from a CUDA graph), the two caches alternating, `--reps` times;
  * the resident bytes of each cache;
  * K4b alone at Llama-3-8B decode heads (32 query / 8 key-value heads): microseconds per call at the ragged kv_len = ctx + 17
    read in place from a cache-shaped buffer, against the aligned kv_len = n = ceil128(ctx + 17) in the same mode and against the
    plain call on n contiguous keys (CUDA-graph replay of 10 calls, the three alternating, min over 5 rounds).
Both caches are filled directly with random keys / values (no prefill through the model: a batch-32 prompt of 32768 tokens does not
fit the activations of the MLP); the MX cache through K5e, its append kernel.

    python tools/dynamic_cache_bench.py [--layers 4] [--batch 1 8 32] [--ctx 1024 4096 32768] [--out profiles/r5_dynamic_cache_decode.json]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from tools import llama_bench  # noqa: E402

HQ, HK, D = 32, 8, 128


def fill(model, cfg, cache, B, L, mx: bool, seed: int) -> None:
    g = torch.Generator(device="cuda").manual_seed(seed)
    for i, block in enumerate(model.model.layers):
        if not mx:
            k = torch.randn(B, HK, L, D, device="cuda", dtype=torch.bfloat16, generator=g)
            cache.update(k, torch.randn(B, HK, L, D, device="cuda", dtype=torch.bfloat16, generator=g), i)
            continue
        for lo in range(0, L, 2048):
            t = min(2048, L - lo)
            q = torch.randn(B, t, HQ, D, device="cuda", dtype=torch.bfloat16, generator=g).transpose(1, 2)
            k = torch.randn(B, t, HK, D, device="cuda", dtype=torch.bfloat16, generator=g).transpose(1, 2)
            v = torch.randn(B, t, HK, D, device="cuda", dtype=torch.bfloat16, generator=g).transpose(1, 2)
            cos = torch.ones(1, t, D, device="cuda", dtype=torch.bfloat16)
            cache.layers[i].mx_append(q, k, v, cos, torch.zeros_like(cos), block.self_attn.qconfig)


def decode_time(model, cfg, caches, B, L, steps, reps):
    tok = torch.randint(0, cfg.vocab_size, (B, 1), device="cuda")
    times = {k: [] for k in caches}
    for r in range(reps + 1):  # (round 0 warms up)
        for kind, cache in caches.items():
            cache.crop(L)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                model(input_ids=tok, past_key_values=cache, use_cache=True)
            e1.record()
            torch.cuda.synchronize()
            if r:
                times[kind].append(round(e0.elapsed_time(e1) / steps, 4))
    return times


def k4b_time(B, L, seed):
    """us per K4b call: ragged kv_len L in place, aligned kv_len n in place, the plain call on n keys"""
    from torchmx_b200 import attention_ops, dtypes
    from torchmx_b200.mx_tensor import MXTensor
    E = dtypes.float8_e4m3
    n = -(-L // 128) * 128
    g = torch.Generator(device="cuda").manual_seed(seed)
    q = MXTensor.to_mx(torch.randn(B, HQ, 1, D, device="cuda", dtype=torch.bfloat16, generator=g), E, 32)
    k = MXTensor.to_mx(torch.randn(B, HK, n, D, device="cuda", dtype=torch.bfloat16, generator=g), E, 32)
    vt = MXTensor.to_mx(torch.randn(B, HK, D, n, device="cuda", dtype=torch.bfloat16, generator=g), E, 32)
    calls = {"ragged_in_place": lambda: attention_ops.flash_attention(q, k, vt, D ** -0.5, None, False, E, 32, kv_len=L),
             "aligned_in_place": lambda: attention_ops.flash_attention(q, k, vt, D ** -0.5, None, False, E, 32, kv_len=n),
             "plain": lambda: attention_ops.flash_attention(q, k, vt, D ** -0.5, None, False, E, 32)}
    graphs = {}
    for name, fn in calls.items():
        assert fn() is not None, name
        graphs[name] = llama_bench.capture(lambda fn=fn: [fn() for _ in range(10)])[0]
    best = {name: [] for name in calls}
    for _ in range(5):
        for name, gr in graphs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            gr.replay()
            e1.record()
            torch.cuda.synchronize()
            best[name].append(e0.elapsed_time(e1) * 100.0)  # ms per 10 calls -> us per call
    return {"n": n, **{name: {"us_min": round(min(v), 2), "spread": round(max(v) / min(v), 3)} for name, v in best.items()}}


@torch.no_grad()
def main(args) -> dict:
    from transformers import DynamicCache
    from torchmx_b200.kv_cache import MXDynamicCache
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    model, cfg, _ = llama_bench.build("8b", args.layers, "float6_e3m2", "float8_e4m3", llm_api=True, mx_attention=True)
    res = {"gpu": smi.splitlines()[0] if smi else "unknown", "model": "8b", "layers": cfg.num_hidden_layers, "weights": "float6_e3m2",
           "activations": "float8_e4m3", "qkvp": "float8_e4m3", "steps_per_run": args.steps, "reps": args.reps,
           "timing": "eager decode steps between CUDA events, caches cropped back to the context before every run; runs alternate bf16 / MX"}
    for B in args.batch:
        for ctx in args.ctx:
            L = ctx + 17
            caches = {"bf16_DynamicCache": DynamicCache(config=cfg), "MXDynamicCache": MXDynamicCache(cfg)}
            for kind, cache in caches.items():
                fill(model, cfg, cache, B, L, kind == "MXDynamicCache", seed=ctx + B)
            entry = {"kv_len": L}
            bytes_ = {kind: llama_bench.kv_cache_bytes(cache) for kind, cache in caches.items()}
            times = decode_time(model, cfg, caches, B, L, args.steps, args.reps)
            for kind in caches:
                entry[kind] = {"ms_per_step": times[kind], "kv_cache_bytes": bytes_[kind]}
            med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
            entry["ms_ratio_median"] = round(med["MXDynamicCache"] / med["bf16_DynamicCache"], 4)
            entry["kv_bytes_ratio"] = round(bytes_["MXDynamicCache"] / bytes_["bf16_DynamicCache"], 4)
            entry["k4b"] = k4b_time(B, L, seed=ctx)
            res[f"b{B}_ctx{ctx}"] = entry
            print(json.dumps({f"b{B}_ctx{ctx}": entry}), flush=True)
            del caches
            torch.cuda.empty_cache()
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--layers", type=int, default=4)
    ap.add_argument("--batch", type=int, nargs="+", default=[1, 8, 32])
    ap.add_argument("--ctx", type=int, nargs="+", default=[1024, 4096, 32768])
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if a.steps > 14:
        ap.error("--steps must stay inside the value block holding ctx + 17 (at most 14), so that the MX cache crops back")
    r = main(a)
    s = json.dumps(r, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
