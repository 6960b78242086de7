"""MX-attention decode of a Llama-3-8B-shaped model (random init; weights fp6_e3m2 / activations fp8_e4m3, e4m3 Q / K / V / P) at
batch 32 with HF's bf16 StaticCache against MXStaticCache, at context 128, 1024 and 4096: ms per decode step from CUDA-graph
replay and the resident bytes of each cache.  Both caches live in the same process and are prefilled with the same prompt; the
timed runs alternate between them, `--reps` times, so the spread of each is visible beside the difference.  The first replayed step
of the two caches is also compared bit for bit.

    python tools/kv_cache_bench.py [--layers N] [--steps 32] [--reps 3] [--out r3.json]
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


@torch.no_grad()
def main(args) -> dict:
    from transformers.cache_utils import StaticCache
    from torchmx_b200.kv_cache import MXStaticCache
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    model, cfg, info = llama_bench.build("8b", args.layers, "float6_e3m2", "float8_e4m3", llm_api=True, mx_attention=True)
    res = {"gpu": smi.splitlines()[0] if smi else "unknown", "model": "8b", "layers": cfg.num_hidden_layers, "batch": args.batch,
           "weights": "float6_e3m2", "activations": "float8_e4m3", "qkvp": "float8_e4m3", "steps_per_run": args.steps, "reps": args.reps,
           "timing": "CUDA-graph replay of one decode step, `steps` replays per run between CUDA events; runs alternate bf16 / MX"}
    B = args.batch
    for ctx in args.ctx:
        cap = -(-(ctx + args.steps + 8) // 128) * 128
        g0 = torch.Generator(device="cuda").manual_seed(ctx)
        prompt = torch.randint(0, cfg.vocab_size, (B, ctx), device="cuda", generator=g0)
        first = torch.randint(0, cfg.vocab_size, (B, 1), device="cuda", generator=g0)
        runs = {}
        for kind, cls in (("bf16_StaticCache", StaticCache), ("MXStaticCache", MXStaticCache)):
            cache = cls(config=cfg, max_cache_len=cap)
            model(input_ids=prompt, past_key_values=cache, use_cache=True, logits_to_keep=1)
            tok = first.clone()

            def step(cache=cache, tok=tok):
                logits = model(input_ids=tok, past_key_values=cache, use_cache=True).logits
                tok.copy_(logits[:, -1].argmax(-1, keepdim=True))
                return logits

            def rewind(cache=cache, tok=tok, kind=kind):
                if kind == "MXStaticCache":
                    cache.crop(ctx)
                else:  # (positions past ctx cleared as well: the V block holding ctx is quantized whole, stale values included)
                    llama_bench.set_len(cache, ctx)
                    for layer in cache.layers:
                        layer.keys[:, :, ctx:].zero_()
                        layer.values[:, :, ctx:].zero_()
                tok.copy_(first)

            rewind()
            g, out = llama_bench.capture(step)
            runs[kind] = (cache, g, out, rewind)
        outs = []
        for kind, (cache, g, out, rewind) in runs.items():
            rewind()
            g.replay()
            outs.append(out.clone())
        entry = {"capacity": cap, "first_step_logits_equal": bool(torch.equal(outs[0], outs[1]))}
        times = {k: [] for k in runs}
        for _ in range(args.reps):
            for kind, (cache, g, out, rewind) in runs.items():
                rewind()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.steps):
                    g.replay()
                e1.record()
                torch.cuda.synchronize()
                times[kind].append(round(e0.elapsed_time(e1) / args.steps, 4))
        for kind, (cache, g, out, rewind) in runs.items():
            entry[kind] = {"ms_per_step": times[kind], "kv_cache_bytes": llama_bench.kv_cache_bytes(cache)}
        entry["kv_bytes_ratio"] = round(entry["MXStaticCache"]["kv_cache_bytes"] / entry["bf16_StaticCache"]["kv_cache_bytes"], 4)
        entry["ms_ratio_median"] = round(sorted(times["MXStaticCache"])[len(times["MXStaticCache"]) // 2]
                                         / sorted(times["bf16_StaticCache"])[len(times["bf16_StaticCache"]) // 2], 4)
        res[f"ctx_{ctx}"] = entry
        print(json.dumps({f"ctx_{ctx}": entry}), flush=True)
        del runs, outs
        torch.cuda.empty_cache()
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--layers", type=int, default=None)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--ctx", type=int, nargs="+", default=[128, 1024, 4096])
    ap.add_argument("--steps", type=int, default=32)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    r = main(a)
    s = json.dumps(r, indent=1)
    print(s)
    if a.out:
        with open(a.out, "w") as f:
            f.write(s + "\n")
