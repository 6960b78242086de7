"""MX-Llama tokens/s (BASELINE.json configs[3] / [4]): a random-init HF LlamaForCausalLM of the named shape,
`quantize_linear_` (weights fp6_e3m2 / activations fp8_e4m3 by default), prefill of one 2048-token prompt and
decode at batch 32 with a pre-filled static KV cache.  Every linear runs K1 (activation quantize) + K3 (MX GEMM).

Timed with CUDA events; "graph" lines replay a captured CUDA graph of the same forward (no host dispatch in the
number), "eager" lines include the Python dispatch of the reference-style module stack.

    python tools/llama_bench.py --model 8b [--layers N] [--prefill 2048] [--batch 32] [--steps 64]

--llm-api --mx-attention --mx-kv-cache keeps the KV cache as MX codes (torchmx_b200.kv_cache.MXStaticCache) instead of HF's bf16
StaticCache; `kv_cache_bytes` is the resident size of the decode cache either way.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FUSE_NORM = os.environ.get("LB_FUSE_NORM", "0") == "1"

SHAPES = {
    "8b": dict(hidden_size=4096, intermediate_size=14336, num_hidden_layers=32, num_attention_heads=32, num_key_value_heads=8, vocab_size=128256),
    "70b": dict(hidden_size=8192, intermediate_size=28672, num_hidden_layers=80, num_attention_heads=64, num_key_value_heads=8, vocab_size=128256),
    "tiny": dict(hidden_size=512, intermediate_size=1024, num_hidden_layers=2, num_attention_heads=8, num_key_value_heads=2, vocab_size=1024),
}


PACK = False


def build(model_name: str, layers: int | None, wdt: str, adt: str, quantize: bool = True, llm_api: bool = False, mx_attention: bool = False,
          fuse_norm: bool | None = None):
    from transformers import LlamaConfig, LlamaForCausalLM

    import torchmx_b200  # noqa: F401
    from torchmx_b200.config import MXConfig, QLinearConfig
    from torchmx_b200.quant_api import quantize_linear_

    kw = dict(SHAPES[model_name])
    if layers:
        kw["num_hidden_layers"] = layers
    cfg = LlamaConfig(max_position_embeddings=8192, rope_theta=500000.0, **kw)
    cfg._attn_implementation = "sdpa"
    torch.manual_seed(0)
    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.bfloat16)
    try:
        with torch.device("cuda"):
            model = LlamaForCausalLM(cfg).eval()
    finally:
        torch.set_default_dtype(old)
    n_lin = sum(1 for m in model.modules() if type(m) is torch.nn.Linear)
    w_elems = sum(m.weight.numel() for m in model.modules() if type(m) is torch.nn.Linear)
    info = {"linears": n_lin, "weight_elements": w_elems}
    if quantize:
        qc = QLinearConfig(weights_config=MXConfig(wdt, 32), activations_config=MXConfig(adt, 32))
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        if llm_api:  # attention / MLP blocks swapped for their MX versions (projection quantization only), then lm_head
            from torchmx_b200.config import QAttentionConfig
            from torchmx_b200.quant_api import quantize_llm_
            e = MXConfig(adt, 32)  # Q, K, V and the attention probabilities as MX operands too (reference :195-243)
            qa = QAttentionConfig(projection_config=qc, query_config=e, key_config=e, value_config=e, attention_weights_config=e) if mx_attention \
                else QAttentionConfig(projection_config=qc)
            quantize_llm_(model, qa, qc, fuse_rmsnorm=FUSE_NORM if fuse_norm is None else fuse_norm)
        else:
            quantize_linear_(model, qc)
        e1.record()
        torch.cuda.synchronize()
        info["quantize_wall_s"] = time.perf_counter() - t0
        info["quantize_gpu_ms"] = e0.elapsed_time(e1)
        bpe = 2 + (0.5 if wdt == "float4_e2m1" else 1) + 1 / 32
        info["quantize_GBps_gpu"] = w_elems * bpe / (info["quantize_gpu_ms"] * 1e-3) / 1e9
    if quantize and PACK:  # reference storage layout dropped: the dense 4 / 6-bit operand stream is the only copy of each weight
        from torchmx_b200.quant_api import pack_linear_
        info["packed_linears"] = pack_linear_(model)
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    info["resident_after_quantize_GB"] = torch.cuda.memory_allocated() / 1e9
    return model, cfg, info


def time_fn(fn, iters: int, warmup: int = 2) -> float:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def set_len(cache, n: int) -> None:
    """Rewind HF's StaticCache (transformers 5.x keeps the write position as a device tensor per layer)."""
    for layer in cache.layers:
        if getattr(layer, "is_initialized", False):
            layer.cumulative_length.fill_(n)


def kv_cache_bytes(cache) -> int:
    """bytes the cache's layers hold: bf16 keys / values, or MX codes, scales and open value blocks"""
    names = ("k_codes", "k_scales", "vt_codes", "vt_scales", "v_open", "keys", "values")
    return sum(t.numel() * t.element_size() for layer in cache.layers for t in (getattr(layer, n, None) for n in names) if isinstance(t, torch.Tensor))


def capture(fn):
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fn()
    return g, out


@torch.no_grad()
def run(args) -> dict:
    from transformers.cache_utils import StaticCache

    if args.mx_kv_cache:
        if not (args.llm_api and args.mx_attention):
            raise SystemExit("--mx-kv-cache needs --llm-api --mx-attention (the cache holds the MX attention operands)")
        from torchmx_b200.kv_cache import MXStaticCache as StaticCache  # noqa: F811
    model, cfg, info = build(args.model, args.layers, args.wdtype, args.adtype, quantize=not args.no_quant, llm_api=args.llm_api, mx_attention=args.mx_attention,
                             fuse_norm=getattr(args, "fuse_norm", None))
    res = {"api": "none (bf16 HF)" if args.no_quant else (("quantize_llm_ + MX attention" if args.mx_attention else "quantize_llm_") if args.llm_api else "quantize_linear_"),
           "kv_cache": "MXStaticCache" if args.mx_kv_cache else "StaticCache", "model": args.model, "layers": cfg.num_hidden_layers, "weights": args.wdtype, "activations": args.adtype, **info}
    dev = "cuda"

    # ---- prefill: one prompt of `prefill` tokens, fresh static cache each run -------------------------------
    P = args.prefill
    ids = torch.randint(0, cfg.vocab_size, (1, P), device=dev)
    cache = StaticCache(config=cfg, max_cache_len=-(-(P + 8) // 128) * 128 if args.mx_attention else P + 8)  # MX attention contractions need a multiple of 128

    def prefill():
        set_len(cache, 0)  # (also for the MX cache: codes left past the prompt are masked, and crop would synchronise inside a capture)
        return model(input_ids=ids, past_key_values=cache, use_cache=True).logits

    ms = time_fn(prefill, args.prefill_iters)
    res["prefill_eager_ms"] = ms
    res["prefill_eager_tok_s"] = P / ms * 1e3
    if not args.no_graph:
        try:
            g, _ = capture(prefill)
            ms = time_fn(g.replay, args.prefill_iters)
            res["prefill_graph_ms"] = ms
            res["prefill_graph_tok_s"] = P / ms * 1e3
            del g
        except Exception as e:  # noqa: BLE001
            res["prefill_graph_error"] = f"{type(e).__name__}: {str(e)[:300]}"
    del cache
    torch.cuda.empty_cache()

    # ---- decode: batch B, KV cache pre-filled with `ctx` tokens per sequence -----------------------------
    B, ctx, steps = args.batch, args.ctx, args.steps
    cache = StaticCache(config=cfg, max_cache_len=-(-(ctx + steps + 8) // 128) * 128 if args.mx_attention else ctx + steps + 8)
    prompt = torch.randint(0, cfg.vocab_size, (B, ctx), device=dev)
    model(input_ids=prompt, past_key_values=cache, use_cache=True)
    tok = torch.randint(0, cfg.vocab_size, (B, 1), device=dev)

    def decode_step():
        logits = model(input_ids=tok, past_key_values=cache, use_cache=True).logits
        tok.copy_(logits[:, -1].argmax(-1, keepdim=True))
        return logits

    def decode_run(step_fn):
        if args.mx_kv_cache:
            cache.crop(ctx)
        else:
            set_len(cache, ctx)
        for _ in range(steps):
            step_fn()

    ms = time_fn(lambda: decode_run(decode_step), 1, warmup=1) / steps
    res["decode_eager_ms_per_step"] = ms
    res["decode_eager_tok_s"] = B / ms * 1e3
    if not args.no_graph:
        try:
            if args.mx_kv_cache:
                cache.crop(ctx)
            else:
                set_len(cache, ctx)
            g, _ = capture(decode_step)
            ms = time_fn(lambda: decode_run(g.replay), 2, warmup=1) / steps
            res["decode_graph_ms_per_step"] = ms
            res["decode_graph_tok_s"] = B / ms * 1e3
        except Exception as e:  # noqa: BLE001
            res["decode_graph_error"] = f"{type(e).__name__}: {str(e)[:300]}"
    res["kv_cache_bytes"] = kv_cache_bytes(cache)
    codes_bytes = info["weight_elements"] * ((0.5 if args.wdtype == "float4_e2m1" else 1) + 1 / 32)
    res["decode_weight_stream_floor_ms"] = codes_bytes / 6.5e12 * 1e3
    from torchmx_b200 import mx_gemm
    res["gemm_stats"] = dict(mx_gemm.stats)
    from torchmx_b200 import attention_ops
    res["attention_stats"] = dict(attention_ops.stats)
    res["resident_after_run_GB"] = torch.cuda.memory_allocated() / 1e9
    res["max_mem_GB"] = torch.cuda.max_memory_allocated() / 1e9
    return res


def run_cfg(**kw) -> dict:
    """`run` with keyword arguments (bench.py calls this in-process): defaults = the command line's"""
    base = dict(model="8b", layers=None, prefill=2048, prefill_iters=5, batch=32, ctx=128, steps=64, wdtype="float6_e3m2", adtype="float8_e4m3",
                no_graph=False, llm_api=False, mx_attention=False, no_quant=False, fuse_norm=None, mx_kv_cache=False)
    base.update(kw)
    return run(argparse.Namespace(**base))


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="8b", choices=list(SHAPES))
    ap.add_argument("--layers", type=int, default=None)
    ap.add_argument("--prefill", type=int, default=2048)
    ap.add_argument("--prefill-iters", type=int, default=5)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--ctx", type=int, default=128)
    ap.add_argument("--steps", type=int, default=64)
    ap.add_argument("--wdtype", default="float6_e3m2")
    ap.add_argument("--adtype", default="float8_e4m3")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--llm-api", action="store_true", help="quantize_llm_ (MX attention / MLP blocks) instead of quantize_linear_")
    ap.add_argument("--mx-attention", action="store_true", help="with --llm-api: quantize Q, K, V and the attention probabilities (MX bmm + fused softmax)")
    ap.add_argument("--mx-kv-cache", action="store_true", help="with --llm-api --mx-attention: the KV cache held as MX codes (MXStaticCache)")
    ap.add_argument("--no-quant", action="store_true", help="plain bf16 HF model (context line, not the product)")
    ap.add_argument("--pack", action="store_true", help="pack_linear_: weights held only as packed tensor-core operands")
    a = ap.parse_args()
    PACK = a.pack
    print(json.dumps(run(a)), flush=True)
