"""K4b (attention_ops.flash_attention, one kernel) against the chain the MX attention block runs without it (K3 bmm -> K4a -> K3 bmm,
with the key / value codes repeated to the query heads) on long key axes, at Llama-3-8B attention shapes (32 query / 8 key-value
heads, head_dim 128, e4m3 Q / K / V / P):
  * causal prefill (the implied-causal path: no mask tensor) of 4096 .. 32768 tokens, batch 1;
  * one unmasked decode step (sdpa with a DynamicCache drops the mask) at batch 32, 4, 2 and 1 against 2048 / 8192 / 32768 keys;
  * K4b alone where the chain cannot run (K4a takes at most 32768 keys): prefill and decode at 65536 and 131072.

Microseconds per call from CUDA-graph replay (one call per graph for the prefill shapes, 10 for decode), the two sides replayed
alternately, min over 5 rounds; the spread (max / min) is reported beside it.  Every working set here except batch-1 decode at
2048 keys is larger than the 126 MB L2.

    python tools/long_attention_time.py [out.json]
"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torchmx_b200  # noqa: E402,F401
from torchmx_b200 import attention_ops, dtypes  # noqa: E402
from torchmx_b200.layers.mx_llama_attention import _repeat_heads  # noqa: E402
from torchmx_b200.mx_tensor import MXTensor  # noqa: E402

HQ, HK, D = 32, 8, 128
E = dtypes.float8_e4m3
SC = D ** -0.5


def graph_of(fn, n):
    fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n):
            fn()
    return g


def compare(fns, n, rounds=5):
    """{name: (min us per call, max / min)} with the graphs of all sides replayed alternately"""
    graphs = {}
    for name, fn in fns.items():
        try:
            graphs[name] = graph_of(fn, n)
        except torch.OutOfMemoryError:
            graphs[name] = None
            torch.cuda.empty_cache()
    ts = {name: [] for name in fns}
    for _ in range(rounds):
        for name, g in graphs.items():
            if g is None:
                continue
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            ts[name].append(e0.elapsed_time(e1) / n * 1e3)
    del graphs
    torch.cuda.empty_cache()
    return {name: ({"us": round(min(t), 1), "spread": round(max(t) / min(t), 3)} if t else "out of memory") for name, t in ts.items()}


def operands(b, q_len, kv_len):
    q = torch.randn(b, HQ, q_len, D, device="cuda", dtype=torch.bfloat16)
    k = torch.randn(b, HK, kv_len, D, device="cuda", dtype=torch.bfloat16)
    v = torch.randn(b, HK, kv_len, D, device="cuda", dtype=torch.bfloat16)
    return MXTensor.to_mx(q, E, 32), MXTensor.to_mx(k, E, 32), MXTensor.to_mx(v.transpose(2, 3).contiguous(), E, 32)


def case(b, q_len, kv_len, with_chain, n):
    Q, K, VT = operands(b, q_len, kv_len)
    causal = q_len > 1
    fns = {"flash": lambda: attention_ops.flash_attention(Q, K, VT, SC, None, causal, E, 32)}
    if with_chain:
        def chain():  # layers/mx_llama_attention.py `_mx_attend` without K4b
            kk, vv = _repeat_heads(K, HQ // HK), _repeat_heads(VT, HQ // HK).transpose(2, 3)
            s = torch.matmul(Q, kk.transpose(2, 3))
            p = attention_ops.softmax_to_mx(s, SC, None, causal, E, 32)
            return torch.matmul(p, vv).transpose(1, 2).contiguous()
        fns["chain"] = chain
    r = compare(fns, n)
    if with_chain and isinstance(r["chain"], dict):
        r["chain_over_flash"] = round(r["chain"]["us"] / r["flash"]["us"], 2)
    r["score_bytes_of_the_chain"] = b * HQ * q_len * kv_len * 2
    del Q, K, VT
    torch.cuda.empty_cache()
    return r


if __name__ == "__main__":
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out = {"gpu": smi.splitlines()[0] if smi else "unknown", "shape": "Llama-3-8B attention (32 q / 8 kv heads, head_dim 128), e4m3 Q / K / V / P"}
    for S in (4096, 8192, 16384, 32768):
        out[f"prefill_causal_s{S}"] = case(1, S, S, True, 1)
    for b in (32, 4, 2, 1):  # (batch x 8 kv heads = CTAs of a K4b decode step: attention_ops.chain_is_faster)
        for kv in (2048, 8192, 32768):
            out[f"decode_b{b}_kv{kv}"] = case(b, 1, kv, True, 10)
    for S in (65536, 131072):
        out[f"prefill_causal_s{S}"] = case(1, S, S, False, 1)
        for b in (32, 1):
            out[f"decode_b{b}_kv{S}"] = case(b, 1, S, False, 10)
    s = json.dumps(out, indent=1)
    print(s)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(s + "\n")
