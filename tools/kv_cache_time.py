"""K5e (glue_ops.rope_quantize_kv: rope + MX KV-cache append + Q quantization, one launch) against the chain it replaces in the MX
attention block with a bf16 StaticCache -- K5b rope, StaticLayer.update (arange + two index_copy_), to_mx(Q), to_mx(whole K cache),
K5d over the whole V cache -- at Llama-3-8B shapes (32 query / 8 key-value heads, head_dim 128, e4m3 Q / K / V):
prefill of 2048 tokens into an empty cache, and decode at batch 32 with C = 256 / 1024 / 4096 (write position C / 2 + 5).

us per step from a CUDA-graph replay of 20 steps (min of 5 replays), and GB/s of the algorithmic bytes of each side (every operand
read once, every result written once).  The decode working sets at C <= 1024 fit the 126 MB L2 between replays; C = 4096 does not.

    python tools/kv_cache_time.py [out.json]
"""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torchmx_b200  # noqa: E402,F401
from torchmx_b200 import dtypes, glue_ops  # noqa: E402
from torchmx_b200.kv_cache import MXStaticLayer  # noqa: E402
from torchmx_b200.mx_tensor import MXTensor  # noqa: E402

HQ, HK, D = 32, 8, 128
E8 = dtypes.float8_e4m3


def timed(f, n=20):
    for _ in range(3):
        f()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(n):
            f()
    ts = []
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1) / n * 1e3)
    return min(ts)


def case(b, t, C, L):
    from transformers.cache_utils import StaticLayer
    qkv = torch.randn(b, t, (HQ + 2 * HK) * D, device="cuda", dtype=torch.bfloat16)
    q, k, v = (z.view(b, t, -1, D).transpose(1, 2) for z in qkv.split([HQ * D, HK * D, HK * D], -1))
    cs = torch.randn(1, t, D, device="cuda", dtype=torch.bfloat16)
    qc = type("Q", (), {})()
    qc.query_config = qc.key_config = qc.value_config = type("C", (), {"elem_dtype": E8, "block_size": 32})()
    mx = MXStaticLayer(C)
    mx._mx_initialize(k, qc)
    mx.cumulative_length.fill_(L)
    args = (mx.cumulative_length, mx.k_codes, mx.k_scales, mx.vt_codes, mx.vt_scales, mx.v_open, (E8, E8, E8))
    us_k5e = timed(lambda: glue_ops.rope_quantize_kv(q, k, v, cs, cs, *args))  # (the position is not advanced: every step writes at L)
    bf = StaticLayer(C)
    bf.update(torch.zeros(b, HK, 1, D, device="cuda", dtype=torch.bfloat16), torch.zeros(b, HK, 1, D, device="cuda", dtype=torch.bfloat16))

    def chain():
        bf.cumulative_length.fill_(L)
        qr, kr = glue_ops.rope(q, k, cs, cs)
        keys, values = bf.update(kr, v)
        MXTensor.to_mx(qr, E8, 32), MXTensor.to_mx(keys, E8, 32), glue_ops.quantize_transposed(values, E8)

    us_chain = timed(chain)
    code = 1 + 1 / 32
    new_in = b * t * (HQ + 2 * HK) * D * 2 + 2 * t * D * 2
    v_blocks = (L + t - 1) // 32 - L // 32 + 1
    by_k5e = new_in + b * HQ * t * D * code + b * HK * t * D * code + b * HK * D * 32 * v_blocks * code + 2 * b * HK * 32 * D * 2
    by_chain = (b * t * (HQ + HK) * D * 2 * 2                   # rope: q, k in, rotated out
                + 2 * b * t * HK * D * 2 * 2                    # cache write: rotated k, v in, cache rows out
                + b * HQ * t * D * (2 + code)                   # to_mx(Q)
                + 2 * b * HK * C * D * (2 + code))              # to_mx(K cache), K5d(V cache)
    return {"K5e_us": round(us_k5e, 2), "K5e_GBps": round(by_k5e / us_k5e / 1e3), "K5e_bytes": int(by_k5e),
            "chain_us": round(us_chain, 2), "chain_GBps": round(by_chain / us_chain / 1e3), "chain_bytes": int(by_chain),
            "speedup": round(us_chain / us_k5e, 2)}


if __name__ == "__main__":
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    out = {"gpu": smi.splitlines()[0] if smi else "unknown", "shape": "Llama-3-8B attention (32 q / 8 kv heads, head_dim 128), e4m3 Q / K / V"}
    out["prefill_2048"] = case(1, 2048, 2048, 0)
    for C in (256, 1024, 4096):
        out[f"decode_b32_C{C}"] = case(32, 1, C, C // 2 + 5)
    s = json.dumps(out, indent=1)
    print(s)
    if len(sys.argv) > 1:
        with open(sys.argv[1], "w") as f:
            f.write(s + "\n")
