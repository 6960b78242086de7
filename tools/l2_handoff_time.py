"""How much of K2's code read K1 hands over through L2, measured as time (ncu, which flushes caches per kernel, cannot show it).

    python tools/l2_handoff_time.py [--parent DIR] [--iters N] [--out profiles/r7_l2_handoff.json]

For each element type on bench.py's 16384 x 16384 bf16 tensor, mean microseconds (CUDA events) of
  (a) K2 right after the K1 that produced its codes, as bench.py runs them;
  (b) K2 after K1 and an unrelated 512 MiB write, so the codes are no longer in L2;
  (c) K1 alone, back to back (the mean over one event pair around `iters` launches).
(b) - (a) is the handoff.  Each tree is measured in a process of its own (the library is loaded once per process): this tree,
and with --parent a checkout of the commit before the L2 hints -- its K1 is the same kernel without hints, its K2 walks forward
without hints, so its (b) - (a) is the no-handoff control.  The two are measured alternately, twice each.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ELEMS = ["float8_e4m3", "float6_e3m2", "float6_e2m3", "float4_e2m1", "int8"]
N = 16384


def measure(root: str, iters: int) -> dict:
    sys.path.insert(0, root)
    import torch
    import torchmx_b200  # noqa: F401
    from torchmx_b200 import _C, dtypes
    from torchmx_b200.mx_tensor import MXTensor
    _C.lib()
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(1234)
    x = torch.randn(N, N, dtype=torch.bfloat16, device=dev, generator=g)
    x *= torch.exp2(torch.randint(-20, 20, (N, 1), device=dev, generator=g).float()).to(torch.bfloat16)
    scrub = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

    def ev():
        return torch.cuda.Event(enable_timing=True)

    out = {}
    for name in ELEMS:
        et = dtypes.STR_TO_SUPPORTED_ELEM_DTYPE[name]
        res = {}
        for case in ("a_after_k1", "b_cold_codes"):
            ts = []
            for i in range(iters + 2):
                m = MXTensor.to_mx(x, et, 32)
                if case == "b_cold_codes":
                    scrub.fill_(i & 0xFF)
                e0, e1 = ev(), ev()
                e0.record()
                y = m.to_dtype(torch.bfloat16)
                e1.record()
                torch.cuda.synchronize()
                if i >= 2:
                    ts.append(e0.elapsed_time(e1) * 1e3)
                del m, y
            res[case + "_k2_us"] = round(statistics.mean(ts), 2)
        # K1 back to back, behind a device-side wait so that host dispatch runs ahead and is not in the number
        ms = [MXTensor.to_mx(x, et, 32) for _ in range(2)]
        torch.cuda._sleep(20_000_000)
        e0, e1 = ev(), ev()
        e0.record()
        for _ in range(iters):
            ms.append(MXTensor.to_mx(x, et, 32))
        e1.record()
        torch.cuda.synchronize()
        res["c_k1_alone_us"] = round(e0.elapsed_time(e1) * 1e3 / iters, 2)
        del ms
        res["handoff_b_minus_a_us"] = round(res["b_cold_codes_k2_us"] - res["a_after_k1_k2_us"], 2)
        out[name] = res
    return out


def card() -> dict:
    import torch
    p = torch.cuda.get_device_properties(0)
    info = {"name": p.name, "l2_cache_bytes": p.L2_cache_size, "sms": p.multi_processor_count}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        info["nvidia_smi_name_power_limit_max_sm_clock"] = q
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi_error"] = str(e)
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent", help="a built checkout of the parent commit to measure beside this tree")
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_l2_handoff.json"))
    ap.add_argument("--measure", metavar="ROOT", help=argparse.SUPPRESS)  # child process: measure the tree at ROOT, print JSON
    args = ap.parse_args()
    if args.measure:
        print(json.dumps(measure(args.measure, args.iters)))
        return
    trees = [("this", ROOT)] + ([("parent", os.path.abspath(args.parent))] if args.parent else [])
    runs = {label: [] for label, _ in trees}
    for _ in range(2):
        for label, root in trees:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--measure", root, "--iters", str(args.iters)],
                               capture_output=True, text=True, check=True)
            runs[label].append(json.loads(r.stdout.strip().splitlines()[-1]))
    result = {"card": card(), "shape": [N, N], "iters_per_case": args.iters, "runs": runs,
              "note": "K2 = dequantize_b32_kernel -> bf16, K1 = quantize_b32_bf16_kernel; (b) writes 512 MiB (torch fill_) between K1 and K2"}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps(result))


if __name__ == "__main__":
    main()
