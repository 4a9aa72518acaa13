"""Times the long-sequence bf16 attention forward (HW > 256 patch tokens: vtp_b200/csrc/attention_long.cu) with CUDA
events, and F.scaled_dot_product_attention on the same bf16 tensors as context.  GPU only.
  python tools/attn_long_bench.py [--reps 20] [--json out.json]
Every input is larger than the B200's 126 MB L2, so the timings include streaming qkv from HBM."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

from vtp_b200 import lib

SHAPES = [  # (B, T, H, prefix)
    (64, 1025, 6, 1),   # VTP-Small trunk at 512x512
    (32, 1025, 16, 1),  # VTP-Large trunk at 512x512
    (128, 577, 6, 1),   # VTP-Small trunk at 384x384
    (8, 4097, 16, 1),   # VTP-Large trunk at 1024x1024
]


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3  # us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    rows = []
    for B, T, H, prefix in SHAPES:
        g = torch.Generator(device="cuda").manual_seed(0)
        qkv = (torch.randn(B * T, 3 * H * 64, device="cuda", generator=g) * 1.5).to(torch.bfloat16)
        out = torch.empty(B * T, H * 64, device="cuda", dtype=torch.bfloat16)
        us = timed(lambda: lib.attention_fwd(qkv, out, B, T, H, prefix=prefix), a.warmup, a.reps)
        q, k, v = [t.transpose(1, 2) for t in qkv.view(B, T, 3, H, 64).unbind(2)]
        us_sdpa = timed(lambda: F.scaled_dot_product_attention(q, k, v), a.warmup, a.reps)
        flop = 4.0 * T * T * 64 * B * H
        row = {"B": B, "T": T, "H": H, "prefix": prefix, "qkv_MB": qkv.numel() * 2 / 2**20, "us": us,
               "tflops": flop / us / 1e6, "sdpa_us": us_sdpa, "sdpa_tflops": flop / us_sdpa / 1e6}
        rows.append(row)
        print(f"B={B:4d} T={T:5d} H={H:2d}: {us:9.1f} us {row['tflops']:6.1f} TFLOP/s   "
              f"(SDPA {us_sdpa:9.1f} us {row['sdpa_tflops']:6.1f} TFLOP/s)", flush=True)
    res = {"device": torch.cuda.get_device_name(), "reps": a.reps, "rows": rows}
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
