"""tcgen05 attention kernels: S = 128 single-tile kernels, the tiled kernels at other lengths and
head sizes, and the eager PyTorch attention they replace (bf16, same tokens), per forward /
backward call; every row carries the card's name and power limit.
CUDA-graph replays; one JSON line per configuration -> gpurun_out/bench_attention.json."""
import json
import math
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from skycomputing_b200.ops import native as nat  # noqa: E402
from tools.triage_gemm import timeit  # noqa: E402


def eager(qkv, B, S, heads):
    H = qkv.shape[1] // 3
    d = H // heads
    q, k, v = qkv.view(B, S, 3, heads, d).permute(2, 0, 3, 1, 4)
    p = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(d), -1)
    return (p @ v).permute(0, 2, 1, 3).reshape(B * S, H)


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader",
                          "-i", str(torch.cuda.current_device())], capture_output=True, text=True)
    name, power = (out.stdout.strip().split(", ") + ["?", "?"])[:2]
    return dict(gpu=name, power_limit=power)


def main():
    rows = []
    heads = 16
    gpu = card()
    # head size 64 at five lengths; the other head sizes at 4096 tokens, S = 128 and 512
    shapes = [(64, S, B) for S, B in ((128, 32), (64, 64), (256, 16), (384, 8), (512, 8))]
    shapes += [(d, S, 4096 // S) for d in (32, 96, 128) for S in (128, 512)]
    for d, S, B in shapes:
        H = heads * d
        torch.manual_seed(0)
        qkv = torch.randn(B * S, 3 * H, device="cuda").bfloat16()
        dctx = torch.randn(B * S, H, device="cuda").bfloat16()
        ctx, lse = nat.attention_fwd(qkv, None, B, S, heads)
        tf = timeit(lambda: nat.attention_fwd(qkv, None, B, S, heads)) * 1e3
        tb = timeit(lambda: nat.attention_bwd(qkv, None, ctx, lse, dctx, B, S, heads)) * 1e3
        te = timeit(lambda: eager(qkv, B, S, heads)) * 1e3
        qg = qkv.clone().requires_grad_(True)

        def eager_fb():
            o = eager(qg, B, S, heads)
            o.backward(dctx)
            qg.grad = None

        teb = timeit(eager_fb, iters=5) * 1e3 - te
        flops_f = 4.0 * B * heads * S * S * d
        row = dict(D=d, S=S, B=B, heads=heads, tokens=B * S,
                   kernels="single-tile" if S == 128 and d == 64 else "tiled",
                   fwd_us=round(tf, 1), bwd_us=round(tb, 1), fwd_tflops=round(flops_f / tf / 1e6, 1),
                   bwd_tflops=round(2.5 * flops_f / tb / 1e6, 1), eager_fwd_us=round(te, 1),
                   eager_bwd_us=round(teb, 1), **gpu)
        rows.append(row)
        print(json.dumps(row), flush=True)
    os.makedirs("gpurun_out", exist_ok=True)
    json.dump(rows, open("gpurun_out/bench_attention.json", "w"), indent=1)


if __name__ == "__main__":
    main()
