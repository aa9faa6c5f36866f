"""Time the fused attention forward / backward at the shapes of the bench workloads.

    python tools/attn_bench.py [B,n,H ...]      (default: cfg3 image/text towers, cfg2 towers)

Prints algorithmic TFLOP/s (4 n^2 64 per (b,h) forward, 10 n^2 64 backward, FA convention)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from x_clip_b200 import kernels as K  # noqa: E402

dev = torch.device("cuda:0")
shapes = [(512, 98, 12), (512, 78, 8), (1024, 32, 8), (1024, 257, 8), (512, 196, 12)]
if len(sys.argv) > 1:
    shapes = [tuple(int(x) for x in a.split(",")) for a in sys.argv[1:]]


def timeit(fn, reps=10):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


for (B, n, H) in shapes:
    g = torch.Generator().manual_seed(0)
    qkv = torch.randn(B * n, 3 * H * 64, generator=g).to(dev).bfloat16()
    d_o = torch.randn(B * n, H * 64, generator=g).to(dev).bfloat16()
    o, lse = K.attn_fwd(qkv, None, B, n, H, 0.125)
    ms_f = timeit(lambda: K.attn_fwd(qkv, None, B, n, H, 0.125))
    ms_b = timeit(lambda: K.attn_bwd(qkv, None, o, d_o, lse, B, n, H, 0.125))
    fl = B * H * n * n * 64.0
    print(f"attn B={B} n={n} H={H}: fwd {ms_f:.3f} ms {4 * fl / ms_f / 1e9:.1f} TFLOP/s | "
          f"bwd {ms_b:.3f} ms {10 * fl / ms_b / 1e9:.1f} TFLOP/s", flush=True)
