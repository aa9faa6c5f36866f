"""Time the pieces of the fused feed-forward block (csrc/ff.cu) and the GEMMs of its backward.

    python tools/ff_bench.py [M,d ...]     (default: cfg3 ViT micro-batch 512, cfg3 text, cfg2 text)"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from x_clip_b200 import kernels as K  # noqa: E402

dev = torch.device("cuda:0")
shapes = [(512 * 98, 768), (512 * 78, 512), (263168, 512)]
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


for (M, d) in shapes:
    g = torch.Generator().manual_seed(0)
    x = torch.randn(M, d, generator=g).to(dev).bfloat16()
    w1 = ((torch.rand(8 * d, d, generator=g) * 2 - 1) / d ** 0.5).to(dev)
    w2 = ((torch.rand(d, 4 * d, generator=g) * 2 - 1) / (4 * d) ** 0.5).to(dev)
    g4 = torch.ones(4 * d, device=dev)
    res = torch.randn(M, d, generator=g).to(dev).bfloat16()
    dx = torch.randn(M, d, generator=g).to(dev).bfloat16()
    w1b = w1.bfloat16()
    w1p, w2g, colvec = K.ff_weights(w1, w2, g4)
    u, hp, rowsum = K.ff_up(x, w1p)
    x2, acc, stats = K.ff_down(hp, w2g, colvec, rowsum, res, 1e-5)
    t = {}
    t["ff_up (fused GEGLU)"] = timeit(lambda: K.ff_up(x, w1p))
    t["ff_down (fused LN)"] = timeit(lambda: K.ff_down(hp, w2g, colvec, rowsum, res, 1e-5))
    t["ff_bwd_prep"] = timeit(lambda: K.ff_bwd_prep(dx, stats))
    t["gemm wgrad up (plain, split-K fp32)"] = timeit(lambda: K.gemm(u, x, a_major=1, b_major=1, accumulate=True))
    t["gemm dgrad up (plain)"] = timeit(lambda: K.gemm(u, w1b, b_major=1))
    dxs, vsum, ab = K.ff_bwd_prep(dx, stats, acc, colvec)
    t["ff_bwd (fused dgrad + LN/GEGLU bwd)"] = timeit(lambda: K.ff_bwd(dx, w2g, u, stats, ab))
    print(f"M={M} d={d}: " + " | ".join(f"{k} {v:.3f} ms" for k, v in t.items()), flush=True)
