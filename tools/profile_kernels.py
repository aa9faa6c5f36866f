"""Stand-alone launches of the hot kernels at benchmark shapes, for `ncu --set full`.

    python tools/profile_kernels.py gemm|attn|nce|rowwise [reps]

gemm : the four GEMM shapes of one text layer at cfg2 (M = 1024*257 tokens, d = 512):
       fwd qkv, fwd ff-up, dgrad ff-up, wgrad ff-up
attn : attention fwd + bwd at B=1024, n=257, h=8 (cfg2 text) and n=33 (cfg2 image)
nce  : logits+InfoNCE fwd/bwd row block at cfg3 per-rank size (4096 x 32768, D = 3*512)
"""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from x_clip_b200 import kernels as K  # noqa: E402


def main():
    what = sys.argv[1]
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    if what == "gemm":
        M, d = 1024 * 257, 512
        x = torch.randn(M, d, device=dev).bfloat16()
        wqkv = torch.randn(3 * d, d, device=dev).bfloat16()
        w1 = torch.randn(8 * d, d, device=dev).bfloat16()
        du = torch.randn(M, 8 * d, device=dev).bfloat16()
        for _ in range(reps):
            K.gemm(x, wqkv)                                   # fwd  [M,512]x[1536,512]
            K.gemm(x, w1)                                     # fwd  [M,512]x[4096,512]
            K.gemm(du, w1, b_major=1)                         # dgrad [M,4096]x[4096,512]
            K.gemm(du, x, a_major=1, b_major=1, accumulate=True)   # wgrad
    elif what == "attn":
        for n in (257, 33):
            B, H = 1024, 8
            qkv = torch.randn(B * n, 3 * H * 64, device=dev).bfloat16()
            mask = torch.rand(B, n, device=dev) > 1e-4
            for _ in range(reps):
                o, lse = K.attn_fwd(qkv, mask, B, n, H, 0.125)
                K.attn_bwd(qkv, mask, o, torch.randn_like(o), lse, B, n, H, 0.125)
    elif what == "nce":
        R, C, D = 4096, 32768, 1536
        a = torch.nn.functional.normalize(torch.randn(R, D, device=dev), dim=-1).bfloat16()
        b = torch.nn.functional.normalize(torch.randn(C, D, device=dev), dim=-1).bfloat16()
        temp = torch.tensor([2.718], device=dev)
        gs = torch.tensor([1.0 / (2 * C)], device=dev)
        for _ in range(reps):
            lse, pos = K.nce_fwd(a, b, temp, 0, False)
            K.nce_bwd(a, b, temp, 0, False, lse, torch.full((C,), lse.mean().item(), device=dev),
                      1.0, 1.0, 2.0, gs)
    elif what == "rowwise":
        M, d = 1024 * 257, 512
        x = torch.randn(M, d, device=dev).bfloat16()
        g = torch.ones(d, device=dev)
        for _ in range(reps):
            out, st, out2, st2 = K.layernorm_fwd(x, g, res=x, g2=g)
            K.layernorm_bwd(x, x, st, g, add=x, dg=torch.zeros(d, device=dev))
    torch.cuda.synchronize()
    print("done", what)


if __name__ == "__main__":
    main()
