"""Fused feed-forward (csrc/ff.cu: GEGLU in the up-projection epilogue, LayerNorm folded into the
down-projection) vs an fp32 torch restatement of x_clip/x_clip.py:180-199 on bf16-rounded operands."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ln(x, g, eps=1e-5):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) * torch.rsqrt(var + eps) * g


@pytest.mark.parametrize("M,d", [(300, 256), (1000, 512), (2 * 98 * 3, 768), (130, 1024), (77, 512),
                                 (148 * 128 * 3 + 40, 512)])   # > 1 tile per CTA pair: the steady-state pipeline
def test_ff_forward_and_w2_gradient(cuda_device, M, d):
    from x_clip_b200 import kernels as K
    dev = cuda_device
    g = torch.Generator().manual_seed(M + d)
    x = torch.randn(M, d, generator=g).to(dev).bfloat16()
    w1 = ((torch.rand(8 * d, d, generator=g) * 2 - 1) / d ** 0.5).to(dev)
    w2 = ((torch.rand(d, 4 * d, generator=g) * 2 - 1) / (4 * d) ** 0.5).to(dev)
    g4 = (1 + 0.1 * torch.randn(4 * d, generator=g)).to(dev)
    res = torch.randn(M, d, generator=g).to(dev).bfloat16()

    w1p, w2g, colvec = K.ff_weights(w1, w2, g4)
    u, hp, rowsum = K.ff_up(x, w1p)
    x2, acc, stats = K.ff_down(hp, w2g, colvec, rowsum, res, 1e-5)
    torch.cuda.synchronize()

    u_ref = x.float() @ w1.bfloat16().float().t()
    val, gate = u_ref[:, :4 * d], u_ref[:, 4 * d:]
    hp_ref = val * torch.nn.functional.gelu(gate)
    assert (u.float() - u_ref).abs().max().item() <= 2e-2 * u_ref.abs().max().item()
    assert (hp.float() - hp_ref).abs().max().item() <= 2e-2 * hp_ref.abs().max().item() + 1e-3
    mu = hp.float().mean(-1)
    rstd = torch.rsqrt(hp.float().var(-1, unbiased=False) + 1e-5)
    assert torch.allclose(stats[:, 0], mu, atol=1e-4, rtol=1e-3)
    assert torch.allclose(stats[:, 1], rstd, rtol=2e-3)
    x2_ref = _ln(hp_ref, g4) @ w2.t() + res.float()
    err = (x2.float() - x2_ref).abs().max().item()
    assert err <= 2e-2 * x2_ref.abs().max().item(), err
    rel = (x2.float() - x2_ref).norm().item() / x2_ref.norm().item()
    assert rel <= 5e-3, rel

    # backward: autograd over the fp32 restatement, on the bf16 activations the kernels saved
    dx = torch.randn(M, d, generator=g).to(dev).bfloat16()
    u_leaf = u.float().requires_grad_(True)
    w2_leaf = w2.clone().requires_grad_(True)
    g4_leaf = g4.clone().requires_grad_(True)
    hp_a = u_leaf[:, :4 * d] * torch.nn.functional.gelu(u_leaf[:, 4 * d:])
    (_ln(hp_a, g4_leaf) @ w2_leaf.t()).backward(dx.float())

    dxs, vsum, ab = K.ff_bwd_prep(dx, stats, acc, colvec)
    du = K.ff_bwd(dx, w2g, u, stats, ab)
    raw = torch.zeros(d, 4 * d, device=dev)
    K.gemm(dxs, hp, a_major=1, b_major=1, out=raw, accumulate=True)
    dg4 = torch.zeros(4 * d, device=dev)
    dw2 = K.ff_w2_grad_post_(raw, vsum, g4, w2, dg4)
    torch.cuda.synchronize()
    for name, got, ref in (("du", du.float(), u_leaf.grad), ("dW2", dw2, w2_leaf.grad), ("dg4", dg4, g4_leaf.grad)):
        rel = (got - ref).norm().item() / ref.norm().item()
        assert rel <= 1.5e-2, (name, rel)
