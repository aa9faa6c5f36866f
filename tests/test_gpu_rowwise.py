"""Row-wise kernels vs fp32 torch autograd of the same (bf16-rounded) inputs."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ln(x, g, eps=1e-5):
    mu = x.mean(-1, keepdim=True)
    var = ((x - mu) ** 2).mean(-1, keepdim=True)
    return (x - mu) * torch.rsqrt(var + eps) * g


def _close(a, b, tol, what=""):
    err = (a.float() - b.float()).abs().max().item()
    ref = b.float().abs().max().item()
    assert err <= tol * max(ref, 1e-3), f"{what}: err {err} vs scale {ref}"


@pytest.mark.parametrize("rows,d", [(1, 256), (77, 512), (1000, 768), (4099, 1024)])
def test_layernorm_fwd_bwd(cuda_device, rows, d):
    from x_clip_b200 import kernels as K
    torch.manual_seed(0)
    x = (torch.randn(rows, d, device=cuda_device) * 2 + 0.5).bfloat16()
    g = 1 + 0.1 * torch.randn(d, device=cuda_device)
    res = torch.randn(rows, d, device=cuda_device).bfloat16()
    out, stats, _, _ = K.layernorm_fwd(x, g, res=res)
    xf = x.float().requires_grad_(True)
    gf = g.clone().requires_grad_(True)
    ref = _ln(xf, gf) + res.float()
    _close(out, ref, 1e-2, "ln fwd")
    assert torch.allclose(stats[:, 0], x.float().mean(-1), atol=1e-4)

    dy = torch.randn(rows, d, device=cuda_device).bfloat16()
    add = torch.randn(rows, d, device=cuda_device).bfloat16()
    dg = torch.zeros(d, device=cuda_device)
    dx = K.layernorm_bwd(dy, x, stats, g, add=add, dg=dg)
    ref.backward(dy.float())
    _close(dx, xf.grad + add.float(), 1.5e-2, "ln dx")
    _close(dg, gf.grad, 5e-3, "ln dg")


def test_layernorm_chain(cuda_device):
    """out = LN(y)*g + x ; out2 = LN(out)*g2 in one pass (attention tail + next pre-norm)."""
    from x_clip_b200 import kernels as K
    torch.manual_seed(1)
    rows, d = 515, 512
    y = torch.randn(rows, d, device=cuda_device).bfloat16()
    x = torch.randn(rows, d, device=cuda_device).bfloat16()
    g = 1 + 0.1 * torch.randn(d, device=cuda_device)
    g2 = 1 + 0.1 * torch.randn(d, device=cuda_device)
    out, stats, out2, stats2 = K.layernorm_fwd(y, g, res=x, g2=g2)
    ref1 = (_ln(y.float(), g) + x.float())
    _close(out, ref1, 1e-2, "chain out")
    ref2 = _ln(out.float(), g2)          # second norm sees the bf16-rounded first output
    _close(out2, ref2, 1e-2, "chain out2")
    assert torch.allclose(stats2[:, 0], out.float().mean(-1), atol=1e-4)


@pytest.mark.parametrize("rows,d", [(4, 256), (1024, 512)])
def test_l2norm(cuda_device, rows, d):
    from x_clip_b200 import kernels as K
    torch.manual_seed(3)
    p = torch.randn(rows, d, device=cuda_device)
    z, zrow, zcol, inv = K.l2norm_fwd(p)
    pf = p.clone().requires_grad_(True)
    ref = torch.nn.functional.normalize(pf, dim=-1)
    assert torch.allclose(z, ref, atol=1e-6)
    hi, lo = zrow[:, :d].float(), zrow[:, d:2 * d].float()
    assert torch.equal(zrow[:, 2 * d:], zrow[:, :d]) and torch.equal(zcol[:, :2 * d], zrow[:, :d].repeat(1, 2))
    assert torch.equal(zcol[:, 2 * d:], zrow[:, d:2 * d])
    assert (hi + lo - ref.detach()).abs().max().item() < 2e-5          # split-bf16 carries ~16 bits
    gram = zrow.float() @ zcol.float().t()
    assert (gram - ref.detach() @ ref.detach().t()).abs().max().item() < 1e-4
    dz = torch.randn(rows, d, device=cuda_device)
    dp = K.l2norm_bwd(dz, z, inv)
    ref.backward(dz)
    _close(dp, pf.grad, 1e-2, "l2norm dp")


def test_cast(cuda_device):
    from x_clip_b200 import kernels as K
    for n in (1, 7, 8, 1000003):
        src = torch.randn(n, device=cuda_device)
        assert torch.equal(K.cast_bf16(src), src.bfloat16())


def test_text_embed_fwd_bwd(cuda_device):
    """[cls | tok[ids] + pos] and its backward (x_clip/x_clip.py:320-332) vs torch autograd."""
    from x_clip_b200 import engine as E
    torch.manual_seed(4)
    B, n, d, vocab = 37, 16, 512, 100
    ids = torch.randint(0, vocab, (B, n), device=cuda_device)
    tok = torch.randn(vocab, d, device=cuda_device, requires_grad=True)
    pos = torch.randn(n + 4, d, device=cuda_device, requires_grad=True)
    cls = torch.randn(d, device=cuda_device, requires_grad=True)
    out = E.TextEmbedFn.apply(ids, tok, pos, cls)
    ref = torch.cat((cls.expand(B, 1, d), tok[ids] + pos[:n]), dim=1)
    assert out.shape == (B, n + 1, d)
    _close(out, ref, 1e-2, "embed fwd")
    dx = torch.randn(B, n + 1, d, device=cuda_device).bfloat16()
    out.backward(dx)
    g = (tok.grad.clone(), pos.grad.clone(), cls.grad.clone())
    tok.grad = pos.grad = cls.grad = None
    ref.backward(dx.float())
    _close(g[0], tok.grad, 1e-5, "dtok")
    _close(g[1], pos.grad, 1e-5, "dpos")
    _close(g[2], cls.grad, 1e-5, "dcls")
