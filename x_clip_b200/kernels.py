"""Tensor-level wrappers over the C-ABI (raw pointers + shapes from torch tensors).

No arithmetic happens here - each function validates devices/dtypes/strides,
allocates outputs through torch's caching allocator and forwards to one
`xclip_*` entry point on torch's current CUDA stream.
"""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib

BF16 = torch.bfloat16
F32 = torch.float32


def _stream(t: torch.Tensor) -> int:
    """Current torch stream of the device the operands live on."""
    return torch.cuda.current_stream(t.device).cuda_stream


class Profiler:
    """Optional per-launch timing (CUDA events on the launching stream) with the ALGORITHMIC
    flops / bytes of each call, used by bench.py for the roofline line.  Off by default."""

    def __init__(self):
        self.enabled = False
        self.records = []          # (family, flops, bytes, start_event, end_event)

    def start(self):
        self.records = []
        self.enabled = True

    def stop(self):
        """-> {family: dict(calls, ms, flops, bytes)}"""
        self.enabled = False
        torch.cuda.synchronize()
        out = {}
        for fam, fl, by, e0, e1 in self.records:
            d = out.setdefault(fam, dict(calls=0, ms=0.0, flops=0.0, bytes=0.0))
            d["calls"] += 1
            d["ms"] += e0.elapsed_time(e1)
            d["flops"] += fl
            d["bytes"] += by
        self.records = []
        return out


PROF = Profiler()


def _call(dev_of: torch.Tensor, family: str, flops: float, nbytes: float, name: str, *args) -> None:
    """Launch on the device of `dev_of` (made current for the call: the library launches on
    cudaGetDevice() and keeps per-device kernel attributes) and on its current torch stream."""
    if dev_of.device.index != torch.cuda.current_device():
        with torch.cuda.device(dev_of.device):
            _call_on_current(family, flops, nbytes, name, *args, _stream(dev_of))
        return
    _call_on_current(family, flops, nbytes, name, *args, _stream(dev_of))


def _call_on_current(family: str, flops: float, nbytes: float, name: str, *args) -> None:
    if not PROF.enabled:
        _lib.call(name, *args)
        return
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    _lib.call(name, *args)
    e1.record()
    PROF.records.append((family, flops, nbytes, e0, e1))


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _need(t: torch.Tensor, dtype, name: str) -> None:
    if not t.is_cuda:
        raise _lib.XClipB200Error(f"{name} must be a CUDA tensor (x_clip_b200 has no CPU path)")
    if t.dtype != dtype:
        raise _lib.XClipB200Error(f"{name} must be {dtype}, got {t.dtype}")


def _rows2d(t: torch.Tensor, name: str) -> None:
    if t.dim() != 2 or t.stride(1) != 1:
        raise _lib.XClipB200Error(f"{name} must be 2-D with a contiguous last dim, got "
                                  f"shape {tuple(t.shape)} strides {t.stride()}")


def gemm(a: torch.Tensor, b: torch.Tensor, *, a_major: int = 0, b_major: int = 0,
         out: Optional[torch.Tensor] = None, out_dtype=BF16, alpha: float = 1.0,
         bias: Optional[torch.Tensor] = None, residual: Optional[torch.Tensor] = None,
         res_row_mod: int = 0, res_row_idx: Optional[torch.Tensor] = None,
         accumulate: bool = False) -> torch.Tensor:
    """out[M,N] (+)= alpha * A @ B^T (+bias) (+residual).  See xclip_gemm_bf16."""
    _need(a, BF16, "a"); _need(b, BF16, "b")
    _rows2d(a, "a"); _rows2d(b, "b")
    if a_major == 0:
        M, K = a.shape
    else:
        K, M = a.shape
    if b_major == 0:
        N, Kb = b.shape
    else:
        Kb, N = b.shape
    if K != Kb:
        raise _lib.XClipB200Error(f"gemm: contraction mismatch {K} vs {Kb}")
    if out is None:
        if accumulate:
            out = torch.zeros((M, N), device=a.device, dtype=F32)
        else:
            out = torch.empty((M, N), device=a.device, dtype=out_dtype)
    _rows2d(out, "out")
    if tuple(out.shape) != (M, N):
        raise _lib.XClipB200Error(f"gemm: out shape {tuple(out.shape)} != {(M, N)}")
    if out.dtype not in (BF16, F32):
        raise _lib.XClipB200Error("gemm: out must be bf16 or f32")
    if bias is not None:
        _need(bias, F32, "bias")
    ldr = 0
    if residual is not None:
        _need(residual, BF16, "residual"); _rows2d(residual, "residual")
        ldr = residual.stride(0)
    if res_row_idx is not None:
        if res_row_idx.dtype != torch.int32 or res_row_idx.numel() != M or not res_row_idx.is_contiguous() \
                or res_row_idx.device != a.device:
            raise _lib.XClipB200Error("gemm: res_row_idx must be a contiguous int32 [M] on the operands' device")
    fam = "gemm_wgrad" if (a_major == 1 and b_major == 1) else ("gemm_dgrad" if b_major == 1 else "gemm_fwd")
    nbytes = 2.0 * (M * K + N * K) + M * N * out.element_size() + (M * N * 2 if residual is not None else 0)
    _call(a, fam, 2.0 * M * N * K, nbytes, "xclip_gemm_bf16", a.data_ptr(), a.stride(0), a_major, b.data_ptr(), b.stride(0),
              b_major, out.data_ptr(), out.stride(0), 1 if out.dtype == F32 else 0, M, N, K,
              float(alpha), _ptr(bias), _ptr(residual), ldr, int(res_row_mod), _ptr(res_row_idx),
              1 if accumulate else 0)
    return out


def cast_bf16(src: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16 copy of a contiguous tensor (weights before they are MMA operands)."""
    _need(src, F32, "src")
    src = src.contiguous()
    dst = torch.empty(src.shape, device=src.device, dtype=BF16)
    if src.numel():
        _call(src, "cast", 0.0, 6.0 * src.numel(), "xclip_cast_f32_bf16", src.data_ptr(), dst.data_ptr(),
              src.numel())
    return dst


def layernorm_fwd(x, g, *, res=None, g2=None, eps=1e-5, want_stats=True):
    """out = LN(x)*g (+res); optionally out2 = LN(out)*g2.  Returns (out, stats, out2, stats2)."""
    _need(x, BF16, "x"); _rows2d(x, "x"); _need(g, F32, "g")
    rows, d = x.shape
    out = torch.empty((rows, d), device=x.device, dtype=BF16)
    stats = torch.empty((rows, 2), device=x.device, dtype=F32) if want_stats else None
    out2 = stats2 = None
    if g2 is not None:
        _need(g2, F32, "g2")
        out2 = torch.empty((rows, d), device=x.device, dtype=BF16)
        stats2 = torch.empty((rows, 2), device=x.device, dtype=F32)
    if res is not None:
        _need(res, BF16, "res"); _rows2d(res, "res")
    passes = 2 + (1 if res is not None else 0) + (1 if g2 is not None else 0)
    _call(x, "layernorm_fwd", 0.0, 2.0 * rows * d * passes, "xclip_layernorm_fwd", x.data_ptr(), x.stride(0), g.data_ptr(), _ptr(res),
              res.stride(0) if res is not None else 0, out.data_ptr(), out.stride(0), _ptr(stats),
              _ptr(g2), _ptr(out2), out2.stride(0) if out2 is not None else 0, _ptr(stats2),
              rows, d, float(eps))
    return out, stats, out2, stats2


def layernorm_bwd(dy, x, stats, g, *, add=None, dg=None):
    """dx = dLN(dy) (+add); dg (fp32 [d]) is accumulated into when given."""
    _need(dy, BF16, "dy"); _need(x, BF16, "x"); _rows2d(dy, "dy"); _rows2d(x, "x")
    rows, d = x.shape
    dx = torch.empty((rows, d), device=x.device, dtype=BF16)
    if add is not None:
        _need(add, BF16, "add"); _rows2d(add, "add")
    _call(dy, "layernorm_bwd", 0.0, 2.0 * rows * d * (3 + (1 if add is not None else 0)),
          "xclip_layernorm_bwd", dy.data_ptr(), dy.stride(0), x.data_ptr(), x.stride(0),
              stats.data_ptr(), g.data_ptr(), _ptr(add), add.stride(0) if add is not None else 0,
              dx.data_ptr(), dx.stride(0), _ptr(dg), rows, d)
    return dx


def l2norm_fwd(p):
    _need(p, F32, "p"); _rows2d(p, "p")
    rows, d = p.shape
    z = torch.empty((rows, d), device=p.device, dtype=F32)
    zrow = torch.empty((rows, 3 * d), device=p.device, dtype=BF16)
    zcol = torch.empty((rows, 3 * d), device=p.device, dtype=BF16)
    inv = torch.empty((rows,), device=p.device, dtype=F32)
    _call(p, "l2norm", 0.0, rows * d * (4 + 4 + 12), "xclip_l2norm_fwd", p.data_ptr(), p.stride(0), z.data_ptr(), zrow.data_ptr(),
              zcol.data_ptr(), inv.data_ptr(), rows, d)
    return z, zrow, zcol, inv


def l2norm_bwd(dz, z, inv):
    _need(dz, F32, "dz"); _need(z, F32, "z")
    dz = dz.contiguous()
    rows, d = z.shape
    dp = torch.empty((rows, d), device=z.device, dtype=BF16)
    _call(dz, "l2norm", 0.0, rows * d * (4 + 4 + 2), "xclip_l2norm_bwd", dz.data_ptr(), z.data_ptr(), inv.data_ptr(), dp.data_ptr(),
              rows, d)
    return dp


def attn_fwd(qkv, key_mask, B, n, heads, scale, causal=False):
    """qkv bf16 [B*n, 3*heads*64] -> (o bf16 [B*n, heads*64], lse f32 [B, heads, n])."""
    _need(qkv, BF16, "qkv"); _rows2d(qkv, "qkv")
    o = torch.empty((B * n, heads * 64), device=qkv.device, dtype=BF16)
    lse = torch.empty((B, heads, n), device=qkv.device, dtype=F32)
    if key_mask is not None:
        if key_mask.dtype != torch.bool or tuple(key_mask.shape) != (B, n) or not key_mask.is_contiguous():
            raise _lib.XClipB200Error("attn_fwd: key_mask must be a contiguous bool [B, n]")
    _call(qkv, "attn_fwd", 4.0 * B * heads * n * n * 64, 2.0 * B * n * heads * 64 * 4, "xclip_attn_fwd", qkv.data_ptr(), qkv.stride(0), _ptr(key_mask), o.data_ptr(),
              o.stride(0), lse.data_ptr(), B, n, heads, float(scale), 1 if causal else 0)
    return o, lse


def attn_bwd(qkv, key_mask, o, d_o, lse, B, n, heads, scale, causal=False):
    _need(d_o, BF16, "d_o"); _rows2d(d_o, "d_o")
    dqkv = torch.empty_like(qkv)
    delta = torch.empty((B, heads, n), device=qkv.device, dtype=F32)
    ws = torch.empty((B * n, heads * 64), device=qkv.device, dtype=F32) if n > 128 else None
    _call(qkv, "attn_bwd", 10.0 * B * heads * n * n * 64, 2.0 * B * n * heads * 64 * 8, "xclip_attn_bwd", qkv.data_ptr(), qkv.stride(0), _ptr(key_mask), o.data_ptr(),
              o.stride(0), d_o.data_ptr(), d_o.stride(0), lse.data_ptr(), delta.data_ptr(),
              dqkv.data_ptr(), dqkv.stride(0), _ptr(ws), B, n, heads, float(scale),
              1 if causal else 0)
    return dqkv


def patchify_gather(img, patch, keep=None):
    """img f32 [B,C,H,W] -> bf16 [B*k, patch*patch*C] (reference (p1 p2 c) order) for the patches
    keep[b, j] (int64 [B,k]) or all patches in order."""
    _need(img, F32, "image")
    img = img.contiguous()
    B, C, H, W = img.shape
    n = (H // patch) * (W // patch)
    k = n if keep is None else keep.shape[1]
    if keep is not None:
        if keep.dtype != torch.int64 or keep.shape[0] != B or keep.device != img.device:
            raise _lib.XClipB200Error("patchify: keep must be int64 [B, k] on the image's device")
        keep = keep.contiguous()
    out = torch.empty((B * k, patch * patch * C), device=img.device, dtype=BF16)
    _call(img, "embed", 0.0, B * k * patch * patch * C * 6.0, "xclip_patchify_gather", img.data_ptr(), B, C, H, W,
          int(patch), _ptr(keep), k, out.data_ptr())
    return out


def scatter_add_rows_(dst, src, idx=None, period=0):
    """dst f32 [V,d] rows idx[r] (int32) or r % period += src bf16 [rows,d]."""
    _need(src, BF16, "src"); _rows2d(src, "src"); _need(dst, F32, "dst")
    rows, d = src.shape
    _call(src, "embed", 0.0, rows * d * 6.0, "xclip_scatter_add_rows", _ptr(idx), int(period), src.data_ptr(),
          src.stride(0), dst.data_ptr(), rows, d, dst.shape[0])
    return dst


def colsum_rows_(dst, src):
    """dst f32 [d] += column sums of src bf16 [rows,d]."""
    _need(src, BF16, "src"); _rows2d(src, "src"); _need(dst, F32, "dst")
    _call(src, "embed", 0.0, src.numel() * 2.0, "xclip_colsum_rows", src.data_ptr(), src.stride(0), dst.data_ptr(),
          src.shape[0], src.shape[1])
    return dst


def ff_weights(w1, w2, g4):
    """bf16 operands of the fused feed-forward: row-permuted up-projection, gain-scaled
    down-projection and its row sums (see xclip_ff_permute_cast / xclip_ff_scale_cast)."""
    _need(w1, F32, "w1"); _need(w2, F32, "w2"); _need(g4, F32, "g4")
    d = w1.shape[1]
    if tuple(w1.shape) != (8 * d, d) or tuple(w2.shape) != (d, 4 * d) or g4.numel() != 4 * d:
        raise _lib.XClipB200Error("ff_weights: shapes must be [8d,d], [d,4d], [4d]")
    w1, w2, g4 = w1.contiguous(), w2.contiguous(), g4.contiguous()
    w1p = torch.empty((8 * d, d), device=w1.device, dtype=BF16)
    w2g = torch.empty((d, 4 * d), device=w1.device, dtype=BF16)
    colvec = torch.empty((d,), device=w1.device, dtype=F32)
    _call(w1, "cast", 0.0, 6.0 * w1.numel(), "xclip_ff_permute_cast", w1.data_ptr(), w1p.data_ptr(), d)
    _call(w2, "cast", 0.0, 6.0 * w2.numel(), "xclip_ff_scale_cast", w2.data_ptr(), g4.data_ptr(),
          w2g.data_ptr(), colvec.data_ptr(), d)
    return w1p, w2g, colvec


def ff_up(x, w1p, need_u=True):
    """x bf16 [M,d] -> (u bf16 [M,8d] = [value|gate] or None, hp bf16 [M,4d], rowsum f32 [M,d/16,2]).
    need_u=False (forward-only sweeps) skips the 8d-wide store of u."""
    _need(x, BF16, "x"); _rows2d(x, "x"); _need(w1p, BF16, "w1p")
    M, d = x.shape
    u = torch.empty((M, 8 * d), device=x.device, dtype=BF16) if need_u else None
    hp = torch.empty((M, 4 * d), device=x.device, dtype=BF16)
    rowsum = torch.empty((M, d // 16, 2), device=x.device, dtype=F32)    # one slot per 64-column box
    _call(x, "ff_up", 2.0 * M * 8 * d * d, 2.0 * (M * d + 8 * d * d + M * (12 if need_u else 4) * d), "xclip_ff_up",
          x.data_ptr(), x.stride(0), w1p.data_ptr(), _ptr(u), u.stride(0) if need_u else 0, hp.data_ptr(),
          hp.stride(0), rowsum.data_ptr(), M, d)
    return u, hp, rowsum


def ff_down(hp, w2g, colvec, rowsum, res, eps):
    """(x2 bf16 [M,d] = LN(hp) g W2^T + res, acc bf16 [M,d], stats f32 [M,2])."""
    _need(hp, BF16, "hp"); _rows2d(hp, "hp"); _need(w2g, BF16, "w2g"); _need(res, BF16, "res"); _rows2d(res, "res")
    M = hp.shape[0]
    d = w2g.shape[0]
    out = torch.empty((M, d), device=hp.device, dtype=BF16)
    acc = torch.empty((M, d), device=hp.device, dtype=BF16)
    stats = torch.empty((M, 2), device=hp.device, dtype=F32)
    _call(hp, "ff_down", 2.0 * M * d * 4 * d, 2.0 * (M * 4 * d + 4 * d * d + 3 * M * d), "xclip_ff_down",
          hp.data_ptr(), hp.stride(0), w2g.data_ptr(), colvec.data_ptr(), rowsum.data_ptr(),
          res.data_ptr(), res.stride(0), out.data_ptr(), out.stride(0), acc.data_ptr(), acc.stride(0),
          stats.data_ptr(), float(eps), M, d)
    return out, acc, stats


def ff_bwd_prep(dx, stats, acc=None, colvec=None):
    """-> (dxs bf16 [M,d] = dx * rstd, vsum f32 [d] = sum_r dxs[r] * mean_r, ab f32 [M,2] or None:
    the two row means of the LayerNorm backward, computed when acc and colvec are given)."""
    _need(dx, BF16, "dx"); _rows2d(dx, "dx"); _need(stats, F32, "stats")
    M, d = dx.shape
    dxs = torch.empty((M, d), device=dx.device, dtype=BF16)
    vsum = torch.zeros((d,), device=dx.device, dtype=F32)
    ab = None
    if acc is not None:
        _need(acc, BF16, "acc"); _rows2d(acc, "acc"); _need(colvec, F32, "colvec")
        ab = torch.empty((M, 2), device=dx.device, dtype=F32)
    _call(dx, "ff_small", 0.0, (4.0 + (2.0 if acc is not None else 0.0)) * M * d, "xclip_ff_bwd_prep",
          dx.data_ptr(), dx.stride(0), stats.data_ptr(), _ptr(acc), acc.stride(0) if acc is not None else 0,
          _ptr(colvec), dxs.data_ptr(), vsum.data_ptr(), _ptr(ab), M, d)
    return dxs, vsum, ab


def ff_bwd(dx, w2g, u, stats, ab):
    """du bf16 [M,8d]: LayerNorm(4d) + GEGLU backward fused into the dgrad GEMM dx @ w2g."""
    _need(dx, BF16, "dx"); _rows2d(dx, "dx"); _need(w2g, BF16, "w2g"); _need(u, BF16, "u"); _rows2d(u, "u")
    _need(stats, F32, "stats"); _need(ab, F32, "ab")
    M, d = dx.shape
    du = torch.empty((M, 8 * d), device=dx.device, dtype=BF16)
    _call(dx, "ff_bwd", 2.0 * M * 4 * d * d, 2.0 * (M * d + 4 * d * d + 16 * M * d), "xclip_ff_bwd",
          dx.data_ptr(), dx.stride(0), w2g.data_ptr(), u.data_ptr(), u.stride(0), stats.data_ptr(),
          ab.data_ptr(), du.data_ptr(), du.stride(0), M, d)
    return du


def ff_w2_grad_post_(raw, vsum, g4, w2=None, dg=None):
    """In place dW2 = g4 * (raw - vsum (x) 1); with w2/dg also accumulates the gain gradient."""
    _need(raw, F32, "raw"); _need(vsum, F32, "vsum"); _need(g4, F32, "g4")
    d = raw.shape[0]
    if w2 is not None:
        _need(w2, F32, "w2"); _need(dg, F32, "dg")
        w2 = w2.contiguous()
    _call(raw, "ff_small", 0.0, (8.0 + (4.0 if w2 is not None else 0.0)) * raw.numel(), "xclip_ff_w2_grad_post",
          raw.data_ptr(), vsum.data_ptr(), g4.data_ptr(), _ptr(w2), _ptr(dg), d)
    return raw


def adamw_step_(p, g, m, v, lr, beta1, beta2, eps, weight_decay, step, grad_scale=1.0):
    """In-place fused AdamW over flat fp32 buffers (see xclip_adamw_step)."""
    for t, nm in ((p, "p"), (g, "g"), (m, "m"), (v, "v")):
        _need(t, F32, nm)
        if not t.is_contiguous() or t.numel() != p.numel():
            raise _lib.XClipB200Error(f"adamw: {nm} must be contiguous with {p.numel()} elements")
    _call(p, "adamw", 0.0, 28.0 * p.numel(), "xclip_adamw_step", p.data_ptr(), g.data_ptr(), m.data_ptr(),
          v.data_ptr(), p.numel(), float(lr), float(beta1), float(beta2), float(eps), float(weight_decay),
          int(step), float(grad_scale))


def rotary_(qkv, n, nslices, cos_tab, sin_tab, inverse=False):
    """In-place rotary embedding of the q | k | v head slices (see xclip_rotary_inplace)."""
    _need(qkv, BF16, "qkv"); _rows2d(qkv, "qkv"); _need(cos_tab, F32, "cos"); _need(sin_tab, F32, "sin")
    if tuple(cos_tab.shape) != (n, 16) or tuple(sin_tab.shape) != (n, 16) or not (
            cos_tab.is_contiguous() and sin_tab.is_contiguous()):
        raise _lib.XClipB200Error("rotary: cos/sin tables must be contiguous [n, 16]")
    _call(qkv, "rotary", 0.0, 4.0 * qkv.shape[0] * nslices * 32, "xclip_rotary_inplace", qkv.data_ptr(),
          qkv.stride(0), qkv.shape[0], int(n), int(nslices), cos_tab.data_ptr(), sin_tab.data_ptr(),
          1 if inverse else 0)
    return qkv


def nce_fwd(a, b, temp_exp, diag_offset, dcl, loss_accum=None, loss_scale=0.0):
    """Row-block InfoNCE forward: (lse [R], pos [R]) for rows a vs all columns b.
    temp_exp: fp32 DEVICE scalar tensor holding exp(temperature)."""
    _need(a, BF16, "a"); _need(b, BF16, "b"); _need(temp_exp, F32, "temp_exp")
    R, D = a.shape
    C = b.shape[0]
    nblk = _lib.load().xclip_nce_num_col_blocks(C)
    part = torch.empty((nblk, R, 2), device=a.device, dtype=F32)
    pos = torch.empty((R,), device=a.device, dtype=F32)
    lse = torch.empty((R,), device=a.device, dtype=F32)
    _call(a, "nce_fwd", 2.0 * R * C * D, 2.0 * (R + C) * D + 8.0 * R, "xclip_nce_fwd", a.data_ptr(), b.data_ptr(), R, C, D, temp_exp.data_ptr(),
              int(diag_offset), 1 if dcl else 0, part.data_ptr(), pos.data_ptr(), lse.data_ptr(),
              _ptr(loss_accum), float(loss_scale))
    return lse, pos


def nce_bwd(a, b, temp_exp, diag_offset, dcl, lse_row, lse_col, w_row, w_col, w_diag, gscale,
            dtemp=None):
    """bf16 temp*g [R, roundup8(C)] (columns >= C are zero); see xclip_nce_bwd."""
    _need(gscale, F32, "gscale")
    R, D = a.shape
    C = b.shape[0]
    ldg = (C + 7) // 8 * 8
    g = torch.empty((R, ldg), device=a.device, dtype=BF16)
    _call(a, "nce_bwd", 2.0 * R * C * D, 2.0 * (R + C) * D + 2.0 * R * C, "xclip_nce_bwd", a.data_ptr(), b.data_ptr(), R, C, D, temp_exp.data_ptr(),
              int(diag_offset), 1 if dcl else 0, _ptr(lse_row), _ptr(lse_col), float(w_row),
              float(w_col), float(w_diag), gscale.data_ptr(), g.data_ptr(), ldg, _ptr(dtemp))
    return g


def filip_segmax(a, b, temp_exp, seg_len, col_mul, col_add):
    """Per row of a and per seg_len-long block of rows of b: max / argmax of temp * <a_r, b_c>."""
    _need(a, BF16, "a"); _need(b, BF16, "b")
    R, D = a.shape
    C = b.shape[0]
    nseg = C // seg_len
    seg_max = torch.empty((R, nseg), device=a.device, dtype=F32)
    seg_arg = torch.empty((R, nseg), device=a.device, dtype=torch.int32)
    _call(a, "filip_segmax", 2.0 * R * C * D, 2.0 * (R + C) * D + 8.0 * R * nseg, "xclip_filip_segmax",
          a.data_ptr(), b.data_ptr(), R, C, D, temp_exp.data_ptr(), int(seg_len), _ptr(col_mul),
          _ptr(col_add), seg_max.data_ptr(), seg_arg.data_ptr())
    return seg_max, seg_arg


def filip_reduce(seg_max, weights, samples, length, nseg, transpose):
    out = torch.empty((nseg, samples) if transpose else (samples, nseg), device=seg_max.device, dtype=F32)
    _call(seg_max, "filip_small", 0.0, 4.0 * seg_max.numel(), "xclip_filip_reduce", seg_max.data_ptr(),
          weights.data_ptr(), samples, length, nseg, out.data_ptr(), 1 if transpose else 0)
    return out


def filip_nce_fwd(s, diag_off, dcl, loss_accum, loss_scale):
    R, C = s.shape
    lse = torch.empty((R,), device=s.device, dtype=F32)
    _call(s, "filip_small", 0.0, 4.0 * s.numel(), "xclip_filip_nce_fwd", s.data_ptr(), R, C,
          int(diag_off), 1 if dcl else 0, lse.data_ptr(), _ptr(loss_accum), float(loss_scale))
    return lse


def filip_nce_bwd(s, lse, diag_off, dcl, gscale):
    R, C = s.shape
    g = torch.empty_like(s)
    _call(s, "filip_small", 0.0, 8.0 * s.numel(), "xclip_filip_nce_bwd", s.data_ptr(), lse.data_ptr(), R,
          C, int(diag_off), 1 if dcl else 0, gscale.data_ptr(), g.data_ptr())
    return g


def filip_expand(seg_arg, seg_max, wmat, rowscale, temp_exp, row0, rows, rows_per_sample, seg_len,
                 nseg, dtemp):
    g = torch.empty((rows, nseg * seg_len), device=seg_arg.device, dtype=BF16)
    _call(seg_arg, "filip_expand", 0.0, 2.0 * g.numel(), "xclip_filip_expand", seg_arg.data_ptr(),
          seg_max.data_ptr(), wmat.data_ptr(), rowscale.data_ptr(), temp_exp.data_ptr(), int(row0),
          int(rows), int(rows_per_sample), int(seg_len), int(nseg), g.data_ptr(), g.stride(0),
          _ptr(dtemp))
    return g


def text_embed_fwd(ids, tok, pos, cls):
    """ids int64 [B,n] -> bf16 [B, n+1, d] = [cls | tok[ids] + pos]."""
    if ids.dtype != torch.int64 or not ids.is_cuda:
        raise _lib.XClipB200Error("text_embed: ids must be a CUDA int64 tensor")
    _need(tok, F32, "token table"); _need(pos, F32, "position table"); _need(cls, F32, "cls token")
    if not (tok.is_contiguous() and pos.is_contiguous() and cls.is_contiguous()):
        raise _lib.XClipB200Error("text_embed: embedding tables must be contiguous")
    ids = ids.contiguous()
    B, n = ids.shape
    vocab, d = tok.shape
    if pos.shape[0] < n or pos.shape[1] != d or cls.numel() != d:
        raise _lib.XClipB200Error("text_embed: table shapes do not match the ids")
    out = torch.empty((B, n + 1, d), device=ids.device, dtype=BF16)
    _call(ids, "embed", 0.0, B * (n + 1) * d * 6.0, "xclip_text_embed_fwd", ids.data_ptr(), tok.data_ptr(),
          pos.data_ptr(), cls.data_ptr(), out.data_ptr(), B, n, d, vocab)
    return out


def text_embed_bwd(ids, dx, vocab, pos_rows):
    ids = ids.contiguous()
    B, n = ids.shape
    d = dx.shape[-1]
    dx = dx.contiguous()
    _need(dx, BF16, "dx")
    dtok = torch.zeros((vocab, d), device=dx.device, dtype=F32)
    dpos = torch.zeros((pos_rows, d), device=dx.device, dtype=F32)
    dcls = torch.zeros((d,), device=dx.device, dtype=F32)
    _call(ids, "embed", 0.0, B * (n + 1) * d * 8.0, "xclip_text_embed_bwd", ids.data_ptr(), dx.data_ptr(),
          dtok.data_ptr(), dpos.data_ptr(), dcls.data_ptr(), B, n, d, vocab)
    return dtok, dpos, dcls
