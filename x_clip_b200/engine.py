"""Forward/backward schedules of the hot path as torch.autograd.Functions.

Each Function is a hand-written schedule of C-ABI kernel calls (x_clip_b200.kernels);
autograd only stitches them to the few torch ops left around them (embedding gather,
patchify, patch-dropout gather).  Activations are bf16, accumulation/statistics fp32,
parameters stay fp32 in the modules (state_dict compatible with the reference) and are
cast to bf16 once per step.

Reference call sites: Transformer.forward x_clip/x_clip.py:274-291 (TransformerFn),
nn.Linear :358,:368 (LinearFn), :713-724 (ProjectL2NormFn), :759-769 + :797-847
(ContrastiveLossFn, with x_clip/distributed.py:41-56 for the gather contract).
"""
from __future__ import annotations

from typing import List, Optional

import torch

from . import kernels as K
from . import distributed as D_

BF16 = torch.bfloat16
F32 = torch.float32
LN_EPS = 1e-5   # the reference's fp32 branch (x_clip.py:118); parameters/outputs are fp32-facing

_scope_cache = None     # dict while a weight_scope() is active, else None


def ff_weights(w1: torch.Tensor, w2: torch.Tensor, g4: torch.Tensor):
    """(w1 permuted bf16, w2*g4 bf16, row sums) for the fused feed-forward; shared inside a
    weight_scope() like weight_bf16."""
    key = ("ff", id(w1), id(w2), id(g4))
    if _scope_cache is not None:
        hit = _scope_cache.get(key)
        if hit is not None and hit[0] is w1:
            return hit[1]
    out = K.ff_weights(w1.detach(), w2.detach(), g4.detach())
    if _scope_cache is not None:
        _scope_cache[key] = (w1, out)
    return out


def weight_bf16(p: torch.Tensor) -> torch.Tensor:
    """bf16 copy of an fp32 parameter (the MMA operand).

    Cast afresh on every call: a cache validated by `p._version` goes stale under `p.data.add_()`
    style updates (Lion/LARS-type optimizers, EMA swaps, clamping), which do not bump the version
    counter - the kernels would silently keep training on old weights.  Forward schedules keep
    the casts they used in `ctx` for their backward (autograd semantics: backward sees the weights
    of its forward).  Only inside an explicit `weight_scope()` - one micro-batched forward or
    backward sweep, during which no optimizer can run - are casts shared between calls."""
    if _scope_cache is not None:
        hit = _scope_cache.get(id(p))
        if hit is not None and hit[0] is p:
            return hit[1]
    w = K.cast_bf16(p.detach())
    if _scope_cache is not None:
        _scope_cache[id(p)] = (p, w)     # holds p: ids cannot be recycled inside the scope
    return w


class weight_scope:
    """Share bf16 weight casts between the encoder calls of ONE sweep over micro-batches.
    `cache`: continue with the casts of an earlier scope (the backward sweep of a step reuses the
    forward sweep's - autograd semantics: backward sees the weights of its forward)."""

    def __init__(self, cache=None):
        self.given = cache

    def __enter__(self):
        global _scope_cache
        self.prev = _scope_cache
        if self.given is not None:
            _scope_cache = self.given
        elif _scope_cache is None:
            _scope_cache = {}
        self.cache = _scope_cache
        return self

    def __exit__(self, *exc):
        global _scope_cache
        _scope_cache = self.prev
        return False


def _wgrad(dy: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """dW[out,in] = dy^T @ x in fp32: both operands consumed MN-major, split-K + atomics."""
    out = torch.zeros((dy.shape[1], x.shape[1]), device=dy.device, dtype=F32)
    K.gemm(dy, x, a_major=1, b_major=1, out=out, accumulate=True)
    return out


# Set by the micro-batched step for every chunk but the last one it back-propagates: transformer
# weight gradients are then accumulated by the kernels straight INTO the existing `.grad` buffers
# (split-K wgrad GEMM with accumulate, gain gradients by atomics) and `None` is returned to autograd -
# no zero-filled temporary, no `grad += new` pass per parameter and chunk.  The last chunk returns
# ordinary gradient tensors, so post-accumulate hooks (GradSync) fire exactly once per step.
_accumulate_into_grad = False
# User option (INTEGRATION.md §3): False sends every chunk's gradients through autograd, so gradient
# hooks fire once per chunk instead of once per step.
INPLACE_GRAD_ACCUMULATION = True


def _grad_target(param: torch.Tensor):
    """`param.grad` when this backward may accumulate into it in place, else None."""
    if not _accumulate_into_grad:
        return None
    g = getattr(param, "grad", None)
    if g is None or g.dtype != F32 or not g.is_contiguous() or g.shape != param.shape or not param.is_leaf:
        return None
    return g


class TransformerFn(torch.autograd.Function):
    """x[B,n,d] (bf16) -> norm_out(blocks(norm_in(x))) (bf16); mask: bool [B,n] or None.

    flat weights = [norm_in.g, norm_out.g] + depth * [g1, wqkv, wo, go, g2, w1, g4, w2].
    causal: the reference's causal mask (x_clip.py:233-236); rot_cos / rot_sin: f32 [n, 16] tables of
    the rotary embedding applied to q, k and v (x_clip.py:221-223) or None.
    """

    @staticmethod
    def forward(ctx, x, mask, heads: int, depth: int, causal: bool, rot_cos, rot_sin, need_bwd: bool,
                *weights):
        B, n, d = x.shape
        M = B * n
        scale = 64 ** -0.5
        g_in, g_out = weights[0], weights[1]
        layers = [weights[2 + 8 * L: 2 + 8 * (L + 1)] for L in range(depth)]
        x_in = x.reshape(M, d)
        if x_in.dtype != BF16:
            x_in = x_in.to(BF16)
        x_in = x_in.contiguous()
        mask_c = None if mask is None else mask.contiguous()

        saved, ff_saved = [], []
        # need_bwd = torch.is_grad_enabled() at the call site (inside forward() it is always off and
        # needs_input_grad ignores no_grad): in the first sweep of the micro-batched step and in
        # inference nothing is kept for a backward, and the 8d-wide u = [value | gate] is not written
        # bf16 MMA operands of this call's weights; backward reuses exactly these (ctx.wb)
        wb = [tuple(weight_bf16(w) for w in (l[1], l[2], l[5])) for l in layers]
        # norm_in fused with the first pre-norm
        xcur, st_in, xn, st1 = K.layernorm_fwd(x_in, g_in, g2=layers[0][0], eps=LN_EPS)
        for L, (g1, wqkv, wo, go, g2, w1, g4, w2) in enumerate(layers):
            bqkv, bo, b1 = wb[L]
            qkv = K.gemm(xn, bqkv)
            if rot_cos is not None:
                K.rotary_(qkv, n, 3 * heads, rot_cos, rot_sin)
            o, lse = K.attn_fwd(qkv, mask_c, B, n, heads, scale, causal)
            y = K.gemm(o, bo)
            # x1 = LN(y)*go + x ; xn2 = LN(x1)*g2   (attention tail + feed-forward pre-norm)
            x1, st_y, xn2, st_x1 = K.layernorm_fwd(y, go, res=xcur, g2=g2, eps=LN_EPS)
            # h below is hp = value*gelu(gate) BEFORE the LayerNorm (the norm is folded into the
            # down-projection)
            w1p, w2g, colvec = ff_weights(w1, w2, g4)
            u, h, rowsum = K.ff_up(xn2, w1p, need_u=need_bwd)
            x2, acc, st_v = K.ff_down(h, w2g, colvec, rowsum, x1, LN_EPS)
            if need_bwd:
                ff_saved.append((w2g, colvec, acc))
            # forward-only sweeps keep NOTHING alive beyond the layer (the list below would otherwise hold
            # every layer's activations until the call returns: ~14 of the 22 d per token-layer)
            if need_bwd:
                saved.append((xcur, st1, xn, qkv, o, lse, y, st_y, x1, st_x1, xn2, u, st_v, h))
            del qkv, o, lse, y, x1, xn2, u, h
            xcur = x2
            if L + 1 < depth:
                xn, st1, _, _ = K.layernorm_fwd(xcur, layers[L + 1][0], eps=LN_EPS)
        out, st_out, _, _ = K.layernorm_fwd(xcur, g_out, eps=LN_EPS)

        ctx.saved = saved
        ctx.tail = (x_in, st_in, xcur, st_out) if need_bwd else None
        ctx.mask = mask_c
        ctx.dims = (B, n, d, heads, depth, scale, causal)
        ctx.rot = (rot_cos, rot_sin)
        ctx.ff_saved = ff_saved
        ctx.weights = weights
        ctx.wb = wb
        return out.view(B, n, d)

    @staticmethod
    def backward(ctx, dout):
        B, n, d, heads, depth, scale, causal = ctx.dims
        rot_cos, rot_sin = ctx.rot
        M = B * n
        weights = ctx.weights
        g_in, g_out = weights[0], weights[1]
        layers = [weights[2 + 8 * L: 2 + 8 * (L + 1)] for L in range(depth)]
        x_in, st_in, x_last, st_out = ctx.tail
        dev = dout.device
        dout = dout.reshape(M, d)
        if dout.dtype != BF16:
            dout = dout.to(BF16)
        dout = dout.contiguous()

        grads: List[Optional[torch.Tensor]] = [None] * len(weights)

        def gain_grad(idx):
            """fp32 accumulator for the gain gradient of weights[idx]: its .grad (in-place mode) or zeros"""
            tgt = _grad_target(weights[idx])
            if tgt is not None:
                return tgt, None
            z = torch.zeros(weights[idx].shape[0], device=dev, dtype=F32)
            return z, z

        def weight_grad(idx, dy_, x_):
            tgt = _grad_target(weights[idx])
            if tgt is not None:
                K.gemm(dy_, x_, a_major=1, b_major=1, out=tgt, accumulate=True)
                return None
            return _wgrad(dy_, x_)

        dg_out, grads[1] = gain_grad(1)
        dx = K.layernorm_bwd(dout, x_last, st_out, g_out, dg=dg_out)
        for L in reversed(range(depth)):
            g1, wqkv, wo, go, g2, w1, g4, w2 = layers[L]
            xcur, st1, xn, qkv, o, lse, y, st_y, x1, st_x1, xn2, u, st_v, h = ctx.saved[L]
            ctx.saved[L] = None
            bqkv, bo, b1 = ctx.wb[L]
            base = 2 + 8 * L
            # feed-forward: x2 = h @ w2^T + x1
            dg4, grads[base + 6] = gain_grad(base + 6)
            # h is the pre-norm hp.  Row means of the LayerNorm backward from d-wide data, the
            # LN + GEGLU backward inside the dgrad GEMM, dW2 / dg4 from dW2g = dxs^T hp - vsum
            w2g, colvec, acc = ctx.ff_saved[L]
            ctx.ff_saved[L] = None
            dxs, vsum, ab = K.ff_bwd_prep(dx, st_v, acc, colvec)
            du = K.ff_bwd(dx, w2g, u, st_v, ab)
            dw2 = K.ff_w2_grad_post_(_wgrad(dxs, h), vsum, g4.detach(), w2.detach(), dg4)
            tgt = _grad_target(w2)
            if tgt is not None:
                tgt.add_(dw2)
                dw2 = None
            grads[base + 7] = dw2
            dxn2 = K.gemm(du, b1, b_major=1)
            grads[base + 5] = weight_grad(base + 5, du, xn2)
            del du
            dg2, grads[base + 4] = gain_grad(base + 4)
            dx1 = K.layernorm_bwd(dxn2, x1, st_x1, g2, add=dx, dg=dg2)
            # attention: x1 = LN(o @ wo^T) * go + x
            dgo, grads[base + 3] = gain_grad(base + 3)
            dy = K.layernorm_bwd(dx1, y, st_y, go, dg=dgo)
            d_o = K.gemm(dy, bo, b_major=1)
            grads[base + 2] = weight_grad(base + 2, dy, o)
            dqkv = K.attn_bwd(qkv, ctx.mask, o, d_o, lse, B, n, heads, scale, causal)
            if rot_cos is not None:      # back through the rotation (its transpose)
                K.rotary_(dqkv, n, 3 * heads, rot_cos, rot_sin, inverse=True)
            dxn = K.gemm(dqkv, bqkv, b_major=1)
            grads[base + 1] = weight_grad(base + 1, dqkv, xn)
            dg1, grads[base + 0] = gain_grad(base + 0)
            dx = K.layernorm_bwd(dxn, xcur, st1, g1, add=dx1, dg=dg1)
        dg_in, grads[0] = gain_grad(0)
        dx_in = K.layernorm_bwd(dx, x_in, st_in, g_in, dg=dg_in)
        ctx.saved = ctx.wb = None
        return (dx_in.view(B, n, d), None, None, None, None, None, None, None, *grads)


class TextEmbedFn(torch.autograd.Function):
    """[cls | token_emb[ids] + abs_pos_emb] -> bf16 [B, n+1, d] (x_clip.py:320-332), one pass."""

    @staticmethod
    def forward(ctx, ids, tok, pos, cls):
        out = K.text_embed_fwd(ids, tok.detach(), pos.detach(), cls.detach())
        ctx.save_for_backward(ids)
        ctx.shapes = (tok.shape[0], pos.shape[0])
        return out

    @staticmethod
    def backward(ctx, dx):
        (ids,) = ctx.saved_tensors
        vocab, pos_rows = ctx.shapes
        if dx.dtype != BF16:
            dx = dx.to(BF16)
        dtok, dpos, dcls = K.text_embed_bwd(ids, dx, vocab, pos_rows)
        return None, dtok, dpos, dcls


class LinearFn(torch.autograd.Function):
    """y = x @ W^T (+ bias) (+ table[row % period])  - x bf16 [M,K], W fp32 [N,K].

    `table` is a positional-embedding table added per row modulo `period` (the vision
    transformer's pos_emb, x_clip.py:382-383) fused in the GEMM epilogue."""

    @staticmethod
    def forward(ctx, x, weight, bias, table):
        x = x.contiguous()
        tbl16 = None if table is None else K.cast_bf16(table.detach())
        wb = weight_bf16(weight)
        y = K.gemm(x, wb, bias=None if bias is None else bias.detach(),
                   residual=tbl16, res_row_mod=0 if table is None else table.shape[0])
        ctx.save_for_backward(x, wb)
        ctx.has_bias = bias is not None
        ctx.period = None if table is None else table.shape[0]
        return y

    @staticmethod
    def backward(ctx, dy):
        x, wb = ctx.saved_tensors
        dy = dy.contiguous()
        if dy.dtype != BF16:
            dy = dy.to(BF16)
        dx = K.gemm(dy, wb, b_major=1) if ctx.needs_input_grad[0] else None
        dw = _wgrad(dy, x)
        db = dy.float().sum(dim=0) if ctx.has_bias else None
        dt = None
        if ctx.period is not None:
            dt = dy.float().view(-1, ctx.period, dy.shape[1]).sum(dim=0)
        return dx, dw, db, dt


class PatchEmbedFn(torch.autograd.Function):
    """tokens = patches @ W^T + bias + pos[index]  (x_clip.py:356-359, :382-383, with the
    PatchDropout selection :134-151 already applied to `patches` and `index`).

    patches bf16 [B*k, patch_dim] come from K.patchify_gather (only the kept patches are read from
    the image); `index` int32 [B*k] is the patch index of every row = the row of the position table
    the GEMM epilogue adds.  Backward: dW by the wgrad GEMM, d bias = column sums, d pos = rows of dy
    scatter-added by `index`; the image needs no gradient."""

    @staticmethod
    def forward(ctx, patches, index, weight, bias, table):
        wb = weight_bf16(weight)
        tbl16 = K.cast_bf16(table.detach())
        y = K.gemm(patches, wb, bias=bias.detach(), residual=tbl16, res_row_idx=index)
        ctx.save_for_backward(patches, index)
        ctx.table_rows = table.shape[0]
        return y

    @staticmethod
    def backward(ctx, dy):
        patches, index = ctx.saved_tensors
        dy = dy.contiguous()
        if dy.dtype != BF16:
            dy = dy.to(BF16)
        dw = _wgrad(dy, patches)
        db = K.colsum_rows_(torch.zeros(dy.shape[1], device=dy.device, dtype=F32), dy)
        dt = K.scatter_add_rows_(torch.zeros((ctx.table_rows, dy.shape[1]), device=dy.device, dtype=F32),
                                 dy, idx=index)
        return None, None, dw, db, dt


class ProjectL2NormFn(torch.autograd.Function):
    """z = normalize(e @ W^T) (x_clip.py:713-715).  Returns (z fp32, zrow, zcol): the last two
    are the split-bf16 MMA operands of the logits contraction (no grad), see xclip_l2norm_fwd."""

    @staticmethod
    def forward(ctx, e, weight):
        e = e.contiguous()
        wb = weight_bf16(weight)
        p = K.gemm(e, wb, out_dtype=F32)
        z, zrow, zcol, inv = K.l2norm_fwd(p)
        ctx.save_for_backward(e, wb, z, inv)
        ctx.mark_non_differentiable(zrow, zcol)
        return z, zrow, zcol

    @staticmethod
    def backward(ctx, dz, _a, _b):
        e, wb, z, inv = ctx.saved_tensors
        dp = K.l2norm_bwd(dz.contiguous().float(), z, inv)
        de = K.gemm(dp, wb, b_major=1) if ctx.needs_input_grad[0] else None
        dw = _wgrad(dp, e)
        return de, dw


class ContrastiveLossFn(torch.autograd.Function):
    """InfoNCE / DCL over all pairs of the GLOBAL batch (x_clip.py:759-769, :813-847).

    Inputs: local unit-norm latents zt, zi [b, D] (fp32, carry the graph), optional extra pair,
    the temperature parameter, and `ops`: per latent set the (zrow, zcol) split-bf16 operands.
    With world size W > 1 one all-gather exchanges the column operands of every set (replacing
    x_clip/distributed.py:14-39), each rank evaluates only its own row blocks, and a second tiny
    all-gather exchanges (lse, pos) so every rank returns the same global loss.  Backward
    reproduces AllGather.backward's contract (distributed.py:50-54): latent grads are
    d loss / d(local latents); d temperature is the full-batch gradient on every rank."""

    @staticmethod
    def forward(ctx, zt, zi, zt_x, zi_x, temperature, ops, dcl: bool, use_gather: bool):
        extra = len(ops) == 4
        rank, world = D_.world() if use_gather else (0, 1)
        b = ops[0][0].shape[0]
        D = ops[0][0].shape[1] // 3
        temp_exp = temperature.detach().float().exp().reshape(1)

        rows = [o[0] for o in ops]                                  # local [b, 3D], [hi|lo|hi]
        cols = D_.gather_rows([o[1] for o in ops]) if world > 1 else [o[1] for o in ops]
        Bg = world * b
        off = rank * b

        # forward row blocks: texts vs all images; images vs all texts (extra latents if any)
        T, I, TX, IX = 0, 1, 2, 3
        lse_t, pos_t = K.nce_fwd(rows[T], cols[I], temp_exp, off, dcl)
        if extra:
            lse_i, pos_i = K.nce_fwd(rows[IX], cols[TX], temp_exp, off, dcl)
        else:
            lse_i, pos_i = K.nce_fwd(rows[I], cols[T], temp_exp, off, dcl)

        stats = torch.stack([lse_t, pos_t, lse_i, pos_i])                      # [4, b]
        gstats = D_.gather_stats(stats) if world > 1 else stats
        loss = ((gstats[0] - gstats[1]).sum() + (gstats[2] - gstats[3]).sum()) / (2.0 * Bg)

        ctx.cfg = (dcl, extra, rank, world, b, D, Bg, off)
        ctx.temp_exp = temp_exp
        ctx.rows, ctx.cols = rows, cols
        ctx.lse = (lse_t, lse_i, gstats[0].contiguous(), gstats[2].contiguous())
        return loss

    @staticmethod
    def backward(ctx, gloss):
        dcl, extra, rank, world, b, D, Bg, off = ctx.cfg
        temp_exp = ctx.temp_exp
        rows, cols = ctx.rows, ctx.cols
        lse_t, lse_i, lse_t_all, lse_i_all = ctx.lse
        gscale = (gloss.detach().float() / (2.0 * Bg)).reshape(1)
        dtemp = torch.zeros(1, device=gloss.device, dtype=F32)
        T, I, TX, IX = 0, 1, 2, 3

        def latent_grad(r, c, lse_row, lse_col, w_row, w_col, w_diag, want_dtemp):
            g = K.nce_bwd(rows[r], cols[c], temp_exp, off, dcl, lse_row, lse_col, w_row, w_col,
                          w_diag, gscale, dtemp if want_dtemp else None)
            # d rows = (temp * g) @ cols_hi ; g is zero-padded to a multiple of 8 columns
            return K.gemm(g, _pad_rows(cols[c][:, :D], g.shape[1]), b_major=1, out_dtype=F32)

        if not extra:
            dzt = latent_grad(T, I, lse_t, lse_i_all, 1.0, 1.0, 2.0, True)
            dzi = latent_grad(I, T, lse_i, lse_t_all, 1.0, 1.0, 2.0, False)
            dzt_x = dzi_x = None
        else:
            dzt = latent_grad(T, I, lse_t, None, 1.0, 0.0, 1.0, True)
            dzi = latent_grad(I, T, None, lse_t_all, 0.0, 1.0, 1.0, False)
            dzi_x = latent_grad(IX, TX, lse_i, None, 1.0, 0.0, 1.0, True)
            dzt_x = latent_grad(TX, IX, None, lse_i_all, 0.0, 1.0, 1.0, False)
        if world > 1:
            D_.all_reduce_sum_(dtemp)       # every rank holds the full-batch d loss / d temperature
        ctx.rows = ctx.cols = None
        return (dzt, dzi, dzt_x, dzi_x, dtemp.reshape(()), None, None, None)


def _pad_rows(m: torch.Tensor, rows: int) -> torch.Tensor:
    """g has roundup8(C) columns; the matching operand needs that many rows (zeros beyond C)."""
    if m.shape[0] == rows:
        return m
    out = torch.zeros((rows, m.shape[1]), device=m.device, dtype=m.dtype)
    out[: m.shape[0]] = m
    return out


def _avail_bytes(dev) -> int:
    """HBM a further allocation can draw on: free device memory + the cached-but-unused part of
    torch's pool (counted at 80 %: cached blocks are not one contiguous range)."""
    free, _ = torch.cuda.mem_get_info(dev)
    cached = torch.cuda.memory_reserved(dev) - torch.cuda.memory_allocated(dev)
    return int(free + 0.8 * max(cached, 0))


# HBM head-room the retention planner leaves untouched: contrastive-loss workspace (g[b, B_g] bf16
# per direction, gathered operands), gradient buckets, allocator slack.
RETAIN_MARGIN_BYTES = 10 << 30
# transient buffers of one chunk's backward (du 8d + a few d-wide rows of one layer) relative to
# the chunk's saved activations (22 d per token-layer x depth)
RETAIN_TRANSIENT_FRAC = 0.15


class _InPlaceGradAccumulation:
    def __init__(self, flag: bool):
        self.flag = flag

    def __enter__(self):
        global _accumulate_into_grad
        self.prev = _accumulate_into_grad
        _accumulate_into_grad = self.flag
        return self

    def __exit__(self, *exc):
        global _accumulate_into_grad
        _accumulate_into_grad = self.prev
        return False


class ChunkedClipLossFn(torch.autograd.Function):
    """Full-batch contrastive loss with micro-batched encoders.

    The reference offers `checkpoint_during_training` (x_clip.py:280-286) to fit large batches;
    here the same need (4096 pairs per GPU for a 32768 global batch) is met by a GradCache-style
    schedule that is mathematically identical to the single-pass step:
      1. encode every chunk -> latents of the whole local batch
      2. one contrastive loss over ALL latents (with the usual cross-rank all-gather)
      3. in backward: d loss / d latents, then back-propagate the matching slice of the latent
         gradient through every chunk's encoders.
    B200-first memory plan: a chunk's saved activations are KEPT from step 1 for as many chunks as
    the 180 GB of HBM hold (`retain`: "auto" measures the first chunk's footprint and plans against
    the free memory; an int fixes the count; 0 = none); only the remaining chunks are encoded
    without saving anything and re-encoded in step 3 (RNG replayed for PatchDropout).  Retained
    chunks cost no extra flops; each re-encoded chunk costs one extra encoder forward."""

    @staticmethod
    def forward(ctx, clip, text, image, text_mask, chunk, temperature, retain="auto"):
        B = text.shape[0]
        dev = text.device
        bounds = [(s, min(s + chunk, B)) for s in range(0, B, chunk)]
        rng_states, zs, opss, kept = [], [], [], []
        foot = None                                   # bytes of one retained chunk's activations
        # "auto" plans ONCE per (batch, chunk size): the first step measures and decides, later steps
        # repeat its decision - the same tensors are then allocated in the same order every step, which
        # is what keeps torch's caching allocator free of fragmentation this close to the HBM limit
        plans = clip.__dict__.setdefault("_retain_plans", {})
        plan_key = (B, chunk, str(dev))
        planned = retain == "auto" and plan_key not in plans
        keep_mask = None                              # a remembered plan: which chunks stay resident
        if retain == "auto" and not planned:
            keep_mask = plans[plan_key]
        oom_fallbacks = 0
        with torch.no_grad(), weight_scope() as wscope:
            for k, (s, e) in enumerate(bounds):
                rng_states.append(torch.cuda.get_rng_state(dev))
                if keep_mask is not None:
                    keep_it = keep_mask[k]
                elif retain == "auto":
                    scale = (e - s) / float(chunk)
                    if foot is None:                  # first chunk: keep it, measure it
                        keep_it = True
                    else:
                        need = foot * scale * (1.0 + RETAIN_TRANSIENT_FRAC) + RETAIN_MARGIN_BYTES
                        keep_it = _avail_bytes(dev) >= need
                else:
                    keep_it = k < int(retain)
                if keep_it:
                    before = torch.cuda.memory_allocated(dev)
                    z = ops = None
                    try:
                        with torch.enable_grad():
                            z, ops = clip._encode_to_latents(text[s:e], image[s:e], text_mask[s:e])
                    except torch.OutOfMemoryError:
                        # the plan was too optimistic (a fragmented cache, memory taken by someone else
                        # since the estimate): this chunk and all later ones are re-encoded in backward
                        z = ops = None
                        retain, keep_mask = 0, None   # (an int plan: nothing further is kept)
                        oom_fallbacks += 1
                    if z is None:
                        torch.cuda.empty_cache()
                        torch.cuda.set_rng_state(rng_states[-1], dev)
                        z, ops = clip._encode_to_latents(text[s:e], image[s:e], text_mask[s:e])
                        kept.append(None)
                        zs.append(z)
                        opss.append(ops)
                        continue
                    kept.append(list(z))
                    if foot is None:
                        foot = max(torch.cuda.memory_allocated(dev) - before, 1)
                        if planned and len(bounds) > 1 and \
                                _avail_bytes(dev) < foot * (1.0 + RETAIN_TRANSIENT_FRAC) + RETAIN_MARGIN_BYTES:
                            kept[-1] = None           # not even a second live chunk fits beside it: let it go
                    z = [t.detach() for t in z]
                else:
                    z, ops = clip._encode_to_latents(text[s:e], image[s:e], text_mask[s:e])
                    kept.append(None)
                zs.append(z)
                opss.append(ops)
        nsets = len(zs[0])
        leaves = [torch.cat([z[j] for z in zs]).detach().requires_grad_(True) for j in range(nsets)]
        ops_all = tuple((torch.cat([o[j][0] for o in opss]), torch.cat([o[j][1] for o in opss]))
                        for j in range(nsets))
        temp_leaf = temperature.detach().requires_grad_(True)
        with torch.enable_grad():
            loss = ContrastiveLossFn.apply(
                leaves[0], leaves[1], leaves[2] if nsets == 4 else None,
                leaves[3] if nsets == 4 else None, temp_leaf, ops_all,
                clip.decoupled_contrastive_learning, clip.requires_all_gather)
        ctx.clip, ctx.inputs = clip, (text, image, text_mask)
        ctx.bounds, ctx.rng_states, ctx.kept = bounds, rng_states, kept
        ctx.graph = (loss, leaves, temp_leaf)
        ctx.weight_casts = wscope.cache
        n_kept = sum(z is not None for z in kept)
        if planned or (oom_fallbacks and plan_key in plans):
            plans[plan_key] = [z is not None for z in kept]    # WHICH chunks stay resident
        clip.last_step_plan = dict(chunks=len(bounds), retained=n_kept, chunk_activation_bytes=foot,
                                   oom_fallbacks=oom_fallbacks)
        return loss.detach()

    @staticmethod
    def backward(ctx, g):
        clip = ctx.clip
        text, image, text_mask = ctx.inputs
        loss, leaves, temp_leaf = ctx.graph
        with torch.enable_grad():
            torch.autograd.backward(loss, g)
        dz = [l.grad for l in leaves]
        dev = text.device
        keep_state = torch.cuda.get_rng_state(dev)
        kept = ctx.kept
        # retained chunks first: their backward releases HBM before any chunk is re-encoded
        order = [k for k in range(len(ctx.bounds)) if kept[k] is not None] + \
                [k for k in range(len(ctx.bounds)) if kept[k] is None]
        with weight_scope(ctx.weight_casts):
            for pos, k in enumerate(order):
                s, e = ctx.bounds[k]
                # parameter gradients accumulate over the chunks; gradient-sync hooks (GradSync)
                # must see a parameter ONCE per step, with its complete gradient: every chunk but
                # the last one processed runs with the hooks deferred (the DDP no_sync convention)
                with torch.enable_grad(), D_.defer_grad_sync(pos != len(order) - 1), \
                        _InPlaceGradAccumulation(INPLACE_GRAD_ACCUMULATION and pos != len(order) - 1):
                    if kept[k] is not None:
                        z, kept[k] = kept[k], None
                    else:
                        torch.cuda.set_rng_state(ctx.rng_states[k], dev)
                        z, _ = clip._encode_to_latents(text[s:e], image[s:e], text_mask[s:e])
                    torch.autograd.backward(list(z), [d[s:e] for d in dz])   # accumulates into .grad
                    del z
        torch.cuda.set_rng_state(keep_state, dev)
        ctx.graph = ctx.inputs = ctx.kept = ctx.weight_casts = None
        return None, None, None, None, None, temp_leaf.grad, None
