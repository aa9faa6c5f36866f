"""Generate tests/golden/*.json by running the REFERENCE (lucidrains/x-clip, imported
read-only from /root/reference) on deterministic protocol weights and inputs.

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

The reference has no tests or golden vectors of its own (SURVEY.md 4), so these files
are what pins oracle/clip_oracle.py.  While generating, the script also cross-checks the
oracle against the live reference (protocol weights AND the reference's native init with
the SURVEY 4 seed protocol) and refuses to write fixtures if they disagree.
"""
from __future__ import annotations

import inspect
import json
import os
import random
import sys
import zlib
from pathlib import Path

import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
REF = Path("/root/reference")
sys.path.insert(0, str(ROOT))

from oracle import clip_oracle as O  # noqa: E402

TINY = dict(dim_text=256, dim_image=256, dim_latent=256, num_text_tokens=128, text_enc_depth=2,
            text_seq_len=16, text_heads=4, visual_enc_depth=2, visual_heads=4,
            visual_image_size=64, visual_patch_size=16)
README = dict(dim_text=512, dim_image=512, dim_latent=512, num_text_tokens=10000,
              text_enc_depth=6, text_seq_len=256, text_heads=8, visual_enc_depth=6,
              visual_image_size=256, visual_patch_size=32, visual_heads=8)

# ViT-B/16-SHAPED towers (cfg3 of BASELINE.json at depth 2): dim_image 768 / 12 heads / 224 px / patch 16
# -> 196 patches (98 kept with the default patch dropout), text 77 tokens + CLS, CLIP-size latent
VITB16_2L = dict(dim_text=512, dim_image=768, dim_latent=512, num_text_tokens=1000, text_enc_depth=2,
                 text_seq_len=77, text_heads=8, visual_enc_depth=2, visual_heads=12,
                 visual_image_size=224, visual_patch_size=16)
# FILIP at the token counts of cfg4: 256 text tokens x 64 (32 with patch dropout) image tokens
FILIP_T256 = dict(dim_text=256, dim_image=256, dim_latent=256, num_text_tokens=512, text_enc_depth=1,
                  text_seq_len=256, text_heads=4, visual_enc_depth=1, visual_heads=4,
                  visual_image_size=256, visual_patch_size=32, use_all_token_embeds=True)

CASES = {
    # name: (cfg overrides, batch, pad_fraction, patch_dropout)
    "tiny_plain": (dict(TINY), 6, 0.2, 0.0),
    "tiny_nomask": (dict(TINY), 5, 0.0, 0.0),
    "tiny_dcl_extra": (dict(TINY, decoupled_contrastive_learning=True, extra_latent_projection=True), 6, 0.2, 0.0),
    "tiny_extra": (dict(TINY, extra_latent_projection=True), 4, 0.1, 0.0),
    "tiny_dcl": (dict(TINY, decoupled_contrastive_learning=True), 4, 0.1, 0.0),
    "tiny_filip": (dict(TINY, use_all_token_embeds=True), 4, 0.25, 0.0),
    "tiny_filip_dcl_extra": (dict(TINY, use_all_token_embeds=True, decoupled_contrastive_learning=True,
                                  extra_latent_projection=True), 4, 0.25, 0.0),
    "tiny_patchdrop": (dict(TINY), 6, 0.2, 0.5),
    "readme_plain": (dict(README), 4, 0.0, 0.0),
    "vitb16_shaped": (dict(VITB16_2L), 4, 0.1, 0.0),          # image attention n = 196, text n = 78
    "vitb16_shaped_drop": (dict(VITB16_2L), 4, 0.1, 0.5),     # image attention n = 98 (cfg3 bench shape)
    "filip_t256": (dict(FILIP_T256), 3, 0.3, 0.0),            # T = 256, I = 64
    "filip_t256_drop": (dict(FILIP_T256), 3, 0.3, 0.5),       # T = 256, I = 32
    "tiny_b64": (dict(TINY), 64, 0.2, 0.0),
    # text-tower variants (SURVEY 8a7 / 8f3): rotary embedding on q, k AND v; causal mask + EOS pooling
    "tiny_rotary": (dict(TINY, text_rotary_pos_emb=True), 6, 0.2, 0.0),
    "tiny_causal": (dict(TINY, text_causal_mask=True, text_eos_id=5), 6, 0.2, 0.0),
    "text77_causal": (dict(VITB16_2L, text_causal_mask=True, text_eos_id=999, visual_enc_depth=1), 4, 0.1, 0.5),                   # batch large enough for the 1e-2 d temperature gate
}
WEIGHT_SEED = 1234
INPUT_SEED = 4321
DROP_SEED = 99


def import_reference():
    if not REF.exists():
        raise SystemExit("/root/reference not present: goldens can only be generated in the build container")
    sys.path.insert(0, str(REF))
    import x_clip  # noqa
    return x_clip


def summ(t: torch.Tensor) -> dict:
    d = t.detach().double().flatten()
    return dict(shape=list(t.shape), sum=d.sum().item(), abs_sum=d.abs().sum().item(),
                sq_sum=(d * d).sum().item(), head=d[:8].tolist())


def build_reference(x_clip, cfg_kwargs, patch_dropout, state):
    clip = x_clip.CLIP(**cfg_kwargs, visual_patch_dropout=patch_dropout)
    full = dict(state)
    for k, v in clip.state_dict().items():        # non-parameter buffers (rotary inv_freq) keep their own values
        if k not in full:
            assert k.endswith("inv_freq"), k
            full[k] = v
    clip.load_state_dict(full, strict=True)
    clip.train()
    # text_causal_mask=True reads an undefined name `b` (x_clip.py:683) where the batch size is meant
    # (SURVEY.md 8c): supply it as a module global - the reference source itself stays untouched
    import x_clip.x_clip as _xc
    _xc.b = None
    return clip


def run_case(x_clip, name, cfg_kwargs, batch, pad_fraction, patch_dropout, grad_sample=0):
    """`grad_sample` > 0: also record each gradient at that many positions (all of a smaller one), drawn
    without replacement from a generator seeded by the case and parameter names."""
    cfg = O.ClipConfig(**cfg_kwargs)
    state = O.protocol_state_dict(cfg, WEIGHT_SEED)
    text, image = O.protocol_inputs(cfg, batch, INPUT_SEED, pad_fraction)
    clip = build_reference(x_clip, cfg_kwargs, patch_dropout, state)

    keep = None
    if patch_dropout > 0:
        n = (cfg.visual_image_size // cfg.visual_patch_size) ** 2
        k = max(1, int(n * (1 - patch_dropout)))
        torch.manual_seed(DROP_SEED)
        keep = torch.randn(batch, n).topk(k, dim=-1).indices   # PatchDropout's draw (x_clip.py:149)
    import x_clip.x_clip as _xc
    _xc.b = batch                                  # see build_reference()
    torch.manual_seed(DROP_SEED)
    loss = clip(text, image, return_loss=True)
    loss.backward()
    grads = {k: p.grad for k, p in clip.named_parameters() if p.grad is not None}

    torch.manual_seed(DROP_SEED)
    with torch.no_grad():
        enc_t, enc_i = clip(text, image, return_encodings=True)
        torch.manual_seed(DROP_SEED)
        lat = clip(text, image, return_latents=True)

    # --- oracle cross-check against the live reference
    p = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    o_loss, parts = O.clip_forward(p, text, image, cfg, keep=keep, return_parts=True)
    o_loss.backward()
    assert abs(o_loss.item() - loss.item()) <= 2e-6 * max(1.0, abs(loss.item())), (name, o_loss.item(), loss.item())
    assert torch.allclose(parts["enc_text"], enc_t, atol=2e-4, rtol=1e-4), name
    assert torch.allclose(parts["enc_image"], enc_i, atol=2e-4, rtol=1e-4), name
    for k, g in grads.items():
        og = p[k].grad
        assert og is not None, (name, k)
        denom = g.norm().item() + 1e-12
        assert (og - g).norm().item() / denom < 2e-4, (name, k, (og - g).norm().item() / denom)

    total = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values())).item()
    out = dict(
        case=name, cfg=cfg_kwargs, batch=batch, pad_fraction=pad_fraction, patch_dropout=patch_dropout,
        weight_seed=WEIGHT_SEED, input_seed=INPUT_SEED, drop_seed=DROP_SEED,
        loss=loss.item(), dtemperature=grads["temperature"].item(), grad_norm=total,
        grad_norms={k: g.double().norm().item() for k, g in grads.items()},
        enc_text=summ(enc_t), enc_image=summ(enc_i),
        latents=[summ(z) for z in lat],
        keep=None if keep is None else keep.tolist(),
        torch_version=torch.__version__,
    )
    if not cfg.use_all_token_embeds:
        out["text_latents"] = lat[0].tolist()
        out["image_latents"] = lat[1].tolist()
    if grad_sample:
        out["grad_samples"] = {}
        for k, g in grads.items():
            gen = torch.Generator().manual_seed(zlib.crc32(f"{name}/{k}".encode()))
            idx = torch.randperm(g.numel(), generator=gen)[:grad_sample].sort().values
            out["grad_samples"][k] = dict(idx=idx.tolist(), val=[float(f"{v:.7g}") for v in g.flatten()[idx].tolist()])
    return out


RANDOM_SEEDS = range(16)


def draw_random_case(rng: random.Random):
    """A small random configuration: widths, head counts, depths, sequence lengths, batch sizes, pad
    fractions, patch dropout and every combination of the loss flags."""
    heads_t, heads_i = rng.choice([1, 2, 4]), rng.choice([1, 2, 4])
    patch = rng.choice([8, 16])
    side = patch * rng.choice([2, 3, 4])
    cfg = dict(dim_text=64 * rng.choice([1, 2, 4]), dim_image=64 * rng.choice([1, 2, 4]),
               dim_latent=64 * rng.choice([1, 2, 4]), num_text_tokens=rng.choice([32, 97, 300]),
               text_enc_depth=rng.choice([1, 2, 3]), text_seq_len=rng.choice([5, 16, 33]), text_heads=heads_t,
               visual_enc_depth=rng.choice([1, 2]), visual_heads=heads_i, visual_image_size=side,
               visual_patch_size=patch)
    flags = dict(decoupled_contrastive_learning=rng.random() < 0.4, extra_latent_projection=rng.random() < 0.4,
                 use_all_token_embeds=rng.random() < 0.3)
    # (FILIP with a causal text tower does not run in the reference itself: 15 text tokens after the CLS
    #  strip against a 16-wide mask, x_clip.py:705 / :806)
    text_kind = rng.choice(["plain", "plain", "rotary"] + ([] if flags["use_all_token_embeds"] else ["causal"]))
    if text_kind == "rotary":
        flags["text_rotary_pos_emb"] = True
    elif text_kind == "causal":
        flags.update(text_causal_mask=True, text_eos_id=cfg["num_text_tokens"] - 1)
    cfg.update({k: v for k, v in flags.items() if v})
    batch = rng.choice([2, 3, 5, 8])
    pad = rng.choice([0.0, 0.2, 0.5])
    n_patches = (side // patch) ** 2
    drop = rng.choice([0.0, 0.0, 0.5]) if n_patches >= 4 else 0.0
    return cfg, batch, pad, drop


def random_cases(x_clip):
    """The reference on the configurations draw_random_case() gives for RANDOM_SEEDS (rng seed 1000 + seed)."""
    torch.set_num_threads(4)
    out = []
    for seed in RANDOM_SEEDS:
        cfg_kwargs, batch, pad, drop = draw_random_case(random.Random(1000 + seed))
        r = run_case(x_clip, f"random_{seed}", cfg_kwargs, batch, pad, drop, grad_sample=16)
        out.append({k: r[k] for k in ("case", "cfg", "batch", "pad_fraction", "patch_dropout", "weight_seed",
                                      "input_seed", "loss", "dtemperature", "grad_norm", "grad_norms", "grad_samples",
                                      "enc_text", "enc_image", "latents", "keep")})
    return out


def reference_signature(x_clip):
    """Keyword names and defaults of the reference's CLIP.__init__ / CLIP.forward, in order; a
    parameter without a default has no "default" entry."""
    def params(fn):
        return [{"name": k} if v.default is inspect.Parameter.empty else {"name": k, "default": v.default}
                for k, v in inspect.signature(fn).parameters.items() if k not in ("self", "kwargs")]
    return {"init": params(x_clip.CLIP.__init__), "forward": params(x_clip.CLIP.forward)}


def multiview_case(x_clip, name, cfg_kwargs, batch, n_aug_text, n_aug_image):
    """aug_text / aug_image views through the reference (x_clip.py:623-650, :851-868) vs the oracle."""
    cfg = O.ClipConfig(**cfg_kwargs)
    state = O.protocol_state_dict(cfg, WEIGHT_SEED)
    views = [O.protocol_inputs(cfg, batch, INPUT_SEED + 17 * v, 0.2) for v in range(1 + max(n_aug_text, n_aug_image))]
    texts = [views[v][0] for v in range(1 + n_aug_text)]
    images = [views[v][1] for v in range(1 + n_aug_image)]
    clip = build_reference(x_clip, cfg_kwargs, 0.0, state)
    loss = clip(texts[0], images[0], return_loss=True,
                aug_text=tuple(texts[1:]) if n_aug_text else None,
                aug_image=tuple(images[1:]) if n_aug_image else None)
    loss.backward()
    grads = {k: p.grad for k, p in clip.named_parameters() if p.grad is not None}
    p = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    o_loss = O.clip_forward_multiview(p, texts, images, cfg, clip.multiview_loss_weight)
    o_loss.backward()
    assert abs(o_loss.item() - loss.item()) <= 3e-6 * max(1.0, abs(loss.item())), (name, o_loss.item(), loss.item())
    for k, g in grads.items():
        assert (p[k].grad - g).norm().item() / (g.norm().item() + 1e-12) < 2e-4, (name, k)
    total = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values())).item()
    return dict(case=name, cfg=cfg_kwargs, batch=batch, n_aug_text=n_aug_text, n_aug_image=n_aug_image,
                view_seed_stride=17, pad_fraction=0.2, weight_seed=WEIGHT_SEED, input_seed=INPUT_SEED,
                multiview_loss_weight=clip.multiview_loss_weight, loss=loss.item(),
                dtemperature=grads["temperature"].item(), grad_norm=total,
                grad_norms={k: g.double().norm().item() for k, g in grads.items()})


def survey_anchor(x_clip, **extra):
    """SURVEY.md 4 protocol: manual_seed(0) -> CLIP(README cfg) -> manual_seed(1) -> inputs."""
    torch.manual_seed(0)
    clip = x_clip.CLIP(**README, visual_patch_dropout=0.0, **extra)
    clip.train()
    torch.manual_seed(1)
    text = torch.randint(0, 10000, (4, 256))
    image = torch.randn(4, 3, 256, 256)
    loss = clip(text, image, return_loss=True)
    loss.backward()
    gn = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in clip.parameters() if p.grad is not None)).item()
    # oracle on the reference's own native-init weights
    cfg = O.ClipConfig(**README, **extra)
    p = {k: v.detach().clone().requires_grad_(True) for k, v in clip.state_dict().items()}
    o_loss = O.clip_forward(p, text, image, cfg)
    o_loss.backward()
    assert abs(o_loss.item() - loss.item()) < 5e-6, (extra, o_loss.item(), loss.item())
    assert abs(p["temperature"].grad.item() - clip.temperature.grad.item()) < 1e-6
    return dict(extra=extra, loss=loss.item(), grad_norm=gn, dtemperature=clip.temperature.grad.item(),
                oracle_loss=o_loss.item())


def _rank_worker(rank, world, cfg_kwargs, state, texts, images, port, q):
    import torch.distributed as dist
    import torch.nn.functional as F
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sys.path.insert(0, str(REF))
    import x_clip
    import x_clip.distributed as xd
    # the reference's distributed.py uses two names it never defines (SURVEY.md 3.4)
    xd.exists = lambda v: v is not None
    xd.F = F
    torch.set_num_threads(2)
    clip = x_clip.CLIP(**cfg_kwargs, visual_patch_dropout=0.0)
    clip.load_state_dict(state)
    clip.train()
    loss = clip(texts[rank], images[rank], return_loss=True)
    loss.backward()
    grads = {k: p.grad for k, p in clip.named_parameters() if p.grad is not None}
    gn = torch.sqrt(sum((g.double() ** 2).sum() for g in grads.values())).item()
    q.put((rank, loss.item(), gn, grads["temperature"].item(),
           {k: g.double().norm().item() for k, g in grads.items()}))
    dist.barrier()
    dist.destroy_process_group()


def sharded_case(name, cfg_kwargs, world=2, per_rank=3):
    import torch.multiprocessing as mp
    cfg = O.ClipConfig(**cfg_kwargs)
    state = O.protocol_state_dict(cfg, WEIGHT_SEED)
    text, image = O.protocol_inputs(cfg, world * per_rank, INPUT_SEED, 0.2)
    texts, images = list(text.chunk(world)), list(image.chunk(world))
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, world, cfg_kwargs, state, texts, images, 29611, q))
             for r in range(world)]
    for pr in procs:
        pr.start()
    res = sorted(q.get(timeout=600) for _ in range(world))
    for pr in procs:
        pr.join()
    ranks = []
    for rank, loss, gn, dtemp, norms in res:
        # oracle's restatement of the per-rank contract
        p = {k: v.clone().requires_grad_(True) for k, v in state.items()}
        o_loss = O.clip_forward_sharded(p, texts, images, cfg, rank)
        o_loss.backward()
        assert abs(o_loss.item() - loss) < 5e-6, (name, rank, o_loss.item(), loss)
        for k, v in norms.items():
            og = p[k].grad
            on = 0.0 if og is None else og.double().norm().item()
            assert abs(on - v) <= 2e-4 * max(v, 1e-6) + 1e-9, (name, rank, k, on, v)
        ranks.append(dict(rank=rank, loss=loss, grad_norm=gn, dtemperature=dtemp, grad_norms=norms))
    return dict(case=name, cfg=cfg_kwargs, world=world, per_rank=per_rank, pad_fraction=0.2,
                weight_seed=WEIGHT_SEED, input_seed=INPUT_SEED, ranks=ranks)


def main():
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    x_clip = import_reference()
    for name, (cfgk, batch, padf, drop) in CASES.items():
        out = run_case(x_clip, name, cfgk, batch, padf, drop)
        (HERE / f"{name}.json").write_text(json.dumps(out))
        print(f"{name}: loss={out['loss']:.7f} grad_norm={out['grad_norm']:.6f} dtemp={out['dtemperature']:.7f}")
    for name, cfgk, na_t, na_i in (("tiny_multiview", dict(TINY), 1, 2),
                                   ("tiny_multiview_dcl_extra", dict(TINY, decoupled_contrastive_learning=True,
                                                                     extra_latent_projection=True), 2, 0)):
        out = multiview_case(x_clip, name, cfgk, 5, na_t, na_i)
        (HERE / f"{name}.json").write_text(json.dumps(out))
        print(f"{name}: loss={out['loss']:.7f} grad_norm={out['grad_norm']:.6f} dtemp={out['dtemperature']:.7f}")
    anchors = [survey_anchor(x_clip),
               survey_anchor(x_clip, decoupled_contrastive_learning=True, extra_latent_projection=True),
               survey_anchor(x_clip, use_all_token_embeds=True)]
    (HERE / "survey_anchors.json").write_text(json.dumps(anchors, indent=1))
    for a in anchors:
        print("anchor", a)
    for name, cfgk in (("sharded_plain", dict(TINY)),
                       ("sharded_dcl_extra", dict(TINY, decoupled_contrastive_learning=True,
                                                  extra_latent_projection=True))):
        out = sharded_case(name, cfgk)
        (HERE / f"{name}.json").write_text(json.dumps(out))
        print(name, [(r["loss"], r["grad_norm"], r["dtemperature"]) for r in out["ranks"]])
    (HERE / "random_cases.json").write_text(json.dumps(random_cases(x_clip), separators=(",", ":")))
    (HERE / "reference_signature.json").write_text(json.dumps(reference_signature(x_clip), indent=1))


if __name__ == "__main__":
    main()
