"""Host-side contract of the drop-in modules (no GPU): parameter tree, flags, error behaviour."""
import pytest
import torch

import x_clip_b200
from oracle import clip_oracle as O

TINY = dict(dim_text=256, dim_image=256, dim_latent=256, num_text_tokens=128, text_enc_depth=2,
            text_seq_len=16, text_heads=4, visual_enc_depth=2, visual_heads=4,
            visual_image_size=64, visual_patch_size=16)


def test_state_dict_matches_reference_names_and_shapes():
    clip = x_clip_b200.CLIP(**TINY)
    want = O.param_shapes(O.ClipConfig(**TINY))
    got = {k: tuple(v.shape) for k, v in clip.state_dict().items()}
    assert got == want
    clip.load_state_dict(O.protocol_state_dict(O.ClipConfig(**TINY), 7), strict=True)


def test_readme_config_parameter_count():
    clip = x_clip_b200.CLIP(dim_text=512, dim_image=512, dim_latent=512, num_text_tokens=10000,
                            text_enc_depth=6, text_seq_len=256, text_heads=8, visual_enc_depth=6,
                            visual_image_size=256, visual_patch_size=32, visual_heads=8)
    n = sum(p.numel() for p in clip.parameters())
    assert abs(n - 58.5e6) < 0.1e6          # SURVEY.md 6: 58.5 M parameters
    assert clip.temperature.item() == 1.0
    assert torch.equal(clip.to_text_latent.weight, clip.to_text_latent_extra.weight)


def test_unknown_kwargs_swallowed_and_asserts_kept():
    x_clip_b200.CLIP(**TINY, some_future_flag=3)
    with pytest.raises(AssertionError):
        x_clip_b200.CLIP(**TINY, visual_has_cls_token=False, text_has_cls_token=False)
    with pytest.raises(AssertionError):
        x_clip_b200.CLIP(**TINY, text_causal_mask=True)          # eos id missing (x_clip.py:480)


@pytest.mark.parametrize("kw", [dict(text_dim_head=32), dict(dim_text=320), dict(sim_reg_loss_weight=0.1),
                                dict(downsample_image_embeds=True, use_all_token_embeds=True),
                                # rotary + causal is broken in the reference itself (x_clip.py:328)
                                dict(text_causal_mask=True, text_eos_id=1, text_rotary_pos_emb=True),
                                # the causal kernels cover <= 128 tokens
                                dict(text_causal_mask=True, text_eos_id=1, text_seq_len=256)])
def test_unsupported_flags_raise_at_construction(kw):
    with pytest.raises(x_clip_b200.Unsupported):
        x_clip_b200.CLIP(**{**TINY, **kw})


def test_aux_loss_heads_construct_on_the_fast_encoders():
    """use_mlm / use_visual_ssl wrap the SAME encoder modules (reference x_clip.py:516-552)."""
    clip = x_clip_b200.CLIP(**TINY, use_mlm=True, use_visual_ssl=True)
    assert clip.mlm.transformer is clip.text_transformer
    assert clip.text_ssl_loss_weight == 0.05 and clip.image_ssl_loss_weight == 0.05


def test_rotary_and_causal_towers_mirror_the_reference_parameter_tree():
    from oracle import clip_oracle as O
    for kw in (dict(text_rotary_pos_emb=True), dict(text_causal_mask=True, text_eos_id=5)):
        clip = x_clip_b200.CLIP(**{**TINY, **kw})
        want = set(O.param_shapes(O.ClipConfig(**{**TINY, **kw})).keys())
        got = set(clip.state_dict().keys())
        assert got - want <= {"text_transformer.rotary_pos_emb.inv_freq"} and not (want - got), (kw, got ^ want)


def test_cpu_inputs_fail_loudly():
    clip = x_clip_b200.CLIP(**TINY)
    text = torch.randint(0, 128, (2, 16))
    img = torch.randn(2, 3, 64, 64)
    with pytest.raises((x_clip_b200.Unsupported, RuntimeError)):
        clip(text, img, return_loss=True)


def test_pluggable_encoders_are_adopted():
    class Enc(torch.nn.Module):
        def forward(self, *a):
            raise RuntimeError("not called here")
    t, i = Enc(), Enc()
    clip = x_clip_b200.CLIP(**TINY, text_encoder=t, image_encoder=i)
    assert clip.text_transformer is t and clip.visual_transformer is i


def test_patch_dropout_matches_reference_recipe():
    pd = x_clip_b200.clip.PatchDropout(0.5)
    pd.train()
    x = torch.randn(3, 16, 8)
    torch.manual_seed(5)
    out = pd(x)
    torch.manual_seed(5)
    idx = torch.randn(3, 16).topk(8, dim=-1).indices          # x_clip.py:148-149
    assert torch.equal(out, x[torch.arange(3)[:, None], idx])
    pd.eval()
    assert pd(x) is x


def test_constructor_and_forward_signatures_match_the_reference():
    """Drop-in surface (SURVEY 8b): same keyword names and defaults as x_clip.CLIP.__init__ /
    forward (x_clip/x_clip.py:413-456, 597-609), as recorded from the reference in
    tests/golden/reference_signature.json."""
    import inspect
    import json
    from pathlib import Path
    import x_clip_b200

    def params(fn):
        return {k: v.default for k, v in inspect.signature(fn).parameters.items()
                if k not in ("self", "kwargs")}

    def recorded(entries):
        return {e["name"]: e.get("default", inspect.Parameter.empty) for e in entries}

    sig = json.loads((Path(__file__).parent / "golden" / "reference_signature.json").read_text())
    ref_init, our_init = recorded(sig["init"]), params(x_clip_b200.CLIP.__init__)
    missing = [k for k in ref_init if k not in our_init]
    assert not missing, f"constructor keywords of the reference missing here: {missing}"
    for k, v in ref_init.items():
        assert our_init[k] == v or (v is inspect.Parameter.empty) == (our_init[k] is inspect.Parameter.empty), \
            f"default of {k}: reference {v!r}, here {our_init[k]!r}"
        if v is not inspect.Parameter.empty:
            assert our_init[k] == v, f"default of {k}: reference {v!r}, here {our_init[k]!r}"
    extra = sorted(set(our_init) - set(ref_init))
    assert extra == ["microbatch", "microbatch_retain"], f"unexpected extra constructor keywords: {extra}"
    ref_fwd, our_fwd = recorded(sig["forward"]), params(x_clip_b200.CLIP.forward)
    assert list(ref_fwd) == list(our_fwd), (list(ref_fwd), list(our_fwd))
    assert ref_fwd == our_fwd
