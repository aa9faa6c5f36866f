"""Cross-check of the CPU oracle against the REFERENCE on randomly drawn small configurations.

tests/golden/random_cases.json holds what the reference computed on each drawn configuration
(tests/golden/make_golden.py, `random_cases`).  The configurations sweep what the named fixtures
(test_oracle_golden.py) cannot enumerate: widths, head counts, depths, sequence lengths, batch sizes,
pad fractions, patch dropout and every combination of the loss flags."""
import importlib.util
import json
import random
from pathlib import Path

import pytest
import torch

from oracle import clip_oracle as O

GOLD = Path(__file__).parent / "golden"


def _mg():
    spec = importlib.util.spec_from_file_location("make_golden", GOLD / "make_golden.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _summ_close(t, ref, tol=2e-4):
    d = t.detach().double().flatten()
    assert list(t.shape) == ref["shape"]
    assert abs(d.sum().item() - ref["sum"]) <= tol * max(1.0, ref["abs_sum"])
    assert abs(d.abs().sum().item() - ref["abs_sum"]) <= tol * max(1.0, ref["abs_sum"])
    assert abs((d * d).sum().item() - ref["sq_sum"]) <= tol * max(1.0, ref["sq_sum"])
    assert torch.allclose(d[:8], torch.tensor(ref["head"], dtype=torch.float64), atol=5e-4, rtol=1e-3)


@pytest.mark.parametrize("seed", range(16))
def test_oracle_equals_live_reference_on_random_configuration(seed):
    mg = _mg()
    out = json.loads((GOLD / "random_cases.json").read_text())[seed]
    assert out["case"] == f"random_{seed}"
    cfg_kwargs, batch, pad, drop = mg.draw_random_case(random.Random(1000 + seed))
    assert (cfg_kwargs, batch, pad, drop) == (out["cfg"], out["batch"], out["pad_fraction"], out["patch_dropout"])
    torch.set_num_threads(4)
    cfg = O.ClipConfig(**cfg_kwargs)
    state = O.protocol_state_dict(cfg, out["weight_seed"])
    text, image = O.protocol_inputs(cfg, batch, out["input_seed"], pad)
    keep = None if out["keep"] is None else torch.tensor(out["keep"])
    p = {k: v.clone().requires_grad_(True) for k, v in state.items()}
    loss, parts = O.clip_forward(p, text, image, cfg, keep=keep, return_parts=True)
    loss.backward()
    assert abs(loss.item() - out["loss"]) <= 2e-6 * max(1.0, abs(out["loss"])), (cfg_kwargs, loss.item(), out["loss"])
    assert abs(p["temperature"].grad.item() - out["dtemperature"]) <= 5e-6
    _summ_close(parts["enc_text"], out["enc_text"])
    _summ_close(parts["enc_image"], out["enc_image"])
    _summ_close(parts["text_latents"], out["latents"][0])
    _summ_close(parts["image_latents"], out["latents"][1])
    total = 0.0
    for k, n in out["grad_norms"].items():
        g = p[k].grad
        assert g is not None, (cfg_kwargs, k)
        gn = g.double().norm().item()
        total += gn * gn
        assert abs(gn - n) <= 5e-4 * max(n, 1e-5) + 1e-8, (cfg_kwargs, k)
        # entries, not only the norm: the reference's gradient at its recorded positions
        smp = out["grad_samples"][k]
        err = (g.double().flatten()[smp["idx"]] - torch.tensor(smp["val"], dtype=torch.float64)).norm().item()
        assert err <= 2e-4 * n + 1e-10, (cfg_kwargs, k, err, n)
    assert abs(total ** 0.5 - out["grad_norm"]) <= 1e-4 * out["grad_norm"]
    # parameters the reference leaves without gradient stay without gradient
    for k, v in p.items():
        if k not in out["grad_norms"]:
            assert v.grad is None or v.grad.abs().max().item() == 0.0, k
