"""Cross-check: the oracle against results of the reference's own modules.  tests/golden/make_golden.py --crosscheck executes
those modules in place on the cases below and stores what they returned in tests/golden/reference_crosscheck.pt, so the
comparison runs without the reference."""
import os

import pytest
import torch

from oracle import edlora_ref as er
from oracle import inject
from oracle import unet as ou

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_crosscheck.pt')


@pytest.fixture(scope='module')
def G():
    return torch.load(GOLD, weights_only=False)


def installer_case():
    """Tiny UNet (seed 3), its rank-4 ED-LoRA (seed 4) and seeded latents / layer-wise embeddings."""
    unet = ou.build_unet(3, ou.TINY)
    lora = inject.random_lora_state(unet, seed=4)
    x = torch.randn(2, 4, 16, 16, generator=torch.Generator().manual_seed(5))
    ehs = torch.randn(2, 4, 77, 768, generator=torch.Generator().manual_seed(6))
    return unet, lora, x, ehs


def quasi_newton_case():
    K = torch.randn(18, 32, generator=torch.Generator().manual_seed(1))
    W0 = torch.randn(24, 32, generator=torch.Generator().manual_seed(2)) * 0.1
    V = K @ (W0 + 0.05 * torch.randn(24, 32, generator=torch.Generator().manual_seed(3))).t()
    return K, V, W0


BIND_CFG = {'<a>': {'concept_token_names': [f'<n{i}>' for i in range(16)]}}
BIND_PROMPTS = ['x <a> y', '<a><a>']
LORA_ALPHA = 0.8
QN_ITERS = 20


def test_reference_installer_and_lora_match_oracle(G):
    g = G['installer']
    unet, lora, x, ehs = installer_case()
    inject.install_edlora_processors(unet)
    assert inject.inject_lora(unet, lora, LORA_ALPHA) == g['n_lora']
    with torch.no_grad():
        y = unet(x, torch.tensor([500, 500]), ehs).sample
    assert ((y - g['out']).norm() / g['out'].norm()).item() < 1e-5


def test_reference_lora_target_selection_matches_trainer_rule():
    """trainer_edlora.py:121-133: every Linear/Conv2d under a module whose class name is `Attention`."""
    u = ou.build_unet(0, ou.TINY)
    names = inject.lora_target_modules(u, 'Attention')
    assert len(names) == 4 * 2 * 4  # 4 transformer blocks x (attn1, attn2) x (to_q,to_k,to_v,to_out.0)
    with torch.device('meta'):
        full = ou.UNet2DConditionModel()
    assert len(inject.lora_target_modules(full, 'Attention')) == 128


def test_reference_bind_and_quasi_newton(G):
    assert er.bind_concept_prompt(BIND_PROMPTS, BIND_CFG) == G['bind_concept_prompt']
    K, V, W0 = quasi_newton_case()
    g = G['quasi_newton']
    assert torch.equal(K, g['K']) and torch.equal(V, g['V']) and torch.equal(W0, g['W0'])
    W = er.update_quasi_newton(K, V, W0, QN_ITERS)
    assert ((W - g['W']).norm() / g['W'].norm()).item() < 1e-5
