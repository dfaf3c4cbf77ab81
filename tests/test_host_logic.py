"""Host-side logic that needs no GPU: weight packing, concat-slot bookkeeping, schedule coefficients, ordering."""
import math

import numpy as np
import pytest
import torch

from oracle import edlora_ref as er
from oracle import inject
from oracle import unet as ou


def test_cross_attention_names_match_reference_order():
    from mos_b200.engine import cross_attention_names
    with torch.device('meta'):
        u = ou.UNet2DConditionModel()
    assert cross_attention_names() == er.cross_attention_layer_order(u)
    with torch.device('meta'):
        t = ou.UNet2DConditionModel(ou.TINY)
    assert cross_attention_names(ou.TINY['block_out_channels'], 1) == er.cross_attention_layer_order(t)


def test_engine_packing_on_cpu():
    from mos_b200.engine import UNetEngine
    u = ou.build_unet(0, ou.TINY)
    lora = inject.random_lora_state(u, seed=10)
    sd = u.state_dict()
    eng = UNetEngine(sd, 2, 16, 16, lora=lora, lora_alpha=0.5, device='cpu', block_out=ou.TINY['block_out_channels'],
                     layers=1)
    tb = 'down_blocks.0.attentions.0.transformer_blocks.0'
    ent = eng.w[tb + '.attn1.qkv']
    assert ent['W'].shape == (960, 320) and ent['lora_down'].shape == (16, 320) and ent['lora_up'].shape == (960, 4)
    assert ent['lora_seg'] == 320
    # fused q|k|v weight rows and LoRA rows land in the right segments
    wq = sd[tb + '.attn1.to_q.weight']
    assert torch.equal(ent['W'][:320].float(), wq.to(eng.ACT).float())
    dv = lora[tb + '.attn1.to_v.lora_down.weight']
    assert torch.equal(ent['lora_down'][8:12].float(), dv.to(eng.ACT).float())
    assert torch.all(ent['lora_down'][12:] == 0)
    uk = lora[tb + '.attn1.to_k.lora_up.weight']
    assert torch.allclose(ent['lora_up'][320:640], uk * 0.5)
    # GEGLU interleave: tile t = [a rows 80t.. | gate rows 1280+80t..]
    ff = eng.w[tb + '.ff1']
    w = sd[tb + '.ff.net.0.proj.weight']
    assert torch.equal(ff['W'][0:80].float(), w[0:80].to(eng.ACT).float())
    assert torch.equal(ff['W'][80:160].float(), w[1280:1360].to(eng.ACT).float())
    assert torch.equal(ff['W'][160:240].float(), w[80:160].to(eng.ACT).float())
    # conv weights are tap-major [Cout, (kh, kw, cin)]
    c1 = eng.w['down_blocks.0.resnets.0.conv1']['W']
    wc = sd['down_blocks.0.resnets.0.conv1.weight']
    assert torch.equal(c1[:, 320:640].float(), wc[:, :, 0, 1].to(eng.ACT).float())
    # merged mode == W + alpha * up @ down (convert_edlora_to_diffusers.py:67-73)
    eng_m = UNetEngine(sd, 2, 16, 16, lora=lora, lora_alpha=0.5, merge_lora=True, device='cpu',
                       block_out=ou.TINY['block_out_channels'], layers=1)
    em = eng_m.w[tb + '.attn2.q']
    assert 'lora_down' not in em
    ref = er.merge_lora_weight(sd[tb + '.attn2.to_q.weight'], lora[tb + '.attn2.to_q.lora_down.weight'],
                               lora[tb + '.attn2.to_q.lora_up.weight'], 0.5)
    assert torch.equal(em['W'].float(), ref.to(eng.ACT).float())


def test_concat_slots_cover_the_unet_skip_wiring():
    from mos_b200.engine import UNetEngine
    with torch.device('meta'):
        u = ou.UNet2DConditionModel()
    sd = {k: torch.zeros(v.shape) for k, v in u.state_dict().items()}
    eng = UNetEngine(sd, 2, 8, 8, device='cpu')
    assert eng.skip_ch == [320, 320, 320, 320, 640, 640, 640, 1280, 1280, 1280, 1280, 1280]
    assert [a + b for a, b in eng.cat_ch] == [2560, 2560, 2560, 2560, 2560, 1920, 1920, 1280, 960, 960, 640, 640]
    # resnet input widths of the up path, as the skeleton defines them
    want = [u.up_blocks[i].resnets[j].conv1.in_channels for i in range(4) for j in range(3)]
    assert [a + b for a, b in eng.cat_ch] == want
    rows = [c.shape[0] for c in eng.cat]
    assert rows == [2 * 1] * 3 + [2 * 4] * 3 + [2 * 16] * 3 + [2 * 64] * 3
    assert eng.temb_total == sum(u.get_submodule(n).time_emb_proj.out_features for n in eng._resnet_names())


def test_product_scheduler_matches_oracle():
    from mos_b200.scheduler import DPMSolverPP2M
    from oracle.schedulers import DPMSolverMultistepScheduler
    for n in (10, 20, 30, 50):
        a, b = DPMSolverPP2M(), DPMSolverMultistepScheduler()
        ts = a.set_timesteps(n)
        b.set_timesteps(n)
        assert np.array_equal(ts, b.timesteps.numpy())       # integer timesteps: bit exact
        for i in range(len(ts)):
            assert np.allclose(a.coefficients(i), b.coefficients(i), rtol=2e-5, atol=1e-6)


def test_missing_library_fails_loudly(monkeypatch, tmp_path):
    from mos_b200 import _lib
    monkeypatch.setattr(_lib, '_lib', None)
    monkeypatch.setattr(_lib, 'LIB_PATH', str(tmp_path / 'nope.so'))
    with pytest.raises(_lib.MosError):
        _lib.lib()


def test_product_bind_concept_prompt_and_boxes_match_reference_golden():
    """bit-exact string / integer outputs of the drop-in functions vs the reference-generated golden"""
    import os
    from mixofshow.pipelines.pipeline_edlora import bind_concept_prompt
    from mixofshow.pipelines.pipeline_regionally_t2iadapter import region_box_indices
    G = torch.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_golden.pt'),
                   weights_only=False)
    g = G['bind_concept_prompt']
    assert bind_concept_prompt(g['prompts'], g['cfg']) == g['out']
    assert bind_concept_prompt(g['prompts'][0], g['cfg']) == g['out_single']
    r = G['region']
    for (H, W, ds, tag), idx in r['box_index_kat'].items():
        boxes = r['boxes'] if tag == 'abut' else r['boxes_overlap']
        assert [region_box_indices(b, H // ds, W // ds) for b in boxes] == [tuple(i) for i in idx]


def test_train_loop_host_logic():
    """train_edlora.py:73-75 total_iter and the linear schedule (diffusers get_scheduler('linear', warmup 0))."""
    import pytest
    import train_edlora as te
    assert te.total_iterations(1000, 4, 1, 1) == 250.0
    assert te.total_iterations(100, 8, 8, 1) == 100 / 64            # fractional, as the reference computes it
    assert te.linear_lr(1e-4, 0, 250) == 1e-4
    assert te.linear_lr(1e-4, 125, 250) == pytest.approx(5e-5)
    assert te.linear_lr(1e-4, 250, 250) == 0.0 and te.linear_lr(1e-4, 300, 250) == 0.0
    from mixofshow.pipelines.trainer_edlora import UNetLoRATrainer
    cfg = {'text_embedding': {'enable_tuning': True, 'lr': 1e-3}, 'text_encoder': {'enable_tuning': False},
           'unet': {'enable_tuning': True, 'lr': 1e-4, 'lora_cfg': {'rank': 4, 'alpha': 1.0, 'where': 'Attention'}}}
    with pytest.raises(NotImplementedError):
        UNetLoRATrainer({}, 2, finetune_cfg=cfg)
    with pytest.raises(ValueError):
        UNetLoRATrainer({}, 2, finetune_cfg=None)


def test_clip_engine_packing_on_cpu():
    """CLIPTextEngine pads 64-dim heads to 80 and 768 / 3072 columns to 800 / 3200 without changing the arithmetic."""
    from transformers import CLIPTextConfig, CLIPTextModel
    from mos_b200.clip_engine import CLIPTextEngine
    cfg = CLIPTextConfig(vocab_size=300, hidden_size=768, intermediate_size=3072, num_hidden_layers=1,
                         num_attention_heads=12, max_position_embeddings=77)
    torch.manual_seed(0)
    m = CLIPTextModel(cfg).eval()
    sd = m.state_dict()
    lora = inject.random_lora_state(m, seed=3, where='CLIPAttention')
    assert len(lora) == 8                                   # q, k, v, out_proj x (down, up)
    eng = CLIPTextEngine(sd, 2, lora=lora, lora_alpha=0.5, device='cpu')
    e = eng.w[0]
    assert e['qkv']['W'].shape == (2880, 768) and e['out']['W'].shape == (800, 960)
    assert e['fc1']['W'].shape == (3200, 768) and e['fc2']['W'].shape == (800, 3200)
    L = 'text_model.encoder.layers.0.'
    x = torch.randn(6, 768)
    for s, pj in enumerate(('q_proj', 'k_proj', 'v_proj')):
        W, b = sd[L + f'self_attn.{pj}.weight'], sd[L + f'self_attn.{pj}.bias']
        ref = x @ W.T + b + 0.5 * (x @ lora[L + f'self_attn.{pj}.lora_down.weight'].T) @ lora[L + f'self_attn.{pj}.lora_up.weight'].T
        Wp = e['qkv']['W'][960 * s:960 * (s + 1)].float()
        t = x @ e['qkv']['lora_down'][4 * s:4 * s + 4].float().T
        got = (x @ Wp.T + e['qkv']['bias'][960 * s:960 * (s + 1)] + t @ e['qkv']['lora_up'][960 * s:960 * (s + 1)].T)
        got = got.view(6, 12, 80)
        assert got[:, :, 64:].abs().max().item() == 0.0     # head pads carry exact zeros
        assert torch.allclose(got[:, :, :64].reshape(6, 768), ref, atol=0.05, rtol=0.05)
    # out_proj reads the padded head layout: zero weight columns at the pads, zero rows 768..799
    a = torch.zeros(6, 12, 80)
    a[:, :, :64] = torch.randn(6, 12, 64)
    ref = a[:, :, :64].reshape(6, 768) @ sd[L + 'self_attn.out_proj.weight'].T + sd[L + 'self_attn.out_proj.bias']
    got = a.reshape(6, 960) @ e['out']['W'].float().T + e['out']['bias']
    assert got[:, 768:].abs().max().item() == 0.0
    assert torch.allclose(got[:, :768], ref, atol=0.05, rtol=0.05)
    # merged mode folds alpha * up @ down into the weight (gradient_fusion.py:99-143)
    em = CLIPTextEngine(sd, 2, lora=lora, lora_alpha=0.5, merge_lora=True, device='cpu').w[0]
    assert 'lora_down' not in em['qkv']
    Wq = sd[L + 'self_attn.q_proj.weight'] + 0.5 * lora[L + 'self_attn.q_proj.lora_up.weight'] @ lora[L + 'self_attn.q_proj.lora_down.weight']
    assert torch.equal(em['qkv']['W'][:960].view(12, 80, 768)[:, :64].reshape(768, 768).float(), Wq.to(torch.bfloat16).float())


def test_regional_script_prepare_text_matches_reference_golden():
    """regionally_controlable_sampling.py:67-94 (the box fractions feed the bit-exact region masks)."""
    import os
    import regionally_controlable_sampling as rcs
    G = torch.load(os.path.join(os.path.dirname(__file__), 'golden', 'reference_golden.pt'))['prepare_text']
    out = rcs.prepare_text('a context prompt', G['prompt_rewrite'], G['height'], G['width'])
    assert out == G['out']                                   # strings and float64 fractions, exactly
    assert rcs.prepare_text('p', '[a]-*-[b]-*-[]', 512, 512) == ('p', [('a', 'b', [0, 0, 1, 1])])
    assert rcs.prepare_text('p', '', 512, 512) == ('p', [])
    a = rcs.parse_args(['--pretrained_model', 'x', '--prompt_rewrite', 'r', '--seed', '3'])
    assert a.seed == 3 and a.height == 768 and a.width == 1536 and a.keypose_adaptor_weight == 1.0


def test_latent_dataset_and_yml_options(tmp_path):
    """`train_edlora.py -opt <yml>` host side: LatentDataset (replace_mapping, dataset_enlarge_ratio, per-rank sharding of one
    shared permutation, drop_last) and the options of a shipped reference yml (`!!float` values, models block = EDLoRATrainer
    keyword arguments)."""
    import inspect
    import os

    import train_edlora as te
    from mixofshow.pipelines.trainer_edlora import EDLoRATrainer
    blob = {'latents': torch.arange(6 * 4 * 2 * 2, dtype=torch.float32).view(6, 4, 2, 2), 'prompts': [f'a <TOK> {i}' for i in range(6)],
            'masks': torch.ones(6, 1, 2, 2)}
    path = str(tmp_path / 'set.pt')
    torch.save(blob, path)
    ds = te.LatentDataset({'path': path, 'replace_mapping': {'<TOK>': '<c1> <c2>'}, 'dataset_enlarge_ratio': 5})
    assert len(ds) == 30 and ds.prompts[3] == 'a <c1> <c2> 3'
    it0, it1 = ds.batches(2, rank=0, world=2, seed=1), ds.batches(2, rank=1, world=2, seed=1)
    seen = []
    for _ in range(7):                       # 30 // 4 = 7 steps per epoch, disjoint shards of one permutation
        b0, b1 = next(it0), next(it1)
        assert b0['images'].shape == (2, 4, 2, 2) and len(b0['prompts']) == 2 and b0['masks'].shape == (2, 1, 2, 2)
        seen += [int(x[0, 0, 0]) // 16 for x in list(b0['images']) + list(b1['images'])]
    assert len(seen) == 28 and max(seen.count(i) for i in range(6)) <= 5
    # the parsed options of the reference's 8101_EDLoRA_potter_Cmix_B4_Repeat500.yml (tests/golden/make_golden.py --crosscheck)
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_crosscheck.pt')
    opt = torch.load(gold, weights_only=False)['train_options']
    assert opt['models']['finetune_cfg']['text_embedding']['lr'] == 1e-3 and opt['train']['emb_norm_threshold'] == 0.55
    params = inspect.signature(EDLoRATrainer.__init__).parameters
    assert all(k in params for k in opt['models']), 'EDLoRATrainer(**opt["models"]) must accept every key of the yml'
