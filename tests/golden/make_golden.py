"""Generate tests/golden/reference_golden.pt by executing the REFERENCE's own Python (read-only, in place, under the
import shims of oracle/ref_shims.py) on seeded synthetic inputs.  Run where a checkout of the reference exists (its
directory in MOS_REFERENCE_ROOT):   python tests/golden/make_golden.py   (--crosscheck: tests/golden/reference_crosscheck.pt)
The reference ships no tests or golden vectors (SURVEY.md §4); these fixtures are what pins the oracle.
Third-party diffusers is absent, so the skeleton the reference code runs on is oracle/unet.py (see its header).
"""
import math
import os
import sys

import torch
import torch.nn as nn

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import ref_shims  # noqa: E402
from oracle import unet as ou  # noqa: E402

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'reference_golden.pt')
CROSS = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'reference_crosscheck.pt')


def gen(seed):
    return torch.Generator().manual_seed(seed)


def q16(t):
    """Round a (large) input to bf16-representable values so it can be stored as bf16 losslessly."""
    return t.to(torch.bfloat16).float()


def pack16(obj):
    """Store bf16-representable fp32 tensors as bf16 (tests call .float() on load)."""
    if torch.is_tensor(obj):
        return obj.to(torch.bfloat16) if (obj.dtype == torch.float32 and torch.equal(obj.to(torch.bfloat16).float(), obj)
                                          and obj.numel() > 4096) else obj
    if isinstance(obj, dict):
        return {k: pack16(v) for k, v in obj.items()}
    if isinstance(obj, list):
        return [pack16(v) for v in obj]
    if isinstance(obj, tuple):
        return tuple(pack16(v) for v in obj)
    return obj


from oracle.train_ref import attn_reg_inputs  # noqa: E402


def golden_attn_reg():
    """T2: EDLoRATrainer.cal_attn_reg (trainer_edlora.py:263-313) executed unbound, + autograd gradients."""
    import types
    tr = ref_shims.load_reference_module('mixofshow/pipelines/trainer_edlora.py')
    out = {}
    for full in (True, False):
        maps, masks, ids, pos = attn_reg_inputs()
        for lst in maps.values():
            for m in lst:
                m.requires_grad_(True)
        me = types.SimpleNamespace(get_all_concept_token_ids=lambda: [49408 + i for i in range(32)],
                                   reg_full_identity=full, attn_reg_weight=0.01)
        loss = tr.EDLoRATrainer.cal_attn_reg(me, maps, masks, ids)
        loss.backward()
        grads = {}
        for place, lst in maps.items():
            for m in lst:
                r = int(math.sqrt(m.shape[1]))
                g = m.grad.view(2, 8, r * r, 77)
                gc = torch.stack([g[i][:, :, pos[i]] for i in range(2)])            # [b, 8, N, 2]
                assert torch.equal(gc[:, :1].expand_as(gc), gc)                     # identical over heads
                other = m.grad.clone().view(2, 8, r * r, 77)
                for i in range(2):
                    other[i][:, :, pos[i]] = 0
                assert other.abs().max().item() == 0                                # only the two concept columns
                if r in grads:
                    assert torch.equal(grads[r], gc[:, 0])                          # identical over a group's layers
                grads[r] = gc[:, 0].clone()
        out['full' if full else 'masked'] = dict(loss=loss.detach(), grads=grads)
    out['pos'] = pos
    # a mask without zeros at the coarsest resolution makes the reference return NaN (skipped by the caller, :257)
    maps, masks, ids, pos = attn_reg_inputs()
    masks[:] = 1.0
    me = types.SimpleNamespace(get_all_concept_token_ids=lambda: [49408 + i for i in range(32)],
                               reg_full_identity=True, attn_reg_weight=0.01)
    out['nan_when_mask_full'] = bool(torch.isnan(tr.EDLoRATrainer.cal_attn_reg(me, maps, masks, ids)))
    return out


def crosscheck():
    """What the reference's own modules return on the cases of tests/test_oracle_vs_reference.py and of the mirror check in
    tests/test_checkpoint_formats.py, and the parsed options of a shipped training yml -> reference_crosscheck.pt."""
    import yaml
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import test_checkpoint_formats as tc
    import test_oracle_vs_reference as tv
    ed = ref_shims.load_reference_module('mixofshow/models/edlora.py')
    pe = ref_shims.load_reference_module('mixofshow/pipelines/pipeline_edlora.py')
    gf = ref_shims.load_reference_module('gradient_fusion.py')
    cv = ref_shims.load_reference_module('mixofshow/utils/convert_edlora_to_diffusers.py')
    G = {}

    unet, lora, x, ehs = tv.installer_case()
    ed.revise_edlora_unet_attention_forward(unet)
    mods = dict(unet.named_modules())
    keep = []
    for k in lora:
        if k.endswith('.lora_down.weight'):
            n = k[:-len('.lora_down.weight')]
            layer = ed.LoRALinearLayer(n, mods[n], rank=4, alpha=tv.LORA_ALPHA)
            layer.lora_down.weight.data = lora[k].clone()
            layer.lora_up.weight.data = lora[n + '.lora_up.weight'].clone()
            keep.append(layer)
    with torch.no_grad():
        G['installer'] = dict(out=unet(x, torch.tensor([500, 500]), ehs).sample, n_lora=len(keep))

    G['bind_concept_prompt'] = pe.bind_concept_prompt(tv.BIND_PROMPTS, tv.BIND_CFG)
    K, V, W0 = tv.quasi_newton_case()
    G['quasi_newton'] = dict(K=K, V=V, W0=W0, W=gf.update_quasi_newton(K, V, W0.clone(), tv.QN_ITERS, 'cpu').detach())

    sds, ckpt = tc.mirror_case()
    merge = {}
    for model_type, sd in sds.items():
        merged = cv.merge_lora_into_weight(sd, ckpt[model_type], model_type=model_type, alpha=tc.MERGE_ALPHA)
        merge[model_type] = tc.merge_samples(sd, merged)
    G['convert'] = dict(merge=merge, load_new_concept=tc.load_concept(cv.load_new_concept, ckpt['new_concept_embedding']))

    with open(os.path.join(ref_shims.REFERENCE_ROOT, 'options/train/EDLoRA/real/8101_EDLoRA_potter_Cmix_B4_Repeat500.yml')) as f:
        opt = yaml.safe_load(f)
    G['train_options'] = dict(models=opt['models'], train=dict(emb_norm_threshold=opt['train']['emb_norm_threshold']))
    torch.save(G, CROSS)
    print('wrote', CROSS, os.path.getsize(CROSS) / 1e6, 'MB')


def main():
    assert ref_shims.reference_available(), 'needs /root/reference'
    if '--crosscheck' in sys.argv:
        crosscheck()
        return
    if '--only-attn-reg' in sys.argv:
        G = torch.load(OUT, weights_only=False)
        G['attn_reg'] = golden_attn_reg()
        torch.save(G, OUT)
        print('updated attn_reg in', OUT)
        return
    ed = ref_shims.load_reference_module('mixofshow/models/edlora.py')
    reg = ref_shims.load_reference_module('mixofshow/pipelines/pipeline_regionally_t2iadapter.py')
    gf = ref_shims.load_reference_module('gradient_fusion.py')
    pe = ref_shims.load_reference_module('mixofshow/pipelines/pipeline_edlora.py')
    cv = ref_shims.load_reference_module('mixofshow/utils/convert_edlora_to_diffusers.py')
    rcs = ref_shims.load_reference_module('regionally_controlable_sampling.py')
    G = {}

    # ---- P1 LoRALinearLayer (edlora.py:221-246) on Linear and 1x1 Conv2d
    torch.manual_seed(0)
    lin = nn.Linear(64, 48)
    x = torch.randn(3, 10, 64, generator=gen(1))
    l = ed.LoRALinearLayer('t', lin, rank=4, alpha=0.7)
    l.lora_up.weight.data = torch.randn(48, 4, generator=gen(2)) * 0.1
    G['lora_linear'] = dict(x=x, w=lin.weight.data.clone(), b=lin.bias.data.clone(),
                            down=l.lora_down.weight.data.clone(), up=l.lora_up.weight.data.clone(), alpha=0.7,
                            y=lin(x).detach())
    conv = nn.Conv2d(32, 24, 1)
    xc = torch.randn(2, 32, 5, 6, generator=gen(3))
    lc = ed.LoRALinearLayer('c', conv, rank=4, alpha=1.3)
    lc.lora_up.weight.data = torch.randn(24, 4, 1, 1, generator=gen(4)) * 0.1
    G['lora_conv'] = dict(x=xc, w=conv.weight.data.clone(), b=conv.bias.data.clone(),
                          down=lc.lora_down.weight.data.clone(), up=lc.lora_up.weight.data.clone(), alpha=1.3,
                          y=conv(xc).detach())

    # ---- P2/P3 processors on the Attention surface (edlora.py:22-173)
    torch.manual_seed(5)
    attn = ou.Attention(320, 128, heads=8, dim_head=40)     # small cross dim keeps the fixture small
    hs = torch.randn(2, 64, 320, generator=gen(6))
    ehs = q16(torch.randn(2, 16, 77, 128, generator=gen(7))[:, :8].contiguous())   # idx 5 of 8 stored layers
    with torch.no_grad():
        out_plain = ed.EDLoRA_AttnProcessor(5)(attn, hs, encoder_hidden_states=ehs)
        seen = {}

        class Ctl:
            def __call__(self, probs, is_cross, place):
                seen['probs'], seen['is_cross'], seen['place'] = probs.clone(), is_cross, place
                return probs
        out_ctl = ed.EDLoRA_Control_AttnProcessor(5, 'down', Ctl())(attn, hs, encoder_hidden_states=ehs)
    G['attn_proc'] = dict(state={k: v.clone() for k, v in attn.state_dict().items()}, hs=hs, ehs=ehs, idx=5,
                          out=out_plain, out_ctl=out_ctl, probs=seen['probs'], is_cross=seen['is_cross'],
                          place=seen['place'])

    # ---- P4 installer ordering (edlora.py:176-218) on the tiny and the full topology (ints / names: bit exact)
    for tag, cfg in (('tiny', ou.TINY), ('sd15', None)):
        torch.manual_seed(0)
        with torch.device('meta'):
            u = ou.UNet2DConditionModel(cfg)
        ed.revise_edlora_unet_attention_forward(u)
        order = {}
        for name, m in u.named_modules():
            if m.__class__.__name__ == 'Attention' and name.endswith('attn2'):
                order[name] = m.processor.cross_attention_idx
        G[f'xattn_order_{tag}'] = order

    # ---- P5 bind_concept_prompt (pipeline_edlora.py:18-29)
    cfgc = {'<potter1>': {'concept_token_names': [f'<new{i}>' for i in range(16)]},
            '<potter2>': {'concept_token_names': [f'<new{16 + i}>' for i in range(16)]}}
    prompts = ['a photo of <potter1> <potter2> in the snow', 'a <potter1>, by <potter2> <potter1>']
    G['bind_concept_prompt'] = dict(cfg=cfgc, prompts=prompts, out=pe.bind_concept_prompt(prompts, cfgc),
                                    out_single=pe.bind_concept_prompt(prompts[0], cfgc))

    # ---- R1 region_rewrite + full regional processor (regional :27-145); boxes from regionally_sample.sh:66-74
    boxes_px = [[4, 7, 1024, 490], [14, 490, 1024, 920], [2, 1302, 1024, 1992]]   # [h0,w0,h1,w1] on 1024x2048
    Hpx, Wpx = 1024, 2048
    boxes = [[b[0] / Hpx, b[1] / Wpx, b[2] / Hpx, b[3] / Wpx] for b in boxes_px]
    boxes_overlap = [boxes[0], [14 / Hpx, 440 / Wpx, 1024 / Hpx, 920 / Wpx], boxes[2]]
    proc = reg.RegionT2I_AttnProcessor(3)
    torch.manual_seed(8)
    attn_r = ou.Attention(320, 128, heads=8, dim_head=40)
    fh, fw = 12, 24
    hs_r = torch.randn(2, fh * fw, 320, generator=gen(9))
    ehs_r = q16(torch.randn(2, 16, 77, 128, generator=gen(10))[:, :4].contiguous())   # idx 3 of 4 stored layers
    region_embs = [q16(torch.randn(2, 4, 77, 128, generator=gen(11))), q16(torch.randn(2, 77, 128, generator=gen(12))),
                   q16(torch.randn(2, 77, 128, generator=gen(13)))]                       # 4-D and 3-D forms (:120-126)
    reg_out = {}
    for tag, bx in (('abut', boxes), ('overlap', boxes_overlap)):
        rl = [(region_embs[i], bx[i]) for i in range(3)]
        with torch.no_grad():
            reg_out[tag] = proc(attn_r, hs_r, encoder_hidden_states=ehs_r, region_list=rl, height=96, width=192)
    torch.manual_seed(18)
    attn_s = ou.Attention(320, None, heads=8, dim_head=40)
    with torch.no_grad():
        self_out = proc(attn_s, hs_r, encoder_hidden_states=None, region_list=[], height=96, width=192)
    # integer KATs of get_region_mask at the four feature resolutions of 768x1536 and of 1024x2048
    kat = {}
    for (H_, W_) in ((768, 1536), (1024, 2048)):
        for ds in (8, 16, 32, 64):
            fh_, fw_ = H_ // ds, W_ // ds
            for tag, bx in (('abut', boxes), ('overlap', boxes_overlap)):
                m = torch.zeros(fh_, fw_)
                idx = []
                for b in bx:
                    sh, sw, eh, ew = math.ceil(b[0] * fh_), math.ceil(b[1] * fw_), math.floor(b[2] * fh_), \
                        math.floor(b[3] * fw_)
                    idx.append((sh, sw, eh, ew))
                kat[(H_, W_, ds, tag)] = idx
    G['region'] = dict(state={k: v.clone() for k, v in attn_r.state_dict().items()}, hs=hs_r, ehs=ehs_r,
                       self_state={k: v.clone() for k, v in attn_s.state_dict().items()},
                       region_embs=region_embs, boxes=boxes, boxes_overlap=boxes_overlap, idx=3, height=96,
                       width=192, out=reg_out, self_out=self_out, box_index_kat=kat)

    # ---- prepare_text (regionally_controlable_sampling.py:67-94)
    pr = ('[a man, in a suit]-*-[ugly, blurry]-*-[4, 7, 1024, 490]|[a woman]-*-[]-*-[14, 490, 1024, 920]')
    try:
        parsed = rcs.prepare_text('a context prompt', pr, 1024, 2048)
        G['prepare_text'] = dict(prompt_rewrite=pr, height=1024, width=2048, out=parsed)
    except Exception as e:  # keep generating the rest; recorded so the test can skip
        G['prepare_text'] = dict(error=repr(e))

    # ---- G1 update_quasi_newton (gradient_fusion.py:38-96), G3 merge (convert_edlora_to_diffusers.py:33-76)
    Kt = torch.randn(30, 64, generator=gen(20))
    W0 = torch.randn(32, 64, generator=gen(21)) * 0.1
    Wt = W0 + torch.randn(32, 64, generator=gen(22)) * 0.05
    Vt = Kt @ Wt.t()
    Wn = gf.update_quasi_newton(Kt, Vt, W0.clone(), 50, 'cpu')
    Kt2 = torch.randn(400, 48, generator=gen(23))
    W02 = torch.randn(40, 48, generator=gen(24)) * 0.1
    Vt2 = Kt2 @ (W02 + torch.randn(40, 48, generator=gen(25)) * 0.05).t() + torch.randn(400, 40, generator=gen(26)) * .01
    Wn2 = gf.update_quasi_newton(Kt2, Vt2, W02.clone(), 50, 'cpu')
    G['quasi_newton'] = dict(K=Kt, V=Vt, W0=W0, Wnew=Wn.detach(), K2=Kt2, V2=Vt2, W02=W02, Wnew2=Wn2.detach())
    sd0 = {'a.to_q.weight': torch.randn(16, 12, generator=gen(30)),
           'b.proj_in.weight': torch.randn(16, 12, 1, 1, generator=gen(31))}
    lsd = {'a.to_q.lora_down.weight': torch.randn(4, 12, generator=gen(32)),
           'a.to_q.lora_up.weight': torch.randn(16, 4, generator=gen(33)),
           'b.proj_in.lora_down.weight': torch.randn(4, 12, 1, 1, generator=gen(34)),
           'b.proj_in.lora_up.weight': torch.randn(16, 4, 1, 1, generator=gen(35))}
    merged = cv.merge_lora_into_weight(sd0, lsd, 'unet', 0.6)
    G['merge_lora'] = dict(sd=sd0, lora=lsd, alpha=0.6, merged=merged)

    # ---- whole tiny UNet: reference processors + reference LoRALinearLayer injection on the skeleton
    from oracle import inject
    u = ou.build_unet(0, ou.TINY)
    ed.revise_edlora_unet_attention_forward(u)
    lora = inject.random_lora_state(u, seed=10)
    mods = dict(u.named_modules())
    keep = []
    for k in lora:
        if k.endswith('.lora_down.weight'):
            name = k[:-len('.lora_down.weight')]
            layer = ed.LoRALinearLayer(name, mods[name], rank=4, alpha=1.0)
            layer.lora_down.weight.data = lora[k].clone()
            layer.lora_up.weight.data = lora[name + '.lora_up.weight'].clone()
            keep.append(layer)
    lat = torch.randn(2, 4, 16, 16, generator=gen(40))
    ehs_u = q16(torch.randn(2, 4, 77, 768, generator=gen(41)))      # the tiny topology has 4 cross-attention layers
    with torch.no_grad():
        y = u(lat, torch.tensor([981, 981]), ehs_u).sample
    G['tiny_unet'] = dict(latents=lat, ehs=ehs_u, t=981, lora_seed=10, unet_seed=0, out=y, n_lora=len(keep))

    # ---- whole tiny UNet through the reference's regional processors + T2I-adapter residuals (regional :88-145,
    #      UNet call at :556-566); 128x256 px -> 16x32 latent
    ur = ou.build_unet(0, ou.TINY)
    reg.revise_regionally_t2iadapter_attention_forward(ur)
    lat_r = torch.randn(2, 4, 16, 32, generator=gen(50))
    ehs_ur = q16(torch.randn(2, 4, 77, 768, generator=gen(51)))
    r_embs = [q16(torch.randn(2, 4, 77, 768, generator=gen(52 + i))) for i in range(3)]
    adapters = [torch.randn(2, 320, 16, 32, generator=gen(60)) * 0.1, torch.randn(2, 640, 8, 16, generator=gen(61)) * 0.1]
    out_r = {}
    for tag, bx in (('abut', boxes), ('overlap', boxes_overlap)):
        rl = [(r_embs[i], bx[i]) for i in range(3)]
        with torch.no_grad():
            out_r[tag] = ur(lat_r, torch.tensor([500, 500]), ehs_ur,
                            cross_attention_kwargs={'region_list': rl, 'height': 128, 'width': 256},
                            down_block_additional_residuals=[a.clone() for a in adapters]).sample
    G['tiny_unet_region'] = dict(latents=lat_r, ehs=ehs_ur, region_embs=r_embs, adapters=adapters, t=500,
                                 height=128, width=256, boxes=boxes, boxes_overlap=boxes_overlap, out=out_r,
                                 unet_seed=0)

    G['attn_reg'] = golden_attn_reg()
    torch.save(pack16(G), OUT)
    print('wrote', OUT, os.path.getsize(OUT) / 1e6, 'MB')


if __name__ == '__main__':
    main()
