"""On-disk / checkpoint plumbing (SURVEY.md 8f rank 3), CPU only: the ED-LoRA delta checkpoint layout
(trainer_edlora.py:358-378, train_edlora.py:168-171) loaded through this repo's `convert_edlora_to_diffusers` mirror into
this repo's containers, cross-checked against what the reference's own file returned (tests/golden/reference_crosscheck.pt)."""
import io
import os

import pytest
import torch

from oracle import inject
from oracle import unet as ou

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_crosscheck.pt')


class FakeTokenizer:
    """the three tokenizer calls load_new_concept makes (convert_edlora_to_diffusers.py:13-15)"""

    def __init__(self, n):
        self.vocab = {f'tok{i}': i for i in range(n)}

    def add_tokens(self, names):
        added = 0
        for n in names:
            if n not in self.vocab:
                self.vocab[n] = len(self.vocab)
                added += 1
        return added

    def convert_tokens_to_ids(self, name):
        return self.vocab[name]

    def __len__(self):
        return len(self.vocab)


def _clip_sd(layers=1, vocab=300):
    from transformers import CLIPTextConfig, CLIPTextModel
    cfg = CLIPTextConfig(vocab_size=vocab, hidden_size=768, intermediate_size=3072, num_hidden_layers=layers,
                         num_attention_heads=12, max_position_embeddings=77)
    torch.manual_seed(0)
    m = CLIPTextModel(cfg).eval()
    return m, {k: v.clone() for k, v in m.state_dict().items()}


def _delta(unet, clip, seed=0):
    g = torch.Generator().manual_seed(seed)
    return {'params': {
        'new_concept_embedding': {'<cat1>': torch.randn(16, 768, generator=g), '<dog2>': torch.randn(16, 768, generator=g)},
        'text_encoder': inject.random_lora_state(clip, seed=seed + 1, where='CLIPAttention'),
        'unet': inject.random_lora_state(unet, seed=seed + 2),
    }}


def test_delta_checkpoint_roundtrip_and_convert_on_b200_containers():
    from types import SimpleNamespace
    from mixofshow.models.clip_b200 import CLIPTextModel
    from mixofshow.models.unet_b200 import UNet2DConditionModel
    from mixofshow.utils.convert_edlora_to_diffusers import convert_edlora
    ref_unet = ou.build_unet(0, ou.TINY)
    clip, clip_sd = _clip_sd()
    ckpt = _delta(ref_unet, clip)
    buf = io.BytesIO()
    torch.save(ckpt, buf)                                    # the `.pth` the reference writes (train_edlora.py:168-171)
    buf.seek(0)
    loaded = torch.load(buf)
    assert set(loaded['params']) == {'new_concept_embedding', 'text_encoder', 'unet'}
    unet = UNet2DConditionModel(block_out_channels=ou.TINY['block_out_channels'],
                                layers_per_block=ou.TINY['layers_per_block'])
    unet.load_state_dict(ref_unet.state_dict())
    pipe = SimpleNamespace(tokenizer=FakeTokenizer(300), text_encoder=CLIPTextModel(clip_sd, device='cpu'), unet=unet)
    w_before = {k: v.clone() for k, v in unet.state_dict().items()}
    pipe, cfg = convert_edlora(pipe, loaded, enable_edlora=True, alpha=0.6)
    # tokens: 16 per concept, ids appended after the original vocabulary, in order
    assert cfg['<cat1>']['concept_token_ids'] == list(range(300, 316))
    assert cfg['<dog2>']['concept_token_names'] == [f'<new{16 + i}>' for i in range(16)]
    table = pipe.text_encoder.get_input_embeddings().weight
    assert table.shape == (332, 768)
    assert torch.equal(table[316:332], loaded['params']['new_concept_embedding']['<dog2>'])
    assert torch.equal(table[:300], clip_sd['text_model.embeddings.token_embedding.weight'])
    # LoRA folded into the UNet / text-encoder weights: W + alpha * up @ down, other tensors untouched
    k = 'down_blocks.0.attentions.0.transformer_blocks.0.attn2.to_k'
    lu = loaded['params']['unet']
    want = w_before[k + '.weight'] + 0.6 * lu[k + '.lora_up.weight'] @ lu[k + '.lora_down.weight']
    assert torch.allclose(pipe.unet.state_dict()[k + '.weight'], want, atol=1e-6)
    assert torch.equal(pipe.unet.state_dict()['conv_in.weight'], w_before['conv_in.weight'])
    q = 'text_model.encoder.layers.0.self_attn.q_proj'
    lt = loaded['params']['text_encoder']
    want = clip_sd[q + '.weight'] + 0.6 * lt[q + '.lora_up.weight'] @ lt[q + '.lora_down.weight']
    assert torch.allclose(pipe.text_encoder.state_dict()[q + '.weight'], want, atol=1e-6)


def test_clip_container_embedding_surface(monkeypatch):
    """Rows written through `.weight.data[...]` (no version counter sees them) must reach the engines: the container
    re-uploads the token table after every hand-out.  The engine is replaced by a recorder (no GPU here)."""
    import mos_b200.clip_engine as ce
    from mixofshow.models.clip_b200 import CLIPTextModel
    calls = []

    class FakeEngine:
        def __init__(self, sd, n, **kw):
            self.n, self.T = n, 77
            calls.append(('build', n, sd['text_model.embeddings.token_embedding.weight'].shape[0]))

        def set_token_embedding(self, table):
            calls.append(('upload', float(table[5, 0]), table.shape[0]))

        def __call__(self, ids):
            return torch.zeros(self.n, 77, 768)

    monkeypatch.setattr(ce, 'CLIPTextEngine', FakeEngine)
    _, sd = _clip_sd()
    te = CLIPTextModel(sd, device='cpu')
    ids = torch.zeros(2, 77, dtype=torch.long)
    assert te(ids)[0].shape == (2, 77, 768)
    te(ids)
    assert calls == [('build', 2, 300)]                       # cached, nothing re-uploaded
    w = te.get_input_embeddings().weight
    w.data[5] = 1.0                                          # in-place row write (trainer_edlora.py:77-82)
    te(ids)
    assert calls[-1] == ('upload', 1.0, 300)
    assert torch.all(te.state_dict()['text_model.embeddings.token_embedding.weight'][5] == 1.0)
    te.resize_token_embeddings(310)
    assert te.get_input_embeddings().weight.shape == (310, 768) and te.config.vocab_size == 310
    te(ids)
    assert calls[-1] == ('build', 2, 310)                     # resize drops the engines
    with pytest.raises(RuntimeError):
        te.load_state_dict({'nope': torch.zeros(1)})


MERGE_ALPHA = 0.7


def mirror_case():
    """Tiny UNet (seed 0) and one-layer CLIP text encoder state dicts, and a seeded delta checkpoint (seed 5)."""
    unet = ou.build_unet(0, ou.TINY)
    clip, clip_sd = _clip_sd()
    return {'unet': unet.state_dict(), 'text_encoder': clip_sd}, _delta(unet, clip, seed=5)['params']


def merge_samples(sd, merged, n=64):
    """The keys of a merged state dict and, for every tensor the merge changed, a fixed seeded sample of its elements."""
    g = torch.Generator().manual_seed(0)
    samples = {}
    for k in sorted(k for k in merged if not torch.equal(merged[k], sd[k])):
        idx = torch.randint(0, merged[k].numel(), (n,), generator=g)
        samples[k] = (idx, merged[k].flatten()[idx].clone())
    return sorted(merged), samples


def load_concept(load_new_concept, embeddings):
    """load_new_concept on the reference's kind of objects (transformers CLIPTextModel + tokenizer stand-in)."""
    from types import SimpleNamespace
    from transformers import CLIPTextConfig, CLIPTextModel
    torch.manual_seed(0)
    m = CLIPTextModel(CLIPTextConfig(vocab_size=300, hidden_size=768, intermediate_size=3072, num_hidden_layers=1,
                                     num_attention_heads=12, max_position_embeddings=77))
    pipe = SimpleNamespace(tokenizer=FakeTokenizer(300), text_encoder=m)
    pipe, cfg = load_new_concept(pipe, embeddings, True)
    return cfg, m.get_input_embeddings().weight.data[300:].clone()


def test_mirror_matches_reference_file_live():
    """The mirror's merge and concept load reproduce what the reference's convert_edlora_to_diffusers.py returned on the same
    case (stored by tests/golden/make_golden.py --crosscheck)."""
    from mixofshow.utils import convert_edlora_to_diffusers as mine
    gold = torch.load(GOLD, weights_only=False)['convert']
    sds, ckpt = mirror_case()
    for model_type, sd in sds.items():
        merged = mine.merge_lora_into_weight(sd, ckpt[model_type], model_type=model_type, alpha=MERGE_ALPHA)
        keys, samples = merge_samples(sd, merged)
        gkeys, gsamples = gold['merge'][model_type]
        assert keys == gkeys and samples.keys() == gsamples.keys()
        assert len(samples) == len(ckpt[model_type]) // 2
        for k, (idx, vals) in samples.items():
            assert torch.equal(idx, gsamples[k][0])
            assert torch.allclose(vals, gsamples[k][1], rtol=1e-6, atol=1e-8), k
    cfg, rows = load_concept(mine.load_new_concept, ckpt['new_concept_embedding'])
    assert cfg == gold['load_new_concept'][0] and torch.equal(rows, gold['load_new_concept'][1])
