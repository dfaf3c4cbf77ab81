"""On-disk model formats of the ED-LoRA ecosystem (SURVEY.md §8f rank 3), host logic only:

  * the diffusers `save_pretrained` directory layout the reference loads with `from_pretrained` (`README.md:146,212`,
    `regionally_controlable_sampling.py:56-63`) and writes at `gradient_fusion.py:811`:
        <dir>/unet/config.json + diffusion_pytorch_model.safetensors (or .bin)
        <dir>/text_encoder/config.json + model.safetensors (or pytorch_model.bin)
  * `<dir>/new_concept_cfg.json` (`gradient_fusion.py:812-813`).
  * a T2I-Adapter directory (`config.json` + `diffusion_pytorch_model.safetensors`, what
    `T2IAdapter.from_pretrained` reads at `regionally_controlable_sampling.py:62-63`).

`load_unet` / `load_text_encoder` build this repo's B200 containers from such a directory; `save_combined_model` writes
one.  diffusers itself is not a dependency: the UNet `config.json` keys are the SD1.5 ones (diffusers 0.19.3), and any
option this path does not implement is rejected loudly instead of being ignored."""
import json
import os

import torch

UNET_WEIGHTS = ('diffusion_pytorch_model.safetensors', 'diffusion_pytorch_model.bin')
TEXT_WEIGHTS = ('model.safetensors', 'pytorch_model.bin')

# SD1.5 `unet/config.json` (diffusers 0.19.3 key names)
UNET_CONFIG_SD15 = {
    '_class_name': 'UNet2DConditionModel', '_diffusers_version': '0.19.3', 'act_fn': 'silu', 'attention_head_dim': 8,
    'block_out_channels': [320, 640, 1280, 1280], 'center_input_sample': False, 'cross_attention_dim': 768,
    'down_block_types': ['CrossAttnDownBlock2D', 'CrossAttnDownBlock2D', 'CrossAttnDownBlock2D', 'DownBlock2D'],
    'downsample_padding': 1, 'flip_sin_to_cos': True, 'freq_shift': 0, 'in_channels': 4, 'layers_per_block': 2,
    'mid_block_scale_factor': 1, 'norm_eps': 1e-05, 'norm_num_groups': 32, 'out_channels': 4, 'sample_size': 64,
    'up_block_types': ['UpBlock2D', 'CrossAttnUpBlock2D', 'CrossAttnUpBlock2D', 'CrossAttnUpBlock2D'],
}
# options that change the arithmetic: only these values are implemented by the B200 engine
_UNET_REQUIRED = {
    'act_fn': 'silu', 'center_input_sample': False, 'downsample_padding': 1, 'flip_sin_to_cos': True, 'freq_shift': 0,
    'mid_block_scale_factor': 1, 'norm_num_groups': 32, 'use_linear_projection': False, 'only_cross_attention': False,
    'dual_cross_attention': False, 'upcast_attention': False, 'resnet_time_scale_shift': 'default',
    'class_embed_type': None, 'addition_embed_type': None, 'encoder_hid_dim': None, 'time_embedding_type': 'positional',
    'conv_in_kernel': 3, 'conv_out_kernel': 3, 'mid_block_type': 'UNetMidBlock2DCrossAttn',
}


def _read_weights(folder, candidates):
    for name in candidates:
        path = os.path.join(folder, name)
        if os.path.isfile(path):
            if name.endswith('.safetensors'):
                from safetensors.torch import load_file
                return load_file(path)
            return torch.load(path, map_location='cpu')
    raise FileNotFoundError(f'none of {candidates} found in {folder}')


def _write_weights(folder, name, state_dict):
    from safetensors.torch import save_file
    os.makedirs(folder, exist_ok=True)
    save_file({k: v.detach().to('cpu').contiguous() for k, v in state_dict.items()}, os.path.join(folder, name))


def check_unet_config(cfg):
    """Reject diffusers UNet options the B200 engine does not implement (instead of silently ignoring them)."""
    for k, want in _UNET_REQUIRED.items():
        if k in cfg and cfg[k] != want and not (want is False and cfg[k] is None):
            raise ValueError(f'unet/config.json: {k}={cfg[k]!r} is not supported on the B200 path (needs {want!r})')
    nb = len(cfg['block_out_channels'])
    down = cfg.get('down_block_types', ['CrossAttnDownBlock2D'] * (nb - 1) + ['DownBlock2D'])
    up = cfg.get('up_block_types', ['UpBlock2D'] + ['CrossAttnUpBlock2D'] * (nb - 1))
    if list(down) != ['CrossAttnDownBlock2D'] * (nb - 1) + ['DownBlock2D'] or \
            list(up) != ['UpBlock2D'] + ['CrossAttnUpBlock2D'] * (nb - 1):
        raise ValueError(f'unsupported block layout: down {down}, up {up}')
    if not isinstance(cfg.get('attention_head_dim', 8), int):
        raise ValueError('per-block attention_head_dim lists are not supported')


def load_unet(model_dir, subfolder='unet'):
    """diffusers-layout directory -> mixofshow.models.unet_b200.UNet2DConditionModel (fp32 parameters on the host; the
    engine packs them to bf16 on first call)."""
    from mixofshow.models.unet_b200 import UNet2DConditionModel
    folder = os.path.join(model_dir, subfolder) if subfolder else model_dir
    with open(os.path.join(folder, 'config.json')) as f:
        cfg = json.load(f)
    check_unet_config(cfg)
    keys = ('in_channels', 'out_channels', 'block_out_channels', 'layers_per_block', 'attention_head_dim',
            'cross_attention_dim', 'norm_num_groups', 'sample_size')
    kw = {k: (tuple(cfg[k]) if isinstance(cfg[k], list) else cfg[k]) for k in keys if k in cfg}
    unet = UNet2DConditionModel(**kw)
    sd = {k: v.to(torch.float32) for k, v in _read_weights(folder, UNET_WEIGHTS).items()}
    unet.load_state_dict(sd)            # strict: a checkpoint of another architecture fails here
    return unet


def save_unet(unet, model_dir, subfolder='unet'):
    folder = os.path.join(model_dir, subfolder) if subfolder else model_dir
    c = unet.config
    cfg = dict(UNET_CONFIG_SD15)
    nb = len(c.block_out_channels)
    cfg.update(in_channels=c.in_channels, out_channels=c.out_channels, block_out_channels=list(c.block_out_channels),
               layers_per_block=c.layers_per_block, attention_head_dim=c.attention_head_dim,
               cross_attention_dim=c.cross_attention_dim, norm_num_groups=c.norm_num_groups, sample_size=c.sample_size,
               down_block_types=['CrossAttnDownBlock2D'] * (nb - 1) + ['DownBlock2D'],
               up_block_types=['UpBlock2D'] + ['CrossAttnUpBlock2D'] * (nb - 1))
    os.makedirs(folder, exist_ok=True)
    with open(os.path.join(folder, 'config.json'), 'w') as f:
        json.dump(cfg, f, indent=2, sort_keys=True)
    _write_weights(folder, UNET_WEIGHTS[0], unet.state_dict())


def load_text_encoder(model_dir, subfolder='text_encoder', **kw):
    """transformers-layout CLIP text encoder directory -> mixofshow.models.clip_b200.CLIPTextModel."""
    from mixofshow.models.clip_b200 import CLIPTextModel
    folder = os.path.join(model_dir, subfolder) if subfolder else model_dir
    with open(os.path.join(folder, 'config.json')) as f:
        cfg = json.load(f)
    if cfg.get('hidden_act', 'quick_gelu') != 'quick_gelu':
        raise ValueError(f"text_encoder/config.json: hidden_act={cfg['hidden_act']!r} is not supported (quick_gelu only)")
    if cfg.get('hidden_size', 768) // cfg.get('num_attention_heads', 12) > 80:
        raise ValueError('head dim > 80 is not supported by the causal attention kernel')
    sd = {k: v.to(torch.float32) for k, v in _read_weights(folder, TEXT_WEIGHTS).items()
          if k.startswith('text_model.') and not k.endswith('position_ids')}
    te = CLIPTextModel(sd, **kw)
    te.hf_config = cfg
    return te


def save_text_encoder(text_encoder, model_dir, subfolder='text_encoder', hf_config=None):
    folder = os.path.join(model_dir, subfolder) if subfolder else model_dir
    cfg = dict(hf_config or getattr(text_encoder, 'hf_config', None) or {})
    sd = text_encoder.state_dict()
    layers = 1 + max(int(k.split('.layers.')[1].split('.')[0]) for k in sd if '.layers.' in k)
    cfg.update(architectures=['CLIPTextModel'], model_type='clip_text_model', hidden_act='quick_gelu',
               vocab_size=sd['text_model.embeddings.token_embedding.weight'].shape[0],
               hidden_size=sd['text_model.embeddings.token_embedding.weight'].shape[1],
               max_position_embeddings=sd['text_model.embeddings.position_embedding.weight'].shape[0],
               intermediate_size=sd['text_model.encoder.layers.0.mlp.fc1.weight'].shape[0], num_hidden_layers=layers)
    cfg.setdefault('num_attention_heads', 12)
    cfg.setdefault('layer_norm_eps', 1e-05)
    os.makedirs(folder, exist_ok=True)
    with open(os.path.join(folder, 'config.json'), 'w') as f:
        json.dump(cfg, f, indent=2, sort_keys=True)
    _write_weights(folder, TEXT_WEIGHTS[0], sd)


VAE_WEIGHTS = ('diffusion_pytorch_model.safetensors', 'diffusion_pytorch_model.bin')
_VAE_REQUIRED = {'act_fn': 'silu', 'norm_num_groups': 32, 'in_channels': 3, 'out_channels': 3}


def load_vae(model_dir, subfolder='vae', device='cuda'):
    """diffusers-layout `vae/` directory (config.json + weights) -> mixofshow.models.vae_b200.AutoencoderKL."""
    from mixofshow.models.vae_b200 import AutoencoderKL
    folder = os.path.join(model_dir, subfolder) if subfolder else model_dir
    with open(os.path.join(folder, 'config.json')) as f:
        cfg = json.load(f)
    for k, want in _VAE_REQUIRED.items():
        if k in cfg and cfg[k] != want:
            raise ValueError(f'vae/config.json: {k}={cfg[k]!r} is not supported on the B200 path (needs {want!r})')
    down = cfg.get('down_block_types')
    if down is not None and any(t != 'DownEncoderBlock2D' for t in down):
        raise ValueError(f'unsupported VAE block layout {down}')
    return AutoencoderKL(_read_weights(folder, VAE_WEIGHTS), block_out_channels=tuple(cfg.get('block_out_channels', (128, 256, 512, 512))),
                         layers_per_block=cfg.get('layers_per_block', 2), latent_channels=cfg.get('latent_channels', 4),
                         scaling_factor=cfg.get('scaling_factor', 0.18215), device=device)


def save_vae(vae, model_dir, subfolder='vae'):
    folder = os.path.join(model_dir, subfolder) if subfolder else model_dir
    c = vae.config
    nb = len(c.block_out_channels)
    cfg = {'_class_name': 'AutoencoderKL', '_diffusers_version': '0.19.3', 'act_fn': 'silu',
           'block_out_channels': list(c.block_out_channels), 'down_block_types': ['DownEncoderBlock2D'] * nb,
           'up_block_types': ['UpDecoderBlock2D'] * nb, 'in_channels': 3, 'out_channels': 3,
           'latent_channels': c.latent_channels, 'layers_per_block': c.layers_per_block, 'norm_num_groups': 32,
           'sample_size': 512, 'scaling_factor': c.scaling_factor}
    os.makedirs(folder, exist_ok=True)
    with open(os.path.join(folder, 'config.json'), 'w') as f:
        json.dump(cfg, f, indent=2, sort_keys=True)
    _write_weights(folder, VAE_WEIGHTS[0], vae.state_dict())


ADAPTER_WEIGHTS = ('diffusion_pytorch_model.safetensors', 'diffusion_pytorch_model.bin')


def load_t2i_adapter(model_dir, device='cuda'):
    """diffusers-layout T2IAdapter directory (config.json + weights, e.g. a local copy of TencentARC/t2iadapter_openpose_sd14v1)
    -> mixofshow.models.adapter_b200.T2IAdapter.  The config is validated by the T2IAdapter constructor."""
    from mixofshow.models.adapter_b200 import T2IAdapter
    if not os.path.isdir(model_dir):
        raise FileNotFoundError(f'T2I-Adapter {model_dir!r} is not a local directory: hub ids are not downloaded; pass a '
                                'directory holding config.json and diffusion_pytorch_model.safetensors')
    with open(os.path.join(model_dir, 'config.json')) as f:
        cfg = json.load(f)
    adapter = T2IAdapter(in_channels=cfg.get('in_channels', 3), channels=cfg.get('channels', [320, 640, 1280, 1280]),
                         num_res_blocks=cfg.get('num_res_blocks', 2), downscale_factor=cfg.get('downscale_factor', 8),
                         adapter_type=cfg.get('adapter_type', 'full_adapter'), device=device)
    adapter.load_state_dict(_read_weights(model_dir, ADAPTER_WEIGHTS))
    return adapter


def save_t2i_adapter(adapter, model_dir):
    c = adapter.config
    cfg = {'_class_name': 'T2IAdapter', '_diffusers_version': '0.19.3', 'adapter_type': c.adapter_type,
           'channels': list(c.channels), 'downscale_factor': c.downscale_factor, 'in_channels': c.in_channels,
           'num_res_blocks': c.num_res_blocks}
    os.makedirs(model_dir, exist_ok=True)
    with open(os.path.join(model_dir, 'config.json'), 'w') as f:
        json.dump(cfg, f, indent=2, sort_keys=True)
    _write_weights(model_dir, ADAPTER_WEIGHTS[0], adapter.state_dict())


def save_combined_model(model_dir, unet, text_encoder, new_concept_cfg, tokenizer=None):
    """What gradient_fusion.py:810-813 (`pipe.save_pretrained`) leaves on disk for the sampling scripts: unet/,
    text_encoder/, new_concept_cfg.json AND the tokenizer that carries the added `<new{k}>` tokens — without it the
    concept tokens would be BPE-split into ordinary sub-tokens on reload and the learned embedding rows never selected.
    (The VAE / scheduler folders of the base model are untouched by the fusion; the caller copies them.)"""
    save_unet(unet, model_dir)
    save_text_encoder(text_encoder, model_dir)
    if tokenizer is not None:
        tokenizer.save_pretrained(os.path.join(model_dir, 'tokenizer'))
    with open(os.path.join(model_dir, 'new_concept_cfg.json'), 'w') as f:
        json.dump(new_concept_cfg, f)


def ensure_concept_tokens(tokenizer, new_concept_cfg):
    """Loader-side guard for fused models: every `concept_token_names[k]` must map to `concept_token_ids[k]`.  A tokenizer
    folder copied from the BASE model lacks the added tokens: they are re-added here in id order and the resulting ids
    are checked against the cfg (raises instead of silently sampling without the concepts)."""
    pairs = sorted({(i, n) for c in new_concept_cfg.values()
                    for i, n in zip(c['concept_token_ids'], c['concept_token_names'])})
    missing = [n for i, n in pairs if tokenizer.convert_tokens_to_ids(n) != i]
    if missing:
        tokenizer.add_tokens([n for _, n in pairs if n in set(missing)])
    bad = [(n, i, tokenizer.convert_tokens_to_ids(n)) for i, n in pairs if tokenizer.convert_tokens_to_ids(n) != i]
    if bad:
        raise ValueError(f'tokenizer does not match new_concept_cfg.json (token, expected id, actual id): {bad[:4]} ... '
                         'load the tokenizer saved next to the fused model')
    return tokenizer


def load_new_concept_cfg(model_dir):
    """regionally_controlable_sampling.py:66-68 / test_edlora.py: {concept: {'concept_token_ids', 'concept_token_names'}}."""
    with open(os.path.join(model_dir, 'new_concept_cfg.json')) as f:
        return json.load(f)
