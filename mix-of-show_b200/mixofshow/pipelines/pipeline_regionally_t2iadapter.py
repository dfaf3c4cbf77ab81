"""Drop-in for the reference's `mixofshow/pipelines/pipeline_regionally_t2iadapter.py`:
`RegionT2I_AttnProcessor`, `revise_regionally_t2iadapter_attention_forward`, `RegionallyT2IAdapterPipeline`.

The region-masked cross-attention (reference :32-86) runs as: one flash cross-attention per region with the region's
own K/V (tcgen05), then `mos_region_combine` (global outside the boxes, mean of covering regions inside).  Box indices
are computed on the host in Python float64 exactly as the reference does (`math.ceil` / `math.floor`), so they are
bit-exact.  Condition images (`*_adapter_input`: PIL images or tensors) are preprocessed as diffusers does and run
through the `keypose_adapter` / `sketch_adapter` attributes (mixofshow.models.adapter_b200.T2IAdapter on the B200);
pre-computed feature maps can be passed as `*_adapter_state` instead.
"""
import ast
import math
from types import SimpleNamespace

import numpy as np
import torch

from mixofshow.pipelines.pipeline_edlora import bind_concept_prompt
from mos_b200 import functional as Fm
from mos_b200 import ops
from mos_b200.scheduler import DPMSolverPP2M


def region_box_indices(box, feat_height, feat_width):
    """(start_h, start_w, end_h, end_w) feature-pixel indices of a fractional box (reference :37-39, :67-68)."""
    start_h, start_w, end_h, end_w = box
    return (math.ceil(start_h * feat_height), math.ceil(start_w * feat_width), math.floor(end_h * feat_height),
            math.floor(end_w * feat_width))


def region_feat_size(height, width, seq_lens):
    downscale = math.sqrt(height * width / seq_lens)               # reference :45
    return int(height // downscale), int(width // downscale)       # reference :48


class RegionT2I_AttnProcessor:
    def __init__(self, cross_attention_idx, attention_op=None):
        self.attention_op = attention_op
        self.cross_attention_idx = cross_attention_idx

    def __call__(self, attn, hidden_states, encoder_hidden_states=None, attention_mask=None, temb=None,
                 **cross_attention_kwargs):
        assert attention_mask is None, 'attention masks are not used by the ED-LoRA path'
        if encoder_hidden_states is None:
            out, _ = Fm.attention_block(attn, hidden_states, None)
            return out
        if len(encoder_hidden_states.shape) == 4:  # multi-layer embedding
            encoder_hidden_states = encoder_hidden_states[:, self.cross_attention_idx, ...]
        seq_lens = hidden_states.shape[1]
        fh, fw = region_feat_size(cross_attention_kwargs['height'], cross_attention_kwargs['width'], seq_lens)
        regions = []
        for region in cross_attention_kwargs['region_list']:
            emb = region[0][:, self.cross_attention_idx, ...] if len(region[0].shape) == 4 else region[0]
            regions.append((emb, region_box_indices(region[1], fh, fw)))
        out, _ = Fm.attention_block(attn, hidden_states, encoder_hidden_states, regions=regions, region_hw=(fh, fw))
        return out


def revise_regionally_t2iadapter_attention_forward(unet):
    def change_forward(unet, count):
        for name, layer in unet.named_children():
            if layer.__class__.__name__ == 'Attention':
                layer.set_processor(RegionT2I_AttnProcessor(count))
                if 'attn2' in name:
                    count += 1
            else:
                count = change_forward(layer, count)
        return count

    cross_attention_idx = change_forward(unet.down_blocks, 0)
    cross_attention_idx = change_forward(unet.mid_block, cross_attention_idx)
    cross_attention_idx = change_forward(unet.up_blocks, cross_attention_idx)
    print(f'Number of attention layer registered {cross_attention_idx}')


def _spatial_weight(feat, base_weight, region_weight_str, height, width):
    """Per-pixel adapter weight with optional per-region overrides '[h0,w0,h1,w1]-w|...' (reference :488-510);
    parsed with ast.literal_eval instead of eval."""
    fh, fw = feat.shape[2:]
    wmap = base_weight * torch.ones(fh, fw, dtype=feat.dtype, device=feat.device)
    if region_weight_str != '':
        for rw in region_weight_str.split('|'):
            region, weight = rw.split('-')
            region, weight = ast.literal_eval(region), ast.literal_eval(weight)
            sh, sw, eh, ew = region
            box = (sh / height, sw / width, eh / height, ew / width)
            a, b, c, d = region_box_indices(box, fh, fw)
            wmap[a:c, b:d] = weight
    return wmap * feat


def _preprocess_adapter_image(image, height, width):
    """diffusers' `_preprocess_adapter_image` (reference :413-423): a PIL image or a list of them -> LANCZOS resize to
    (width, height) -> fp32 NCHW in [0, 1] (a grayscale image gets one channel); tensors pass through untouched."""
    import PIL.Image
    if isinstance(image, torch.Tensor):
        return image
    if isinstance(image, PIL.Image.Image):
        image = [image]
    if not (isinstance(image, (list, tuple)) and image and all(isinstance(i, PIL.Image.Image) for i in image)):
        raise TypeError(f'adapter input must be a PIL image, a list of PIL images or a tensor, got {type(image)}')
    arrs = [np.array(i.resize((width, height), resample=PIL.Image.LANCZOS)) for i in image]
    arrs = [a[None, ..., None] if a.ndim == 2 else a[None] for a in arrs]
    x = np.concatenate(arrs, axis=0).astype(np.float32) / 255.0
    return torch.from_numpy(x.transpose(0, 3, 1, 2).copy())


class RegionallyT2IAdapterPipeline:
    def __init__(self, vae=None, text_encoder=None, tokenizer=None, unet=None, scheduler=None, safety_checker=None,
                 feature_extractor=None, requires_safety_checker: bool = False):
        assert unet is not None
        self.vae, self.text_encoder, self.tokenizer, self.unet = vae, text_encoder, tokenizer, unet
        self.scheduler = scheduler if scheduler is not None else DPMSolverPP2M()
        # diffusers: 2 ** (len(vae.config.block_out_channels) - 1); 8 for SD1.5 (and when no VAE is attached)
        self.vae_scale_factor = 2 ** (len(vae.config.block_out_channels) - 1) if vae is not None else 8
        self.new_concept_cfg = None
        self.keypose_adapter = self.sketch_adapter = None
        self.device = torch.device('cuda')
        revise_regionally_t2iadapter_attention_forward(self.unet)     # reference :210

    def to(self, device):
        self.device = torch.device(device)
        return self

    def set_new_concept_cfg(self, new_concept_cfg=None):
        self.new_concept_cfg = new_concept_cfg

    def _embed(self, prompts, device):
        ids = self.tokenizer(prompts, padding='max_length', max_length=self.tokenizer.model_max_length,
                             truncation=True, return_tensors='pt').input_ids
        return self.text_encoder(ids.to(device), attention_mask=None)[0]

    # reference :215-299
    def _encode_region_prompt(self, prompt, new_concept_cfg, device, num_images_per_prompt,
                              do_classifier_free_guidance, negative_prompt=None, prompt_embeds=None,
                              negative_prompt_embeds=None, height=512, width=512, region_list=None):
        if prompt is not None and isinstance(prompt, str):
            batch_size = 1
        elif prompt is not None and isinstance(prompt, list):
            batch_size = len(prompt)
        else:
            batch_size = prompt_embeds.shape[0] // (2 if do_classifier_free_guidance else 1)
        assert batch_size == 1, 'only sample one prompt once in this version'
        if prompt_embeds is None:
            if self.tokenizer is None or self.text_encoder is None:
                raise ValueError('no tokenizer / text_encoder supplied: pass prompt_embeds and region_list embeddings')
            context_prompt, region_list = prompt[0][0], list(prompt[0][1])
            e = self._embed(bind_concept_prompt([context_prompt], new_concept_cfg), device)
            prompt_embeds = e.reshape(batch_size, -1, *e.shape[1:])
            layer_num, seq_len = prompt_embeds.shape[1:3]
            if negative_prompt is None:
                negative_prompt = [''] * batch_size
            ne = self._embed(negative_prompt, device).view(batch_size, 1, seq_len, -1).repeat(1, layer_num, 1, 1)
            prompt_embeds = torch.cat([ne, prompt_embeds])
            for idx, (region_prompt, region_neg_prompt, pos) in enumerate(region_list):
                re_ = self._embed(bind_concept_prompt([region_prompt], new_concept_cfg), device)
                re_ = re_.reshape(batch_size, -1, *re_.shape[1:])
                if region_neg_prompt is None:
                    region_neg_prompt = [''] * batch_size
                rn = self._embed(region_neg_prompt, device).view(batch_size, 1, seq_len, -1).repeat(1, layer_num, 1, 1)
                region_list[idx] = (torch.cat([rn, re_]), pos)
        return prompt_embeds, region_list

    def _run_adapter(self, adapter, kind, adapter_input, height, width, latent_hw):
        """reference :413-423 + :474-482: preprocess the condition and run the adapter once."""
        if adapter is None:
            raise ValueError(f'{kind}_adapter_input given but pipe.{kind}_adapter is not set')
        x = _preprocess_adapter_image(adapter_input, height, width).to(self.device, adapter.dtype)
        state = adapter(x)
        if tuple(state[0].shape[-2:]) != tuple(latent_hw):
            raise ValueError(f'{kind} adapter features are {tuple(state[0].shape[-2:])}, the latents {tuple(latent_hw)}: '
                             'the adapter downscale factor must equal the VAE scale factor')
        return state

    @torch.no_grad()
    def decode_latents(self, latents, output_type='pil'):
        """latents -> images through the VAE: a list of PIL images, or an NHWC numpy array for output_type='np'."""
        if self.vae is None:
            raise ValueError("no VAE supplied: use output_type='latent'")
        image = self.vae.decode(latents / 0.18215).sample
        image = (image / 2 + 0.5).clamp(0, 1).cpu().permute(0, 2, 3, 1).float().numpy()
        if output_type == 'pil':
            from mixofshow.pipelines.pipeline_edlora import numpy_to_pil
            image = numpy_to_pil(image)
        return image

    @torch.no_grad()
    def __call__(self, prompt=None, keypose_adapter_input=None, keypose_adaptor_weight=1.0,
                 region_keypose_adaptor_weight='', sketch_adapter_input=None, sketch_adaptor_weight=1.0,
                 region_sketch_adaptor_weight='', height=None, width=None, num_inference_steps: int = 50,
                 guidance_scale: float = 7.5, negative_prompt=None, num_images_per_prompt=1, eta: float = 0.0,
                 generator=None, latents=None, prompt_embeds=None, negative_prompt_embeds=None, output_type='pil',
                 return_dict: bool = True, callback=None, callback_steps: int = 1, cross_attention_kwargs=None,
                 region_list=None, keypose_adapter_state=None, sketch_adapter_state=None):
        """Extra (B200) arguments: `region_list` = [(region_embeds [2,16,77,768], box fractions)] and
        `*_adapter_state` = precomputed T2I-Adapter feature maps (4 NCHW tensors), for use without CLIP / adapters."""
        device = self.device
        do_cfg = guidance_scale > 1.0
        assert self.new_concept_cfg is not None
        prompt_embeds, region_list = self._encode_region_prompt(
            prompt, self.new_concept_cfg, device, num_images_per_prompt, do_cfg, negative_prompt,
            prompt_embeds=prompt_embeds, negative_prompt_embeds=negative_prompt_embeds, height=height, width=width,
            region_list=region_list)
        self.scheduler.set_timesteps(num_inference_steps, device=device)
        timesteps = [int(t) for t in self.scheduler.timesteps]
        h, w = height // self.vae_scale_factor, width // self.vae_scale_factor
        shape = (1, self.unet.config.in_channels, h, w)
        if latents is None:
            latents = torch.randn(shape, generator=generator, device=generator.device if generator is not None
                                  else 'cpu')
        latents = (latents.to(device, torch.float32) * self.scheduler.init_noise_sigma).contiguous()

        if keypose_adapter_state is None and keypose_adapter_input is not None:
            keypose_adapter_state = self._run_adapter(self.keypose_adapter, 'keypose', keypose_adapter_input, height, width,
                                                      (h, w))
        if sketch_adapter_state is None and sketch_adapter_input is not None:
            sketch_adapter_state = self._run_adapter(self.sketch_adapter, 'sketch', sketch_adapter_input, height, width,
                                                     (h, w))
        adapter_state = None
        if keypose_adapter_state is not None or sketch_adapter_state is not None:
            n = len(keypose_adapter_state) if keypose_adapter_state is not None else len(sketch_adapter_state)
            adapter_state = []
            for i in range(n):
                fk = fs = 0
                if keypose_adapter_state is not None:
                    fk = _spatial_weight(keypose_adapter_state[i], keypose_adaptor_weight,
                                         region_keypose_adaptor_weight, height, width)
                if sketch_adapter_state is not None:
                    fs = _spatial_weight(sketch_adapter_state[i], sketch_adaptor_weight, region_sketch_adaptor_weight,
                                         height, width)
                v = fk + fs
                adapter_state.append(torch.cat([v] * 2, dim=0) if do_cfg else v)

        x0_prev = torch.zeros_like(latents)
        kwargs = {'region_list': region_list, 'height': height, 'width': width}
        # one prepared session (reference loop :548-580): region embeddings / boxes and the adapter residuals are
        # step-invariant and uploaded once; a step is one graph replay + one fused CFG / DPM-Solver++ kernel
        sess = self.unet.session(2 if do_cfg else 1, h, w, device, prompt_embeds, kwargs, adapter_state)
        unet_in = sess.latents_in
        unet_in.copy_(torch.cat([latents] * 2) if do_cfg else latents)
        sess.t_in.fill_(float(timesteps[0]))
        for i, t in enumerate(timesteps):
            noise_pred = sess.step()
            t_next = float(timesteps[i + 1]) if i + 1 < len(timesteps) else 0.0
            ops.cfg_dpmpp_step(noise_pred, latents, x0_prev, unet_in.view(-1), cfg=do_cfg,
                               guidance=float(guidance_scale), coef=self.scheduler.coefficients(i), t_out=sess.t_in,
                               t_next=t_next)
            if callback is not None and i % callback_steps == 0:
                callback(i, t, latents)
        image = latents if output_type == 'latent' else self.decode_latents(latents, output_type)
        if not return_dict:
            return (image, None)
        return SimpleNamespace(images=image, nsfw_content_detected=None)
