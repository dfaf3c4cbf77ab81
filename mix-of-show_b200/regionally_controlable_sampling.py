"""B200 mirror of the reference's `regionally_controlable_sampling.py` entry script (BASELINE config 4): region-string
parsing, model loading from a fused `combined_model_*` directory, condition images, and the sampling call.  Host logic only;
the UNet loop runs on `RegionallyT2IAdapterPipeline` (mixofshow/pipelines/pipeline_regionally_t2iadapter.py) and the
T2I-Adapters on `mixofshow.models.adapter_b200.T2IAdapter`.

Conditions are images (`--sketch_condition` / `--keypose_condition`, run through the adapters of `--sketch_adapter` /
`--keypose_adapter DIR`: local diffusers T2IAdapter directories, where the reference names hub ids) or pre-computed adapter
feature maps (`--*_adapter_state file.pt`).  The result is always written as latents; with `--vae_model DIR` (a directory
holding `vae/`) it is also decoded and saved as a PNG with its config `.txt`, as the reference does."""
import argparse
import ast
import hashlib
import json
import os

import torch


def prepare_text(prompt, region_prompts, height, width):
    """regionally_controlable_sampling.py:67-94.  region_prompts:
    '[subject1]-*-[negative1]-*-[h0, w0, h1, w1]|[subject2]-*-[negative2]-*-[...]' (pixel boxes; '[]' = whole image) ->
    (prompt, [(region prompt, region negative prompt, [h0/H, w0/W, h1/H, w1/W]), ...]).  The box arithmetic is Python
    float division exactly as in the reference (the fractions feed the bit-exact ceil/floor of the region masks)."""
    region_collection = []
    for region in region_prompts.split('|'):
        if region == '':
            break
        prompt_region, neg_prompt_region, pos = region.split('-*-')
        prompt_region = prompt_region.replace('[', '').replace(']', '')
        neg_prompt_region = neg_prompt_region.replace('[', '').replace(']', '')
        pos = list(ast.literal_eval(pos))          # the reference uses eval(); the strings are list literals
        if len(pos) == 0:
            pos = [0, 0, 1, 1]
        else:
            pos[0], pos[2] = pos[0] / height, pos[2] / height
            pos[1], pos[3] = pos[1] / width, pos[3] / width
        region_collection.append((prompt_region, neg_prompt_region, pos))
    return (prompt, region_collection)


def build_model(pretrained_model, device='cuda', tokenizer=None, vae_model=None):
    """reference :55-64: pipeline + new_concept_cfg.json from a fused model directory (+ the VAE of `vae_model/vae`)."""
    from mixofshow.pipelines.pipeline_regionally_t2iadapter import RegionallyT2IAdapterPipeline
    from mixofshow.utils import model_io
    assert os.path.exists(os.path.join(pretrained_model, 'new_concept_cfg.json'))
    unet = model_io.load_unet(pretrained_model)
    text_encoder = model_io.load_text_encoder(pretrained_model, device=device)
    if tokenizer is None:
        from transformers import CLIPTokenizer
        tokenizer = CLIPTokenizer.from_pretrained(pretrained_model, subfolder='tokenizer')
    new_concept_cfg = model_io.load_new_concept_cfg(pretrained_model)
    model_io.ensure_concept_tokens(tokenizer, new_concept_cfg)      # the fused model's added `<new{k}>` tokens
    vae = model_io.load_vae(vae_model, device=device) if vae_model is not None else None
    pipe = RegionallyT2IAdapterPipeline(vae=vae, text_encoder=text_encoder, tokenizer=tokenizer, unet=unet).to(device)
    pipe.set_new_concept_cfg(new_concept_cfg)
    return pipe


def sample_image(pipe, input_prompt, input_neg_prompt=None, generator=None, num_inference_steps=50, guidance_scale=7.5,
                 **extra_kargs):
    """reference :14-52 (adapter states / weights travel in extra_kargs: keypose_adapter_state=..., sketch_adaptor_weight=...)."""
    return pipe(prompt=input_prompt, negative_prompt=input_neg_prompt, generator=generator, guidance_scale=guidance_scale,
                num_inference_steps=num_inference_steps, **extra_kargs).images


def parse_args(argv=None):
    parser = argparse.ArgumentParser('', add_help=False)
    parser.add_argument('--pretrained_model', required=True, type=str)
    parser.add_argument('--sketch_condition', default=None, type=str, help="sketch image ('' or a missing file: skipped)")
    parser.add_argument('--sketch_adapter', default=None, type=str, help='local diffusers T2IAdapter directory (sketch)')
    parser.add_argument('--keypose_condition', default=None, type=str, help="pose image ('' or a missing file: skipped)")
    parser.add_argument('--keypose_adapter', default=None, type=str, help='local diffusers T2IAdapter directory (key pose)')
    parser.add_argument('--vae_model', default=None, type=str, help='directory holding vae/: also decode and save a PNG')
    parser.add_argument('--sketch_adapter_state', default=None, type=str, help='torch file: 4 pre-computed sketch adapter maps')
    parser.add_argument('--sketch_adaptor_weight', default=1.0, type=float)
    parser.add_argument('--region_sketch_adaptor_weight', default='', type=str)
    parser.add_argument('--keypose_adapter_state', default=None, type=str, help='torch file: 4 pre-computed keypose adapter maps')
    parser.add_argument('--keypose_adaptor_weight', default=1.0, type=float)
    parser.add_argument('--region_keypose_adaptor_weight', default='', type=str)
    parser.add_argument('--height', default=768, type=int)
    parser.add_argument('--width', default=1536, type=int)
    parser.add_argument('--save_dir', default=None, type=str)
    parser.add_argument('--prompt', default='photo of a toy', type=str)
    parser.add_argument('--negative_prompt', default='', type=str)
    parser.add_argument('--prompt_rewrite', default='', type=str)
    parser.add_argument('--seed', default=16141, type=int)
    parser.add_argument('--suffix', default='', type=str)
    parser.add_argument('--num_inference_steps', default=50, type=int)       # the reference samples with 50 steps (:38)
    return parser.parse_args(argv)


def load_conditions(args):
    """reference :121-139: {'sketch': PIL 'L' image or None, 'keypose': PIL 'RGB' image or None} and the sampling
    (height, width): the conditions' size when one is used, else --height / --width.  A condition path that is '' or
    does not exist is skipped.  Raises ValueError (before any model is loaded) when a used condition has no adapter
    directory or comes with a pre-computed state of the same kind, or when the two conditions differ in size."""
    from PIL import Image
    conds = {}
    for kind, mode in (('sketch', 'L'), ('keypose', 'RGB')):
        path = getattr(args, f'{kind}_condition')
        if path is None or not os.path.exists(path):
            conds[kind] = None
            print(f'skip {kind} condition')
            continue
        if getattr(args, f'{kind}_adapter') is None:
            raise ValueError(f'--{kind}_condition needs --{kind}_adapter DIR (a local T2IAdapter directory)')
        if getattr(args, f'{kind}_adapter_state') is not None:
            raise ValueError(f'--{kind}_condition and --{kind}_adapter_state are exclusive: give one of them')
        conds[kind] = Image.open(path).convert(mode)
        print(f'use {kind} condition')
    sizes = {c.size for c in conds.values() if c is not None}
    if len(sizes) > 1:
        raise ValueError(f'conditions should be same size, got {sorted(sizes)} (width, height)')
    if sizes:
        width, height = sizes.pop()
        return conds, height, width
    return conds, args.height, args.width


def save_image(args, image, save_prompt):
    """reference :164-187: <save_dir>/seed_<seed>/<prompt>---<suffix>---<hash>.png and the .txt of its config lines."""
    configs = [
        f'pretrained_model: {args.pretrained_model}\n',
        f'context_prompt: {args.prompt}\n', f'neg_context_prompt: {args.negative_prompt}\n',
        f'sketch_condition: {args.sketch_condition}\n', f'sketch_adaptor_weight: {args.sketch_adaptor_weight}\n',
        f'region_sketch_adaptor_weight: {args.region_sketch_adaptor_weight}\n',
        f'keypose_condition: {args.keypose_condition}\n', f'keypose_adaptor_weight: {args.keypose_adaptor_weight}\n',
        f'region_keypose_adaptor_weight: {args.region_keypose_adaptor_weight}\n', f'random seed: {args.seed}\n',
        f'prompt_rewrite: {args.prompt_rewrite}\n'
    ]
    hash_code = hashlib.sha256(''.join(configs).encode('utf-8')).hexdigest()[:8]
    save_name = f"{save_prompt.replace(' ', '_')}---{args.suffix}---{hash_code}.png"
    save_dir = os.path.join(args.save_dir, f'seed_{args.seed}')
    os.makedirs(save_dir, exist_ok=True)
    save_path = os.path.join(save_dir, save_name)
    image.save(save_path)
    with open(save_path.replace('.png', '.txt'), 'w') as fw:
        fw.writelines(configs)
    return save_path


def main(argv=None):
    args = parse_args(argv)
    conds, height, width = load_conditions(args)
    device = torch.device('cuda')
    pipe = build_model(args.pretrained_model, device, vae_model=args.vae_model)
    kwargs = {'height': height, 'width': width, 'output_type': 'latent'}
    for kind in ('sketch', 'keypose'):
        path = getattr(args, f'{kind}_adapter_state')
        if path is not None:
            kwargs[f'{kind}_adapter_state'] = torch.load(path)
        if conds[kind] is not None:
            from mixofshow.models.adapter_b200 import T2IAdapter
            setattr(pipe, f'{kind}_adapter', T2IAdapter.from_pretrained(getattr(args, f'{kind}_adapter')).to(device))
            kwargs[f'{kind}_adapter_input'] = [conds[kind]]
        kwargs[f'{kind}_adaptor_weight'] = getattr(args, f'{kind}_adaptor_weight')
        kwargs[f'region_{kind}_adaptor_weight'] = getattr(args, f'region_{kind}_adaptor_weight')
    input_prompt = [prepare_text(args.prompt, args.prompt_rewrite, height, width)]
    latents = sample_image(pipe, input_prompt=input_prompt, input_neg_prompt=[args.negative_prompt],
                           generator=torch.Generator('cpu').manual_seed(args.seed),
                           num_inference_steps=args.num_inference_steps, **kwargs)
    if args.save_dir is not None:
        os.makedirs(args.save_dir, exist_ok=True)
        out = os.path.join(args.save_dir, f'latents---{args.seed}{"---" + args.suffix if args.suffix else ""}.pt')
        torch.save({'latents': latents.cpu(), 'config': vars(args)}, out)
        with open(os.path.join(args.save_dir, 'config.json'), 'w') as f:
            json.dump(vars(args), f)
        print(f'save to: {out}')
        if pipe.vae is not None:
            print(f'save to: {save_image(args, pipe.decode_latents(latents)[0], input_prompt[0][0])}')
    return latents


if __name__ == '__main__':
    main()
