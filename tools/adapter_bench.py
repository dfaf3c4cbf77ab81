#!/usr/bin/env python
"""tools/adapter_bench.py — time the T2I-Adapters on the B200.

  1. Both sd14v1 adapter shapes (key pose: 3 input channels, sketch: 1), batch 1, at 768 x 1536 (BASELINE config 4) and
     1024 x 2048 (the reference's `_2x` conditions): `T2IAdapter(x)` timed with CUDA events over --iters calls after
     --warmup calls.  FLOP are counted from the layer shapes (2 * M * N * K per convolution).
  2. One 30-step RegionallyT2IAdapterPipeline call at 768 x 1536 (full SD1.5 topology, 3 regions, CFG 7.5) given both
     condition images, against the same call given pre-computed adapter states.

Random-init weights (seeded); the card name and power limit are read in the same run.  Prints one JSON line.
  python tools/adapter_bench.py [--iters 50] [--warmup 5] [--no-pipeline]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, 'mix-of-show_b200')):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

CHANNELS = (320, 640, 1280, 1280)


def adapter_flop(cin, height, width, channels=CHANNELS, num_res_blocks=2, f=8):
    """Multiply-adds x 2 of every convolution of a 'full_adapter' T2IAdapter at batch 1."""
    h, w = height // f, width // f
    flop = 2 * h * w * channels[0] * 9 * cin * f * f
    for i, c in enumerate(channels):
        if i > 0:
            h, w = (h + 1) // 2, (w + 1) // 2
            if channels[i - 1] != c:
                flop += 2 * h * w * c * channels[i - 1]
        flop += num_res_blocks * 2 * h * w * c * (9 * c + c)
    return flop


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader'], capture_output=True,
                       text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name()


def time_adapters(iters, warmup):
    from mixofshow.models.adapter_b200 import T2IAdapter
    rows = []
    for kind, cin in (('keypose', 3), ('sketch', 1)):
        ad = T2IAdapter(in_channels=cin)
        for height, width in ((768, 1536), (1024, 2048)):
            x = torch.rand(1, cin, height, width, generator=torch.Generator().manual_seed(cin)).cuda()
            for _ in range(warmup):
                ad(x)
            torch.cuda.synchronize()
            t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            t0.record()
            for _ in range(iters):
                ad(x)
            t1.record()
            torch.cuda.synchronize()
            ms = t0.elapsed_time(t1) / iters
            flop = adapter_flop(cin, height, width)
            rows.append({'adapter': kind, 'height': height, 'width': width, 'ms': round(ms, 3), 'gflop': round(flop / 1e9, 1),
                         'tflops': round(flop / ms / 1e9, 1), 'launches': ad._engine.launches})
            print(f'{kind:8s} {height}x{width}: {ms:.3f} ms  {flop / 1e9:.1f} GFLOP  {flop / ms / 1e9:.1f} TFLOP/s  '
                  f'{ad._engine.launches} launches', flush=True)
    return rows


def time_pipeline(steps=30):
    from PIL import Image

    from mixofshow.models.adapter_b200 import T2IAdapter
    from mixofshow.models.unet_b200 import UNet2DConditionModel
    from mixofshow.pipelines.pipeline_regionally_t2iadapter import RegionallyT2IAdapterPipeline, _preprocess_adapter_image
    from oracle import unet as ou
    height, width = 768, 1536
    unet = UNet2DConditionModel()
    unet.load_state_dict(ou.build_unet(0, None).state_dict())
    pipe = RegionallyT2IAdapterPipeline(unet=unet).to('cuda')
    pipe.set_new_concept_cfg({})
    pipe.keypose_adapter, pipe.sketch_adapter = T2IAdapter(in_channels=3), T2IAdapter(in_channels=1)
    cond = os.path.join(ROOT, 'tests', 'golden', 'conditions')
    pose = Image.open(os.path.join(cond, 'harry+catA+dogA_pose.png')).convert('RGB')
    sketch = Image.open(os.path.join(cond, 'harry+catA+dogA_sketch.png')).convert('L')
    g = lambda s: torch.Generator().manual_seed(s)
    boxes = [[3, 5, 768, 368], [11, 368, 768, 690], [2, 977, 768, 1494]]
    regs = [(torch.randn(2, 16, 77, 768, generator=g(5 + i)).cuda(), (b[0] / height, b[1] / width, b[2] / height, b[3] / width))
            for i, b in enumerate(boxes)]
    common = dict(prompt_embeds=torch.randn(2, 16, 77, 768, generator=g(4)).cuda(), region_list=regs, height=height,
                  width=width, num_inference_steps=steps, guidance_scale=7.5, output_type='latent')
    lat = torch.randn(1, 4, height // 8, width // 8, generator=g(3))
    states = {k: pipe.__dict__[f'{k}_adapter'](_preprocess_adapter_image(img, height, width).cuda())
              for k, img in (('keypose', pose), ('sketch', sketch))}
    legs = {'conditions': dict(keypose_adapter_input=[pose], sketch_adapter_input=[sketch]),
            'states': dict(keypose_adapter_state=states['keypose'], sketch_adapter_state=states['sketch'])}
    out = {}
    for rep in range(3):                       # first round warms both legs (engines, graphs); alternate the legs
        for name, kw in legs.items():
            torch.cuda.synchronize()
            t = time.perf_counter()
            pipe(latents=lat.clone(), **common, **kw)
            torch.cuda.synchronize()
            if rep > 0:
                out.setdefault(name, []).append(time.perf_counter() - t)
    res = {k: round(min(v) * 1e3, 1) for k, v in out.items()}
    print(f'{steps}-step pipeline call at {height}x{width}: with conditions {res["conditions"]} ms, with pre-computed '
          f'states {res["states"]} ms', flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--no-pipeline', action='store_true')
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('adapter_bench.py needs a GPU')
    torch.backends.cuda.matmul.allow_tf32 = False
    gpu = card()
    print(f'card: {gpu}', flush=True)
    result = {'card': gpu, 'adapters': time_adapters(a.iters, a.warmup)}
    if not a.no_pipeline:
        result['pipeline_30_steps_ms'] = time_pipeline()
    print(json.dumps(result))


if __name__ == '__main__':
    main()
