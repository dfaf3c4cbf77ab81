#!/usr/bin/env python
"""bench.py — BASELINE.json metric: SD1.5 UNet + ED-LoRA denoise steps/sec @512x512, bf16, on N B200s.

One "step" = one denoise step of EDLoRAPipeline (mixofshow/pipelines/pipeline_edlora.py:273-290): CFG batch-2 UNet
forward (un-merged rank-4 ED-LoRA on all 128 attention linears, layer-wise text embeddings) + CFG combine +
DPM-Solver++(2M) update.  Synthetic data: random-init SD1.5-topology weights (seed 0), random latents / embeddings.

  python bench.py --gpus N --steps K --warmup W          (N > 1: launched by torchrun, one rank per GPU, replicas)
  python bench.py --impl reference ...                    CPU arm: the fp32 oracle port of the reference path
  python bench.py ... --dump-outputs DIR                  also write what the last timed step of each leg computed

Prints ONE JSON line.  With the same arguments every input is the same from run to run (fixed seeds), so the arrays
--dump-outputs writes let two builds be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, 'mix-of-show_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

METRIC = 'SD1.5 UNet+ED-LoRA denoise steps/sec @512x512 bf16'
UNIT = 'denoise_steps/s'
WORKLOAD = ('EDLoRAPipeline denoise step: SD1.5 UNet 512x512 (latent 64x64), CFG batch 2, un-merged rank-4 ED-LoRA on '
            '128 attention linears, 16 layer-wise text embeddings [2,16,77,768] (their K/V projections computed once per '
            'prompt, not per step), DPM-Solver++(2M) update')
CPU_THREADS = None
FLOPS_PER_STEP = 2 * 0.8044e12  # algorithmic FLOPs of one CFG denoise step (SURVEY.md §8d)
DUMP_BYTES = 64 << 20           # --dump-outputs writes at most this much


def load_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            p = json.load(f)
        return {'tflops': float(p['bf16_tflops_sustained']), 'hbm': float(p['hbm_gbs']), 'src': 'measured'}
    except Exception:
        return {'tflops': 1400.0, 'hbm': 6650.0, 'src': 'fallback'}


def dump_outputs(path, arrays):
    """Write each array as <path>/<name>.npy in float32.  An array larger than its equal share of DUMP_BYTES is replaced by a
    fixed sample of its flattened elements: the first `share` positions of a seed-0 permutation, in ascending order."""
    import numpy as np
    import torch
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // 4 // len(arrays)
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() > share:
            idx = torch.randperm(a.numel(), generator=torch.Generator().manual_seed(0))[:share].sort().values
            a = a.reshape(-1)[idx]
        np.save(os.path.join(path, name + '.npy'), a.numpy())


# ----------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--id={self.index}', f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for s in self.samples:
            f = [x.strip() for x in s.split(',')]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ----------------------------------------------------------------------------------------------- workload
TINY = dict(block_out_channels=(320, 640), layers_per_block=1)       # --tiny debug topology (2-level UNet)


def build_workload(tiny=False, images=1):
    """Synthetic model + inputs for both arms WITHOUT touching oracle/: SD1.5-topology weights from this package's own
    `UNet2DConditionModel` container (PyTorch default inits under manual_seed(0), diffusers parameter names), a rank-4
    ED-LoRA on every attention projection (down ~ kaiming-uniform(a=sqrt(5)) as edlora.py:238, up ~ N(0, 0.02^2) so the
    low-rank path is exercised, SURVEY.md 8d) and random latents / layer-wise text embeddings."""
    import torch
    from mixofshow.models.unet_b200 import UNet2DConditionModel
    cfg = TINY if tiny else None
    torch.manual_seed(0)
    model = UNet2DConditionModel(**(cfg or {}))
    sd = {k: v.detach().clone() for k, v in model.state_dict().items()}
    del model
    lora = random_unet_lora(sd, cfg, seed=10)
    H = W = 64
    lat = torch.randn(images, 4, H, W, generator=torch.Generator().manual_seed(1))
    ehs = torch.randn(2 * images, 16, 77, 768, generator=torch.Generator().manual_seed(2))   # [uncond x n | cond x n]
    return sd, lora, lat, ehs, cfg


def random_unet_lora(sd, cfg=None, seed=10):
    """A random rank-4 ED-LoRA on every attention projection of `sd` (reference key layout: <module>.lora_down.weight
    [4, in], <module>.lora_up.weight [out, 4]); down ~ kaiming-uniform(a=sqrt(5)) (edlora.py:238), up ~ N(0, 0.02^2)."""
    import math

    import torch
    from mos_b200.engine import cross_attention_names
    g = torch.Generator().manual_seed(seed)
    names = cross_attention_names(cfg['block_out_channels'], cfg['layers_per_block']) if cfg else cross_attention_names()
    lora = {}
    for an in names:
        tb = an[:-len('.attn2')]
        for a in ('attn1', 'attn2'):
            for pj in ('to_q', 'to_k', 'to_v', 'to_out.0'):
                m = f'{tb}.{a}.{pj}'
                cout, cin = sd[m + '.weight'].shape
                lora[m + '.lora_down.weight'] = (torch.rand(4, cin, generator=g) * 2 - 1) / math.sqrt(cin)
                lora[m + '.lora_up.weight'] = torch.randn(cout, 4, generator=g) * 0.02
    return lora


def build_pipeline(sd, lora, cfg, dev):
    """The drop-in objects a user of the reference holds: B200 UNet container + LoRALinearLayer on all 128 attention
    projections (trainer_edlora.py:121-133 / convert_edlora_to_diffusers.py) + EDLoRAPipeline."""
    import contextlib
    import io

    import torch
    from mixofshow.models.edlora import LoRALinearLayer
    from mixofshow.models.unet_b200 import UNet2DConditionModel
    from mixofshow.pipelines.pipeline_edlora import EDLoRAPipeline
    unet = UNet2DConditionModel(**(cfg or {}))
    unet.load_state_dict(sd)
    mods = dict(unet.named_modules())
    with torch.no_grad():
        for k in lora:
            if k.endswith('.lora_down.weight'):
                name = k[:-len('.lora_down.weight')]
                layer = LoRALinearLayer(name, mods[name], rank=4, alpha=1.0)
                layer.lora_down.weight.copy_(lora[k])
                layer.lora_up.weight.copy_(lora[name + '.lora_up.weight'])
    with contextlib.redirect_stdout(io.StringIO()):      # the installers print a registration count (as the reference)
        pipe = EDLoRAPipeline(unet=unet).to(dev)
    pipe.set_new_concept_cfg({})
    return pipe


def build_cpu_reference(sd, lora, cfg):
    """CPU arm only: the fp32 oracle port of the reference path (oracle/ is test / baseline infrastructure), loaded with
    the SAME synthetic weights as the GPU arm."""
    from oracle import inject
    from oracle import unet as ou
    with __import__('torch').no_grad():
        unet = ou.UNet2DConditionModel(ou.TINY if cfg else None)
        unet.load_state_dict(sd)
    unet.eval()
    inject.install_edlora_processors(unet)
    return unet


def pick_cpu_threads():
    """Thread count of the CPU arm: PINNED to min(32, host CPUs) so that both arms of every run (and every round) use the
    same count.  (Round 1 picked the fastest of {8..128} per run; the pick flipped between 32 / 64 / 128 threads and the
    baseline moved 0.13-0.28 steps/s with it.  32 was the most frequent winner on the 128-thread GPU host: fp32 convs of
    this size stop scaling there and oversubscription costs an order of magnitude.)"""
    import torch
    n = min(32, os.cpu_count() or 1)
    torch.set_num_threads(n)
    return n


def cpu_reference_steps(unet, lora, lat, ehs, steps, warmup, budget_s):
    """Time the reference path on host cores: fp32 oracle UNet (reference processors' restatement + LoRA) + CFG +
    DPM-Solver++ per step.  Returns (steps_run, seconds)."""
    import torch
    from oracle import edlora_ref as er
    from oracle import inject
    from oracle.schedulers import DPMSolverMultistepScheduler
    inject.inject_lora(unet, lora, 1.0)
    global CPU_THREADS
    CPU_THREADS = pick_cpu_threads()
    sched = DPMSolverMultistepScheduler()
    sched.set_timesteps(50)
    latents = lat.clone()

    def one(i):
        nonlocal latents
        t = int(sched.timesteps[i])
        with torch.no_grad():
            eps = unet(torch.cat([latents] * 2), torch.tensor([t, t]), ehs).sample
        latents = sched.step(er.cfg_combine(eps, 7.5), t, latents).prev_sample

    i = 0
    for _ in range(warmup):
        one(i)
        i += 1
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        one(i)
        i += 1
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    return done, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--tiny', action='store_true', help='debug: 2-level UNet')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--act-dtype', default='fp16', choices=['fp16', 'bf16'],
                    help='operand type (weights and activations) of the sampling engine.  fp16 (default) is the reference\'s '
                         'own sampling precision and meets the 1e-3 latent tolerance at guidance 7.5; bf16 runs at the same '
                         'speed but measures 2.8e-3 (tests/test_unet_gpu.py, profiles/README.md)')
    ap.add_argument('--no-train', action='store_true', help='skip the data-parallel training leg (extra.train)')
    ap.add_argument('--train-batch', type=int, default=8, help='per-GPU batch of the training leg (BASELINE config 5: 8)')
    ap.add_argument('--images', type=int, default=1,
                    help='images denoised together per step (default 1 = the BASELINE workload; > 1 is a separate, '
                         'labelled throughput mode: value counts image-steps)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps write, as DIR/<name>.npy (float32, 64 MB at most), what the last timed step '
                         'of each leg returned: latents and eps of the device-resident loop, the latents of the '
                         'EDLoRAPipeline call, the trainable parameters and loss of the training leg')
    args = ap.parse_args()
    if args.dump_outputs and args.impl != 'b200':
        ap.error('--dump-outputs writes the outputs of the b200 implementation')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    import torch

    if args.impl == 'reference':
        if rank != 0:
            return
        sd, lora, lat, ehs, cfg = build_workload(args.tiny)
        unet = build_cpu_reference(sd, lora, cfg)
        done, secs = cpu_reference_steps(unet, lora, lat, ehs, args.steps, min(args.warmup, 1), budget_s=240.0)
        v = done / secs
        print(json.dumps({
            'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': done,
            'warmup': min(args.warmup, 1), 'ms_per_step': 1e3 * secs / done, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
            'config': {'workload': WORKLOAD, 'note': 'CPU oracle port of the reference path (diffusers absent); '
                       'steps capped to a 240 s budget'},
            'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': CPU_THREADS, 'host_cpus': os.cpu_count(), 'kind': 'port',
                             'sample': f'{done} full CFG denoise steps after {min(args.warmup, 1)} warm-up'},
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        }))
        return

    assert torch.cuda.is_available(), 'bench.py needs a GPU (no CPU fallback for the product path)'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=dev)
    from mos_b200 import ops
    from mos_b200.scheduler import DPMSolverPP2M

    sd, lora, lat, ehs, cfg = build_workload(args.tiny, args.images)
    n_img = args.images
    B, H, W = 2 * n_img, lat.shape[2], lat.shape[3]
    # The reference-facing objects (SURVEY.md 8b): the UNet container with a LoRALinearLayer on every attention projection
    # (installed as trainer_edlora.py:121-133 does) inside an EDLoRAPipeline.  Both legs below run on the engine this
    # container packs: `value` replays its prepared session directly (inputs resident in HBM), `e2e` is the user's call.
    pipe = build_pipeline(sd, lora, cfg, dev)
    unet = pipe.unet
    unet.act_dtype = torch.float16 if args.act_dtype == 'fp16' else torch.bfloat16
    sess = unet.session(B, H, W, dev, ehs.to(dev))
    eng = sess.eng
    nx = len(eng.xattn_names)
    sched = DPMSolverPP2M()
    total_steps = args.warmup + args.steps
    sched.set_timesteps(max(50, total_steps))
    ts = [float(t) for t in sched.timesteps]

    latents = lat.to(dev).clone()
    x0_prev = torch.zeros_like(latents)
    unet_in = eng.in_latents.view(-1)

    def reset():
        latents.copy_(lat.to(dev))
        x0_prev.zero_()
        eng.in_latents.copy_(torch.cat([latents, latents]))
        eng.in_t.fill_(ts[0])

    def step(i):
        eng.run()
        nxt = ts[i + 1] if i + 1 < len(ts) else 0.0
        ops.cfg_dpmpp_step(eng.out_eps, latents, x0_prev, unet_in, cfg=True, guidance=7.5,
                           coef=sched.coefficients(i), t_out=eng.in_t, t_next=nxt)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---------------- device-resident throughput (`value`)
    reset()
    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.warmup, total_steps):
        step(i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    launches = (eng.launches + 1) * args.steps
    outputs = {'latents': latents.clone(), 'eps': eng.out_eps.clone()} if args.dump_outputs and rank == 0 else None

    # ---------------- end-to-end through the public API (`e2e`): EDLoRAPipeline.__call__ on HOST tensors.  One call =
    # one image = `steps` denoise steps; per call the latents and the prompt embeddings travel host -> device (pinned
    # memory), per step the callback reads the current latents back into pinned host memory (progress preview, the
    # reference's `callback(i, t, latents)` hook, pipeline_edlora.py:298-300) and the final latents come back at the end.
    h_lat = lat.clone().pin_memory()
    h_cond = ehs[n_img:].clone().pin_memory()                      # [n, 16, 77, 768] layer-wise prompt embeddings
    h_neg = ehs[:n_img, 0].clone().pin_memory()                    # [n, 77, 768] negative-prompt embeddings
    h_step = torch.empty_like(h_lat).pin_memory()
    h_out = torch.empty_like(h_lat).pin_memory()

    def cb(i, t, latents_dev):
        h_step.copy_(latents_dev, non_blocking=True)

    def pipeline_call(steps):
        out = pipe(prompt_embeds=h_cond, negative_prompt_embeds=h_neg, latents=h_lat, num_inference_steps=steps,
                   guidance_scale=7.5, output_type='latent', callback=cb, callback_steps=1)
        h_out.copy_(out.images, non_blocking=True)
        torch.cuda.current_stream().synchronize()   # the caller consumes the image on the host
        return h_out

    pipeline_call(max(args.warmup, 3))
    barrier()
    t0 = time.perf_counter()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    e2e_out = pipeline_call(args.steps)
    g1.record()
    barrier()
    if outputs is not None:
        outputs['e2e_latents'] = e2e_out.clone()
    e2e_ms = max(g0.elapsed_time(g1), 1e3 * (time.perf_counter() - t0))
    clocks = sampler.stop() if rank == 0 else None      # sampled over both timed regions (device-resident and e2e)
    per_call_h2d = h_lat.numel() * 4 + h_cond.numel() * 4 + h_neg.numel() * 4
    h2d = per_call_h2d / args.steps
    d2h = h_step.numel() * 4 + h_out.numel() * 4 / args.steps

    # ---------------- per-kernel roofline of the dominant kernel (tcgen05 GEMM / implicit-GEMM conv), eager mode
    used_graph = eng.graph is not None
    roof = None
    if rank == 0:
        roof = gemm_roofline(eng, ops, torch)

    # ---------------- data-parallel ED-LoRA training leg (BASELINE configs 2 / 5): the path that actually shards
    train = None
    if not args.no_train:
        del pipe, unet, sess, eng
        torch.cuda.empty_cache()
        try:
            train = train_leg(args, rank, world, dev, sd, lora, cfg, outputs)
        except Exception as exc:                     # the headline line must still print; the failure is reported, not hidden
            import traceback
            traceback.print_exc()
            train = {'error': f'{type(exc).__name__}: {exc}'[:400]}

    if world > 1:
        tt = torch.tensor([ms, e2e_ms], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms, e2e_ms = tt[0].item(), tt[1].item()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    value = world * n_img * args.steps / (ms / 1e3)
    e2e_value = world * n_img * args.steps / (e2e_ms / 1e3)
    out = {
        'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': args.act_dtype, 'data': 'synthetic',
        'config': {'workload': WORKLOAD,
                   'precision': ('fp16 tensor-core operands (weights + activations), fp32 accumulation / statistics / softmax: '
                                 'the reference\'s own sampling precision (README.md:146 torch_dtype=float16); same tcgen05 '
                                 'kind::f16 rate as bf16.  bf16 operands (--act-dtype bf16) run at the same speed but miss the '
                                 '1e-3 latent tolerance at guidance 7.5 (2.8e-3)') if args.act_dtype == 'fp16' else
                                'bf16 operands, fp32 accumulation', 'parallelism': f'replicas x{world} (independent images per GPU, no data-path '
                   'collective; SURVEY.md 8e)', 'l2': 'inputs larger than L2: 1.72 GB of 16-bit weights streamed per '
                   'step vs 126 MB L2, no explicit flush', 'cuda_graph': bool(used_graph), 'images_per_step': n_img},
        'clocks': clocks,
        'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                'ms_per_step': e2e_ms / args.steps,
                'api': "EDLoRAPipeline.__call__(prompt_embeds=, negative_prompt_embeds=, latents=, num_inference_steps=steps, "
                       "guidance_scale=7.5, output_type='latent', callback=) on pinned HOST tensors; one call of `steps` steps",
                'h2d_bytes_per_call': per_call_h2d},
        'gpu_launches': launches,
        'step_tflops': FLOPS_PER_STEP * value / world / 1e12 if not args.tiny else None,   # per GPU, all images
    }
    if train is not None:
        out['extra'] = {'train': train}
    if roof is not None:
        frac = roof['achieved'] / peaks['tflops']
        out['roofline'] = {'bound': 'tensor', 'achieved': roof['achieved'], 'peak': peaks['tflops'], 'unit': 'TFLOP/s',
                           'frac': frac, **gemm_traffic(),
                           'method': 'T(graph step) - T(graph step without gemm launches), CUDA events',
                           'peak_source': peaks['src'] + ' (bf16_tflops_sustained)',
                           'kernel': 'mos::gemm_kernel (tcgen05 GEMM + implicit-GEMM conv3x3)',
                           'launches_per_step': roof['launches'], 'kernel_ms_per_step': roof['ms'],
                           'algorithmic_gflop_per_step': roof['gflop']}
    if world == 1 and not args.no_cpu_baseline and n_img == 1:
        unet = build_cpu_reference(sd, lora, cfg)
        done, secs = cpu_reference_steps(unet, lora, lat, ehs, 2, 1, budget_s=60.0)
        out['cpu_baseline'] = {'value': done / secs, 'unit': UNIT, 'cores': CPU_THREADS, 'host_cpus': os.cpu_count(),
                               'kind': 'port',
                               'sample': f'{done} full CFG denoise steps (same workload, fp32 oracle) after 1 warm-up'}
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


def synthetic_clip_state(n_new_tokens=32, seed=11):
    """Random-init CLIP text encoder at the SD1.5 sizes (12 layers, width 768, 12 heads, 49408 tokens + the new-concept rows),
    transformers parameter names; init scales of transformers' CLIPTextModel (N(0, 0.02) embeddings / projections)."""
    import torch
    g = torch.Generator().manual_seed(seed)
    C, I, L = 768, 3072, 12
    sd = {'text_model.embeddings.token_embedding.weight': torch.randn(49408 + n_new_tokens, C, generator=g) * 0.02,
          'text_model.embeddings.position_embedding.weight': torch.randn(77, C, generator=g) * 0.02,
          'text_model.final_layer_norm.weight': torch.ones(C), 'text_model.final_layer_norm.bias': torch.zeros(C)}
    for i in range(L):
        p = f'text_model.encoder.layers.{i}.'
        for n in ('layer_norm1', 'layer_norm2'):
            sd[p + n + '.weight'], sd[p + n + '.bias'] = torch.ones(C), torch.zeros(C)
        for n in ('q_proj', 'k_proj', 'v_proj', 'out_proj'):
            sd[p + f'self_attn.{n}.weight'] = torch.randn(C, C, generator=g) * C ** -0.5 * 0.6
            sd[p + f'self_attn.{n}.bias'] = torch.zeros(C)
        sd[p + 'mlp.fc1.weight'], sd[p + 'mlp.fc1.bias'] = torch.randn(I, C, generator=g) * C ** -0.5 * 0.6, torch.zeros(I)
        sd[p + 'mlp.fc2.weight'], sd[p + 'mlp.fc2.bias'] = torch.randn(C, I, generator=g) * I ** -0.5 * 0.6, torch.zeros(C)
    return sd


def train_leg(args, rank, world, dev, sd, lora, cfg, outputs=None):
    """BASELINE config 5 (config 2 at N = 1): data-parallel ED-LoRA training, the path that actually shards.  Every rank runs
    the captured step of `EDLoRATrainer.forward` + `loss.backward()` (trainer_edlora.py:218-261, train_edlora.py:120-123) on
    ITS shard of the global batch (per-GPU batch fixed: weak scaling): CLIP text encoder forward (16 layer-wise prompts per
    sample, CLIPAttention LoRA) -> UNet forward (Attention LoRA) -> masked MSE + attention regulariser -> UNet backward ->
    CLIP backward; then the step's ONE collective - an NCCL all-reduce (sum, fp32) of the flat gradient buffer [32 concept
    embedding rows | CLIP LoRA | UNet LoRA | loss, Norm_mean] - then the fused flat AdamW on the three learning-rate groups
    and the LoRA re-pack (train_edlora.py:57,105-158; SURVEY.md 8e).  The VAE encoder runs upstream (latents in).  Timed
    with CUDA events, max over ranks; the all-reduce alone is timed separately.  `outputs`, when given, receives the
    trainable parameters and the loss after the last timed step."""
    import math

    import torch
    import torch.distributed as dist
    from mos_b200 import dp
    from mos_b200.clip_train_engine import CLIPTrainEngine
    from mos_b200.train_engine import TrainEngine
    kw = dict(block_out=cfg['block_out_channels'], layers=cfg['layers_per_block']) if cfg else {}
    B = args.train_batch
    tsd = synthetic_clip_state()
    g0 = torch.Generator().manual_seed(12)
    tlora = {}
    for i in range(12):
        for pj in ('q_proj', 'k_proj', 'v_proj', 'out_proj'):
            m = f'text_model.encoder.layers.{i}.self_attn.{pj}'
            tlora[m + '.lora_down.weight'] = (torch.rand(4, 768, generator=g0) * 2 - 1) / math.sqrt(768)
            tlora[m + '.lora_up.weight'] = torch.randn(768, 4, generator=g0) * 0.02
    concept_ids = list(range(49408, 49408 + 32))
    n_text = CLIPTrainEngine.lora_param_count(12, 768, 960)
    n_unet = sum(v.numel() for v in lora.values())
    state = dp.FlatTrainState(len(concept_ids), 768, n_text, n_unet, lrs=(1e-3, 1e-5, 1e-4), device=dev)
    eng = TrainEngine(sd, B, 64, 64, lora=lora, attn_reg_weight=0.01, reg_full_identity=False, state=state,
                      state_offset=state.group_end[1], text_grad=True, device=dev, **kw)
    nx = len(eng.xattn_names)
    text = CLIPTrainEngine(tsd, nx * B, lora=tlora, lora_alpha=1.0, concept_token_ids=concept_ids, state=state, emb_offset=0,
                           lora_offset=state.group_end[0], device=dev)
    eng.attach_text_engine(text)
    g = torch.Generator().manual_seed(100 + rank)              # per-rank data (train_edlora.py:48,70)
    x0 = torch.randn(B, 4, 64, 64, generator=g).to(dev)
    noise = torch.randn(B, 4, 64, 64, generator=g).to(dev)
    t = torch.randint(0, 1000, (B,), generator=g).to(dev)
    ids = torch.randint(1000, 40000, (nx, B, 77), generator=g)    # layer-major [16, B, 77]: BOS, 8 words incl. the two
    ids[:, :, 0] = 49406                                           # layer-wise concept tokens at positions 2 and 3, EOS padding
    ids[:, :, 9:] = 49407
    for l in range(nx):
        ids[l, :, 2], ids[l, :, 3] = concept_ids[l % 16], concept_ids[16 + l % 16]
    ids = ids.reshape(nx * B, 77)
    masks = torch.zeros(B, 1, 64, 64)
    masks[:, :, 8:56, 16:48] = 1.0                               # SURVEY.md 8d config 2
    masks = masks.to(dev)
    pos = [[2, 3]] * B

    def step():
        out = eng.forward_backward(x0, noise, t, None, masks, token_pos=pos, text_ids=ids)
        scale = dp.allreduce_flat_device(state, out[0:1])
        dp.optimizer_step(state, scale)
        eng.refresh_lora()
        text.refresh_lora()

    def sync():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    steps, warm = args.steps, 3
    for _ in range(warm):
        step()
    sync()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    sync()
    ms = e0.elapsed_time(e1) / steps
    if outputs is not None:
        outputs['train_params'] = state.params.clone()
        outputs['train_loss'] = state.grads[state.n:state.n + 1] / world
    # the collective alone (same buffer size, back to back)
    a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    scratch = state.grads.clone()
    reps = 20
    a0.record()
    for _ in range(reps):
        if world > 1:
            dist.all_reduce(scratch, op=dist.ReduceOp.SUM)
    a1.record()
    sync()
    ar_us = a0.elapsed_time(a1) / reps * 1e3 if world > 1 else 0.0
    # replicas must hold bit-identical parameters after the steps (same init, same reduced gradient on every rank)
    identical = True
    tt = torch.tensor([ms, ar_us], device=dev)
    if world > 1:
        hi, lo = state.params.clone(), state.params.clone()
        dist.all_reduce(hi, op=dist.ReduceOp.MAX)
        dist.all_reduce(lo, op=dist.ReduceOp.MIN)
        identical = bool(torch.equal(hi, lo))
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    ms, ar_us = tt[0].item(), tt[1].item()
    loss = state.grads[state.n].item() / world
    # SURVEY.md 8d: UNet fwd + dX-only bwd + LoRA dW = 1.61 TFLOP, CLIP x16 sequences fwd + bwd = 0.42 TFLOP per sample
    per_sample_tflop = 1.61 + 0.42 if not cfg else None
    return {'metric': 'ED-LoRA train samples/sec (train_edlora step: CLIP text encoder x16 + SD1.5 UNet @512x512, bf16; text-'
                      'embedding rows, CLIPAttention LoRA and UNet Attention LoRA trained; forward + masked MSE + attention '
                      'regulariser + backward + all-reduce + AdamW)',
            'value': B * world / ms * 1e3, 'unit': 'samples/s', 'n_gpus': world, 'ms_per_step': ms, 'steps': steps,
            'warmup': warm, 'batch_per_gpu': B, 'global_batch': B * world, 'scaling': 'weak',
            'collective': 'ONE NCCL all-reduce (sum, fp32) of the flat gradient buffer per optimiser step',
            'allreduce_bytes_per_step': (state.n + 2) * 4, 'allreduce_us': ar_us,
            'trainable_params': {'embedding_rows': len(concept_ids) * 768, 'clip_lora_padded': n_text, 'unet_lora': n_unet},
            'params_bit_identical_across_ranks': identical, 'mean_loss': loss,
            'step_tflops_per_gpu': (per_sample_tflop * B / (ms * 1e-3)) if per_sample_tflop else None,
            'kernel_launches_per_step': eng.launches + text.launches,
            'data': 'synthetic (per-rank seeds): latents, token ids, masks; VAE encode upstream'}


def gemm_traffic():
    """`roofline.traffic`: dram__bytes_read.sum + dram__bytes_write.sum per launch of mos::gemm_kernel, read from the
    committed summary of the round's `ncu --set full` capture (profiles/r2_kernels_summary.json, written by
    tools/ncu_summary.py from the .ncu-rep) - not a literal in this file.  null when the summary is absent."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'r2_kernels_summary.json')) as f:
            rows = [r for r in json.load(f)['kernels'] if 'gemm_kernel' in r['kernel']]
        vals = [r['dram_bytes'] for r in rows if r.get('dram_bytes') is not None]
        if not vals:
            return {'traffic': None}
        # algorithmic operand bytes of the captured launches (tools/ncu_targets.py, in launch order, two launches each): unique
        # A + W bytes read once; the 16-bit output tile normally stays in the 126 MB L2 within the capture window
        algo = {'conv3x3 8192x320x2880 (1-CTA)': (8192 * 320 + 320 * 2880) * 2, 'conv3x3 8192x320x2880 (CTA pair)': (8192 * 320 + 320 * 2880) * 2,
                '8192x320x320 +LoRA +residual': (8192 * 320 * 2 + 320 * 320 + 16 * 320) * 2, 'GEGLU 8192x2560x320': (8192 * 320 + 2560 * 320) * 2,
                'conv3x3 split-K 512x1280x11520': (512 * 1280 + 1280 * 11520) * 2}
        names = [n for n in algo for _ in range(2)]
        per = ', '.join(f"{n}: {r['dram_bytes'] / 1e6:.1f} MB measured / {algo[n] / 1e6:.1f} MB algorithmic"
                        for n, r in zip(names, rows) if r.get('dram_bytes') is not None) if len(rows) == len(names) else ''
        return {'traffic': sum(vals) / len(vals),
                'traffic_note': f'mean dram__bytes_read+write over the {len(vals)} gemm_kernel launches of the ncu --set full '
                                'capture of tools/ncu_targets.py: profiles/r2_kernels_summary.json' + ('; ' + per if per else '')}
    except Exception:
        return {'traffic': None}


def gemm_roofline(eng, ops, torch):
    """Device time of the dominant kernel family (mos::gemm_kernel: tcgen05 GEMM + implicit-GEMM conv) inside the
    real captured step, measured live with CUDA events on the launching stream as a difference of graph replays:
    T(full step) - T(same step without the gemm launches).  (Per-launch events in eager mode would time the Python
    launch path, not the kernel; nsys is not available.)  Algorithmic FLOPs = sum 2*M*N*K over the step's launches
    (LoRA rank columns, padding, split-K re-reads excluded)."""
    flops = []
    orig = ops.gemm

    def counting(A, W, out=None, **kw):
        conv = kw.get('conv')
        M = conv[0] * conv[1] * conv[2] if conv is not None else (kw.get('M') or A.shape[0])
        flops.append(2.0 * M * W.shape[0] * W.shape[1])
        return orig(A, W, out, **kw)

    ops.gemm = counting
    try:
        eng._run()
        torch.cuda.synchronize()
    finally:
        ops.gemm = orig
    launches, fl = len(flops), sum(flops)

    def replay_ms(skip, reps=20):
        eng.skip = set(skip)
        eng.graph = None
        eng.run()
        eng.run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            eng.run()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    t_full = replay_ms([])
    t_wo = replay_ms(['gemm'])
    eng.skip = set()
    eng.graph = None
    ms = max(t_full - t_wo, 1e-6)
    return {'achieved': fl / (ms * 1e-3) / 1e12, 'ms': ms, 'launches': launches, 'gflop': fl / 1e9,
            'step_ms_graph_only': t_full}


if __name__ == '__main__':
    main()
