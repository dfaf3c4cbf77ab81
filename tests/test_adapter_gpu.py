"""T2I-Adapter on the B200 against the fp32 oracle (oracle/adapter.py, run on the GPU with TF32 off): the two layout kernels,
the ReLU epilogue of the GEMM, the whole network at the sampling sizes of the reference, the regional pipeline fed with
condition images, and the entry script end to end.

Tolerances (rel-L2 = ||a-b|| / ||b||): pixel unshuffle bit-exact (a copy with one fp32 -> fp16 rounding); average pool
within 1 fp16 ulp (fp32 sum, one rounding); GEMM epilogue 6e-4 (fp16 operands, tests/test_gemm_gpu.py); adapter feature maps
5e-3 (fp16 operands through 21 layers; the VAE reaches 2.3e-3); 3-step pipeline latents 5e-3 (tests/test_regional_gpu.py)."""
import os

import pytest
import torch
import torch.nn.functional as F
from PIL import Image

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
COND = os.path.join(HERE, 'golden', 'conditions')


def rel_l2(a, b):
    a, b = a.float().cpu(), b.float().cpu()
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def _condition(kind, height, width, batch=1):
    """The reference's condition images resized to (height, width); batch 2 adds the mirrored image."""
    from mixofshow.pipelines.pipeline_regionally_t2iadapter import _preprocess_adapter_image
    img = Image.open(os.path.join(COND, f'harry+catA+dogA_{kind}.png')).convert('L' if kind == 'sketch' else 'RGB')
    imgs = [img, img.transpose(Image.FLIP_LEFT_RIGHT)][:batch]
    return _preprocess_adapter_image(imgs, height, width)


@pytest.mark.parametrize('C', [1, 3])
def test_pixel_unshuffle_bit_exact(cuda, C):
    from mos_b200 import ops
    B, H, W, r = 2, 48, 80, 8
    x = torch.rand(B, C, H, W, generator=torch.Generator().manual_seed(C)).to(cuda)
    K = C * r * r
    y = torch.full((B * (H // r) * (W // r), K + 64), 7.0, device=cuda, dtype=torch.float16)
    ops.pixel_unshuffle(x, y, r=r)
    ref = F.pixel_unshuffle(x, r).half().permute(0, 2, 3, 1).reshape(-1, K)
    assert torch.equal(y[:, :K].view(torch.int16), ref.view(torch.int16))
    assert bool((y[:, K:] == 7).all())                     # pitch columns untouched
    with pytest.raises(ValueError):
        ops.pixel_unshuffle(x[:, :, :44].contiguous(), y, r=r)


@pytest.mark.parametrize('H,W', [(8, 12), (7, 9), (5, 6), (1, 3)])
def test_avgpool2x2_ceil_mode(cuda, H, W):
    from mos_b200 import ops
    B, C, ld = 2, 320, 336
    x = torch.randn(B * H * W, ld, generator=torch.Generator().manual_seed(H * W)).to(cuda).half()
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    y = torch.zeros(B * Ho * Wo, ld, device=cuda, dtype=torch.float16)
    ops.avgpool2x2(x, y, B=B, H=H, W=W, C=C)
    xn = x[:, :C].float().view(B, H, W, C).permute(0, 3, 1, 2)
    ref = F.avg_pool2d(xn, 2, 2, ceil_mode=True).permute(0, 2, 3, 1).reshape(-1, C).half()
    ulp = (torch.nextafter(ref.abs(), torch.tensor(float('inf'), device=cuda, dtype=torch.float16)) - ref.abs()).float()
    err = (y[:, :C].float() - ref.float()).abs()
    print(f'avgpool {H}x{W}: max error {float((err / ulp).max()):.2f} ulp')
    assert bool((err <= ulp).all())


@pytest.mark.parametrize('residual', [False, True])
@pytest.mark.parametrize('kind', ['plain', 'plain_pair', 'conv64'])
def test_gemm_relu_epilogue(cuda, kind, residual):
    from mos_b200 import ops
    g = torch.Generator().manual_seed(11)
    N = 320
    if kind == 'conv64':                                  # adapter conv_in of a sketch: C = 1 * 8^2
        B, H, Wd, C = 2, 12, 20, 64
        x = torch.rand(B, H, Wd, C, generator=g).to(cuda).half()
        w = (torch.randn(N, C, 3, 3, generator=g) * (9 * C) ** -0.5).to(cuda).half()
        A, Wp, M = x, w.permute(0, 2, 3, 1).reshape(N, 9 * C).contiguous(), B * H * Wd
        acc = F.conv2d(x.float().permute(0, 3, 1, 2), w.float(), padding=1).permute(0, 2, 3, 1).reshape(M, N)
        kw = dict(conv=(B, H, Wd, C))
    else:
        M, K = 512, 640
        A = torch.randn(M, K, generator=g).to(cuda).half()
        Wp = (torch.randn(N, K, generator=g) * K ** -0.5).to(cuda).half()
        acc = A.float() @ Wp.float().t()
        kw = dict(pair_mode=1 if kind == 'plain_pair' else 2)
    bias = torch.randn(N, generator=g).to(cuda) * 0.5
    res = torch.randn(M, N, generator=g).to(cuda).half() if residual else None
    out = torch.empty(M, N, device=cuda, dtype=torch.float16)
    ops.gemm(A, Wp, out, bias=bias, residual=res, act='relu', **kw)
    ref = torch.relu(acc + bias) + (res.float() if residual else 0)
    e = rel_l2(out, ref)
    print(f'relu epilogue {kind} residual={residual}: rel-L2 {e:.2e}')
    assert e < 6e-4
    if not residual:
        assert float(out.min()) == 0.0


@pytest.mark.parametrize('size', [(512, 512, 2), (768, 1536, 1), (1024, 2048, 1), (288, 288, 1)],
                         ids=['512x512_b2', '768x1536', '1024x2048', '288x288'])
@pytest.mark.parametrize('cin', [1, 3])
def test_adapter_vs_oracle(cuda, cin, size):
    from mixofshow.models.adapter_b200 import T2IAdapter
    from oracle import adapter as oa
    height, width, B = size
    ref = oa.build_adapter(cin, in_channels=cin).to(cuda)
    ad = T2IAdapter(in_channels=cin)
    ad.load_state_dict(ref.state_dict())
    x = _condition('sketch' if cin == 1 else 'pose', height, width, B).to(cuda)
    with torch.no_grad():
        exp = ref(x)
    got = ad(x)
    errs = [rel_l2(a, b) for a, b in zip(got, exp)]
    print(f'adapter in={cin} {height}x{width} B={B}: launches {ad._engine.launches}, rel-L2 per level '
          + ', '.join(f'{e:.2e}' for e in errs))
    assert [tuple(t.shape) for t in got] == [tuple(t.shape) for t in exp]
    assert all(t.dtype == torch.float32 and t.is_cuda and t.is_contiguous() for t in got)
    assert max(errs) <= 5e-3
    if B == 2:      # distinct images stay distinct
        assert rel_l2(got[0][1], got[0][0]) > 1e-2


def test_pipeline_with_condition_images(cuda):
    """RegionallyT2IAdapterPipeline given PIL key-pose and sketch conditions and B200 adapters, against the same pipeline given
    the oracle adapters' feature maps of the preprocessed images as `*_adapter_state`."""
    from mixofshow.models.adapter_b200 import T2IAdapter
    from mixofshow.models.unet_b200 import UNet2DConditionModel
    from mixofshow.pipelines.pipeline_regionally_t2iadapter import RegionallyT2IAdapterPipeline, _preprocess_adapter_image
    from oracle import adapter as oa
    from oracle import unet as ou
    height, width = 192, 384
    h, w = height // 8, width // 8
    ref_unet = ou.build_unet(0, ou.TINY)
    unet = UNet2DConditionModel(block_out_channels=ou.TINY['block_out_channels'], layers_per_block=ou.TINY['layers_per_block'])
    unet.load_state_dict(ref_unet.state_dict())
    pipe = RegionallyT2IAdapterPipeline(unet=unet).to('cuda')
    pipe.set_new_concept_cfg({})
    refs = {k: oa.build_adapter(s, in_channels=c, channels=(320, 640)).to(cuda) for k, s, c in (('keypose', 21, 3), ('sketch', 22, 1))}
    for k, r in refs.items():
        a = T2IAdapter(in_channels=r.adapter.conv_in.in_channels // 64, channels=[320, 640])
        a.load_state_dict(r.state_dict())
        setattr(pipe, f'{k}_adapter', a)
    src = {k: Image.open(os.path.join(COND, f'harry+catA+dogA_{n}.png')).convert(m)
           for k, n, m in (('keypose', 'pose', 'RGB'), ('sketch', 'sketch', 'L'))}
    g = lambda s: torch.Generator().manual_seed(s)
    lat = torch.randn(1, 4, h, w, generator=g(3))
    ehs = torch.randn(2, 16, 77, 768, generator=g(4))
    regs = [(torch.randn(2, 16, 77, 768, generator=g(5 + i)).cuda(), b)
            for i, b in enumerate([(0.0, 0.0, 1.0, 0.45), (0.0, 0.5, 1.0, 1.0)])]
    common = dict(prompt_embeds=ehs.cuda(), region_list=regs, height=height, width=width, num_inference_steps=3,
                  guidance_scale=7.5, output_type='latent', keypose_adaptor_weight=0.8, sketch_adaptor_weight=0.6,
                  region_sketch_adaptor_weight='[0,0,192,180]-1.3')

    def run(**kw):
        return pipe(latents=lat.clone(), **common, **kw).images

    got = run(keypose_adapter_input=[src['keypose']], sketch_adapter_input=[src['sketch']])
    with torch.no_grad():
        states = {k: refs[k](_preprocess_adapter_image([src[k]], height, width).to(cuda)) for k in refs}
    exp = run(keypose_adapter_state=states['keypose'], sketch_adapter_state=states['sketch'])
    e = rel_l2(got, exp)
    print(f'pipeline with condition images vs oracle adapter states: latents rel-L2 {e:.3e}')
    assert torch.isfinite(got).all() and e <= 5e-3
    other = run(keypose_adapter_input=[src['keypose']], sketch_adapter_input=[src['sketch'].transpose(Image.FLIP_TOP_BOTTOM)])
    moved = rel_l2(other, got)
    print(f'a different sketch moves the latents by rel-L2 {moved:.3e}')
    assert moved > 1e-3


def test_cli_end_to_end(cuda, tmp_path):
    import json

    import regionally_controlable_sampling as rcs
    from mixofshow.models.adapter_b200 import T2IAdapter
    from mixofshow.models.vae_b200 import AutoencoderKL
    from mixofshow.utils import model_io
    from oracle import adapter as oa
    from oracle import vae as ov
    from synth import make_pretrained_dir
    base = make_pretrained_dir(str(tmp_path / 'base'), with_vae=False)
    json.dump({}, open(os.path.join(base, 'new_concept_cfg.json'), 'w'))
    # a VAE with SD1.5's scale factor 8 (four levels) so that latents and adapter features line up
    vcfg = dict(block_out_channels=(128, 128, 128, 256), layers_per_block=1)
    vref = ov.build_vae(5, vcfg)
    model_io.save_vae(AutoencoderKL({k: v.detach() for k, v in vref.state_dict().items()}, device='cpu', **vcfg),
                      str(tmp_path / 'vae8'))
    dirs = {}
    for kind, cin, seed in (('sketch', 1, 31), ('keypose', 3, 32)):
        a = T2IAdapter(in_channels=cin, channels=[320, 640])
        a.load_state_dict(oa.build_adapter(seed, in_channels=cin, channels=(320, 640)).state_dict())
        dirs[kind] = str(tmp_path / f'{kind}_adapter')
        model_io.save_t2i_adapter(a, dirs[kind])
    size = (256, 128)                                     # (width, height) of the conditions
    sk = Image.open(os.path.join(COND, 'harry+catA+dogA_sketch.png')).resize(size)
    sk.save(tmp_path / 'sketch.png')
    Image.open(os.path.join(COND, 'harry+catA+dogA_pose.png')).resize(size).save(tmp_path / 'pose.png')
    save = str(tmp_path / 'out')
    lat = rcs.main(['--pretrained_model', base, '--prompt', 'two animals', '--negative_prompt', 'blurry',
                    '--prompt_rewrite', '[a cat]-*-[blurry]-*-[0,0,128,120]|[a dog]-*-[blurry]-*-[0,130,128,256]',
                    '--sketch_condition', str(tmp_path / 'sketch.png'), '--sketch_adapter', dirs['sketch'],
                    '--keypose_condition', str(tmp_path / 'pose.png'), '--keypose_adapter', dirs['keypose'],
                    '--vae_model', str(tmp_path / 'vae8'), '--num_inference_steps', '3', '--save_dir', save,
                    '--seed', '9', '--suffix', 'e2e'])
    assert tuple(lat.shape) == (1, 4, 16, 32) and torch.isfinite(lat).all()
    assert os.path.exists(os.path.join(save, 'latents---9---e2e.pt')) and os.path.exists(os.path.join(save, 'config.json'))
    pngs = [f for f in os.listdir(os.path.join(save, 'seed_9')) if f.endswith('.png')]
    assert len(pngs) == 1 and pngs[0].startswith('two_animals---e2e---')
    assert Image.open(os.path.join(save, 'seed_9', pngs[0])).size == size
    txt = open(os.path.join(save, 'seed_9', pngs[0].replace('.png', '.txt'))).read()
    assert 'sketch_condition: ' + str(tmp_path / 'sketch.png') in txt and 'random seed: 9' in txt
