"""T2I-Adapter host logic without a GPU: the diffusers directory format, the oracle's parameter count, config rejections,
condition-image preprocessing, the entry script's condition validation and the C-ABI validation of the ReLU epilogue."""
import ctypes
import json
import math
import os

import numpy as np
import pytest
import torch
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))


def _args(extra):
    import regionally_controlable_sampling as rcs
    return rcs.parse_args(['--pretrained_model', '/nonexistent'] + extra)


def _png(path, size, mode='RGB'):
    Image.new(mode, size, 255 if mode == 'L' else (255, 255, 255)).save(path)
    return str(path)


def test_save_load_round_trip(tmp_path):
    from mixofshow.models.adapter_b200 import T2IAdapter
    from mixofshow.utils import model_io
    from oracle import adapter as oa
    ref = oa.build_adapter(3, in_channels=1, channels=(320, 640))
    a = T2IAdapter(in_channels=1, channels=[320, 640])
    a.load_state_dict(ref.state_dict())
    model_io.save_t2i_adapter(a, str(tmp_path))
    cfg = json.load(open(tmp_path / 'config.json'))
    assert cfg['adapter_type'] == 'full_adapter' and cfg['channels'] == [320, 640] and cfg['in_channels'] == 1
    assert cfg['num_res_blocks'] == 2 and cfg['downscale_factor'] == 8
    assert os.path.exists(tmp_path / 'diffusion_pytorch_model.safetensors')
    b = T2IAdapter.from_pretrained(str(tmp_path), torch_dtype=torch.float16)
    assert vars(b.config) == vars(a.config) and b.dtype == torch.float16 and b.to('cuda') is b
    sd, want = b.state_dict(), ref.state_dict()
    assert set(sd) == set(want)
    assert all(torch.equal(sd[k], want[k]) for k in want)


def test_parameter_counts():
    from mixofshow.models.adapter_b200 import T2IAdapter, param_shapes
    from oracle import adapter as oa
    for cin, n in ((3, 77_369_280), (1, 77_000_640)):
        assert sum(p.numel() for p in oa.build_adapter(0, cin).parameters()) == n
        shapes = param_shapes(cin, [320, 640, 1280, 1280], 2, 8)
        assert sum(math.prod(s) for s in shapes.values()) == n
    # the default-initialised drop-in carries the oracle's key set and shapes
    ref = oa.build_adapter(0, 1, channels=(320, 640, 640))
    a = T2IAdapter(in_channels=1, channels=[320, 640, 640])
    assert {k: tuple(v.shape) for k, v in a.state_dict().items()} == {k: tuple(v.shape) for k, v in ref.state_dict().items()}


def test_config_rejections(tmp_path):
    from mixofshow.models.adapter_b200 import T2IAdapter
    from mixofshow.utils import model_io
    with pytest.raises(ValueError, match='light_adapter'):
        T2IAdapter(adapter_type='light_adapter')
    with pytest.raises(ValueError, match='multiples of 160'):
        T2IAdapter(channels=[320, 600])
    with pytest.raises(ValueError, match='multiple of 64'):
        T2IAdapter(in_channels=1, downscale_factor=4)
    with pytest.raises(FileNotFoundError, match='local directory'):
        model_io.load_t2i_adapter('TencentARC/t2iadapter_openpose_sd14v1')
    json.dump({'adapter_type': 'light_adapter', 'channels': [320, 640, 1280], 'in_channels': 3}, open(tmp_path / 'config.json', 'w'))
    with pytest.raises(ValueError, match='light_adapter'):
        model_io.load_t2i_adapter(str(tmp_path))
    a = T2IAdapter(in_channels=1, channels=[320])
    with pytest.raises(KeyError):
        a.load_state_dict({k: v for k, v in a.state_dict().items() if 'block2' not in k})


def test_preprocess_adapter_image():
    from mixofshow.pipelines.pipeline_regionally_t2iadapter import _preprocess_adapter_image
    sketch = Image.open(os.path.join(HERE, 'golden', 'conditions', 'harry+catA+dogA_sketch.png'))
    L, rgb = sketch.convert('L'), sketch.convert('RGB')
    x = _preprocess_adapter_image(L, 96, 200)
    assert x.dtype == torch.float32 and tuple(x.shape) == (1, 1, 96, 200)
    exp = np.array(L.resize((200, 96), resample=Image.LANCZOS)).astype(np.float32) / 255.0
    assert torch.equal(x[0, 0], torch.from_numpy(exp))
    y = _preprocess_adapter_image(rgb, 96, 200)
    assert tuple(y.shape) == (1, 3, 96, 200) and 0 <= float(y.min()) and float(y.max()) <= 1
    exp = np.array(rgb.resize((200, 96), resample=Image.LANCZOS)).astype(np.float32) / 255.0
    assert torch.equal(y[0], torch.from_numpy(exp).permute(2, 0, 1))
    z = _preprocess_adapter_image([rgb, rgb.transpose(Image.FLIP_LEFT_RIGHT)], 96, 200)
    assert tuple(z.shape) == (2, 3, 96, 200) and torch.equal(z[0], y[0]) and torch.equal(z[1], y[0].flip(-1))
    t = torch.rand(1, 3, 64, 64)
    assert _preprocess_adapter_image(t, 96, 200) is t


def test_cli_conditions(tmp_path):
    import regionally_controlable_sampling as rcs
    pose = _png(tmp_path / 'pose.png', (256, 128))
    sketch = _png(tmp_path / 'sketch.png', (256, 128), 'L')
    other = _png(tmp_path / 'other.png', (128, 128))
    # '' and a missing file are skipped: the sampling size stays --height / --width
    conds, h, w = rcs.load_conditions(_args(['--sketch_condition', '', '--keypose_condition', str(tmp_path / 'no.png'),
                                             '--height', '64', '--width', '96']))
    assert conds == {'sketch': None, 'keypose': None} and (h, w) == (64, 96)
    conds, h, w = rcs.load_conditions(_args(['--sketch_condition', sketch, '--sketch_adapter', 'a',
                                             '--keypose_condition', pose, '--keypose_adapter', 'b']))
    assert conds['sketch'].mode == 'L' and conds['keypose'].mode == 'RGB' and (h, w) == (128, 256)
    with pytest.raises(ValueError, match='same size'):
        rcs.load_conditions(_args(['--sketch_condition', sketch, '--sketch_adapter', 'a',
                                   '--keypose_condition', other, '--keypose_adapter', 'b']))
    # refused by main() before any model is loaded or CUDA is touched
    with pytest.raises(ValueError, match='--keypose_adapter'):
        rcs.main(['--pretrained_model', '/nonexistent', '--keypose_condition', pose])
    with pytest.raises(ValueError, match='exclusive'):
        rcs.main(['--pretrained_model', '/nonexistent', '--sketch_condition', sketch, '--sketch_adapter', 'a',
                  '--sketch_adapter_state', 'state.pt'])


@pytest.fixture(scope='module')
def lib():
    import __graft_entry__ as g
    g.build()
    from mos_b200 import _lib
    return _lib.lib()


def test_gemm_act_field_and_validation(lib):
    """`act` is the trailing field of mos_gemm_args; the ReLU epilogue is refused with split-K / geglu / head-split / LoRA /
    fp32 output before any CUDA call."""
    from mos_b200 import _lib
    assert _lib.GemmArgs._fields_[-1] == ('act', ctypes.c_int32)
    assert _lib.GemmArgs.act.offset == _lib.GemmArgs.prefetch_bytes.offset + 8
    assert (_lib.MOS_ACT_NONE, _lib.MOS_ACT_RELU) == (0, 1)

    def args(**kw):
        a = _lib.GemmArgs()
        a.A, a.W, a.out, a.partial = 256, 256, 256, 256
        a.M, a.N, a.K, a.lda, a.ldc = 128, 160, 64, 64, 160
        a.a_dtype = a.w_dtype = _lib.MOS_DT_F16
        a.act = _lib.MOS_ACT_RELU
        for k, v in kw.items():
            setattr(a, k, v)
        return a

    for kw in (dict(splits=2), dict(geglu=1), dict(out_mode=_lib.MOS_OUT_HEADS, heads=1, head_dim=160, tokens_per_batch=128),
               dict(lora_down=256, lora_up=256, lora_seg=160), dict(out_mode=_lib.MOS_OUT_F32)):
        assert lib.mos_gemm_bf16(ctypes.byref(args(**kw)), None) == -1, kw
        assert b'act needs' in lib.mos_last_error(), kw
    assert lib.mos_gemm_bf16(ctypes.byref(args(act=7)), None) == -1 and b'MOS_ACT' in lib.mos_last_error()
