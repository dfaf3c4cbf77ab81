"""Drop-in for the adapters the reference attaches to its regional pipeline (diffusers `T2IAdapter`, loaded at
regionally_controlable_sampling.py:62-63 and called at mixofshow/pipelines/pipeline_regionally_t2iadapter.py:474-482):
same constructor arguments, diffusers parameter names, `from_pretrained` from a local directory, and `adapter(x)` returning
one fp32 NCHW feature map per level — running on `mos_b200.adapter_engine.AdapterEngine` (fp16 weights, inference only:
the adapters are frozen in every reference workflow).  Only adapter_type='full_adapter' (both sd14v1 checkpoints) exists."""
import math
from types import SimpleNamespace

import torch


def param_shapes(in_channels, channels, num_res_blocks, downscale_factor):
    """diffusers key -> shape of every parameter of a 'full_adapter' T2IAdapter."""
    shapes = {'adapter.conv_in.weight': (channels[0], in_channels * downscale_factor ** 2, 3, 3),
              'adapter.conv_in.bias': (channels[0],)}
    for i, c in enumerate(channels):
        if i > 0 and channels[i - 1] != c:
            shapes[f'adapter.body.{i}.in_conv.weight'] = (c, channels[i - 1], 1, 1)
            shapes[f'adapter.body.{i}.in_conv.bias'] = (c,)
        for j in range(num_res_blocks):
            p = f'adapter.body.{i}.resnets.{j}'
            shapes.update({p + '.block1.weight': (c, c, 3, 3), p + '.block1.bias': (c,),
                           p + '.block2.weight': (c, c, 1, 1), p + '.block2.bias': (c,)})
    return shapes


class T2IAdapter:
    def __init__(self, in_channels=3, channels=(320, 640, 1280, 1280), num_res_blocks=2, downscale_factor=8,
                 adapter_type='full_adapter', device='cuda'):
        if adapter_type != 'full_adapter':
            raise ValueError(f"T2IAdapter: adapter_type={adapter_type!r} is not supported (only 'full_adapter')")
        channels = [int(c) for c in channels]
        if not channels or any(c <= 0 or c % 160 for c in channels):
            raise ValueError(f'T2IAdapter: channels={channels} must be positive multiples of 160 (the GEMM tile width)')
        if (in_channels * downscale_factor ** 2) % 64:
            raise ValueError(f'T2IAdapter: in_channels * downscale_factor^2 = {in_channels * downscale_factor ** 2} must be '
                             'a multiple of 64 (the GEMM k block)')
        self.config = SimpleNamespace(in_channels=in_channels, channels=channels, num_res_blocks=num_res_blocks,
                                      downscale_factor=downscale_factor, adapter_type=adapter_type)
        self.device = torch.device(device)
        self.dtype = torch.float16
        # PyTorch's default Conv2d initialisation (diffusers constructs the modules the same way)
        self._sd = {}
        for k, shape in param_shapes(in_channels, channels, num_res_blocks, downscale_factor).items():
            fan_in = math.prod(shape[1:]) if k.endswith('.weight') else math.prod(self._sd[k[:-4] + 'weight'].shape[1:])
            self._sd[k] = torch.empty(shape).uniform_(-fan_in ** -0.5, fan_in ** -0.5)
        self._engine = None

    @classmethod
    def from_pretrained(cls, pretrained_model_name_or_path, torch_dtype=None, **kw):
        """diffusers call shape (regionally_controlable_sampling.py:62-63); the path must be a local directory."""
        from mixofshow.utils.model_io import load_t2i_adapter
        return load_t2i_adapter(pretrained_model_name_or_path, **{k: v for k, v in kw.items() if k == 'device'})

    def to(self, *a, **k):
        return self

    def eval(self):
        return self

    def state_dict(self):
        return dict(self._sd)

    def parameters(self):
        return iter(self._sd.values())

    def load_state_dict(self, state_dict, strict=True):
        c = self.config
        want = param_shapes(c.in_channels, c.channels, c.num_res_blocks, c.downscale_factor)
        missing, unexpected = sorted(set(want) - set(state_dict)), sorted(set(state_dict) - set(want))
        if missing or unexpected:
            raise KeyError(f'T2IAdapter.load_state_dict: missing {missing[:4]}, unexpected {unexpected[:4]}')
        bad = [k for k, s in want.items() if tuple(state_dict[k].shape) != s]
        if bad:
            raise ValueError(f'T2IAdapter.load_state_dict: shape mismatch at {bad[:4]}')
        self._sd = {k: state_dict[k].detach().to('cpu', torch.float32).clone() for k in want}
        self._engine = None

    def _get_engine(self):
        if self._engine is None:
            from mos_b200.adapter_engine import AdapterEngine
            c = self.config
            self._engine = AdapterEngine(self._sd, in_channels=c.in_channels, channels=c.channels,
                                         num_res_blocks=c.num_res_blocks, downscale_factor=c.downscale_factor,
                                         device=self.device)
        return self._engine

    @torch.no_grad()
    def __call__(self, x):
        """x [B, in_channels, H, W] in [0, 1] -> [fp32 NCHW [B, channels[l], h_l, w_l] for each level] on the device."""
        eng = self._get_engine()
        feats = eng.forward(x)
        B = x.shape[0]
        h, w = x.shape[2] // self.config.downscale_factor, x.shape[3] // self.config.downscale_factor
        out = []
        for l, f in enumerate(feats):
            if l > 0:
                h, w = (h + 1) // 2, (w + 1) // 2
            out.append(f.view(B, h, w, -1).permute(0, 3, 1, 2).to(torch.float32, memory_format=torch.contiguous_format))
        return out

    forward = __call__
