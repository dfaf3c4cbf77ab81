"""ORACLE (test infrastructure, never imported by the product path).

Plain-PyTorch fp32 restatement of the T2I-Adapter the reference loads at regionally_controlable_sampling.py:62-63
(`T2IAdapter.from_pretrained('TencentARC/t2iadapter_openpose_sd14v1' | '..._sketch_sd14v1')`) and runs once per condition
image at mixofshow/pipelines/pipeline_regionally_t2iadapter.py:474-482: diffusers-0.19.3 `T2IAdapter` with
adapter_type='full_adapter' (the format of both sd14v1 checkpoints):

    PixelUnshuffle(f) -> conv_in (3x3, in_channels*f^2 -> channels[0])
    -> body[i]: [AvgPool2d(2, 2, ceil_mode=True) if i > 0] [in_conv 1x1 if the width changes]
                num_res_blocks x (x + block2(relu(block1(x))))   (block1 3x3, block2 1x1)
    -> one feature map per level.

Parameter names equal diffusers' (`adapter.conv_in.*`, `adapter.body.{i}.in_conv.*`, `adapter.body.{i}.resnets.{j}.block{1,2}.*`).

PARITY PINNING: diffusers is not installed here and the reference holds no golden vector for this network, so this
restatement of the published algorithm is "parity unpinned" against diffusers itself, exactly like oracle/unet.py and
oracle/vae.py.
"""
import torch
import torch.nn as nn
import torch.nn.functional as F

SD14_CHANNELS = (320, 640, 1280, 1280)


class AdapterResnetBlock(nn.Module):
    def __init__(self, channels):
        super().__init__()
        self.block1 = nn.Conv2d(channels, channels, 3, padding=1)
        self.block2 = nn.Conv2d(channels, channels, 1)

    def forward(self, x):
        return x + self.block2(F.relu(self.block1(x)))


class AdapterBlock(nn.Module):
    def __init__(self, cin, cout, num_res_blocks, down):
        super().__init__()
        self.down = down
        self.in_conv = nn.Conv2d(cin, cout, 1) if cin != cout else None
        self.resnets = nn.Sequential(*[AdapterResnetBlock(cout) for _ in range(num_res_blocks)])

    def forward(self, x):
        if self.down:
            x = F.avg_pool2d(x, 2, 2, ceil_mode=True)
        if self.in_conv is not None:
            x = self.in_conv(x)
        return self.resnets(x)


class FullAdapter(nn.Module):
    def __init__(self, in_channels=3, channels=SD14_CHANNELS, num_res_blocks=2, downscale_factor=8):
        super().__init__()
        self.f = downscale_factor
        self.conv_in = nn.Conv2d(in_channels * downscale_factor ** 2, channels[0], 3, padding=1)
        self.body = nn.ModuleList([AdapterBlock(channels[0], channels[0], num_res_blocks, False)] +
                                  [AdapterBlock(channels[i - 1], channels[i], num_res_blocks, True)
                                   for i in range(1, len(channels))])

    def forward(self, x):
        x = self.conv_in(F.pixel_unshuffle(x, self.f))
        feats = []
        for blk in self.body:
            x = blk(x)
            feats.append(x)
        return feats


class T2IAdapter(nn.Module):
    def __init__(self, in_channels=3, channels=SD14_CHANNELS, num_res_blocks=2, downscale_factor=8):
        super().__init__()
        self.adapter = FullAdapter(in_channels, channels, num_res_blocks, downscale_factor)

    def forward(self, x):
        return self.adapter(x)


def build_adapter(seed=0, in_channels=3, channels=SD14_CHANNELS, num_res_blocks=2, downscale_factor=8):
    """Seeded fp32 adapter with PyTorch's default Conv2d initialisation."""
    torch.manual_seed(seed)
    return T2IAdapter(in_channels, tuple(channels), num_res_blocks, downscale_factor).eval()
