"""AdapterEngine — the T2I-Adapter ('full_adapter', diffusers T2IAdapter) on B200, built only from libmos_sm100 kernels.
Owns the call the reference makes once per condition image:

    keypose_adapter_state = self.keypose_adapter(keypose_input)     mixofshow/pipelines/pipeline_regionally_t2iadapter.py:474-482

PixelUnshuffle(f) writes the NHWC rows conv_in reads (mos_pixel_unshuffle); every 3x3 convolution is the implicit-GEMM conv
of mos_gemm_bf16 (resnet block1 with the ReLU epilogue), every 1x1 convolution a plain GEMM (block2 with the residual
epilogue), and the level change is mos_avgpool2x2 (ceil mode).  Activations and weights are fp16, accumulation fp32.
No CPU / PyTorch fallback: every arithmetic op is a C-ABI call.
"""
import torch

from . import ops

F16 = torch.float16
F32 = torch.float32


class AdapterEngine:
    def __init__(self, state_dict, *, in_channels=3, channels=(320, 640, 1280, 1280), num_res_blocks=2, downscale_factor=8,
                 device='cuda'):
        """state_dict: diffusers-named tensors of T2IAdapter (`adapter.conv_in.*`, `adapter.body.{i}...`).  Weights are
        packed once; activation buffers are allocated per input shape (B, H, W) on first use."""
        self.dev = torch.device(device)
        self.cin, self.ch, self.nres, self.f = in_channels, tuple(channels), num_res_blocks, downscale_factor
        self.K0 = in_channels * downscale_factor ** 2
        assert self.K0 % ops.BK == 0 and all(c % ops.BN == 0 for c in self.ch)
        self.w, self.bufs = {}, {}
        self.launches = 0
        self._pack('conv_in', state_dict, 'adapter.conv_in')
        for i, c in enumerate(self.ch):
            if i > 0 and self.ch[i - 1] != c:
                self._pack(f'{i}.in_conv', state_dict, f'adapter.body.{i}.in_conv')
            for j in range(self.nres):
                for b in ('block1', 'block2'):
                    self._pack(f'{i}.{j}.{b}', state_dict, f'adapter.body.{i}.resnets.{j}.{b}')

    def _pack(self, key, sd, name):
        """Conv2d [N, C, k, k] -> fp16 [N, k*k*C] (3x3 tap-major: column (kh*3 + kw)*C + c; 1x1: [N, C]) + fp32 bias."""
        W = sd[name + '.weight'].detach().to(self.dev, F32)
        self.w[key] = {'W': W.permute(0, 2, 3, 1).reshape(W.shape[0], -1).to(F16).contiguous(),
                       'bias': sd[name + '.bias'].detach().to(self.dev, F32).contiguous()}

    def buf(self, key, name, shape):
        k = (key, name)
        if k not in self.bufs:
            self.bufs[k] = torch.empty(shape, device=self.dev, dtype=F16)
        return self.bufs[k]

    def gemm(self, A, key, out, **kw):
        ent = self.w[key]
        ops.gemm(A, ent['W'], out, bias=ent['bias'], **kw)
        self.launches += 1
        return out

    @torch.no_grad()
    def forward(self, images):
        """images [B, in_channels, H, W] in [0, 1] (H, W multiples of the downscale factor) -> one fp16 NHWC feature map
        [B*h_l*w_l, channels[l]] per level (h_0 = H/f, h_l = ceil(h_{l-1}/2)).  The maps are this engine's buffers for
        the shape: valid until the next call with the same (B, H, W)."""
        B, cin, H, W = images.shape
        if cin != self.cin:
            raise ValueError(f'T2I-Adapter: {cin} input channels, the adapter expects {self.cin}')
        if H % self.f or W % self.f:
            raise ValueError(f'T2I-Adapter: image size {H}x{W} must be a multiple of the downscale factor {self.f}')
        key = (B, H, W)
        self.launches = 0
        h, w = H // self.f, W // self.f
        x0 = self.buf(key, 'unshuffle', (B * h * w, self.K0))
        ops.pixel_unshuffle(images.to(self.dev, F32).contiguous(), x0, r=self.f)
        self.launches += 1
        x = self.gemm(x0, 'conv_in', self.buf(key, 'conv_in', (B * h * w, self.ch[0])), conv=(B, h, w, self.K0))
        feats = []
        for i, c in enumerate(self.ch):
            if i > 0:
                cp = self.ch[i - 1]
                h2, w2 = (h + 1) // 2, (w + 1) // 2
                pooled = self.buf(key, f'{i}.pool', (B * h2 * w2, cp))
                ops.avgpool2x2(x, pooled, B=B, H=h, W=w, C=cp)
                self.launches += 1
                h, w, x = h2, w2, pooled
                if cp != c:
                    x = self.gemm(x, f'{i}.in_conv', self.buf(key, f'{i}.in_conv', (B * h * w, c)))
            M = B * h * w
            t = self.buf(key, f'{i}.t', (M, c))
            for j in range(self.nres):
                self.gemm(x, f'{i}.{j}.block1', t, conv=(B, h, w, c), act='relu')
                x = self.gemm(t, f'{i}.{j}.block2', self.buf(key, f'{i}.x{j % 2}', (M, c)), residual=x)
            feats.append(x)
        return feats
