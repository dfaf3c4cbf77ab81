// adapter.cu — the two layout kernels of the T2I-Adapter ('full_adapter', diffusers T2IAdapter) that the GEMM does not
// cover: PixelUnshuffle of the fp32 condition image straight into the NHWC rows conv_in reads, and the ceil-mode 2x2
// average pool between levels.  Both are bandwidth-bound glue run once per condition image.
#include "common.h"
#include "tc.cuh"

namespace mos {

#define STREAM(s) reinterpret_cast<cudaStream_t>(s)
static inline unsigned nblk(long long total, int threads) { return (unsigned)((total + threads - 1) / threads); }

// y[(b, ho, wo), c*r*r + i*r + j] = x[b, c, ho*r + i, wo*r + j]; one thread writes 8 consecutive output channels
template <bool F16>
__global__ void pixel_unshuffle_kernel(const float* __restrict__ x, int B, int C, int H, int W, int r,
                                       __nv_bfloat16* __restrict__ y, long long ldy) {
  pdl_wait();
  pdl_launch_dependents();
  const int Ho = H / r, Wo = W / r, Co = C * r * r, oct = Co / 8;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)B * Ho * Wo * oct) return;
  const int o = (int)(idx % oct);
  const long long pix = idx / oct;
  const int wo = (int)(pix % Wo);
  const int ho = (int)((pix / Wo) % Ho);
  const int b = (int)(pix / ((long long)Wo * Ho));
  float v[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = o * 8 + e;
    const int c = k / (r * r), i = (k / r) % r, j = k % r;
    v[e] = __ldg(x + (((long long)b * C + c) * H + ho * r + i) * W + wo * r + j);
  }
  uint4 u;
  u.x = pack16x2<F16>(v[0], v[1]);
  u.y = pack16x2<F16>(v[2], v[3]);
  u.z = pack16x2<F16>(v[4], v[5]);
  u.w = pack16x2<F16>(v[6], v[7]);
  *reinterpret_cast<uint4*>(y + pix * ldy + o * 8) = u;
}

// y[b, ho, wo, :] = mean of x[b, 2ho + {0,1}, 2wo + {0,1}, :] over the taps inside the input (ceil_mode, no padding)
template <bool F16>
__global__ void avgpool2x2_kernel(const __nv_bfloat16* __restrict__ x, long long ldx, int B, int H, int W, int C,
                                  __nv_bfloat16* __restrict__ y, long long ldy) {
  pdl_wait();
  pdl_launch_dependents();
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2, oct = C / 8;
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)B * Ho * Wo * oct) return;
  const int o = (int)(idx % oct);
  const long long pix = idx / oct;
  const int wo = (int)(pix % Wo);
  const int ho = (int)((pix / Wo) % Ho);
  const int b = (int)(pix / ((long long)Wo * Ho));
  const int nh = min(2, H - 2 * ho), nw = min(2, W - 2 * wo);
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int i = 0; i < nh; ++i)
    for (int j = 0; j < nw; ++j) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + (((long long)b * H + 2 * ho + i) * W + 2 * wo + j) * ldx + o * 8));
      const uint32_t w4[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = unpack16x2<F16>(w4[e]);
        acc[2 * e] += f.x;
        acc[2 * e + 1] += f.y;
      }
    }
  const float n = (float)(nh * nw);
  uint4 u;
  u.x = pack16x2<F16>(acc[0] / n, acc[1] / n);
  u.y = pack16x2<F16>(acc[2] / n, acc[3] / n);
  u.z = pack16x2<F16>(acc[4] / n, acc[5] / n);
  u.w = pack16x2<F16>(acc[6] / n, acc[7] / n);
  *reinterpret_cast<uint4*>(y + pix * ldy + o * 8) = u;
}

}  // namespace mos

using namespace mos;

extern "C" int mos_pixel_unshuffle(const float* x, int32_t B, int32_t C, int32_t H, int32_t W, int32_t r, void* y,
                                   int64_t ldy, int32_t act_dtype, void* stream) {
  MOS_CHECK_ARG(x && y && B > 0 && C > 0 && r > 0 && H > 0 && W > 0, "mos_pixel_unshuffle: bad arguments");
  MOS_CHECK_ARG(H % r == 0 && W % r == 0, "mos_pixel_unshuffle: H=%d and W=%d must be multiples of r=%d", H, W, r);
  MOS_CHECK_ARG((C * r * r) % 8 == 0 && ldy >= (int64_t)C * r * r && ldy % 8 == 0,
                "mos_pixel_unshuffle: C*r*r=%d must be a multiple of 8 and ldy=%lld >= it, a multiple of 8", C * r * r,
                (long long)ldy);
  MOS_CHECK_DTYPE(act_dtype, "mos_pixel_unshuffle");
  const long long total = (long long)B * (H / r) * (W / r) * (C * r * r / 8);
  MOS_CHECK_CUDA(launch_pdl(act_dtype ? pixel_unshuffle_kernel<true> : pixel_unshuffle_kernel<false>, dim3(nblk(total, 256)),
                            dim3(256), 0, STREAM(stream), x, (int)B, (int)C, (int)H, (int)W, (int)r,
                            reinterpret_cast<__nv_bfloat16*>(y), (long long)ldy));
  return MOS_OK;
}

extern "C" int mos_avgpool2x2(const void* x, int64_t ldx, int32_t B, int32_t H, int32_t W, int32_t C, void* y, int64_t ldy,
                              int32_t act_dtype, void* stream) {
  MOS_CHECK_ARG(x && y && B > 0 && H > 0 && W > 0 && C > 0, "mos_avgpool2x2: bad arguments");
  MOS_CHECK_ARG(C % 8 == 0 && ldx % 8 == 0 && ldy % 8 == 0 && ldx >= C && ldy >= C,
                "mos_avgpool2x2: C=%d, ldx=%lld, ldy=%lld must be multiples of 8 with ldx, ldy >= C", C, (long long)ldx,
                (long long)ldy);
  MOS_CHECK_DTYPE(act_dtype, "mos_avgpool2x2");
  const long long total = (long long)B * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8);
  MOS_CHECK_CUDA(launch_pdl(act_dtype ? avgpool2x2_kernel<true> : avgpool2x2_kernel<false>, dim3(nblk(total, 256)), dim3(256),
                            0, STREAM(stream), reinterpret_cast<const __nv_bfloat16*>(x), (long long)ldx, (int)B, (int)H,
                            (int)W, (int)C, reinterpret_cast<__nv_bfloat16*>(y), (long long)ldy));
  return MOS_OK;
}
