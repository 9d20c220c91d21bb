// DenseNet plugin kernels (the reference's model/densenet.py, torchvision's _DenseLayer / _Transition), inference.
//   bn_relu               norm1 + relu1 of a dense layer: the first `channels` channels of the block's concatenation buffer, BN folded to
//                         scale/shift, ReLU, written fp16 into a scratch buffer whose extra channels up to `channels_padded` are zeros, so the
//                         bottleneck 1x1 conv reads a Cin that is a multiple of 32 against a zero-padded weight.
//   bn_relu_avgpool2x2    a transition's norm + relu + AvgPool2d(2, 2), the pool moved before the transition's 1x1 conv (a 1x1 conv is
//                         per-pixel linear, so pool(conv(a)) == conv(pool(a)) in real arithmetic; 4x fewer MMAs).
// The convs are yb_conv_bn_act_fwd; the stem and the max-pool are resnet_ops.cu's.
#include "yb_common.h"
#include <cuda_fp16.h>
#include <stdint.h>

namespace yb {

namespace {

constexpr int kThreads = 256;

// grid size of the grid-stride loops: enough CTAs to fill the GPU, few enough that each amortises its scale/shift load
unsigned grid_for(long long work) {
  const long long blocks = (work + kThreads - 1) / kThreads;
  const long long cap = static_cast<long long>(sm_count()) * 8;
  return static_cast<unsigned>(blocks < cap ? blocks : cap);
}

__device__ __forceinline__ float bn_relu1(float v, float s, float t) { return fmaxf(fmaf(v, s, t), 0.f); }

// scale[c..c+8) and shift[c..c+8) from shared memory
__device__ __forceinline__ void load_st8(const float* ss, int channels, int c, float (&s)[8], float (&t)[8]) {
  const float4 s0 = *reinterpret_cast<const float4*>(ss + c), s1 = *reinterpret_cast<const float4*>(ss + c + 4);
  const float4 t0 = *reinterpret_cast<const float4*>(ss + channels + c), t1 = *reinterpret_cast<const float4*>(ss + channels + c + 4);
  s[0] = s0.x; s[1] = s0.y; s[2] = s0.z; s[3] = s0.w; s[4] = s1.x; s[5] = s1.y; s[6] = s1.z; s[7] = s1.w;
  t[0] = t0.x; t[1] = t0.y; t[2] = t0.z; t[3] = t0.w; t[4] = t1.x; t[5] = t1.y; t[6] = t1.z; t[7] = t1.w;
}

__device__ __forceinline__ void load_scale_shift(float* ss, const float* __restrict__ scale, const float* __restrict__ shift, int channels) {
  for (int i = threadIdx.x; i < channels; i += blockDim.x) {
    ss[i] = __ldg(scale + i);
    ss[channels + i] = __ldg(shift + i);
  }
  __syncthreads();
}

}  // namespace

// one thread per 8 channels of one pixel; (pixel, channel group) advance by the grid stride without a division
__global__ void __launch_bounds__(kThreads) bn_relu_kernel(const __half* __restrict__ x, int x_ld, const float* __restrict__ scale,
                                                           const float* __restrict__ shift, __half* __restrict__ y, int y_ld, long long pixels,
                                                           int channels, int groups_padded) {
  extern __shared__ float ss[];            // [2][channels]: scale, shift
  load_scale_shift(ss, scale, shift, channels);
  const int groups = channels >> 3;
  const long long total = pixels * groups_padded;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  long long p = idx / groups_padded;
  int g = static_cast<int>(idx - p * groups_padded);
  const long long dp = stride / groups_padded;
  const int dg = static_cast<int>(stride - dp * groups_padded);
  for (; idx < total; idx += stride) {
    uint4 out = make_uint4(0u, 0u, 0u, 0u);
    if (g < groups) {
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(x + p * x_ld + g * 8));
      float s[8], t[8];
      load_st8(ss, channels, g * 8, s, t);
      const __half2* hv = reinterpret_cast<const __half2*>(&v);
      __half2* ho = reinterpret_cast<__half2*>(&out);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 f = __half22float2(hv[e]);
        ho[e] = __floats2half2_rn(bn_relu1(f.x, s[2 * e], t[2 * e]), bn_relu1(f.y, s[2 * e + 1], t[2 * e + 1]));
      }
    }
    *reinterpret_cast<uint4*>(y + p * y_ld + g * 8) = out;
    p += dp;
    g += dg;
    if (g >= groups_padded) { g -= groups_padded; ++p; }
  }
}

int bn_relu(const void* x, int x_ld, const float* scale, const float* shift, void* y, int y_ld, long long pixels, int channels, int channels_padded,
            cudaStream_t stream) {
  YB_REQUIRE(x && y && scale && shift && pixels > 0 && channels > 0, "bn_relu: bad argument");
  YB_REQUIRE(channels % 8 == 0 && x_ld % 8 == 0 && y_ld % 8 == 0 && channels_padded % 8 == 0,
             "bn_relu: channels=%d, channels_padded=%d, x_ld=%d, y_ld=%d must be multiples of 8", channels, channels_padded, x_ld, y_ld);
  YB_REQUIRE(channels_padded >= channels && x_ld >= channels && y_ld >= channels_padded,
             "bn_relu: channels=%d, channels_padded=%d, x_ld=%d, y_ld=%d", channels, channels_padded, x_ld, y_ld);
  YB_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(scale) & 15) == 0 && (reinterpret_cast<uintptr_t>(shift) & 15) == 0,
             "bn_relu: pointers must be 16B aligned");
  const int smem = 2 * channels * static_cast<int>(sizeof(float));
  YB_REQUIRE(smem <= 48 * 1024, "bn_relu: %d channels exceed the shared-memory scale/shift table", channels);
  const int groups_padded = channels_padded / 8;
  bn_relu_kernel<<<grid_for(pixels * groups_padded), kThreads, smem, stream>>>(static_cast<const __half*>(x), x_ld, scale, shift, static_cast<__half*>(y), y_ld,
                                                                              pixels, channels, groups_padded);
  return check_launch("bn_relu_kernel");
}

// y[b, oy, ox, c] = 0.25 * sum over the 2x2 window of relu(x * scale + shift), summed in fp32; one thread per 8 channels of one output pixel
__global__ void __launch_bounds__(kThreads) bn_relu_avgpool2x2_kernel(const __half* __restrict__ x, int x_ld, const float* __restrict__ scale,
                                                                      const float* __restrict__ shift, __half* __restrict__ y, int height, int width,
                                                                      int out_pixels, int channels) {
  extern __shared__ float ss[];
  load_scale_shift(ss, scale, shift, channels);
  const int groups = channels >> 3;
  const int oh = height >> 1, ow = width >> 1;
  const long long total = static_cast<long long>(out_pixels) * groups;
  const long long stride = static_cast<long long>(gridDim.x) * blockDim.x;
  long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  int q = static_cast<int>(idx / groups);
  int g = static_cast<int>(idx - static_cast<long long>(q) * groups);
  const int dq = static_cast<int>(stride / groups);
  const int dg = static_cast<int>(stride - static_cast<long long>(dq) * groups);
  for (; idx < total; idx += stride) {
    const int ox = q % ow;
    const int r = q / ow;                   // b * oh + oy
    const int oy = r % oh, b = r / oh;
    float s[8], t[8];
    load_st8(ss, channels, g * 8, s, t);
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[e] = 0.f;
#pragma unroll
    for (int dy = 0; dy < 2; ++dy) {
#pragma unroll
      for (int dx = 0; dx < 2; ++dx) {
        const long long pix = (static_cast<long long>(b) * height + 2 * oy + dy) * width + 2 * ox + dx;
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(x + pix * x_ld + g * 8));
        const __half2* hv = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __half22float2(hv[e]);
          acc[2 * e] += bn_relu1(f.x, s[2 * e], t[2 * e]);
          acc[2 * e + 1] += bn_relu1(f.y, s[2 * e + 1], t[2 * e + 1]);
        }
      }
    }
    uint4 out;
    __half2* ho = reinterpret_cast<__half2*>(&out);
#pragma unroll
    for (int e = 0; e < 4; ++e) ho[e] = __floats2half2_rn(0.25f * acc[2 * e], 0.25f * acc[2 * e + 1]);
    *reinterpret_cast<uint4*>(y + static_cast<long long>(q) * channels + g * 8) = out;
    q += dq;
    g += dg;
    if (g >= groups) { g -= groups; ++q; }
  }
}

int bn_relu_avgpool2x2(const void* x, int x_ld, const float* scale, const float* shift, void* y, int batch, int height, int width, int channels,
                       cudaStream_t stream) {
  YB_REQUIRE(x && y && scale && shift && batch > 0 && channels > 0, "bn_relu_avgpool2x2: bad argument");
  YB_REQUIRE(height >= 2 && width >= 2, "bn_relu_avgpool2x2: %dx%d input has no 2x2 window", height, width);
  YB_REQUIRE(channels % 8 == 0 && x_ld % 8 == 0 && x_ld >= channels, "bn_relu_avgpool2x2: channels=%d, x_ld=%d must be multiples of 8", channels, x_ld);
  YB_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0 &&
                 (reinterpret_cast<uintptr_t>(scale) & 15) == 0 && (reinterpret_cast<uintptr_t>(shift) & 15) == 0,
             "bn_relu_avgpool2x2: pointers must be 16B aligned");
  const int smem = 2 * channels * static_cast<int>(sizeof(float));
  YB_REQUIRE(smem <= 48 * 1024, "bn_relu_avgpool2x2: %d channels exceed the shared-memory scale/shift table", channels);
  const long long out_pixels = static_cast<long long>(batch) * (height / 2) * (width / 2);
  YB_REQUIRE(out_pixels * (channels / 8) < (1ll << 31), "bn_relu_avgpool2x2: too many outputs");
  bn_relu_avgpool2x2_kernel<<<grid_for(out_pixels * (channels / 8)), kThreads, smem, stream>>>(
      static_cast<const __half*>(x), x_ld, scale, shift, static_cast<__half*>(y), height, width, static_cast<int>(out_pixels), channels);
  return check_launch("bn_relu_avgpool2x2_kernel");
}

}  // namespace yb
