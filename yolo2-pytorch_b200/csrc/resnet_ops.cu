// ResNet plugin kernels (SURVEY 8f rank 4; /root/reference model/resnet.py:28-147), inference.  The stem and the max-pool are also
// DenseNet's (model/densenet.py:34-39): a 96-wide stem for densenet161, and the max-pool writes into a slice of the first dense block's buffer.
//   stem7x7     nn.Conv2d(3, 64, 7, stride 2, pad 3) + BatchNorm2d + ReLU (:107-109): fp32 NCHW image in, fp16 NHWC out -- the layout boundary.
//   maxpool3x3  nn.MaxPool2d(3, stride 2, pad 1) (:110) on fp16 NHWC.
//   subsample2  x[:, ::2, ::2, :]: a stride-2 conv with "same" padding equals its stride-1 form at the even pixels, so the three stride-2 3x3
//               convs and the 1x1 stride-2 downsample convs (:33,:39,:65,:73) run on the stride-1 tcgen05 kernel + this selection.
//   add_relu    out += residual; relu (:58-59, :100-101).
// The 3x3 / 1x1 convs themselves (with folded BN and ReLU or identity) are yb_conv_bn_act_fwd.
#include "yb_common.h"
#include <cuda_fp16.h>
#include <stdint.h>

namespace yb {

constexpr int kStemTaps = 147;

// one thread per output pixel, all kOut channels in registers; weights [tap][kOut] in shared memory (tap = ci*49 + r*7 + s).
// kOut = 64 is ResNet's and DenseNet-121/169/201's stem, 96 is DenseNet-161's.
template <int kOut>
__global__ void __launch_bounds__(128) stem7x7_kernel(const float* __restrict__ x, const float* __restrict__ w, const float* __restrict__ scale,
                                                      const float* __restrict__ shift, __half* __restrict__ y, int batch, int height, int width) {
  extern __shared__ float ws[];            // [147][kOut]
  for (int i = threadIdx.x; i < kStemTaps * kOut; i += blockDim.x) ws[i] = w[(i % kOut) * kStemTaps + i / kOut];
  __syncthreads();
  const int oh = height >> 1, ow = width >> 1;
  const long long total = static_cast<long long>(batch) * oh * ow;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int px = static_cast<int>(idx % ow);
  const long long t = idx / ow;
  const int py = static_cast<int>(t % oh);
  const long long img = t / oh;
  float acc[kOut];
#pragma unroll
  for (int i = 0; i < kOut; ++i) acc[i] = 0.f;
  for (int ci = 0; ci < 3; ++ci) {
    const float* xp = x + (img * 3 + ci) * height * width;
    for (int r = 0; r < 7; ++r) {
      const int iy = 2 * py - 3 + r;
      if (iy < 0 || iy >= height) continue;
#pragma unroll
      for (int s = 0; s < 7; ++s) {
        const int ix = 2 * px - 3 + s;
        const float v = (ix >= 0 && ix < width) ? __ldg(xp + static_cast<long long>(iy) * width + ix) : 0.f;
        const float4* wp = reinterpret_cast<const float4*>(ws + (ci * 49 + r * 7 + s) * kOut);
#pragma unroll
        for (int q = 0; q < kOut / 4; ++q) {
          const float4 wv = wp[q];
          acc[4 * q] = fmaf(v, wv.x, acc[4 * q]); acc[4 * q + 1] = fmaf(v, wv.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(v, wv.z, acc[4 * q + 2]); acc[4 * q + 3] = fmaf(v, wv.w, acc[4 * q + 3]);
        }
      }
    }
  }
  uint4* dst = reinterpret_cast<uint4*>(y + idx * kOut);
#pragma unroll
  for (int q = 0; q < kOut / 8; ++q) {
    uint4 pk;
    __half2* h = reinterpret_cast<__half2*>(&pk);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int c = q * 8 + 2 * e;
      h[e] = __floats2half2_rn(fmaxf(acc[c] * __ldg(scale + c) + __ldg(shift + c), 0.f), fmaxf(acc[c + 1] * __ldg(scale + c + 1) + __ldg(shift + c + 1), 0.f));
    }
    dst[q] = pk;
  }
}

template <int kOut>
static int stem7x7_launch(const float* x, const float* w, const float* scale, const float* shift, void* y, int batch, int height, int width,
                          cudaStream_t stream) {
  YB_REQUIRE(x && w && scale && shift && y && batch > 0 && height % 2 == 0 && width % 2 == 0, "stem7x7: bad argument");
  const int smem = kStemTaps * kOut * static_cast<int>(sizeof(float));
  static bool attr_set = false;
  if (!attr_set) {
    YB_CUDA(cudaFuncSetAttribute(stem7x7_kernel<kOut>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    attr_set = true;
  }
  const long long total = static_cast<long long>(batch) * (height / 2) * (width / 2);
  stem7x7_kernel<kOut><<<static_cast<unsigned>((total + 127) / 128), 128, smem, stream>>>(x, w, scale, shift, reinterpret_cast<__half*>(y), batch, height, width);
  return check_launch("stem7x7_kernel");
}

int stem7x7(const float* x, const float* w, const float* scale, const float* shift, void* y, int batch, int height, int width, cudaStream_t stream) {
  return stem7x7_launch<64>(x, w, scale, shift, y, batch, height, width, stream);
}

int stem7x7_96(const float* x, const float* w, const float* scale, const float* shift, void* y, int batch, int height, int width, cudaStream_t stream) {
  return stem7x7_launch<96>(x, w, scale, shift, y, batch, height, width, stream);
}

__device__ __forceinline__ uint4 hmax8_(uint4 a, uint4 b) {
  uint4 r;
  const __half2* pa = reinterpret_cast<const __half2*>(&a);
  const __half2* pb = reinterpret_cast<const __half2*>(&b);
  __half2* pr = reinterpret_cast<__half2*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) pr[i] = __hmax2(pa[i], pb[i]);
  return r;
}

// nn.MaxPool2d(kernel_size=3, stride=2, padding=1): out[oy, ox] = max over the in-range pixels of rows 2oy-1..2oy+1, columns 2ox-1..2ox+1,
// written to channels [y_ch_off, y_ch_off + channels) of an output whose pixels are y_ld channels apart
__global__ void maxpool3x3_s2_kernel(const __half* __restrict__ x, __half* __restrict__ y, int batch, int height, int width, int channels, int y_ld,
                                     int y_ch_off) {
  const int c8 = channels >> 3;
  const int oh = (height + 1) / 2, ow = (width + 1) / 2;
  const long long total = static_cast<long long>(batch) * oh * ow * c8;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int cg = static_cast<int>(idx % c8);
  long long t = idx / c8;
  const long long pix = t;
  const int px = static_cast<int>(t % ow); t /= ow;
  const int py = static_cast<int>(t % oh);
  const long long img = t / oh;
  bool any = false;
  uint4 m = make_uint4(0u, 0u, 0u, 0u);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const int iy = 2 * py - 1 + r;
    if (iy < 0 || iy >= height) continue;
#pragma unroll
    for (int s = 0; s < 3; ++s) {
      const int ix = 2 * px - 1 + s;
      if (ix < 0 || ix >= width) continue;
      const uint4 v = __ldg(reinterpret_cast<const uint4*>(x + ((img * height + iy) * width + ix) * channels + cg * 8));
      m = any ? hmax8_(m, v) : v;
      any = true;
    }
  }
  *reinterpret_cast<uint4*>(y + pix * y_ld + y_ch_off + cg * 8) = m;
}

int maxpool3x3_s2_strided(const void* x, void* y, int batch, int height, int width, int channels, int y_ld, int y_ch_off, cudaStream_t stream) {
  YB_REQUIRE(x && y && batch > 0 && height > 0 && width > 0 && channels > 0 && channels % 8 == 0, "maxpool3x3_s2: bad argument");
  YB_REQUIRE(y_ld % 8 == 0 && y_ch_off % 8 == 0 && y_ch_off >= 0 && y_ch_off + channels <= y_ld,
             "maxpool3x3_s2: y_ld=%d / y_ch_off=%d must be multiples of 8 holding %d channels", y_ld, y_ch_off, channels);
  YB_REQUIRE((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0, "maxpool3x3_s2: x/y must be 16B aligned");
  const long long total = static_cast<long long>(batch) * ((height + 1) / 2) * ((width + 1) / 2) * (channels / 8);
  maxpool3x3_s2_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(reinterpret_cast<const __half*>(x), reinterpret_cast<__half*>(y), batch, height,
                                                                                      width, channels, y_ld, y_ch_off);
  return check_launch("maxpool3x3_s2_kernel");
}

int maxpool3x3_s2(const void* x, void* y, int batch, int height, int width, int channels, cudaStream_t stream) {
  return maxpool3x3_s2_strided(x, y, batch, height, width, channels, channels, 0, stream);
}

// y[b, oy, ox, :] = x[b, 2oy, 2ox, :]
__global__ void subsample2_kernel(const __half* __restrict__ x, __half* __restrict__ y, int batch, int height, int width, int channels) {
  const int c8 = channels >> 3;
  const int oh = (height + 1) / 2, ow = (width + 1) / 2;
  const long long total = static_cast<long long>(batch) * oh * ow * c8;
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int cg = static_cast<int>(idx % c8);
  long long t = idx / c8;
  const int px = static_cast<int>(t % ow); t /= ow;
  const int py = static_cast<int>(t % oh);
  const long long img = t / oh;
  reinterpret_cast<uint4*>(y)[idx] = __ldg(reinterpret_cast<const uint4*>(x + ((img * height + 2 * py) * width + 2 * px) * channels + cg * 8));
}

int subsample2(const void* x, void* y, int batch, int height, int width, int channels, cudaStream_t stream) {
  YB_REQUIRE(x && y && batch > 0 && height > 0 && width > 0 && channels % 8 == 0, "subsample2: bad argument");
  const long long total = static_cast<long long>(batch) * ((height + 1) / 2) * ((width + 1) / 2) * (channels / 8);
  subsample2_kernel<<<static_cast<unsigned>((total + 255) / 256), 256, 0, stream>>>(reinterpret_cast<const __half*>(x), reinterpret_cast<__half*>(y), batch, height, width,
                                                                                   channels);
  return check_launch("subsample2_kernel");
}

// out = relu(a + b), fp16, fp32 add, 8 elements per thread
__global__ void add_relu_kernel(const uint4* __restrict__ a, const uint4* __restrict__ b, uint4* __restrict__ out, long long n8) {
  const long long idx = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= n8) return;
  const uint4 va = __ldg(a + idx), vb = __ldg(b + idx);
  const __half2* pa = reinterpret_cast<const __half2*>(&va);
  const __half2* pb = reinterpret_cast<const __half2*>(&vb);
  uint4 r;
  __half2* pr = reinterpret_cast<__half2*>(&r);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 fa = __half22float2(pa[i]), fb = __half22float2(pb[i]);
    pr[i] = __floats2half2_rn(fmaxf(fa.x + fb.x, 0.f), fmaxf(fa.y + fb.y, 0.f));
  }
  out[idx] = r;
}

int add_relu(const void* a, const void* b, void* out, long long count, cudaStream_t stream) {
  YB_REQUIRE(a && b && out && count > 0 && count % 8 == 0, "add_relu: count must be a positive multiple of 8");
  const long long n8 = count / 8;
  add_relu_kernel<<<static_cast<unsigned>((n8 + 255) / 256), 256, 0, stream>>>(static_cast<const uint4*>(a), static_cast<const uint4*>(b), static_cast<uint4*>(out), n8);
  return check_launch("add_relu_kernel");
}

}  // namespace yb
