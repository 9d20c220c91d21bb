// Photometric training augmentations (the reference's transform/image.py:32-99, applied per resized image by utils/data.py:121)
// for a batch of same-size uint8 HWC frames in ONE launch, each image with its own parameters.  Stages, in this order, each optional:
//   1. box blur (kx, ky)      RandomBlur  (:42-49)  cv2.blur(img, (kx, ky)): anchor (kx / 2, ky / 2), BORDER_REFLECT_101
//   2. BGR -> HSV             BGR2HSV     (:32-34)  cv2 COLOR_BGR2HSV, 8-bit (H in 0..179)
//   3. per-channel table      RandomHue / RandomSaturation / RandomBrightness (:52-88), composed on the host
//   4. HSV -> RGB             HSV2RGB     (:37-39)  cv2 COLOR_HSV2RGB, 8-bit
//   5. per-channel table      RandomGamma (:91-98)
// Exactness contract (cv2 4.13, checked exhaustively against cv2 itself by the oracle, oracle/photometric.py):
//   blur: integer window sum S over area a = kx * ky, out = (S + a / 2) / a, except for a = 2, 4, 8, 16 where cv2's fixed-point
//         divide gives (S + a / 2 + 1) / a; saturated to 255.  The one intended difference: cv2 wraps an area-2 sum of 510 to 0 in
//         its scalar tail loop (white pixel pairs turn black depending on the row width); here it saturates to 255.
//   BGR2HSV: cv2's integer path with its 12-bit reciprocal tables sdiv[i] = rint((255 << 12) / i), hdiv[i] = rint((180 << 12) / 6i).
//   HSV2RGB: float32 in the operation order of cv2's per-pixel path -- h * (6 / 180), s and v * (1 / 255), sector = trunc(h),
//            f = h - sector, tab = {v, v(1 - s), v * fma(-s, f, 1), v * fma(-s, 1 - f, 1)}, then rint(x * 255).  cv2's vectorised
//            body truncates x * 255 instead (its result depends on where a pixel falls in the row); the rounding path is restated.
// Each block owns a TH x TW output tile of one image: the tile plus its blur halo is loaded once into shared memory with 16-byte
// loads (rows and columns reflected at the frame border), the separable box sums run in integers from shared memory, the image's
// tables are staged in shared memory, and the tile leaves through a shared-memory staging buffer with 16-byte stores.
#include "yb_common.h"
#include <stdint.h>

namespace yb {

namespace {

constexpr int kTW = 32, kTH = 32, kThreads = 256, kMaxK = 15;
constexpr int kInRows = kTH + kMaxK - 1;
constexpr int kInPitch = 160;   // >= (kTW + kMaxK - 1) * 3 + 15, rounded up to 16
constexpr int kOutPitch = 112;  // >= kTW * 3 + 15, rounded up to 16
constexpr int kColW = kTW + kMaxK - 1;

__device__ __forceinline__ int reflect101(int p, int n) {
  if (n == 1) return 0;
  while (p < 0 || p >= n) p = p < 0 ? -p : 2 * n - 2 - p;
  return p;
}

// Copy the bytes [g, g + len) of global memory into shared memory `s` laid out so that s[k] holds byte (g & ~15) + k: whole
// 16-byte chunks move as uint4, the partial chunks at either end byte by byte.  Only bytes inside the range are touched.
__device__ __forceinline__ void load_chunk(const uint8_t* g, int len, uint8_t* s, int chunk) {
  const uintptr_t a0 = reinterpret_cast<uintptr_t>(g) & ~static_cast<uintptr_t>(15);
  const uintptr_t lo = reinterpret_cast<uintptr_t>(g), hi = lo + len;
  const uintptr_t c = a0 + 16 * static_cast<uintptr_t>(chunk);
  if (c >= lo && c + 16 <= hi) {
    *reinterpret_cast<uint4*>(s + 16 * chunk) = *reinterpret_cast<const uint4*>(c);
  } else {
    for (int k = 0; k < 16; ++k)
      if (c + k >= lo && c + k < hi) s[16 * chunk + k] = *reinterpret_cast<const uint8_t*>(c + k);
  }
}

__device__ __forceinline__ void store_chunk(uint8_t* g, int len, const uint8_t* s, int chunk) {
  const uintptr_t a0 = reinterpret_cast<uintptr_t>(g) & ~static_cast<uintptr_t>(15);
  const uintptr_t lo = reinterpret_cast<uintptr_t>(g), hi = lo + len;
  const uintptr_t c = a0 + 16 * static_cast<uintptr_t>(chunk);
  if (c >= lo && c + 16 <= hi) {
    *reinterpret_cast<uint4*>(c) = *reinterpret_cast<const uint4*>(s + 16 * chunk);
  } else {
    for (int k = 0; k < 16; ++k)
      if (c + k >= lo && c + k < hi) *reinterpret_cast<uint8_t*>(c + k) = s[16 * chunk + k];
  }
}

__device__ __forceinline__ int chunks_of(const uint8_t* g, int len) {
  const uintptr_t a0 = reinterpret_cast<uintptr_t>(g) & ~static_cast<uintptr_t>(15);
  return static_cast<int>((reinterpret_cast<uintptr_t>(g) + len - a0 + 15) / 16);
}

__device__ __forceinline__ void bgr2hsv(int b, int g, int r, const int* sdiv, const int* hdiv, int& h, int& s, int& v) {
  v = max(max(b, g), r);
  const int diff = v - min(min(b, g), r);
  s = (diff * sdiv[v] + (1 << 11)) >> 12;
  int hh = v == r ? g - b : (v == g ? b - r + 2 * diff : r - g + 4 * diff);
  hh = (hh * hdiv[diff] + (1 << 11)) >> 12;
  h = hh < 0 ? hh + 180 : hh;
}

__device__ __forceinline__ int unit_to_u8(float x) {
  const int q = __float2int_rn(__fmul_rn(x, 255.f));
  return q < 0 ? 0 : (q > 255 ? 255 : q);
}

__device__ __forceinline__ void hsv2rgb(int h8, int s8, int v8, int& r, int& g, int& b) {
  const float hscale = __fdiv_rn(6.f, 180.f), inv255 = __fdiv_rn(1.f, 255.f);
  const float h = __fmul_rn(static_cast<float>(h8), hscale);
  const float s = __fmul_rn(static_cast<float>(s8), inv255);
  const float v = __fmul_rn(static_cast<float>(v8), inv255);
  int sector = static_cast<int>(truncf(h));
  const float f = __fsub_rn(h, static_cast<float>(sector));
  if (sector < 0 || sector >= 6) sector = 0;
  const float t1 = __fmul_rn(v, __fsub_rn(1.f, s));
  const float t2 = __fmul_rn(v, __fmaf_rn(-s, f, 1.f));
  const float t3 = __fmul_rn(v, __fmaf_rn(-s, __fsub_rn(1.f, f), 1.f));
  // cv2's sector_data {b, g, r} = {1,3,0} {1,0,2} {3,0,1} {0,2,1} {0,1,3} {2,1,0}, one nibble per sector
  auto pick = [&](int packed) {
    const int k = (packed >> (4 * sector)) & 3;
    return k == 0 ? v : (k == 1 ? t1 : (k == 2 ? t2 : t3));
  };
  b = unit_to_u8(pick(0x200311));
  g = unit_to_u8(pick(0x112003));
  r = unit_to_u8(pick(0x031120));
}

__global__ void __launch_bounds__(kThreads) photometric_u8_kernel(const uint8_t* src, uint8_t* dst, int height,
                                                                   int width, int tiles_x, const int* __restrict__ blur_k, int to_hsv,
                                                                   const uint8_t* __restrict__ lut_hsv, int to_rgb,
                                                                   const uint8_t* __restrict__ lut_out) {
  __shared__ __align__(16) uint8_t s_in[kInRows * kInPitch];
  __shared__ __align__(16) uint8_t s_out[kTH * kOutPitch];
  __shared__ uint16_t s_col[kTH * kColW * 3];
  __shared__ int s_div[2][256];
  __shared__ uint8_t s_lut[2][3][256];
  __shared__ int s_delta[kInRows];

  const int img = blockIdx.y;
  const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
  const int x0 = tx * kTW, y0 = ty * kTH;
  const int tw = min(kTW, width - x0), th = min(kTH, height - y0);
  int kx = 1, ky = 1;
  if (blur_k != nullptr) { kx = blur_k[2 * img]; ky = blur_k[2 * img + 1]; }
  if (kx < 1 || kx > kMaxK || ky < 1 || ky > kMaxK) return;  // never index past the shared tiles (the host wrappers reject these)
  const int ax = kx / 2, ay = ky / 2;
  const long long row_bytes = 3ll * width;
  const uint8_t* frame = src + static_cast<long long>(img) * height * row_bytes;
  uint8_t* out_frame = dst + static_cast<long long>(img) * height * row_bytes;

  // tables
  for (int i = threadIdx.x; i < 256; i += kThreads) {
    if (to_hsv) {
      const double d = static_cast<double>(i > 0 ? i : 1);
      s_div[0][i] = i > 0 ? __double2int_rn(static_cast<double>(255 << 12) / d) : 0;
      s_div[1][i] = i > 0 ? __double2int_rn(static_cast<double>(180 << 12) / (6.0 * d)) : 0;
    }
    for (int c = 0; c < 3; ++c) {
      s_lut[0][c][i] = lut_hsv != nullptr ? lut_hsv[(static_cast<long long>(img) * 3 + c) * 256 + i] : static_cast<uint8_t>(i);
      s_lut[1][c][i] = lut_out != nullptr ? lut_out[(static_cast<long long>(img) * 3 + c) * 256 + i] : static_cast<uint8_t>(i);
    }
  }

  // input rows y0 - ay .. y0 + th - 1 + (ky - 1 - ay), reflected; columns [cs, ce) of each (reflection happens when reading)
  const int in_rows = th + ky - 1;
  const int cs = max(0, x0 - ax), ce = min(width, x0 + tw + (kx - 1 - ax));
  const int span = (ce - cs) * 3;
  const int max_chunks = (span + 15 + 15) / 16;  // a row's chunk count depends on its alignment: the worst case, <= kInPitch / 16
  for (int i = threadIdx.x; i < in_rows * max_chunks; i += kThreads) {
    const int r = i / max_chunks, chunk = i - r * max_chunks;
    const uint8_t* g = frame + reflect101(y0 - ay + r, height) * row_bytes + 3ll * cs;
    if (chunk == 0) s_delta[r] = static_cast<int>(reinterpret_cast<uintptr_t>(g) & 15);
    if (chunk < chunks_of(g, span)) load_chunk(g, span, s_in + r * kInPitch, chunk);
  }
  __syncthreads();

  // vertical window sums over the tile's columns plus the horizontal halo (column j is x = x0 - ax + j, reflected)
  const bool blur = kx * ky > 1;
  const int cols = tw + kx - 1;
  if (blur) {
    for (int i = threadIdx.x; i < th * cols * 3; i += kThreads) {
      const int r = i / (cols * 3), rem = i - r * cols * 3, j = rem / 3, c = rem - j * 3;
      const int off = (reflect101(x0 - ax + j, width) - cs) * 3 + c;
      int sum = 0;
      for (int k = 0; k < ky; ++k) sum += s_in[(r + k) * kInPitch + s_delta[r + k] + off];
      s_col[(r * kColW + j) * 3 + c] = static_cast<uint16_t>(sum);
    }
    __syncthreads();
  }

  const int area = kx * ky;
  const int bump = (area == 2 || area == 4 || area == 8 || area == 16) ? 1 : 0;
  const unsigned magic = static_cast<unsigned>((0x100000000ull + area - 1) / area);  // ceil(2^32 / a): exact for sums < 2^16
  uint8_t* out_row0 = out_frame + static_cast<long long>(y0) * row_bytes + 3ll * x0;
  const int out_delta0 = static_cast<int>(reinterpret_cast<uintptr_t>(out_row0) & 15);
  const int out_step = static_cast<int>(row_bytes & 15);
  for (int p = threadIdx.x; p < th * tw; p += kThreads) {
    const int r = p / tw, x = p - r * tw;
    int px[3];
    if (blur) {
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        unsigned sum = 0;
        for (int k = 0; k < kx; ++k) sum += s_col[(r * kColW + x + k) * 3 + c];
        const unsigned q = __umulhi(sum + static_cast<unsigned>(area / 2 + bump), magic);
        px[c] = q > 255u ? 255 : static_cast<int>(q);
      }
    } else {
      const uint8_t* sp = s_in + r * kInPitch + s_delta[r] + (x0 + x - cs) * 3;
      px[0] = sp[0]; px[1] = sp[1]; px[2] = sp[2];
    }
    if (to_hsv) bgr2hsv(px[0], px[1], px[2], s_div[0], s_div[1], px[0], px[1], px[2]);
#pragma unroll
    for (int c = 0; c < 3; ++c) px[c] = s_lut[0][c][px[c]];
    if (to_rgb) hsv2rgb(px[0], px[1], px[2], px[0], px[1], px[2]);
    const int od = (out_delta0 + r * out_step) & 15;
    uint8_t* op = s_out + r * kOutPitch + od + x * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) op[c] = s_lut[1][c][px[c]];
  }
  __syncthreads();

  const int out_span = tw * 3;
  const int out_chunks = (out_span + 15 + 15) / 16;
  for (int i = threadIdx.x; i < th * out_chunks; i += kThreads) {
    const int r = i / out_chunks, chunk = i - r * out_chunks;
    uint8_t* g = out_row0 + r * row_bytes;
    if (chunk < chunks_of(g, out_span)) store_chunk(g, out_span, s_out + r * kOutPitch, chunk);
  }
}

}  // namespace

int photometric_u8(const void* src, void* dst, int batch, int height, int width, const int* blur_k, int to_hsv, const unsigned char* lut_hsv,
                   int to_rgb, const unsigned char* lut_out, cudaStream_t stream) {
  YB_REQUIRE(src && dst && batch > 0 && height > 0 && width > 0 && batch <= 65535, "photometric_u8: bad argument");
  YB_REQUIRE(blur_k == nullptr || src != dst, "photometric_u8: src and dst must not alias when the blur is on");
  const int tiles_x = (width + kTW - 1) / kTW, tiles_y = (height + kTH - 1) / kTH;
  YB_REQUIRE(static_cast<long long>(tiles_x) * tiles_y < (1ll << 31), "photometric_u8: frame too large");
  photometric_u8_kernel<<<dim3(tiles_x * tiles_y, batch), kThreads, 0, stream>>>(
      static_cast<const uint8_t*>(src), static_cast<uint8_t*>(dst), height, width, tiles_x, blur_k, to_hsv != 0, lut_hsv, to_rgb != 0, lut_out);
  return check_launch("photometric_u8_kernel");
}

}  // namespace yb
