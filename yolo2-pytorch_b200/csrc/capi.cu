// extern "C" surface of libyolo2_b200.so (declared in include/yolo2_b200.h) + shared host helpers.
#include "../../include/yolo2_b200.h"
#include "yb_common.h"
#include <stdarg.h>
#include <stdint.h>

namespace yb {

char* err_buf() {
  static thread_local char buf[512] = {0};
  return buf;
}

int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(err_buf(), 512, fmt, ap);
  va_end(ap);
  return code;
}

int check_launch(const char* what) {
  const cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(static_cast<int>(e), "%s: %s", what, cudaGetErrorString(e));
  return 0;
}

int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

static int* g_dbg_host = nullptr;
static int* g_dbg_dev = nullptr;

int* debug_word_device() {
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* h = nullptr;
    if (cudaHostAlloc(&h, 4 * sizeof(int), cudaHostAllocMapped) == cudaSuccess) {
      memset(h, 0, 4 * sizeof(int));
      void* d = nullptr;
      if (cudaHostGetDevicePointer(&d, h, 0) == cudaSuccess) {
        g_dbg_host = static_cast<int*>(h);
        g_dbg_dev = static_cast<int*>(d);
      }
    } else {
      cudaGetLastError();
    }
  }
  return g_dbg_dev;
}

// implemented in the kernel translation units
long long conv_workspace_bytes();
int conv_igemm_forward(const void*, const void*, const float*, const float*, float, void*, int, int, int, int, int, int, int, long long,
                       int, int, int, void*, long long, double*, int, int, cudaStream_t);
int pack_weight_split(const float*, void*, int, int, int, int, int, cudaStream_t);
int maxpool2x2_split(const void*, void*, int, int, int, int, int, int, int, int, cudaStream_t);
int conv_ref_forward(const void*, const void*, const float*, const float*, float, void*, int, int, int, int, int, int, int, long long,
                     int, int, cudaStream_t);
int pack_weight(const float*, void*, int, int, int, int, int, cudaStream_t);
int pack_weights_batch(const void*, int, int, cudaStream_t);
void conv_set_trace(void*);
int bn_fold(const float*, const float*, const float*, const float*, float, float*, float*, int, cudaStream_t);
int conv0_tc_forward(const void*, int, const float*, const float*, const float*, float, void*, int, int, int, int, int, double*, cudaStream_t);
int maxpool2x2(const void*, void*, int, int, int, int, int, cudaStream_t);
int maxpool2x2_s1(const void*, void*, int, int, int, int, int, cudaStream_t);
int maxpool2x2_s1_bwd(const void*, const void*, void*, int, int, int, int, cudaStream_t);
int reorg_nhwc(const void*, void*, int, int, int, int, int, int, int, cudaStream_t);
int reorg_nchw(const float*, float*, int, int, int, int, int, int, cudaStream_t);
int decode_forward(const float*, const float*, float*, float*, float*, float*, float*, float*, float*, int, int, int, int, int,
                   cudaStream_t);
int filter_nms(const float*, const float*, const float*, const float*, int, int, int, int, float, float, float, int, int*, int*, int*,
               int*, int*, int*, int*, float*, int, int*, int*, float*, cudaStream_t);
int iou_matrix(const float*, const float*, const float*, const float*, float*, int, int, int, float, cudaStream_t);
int region_loss_forward(const float*, const float*, const float*, const float*, const long long*, int, int, int, int, int, int, float, int,
                        float*, unsigned char*, unsigned char*, float*, int*, float*, float*, float*, cudaStream_t);
int region_loss_backward(const float*, const float*, const float*, float*, int, int, int, int, int, cudaStream_t);
int bn_stats(const void*, long long, long long, int, double*, cudaStream_t);
int bn_finalize(double*, long long, int, float, float, float*, float*, float*, float*, cudaStream_t);
int bn_act_apply(const void*, long long, const float*, const float*, const float*, const float*, float, void*, long long, int, int, int, int, int,
                 int, cudaStream_t);
int bn_act_bwd(int, const void*, long long, const float*, const float*, const float*, const float*, float, const void*, long long, int,
               const void*, long long, int, int, int, int, int, int, double*, void*, long long, int, cudaStream_t);
int bn_param_grad(double*, int, float*, float*, int, float, cudaStream_t);
int reorg_bwd(const void*, long long, int, void*, int, int, int, int, cudaStream_t);
int head_grad_prepare(const float*, void*, float*, int, int, int, int, cudaStream_t);
int conv0_wgrad(const float*, const void*, float*, int, int, int, cudaStream_t);
int conv0_wgrad_bn(const float*, const void*, const void*, long long, int, const float*, const float*, const float*, const float*, float, const double*, float*, int, int, int,
                   cudaStream_t);
int resize_batch_u8(const void*, const long long*, const int*, void*, int, int, int, int, float*, float*, int, cudaStream_t);
int totensor_u8(const void*, float*, int, int, int, cudaStream_t);
int warp_affine_u8(const void*, int, int, void*, int, int, const double*, const int*, cudaStream_t);
int resize_aug_batch_u8(const void*, const long long*, const int*, const int*, const float*, const unsigned char*, void*, int, int, int, int, float*, float*,
                        int, cudaStream_t);
int photometric_u8(const void*, void*, int, int, int, const int*, int, const unsigned char*, int, const unsigned char*, cudaStream_t);
int eval_match(const float*, const float*, const int*, const int*, const float*, const float*, const int*, const int*, int, int, int, float, float,
               unsigned char*, cudaStream_t);
int unpack_wgrad(const float*, float*, int, int, int, float, cudaStream_t);
int grad_guard(float*, long long, float*, int, cudaStream_t);
int conv_wgrad_forward(const void*, const void*, float*, int, int, int, int, int, int, int, int, cudaStream_t);
int stem7x7(const float*, const float*, const float*, const float*, void*, int, int, int, cudaStream_t);
int stem7x7_96(const float*, const float*, const float*, const float*, void*, int, int, int, cudaStream_t);
int maxpool3x3_s2(const void*, void*, int, int, int, int, cudaStream_t);
int maxpool3x3_s2_strided(const void*, void*, int, int, int, int, int, int, cudaStream_t);
int bn_relu(const void*, int, const float*, const float*, void*, int, long long, int, int, cudaStream_t);
int bn_relu_avgpool2x2(const void*, int, const float*, const float*, void*, int, int, int, int, cudaStream_t);
int subsample2(const void*, void*, int, int, int, int, cudaStream_t);
int add_relu(const void*, const void*, void*, long long, cudaStream_t);
int comm_version(int*);
int comm_unique_id(void*);
int comm_init(void**, int, const void*, int);
int comm_destroy(void*);
int allreduce_bucket(void*, void*, long long, int, cudaStream_t);
int broadcast_buffer(void*, void*, long long, int, int, cudaStream_t);
int mb_conv0(const float*, const float*, const float*, const float*, void*, int, int, int, int, int, cudaStream_t);
int dwconv3x3_split(const void*, const float*, const float*, const float*, void*, int, int, int, int, int, cudaStream_t);
int dwconv3x3(const void*, const float*, const float*, const float*, void*, int, int, int, int, int, int, cudaStream_t);
int dw_dgrad(const void*, const float*, void*, int, int, int, int, int, cudaStream_t);
int dw_wgrad(const void*, const void*, float*, int, int, int, int, int, cudaStream_t);
int mb_conv0_wgrad(const float*, const void*, float*, int, int, int, cudaStream_t);

}  // namespace yb

#define S(stream) static_cast<cudaStream_t>(stream)

extern "C" {

int yb_version(void) { return 100; }

const char* yb_last_error(void) { return yb::err_buf(); }

int yb_debug_read(int out[4]) {
  if (out == nullptr) return YB_ERR_BAD_ARG;
  if (yb::g_dbg_host == nullptr) { out[0] = out[1] = out[2] = out[3] = 0; return 0; }
  for (int i = 0; i < 4; ++i) { out[i] = yb::g_dbg_host[i]; yb::g_dbg_host[i] = 0; }
  return 0;
}

int yb_conv_set_trace(void* dev_buf) { yb::conv_set_trace(dev_buf); return 0; }

int yb_pack_weight_f16(const float* w_oihw, void* w_f16, int cout, int cin, int ksize, int mode, yb_stream_t stream) {
  return yb::pack_weight(w_oihw, w_f16, cout, cin, ksize, mode, 0, S(stream));
}

int yb_bn_fold(const float* gamma, const float* beta, const float* running_mean, const float* running_var, float eps, float* scale,
               float* shift, int channels, yb_stream_t stream) {
  return yb::bn_fold(gamma, beta, running_mean, running_var, eps, scale, shift, channels, S(stream));
}

int yb_conv0_bn_leaky_pool_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, float slope,
                               void* y_nhwc_f16, int batch, int height, int width, int cout, yb_stream_t stream) {
  return yb::conv0_tc_forward(x_nchw, 0, w_oihw, scale, shift, slope, y_nhwc_f16, batch, height, width, cout, 0, nullptr, S(stream));
}

int yb_conv0_u8_bn_leaky_pool_fwd(const unsigned char* x_nhwc_u8, const float* w_oihw, const float* scale, const float* shift,
                                  float slope, void* y_nhwc_f16, int batch, int height, int width, int cout, yb_stream_t stream) {
  return yb::conv0_tc_forward(x_nhwc_u8, 1, w_oihw, scale, shift, slope, y_nhwc_f16, batch, height, width, cout, 0, nullptr, S(stream));
}

int yb_conv_bn_act_fwd(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch,
                       int height, int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int out_mode,
                       int flags, yb_stream_t stream) {
  return yb::conv_igemm_forward(x, w, scale, shift, slope, y, batch, height, width, cin, cout, ksize, x_ld, y_ld, y_ch_off, out_mode,
                                flags, nullptr, 0, nullptr, 0, -1, S(stream));
}

int yb_conv_bn_act_stats_fwd(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch,
                             int height, int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int flags,
                             double* sums, yb_stream_t stream) {
  return yb::conv_igemm_forward(x, w, scale, shift, slope, y, batch, height, width, cin, cout, ksize, x_ld, y_ld, y_ch_off, 0, flags, nullptr, 0,
                                sums, 0, -1, S(stream));
}

long long yb_conv_workspace_bytes(void) { return yb::conv_workspace_bytes(); }

int yb_conv_bn_act_fwd_ws(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch,
                          int height, int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int out_mode,
                          int flags, void* workspace, long long workspace_bytes, yb_stream_t stream) {
  return yb::conv_igemm_forward(x, w, scale, shift, slope, y, batch, height, width, cin, cout, ksize, x_ld, y_ld, y_ch_off, out_mode,
                                flags, workspace, workspace_bytes, nullptr, 0, -1, S(stream));
}

int yb_conv_bn_act_split_fwd(const void* x, const void* w_split, const float* scale, const float* shift, float slope, void* y, int batch,
                             int height, int width, int k_channels, int a_channels, int cout, int ksize, int x_ld, long long y_ld,
                             int y_ch_off, int lo_ch_off, int out_mode, int flags, void* workspace, long long workspace_bytes,
                             yb_stream_t stream) {
  return yb::conv_igemm_forward(x, w_split, scale, shift, slope, y, batch, height, width, k_channels, cout, ksize, x_ld, y_ld, y_ch_off,
                                out_mode, flags, workspace, workspace_bytes, nullptr, a_channels, lo_ch_off, S(stream));
}

int yb_pack_weight_split_f16(const float* w_oihw, void* w_f16, int cout, int cin, int ksize, int segments, int lo_mask, yb_stream_t stream) {
  return yb::pack_weight_split(w_oihw, w_f16, cout, cin, ksize, segments, lo_mask, S(stream));
}

int yb_maxpool2x2_split_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, int x_lo_off, int y_ld,
                            int y_lo_off, yb_stream_t stream) {
  return yb::maxpool2x2_split(x, y, batch, height, width, channels, x_ld, x_lo_off, y_ld, y_lo_off, S(stream));
}

int yb_conv_ref_fwd(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch, int height,
                    int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int out_mode, yb_stream_t stream) {
  return yb::conv_ref_forward(x, w, scale, shift, slope, y, batch, height, width, cin, cout, ksize, x_ld, y_ld, y_ch_off, out_mode,
                              S(stream));
}

int yb_maxpool2x2_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, yb_stream_t stream) {
  return yb::maxpool2x2(x, y, batch, height, width, channels, x_ld, S(stream));
}

int yb_maxpool2x2_s1_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, yb_stream_t stream) {
  return yb::maxpool2x2_s1(x, y, batch, height, width, channels, x_ld, S(stream));
}

int yb_maxpool2x2_s1_bwd_f16(const void* x, const void* dy, void* dx, int batch, int height, int width, int channels, yb_stream_t stream) {
  return yb::maxpool2x2_s1_bwd(x, dy, dx, batch, height, width, channels, S(stream));
}

int yb_reorg_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, int y_ld, int y_ch_off,
                 yb_stream_t stream) {
  return yb::reorg_nhwc(x, y, batch, height, width, channels, x_ld, y_ld, y_ch_off, S(stream));
}

int yb_reorg_f32_nchw(const float* x, float* y, int batch, int channels, int height, int width, int stride_h, int stride_w,
                      yb_stream_t stream) {
  return yb::reorg_nchw(x, y, batch, channels, height, width, stride_h, stride_w, S(stream));
}

int yb_decode_fwd(const float* feature, const float* anchors_hw, float* iou, float* center_offset, float* size_norm, float* yx_min,
                  float* yx_max, float* logits, float* prob, int batch, int rows, int cols, int num_anchors, int num_cls,
                  yb_stream_t stream) {
  return yb::decode_forward(feature, anchors_hw, iou, center_offset, size_norm, yx_min, yx_max, logits, prob, batch, rows, cols,
                            num_anchors, num_cls, S(stream));
}

int yb_filter_nms(const float* score, const float* yx_min, const float* yx_max, const float* prob, int batch, int n, int num_cls,
                  int mode, float threshold, float threshold_cls, float overlap, int limit, int* n_filtered, int* n_keep,
                  int* keep_idx, int* keep_box, int* n_det, int* det_keep, int* det_cls, float* det_score, int det_cap,
                  int* filt_box, int* best_cls, float* best_prob, yb_stream_t stream) {
  return yb::filter_nms(score, yx_min, yx_max, prob, batch, n, num_cls, mode, threshold, threshold_cls, overlap, limit, n_filtered,
                        n_keep, keep_idx, keep_box, n_det, det_keep, det_cls, det_score, det_cap, filt_box, best_cls, best_prob,
                        S(stream));
}

int yb_iou_matrix(const float* yx_min1, const float* yx_max1, const float* yx_min2, const float* yx_max2, float* out, int batch,
                  int n1, int n2, float min_union, yb_stream_t stream) {
  return yb::iou_matrix(yx_min1, yx_max1, yx_min2, yx_max2, out, batch, n1, n2, min_union, S(stream));
}

int yb_region_loss_fwd(const float* feature, const float* anchors_hw, const float* gt_yx_min, const float* gt_yx_max,
                       const long long* gt_cls, int batch, int rows, int cols, int num_anchors, int num_cls, int num_gt, float threshold,
                       int cross_entropy, float* losses, unsigned char* positive, unsigned char* negative, float* best_iou, int* pos_count,
                       float* partial, float* grad_terms, float* grad_bg, yb_stream_t stream) {
  return yb::region_loss_forward(feature, anchors_hw, gt_yx_min, gt_yx_max, gt_cls, batch, rows, cols, num_anchors, num_cls, num_gt,
                                 threshold, cross_entropy, losses, positive, negative, best_iou, pos_count, partial, grad_terms, grad_bg,
                                 S(stream));
}

int yb_region_loss_bwd(const float* grad_terms, const float* grad_bg, const float* weights5, float* dfeature, int batch, int rows, int cols,
                       int num_anchors, int num_cls, yb_stream_t stream) {
  return yb::region_loss_backward(grad_terms, grad_bg, weights5, dfeature, batch, rows, cols, num_anchors, num_cls, S(stream));
}

int yb_conv0_raw_fwd(const float* x_nchw, const float* w_oihw, void* z_nhwc_f16, int batch, int height, int width, int cout,
                     yb_stream_t stream) {
  return yb::conv0_tc_forward(x_nchw, 0, w_oihw, nullptr, nullptr, 1.f, z_nhwc_f16, batch, height, width, cout, 1, nullptr, S(stream));
}

int yb_conv0_raw_stats_fwd(const float* x_nchw, const float* w_oihw, void* z_nhwc_f16, double* sums, int batch, int height, int width, int cout,
                           yb_stream_t stream) {
  return yb::conv0_tc_forward(x_nchw, 0, w_oihw, nullptr, nullptr, 1.f, z_nhwc_f16, batch, height, width, cout, 1, sums, S(stream));
}

int yb_pack_weights_batch(const yb_pack_unit* units_dev, int num_units, int total_blocks, yb_stream_t stream) {
  return yb::pack_weights_batch(units_dev, num_units, total_blocks, S(stream));
}

int yb_pack_weight_dgrad_f16(const float* w_oihw, void* w_f16, int cout, int cin, int ksize, int cout_pad, yb_stream_t stream) {
  return yb::pack_weight(w_oihw, w_f16, cout, cin, ksize, 1, cout_pad, S(stream));
}

int yb_bn_stats(const void* z, long long ld, long long rows, int channels, double* sums, yb_stream_t stream) {
  return yb::bn_stats(z, ld, rows, channels, sums, S(stream));
}

int yb_bn_finalize(double* sums, long long rows, int channels, float eps, float momentum, float* running_mean, float* running_var,
                   float* mean, float* invstd, yb_stream_t stream) {
  return yb::bn_finalize(sums, rows, channels, eps, momentum, running_mean, running_var, mean, invstd, S(stream));
}

int yb_bn_act_apply(const void* z, long long ld_z, const float* mean, const float* invstd, const float* gamma, const float* beta,
                    float slope, void* a, long long ld_a, int a_ch_off, int batch, int height, int width, int channels, int pool,
                    yb_stream_t stream) {
  return yb::bn_act_apply(z, ld_z, mean, invstd, gamma, beta, slope, a, ld_a, a_ch_off, batch, height, width, channels, pool, S(stream));
}

int yb_bn_act_bwd(int mode, const void* z, long long ld_z, const float* mean, const float* invstd, const float* gamma, const float* beta,
                  float slope, const void* da, long long ld_da, int da_off, const void* dap, long long ld_dap, int dap_off, int batch,
                  int height, int width, int channels, int window, double* sums, void* dz, long long ld_dz, int has_bn, yb_stream_t stream) {
  return yb::bn_act_bwd(mode, z, ld_z, mean, invstd, gamma, beta, slope, da, ld_da, da_off, dap, ld_dap, dap_off, batch, height, width,
                        channels, window, sums, dz, ld_dz, has_bn, S(stream));
}

int yb_bn_param_grad(double* sums, int channels, float* dgamma, float* dbeta, int reset, float scale, yb_stream_t stream) {
  return yb::bn_param_grad(sums, channels, dgamma, dbeta, reset, scale, S(stream));
}

int yb_reorg_bwd_f16(const void* dy, long long ld_dy, int dy_off, void* dx, int batch, int height, int width, int channels,
                     yb_stream_t stream) {
  return yb::reorg_bwd(dy, ld_dy, dy_off, dx, batch, height, width, channels, S(stream));
}

int yb_head_grad_prepare(const float* dfeature, void* dz_nhwc_f16, float* dbias, int batch, int channels, int channels_pad, int cells,
                         yb_stream_t stream) {
  return yb::head_grad_prepare(dfeature, dz_nhwc_f16, dbias, batch, channels, channels_pad, cells, S(stream));
}

int yb_conv0_wgrad(const float* x_nchw, const void* dz_nhwc_f16, float* dw_oihw, int batch, int height, int width, yb_stream_t stream) {
  return yb::conv0_wgrad(x_nchw, dz_nhwc_f16, dw_oihw, batch, height, width, S(stream));
}

int yb_conv0_wgrad_bn(const float* x_nchw, const void* z_nhwc_f16, const void* dap, long long ld_dap, int dap_off, const float* mean, const float* invstd,
                      const float* gamma, const float* beta, float slope, const double* sums, float* dw_oihw, int batch, int height, int width,
                      yb_stream_t stream) {
  return yb::conv0_wgrad_bn(x_nchw, z_nhwc_f16, dap, ld_dap, dap_off, mean, invstd, gamma, beta, slope, sums, dw_oihw, batch, height, width, S(stream));
}

int yb_conv_wgrad(const void* x, const void* dz, float* dw_krsc, int batch, int height, int width, int cin, int cout, int ksize, int x_ld,
                  int dz_ld, yb_stream_t stream) {
  return yb::conv_wgrad_forward(x, dz, dw_krsc, batch, height, width, cin, cout, ksize, x_ld, dz_ld, S(stream));
}

int yb_unpack_wgrad(const float* dw_krsc, float* dw_oihw, int cout, int cin, int ksize, float scale, yb_stream_t stream) {
  return yb::unpack_wgrad(dw_krsc, dw_oihw, cout, cin, ksize, scale, S(stream));
}

int yb_grad_guard(float* grads, long long count, float* found_inf, int zero_if_found, yb_stream_t stream) {
  return yb::grad_guard(grads, count, found_inf, zero_if_found, S(stream));
}

int yb_resize_batch_u8(const void* src, const long long* src_off, const int* src_hw, void* dst, int batch, int height, int width, int swap_rb,
                       float* yx_min, float* yx_max, int slots, yb_stream_t stream) {
  return yb::resize_batch_u8(src, src_off, src_hw, dst, batch, height, width, swap_rb, yx_min, yx_max, slots, S(stream));
}

int yb_resize_aug_batch_u8(const void* src, const long long* src_off, const int* src_hw, const int* crop, const float* margin, const unsigned char* flip,
                           void* dst, int batch, int height, int width, int swap_rb, float* yx_min, float* yx_max, int slots, yb_stream_t stream) {
  return yb::resize_aug_batch_u8(src, src_off, src_hw, crop, margin, flip, dst, batch, height, width, swap_rb, yx_min, yx_max, slots, S(stream));
}

int yb_warp_affine_u8(const void* src, int src_h, int src_w, void* dst, int dst_h, int dst_w, const double* inverse_matrix6, const int* fill3,
                      yb_stream_t stream) {
  return yb::warp_affine_u8(src, src_h, src_w, dst, dst_h, dst_w, inverse_matrix6, fill3, S(stream));
}

int yb_totensor_u8(const void* src_nhwc_u8, float* dst_nchw_f32, int batch, int height, int width, yb_stream_t stream) {
  return yb::totensor_u8(src_nhwc_u8, dst_nchw_f32, batch, height, width, S(stream));
}

int yb_photometric_u8(const void* src, void* dst, int batch, int height, int width, const int* blur_k, int to_hsv, const unsigned char* lut_hsv,
                      int to_rgb, const unsigned char* lut_out, yb_stream_t stream) {
  return yb::photometric_u8(src, dst, batch, height, width, blur_k, to_hsv, lut_hsv, to_rgb, lut_out, S(stream));
}

int yb_eval_match(const float* det_yx_min, const float* det_yx_max, const int* det_cls, const int* det_off, const float* gt_yx_min,
                  const float* gt_yx_max, const int* gt_cls, const int* gt_off, int batch, int num_cls, int max_gt, float threshold, float min_union,
                  unsigned char* tp, yb_stream_t stream) {
  return yb::eval_match(det_yx_min, det_yx_max, det_cls, det_off, gt_yx_min, gt_yx_max, gt_cls, gt_off, batch, num_cls, max_gt, threshold, min_union, tp,
                        S(stream));
}

int yb_mb_conv0_bn_relu_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_nhwc_f16, int batch,
                            int height, int width, yb_stream_t stream) {
  return yb::mb_conv0(x_nchw, w_oihw, scale, shift, y_nhwc_f16, batch, height, width, 0, 0, S(stream));
}

int yb_mb_conv0_split_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_hi_lo, int batch, int height, int width,
                          yb_stream_t stream) {
  return yb::mb_conv0(x_nchw, w_oihw, scale, shift, y_hi_lo, batch, height, width, 0, 1, S(stream));
}

int yb_dwconv3x3_split_fwd(const void* x_hi_lo, const float* w_c9, const float* scale, const float* shift, void* y_hi_lo, int batch, int height, int width,
                           int channels, int stride, yb_stream_t stream) {
  return yb::dwconv3x3_split(x_hi_lo, w_c9, scale, shift, y_hi_lo, batch, height, width, channels, stride, S(stream));
}

int yb_mb_conv0_raw_fwd(const float* x_nchw, const float* w_oihw, void* z_nhwc_f16, int batch, int height, int width, yb_stream_t stream) {
  return yb::mb_conv0(x_nchw, w_oihw, nullptr, nullptr, z_nhwc_f16, batch, height, width, 1, 0, S(stream));
}

int yb_mb_conv0_wgrad(const float* x_nchw, const void* dz_nhwc_f16, float* dw_oihw, int batch, int height, int width, yb_stream_t stream) {
  return yb::mb_conv0_wgrad(x_nchw, dz_nhwc_f16, dw_oihw, batch, height, width, S(stream));
}

int yb_dwconv3x3_raw_fwd(const void* x, const float* w_c9, void* z, int batch, int height, int width, int channels, int stride, yb_stream_t stream) {
  return yb::dwconv3x3(x, w_c9, nullptr, nullptr, z, batch, height, width, channels, stride, 1, S(stream));
}

int yb_dwconv3x3_dgrad(const void* dz, const float* w_c9, void* da, int batch, int height, int width, int channels, int stride, yb_stream_t stream) {
  return yb::dw_dgrad(dz, w_c9, da, batch, height, width, channels, stride, S(stream));
}

int yb_dwconv3x3_wgrad(const void* a, const void* dz, float* dw_c9, int batch, int height, int width, int channels, int stride, yb_stream_t stream) {
  return yb::dw_wgrad(a, dz, dw_c9, batch, height, width, channels, stride, S(stream));
}

int yb_dwconv3x3_bn_relu_fwd(const void* x, const float* w_c9, const float* scale, const float* shift, void* y, int batch, int height,
                             int width, int channels, int stride, yb_stream_t stream) {
  return yb::dwconv3x3(x, w_c9, scale, shift, y, batch, height, width, channels, stride, 0, S(stream));
}

int yb_stem7x7_bn_relu_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_nhwc_f16, int batch, int height, int width,
                           yb_stream_t stream) {
  return yb::stem7x7(x_nchw, w_oihw, scale, shift, y_nhwc_f16, batch, height, width, S(stream));
}

int yb_maxpool3x3_s2_f16(const void* x, void* y, int batch, int height, int width, int channels, yb_stream_t stream) {
  return yb::maxpool3x3_s2(x, y, batch, height, width, channels, S(stream));
}

int yb_stem7x7_96_bn_relu_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_nhwc_f16, int batch, int height,
                              int width, yb_stream_t stream) {
  return yb::stem7x7_96(x_nchw, w_oihw, scale, shift, y_nhwc_f16, batch, height, width, S(stream));
}

int yb_maxpool3x3_s2_strided_f16(const void* x, void* y, int batch, int height, int width, int channels, int y_ld, int y_ch_off, yb_stream_t stream) {
  return yb::maxpool3x3_s2_strided(x, y, batch, height, width, channels, y_ld, y_ch_off, S(stream));
}

int yb_bn_relu_f16(const void* x, int x_ld, const float* scale, const float* shift, void* y, int y_ld, long long pixels, int channels, int channels_padded,
                   yb_stream_t stream) {
  return yb::bn_relu(x, x_ld, scale, shift, y, y_ld, pixels, channels, channels_padded, S(stream));
}

int yb_bn_relu_avgpool2x2_f16(const void* x, int x_ld, const float* scale, const float* shift, void* y, int batch, int height, int width, int channels,
                              yb_stream_t stream) {
  return yb::bn_relu_avgpool2x2(x, x_ld, scale, shift, y, batch, height, width, channels, S(stream));
}

int yb_subsample2_f16(const void* x, void* y, int batch, int height, int width, int channels, yb_stream_t stream) {
  return yb::subsample2(x, y, batch, height, width, channels, S(stream));
}

int yb_add_relu_f16(const void* a, const void* b, void* out, long long count, yb_stream_t stream) { return yb::add_relu(a, b, out, count, S(stream)); }

int yb_comm_version(int* nccl_version) { return yb::comm_version(nccl_version); }

int yb_comm_unique_id(void* id128) { return yb::comm_unique_id(id128); }

int yb_comm_init(void** comm, int nranks, const void* id128, int rank) { return yb::comm_init(comm, nranks, id128, rank); }

int yb_comm_destroy(void* comm) { return yb::comm_destroy(comm); }

int yb_allreduce_bucket(void* comm, void* buf, long long count, int dtype, yb_stream_t stream) {
  return yb::allreduce_bucket(comm, buf, count, dtype, S(stream));
}

int yb_broadcast_buffer(void* comm, void* buf, long long count, int dtype, int root, yb_stream_t stream) {
  return yb::broadcast_buffer(comm, buf, count, dtype, root, S(stream));
}

}  // extern "C"
