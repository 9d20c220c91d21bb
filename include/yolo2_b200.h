/* libyolo2_b200.so -- C ABI of the B200-native YOLOv2 hot path.
 *
 * Drop-in boundary for the Darknet-19 detection path of ruiminshen/yolo2-pytorch.  The reference
 * has no FFI of its own (it is pure Python over torch, SURVEY.md section 8b); each entry point below
 * names the reference Python interface it replaces (file:line under /root/reference) -- these
 * are the calls a maintainer would bind with ctypes (INTEGRATION.md shows the stubs).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer owned by the caller
 *     (PyTorch owns all storage); the library never allocates or frees device memory that
 *     outlives the call and never touches the default stream unless `stream` is NULL;
 *   - `stream` is a cudaStream_t passed as void*; all work is asynchronous on it;
 *   - return value: 0 = success, >0 = cudaError_t, <0 = library error (YB_ERR_*); a human
 *     readable message for the calling thread is returned by yb_last_error();
 *   - there is NO CPU fallback and no silent dispatch: unsupported shapes are errors.
 *   - activations inside the backbone are fp16 NHWC ("x_ld" = elements between consecutive
 *     pixels, so a tensor may be a channel slice of a wider buffer); the tensors the reference's
 *     callers see (input image batch, head feature map, decode outputs) are fp32 in the
 *     reference's own layouts.
 */
#ifndef YOLO2_B200_H_
#define YOLO2_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef void* yb_stream_t; /* cudaStream_t */

#define YB_ERR_BAD_ARG (-1)
#define YB_ERR_UNSUPPORTED (-2)
#define YB_ERR_DRIVER (-3)

/* yb_conv_bn_act_fwd out_mode */
#define YB_OUT_F16_NHWC 0
#define YB_OUT_F32_NCHW 1
/* yb_conv_bn_act_fwd flags */
#define YB_CONV_A_TILED 1      /* 1x1 only: fetch A with a plain 2-D tiled TMA instead of im2col mode */
#define YB_CONV_WIDE_N 2       /* allow the 128x256 tile when Cout % 256 == 0 */
#define YB_CONV_FORCE_BN(bn) ((bn) << 8) /* testing: force BLOCK_N in {64,128,256} */
#define YB_CONV_POOL2X2 16     /* also apply MaxPool2d(2): y is [B,H/2,W/2,Cout]; implemented for the 3x3 Cin=32 layer (layers1.2) */
#define YB_CONV_C32_IM2COL 32  /* testing: Cin=32 3x3 through the im2col small-K kernel instead of the halo-tile kernel */
#define YB_CONV_NO_STREAMK 8   /* never split tiles along K even when a workspace is supplied */
#define YB_CONV_FORCE_STREAMK (1 << 30) /* testing: split along K whenever the shape allows it */
#define YB_CONV_NO_SMALLK (1 << 28)     /* testing: route Cin=32 3x3 layers through the generic kernel */
#define YB_CONV_PLAIN_STORE (1 << 29)   /* testing: small-K kernel writes with per-thread stores instead of a TMA store */
/* yb_filter_nms mode */
#define YB_FILTER_THRESHOLD 0  /* detect/fix = 0: iou > detect/threshold            (detect.py:56) */
#define YB_FILTER_FIX 1        /* detect/fix = 1: iou * max prob > threshold_cls    (detect.py:54) */
#define YB_FILTER_NONE 2       /* plain utils.postprocess.nms over all n boxes */

int yb_version(void);
const char* yb_last_error(void);
/* Reads (and clears) the host-mapped debug word a kernel writes before it traps on a pipeline
 * time-out: out[0] = 0x0BADxxxx code, out[1] = block, out[2] = thread, out[3] = parity. */
int yb_debug_read(int out[4]);
/* Profiling aid (tools/conv_trace.py): when dev_buf (768 x uint64, device memory) is non-NULL, block 0 of the
 * tcgen05 conv kernels records clock64() per pipeline event: [0,256) TMA producer, [256,512) MMA issuer,
 * [512,768) epilogue.  NULL switches it off (the default). */
int yb_conv_set_trace(void* dev_buf);

/* ---- parameter preparation ---------------------------------------------------------------- */
/* nn.Conv2d weight [Cout,Cin,k,k] fp32 (model/yolo2.py:57) -> fp16 [Cout][k][k][Cin] (mode 0), or
 * the rotated/transposed data-gradient operand [Cin][k][k][Cout] (mode 1). */
int yb_pack_weight_f16(const float* w_oihw, void* w_f16, int cout, int cin, int ksize, int mode, yb_stream_t stream);
/* nn.BatchNorm2d in eval mode (model/yolo2.py:58): scale = gamma / sqrt(var + eps), shift = beta - mean * scale. */
int yb_bn_fold(const float* gamma, const float* beta, const float* running_mean, const float* running_var, float eps, float* scale,
               float* shift, int channels, yb_stream_t stream);

/* ---- backbone: model.yolo2.Conv2d.forward (model/yolo2.py:61-65), nn.MaxPool2d (:79), reorg (:33-46) */
/* layers1.0 + its MaxPool: x fp32 NCHW [B,3,H,W] (the caller's tensor) -> y fp16 NHWC [B,H/2,W/2,32].
 * H % 16 == 0, W % 32 == 0. */
int yb_conv0_bn_leaky_pool_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, float slope,
                               void* y_nhwc_f16, int batch, int height, int width, int cout, yb_stream_t stream);
/* Same layer fed by raw frames: x uint8 NHWC [B,H,W,3] (RGB), scaled by 1/255 in the kernel --
 * replaces the host-side torchvision ToTensor the reference runs per frame (detect.py:144-145,
 * transform/__init__.py) and cuts the host->device copy 4x. */
int yb_conv0_u8_bn_leaky_pool_fwd(const unsigned char* x_nhwc_u8, const float* w_oihw, const float* scale, const float* shift,
                                  float slope, void* y_nhwc_f16, int batch, int height, int width, int cout, yb_stream_t stream);
/* k in {1,3}, stride 1, pad (k-1)/2 conv + per-channel scale/shift + leaky(slope) as a tcgen05
 * implicit GEMM.  x: fp16 NHWC [B,H,W,Cin] with pixel pitch x_ld; w: fp16 [Cout][k][k][Cin];
 * y: fp16 NHWC (pixel pitch y_ld, first channel y_ch_off) or fp32 NCHW [B,Cout,H,W].
 * slope = 1 disables the activation; the head passes scale = 1, shift = bias. */
int yb_conv_bn_act_fwd(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch,
                       int height, int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int out_mode,
                       int flags, yb_stream_t stream);
/* Same conv with a caller-owned scratch buffer (yb_conv_workspace_bytes() bytes, 256 B aligned, ZERO-FILLED ONCE when it
 * is allocated; one per stream -- launches that may overlap must not share it).  With it the library may run the layer
 * stream-K: tiles x K-blocks are divided evenly over all SMs and tiles cut by a boundary are summed through the buffer,
 * which keeps every SM busy on the 13x13 / 26x26 layers whose tile count does not fill the GPU.  NULL = plain tiles. */
/* Training forward: yb_conv_bn_act_fwd (fp16 NHWC output) that ALSO adds the per-channel sum and sum of squares of the stored
 * (fp16-rounded) outputs into sums[0..Cout) / sums[Cout..2Cout) (double, zero on entry: the contract of yb_bn_stats), reduced in
 * the epilogue with warp shuffles -- train-mode BatchNorm statistics (model/yolo2.py:58) without a second pass over z.  Not for
 * the Cin = 32 3x3 layer (halo-tile kernel). */
int yb_conv_bn_act_stats_fwd(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch,
                             int height, int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int flags,
                             double* sums, yb_stream_t stream);
long long yb_conv_workspace_bytes(void);
int yb_conv_bn_act_fwd_ws(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch,
                          int height, int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int out_mode,
                          int flags, void* workspace, long long workspace_bytes, yb_stream_t stream);
/* Split-precision ("strict") form of the same unit, for callers that need the reference's fp32 results to 1e-3 end to end
 * (model/yolo2.py:125-130 runs in fp32; 23 fp16-operand layers drift 1.6e-3).  The GEMM's reduction dimension is a concatenation
 * of fp16 terms accumulated in one fp32 TMEM accumulator:  A = [a_hi | a_lo | a_hi],  W = [w_hi | w_hi | w_lo]  (or the two-term
 * forms [a_hi | a_lo] x [w_hi | w_hi] and [a_hi | a_hi] x [w_hi | w_lo]).
 *   x        fp16 NHWC, pixel pitch x_ld, holding a_channels channels: C (hi only) or 2C ([hi | lo] of the same pixel);
 *   w_split  fp16 [Cout][k][k][k_channels] from yb_pack_weight_split_f16 (k_channels = 2C or 3C; channel offsets >= a_channels
 *            wrap around to the start of the pixel's channels, which is how a_hi is read twice);
 *   lo_ch_off >= 0: besides y = fp16(v) at y_ch_off also stores fp16(v - fp32(fp16(v))) at channel lo_ch_off of the same pixel
 *            (fp16 NHWC output only), so the next layer can read [hi | lo]; -1: plain output.
 * Everything else as yb_conv_bn_act_fwd_ws (workspace may be NULL). */
int yb_conv_bn_act_split_fwd(const void* x, const void* w_split, const float* scale, const float* shift, float slope, void* y, int batch,
                             int height, int width, int k_channels, int a_channels, int cout, int ksize, int x_ld, long long y_ld,
                             int y_ch_off, int lo_ch_off, int out_mode, int flags, void* workspace, long long workspace_bytes,
                             yb_stream_t stream);
/* B operand of yb_conv_bn_act_split_fwd: out[co][r][s][seg*Cin + ci], seg in [0, segments): fp16(w), or where bit seg of lo_mask is
 * set fp16(w - fp32(fp16(w))).  (segments, lo_mask) = (2, 0) activation split, (2, 2) weight split, (3, 4) both. */
int yb_pack_weight_split_f16(const float* w_oihw, void* w_f16, int cout, int cin, int ksize, int segments, int lo_mask, yb_stream_t stream);
/* nn.MaxPool2d(2) (model/yolo2.py:79) on split activations: hi at channel c, lo at c + *_lo_off of the same pixel; the window element
 * with the largest hi + lo wins and its pair is copied. */
int yb_maxpool2x2_split_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, int x_lo_off, int y_ld,
                            int y_lo_off, yb_stream_t stream);
/* Same contract on CUDA cores (one thread per output): test/bisect utility, not a product path. */
int yb_conv_ref_fwd(const void* x, const void* w, const float* scale, const float* shift, float slope, void* y, int batch, int height,
                    int width, int cin, int cout, int ksize, int x_ld, long long y_ld, int y_ch_off, int out_mode, yb_stream_t stream);
int yb_maxpool2x2_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, yb_stream_t stream);
/* model.yolo2.Tiny: ConstantPad2d((0,1,0,1), float32 min) + MaxPool2d(2, stride=1) (model/yolo2.py:150-151): [B,H,W,C] -> [B,H,W,C]. */
int yb_maxpool2x2_s1_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, yb_stream_t stream);
/* Backward of that pooling (training of model.yolo2.Tiny): dx = gradient routed to the first maximum of every window; x is the pooling INPUT. */
int yb_maxpool2x2_s1_bwd_f16(const void* x, const void* dy, void* dx, int batch, int height, int width, int channels, yb_stream_t stream);
/* space-to-depth(2) on fp16 NHWC into channels [y_ch_off, y_ch_off + 4C) of a y_ld-wide buffer
 * (this plus y_ch_off of the conv replaces torch.cat, model/yolo2.py:129). */
int yb_reorg_f16(const void* x, void* y, int batch, int height, int width, int channels, int x_ld, int y_ld, int y_ch_off,
                 yb_stream_t stream);
/* model.yolo2.reorg(x, stride_h, stride_w) on the caller's fp32 NCHW tensors (model/yolo2.py:33-46). */
int yb_reorg_f32_nchw(const float* x, float* y, int batch, int channels, int height, int width, int stride_h, int stride_w,
                      yb_stream_t stream);

/* ---- head: model.Inference.forward (model/__init__.py:117-135) + F.softmax (detect.py:152) ---- */
/* feature fp32 [B, A*(5+C), rows, cols]; anchors fp32 [A,2] (height,width).  Outputs: iou [B,cells,A],
 * center_offset/size_norm/yx_min/yx_max [B,cells,A,2], logits/prob [B,cells,A,C] (prob may be NULL;
 * logits may be NULL when num_cls == 1). */
int yb_decode_fwd(const float* feature, const float* anchors_hw, float* iou, float* center_offset, float* size_norm, float* yx_min,
                  float* yx_max, float* logits, float* prob, int batch, int rows, int cols, int num_anchors, int num_cls,
                  yb_stream_t stream);

/* ---- detection post-filter: detect.filter_visible + utils.postprocess.nms + detect.postprocess
 *      (detect.py:51-80, utils/postprocess.py:23-49), one CTA per image, no host sync ---------- */
/* score [B,n], yx_min/yx_max [B,n,2], prob [B,n,C] (NULL for YB_FILTER_NONE).
 * n_filtered[B]; n_keep[B]; keep_idx[B,limit] = indices into the filtered arrays in descending
 * score order (exactly the list utils.postprocess.nms returns); keep_box[B,limit] = the same as
 * indices into the n input boxes.  If n_det != NULL (fix mode): the (kept box, class) pairs with
 * iou*prob > threshold_cls in mask.nonzero() order: det_keep (rank in the keep list), det_cls,
 * det_score, each [B,det_cap]; n_det[B].  Optional (NULL to skip): filt_box[B,n] = input box of each
 * filtered rank (ascending, the order detect.filter_visible returns), best_cls/best_prob[B,n] =
 * torch.max(prob, -1) per input box (detect.py:52). */
int yb_filter_nms(const float* score, const float* yx_min, const float* yx_max, const float* prob, int batch, int n, int num_cls,
                  int mode, float threshold, float threshold_cls, float overlap, int limit, int* n_filtered, int* n_keep,
                  int* keep_idx, int* keep_box, int* n_det, int* det_keep, int* det_cls, float* det_score, int det_cap,
                  int* filt_box, int* best_cls, float* best_prob, yb_stream_t stream);
/* utils.iou.torch.iou_matrix / batch_iou_matrix (utils/iou/torch.py:47-61,139-153): out [B,n1,n2]. */
int yb_iou_matrix(const float* yx_min1, const float* yx_max1, const float* yx_min2, const float* yx_max2, float* out, int batch,
                  int n1, int n2, float min_union, yb_stream_t stream);

/* ---- training: region loss, model.loss + iou_match / fit_positive / fill_norm (model/__init__.py:59-107,138-167) ---- */
/* feature fp32 [B,A*(5+C),rows,cols] (the head output); GT in GRID units (train.norm_data, train.py:57-62):
 * gt_yx_min/gt_yx_max [B,G,2], gt_cls int64 [B,G], zero-padded slots allowed (utils/data.py:38-41).
 * Outputs: losses[5] = (foreground, background, center, size, cls), each already / (B*cells*A); positive /
 * negative uint8 [B,cells,A]; best_iou [B,cells,A]; and the UNWEIGHTED per-term gradients w.r.t. feature
 * (grad_terms: feature layout, grad_bg [B,A,cells]) consumed by yb_region_loss_bwd.  pos_count[B] and
 * partial[B*5] are scratch.  cross_entropy: train/cross_entropy (config.ini:77). */
int yb_region_loss_fwd(const float* feature, const float* anchors_hw, const float* gt_yx_min, const float* gt_yx_max,
                       const long long* gt_cls, int batch, int rows, int cols, int num_anchors, int num_cls, int num_gt, float threshold,
                       int cross_entropy, float* losses, unsigned char* positive, unsigned char* negative, float* best_iou, int* pos_count,
                       float* partial, float* grad_terms, float* grad_bg, yb_stream_t stream);
/* dfeature = sum_k weights5[k] * d loss_k / d feature; weights5 is a DEVICE array (hparam * upstream grad, train.py:348-351). */
int yb_region_loss_bwd(const float* grad_terms, const float* grad_bg, const float* weights5, float* dfeature, int batch, int rows, int cols,
                       int num_anchors, int num_cls, yb_stream_t stream);

/* ---- training: what torch autograd runs for the backbone in the reference (train.py:344-351) ------------------
 * Forward (train mode) of one model.yolo2.Conv2d unit = yb_conv_bn_act_fwd with scale = 1, shift = 0, slope = 1
 * (raw conv output z, fp16 NHWC; yb_conv_bn_act_stats_fwd also produces the statistics) -> yb_bn_stats -> yb_bn_finalize (batch mean / invstd, running-stat update with
 * momentum 0.01, model/yolo2.py:58) -> yb_bn_act_apply (normalise + leaky [+ MaxPool2d(2)]).
 * Backward of the unit = yb_bn_act_bwd mode 0 (reduce) -> yb_bn_param_grad (dgamma, dbeta) -> yb_bn_act_bwd mode 1
 * (dz) -> yb_conv_bn_act_fwd on dz with yb_pack_weight_dgrad_f16 weights (data gradient) + yb_conv_wgrad /
 * yb_unpack_wgrad (weight gradient).  All activations / gradients fp16 NHWC, statistics in double, parameter
 * gradients fp32 in the reference's OIHW layout. */
/* layers1.0 in train mode: raw conv output, unpooled fp16 NHWC [B,H,W,32]. */
int yb_conv0_raw_fwd(const float* x_nchw, const float* w_oihw, void* z_nhwc_f16, int batch, int height, int width, int cout,
                     yb_stream_t stream);
/* the same with the BatchNorm batch statistics of z fused in: sums (double [2][32], the yb_bn_stats layout) += sum z, sum z^2 of the stored fp16
 * values.  H % 32 == 0 and W % 16 == 0. */
int yb_conv0_raw_stats_fwd(const float* x_nchw, const float* w_oihw, void* z_nhwc_f16, double* sums, int batch, int height, int width, int cout,
                           yb_stream_t stream);
/* data-gradient operand of a conv: fp16 [Cin][k][k][cout_pad], rotated 180 degrees, Cout zero-padded to cout_pad. */
int yb_pack_weight_dgrad_f16(const float* w_oihw, void* w_f16, int cout, int cin, int ksize, int cout_pad, yb_stream_t stream);
/* Both operands of many units in ONE launch (a training step re-packs every weight: the optimizer just changed them).  `units_dev` is a DEVICE array;
 * unit i owns blocks [block0, block0 + ceil(cout_pad / 64) * ci_blocks) with ci_blocks = ceil(cin / (ksize == 3 ? 32 : 256)); block0 ascending from 0;
 * cin and cout_pad even; out_fwd = the yb_pack_weight_f16 layout, out_dgrad = the yb_pack_weight_dgrad_f16 layout, either may be NULL. */
typedef struct yb_pack_unit {
  const float* w_oihw;
  void* out_fwd;
  void* out_dgrad;
  int cout, cin, ksize, cout_pad, block0, ci_blocks;
} yb_pack_unit;
int yb_pack_weights_batch(const yb_pack_unit* units_dev, int num_units, int total_blocks, yb_stream_t stream);
/* sums[0..C) += sum z, sums[C..2C) += sum z^2 over `rows` pixels (double, must be zero on entry; finalize re-zeroes). */
int yb_bn_stats(const void* z, long long ld, long long rows, int channels, double* sums, yb_stream_t stream);
int yb_bn_finalize(double* sums, long long rows, int channels, float eps, float momentum, float* running_mean, float* running_var,
                   float* mean, float* invstd, yb_stream_t stream);
int yb_bn_act_apply(const void* z, long long ld_z, const float* mean, const float* invstd, const float* gamma, const float* beta,
                    float slope, void* a, long long ld_a, int a_ch_off, int batch, int height, int width, int channels, int pool,
                    yb_stream_t stream);
/* Backward through leaky + BN (+ pooling).  The gradient w.r.t. the unit's activated output arrives as `da`
 * (unpooled, [B,H,W,*], may be NULL) and/or `dap` (through the unit's MaxPool2d(2), [B,H/2,W/2,*], routed to the
 * first maximum of each window; requires window = 1).  mode 0: sums += (sum dy, sum dy*xhat); mode 1: write dz.
 * has_bn = 0: unit without BatchNorm (bias gradient = sums[0..C)). */
int yb_bn_act_bwd(int mode, const void* z, long long ld_z, const float* mean, const float* invstd, const float* gamma, const float* beta,
                  float slope, const void* da, long long ld_da, int da_off, const void* dap, long long ld_dap, int dap_off, int batch,
                  int height, int width, int channels, int window, double* sums, void* dz, long long ld_dz, int has_bn, yb_stream_t stream);
/* dgamma = scale * sums[C..2C), dbeta = scale * sums[0..C) (scale = 1 / loss scale: gradients travel in fp16 multiplied by a static
 * loss scale); reset = 1 re-zeroes the accumulators for the next step. */
int yb_bn_param_grad(double* sums, int channels, float* dgamma, float* dbeta, int reset, float scale, yb_stream_t stream);
/* backward of model.yolo2.reorg + torch.cat (model/yolo2.py:33-46,129): un-permute channels [dy_off, dy_off+4C). */
int yb_reorg_bwd_f16(const void* dy, long long ld_dy, int dy_off, void* dx, int batch, int height, int width, int channels,
                     yb_stream_t stream);
/* head: dfeature fp32 NCHW [B,C,S,S] -> fp16 NHWC [B,S,S,channels_pad] (zero padded) + conv bias gradient [C]. */
int yb_head_grad_prepare(const float* dfeature, void* dz_nhwc_f16, float* dbias, int batch, int channels, int channels_pad, int cells,
                         yb_stream_t stream);
/* layers1.0 weight gradient [32,3,3,3] from the fp32 NCHW image and dz fp16 NHWC [B,H,W,32]. */
int yb_conv0_wgrad(const float* x_nchw, const void* dz_nhwc_f16, float* dw_oihw, int batch, int height, int width, yb_stream_t stream);
/* The same with the second pass of that layer's BatchNorm + leaky + 2x2 max-pool backward fused in (yb_bn_act_bwd mode 1, pooled gradient only):
 * reads the raw conv output z [B,H,W,32] and the gradient of the pooled activation dap [B,H/2,W/2,ld_dap] at channel dap_off, `sums` = the
 * double [2][32] of yb_bn_act_bwd mode 0; dz is formed in shared memory and never written (the image needs no data gradient). */
int yb_conv0_wgrad_bn(const float* x_nchw, const void* z_nhwc_f16, const void* dap, long long ld_dap, int dap_off, const float* mean, const float* invstd,
                      const float* gamma, const float* beta, float slope, const double* sums, float* dw_oihw, int batch, int height, int width,
                      yb_stream_t stream);
/* tcgen05 weight gradient: dw_krsc fp32 [Cout][k][k][Cin] (overwritten) from x fp16 NHWC [B,H,W,x_ld] and dz fp16 [B,H,W,dz_ld]. */
int yb_conv_wgrad(const void* x, const void* dz, float* dw_krsc, int batch, int height, int width, int cin, int cout, int ksize, int x_ld,
                  int dz_ld, yb_stream_t stream);
/* fp32 [Cout][k][k][Cin] (yb_conv_wgrad's layout) -> the reference's OIHW parameter-gradient layout, multiplied by `scale`. */
int yb_unpack_wgrad(const float* dw_krsc, float* dw_oihw, int cout, int cin, int ksize, float scale, yb_stream_t stream);

/* Guard of the fp16 / static-loss-scale backward (the reference trains in fp32 and has no such failure mode): found_inf[0] (device
 * float) = 1 if any of the `count` fp32 gradient values is inf / NaN, else 0; with zero_if_found the whole buffer is cleared in that case
 * so the optimizer takes a null step instead of absorbing the overflow into its state.  Asynchronous, no host sync, capturable. */
int yb_grad_guard(float* grads, long long count, float* found_inf, int zero_if_found, yb_stream_t stream);

/* ---- GPU input pipeline (SURVEY 8f rank 2; transform/resize/image.py:23-24, transform/resize/label.py:25-31, transform/image.py:27-29) ----
 * A batch of decoded uint8 HWC frames of DIFFERENT sizes -> [B,height,width,3] uint8 in one launch: cv2.resize(image, (width, height))
 * (8-bit INTER_LINEAR, bit-exact) + optional BGR->RGB swap.  src = packed frames, image i starts at byte src_off[i] and is
 * src_hw[2i] x src_hw[2i+1] pixels.  Optional boxes yx_min / yx_max [B,slots,2] (pixels of the source frame) are scaled in place by
 * (height / src_h, width / src_w).  The output feeds yb_conv0_u8_bn_leaky_pool_fwd (which applies ToTensor's 1/255). */
int yb_resize_batch_u8(const void* src, const long long* src_off, const int* src_hw, void* dst, int batch, int height, int width, int swap_rb,
                       float* yx_min, float* yx_max, int slots, yb_stream_t stream);

/* The training form of the same launch: out = cv2.resize(crop(flip(frame))) -- `transform.augmentation.flip_horizontally`
 * (transform/augmentation.py:87-95, cv2.flip(image, 1)) then `transform.resize.label.random_crop` (transform/resize/label.py:58-75: the
 * window image[y0:y1, x0:x1], then `rescale`), the default `resize_train` of config.ini:48.  flip: uint8[B] (NULL = none); crop: int[B][4] =
 * (y0, x0, y1, x1) in the flipped frame (NULL = whole frame); margin: float[B][2], the reference's un-truncated float32 crop origin that it
 * subtracts from the boxes.  Boxes are transformed in the reference's order and float32 arithmetic (flip, crop, scale).  Bit-exact with
 * cv2 for the pixels: both augmentations are index transforms on the source of the same resize. */
int yb_resize_aug_batch_u8(const void* src, const long long* src_off, const int* src_hw, const int* crop, const float* margin, const unsigned char* flip,
                           void* dst, int batch, int height, int width, int swap_rb, float* yx_min, float* yx_max, int slots, yb_stream_t stream);

/* cv2.warpAffine(frame, M, (dst_w, dst_h), INTER_LINEAR, BORDER_CONSTANT, fill) on one uint8 HWC frame, bit-exact: the image half of
 * `transform.augmentation.Rotator.__call__` / `random_rotate` (transform/augmentation.py:46-49,61-76) and of `transform.resize.image.fixed`
 * when it shrinks (transform/resize/image.py:36-46).  inverse_matrix6 / fill3 are HOST pointers: the 2x3 matrix already inverted the way
 * OpenCV does it (double), and the border colour per channel. */
int yb_warp_affine_u8(const void* src, int src_h, int src_w, void* dst, int dst_h, int dst_w, const double* inverse_matrix6, const int* fill3,
                      yb_stream_t stream);

/* torchvision ToTensor for a batch (the `transform_tensor` step, utils/data.py:120-121): uint8 NHWC [B,H,W,3] -> fp32 NCHW [B,3,H,W],
 * value / 255.  Only the training path needs the fp32 image (inference reads the uint8 frames in the first conv kernel). */
int yb_totensor_u8(const void* src_nhwc_u8, float* dst_nchw_f32, int batch, int height, int width, yb_stream_t stream);

/* Photometric training augmentations of transform/image.py:32-99 (RandomBlur, BGR2HSV, RandomHue, RandomSaturation, RandomBrightness,
 * HSV2RGB, RandomGamma; applied per resized image at utils/data.py:121) for a batch of same-size uint8 HWC frames [B,height,width,3] in
 * one launch, each image with its own parameters.  Stages in this order, each optional:
 *   blur_k  int[B][2] (kx, ky), 1 <= k <= 15 (NULL = no blur): cv2.blur(img, (kx, ky)), BORDER_REFLECT_101; src and dst must not alias
 *   to_hsv  cv2 COLOR_BGR2HSV, 8-bit (H in 0..179), bit-exact
 *   lut_hsv uint8[B][3][256] (NULL = identity): per-image, per-channel table (hue / saturation / brightness, composed on the host)
 *   to_rgb  cv2 COLOR_HSV2RGB, 8-bit, bit-exact
 *   lut_out uint8[B][3][256] (NULL = identity): per-image, per-channel table (gamma)
 * All pointers are device pointers.  The blur is cv2's arithmetic with one intended difference: an area-2 window of two 255s gives 255
 * (cv2 wraps it to 0 in its scalar tail loop, so its result depends on the row width).  Images whose (kx, ky) lie outside 1..15 are
 * left unwritten; the Python wrappers reject such draws before the launch. */
int yb_photometric_u8(const void* src, void* dst, int batch, int height, int width, const int* blur_k, int to_hsv, const unsigned char* lut_hsv,
                      int to_rgb, const unsigned char* lut_out, yb_stream_t stream);

/* ---- evaluation matching (SURVEY 8f rank 3; eval.py:57-75 `_matching`/`matching`, called per image and class at eval.py:210-216) ----
 * Segmented batch: image i owns detections [det_off[i], det_off[i+1]) (descending score within the image, as postprocess returns
 * them) and ground-truth boxes [gt_off[i], gt_off[i+1]); boxes are (y, x) float pairs, classes int32.  tp[d] = 1 iff detection d's
 * best-IoU ground truth of its own class (ties: lowest index) has IoU > threshold and was not claimed by an earlier detection of
 * the image.  IoU uses the reference's operation order (utils/iou/torch.py:24-61) with min_union = float32 eps. */
int yb_eval_match(const float* det_yx_min, const float* det_yx_max, const int* det_cls, const int* det_off, const float* gt_yx_min,
                  const float* gt_yx_max, const int* gt_cls, const int* gt_off, int batch, int num_cls, int max_gt, float threshold, float min_union,
                  unsigned char* tp, yb_stream_t stream);

/* ---- MobileNet plugin (model/mobilenet.py:25-85), inference ------------------------------------------------- */
/* conv_bn(3,32,stride 2) + BN + ReLU: x fp32 NCHW [B,3,H,W] -> y fp16 NHWC [B,H/2,W/2,32] (model/mobilenet.py:25-30). */
int yb_mb_conv0_bn_relu_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_nhwc_f16, int batch,
                            int height, int width, yb_stream_t stream);
/* conv_dw: depthwise 3x3 (stride 1 or 2, pad 1) + BN + ReLU on fp16 NHWC; w fp32 [C][9] (model/mobilenet.py:33-38). */
int yb_dwconv3x3_bn_relu_fwd(const void* x, const float* w_c9, const float* scale, const float* shift, void* y, int batch, int height,
                             int width, int channels, int stride, yb_stream_t stream);

/* ---- ResNet plugin (model/resnet.py:28-147), inference --------------------------------------------------------
 * stem: nn.Conv2d(3, 64, 7, stride 2, pad 3) + BatchNorm2d + ReLU (:107-109), x fp32 NCHW -> y fp16 NHWC [B,H/2,W/2,64]; nn.MaxPool2d(3, 2, 1) (:110);
 * x[:, ::2, ::2, :] -- a stride-2 "same" conv is its stride-1 form at the even pixels, so the stride-2 3x3 / 1x1 convs of the blocks (:33,:39,:65,:73)
 * run on yb_conv_bn_act_fwd + this selection; out = relu(a + b), the residual join (:58-59,:100-101). */
int yb_stem7x7_bn_relu_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_nhwc_f16, int batch, int height, int width,
                           yb_stream_t stream);
int yb_maxpool3x3_s2_f16(const void* x, void* y, int batch, int height, int width, int channels, yb_stream_t stream);
int yb_subsample2_f16(const void* x, void* y, int batch, int height, int width, int channels, yb_stream_t stream);
int yb_add_relu_f16(const void* a, const void* b, void* out, long long count, yb_stream_t stream);

/* ---- DenseNet plugin (model/densenet.py:29-117, torchvision's _DenseLayer / _Transition), inference -------------------------------------
 * The stem is yb_stem7x7_bn_relu_fwd (64 outputs: densenet121/169/201) or yb_stem7x7_96_bn_relu_fwd (96 outputs: densenet161), same contract.
 * yb_maxpool3x3_s2_strided_f16: yb_maxpool3x3_s2_f16 writing channels [y_ch_off, y_ch_off + channels) of an fp16 NHWC output of pitch y_ld (the first
 * dense block's concatenation buffer); yb_maxpool3x3_s2_f16 is its y_ld = channels, y_ch_off = 0 case.
 * yb_bn_relu_f16: y[p, c] = fp16(max(fmaf(x[p, c], scale[c], shift[c]), 0)) for c < channels, 0 for channels <= c < channels_padded; x and y fp16 with
 * pixel pitches x_ld / y_ld.  channels, channels_padded, x_ld, y_ld multiples of 8, pointers 16B aligned, else YB_ERR_BAD_ARG.
 * yb_bn_relu_avgpool2x2_f16: y[b, oy, ox, c] = fp16(0.25 * sum over rows 2oy..2oy+1, columns 2ox..2ox+1 of relu(fmaf(x, scale, shift))), summed in
 * fp32; x [B,H,W] of pitch x_ld, y contiguous [B, H/2, W/2, channels] (odd sizes floor, as AvgPool2d(2, 2)). */
int yb_stem7x7_96_bn_relu_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_nhwc_f16, int batch, int height,
                              int width, yb_stream_t stream);
int yb_maxpool3x3_s2_strided_f16(const void* x, void* y, int batch, int height, int width, int channels, int y_ld, int y_ch_off, yb_stream_t stream);
int yb_bn_relu_f16(const void* x, int x_ld, const float* scale, const float* shift, void* y, int y_ld, long long pixels, int channels, int channels_padded,
                   yb_stream_t stream);
int yb_bn_relu_avgpool2x2_f16(const void* x, int x_ld, const float* scale, const float* shift, void* y, int batch, int height, int width, int channels,
                              yb_stream_t stream);

/* Training of the MobileNet plugin: what torch autograd does for conv_bn / conv_dw (model/mobilenet.py:25-38).  The raw forms return the conv
 * output before BatchNorm / ReLU (train-mode statistics come from yb_bn_stats / yb_bn_finalize, the activation from yb_bn_act_apply with slope 0);
 * height / width are always those of the conv INPUT.  dgrad: da fp16 [B,H,W,C] from dz fp16 [B,H/stride,W/stride,C]; wgrad: dw fp32 [C][9]
 * (overwritten) from the input activation a and dz; first layer: dw fp32 OIHW [32,3,3,3] (overwritten) from the fp32 NCHW image and dz. */
/* Strict-precision forms of the two MobileNet-specific layers (`[b200] precision = strict` on this plugin): activations are [hi | lo] fp16 pairs,
 * y_hi_lo = [B,H/2,W/2,64] for the first conv, x_hi_lo [B,H,W,2C] -> y_hi_lo [B,H/stride,W/stride,2C] for the depthwise conv (computed on hi + lo in
 * fp32); the pointwise convs and the head run yb_conv_bn_act_split_fwd. */
int yb_mb_conv0_split_fwd(const float* x_nchw, const float* w_oihw, const float* scale, const float* shift, void* y_hi_lo, int batch, int height, int width,
                          yb_stream_t stream);
int yb_dwconv3x3_split_fwd(const void* x_hi_lo, const float* w_c9, const float* scale, const float* shift, void* y_hi_lo, int batch, int height, int width,
                           int channels, int stride, yb_stream_t stream);
int yb_mb_conv0_raw_fwd(const float* x_nchw, const float* w_oihw, void* z_nhwc_f16, int batch, int height, int width, yb_stream_t stream);
int yb_mb_conv0_wgrad(const float* x_nchw, const void* dz_nhwc_f16, float* dw_oihw, int batch, int height, int width, yb_stream_t stream);
int yb_dwconv3x3_raw_fwd(const void* x, const float* w_c9, void* z, int batch, int height, int width, int channels, int stride, yb_stream_t stream);
int yb_dwconv3x3_dgrad(const void* dz, const float* w_c9, void* da, int batch, int height, int width, int channels, int stride, yb_stream_t stream);
int yb_dwconv3x3_wgrad(const void* a, const void* dz, float* dw_c9, int batch, int height, int width, int channels, int stride, yb_stream_t stream);

/* ---- data-parallel gradient exchange (replaces nn.DataParallel's replicate / gather / reduce_add_coalesced, train.py:65-71) ----
 * One process per GPU.  The communicator is an NCCL communicator owned by this library (NCCL is bound with dlopen at the first
 * call: the libnccl.so.2 already in the process -- PyTorch ships one -- else the system's, else $YB_NCCL_PATH).
 *   yb_comm_unique_id   rank 0 creates the 128-byte rendezvous id; the caller ships it to the other ranks (any side channel);
 *   yb_comm_init        collective over all ranks, with the current CUDA device bound to the calling process' GPU;
 *   yb_allreduce_bucket in-place SUM over ranks of `count` elements of one gradient bucket, asynchronous on `stream` (the caller
 *                       orders it after the kernels that fill the bucket with CUDA events; capturable into a CUDA graph).  The
 *                       1/world of the average is folded into the gradient kernels' un-scaling (yb_unpack_wgrad `scale`, ...);
 *   yb_broadcast_buffer root's buffer to every rank (initial parameters / buffers, as DataParallel replicates GPU 0's);
 *   yb_comm_destroy     after every CUDA graph that captured a collective has been destroyed.
 * dtype: 0 = float32, 1 = float16, 2 = bfloat16, 3 = int32. */
int yb_comm_version(int* nccl_version);
int yb_comm_unique_id(void* id128);
int yb_comm_init(void** comm, int nranks, const void* id128, int rank);
int yb_comm_destroy(void* comm);
int yb_allreduce_bucket(void* comm, void* buf, long long count, int dtype, yb_stream_t stream);
int yb_broadcast_buffer(void* comm, void* buf, long long count, int dtype, int root, yb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* YOLO2_B200_H_ */
