/*
 * vps_b200.h -- C ABI of libvps_b200.so (sm_100a kernels for the FuseTrack frame-pair path).
 *
 * Every entry point takes plain device pointers, sizes and a cudaStream_t (as void*), returns an
 * int status (0 = ok, negative = VPS_E_*), never throws across the ABI and never frees caller
 * memory.  Each declaration cites the reference interface (file:line under mcahny/vps) it replaces.
 *
 * Tensor convention (differs from the reference on purpose): activations are NHWC ("pixel-major")
 * with an explicit per-pixel channel stride `cs`, so a channel slice of a concat buffer is a view
 * (ptr + c_off, cs = total channels).  address(n,y,x,c) = ptr + ((n*h + y)*w + x)*cs + c.
 * dtype: VPS_F32 or VPS_BF16.  The boundary tensors of the detector (images in, label maps out)
 * stay NCHW fp32 / int64 exactly as in the reference; the layout conversion is one kernel each way.
 */
#ifndef VPS_B200_H_
#define VPS_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VPS_OK 0
#define VPS_E_ARG (-1)     /* bad argument / unsupported geometry */
#define VPS_E_CUDA (-2)    /* a CUDA runtime / driver call failed (see vps_last_error) */
#define VPS_E_NODEV (-3)   /* no sm_100 device */

#define VPS_F32 0
#define VPS_BF16 1

#define VPS_ACT_NONE 0
#define VPS_ACT_RELU 1
#define VPS_ACT_LRELU 2    /* negative slope in vps_conv_args.slope (reference uses 0.1) */
#define VPS_ACT_SIGMOID 3

typedef struct vps_tensor {
  void* ptr;
  int32_t n, h, w, c;   /* logical NHWC extent */
  int32_t cs;           /* channel stride: elements between consecutive pixels (>= c) */
  int32_t dtype;        /* VPS_F32 | VPS_BF16 */
} vps_tensor;

/* ---- library ------------------------------------------------------------------------------- */
const char* vps_last_error(void);
int vps_version(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches claim) */
int64_t vps_launch_count(void);
/* a CUDA-graph replay re-launches kernels without going through the C entry points: the caller reports them */
void vps_add_launch_count(int64_t n);

/* ---- dense contractions -------------------------------------------------------------------- */
/*
 * Convolution as implicit GEMM.  Replaces every nn.Conv2d / ConvTranspose2d / nn.Linear call on
 * the path (cuDNN/cuBLAS in the reference; e.g. resnet.py:506-517, fpn.py:100-139,
 * tcea_modules.py:50-78, FlowNetS.py:62-94, convfc_bbox_head.py:132-168, fcn_mask_head.py:94-103)
 * and the GEMM half of DCNv1 (deform_conv_cuda.cpp:231-236).
 *
 *   y[n, oy*oy_mul+oy_off, ox*ox_mul+ox_off, co] =
 *       act( bias[co] + sum_{r,s,ci} x[n, oy*sh - ph + r, ox*sw - pw + s, ci] * W[co,r,s,ci] ) (+ res)
 *
 * for oy < oh, ox < ow.  Out-of-range input taps read zero.  (oy_mul,oy_off,...) let a transposed
 * convolution run as stride-phase sub-convolutions writing interleaved output pixels.
 *
 * vps_conv2d_tc   : bf16 operands, fp32 accumulation on tcgen05 tensor cores (TMA im2col tiles,
 *                   accumulators in TMEM).  w = bf16 [cout_pad][kh*kw*cin_pad] (ci fastest,
 *                   cin_pad = cin rounded up to cin_gran (64 or 16), cout_pad to 16), from vps_pack_weights_tc.
 *                   x must be VPS_BF16 with cs % 8 == 0 and 16-byte aligned ptr.
 * vps_conv2d_simt : fp32 (or bf16 storage) direct convolution on CUDA cores with fp32 FMA --
 *                   the parity-mode path and the path for tiny channel counts.
 *                   w = f32 [kh][kw][cin][cout].
 */
typedef struct vps_conv_args {
  vps_tensor x, y, res;       /* res.ptr == NULL: no residual.  res is added AFTER act when
                                 res_after_act != 0, else before (ResNet: add then ReLU). */
  const void* w;
  const float* bias;          /* [cout] fp32 or NULL */
  int32_t kh, kw, sh, sw, ph, pw;
  int32_t oh, ow;
  int32_t oy_mul, oy_off, ox_mul, ox_off;
  int32_t cin, cout;
  int32_t act;
  float slope;
  int32_t res_after_act;
  float out_scale;            /* y = out_scale * act(...) ; 1.0 normally (FlowNet2 div_flow folds here) */
  int32_t cin_gran;           /* tc only: 64 (default, 0) or 16 = channel granularity of the packed weights / K step */
} vps_conv_args;

int vps_conv2d_tc(const vps_conv_args* a, void* stream);
/* up to 4 problems sharing x / y / geometry / bias / activation and differing in w, (ph,pw) and (oy_off,ox_off):
 * the stride phases of a ConvTranspose2d (submodules.py:33-37, fcn_mask_head.py:66-71) in one persistent launch. */
int vps_conv2d_tc_multi(const vps_conv_args* a, int nprob, void* stream);
int vps_conv2d_simt(const vps_conv_args* a, void* stream);
/* OIHW fp32 (torch layout, on device) -> packed layouts.  scale[cout] (may be NULL) is folded in
 * (frozen BatchNorm: resnet.py:519-526).  transposed != 0: src is IOHW (ConvTranspose2d). */
int vps_pack_weights_tc(const float* w_oihw, const float* scale, void* dst_bf16, int cout, int cin,
                        int kh, int kw, int transposed, int cin_gran, void* stream);
int vps_pack_weights_simt(const float* w_oihw, const float* scale, float* dst, int cout, int cin,
                          int kh, int kw, int transposed, void* stream);
/* bytes of the packed tc weight buffer */
int64_t vps_packed_tc_bytes(int cout, int cin, int kh, int kw, int cin_gran);

/* ---- fp32-parity tensor-core convolution ("tc32" precision) ------------------------------------
 * Same contract as vps_conv2d_tc, but x (and y, res) are fp32: the reference's convolutions are fp32 cuDNN calls
 * (resnet.py:506-517, flownet2.py:133-198, fpn.py:100-139 ...) and north_star asks for label maps / ids bit-exact.
 * Each operand is split on the fly into two fp16 planes, v = A + 2^-11 * A2 with A = fp16(v), A2 = fp16(2^11 (v - A)),
 * and three tcgen05 products
 *   A*B + 2^-11 * (A2*B + A*B2)
 * are summed (~2^-21 relative per product, 3 tensor-core passes; below 2^-14 an operand carries an absolute error of
 * 2^-36).  Because tcgen05.mma truncates when it adds into its accumulator, the main product is accumulated in short chains
 * that are promoted to round-to-nearest register sums (conv_tc32.cu).  Weights are pre-split by vps_pack_weights_tc32 into
 * two fp16 planes [B | B2]; the nprob stride phases of a transposed convolution share ONE packed buffer (args[i].w
 * identical, problem i = plane slice i).
 * |value| > 65504 (or NaN) in x or w saturates the fp16 planes (the result is then wrong) and is counted:
 * vps_tc32_overflow(reset) returns the count (device sync) -- callers must treat non-zero as an error. */
int vps_conv2d_tc32(const vps_conv_args* a, void* stream);
int vps_conv2d_tc32_multi(const vps_conv_args* a, int nprob, void* stream);
int vps_pack_weights_tc32(const float* w_oihw, const float* scale, void* dst, int cout, int cin, int kh, int kw,
                          int transposed, int prob, int nprob, void* stream);
int64_t vps_packed_tc32_bytes(int cout, int cin, int kh, int kw, int nprob);
int vps_tc32_overflow(int reset);
/* fused DCNv1 3x3 in the tc32 precision (deform_conv.py:15-87 forward; deform_conv_cuda.cpp:152-260 = deformable_im2col +
 * GEMM): the sampling warps write the split operand planes straight into the tensor-core ring, no column matrix.
 * x fp32 NHWC (c % 32 == 0), offset fp32 NHWC [..,18], w = vps_pack_weights_tc32 buffer of the [cout,cin,3,3] kernel. */
int vps_deform_conv_tc32(const vps_tensor* x, const vps_tensor* offset, const void* w, int cout, const vps_tensor* y,
                         void* stream);

/* explicit im2col for small-cin layers feeding vps_conv2d_tc as a 1x1 conv: cols is NHWC
 * [n, oh, ow, kpad] with k = (r*kw+s)*cin + ci, zero padded to cols.c. */
int vps_im2col(const vps_tensor* x, const vps_tensor* cols, int kh, int kw, int sh, int sw, int ph,
               int pw, void* stream);

/* ---- FlowNet2 native ops --------------------------------------------------------------------- */
/* correlation_cuda.forward (correlation_cuda.cc:10-87, correlation_cuda_kernel.cu:74-147),
 * kernel_size 1.  out channel (tj+R)*D+(ti+R), R = max_disp/stride2, D = 2R+1; out = sum_c / C.
 * Optional fused LeakyReLU (FlowNetC.py:33,87).  f1,f2,out NHWC. */
int vps_correlation(const vps_tensor* f1, const vps_tensor* f2, const vps_tensor* out, int pad,
                    int max_disp, int stride1, int stride2, int act, float slope, void* stream);
/* the two implementations behind vps_correlation: banded GEMM on tcgen05 (bf16 features, C % 64 == 0, C <= 256,
 * the (pad 20, d 20, s2 2) and (pad 4, d 4, s2 1) call sites) and the CUDA-core kernel (any dtype; parity mode). */
int vps_correlation_tc(const vps_tensor* f1, const vps_tensor* f2, const vps_tensor* out, int pad,
                       int max_disp, int stride1, int stride2, int act, float slope, void* stream);
int vps_correlation_simt(const vps_tensor* f1, const vps_tensor* f2, const vps_tensor* out, int pad,
                         int max_disp, int stride1, int stride2, int act, float slope, void* stream);
/* correlation of fp32 features on the tensor cores in the parity precision (tc32): operands split into fp16 planes
 * (v = hi + 2^-11 lo), three banded-GEMM passes (hi.hi + 2^-11 (hi.lo + lo.hi)) accumulated in the fp32 output.  Same call sites /
 * geometries as vps_correlation_tc (correlation_cuda.cc:10-87); ws = vps_correlation_tc32_ws_bytes(f1) bytes, 256-byte aligned. */
int64_t vps_correlation_tc32_ws_bytes(const vps_tensor* f1);
int vps_correlation_tc32(const vps_tensor* f1, const vps_tensor* f2, const vps_tensor* out, int pad, int max_disp, int stride1,
                         int stride2, int act, float slope, void* ws, void* stream);

/* resample2d_cuda.forward (resample2d_cuda.cc:6-31, resample2d_kernel.cu:16-71): bilinear warp by
 * pixel-unit flow (channel 0 = x), border-clamped taps, kernel_size 1. */
int vps_resample2d(const vps_tensor* src, const vps_tensor* flow, const vps_tensor* out, void* stream);
/* channelnorm_cuda.forward (channelnorm_cuda.cc:6-30, channelnorm_kernel.cu:19-60): sqrt(sum_c x^2);
 * computes the norm of (a - b) when b != NULL (fuses flownet2.py:147-148). out has 1 channel. */
int vps_channelnorm(const vps_tensor* a, const vps_tensor* b, const vps_tensor* out, void* stream);

/* compute_flow head (panoptic_fusetrack.py:119-121 denormalize, flownet2.py:135-139): rgb = img*std+mean
 * for both NCHW fp32 frames, per-channel mean over both frames, x = (rgb - mean)/rgb_max -> NHWC [1,H,W,6]
 * (img 0..2, ref 3..5).  std3/mean3 are HOST arrays of 3 floats; sums_ws = 3 device doubles. */
int vps_flownet_input(const float* img_nchw, const float* ref_nchw, int H, int W, const float* std3,
                      const float* mean3, float rgb_max, double* sums_ws, const vps_tensor* x, void* stream);

/* Fused construction of FlowNet2's stage inputs (flownet2.py:142-153): cat[12] = (x6 | resample2d(img1 = x6[3:6], flow) |
 * flow / div | channelnorm(img0 - resampled)) with flow = bilinear upsample (align_corners False) of flow_lo [n,h,w,2] f32
 * times mul; inv = 1 / div_flow.  One pass, one whole-pixel store; bit-identical to vps_resize_bilinear + vps_axpby +
 * vps_resample2d + vps_channelnorm.  cat must be a full buffer (its channel padding is zeroed). */
int vps_flownet_stage(const vps_tensor* x6, const vps_tensor* flow_lo, float mul, float inv, const vps_tensor* cat, void* stream);
/* concat3 of flownet2.py:176-189: cat[11] = (img0 | sd_flow | s2_flow | |sd_flow| | |s2_flow| | |img0 - warp(img1, sd_flow)| |
 * |img0 - warp(img1, s2_flow)|), the flows being nearest-upsampled low-resolution f32 flows times mul_s2 / mul_sd. */
int vps_flownet_cat3(const vps_tensor* x6, const vps_tensor* s2_flow_lo, const vps_tensor* sd_flow_lo, float mul_s2, float mul_sd,
                     const vps_tensor* cat, void* stream);

/* nn.ConvTranspose2d(2, 2, 4, 2, 1): the `upsampled_flow*_to_*` layers of every FlowNet (FlowNetS.py:45-48,
 * FlowNetC.py:48-51, FlowNetSD.py:45-48, FlowNetFusion.py:34-35).  w_iohw_host = 64 HOST floats [ci][co][ky][kx],
 * bias_host = 2 HOST floats or NULL (they travel as kernel arguments); x [n,h,w,2] -> y [n,2h,2w,2] (a concat slice). */
int vps_flow_deconv(const vps_tensor* x, const float* w_iohw_host, const float* bias_host, const vps_tensor* y,
                    void* stream);

/* ---- layout / pointwise / resampling --------------------------------------------------------- */
int vps_nchw_to_nhwc(const float* src, const vps_tensor* dst, void* stream);   /* src [n,c,h,w] f32 */
int vps_nhwc_to_nchw(const vps_tensor* src, float* dst, void* stream);
/* dst = alpha * src (+ beta) channel-slice copy with dtype conversion */
int vps_copy_scale(const vps_tensor* src, const vps_tensor* dst, float alpha, void* stream);
/* out = a*alpha + b*beta (b may be NULL) */
int vps_axpby(const vps_tensor* a, const vps_tensor* b, const vps_tensor* out, float alpha, float beta,
              void* stream);
/* F.interpolate bilinear align_corners=False (torch semantics incl. scale = in/out), out size from `out`;
 * result multiplied by `mul` (panoptic_fusetrack.py:141-142, upsnetFPN.py:74-80, flownet2.py:45,57). */
int vps_resize_bilinear(const vps_tensor* src, const vps_tensor* out, float mul, void* stream);
/* F.interpolate nearest: src index = floor(dst * in/out) (fpn.py:112-113, flownet2.py:72-73);
 * accumulate != 0: out += (FPN top-down add). */
int vps_resize_nearest(const vps_tensor* src, const vps_tensor* out, float mul, int accumulate, void* stream);
/* space-to-depth, block 2: y[n,Y,X,(dy*2+dx)*C+c] = x[n,2Y+dy,2X+dx,c].  Lets the 7x7 stride-2 stem convolutions
 * (resnet.py:436-451, FlowNetC.py:20 / FlowNetS.py:20 conv1) run as 4x4 stride-1 implicit GEMMs on the tensor cores. */
int vps_space_to_depth2(const vps_tensor* x, const vps_tensor* y, void* stream);
/* second half of a 3x3 / stride 1 / pad 1 convolution with <= 3 output channels (FlowNet2 predict_flow*, submodules.py:27-28)
 * whose first half ran as a 1x1 convolution with the taps on the output-channel axis (z[p][t*cout+co], t = 3*r+s):
 * out[n,y,x,co] = act(bias[co] + sum_t z[n, y+r-1, x+s-1, t*cout+co]) * out_scale, zero outside the map.  fp32 tensors. */
int vps_tap_gather3x3(const vps_tensor* z, const vps_tensor* out, const float* bias, int act, float slope, float out_scale,
                      void* stream);
/* max / avg pool (resnet.py:451, tcea_modules.py:27-28; avg = count_include_pad) */
int vps_pool2d(const vps_tensor* src, const vps_tensor* out, int k, int s, int p, int is_avg, void* stream);
/* GroupNorm(groups, eps) + optional ReLU (upsnetFPN.py:42-51) */
int vps_groupnorm(const vps_tensor* x, const vps_tensor* y, const float* gamma, const float* beta, int groups,
                  float eps, int relu, void* stream);

/* ---- BFPTcea -------------------------------------------------------------------------------- */
/* gather: mean over levels of nearest-upsampled maps (bfp_tcea.py:96-109), refine_level 0 */
int vps_bfp_gather(const vps_tensor* levels, int nlev, const vps_tensor* out, void* stream);
/* scatter: out_i = adaptive_max_pool2d(bsf, size_i) + in_i (bfp_tcea.py:141-147) */
int vps_bfp_scatter(const vps_tensor* bsf, const vps_tensor* in, const vps_tensor* out, void* stream);
/* WarpingLayer (flow_modules.py:126-148): grid_sample(bilinear, zeros, align_corners=False) at
 * ix = (x + fx) * W/(W-1) - 0.5 */
int vps_flow_warp(const vps_tensor* src, const vps_tensor* flow, const vps_tensor* out, void* stream);
/* TCEA temporal attention (tcea_modules.py:52-61): out[:, f*C:(f+1)*C] = fea_f * sigmoid(sum_c emb_f*emb_ref) */
int vps_tcea_temporal(const vps_tensor* fea0, const vps_tensor* fea1, const vps_tensor* emb0,
                      const vps_tensor* emb1, const vps_tensor* emb_ref, const vps_tensor* out, void* stream);
/* fea * sigmoid(att) * 2 + att_add (tcea_modules.py:75-77) */
int vps_tcea_combine(const vps_tensor* fea, const vps_tensor* att, const vps_tensor* att_add,
                     const vps_tensor* out, void* stream);

/* ---- DCNv1 ---------------------------------------------------------------------------------- */
/* Fused DCNv1 forward (deform_conv.py:15-87 -> deform_conv_cuda.cpp forward, deformable_im2col + GEMM) for the
 * configuration the FuseTrack path uses: 3x3, stride 1, pad 1, dilation 1, 1 group, 1 deformable group, no bias.
 * x bf16 NHWC (cin %% 64 == 0), offset f32 NHWC [.., >= 18] = (dy, dx) per tap, w = vps_pack_weights_tc layout of the
 * OIHW kernel (cin_gran 64), y bf16 or f32 NHWC with cout <= 256 channels.  The sampled columns go straight into the
 * tensor-core operand ring in shared memory; same bf16 columns as vps_deform_im2col + vps_conv2d_tc (1x1), summed over
 * K chunk-major instead of tap-major (results agree to one bf16 rounding). */
int vps_deform_conv_tc(const vps_tensor* x, const vps_tensor* offset, const void* w, int cout, const vps_tensor* y,
                       void* stream);
/* deformable_im2col (deform_conv_cuda_kernel.cu:83-113,189-242), 3x3 stride 1 pad 1 dil 1,
 * deformable_group 1.  offset NHWC [n,h,w,18] (ch 2k = dy, 2k+1 = dx); cols NHWC [n,h,w,9*c] (k-major). */
int vps_deform_im2col(const vps_tensor* x, const vps_tensor* offset, const vps_tensor* cols, void* stream);

/* ---- detection ops --------------------------------------------------------------------------- */
/* RoIAlign legacy mmdet v1 (roi_align_kernel.cu:16-128) with FPN level mapping
 * (single_level.py:54-73, finest_scale 56), all levels in one launch.  feats: nlev NHWC maps,
 * strides[nlev]; rois device f32 [nroi,5] (batch,x1,y1,x2,y2); out NHWC [>=nroi, ps, ps, c]
 * (flattened (ph,pw,c): the FC weights are permuted to this order at pack time).
 * nroi_dev (may be NULL) = device int holding the valid count; rows beyond it are zero-filled. */
int vps_roi_align(const vps_tensor* feats, const int* strides, int nlev, const float* rois, int nroi,
                  const int* nroi_dev, const vps_tensor* out, int sample_num, void* stream);
/* stable descending radix sort of float keys with their original indices (ties keep ascending index:
 * the pinned version of the reference's unspecified topk / argsort tie order, SURVEY A.9).
 * ws must hold at least n*4 + 256 + cub temp bytes (n*24 + 64 KiB is always enough). */
int vps_sort_desc(const float* keys, float* keys_out, int32_t* idx_out, int n, void* ws, int64_t ws_bytes,
                  void* stream);
/* RPN objectness (rpn_head.py:69-72): sigmoid of an NHWC score map, flattened in the reference's
 * (h, w, anchor) order into dst[h*w*c]. */
int vps_sigmoid_flat(const vps_tensor* src, float* dst, void* stream);
/* RPN per-level candidate decode (rpn_head.py:73-85 + delta2bbox transforms.py:34-68, means 0 stds 1):
 * for the top k sorted flat indices: anchor from index, decode, clamp to the image;
 * dets [k,5] = (x1,y1,x2,y2,score) in score order. */
int vps_rpn_decode(const float* scores_sorted, const int32_t* idx_sorted, int k, const vps_tensor* deltas,
                   int feat_h, int feat_w, int stride, const float* base_anchors, int num_anchors,
                   float img_h, float img_w, float* dets, void* stream);
/* greedy NMS (nms_kernel.cu:13-131 / upsnet nms_kernel.cu:40-150): dets [n,5] already sorted by score
 * (descending); IoU with +1 extents, suppress when IoU > thr.  Bitmask kernel + the reference's host
 * greedy loop run as a single-block device pass: no D2H.  keep_idx[0..*nkeep) = kept positions,
 * ascending (= score order).  If n_dev != NULL the valid count is read from it (<= n).
 * ws >= n * ceil(n/64) * 8 bytes. */
int vps_nms(const float* dets, int n, const int* n_dev, float thr, int32_t* keep_idx, int* nkeep,
            void* ws, int64_t ws_bytes, void* stream);
/* nb (<= 8) independent NMS problems in one launch pair -- the per-level NMS of get_bboxes_single
 * (rpn_head.py:55-104): problem b = rows [b*seg, b*seg + ns[b]) of dets (ns = host array; n_dev, if given, is a device
 * array of nb valid counts), keep_idx + b*seg / nkeep[b] its result.  ws >= nb * seg * ceil(max ns / 64) * 8 bytes. */
int vps_nms_batch(const float* dets, int nb, int seg, const int* ns, const int* n_dev, float thr,
                  int32_t* keep_idx, int* nkeep, void* ws, int64_t ws_bytes, void* stream);
/* dst[i,:] = src[idx[i],:] for i < n (valid count from n_dev if given; rows beyond are zeroed) */
int vps_gather_rows(const float* src, const int32_t* idx, int n, const int* n_dev, int width, float* dst,
                    void* stream);
/* MaskROI pre-NMS (mask_roi.py:37-93 + upsnet bbox_transform.py:290-330 weights (10,10,5,5) +
 * clip_boxes :45-60): slot (roi*8 + class-1) of cand [nroi*8,5] gets the decoded, clipped box and
 * softmax prob if prob > score_thr, else prob = -1 (class-agnostic fold order, deterministic);
 * *ncand = number of valid slots. */
int vps_maskroi_candidates(const float* rois, const float* cls_score, const float* bbox_pred,
                           int row_stride /* floats between consecutive RoI rows of cls_score / bbox_pred */, int nroi,
                           const int* nroi_dev, int num_classes, float score_thr, float img_h, float img_w,
                           float* cand, int32_t* cand_cls, float* cand_prob, int* ncand, void* stream);
/* tracker (track_head.py:73-132, panoptic_fusetrack.py:412-469): dots = emb . ref_emb^T,
 * comp = log_softmax([0|dots]) + c0*log(p) + c1*[0|IoU] + c2*[1|label eq], row argmax (first max),
 * then the sequential id-assignment loop on one device thread.  Outputs det_obj_ids[k], match_ids[k],
 * comp_scores [k,m+1], mem_src[cap] (detection whose RoI features/box end in memory slot j, -1 =
 * unchanged) and *new_m.  ws >= (k*m + k + 2*cap)*4 bytes. */
int vps_track_assign(const float* emb, const float* ref_emb, int k, int m, int dim, const float* det_boxes,
                     const float* ref_boxes, const int32_t* det_labels, const int32_t* ref_labels,
                     const float* cls_prob, float c0, float c1, float c2, int cap, int32_t* det_obj_ids,
                     int32_t* match_ids, float* comp_scores, int32_t* mem_src, int* new_m, void* ws,
                     int64_t ws_bytes, void* stream);

/* RPN tail (rpn_head.py:94-103): dets_cat = nlev segments of `seg` rows [x1,y1,x2,y2,score] with counts[l]
 * valid rows each; stable top-`cap` by score -> proposals [cap,5] and rois [cap,5] = (0,x1,y1,x2,y2)
 * (bbox2roi, transforms.py:106-125); *total = min(cap, sum counts).  Workspaces: scores_ws/scores_sorted_ws
 * [nlev*seg] f32, idx_sorted_ws [nlev*seg] i32, sort_ws as for vps_sort_desc. */
int vps_rpn_finalize(const float* dets_cat, const int* counts, int nlev, int seg, int cap, float* scores_ws,
                     float* scores_sorted_ws, int32_t* idx_sorted_ws, void* sort_ws, int64_t sort_ws_bytes,
                     float* proposals, float* rois, int* total, void* stream);
/* MaskROI tail (mask_roi.py:95-147): NMS survivors `keep[0..*nkeep)` (positions in the score-sorted candidate
 * list) -> max_det rule (scores >= the max_det-th best) -> det_rois [cap,5] (batch 0), cls_idx, cls_prob;
 * kout[0] = k, kout[1] = 1 when the dummy "no detection" result (score 1, zero box, class 0) was emitted. */
int vps_maskroi_finalize(const float* cand_sorted, const int32_t* slot_sorted, const int32_t* cand_cls,
                         const int32_t* keep, const int* nkeep, int max_det, int cap, float* det_rois,
                         int32_t* cls_idx, float* cls_prob, int* kout, void* stream);
/* det_bboxes = roi2bbox(det_rois) (transforms.py:128-135) and det_labels = cls_idx - 1
 * (panoptic_fusetrack.py:386-389): det_rois [cap,5] -> boxes [cap,4], labels [cap]. */
int vps_det_split(const float* det_rois, const int32_t* cls_idx, int cap, float* boxes, int32_t* labels,
                  void* stream);
/* mask_score.gather(1, cls_idx) (panoptic_fusetrack.py:566-568): logits NHWC [>=k,ms,ms,9] -> out f32 [k,ms,ms] */
int vps_select_class(const vps_tensor* logits, const int32_t* cls_idx, int k, float* out, void* stream);
/* tracker memory update (panoptic_fusetrack.py:441-443,458-459,467-469): for j < *new_m with mem_src[j] >= 0:
 * mem_feats[j] <- det_feats[mem_src[j]], mem_boxes likewise, mem_labels only for appended slots (j >= old_m). */
int vps_track_update(void* mem_feats, const void* det_feats, int dtype, int64_t feat_len, float* mem_boxes,
                     const float* det_boxes, int32_t* mem_labels, const int32_t* det_labels,
                     const int32_t* mem_src, int old_m, int cap, const int* new_m_dev, void* stream);

/* ---- panoptic fusion ------------------------------------------------------------------------- */
/* MaskRemoval (mask_removal.py:29-92): boxes [k,4] f32, mask_logit [k,ms,ms] f32, cls_idx[k] (1-based),
 * order[k] = detection indices sorted by prob (descending, stable).  cv2.resize(INTER_LINEAR) of each
 * 28x28 logit map is evaluated on the fly; occ = uint8 [num_things,H,W] class occupancy workspace.
 * Outputs keep_flag[k] (sorted order), keep_sorted[0..*nkeep) = kept detection indices in sorted order.
 * counters: uint32 [2k] workspace. */
int vps_mask_removal(const float* boxes, const int32_t* order, int k, const int* k_dev,
                     const float* mask_logit, int msize, const int32_t* cls_idx, int H, int W, float frac_thr,
                     uint8_t* occ, int num_things, unsigned int* counters, int32_t* keep_flag,
                     int32_t* keep_sorted, int* nkeep, void* stream);
/* final fusion (SegTerm unary_logits.py:81-108, paste mask_removal.py:86, argmax
 * panoptic_fusetrack.py:588-593): per full-resolution pixel, fcn_output = bilinear x4 of fcn_score
 * (upsnetFPN.py:59,80) computed in registers; pano_out = argmax over [stuff(num_stuff) | kept
 * instances (seg term + pasted mask logit)], sem_out = argmax over all classes; [H,W] each, stored as int64
 * (label_bytes 8, the dtype torch.max returns in the reference) or uint8 (label_bytes 1, same values, 8x less D2H).
 * dummy != 0: the MaskROI "no detection" result (one all-zero instance channel). */
int vps_panoptic_fuse(const vps_tensor* fcn_score, const float* boxes, const int32_t* cls_idx,
                      const float* mask_logit, int msize, const int32_t* keep_sorted, const int* nkeep_dev,
                      int kcap, int num_stuff, int dummy, int H, int W, void* pano_out, void* sem_out,
                      int label_bytes, void* stream);

/* ---- SURVEY 8f rank 1: the step right after the hot path ------------------------------------------------------
 * get_unified_pan_result for ONE frame (tools/dataset/cityscapes_vps.py:183-224): seg / pan = the [H,W] label maps of
 * simple_test (uint8, or int64 of which the low byte is used -- the reference's collector casts to uint8,
 * tools/test_vpq.py:52-56); cls_ind[k] = panoptic_cls_inds, obj_id[k] = track ids after the reference's duplicate
 * re-numbering (host state, see vps_b200/postproc.py) or NULL -- both are HOST arrays (k <= 256, passed to the kernel by
 * value); id_last_stuff = num_seg_classes - num_classes (10).
 * out = uint8 [H,W,3] = (semantic, instance rank, track id + 1).  One histogram pass + a 256-entry look-up-table pass;
 * ws >= vps_unify_pan_ws_bytes() bytes, 16-byte aligned. */
int64_t vps_unify_pan_ws_bytes(void);
int vps_unify_pan(const void* seg, const void* pan, int label_bytes, int H, int W, const int32_t* cls_ind,
                  const int32_t* obj_id, int k, int id_last_stuff, int stuff_area_limit, uint8_t* out, void* ws,
                  int64_t ws_bytes, void* stream);
/* 1 if the last vps_unify_pan call on `ws` met a panoptic instance id without a cls_ind entry (the reference raises
 * IndexError there, cityscapes_vps.py:197); synchronises `stream` */
int vps_unify_pan_error(const void* ws, void* stream);
int64_t vps_unify_pan_error_offset(void);   /* byte offset of that flag (int32) inside ws, for asynchronous read-back */

/* ---- SURVEY 8f rank 2: pixel-level step of the VPQ evaluator (tools/eval_vpq.py:138-145) --------------------------
 * np.unique(gt.astype(uint64) * offset + pred, return_counts=True) over a tube of id maps (npix = nframes*H*W, device
 * uint32): pairs_out (ascending) / counts_out must have room for npix entries, *nruns_dev receives the number of distinct
 * pairs.  64-bit radix sort + run-length encode; ws >= vps_tube_confusion_ws_bytes(npix), 256-byte aligned.
 * vps_rgb_to_id decodes an RGB-coded id image [npix,3] (r + 256 g + 65536 b, eval_vpq.py:87-89). */
int64_t vps_tube_confusion_ws_bytes(int64_t npix);
int vps_tube_confusion(const uint32_t* gt_ids, const uint32_t* pred_ids, int64_t npix, uint64_t offset, uint64_t* pairs_out,
                       uint32_t* counts_out, int* nruns_dev, void* ws, int64_t ws_bytes, void* stream);
int vps_rgb_to_id(const uint8_t* rgb, int64_t npix, uint32_t* ids, void* stream);
/* segment ids of a unified 3-channel result [npix,3] (vps_unify_pan): the segmentation converter_2ch_track_core
 * (tools/dataset/cityscapes_vps.py:104-140) produces through panopticapi's colours -- ONE segment per stuff category
 * (semantic < num_stuff: id 1000 * semantic + 1, whatever the track channel holds), one per (thing category, track) key
 * (id 1000 * semantic + track + 1), VOID (semantic 255) -> 0 */
int vps_pan2ch_ids(const uint8_t* pan_2ch, int64_t npix, int num_stuff, uint32_t* ids, void* stream);

/* ---- input stage (SURVEY 8f rank 4) -----------------------------------------------------------------------------------------
 * Normalize (mmcv.imnormalize: float32, BGR->RGB, (x - mean) / std; transforms.py:295-318) + Pad(size_divisor) (zero pad bottom /
 * right, :238-270) + ImageToTensor (HWC -> CHW, formating.py:46-68) of one uint8 HWC BGR frame in one pass: out is fp32 NCHW
 * [1,3,hp,wp].  mean3 / std3 are HOST arrays in output-channel order (RGB when to_rgb).  Bit-identical to the numpy arithmetic. */
int vps_preprocess_u8(const uint8_t* bgr_hwc, int h, int w, const float* mean3, const float* std3, int to_rgb,
                      float* out_nchw, int hp, int wp, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VPS_B200_H_ */
