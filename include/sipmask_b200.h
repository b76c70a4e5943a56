/*
 * sipmask_b200 - C ABI of the B200-native SipMask inference hot path.
 *
 * Drop-in boundary (SURVEY.md §8b).  Every entry point replaces one native
 * (pybind) entry point or one python/ATen call sequence of the reference
 * (JialeCao001/SipMask @ bc63fa9, paths relative to SipMask-mmdetection/mmdet/).
 *
 * Conventions
 *   - extern "C", plain pointers + sizes, no torch types.
 *   - all pointers are DEVICE pointers unless named host_*; the caller owns every
 *     buffer including workspaces (query with *_workspace_bytes); the library never
 *     allocates or frees device memory and never synchronises the device.
 *   - every launch goes to the caller's `stream` (the reference's CropSplit launches on
 *     the legacy default stream, ops/crop/src/crop_split_cuda_kernel.cu:77 - fixed here).
 *   - return 0 on success, a negative SMB_E* code otherwise; smb_last_error() gives a
 *     thread-local message.  (The reference only printf()s CUDA launch errors,
 *     crop_split_cuda_kernel.cu:81-85.)
 *   - dtype codes: SMB_F32 = 0, SMB_F16 = 1.
 */
#ifndef SIPMASK_B200_H_
#define SIPMASK_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* smb_stream_t; /* == cudaStream_t */

#define SMB_OK 0
#define SMB_EINVAL (-1)   /* bad argument / unsupported shape */
#define SMB_ECUDA (-2)    /* CUDA runtime / driver error      */
#define SMB_EWORKSPACE (-3) /* workspace too small            */
#define SMB_EARCH (-4)    /* device is not sm_100             */

#define SMB_F32 0
#define SMB_F16 1

const char* smb_last_error(void);
int smb_version(void);
/* 0 if the current device can run the sm_100a kernels, SMB_EARCH otherwise. */
int smb_check_device(void);

/* ------------------------------------------------------------------ mask assembly
 * Replaces sipmask_head.py:615-627: 4x (protos @ cof_k^T) -> sigmoid -> stack ->
 * CropSplit(ops/crop/src/crop_split_cuda_kernel.cu:19-59) -> permute, as ONE kernel
 * that evaluates only the selected sub-region's dot product for in-box pixels.
 *   protos : [32,H,W] (layout_hwc=0, the reference's `feat_mask`) or [H,W,32] (layout_hwc=1)
 *   cofs   : [N,128] fp32, per detection (00|01|10|11 blocks of 32, sipmask_head.py:616-619)
 *   boxes  : [N,4] fp32 image-space boxes; rois = boxes * box_scale (sipmask_head.py:623,
 *            box_scale = scale_factor / 2), per-coordinate box_scale[4]
 *   out    : [N,H,W] (fp32 or fp16) = the reference's pos_masks.permute(2,0,1)
 */
int smb_mask_assemble(const void* protos, int protos_dtype, int layout_hwc,
                      const float* cofs, const float* boxes, const float* host_box_scale4,
                      void* out, int out_dtype, int H, int W, int N, smb_stream_t stream);

/* Bilinear resize (align_corners=False) + `> thr` of pos_masks (sipmask_head.py:630-633), pasted top-left into
 * [N,out_h,out_w] and truncated (sipmask_head.py:648-654).  The reference interpolates by 2/scale_factor (per axis
 * scale_factor[3:1:-1] on the SSD path): the caller passes the interpolated size (full_h, full_w) =
 * (floor(H * 2/sf_h), floor(W * 2/sf_w)) and the source step per output pixel (ry, rx): src = (dst + 0.5) * r - 0.5 with
 * r = 1 / (2/sf) (what F.interpolate(scale_factor=...) does in PyTorch >= 1.6), or r <= 0 for in/out
 * (recompute_scale_factor=True, the behaviour of PyTorch <= 1.5, the version range the reference README pins).
 *   pos : [N,H,W] fp32/fp16      out_u8 : [N,out_h,out_w] uint8 {0,1}; pixels beyond (full_h, full_w) are 0. */
int smb_mask_resize_threshold(const void* pos, int pos_dtype, uint8_t* out_u8, int N, int H, int W, int full_h,
                              int full_w, float ry, float rx, int out_h, int out_w, float thr, smb_stream_t stream);
/* Bit-packed variant: out_bits [N,out_h,ceil(out_w/32)] uint32, pixel x = bit (x & 31) of word (x >> 5). */
int smb_mask_resize_threshold_pack(const void* pos, int pos_dtype, uint32_t* out_bits, int N, int H, int W,
                                   int full_h, int full_w, float ry, float rx, int out_h, int out_w, float thr,
                                   smb_stream_t stream);
/* scale_factor == 1 shorthands: full size = (2H, 2W). */
int smb_mask_upsample2_threshold(const void* pos, int pos_dtype, uint8_t* out_u8, int N, int H, int W,
                                 int out_h, int out_w, float thr, smb_stream_t stream);
int smb_mask_upsample2_threshold_pack(const void* pos, int pos_dtype, uint32_t* out_bits, int N, int H, int W,
                                      int out_h, int out_w, float thr, smb_stream_t stream);

/* SipMask++ mask rescoring (sipmask_head.py:200-219,635-643; SURVEY.md 8a-10).
 * smb_conv3x3s2_relu_f32: one ConvModule of `convs_scoring`: NCHW fp32 conv3x3, stride 2, padding 0, + bias, ReLU;
 *   in [N,Cin,H,W] -> out [N,Cout,(H-3)/2+1,(W-3)/2+1], weight [Cout,Cin,3,3].
 * smb_mask_rescore: relu(mask_scoring 1x1) -> global max-pool -> the detection's own class -> times det[:,4]:
 *   feat [N,C,h,w], weight1x1 [num_classes,C], labels int64 [N], det [N,5], n_valid device int (or NULL) -> scores [N]. */
int smb_conv3x3s2_relu_f32(const float* in, const float* weight, const float* bias, float* out, int N, int Cin, int H,
                           int W, int Cout, smb_stream_t stream);
int smb_mask_rescore(const float* feat, int N, int C, int h, int w, const float* weight1x1, const float* bias1x1,
                     int num_classes, const int64_t* labels, const float* det, const int* n_valid, float* scores,
                     smb_stream_t stream);

/* COCO RLE of bit-packed masks on the device (replaces the per-detection `masks[i].cpu().numpy()` + pycocotools
 * `mask_util.encode(order='F')` tail, sipmask_head.py:645-657; SURVEY.md 8f-1).
 *   mask_bits : [N, mask_h, words] uint32 (pixel x = bit x&31 of word x>>5), cropped to the top-left H x W (= ori_shape)
 *   n_valid   : device int (number of valid detections, may be NULL = N)
 *   counts    : [N, cap] uint32 run lengths in COLUMN-major order, starting with the zeros run
 *   n_counts  : [N] int32: number of runs, 0 for det >= *n_valid, or -(boundaries+1) if cap was too small */
int smb_mask_rle_counts(const uint32_t* mask_bits, int N, int mask_h, int words, int H, int W, const int* n_valid,
                        uint32_t* counts, int cap, int* n_counts, smb_stream_t stream);
/* HOST helper (plain C, no CUDA): pycocotools' rleToString of `n` run lengths; returns the length written, -1 if cap is
 * too small.  counts is a host pointer. */
int smb_rle_to_string(const uint32_t* host_counts, int n, char* host_out, int cap);

/* Fully fused mask path (sipmask_head.py:609-633,648-654): prototypes -> selected sub-region dot product -> sigmoid ->
 * crop -> bilinear resize to (full_h, full_w) -> `> thr` -> bit-pack into [N,out_h,ceil(out_w/32)] (a memset node zero-fills
 * the planes, one kernel writes the words that intersect a box).  pos_masks is never written to memory.
 * Same arguments as smb_mask_assemble; resize / output as smb_mask_resize_threshold_pack.  Shrinking by more than 4x
 * (scale_factor > 8) returns SMB_EINVAL. */
int smb_mask_assemble_pack(const void* protos, int protos_dtype, int layout_hwc, const float* cofs, const float* boxes,
                           const float* host_box_scale4, uint32_t* out_bits, int H, int W, int N, int full_h, int full_w,
                           float ry, float rx, int out_h, int out_w, float thr, smb_stream_t stream);

/* fp16 prototypes run the tensor-core variants of smb_mask_assemble / smb_mask_assemble_pack (mma.sync dot products with
 * the fp32 coefficients split into fp16 hi + lo; same crop geometry, mask values within ~1e-6 of the scalar kernels).
 * on = 1 / 0 selects them / the scalar-fmaf kernels for later calls, on < 0 only queries; returns the previous setting
 * (initial value: environment SMB_MASK_MMA, else the build default). */
int smb_mask_set_tensor_dot(int on);

/* ------------------------------------------------------------------ CropSplit (operator API)
 * Replaces crop_split_cuda.crop_split_cuda_forward(data, rois, out, H, W, c, n)
 * (ops/crop/src/crop_split_cuda.cpp:14-36).  data [c*c,H,W,N], rois [N,4], out [H,W,N]; c == 2.
 */
int smb_crop_split_forward(const void* data, const void* rois, void* out, int dtype,
                           int H, int W, int c, int N, smb_stream_t stream);

/* Training-side companions (SURVEY 8f-4).  smb_crop_split_backward replaces crop_split_cuda_backward
 * (ops/crop/src/crop_split_cuda_kernel.cu:90-163): top_grad [H,W,N] -> bottom_grad [c*c,H,W,N], every element written
 * (the reference zero-initialises and atomically adds).  smb_crop_split_gt replaces crop_split_gt_cuda_forward AND
 * _backward (ops/crop/src/crop_split_gt_cuda_kernel.cu:19-49,76-104): out[h,w,n] = data[h,w,n] inside roi n, else 0. */
int smb_crop_split_backward(const void* top_grad, const void* rois, void* bottom_grad, int dtype, int H, int W, int c, int N,
                            smb_stream_t stream);
int smb_crop_split_gt(const void* data, const void* rois, void* out, int dtype, int H, int W, int N, smb_stream_t stream);

/* ------------------------------------------------------------------ NMS (operator API)
 * Replaces nms_cuda.nms(dets, thr) (ops/nms/src/nms_kernel.cu:71-138) without the D2H bitmask copy
 * and host sweep.  dets [n,5] fp32; keep_out [n] int64 receives ORIGINAL indices ascending;
 * n_keep_out device int32.  cmp_ge: 0 = suppress IoU > thr (CUDA ref), 1 = IoU >= thr (CPU ref).
 * n <= 8192.
 */
int smb_nms(const float* dets, int n, float iou_thr, int cmp_ge, int plus_one,
            int64_t* keep_out, int* n_keep_out, smb_stream_t stream);

/* ------------------------------------------------------------------ decode + per-level top-k
 * Replaces sipmask_head.py:556-592 (sigmoid, max_c(score*ctr) top-k per level, distance2bbox
 * core/bbox/transforms.py:202-223, concat, /scale_factor, no bg column).
 * Level l has hw[l] locations on a w[l]-wide grid with stride[l]; its tensors are channel-last:
 *   cls[l] : [hw,C] fp32 logits with row pitch cls_pitch (elements);  ctr[l] : [hw] pitch ctr_pitch
 *   box[l] : [hw,4] fp32 distances (already x stride) with row pitch box_pitch
 * Outputs (n_total = sum_l min(hw[l], nms_pre) when nms_pre > 0):
 *   cand_boxes [n_total,4], cand_scores [n_total,C] (sigmoid), cand_ctr [n_total] (sigmoid),
 *   cand_loc [n_total] int32 = level-concatenated location index (for gathering coefficients).
 */
typedef struct {
  const float* cls; const float* ctr; const float* box;
  int cls_pitch, ctr_pitch, box_pitch;
  int h, w, stride;
  float box_scale, box_mul; /* distance = (box * box_scale) * box_mul : (1,1) for the reference's bbox_preds,
                               (Scale_l, stride_l) when `box` is the raw fcos_reg output (sipmask_head.py:261,268) */
} smb_level_t;

size_t smb_decode_workspace_bytes(int num_levels, const smb_level_t* host_levels, int nms_pre);
int smb_decode_topk(int num_levels, const smb_level_t* host_levels, int num_classes, int nms_pre,
                    int img_h, int img_w, const float* host_scale4 /* scale_factor per coordinate (boxes are divided by it), or NULL */,
                    float* cand_boxes, float* cand_scores, float* cand_ctr, int* cand_loc,
                    void* workspace, size_t workspace_bytes, smb_stream_t stream);

/* ------------------------------------------------------------------ multi-class NMS
 * Replaces core/post_processing/bbox_nms.py:79-146 (python loop over classes, one nms_cuda +
 * D2H + host sweep per class) with two launches and no host sync.
 *   boxes [n,4], scores [n,C] (raw sigmoid, no bg column), ctr [n] (score factor)
 *   det_out [max_num,5] (x1,y1,x2,y2,score*ctr), label_out [max_num] int64 (0-based),
 *   idx_out [max_num] int64 (row of boxes), count_out device int32.
 * Order: class-major / ascending row when total <= max_num, else descending score
 * (ties: class-major order) - bbox_nms.py:135-140.   n <= 4096, max_num <= 1024.
 */
size_t smb_multiclass_nms_workspace_bytes(int n, int num_classes);
int smb_multiclass_nms(const float* boxes, const float* scores, const float* ctr, int n, int num_classes,
                       float score_thr, float iou_thr, int max_num, int cmp_ge,
                       float* det_out, int64_t* label_out, int64_t* idx_out, int* count_out,
                       void* workspace, size_t workspace_bytes, smb_stream_t stream);

/* ------------------------------------------------------------------ fast NMS (SSD / VIS path)
 * Replaces SipMaskHead.fast_nms (sipmask_head.py:868-910): per-class descending sort, top_k,
 * IoU without +1 (:912-959), triu, column max, `iou_max <= thr && score > score_thr`, global
 * descending sort, first max_num.   scores [n,C] sigmoid, ctr [n]; n <= 4096, top_k <= 256.
 */
size_t smb_fast_nms_workspace_bytes(int n, int num_classes, int top_k);
int smb_fast_nms(const float* boxes, const float* scores, const float* ctr, int n, int num_classes,
                 float score_thr, float iou_thr, int top_k, int max_num,
                 float* det_out, int64_t* label_out, int64_t* idx_out, int* count_out,
                 void* workspace, size_t workspace_bytes, smb_stream_t stream);

/* The gather between NMS and mask assembly (mlvl_cofs[idxs_keep], det_bboxes[:, :4]; sipmask_head.py:612,623) in one launch:
 * det_cofs[i,:] = cof_src[cand_loc[idx[i]],:] (row pitch cof_pitch floats), det_boxes[i,:] = det[i,:4] for i < *count,
 * zeros after; loc_out (may be NULL) receives the level-concatenated location of each kept detection (-1 after count).
 * cof_src is either one image's level-concatenated [tot, pitch] buffer (num_levels = 0) or a batched level-major buffer
 * [level][n_img][hw_l][pitch] with host_level_hw[l] = h_l * w_l, of which image `img` is gathered. */
int smb_gather_det_inputs(const float* cof_src, int cof_pitch, const int* cand_loc, const int64_t* idx, const float* det,
                          const int* count_dev, int max_rows, int row_elems, float* det_cofs, float* det_boxes,
                          int64_t* loc_out, int num_levels, const int* host_level_hw, int n_img, int img, smb_stream_t stream);

/* SipMask-VIS `extract_box_feature_center_single` (SipMask-VIS/mmdet/models/anchor_heads/sipmask_head.py:609-613,768-781):
 * out[i,:] = track[floor((y1+y2)*sy/2/stride), floor((x1+x2)*sx/2/stride), :] for i < *count, zeros after.
 * track [h,w,C] fp32 channel-last (the `sipmask_track` output), det [max_rows,5], (sx, sy) = scale_factor when the
 * detections were rescaled (res_det_bboxes = det * scale_factor), feat_stride = 8. */
int smb_gather_track_feats(const float* track, int h, int w, int C, const float* det, const int* count_dev, int max_rows,
                           float scale_x, float scale_y, float feat_stride, float* out, smb_stream_t stream);

/* HOST helper (plain C++, no CUDA): one frame of the SipMask-VIS tracker association (SipMask-VIS/mmdet/models/anchor_heads/
 * sipmask_head.py:544-562,612-667) on host arrays.  State = the tracked objects' boxes [capacity,5], labels [capacity],
 * features [capacity,feat_dim], of which the first n_prev are valid; updated in place.  host_ids_out [n] receives the object
 * ids (-1: lost the claim).  Returns the new number of tracked objects, or a negative SMB_E* code. */
int smb_track_step(const float* host_det, const int64_t* host_labels, const float* host_feats, int n, int feat_dim,
                   float* host_prev_det, int64_t* host_prev_labels, float* host_prev_feats, int n_prev, int capacity,
                   const float* host_match_coeff3, int32_t* host_ids_out);

/* gather rows: dst[i,:] = src[idx[i],:] for i < *count (device count), zero otherwise. */
int smb_gather_rows_f32(const float* src, int src_pitch, const int64_t* idx, const int* count_dev,
                        int max_rows, int row_elems, float* dst, smb_stream_t stream);

/* ------------------------------------------------------------------ convolution engine (tcgen05)
 * Replaces every nn.Conv2d (+ folded eval BatchNorm, bias, residual add, ReLU) on the path
 * (models/backbones/resnet.py:203-239, models/necks/fpn.py:138-178, ops/conv_module.py:124-132,
 * anchor_heads/sipmask_head.py:241-287) with one implicit-GEMM kernel:
 *   D[pixels, Cout] = sum_{taps, Cin} A[pixel + tap, Cin] * Wt[Cout, tap, Cin]
 * A is the NHWC fp16 activation read through TMA tensor maps (one 2D-patch box per tap; zero
 * fill outside the image gives the padding), W is [Cout, taps*Cin] fp16 K-major, the fp32
 * accumulator lives in TMEM (tcgen05.mma cta_group::1, M=128), the epilogue applies
 * scale/bias (folded BN), residual, ReLU, optional GroupNorm statistics, and writes NHWC.
 */
typedef struct smb_conv_plan smb_conv_plan_t;

typedef struct {
  int N, H, W, Cin;          /* input  NHWC (Cin % 64 == 0, or Cin == 8-padded stem handled internally) */
  int Cout;                  /* multiple of 16, <= 256 per N-tile (larger Cout is tiled) */
  int kh, kw, stride, pad;   /* 1x1/3x3 stride 1|2, pad = k/2 ; 7x7/2 stem uses the dedicated plan */
  int relu;                  /* apply ReLU in the epilogue */
  int has_bias;              /* per-channel fp32 bias (folded BN shift / conv bias) */
  int has_residual;          /* add an NHWC fp16 tensor of the output shape before ReLU */
  int residual_upsample;     /* residual is the coarser FPN level: nearest-neighbour gather (fpn.py:149-152) */
  int res_h, res_w;          /* residual spatial size when residual_upsample */
  int out_dtype;             /* SMB_F16 or SMB_F32 */
  int gn_stats;              /* accumulate per-(image,group) {sum*2^20, sumsq*2^16} as int64 fixed point into stats[N*32*2]
                                (integer atomics: bit-reproducible run to run) */
  int in_pitch, out_pitch;   /* channel pitch (elements) of input / output rows; 0 = dense */
} smb_conv_desc_t;

int smb_conv_plan_create(const smb_conv_desc_t* desc, const void* in, const void* weight, void* out,
                         smb_conv_plan_t** plan_out);

/* One launch over several feature-pyramid levels that share the weights (the FCOS towers / heads are applied to
 * P3..P7 in a python loop in the reference, sipmask_head.py:250-271).  desc->H/W are ignored; stride must be 1.
 * Per-level residual / gn_stats pointers are baked into the plan (pass NULLs to smb_conv_run). */
typedef struct {
  const void* in; void* out;
  const void* residual; void* gn_stats;
  int H, W, res_h, res_w;
} smb_conv_level_t;
int smb_conv_plan_create_multi(const smb_conv_desc_t* desc, int num_levels, const smb_conv_level_t* levels,
                               const void* weight, smb_conv_plan_t** plan_out);
void smb_conv_plan_destroy(smb_conv_plan_t* plan);
/* Cap the persistent grid of a plan (multiple of its cluster size), so that independent convolutions launched on
 * different streams share the GPU instead of running one after the other with half-empty last waves. */
int smb_conv_plan_set_max_ctas(smb_conv_plan_t* plan, int max_ctas);
/* Planner knob for plans created AFTER the call: the N tile is the largest of {256,128,64} that still yields at least
 * `min_tiles` output tiles (default 48; <= 0 restores the default).  Small values favour fat tiles (fewer bytes through
 * L2 -> SM per FLOP), large values favour occupancy of a single stream.  Returns the previous value. */
int smb_conv_set_min_tiles(int min_tiles);
/* Read-only view of what the planner chose for a plan (tests pin the branch a shape is meant to reach).  Writes the
 * first min(n, 11) of, in this order:
 *   n_tile, n_tiles_n, tiles_m, pair (cta_group::2), cluster (CTAs per cluster), grid (CTAs launched, after
 *   smb_conv_plan_set_max_ctas), out_tma (TMA-store epilogue), res_tma (TMA-staged residual), stage_slots,
 *   epi_split (split epilogue chosen at plan time; smb_conv_run falls back to the lockstep epilogue when alpha != 1,
 *   there is no bias or the bias is not 16-byte aligned), small (conv1x1_small_kernel).
 * Returns the number of fields the library knows (11), or a negative SMB_E* code. */
int smb_conv_plan_info(const smb_conv_plan_t* plan, int* out, int n);
/* out = relu?( (acc + bias) * alpha + residual ); alpha carries the per-level `Scale` of fcos_reg
 * (sipmask_head.py:261, ops/scale.py:12-15). */
int smb_conv_run(const smb_conv_plan_t* plan, const float* bias, const void* residual, void* gn_stats,
                 float alpha, smb_stream_t stream);

/* ------------------------------------------------------------------ elementwise / gather kernels (NHWC fp16) */
/* GroupNorm(32 groups, eps) + ReLU applied in place from precomputed per-(image,group) sum/sumsq
 * (ops/norm.py:43-49 + conv_module.py:124-132).  x [N*HW, C] fp16. */
int smb_groupnorm_relu_apply(void* x, int n_img, int hw, int C, int pitch, const void* stats /* int64 [n_img*32*2] */,
                             const float* gamma, const float* beta, float eps, int relu, smb_stream_t stream);
/* stats for a tensor that did not come out of smb_conv_run (e.g. DCN output computed elsewhere). */
int smb_groupnorm_stats(const void* x, int n_img, int hw, int C, int pitch, void* stats /* int64 */, smb_stream_t stream);

/* Deformable im2col (ops/dcn/src/deform_conv_cuda_kernel.cu:85-115,191-243), channel-last:
 *   x [H,W,C] fp16, offset [H,W,dg*18] fp32 (per dg: 2*(i*3+j)=dh, +1=dw) with pitch off_pitch
 *   -> col [H*W, 9*C] fp16, K index = tap*C + c (3x3, stride 1, pad 1, dil 1). */
int smb_deform_im2col(const void* x, const float* offset, int off_pitch, void* col,
                      int n_img, int H, int W, int C, int deformable_groups, smb_stream_t stream);

/* FeatureAlign.conv_offset (sipmask_head.py:30-33,50): off[pix,o] = sum_k W[o,k] * (bbox[pix,k] * scale), fp32. */
int smb_offset_conv1x1(const float* bbox, int bbox_pitch, float scale, const float* weight, int n_off, float* off,
                       long long npix, smb_stream_t stream);

/* Multi-level (batched over feature-pyramid levels, shared parameters) variants of the three kernels above:
 * one launch instead of one per level.  Pointer arrays are HOST arrays of device pointers. */
int smb_groupnorm_relu_apply_multi(int num_levels, void* const* xs, const void* const* stats, const int* Hs, const int* Ws,
                                   int n_img, int C, int pitch, const float* gamma, const float* beta, float eps, int relu,
                                   smb_stream_t stream);
int smb_offset_conv1x1_multi(int num_levels, const float* const* bboxes, int bbox_pitch, const float* scales,
                             const float* weight, int n_off, float* const* offs, const int* Hs, const int* Ws, int n_img,
                             smb_stream_t stream);
int smb_deform_im2col_multi(int num_levels, const void* const* xs, const float* const* offs, int off_pitch,
                            void* const* cols, const int* Hs, const int* Ws, int n_img, int C, int deformable_groups,
                            smb_stream_t stream);

/* MaxPool2d(3, 2, 1) (backbones/resnet.py:460), NHWC fp16. */
int smb_maxpool3x3s2(const void* x, void* y, int N, int H, int W, int C, smb_stream_t stream);

/* Bilinear upsample by an integer factor, align_corners=False (sipmask_head.py:279,285), NHWC fp16,
 * writing into a channel slice of a wider tensor (out_pitch, out_choff) so torch.cat is free.
 * y is [N, out_h, out_w, out_pitch]: the top-left out_h x out_w (<= H*factor x W*factor) of the upsampled map, so a
 * level whose upsampled size exceeds the P3 map it is concatenated to is cropped instead of written past y;
 * factor 1 (a channel copy) needs out_h == H, out_w == W. */
int smb_upsample_bilinear(const void* x, int in_pitch, void* y, int out_pitch, int out_choff,
                          int N, int H, int W, int C, int factor, int out_h, int out_w, int relu, smb_stream_t stream);

/* Image preparation: NCHW fp32 -> zero-padded NHWC8 fp16 [N, H+6, W+8, 8] for the 7x7/2 stem. */
int smb_image_to_nhwc8(const float* img, void* out, int N, int H, int W, smb_stream_t stream);

/* Test-time image pipeline on the device (SURVEY.md 8f-3; transforms.py:97-110 Resize(keep_ratio), :335-363 Normalize
 * (std = 1, to_rgb = False), :274-300 Pad(32); mmcv.imrescale -> cv2.resize(INTER_LINEAR) restated bit-exactly):
 *   src       : uint8 BGR HWC [src_h, src_w, 3] device image, row pitch in bytes
 *   dst_h/w   : resized size (mmcv rule: int(h * s + 0.5), s = min(max_long / max(h, w), max_short / min(h, w)))
 *   out_nhwc8 : the stem's input [H+6, W+8, 8] fp16 (pixel (y,x) at (y+3, x+3)), H x W = padded size >= dst; everything
 *               outside the resized image is zero (= zero padding AFTER mean subtraction, as in the reference) */
int smb_preprocess_u8(const uint8_t* src, int src_h, int src_w, int src_pitch_bytes, int dst_h, int dst_w,
                      const float* host_mean3, void* out_nhwc8, int H, int W, smb_stream_t stream);

/* Stem 7x7/2 conv (3->64) + folded BN + ReLU on the padded NHWC8 image (backbones/resnet.py:448-460). */
int smb_stem_plan_create(int N, int H, int W, const void* img_nhwc8, const void* weight448, void* out,
                         smb_conv_plan_t** plan_out);
/* Space-to-depth form of the same stem (K = 256 instead of 448): the image is stored as [N, H/2+3, W/2+4, 16] fp16 with
 * element (Y, X, (dy*2+dx)*4 + c) = padded pixel (2Y+dy, 2X+dx) channel c (smb_image_to_s2d16 / smb_preprocess_u8_s2d), the
 * weights as [64, 4*64] with K = a*64 + b*16 + (dy*2+dx)*4 + c for filter tap (r, s) = (2a+dy, 2b+dx). */
int smb_stem_plan_create_s2d(int N, int H, int W, const void* img_s2d16, const void* weight256, void* out,
                             smb_conv_plan_t** plan_out);
int smb_image_to_s2d16(const float* img_nchw_f32, void* out_s2d16, int N, int H, int W, smb_stream_t stream);
int smb_preprocess_u8_s2d(const uint8_t* src, int src_h, int src_w, int src_pitch_bytes, int dst_h, int dst_w,
                          const float* host_mean3, void* out_s2d16, int H, int W, smb_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SIPMASK_B200_H_ */
