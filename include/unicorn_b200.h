/* unicorn_b200 — C ABI of the B200-native Unicorn per-frame inference hot path.
 *
 * Every entry point takes plain device pointers, sizes and a CUDA stream (passed as void* so the header
 * needs no CUDA include).  No entry point allocates, synchronises or keeps state between calls (apart from
 * a lazily resolved driver entry point), so all of them are CUDA-graph capturable.  All return 0 on success
 * and a negative UC_E* / positive cudaError_t code otherwise; uc_last_error() gives the text.
 * There is NO CPU fallback: on a machine without an sm_100 device every launch returns an error.
 *
 * Reference interfaces replaced (paths relative to MasterBin-IIAU/Unicorn):
 *   uc_msda_forward_*      unicorn/models/ops/src/ms_deform_attn.h:20-39  (ms_deform_attn_forward)
 *                          -> unicorn/models/ops/src/cuda/ms_deform_attn_cuda.cu:20-80
 *                          -> ms_deformable_im2col_gpu_kernel, ms_deform_im2col_cuda.cuh:237-299
 *   uc_conv2d              nn.Conv2d / nn.Linear call sites of the backbone, neck, heads:
 *                          backbone/convnext.py:41-54,82-87; network_blocks.py:50-51; unicorn.py:36-44;
 *                          unicorn_head.py:267-336; ops/modules/ms_deform_attn.py:94-113
 *   uc_stem_ln             backbone/convnext.py:77-80 (conv4x4s4 + channels_first LayerNorm)
 *   uc_dwconv7_ln          backbone/convnext.py:43-45 (dwconv 7x7 + LayerNorm)
 *   uc_layernorm           backbone/convnext.py:176-184; deformable_transformer.py:113,121
 *   uc_groupnorm_*         GroupNorm(16,eps 1e-3) from exp/unicorn_track.py:450-470; unicorn.py:38
 *   uc_corr_propagate      external/lib/test/tracker/unicorn_sot.py:95-100, unicorn_vos.py:171-181
 *   uc_head_decode         unicorn_head.py:332-334,467-482
 *   uc_nms_*               utils/boxes.py:33-77 (torchvision.ops.batched_nms)
 */
#ifndef UNICORN_B200_H_
#define UNICORN_B200_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define UC_API __attribute__((visibility("default")))
#else
#define UC_API
#endif

#define UC_OK 0
#define UC_EINVAL (-1)   /* bad argument (shape / alignment / dtype) */
#define UC_EDRIVER (-2)  /* driver entry point (cuTensorMapEncodeTiled) unavailable */
#define UC_ENODEV (-3)   /* no sm_100 device */

/* dtypes of activation tensors */
#define UC_BF16 0
#define UC_F32 1
#define UC_F16 2

/* fused activations */
#define UC_ACT_NONE 0
#define UC_ACT_RELU 1
#define UC_ACT_GELU 2 /* exact erf GELU (nn.GELU()), evaluated as x*sigmoid(x*P(x^2)), |error| < 4e-6 */
#define UC_ACT_SILU 3
#define UC_ACT_SIGMOID 4

UC_API const char* uc_last_error(void);
UC_API int uc_version(void);
/* 0 if the current device is sm_100 and the driver entry points resolve, else a UC_E* code */
UC_API int uc_check_device(void);

/* Dense convolution / linear layer as an implicit GEMM on tcgen05 tensor cores (TMA-fed, TMEM accumulators).
 *   x : NHWC activations, 16-bit (bf16 or f16 per x_dtype), pixel stride ldx elements (ldx >= Cin, ldx % 8 == 0)
 *   w : packed weights [Cout][KH*KW][Cin] in the same 16-bit type as x (K-major)
 *   y : NHWC output, pixel stride ldy, dtype y_dtype; y = act(conv(x) + bias) ; then y = res + gamma * y if given
 * A Linear layer on [M, Cin] rows is B=1, H=1, W=M, KH=KW=1.  stride in {1,2}; pad < KH.
 * Cin % 8 == 0, Cout % 8 == 0 (pad the weight rows / output channels otherwise).  Outputs (and residuals) whose rows start on
 * 32-byte boundaries (ldy * sizeof % 32 == 0, y % 32 == 0) are written with one 256-bit store per 16 channels; other
 * layouts fall back to 128-bit stores.  Every launch is CUDA-graph capturable and uses programmatic dependent launch.
 */
typedef struct UcConv2d {
  const void* x;
  int x_dtype;
  int B, H, W, Cin, ldx;
  const void* w;
  int Cout, KH, KW, stride, pad;
  const float* bias;  /* [Cout] or NULL */
  int act;            /* UC_ACT_* */
  const float* gamma; /* [Cout] layer scale or NULL */
  const void* res;    /* residual, 16-bit like x, rows of ldres elements, or NULL */
  int ldres;
  void* y;
  int ldy;
  int y_dtype;
  int block_n; /* 0 = auto; else force the N tile (16,32,64,96,128,192,256); +1000 (1128,1192,1256) = the
                  cta_group::2 variant: an SM pair computes a 256 x N tile with one pair-MMA stream */
  /* Optional GroupNorm statistics of the (pre-activation) output, accumulated per (image, group):
   * gn_stats[b][g] = {sum, sumsq} as int64 fixed point (value * 2^22; integer atomics => order independent,
   * bit-reproducible); must be zeroed by the caller; NULL = off.  Consumed by uc_groupnorm_apply. */
  void* gn_stats;
  int gn_groups;
  /* Optional LayerNorm folded into a 1x1 conv (ConvNeXt block, convnext.py:45-46): x is the UN-normalised map, w = W * diag(ln_w),
   * bias = W @ ln_b + b, col_s[n] = sum_k w[n][k] (of the 16-bit weights), row_stats = per-pixel {sum, sumsq} over Cin of x as
   * written by uc_dwconv7 (int64 fixed point 2^22): y = act(rstd * (w x) - rstd * mu * col_s + bias).  NULL = off. */
  const void* row_stats;
  const float* col_s;
  float row_eps;
} UcConv2d;
UC_API int uc_conv2d(const UcConv2d* d, void* stream);

/* ConvNeXt stem: Conv2d(3,C0,k4,s4)+bias then channels_first LayerNorm (backbone/convnext.py:77-80,179-184).
 * img: fp32 NCHW [B,3,H,W] (PreprocessorX output, unicorn_sot.py:114-123) or, with img_is_u8_hwc = 1, the uint8 HWC
 * BGR frame [B,H,W,3] as cv2 delivers it (the permute / float conversion is fused into the load);
 * w48 fp32 [48][C0] with k=(ci*4+kh)*4+kw; out NHWC bf16 [B,H/4,W/4,C0]. */
UC_API int uc_stem_ln(const void* img, int img_is_u8_hwc, const float* w48, const float* bias, const float* lnw, const float* lnb,
                      void* out_bf16, int B, int H, int W, int C0, float eps, void* stream);

/* ConvNeXt block front half in ONE launch: depthwise 7x7 (pad 3)+bias then LayerNorm over C (convnext.py:43-45); the
 * intermediate map stays in shared memory (C % 64 == 0; other C use a one-warp-row kernel).  Not in place.  The engine uses
 * uc_dwconv7 + uc_layernorm instead, which is faster on ConvNeXt-L's shapes (DESIGN.md 4.3).
 * x,y NHWC bf16 contiguous [B,H,W,C]; w49 fp32 [49][C] (k = kh*7+kw). */
UC_API int uc_dwconv7_ln(const void* x_bf16, const float* w49, const float* bias, const float* lnw, const float* lnb,
                         void* y_bf16, int B, int H, int W, int C, float eps, void* stream);

/* Depthwise 7x7 (pad 3) + bias of the ConvNeXt block (convnext.py:43), TMA staged (csrc/dwconv_tma.cu); follow with uc_layernorm,
 * or give ln_stats and fold the LayerNorm into pwconv1 (UcConv2d.row_stats).  x, y NHWC bf16 contiguous, not in place; w49 fp32 [49][C].
 * ln_stats (optional, may be NULL): [B*H*W][2] int64 fixed point (value * 2^22), zeroed by the caller; receives the per-pixel
 * {sum, sum of squares} over C of the stored outputs.  work_counter (optional, may be NULL): one device int, ZERO before the launch,
 * used to hand out the tiles dynamically (balanced SM loads on small maps); NULL = static round-robin. */
UC_API int uc_dwconv7(const void* x_bf16, const float* w49, const float* bias, void* y_bf16, int B, int H, int W, int C,
                      void* ln_stats, int* work_counter, void* stream);

/* The same depthwise 7x7 + bias on tensor cores (csrc/dwconv_mma.cu): every filter row is a banded 16 x 8 Toeplitz block applied with
 * mma.sync.m16n8k16 to a channel-planar copy of the input tile.  qtab = per 32-channel chunk {int32 [32][7][8]: the filter as bf16
 * tap pairs {f[kh][j-1], f[kh][j]}, j = 0..7, zero outside the row; fp32 [32]: the biases}, zero for the channels that pad C to a
 * multiple of 32 (unicorn_b200.ops.pack_dw_weight_mma); C % 8 == 0.  Same x / y / work_counter conventions as uc_dwconv7; no ln_stats. */
UC_API int uc_dwconv7_mma(const void* x_bf16, const void* qtab, void* y_bf16, int B, int H, int W, int C, int* work_counter, void* stream);

/* Fused back half of a ConvNeXt block (unicorn/models/backbone/convnext.py:45-52: norm -> pwconv1 -> GELU -> pwconv2 -> gamma ->
 * residual) in one launch, for C = 96 / 192 / 256 / 384 (uc_convnext_mlp_supported): x[M][C] += gamma * (W2 . GELU(W1f . LN0(t) + c1) + b2), LN0 =
 * LayerNorm without affine (eps = ln_eps) over the C channels of a row of t[M][C] (the depthwise-conv output), W1f[4C][C] = pwconv1
 * weight with the LayerNorm weight folded in (W1 diag(g)), c1[4C] = b1 + W1 beta, W2[C][4C].  bf16 maps and weights, fp32 vectors;
 * t / weights 16-byte, x / vectors 32-byte aligned.  The 4C hidden activations stay in shared / tensor memory (csrc/mlp_fused.cu). */
UC_API int uc_convnext_mlp_supported(int C);
UC_API int uc_convnext_mlp(const void* t_bf16, const void* w1f_bf16, const float* c1, const void* w2_bf16, const float* b2, const float* gamma,
                           void* x_bf16, int M, int C, float ln_eps, void* stream);

/* Row LayerNorm: y[m,:] = LN(x[m,:] + res[m,:]) * w + b  (res may be NULL).  16-bit rows with element strides.
 * convnext.py:176-184 (downsample / out norms), deformable_transformer.py:113,121,127-130 (post-norm). */
UC_API int uc_layernorm(const void* x, int ldx, const void* res, int ldres, const float* w, const float* b, void* y,
                        int ldy, long M, int C, float eps, int dtype, void* stream);

/* GroupNorm apply with the statistics accumulated by uc_conv2d (gn_stats = [B][G]{sum,sumsq}):
 * y = act((x-mean)*rstd*w+b) [+ prior[pix]*beta[c]] ; optional second output y2 = y + add2.
 * network_blocks.py:50-51 with exp/unicorn_track.py:450-470 (GN16, eps 1e-3, SiLU); unicorn.py:38 (GN32, eps 1e-5);
 * unicorn_head.py:272-275 (prior fusion).  x,y,add2,y2 bf16 NHWC with pixel strides. */
UC_API int uc_groupnorm_apply(const void* x, int ldx, const void* stats, const float* w, const float* b, void* y,
                              int ldy, int B, long HW, int C, int G, float eps, int act, const float* prior,
                              const float* beta, const void* add2, int ldadd2, void* y2, int ldy2, void* stream);

/* dst[b,oh,ow,:C] = src[b,oh/up,ow/up,:C], up in {1,2} (nearest upsample + concat slice; yolo_pafpn_new.py:139-146). */
UC_API int uc_copy_upsample(const void* src, int lds, void* dst, int ldd, int B, int Hs, int Ws, int C, int up, void* stream);
/* nn.PixelShuffle(2) in NHWC (unicorn.py:41): in [B,H,W,4*Co] -> out [B,2H,2W,Co], 16-bit. */
UC_API int uc_pixel_shuffle2(const void* in, int ldi, void* out, int ldo, int B, int H, int W, int Co, void* stream);
/* F.interpolate(bilinear, align_corners=False) on fp32 planes [P,Hs,Ws]->[P,Hd,Wd]; scale_* = 1/scale_factor or 0. */
UC_API int uc_bilinear_f32(const float* src, float* dst, int P, int Hs, int Ws, int Hd, int Wd, float scale_h,
                           float scale_w, void* stream);
/* Letterbox preprocessing on the device (PreprocessorX.process, external/lib/test/tracker/unicorn_sot.py:114-123; preproc,
 * unicorn/data/data_augment.py:194-214): dst[0:rh,0:rw] = cv2.resize(src,(rw,rh),INTER_LINEAR) — bit-exact restatement of
 * OpenCV's 8-bit fixed-point bilinear —, the rest = pad (114); swap_rb does cv2.COLOR_RGB2BGR.  uint8 HWC, 3 channels. */
UC_API int uc_letterbox_u8(const uint8_t* src_hwc, int Hs, int Ws, uint8_t* dst_hwc, int Hd, int Wd, int rh, int rw,
                           int swap_rb, int pad, void* stream);
UC_API int uc_add(const void* a, int lda, const void* b, int ldb, void* y, int ldy, long M, int C, int dtype, void* stream);
/* Conditional strided row copy decided on the device: rows are copied when (*flag_dev != 0) != invert.  The MOT drivers use it for
 * "pre_dict = cur_dict only when this frame produced detections" (unicorn/evaluators/mot_evaluator.py:1005,1014-1020) so that the
 * frame needs no host decision (CUDA-graph replay).  16-byte aligned rows / strides. */
UC_API int uc_copy_rows_if(const int* flag_dev, int invert, const void* src, long src_ld_bytes, void* dst, long dst_ld_bytes, long rows,
                           int row_bytes, void* stream);
UC_API int uc_nchw_f32_to_nhwc(const float* src, void* dst, int ldd, int B, int C, long HW, int dtype, void* stream);
UC_API int uc_nhwc_to_nchw_f32(const void* src, int lds, float* dst, int B, int C, long HW, int dtype, void* stream);

/* Drop-in for MultiScaleDeformableAttention.ms_deform_attn_forward (ops/src/ms_deform_attn.h:20-39):
 * value [B,S,M,D] f32, spatial_shapes [L,2] i64 (device), level_start_index [L] i64 (device),
 * sampling_loc [B,Lq,M,L,P,2] f32 normalised (x,y), attn_weight [B,Lq,M,L,P] f32 -> out [B,Lq,M*D] f32. */
UC_API int uc_msda_forward_f32(const float* value, const int64_t* spatial_shapes, const int64_t* level_start_index,
                               const float* sampling_loc, const float* attn_weight, int B, int S, int M, int D, int L,
                               int Lq, int P, float* out, void* stream);
/* Fused form used by the B200 path (B=1, head dim 32): value bf16 [S, M*32]; offlog f32 [Lq, ld] = raw
 * sampling_offsets (M*L*P*2) followed by attention logits (M*L*P); queries = concatenated level grids;
 * level_hw host int[2L] (h,w).  out bf16 [Lq, M*32]. */
UC_API int uc_msda_fused_bf16(const void* value, const float* offlog, int ld_offlog, void* out, const int* level_hw,
                              int L, int M, int P, void* stream);

/* Fused correlation + softmax over reference positions + label propagation
 * (external/lib/test/tracker/unicorn_sot.py:95-100; unicorn_vos.py:171-181):
 *   out[o,j] = sum_i values[o,i] * softmax_i(<embed_ref[i,:], embed_cur[j,:]>)
 * embed_* [n, C=128] 16-bit rows (NHWC embedding maps), values f32 [n_obj, ldv], out f32 [n_obj, ldo]; n_obj <= 8. */
UC_API int uc_corr_propagate(const void* embed_ref, int ld_ref, int n_ref, const void* embed_cur, int ld_cur, int n_cur,
                             int C, int dtype, const float* values, int ldv, int n_obj, float* out, int ldo, void* stream);

/* Head decode (unicorn_head.py:332-334,467-482): per level regobj f32 [HW, ld_ro] = reg(4), obj logit;
 * cls f32 [HW, ld_cls] = class logits.  regobj/cls/hw/strides are HOST arrays of 3 device pointers / ints.
 * out f32 [sum HW, 5+ncls] = cx,cy,w,h,sigmoid(obj),sigmoid(cls..). */
UC_API int uc_head_decode(const float* const* regobj, const float* const* cls, const int* hw, const int* strides,
                          int ld_ro, int ld_cls, int ncls, float* out, void* stream);

/* postprocess (utils/boxes.py:33-77) on the device: out_dets f32 [<=A, 7] rows (x1,y1,x2,y2,obj,cls_conf,cls_id)
 * in descending score order, *out_count (device int) = number of rows.  max_keep > 0 stops the greedy scan once that
 * many boxes are kept: the rows returned are exactly the first max_keep rows of the full result (the SOT driver only
 * consumes output[:max_inst], external/lib/test/tracker/unicorn_sot.py:69-70); max_keep <= 0 = no limit.
 * out_anchor (device int[A], may be NULL) receives the anchor index of every returned row — what postprocess_inst
 * (utils/boxes.py:125-128) needs to pick each instance's location / dynamic parameters / FPN level. */
UC_API long uc_postprocess_workspace_bytes(int max_anchors);
UC_API int uc_postprocess(const float* pred, int A, int ncls, float conf_thre, float nms_thre, int max_keep, void* workspace,
                          long workspace_bytes, float* out_dets, int* out_count, int* out_anchor, void* stream);

/* Instance-embedding sampling at box centres (unicorn/evaluators/mot_evaluator.py:1024-1034): embed NHWC 16-bit
 * [h,w,C] (pixel stride ld), boxes f32 [n,ldb] xyxy in network-input pixels, stride = 8; grid_sample(bilinear,
 * border, align_corners=False) semantics incl. the reference's clamp/normalise step.  n = min(*count_dev, n_max)
 * (count_dev may be NULL).  out f32 [n_max, C]. */
UC_API int uc_sample_embed(const void* embed, int ld, int h, int w, int C, int dtype, const float* boxes, int ldb,
                           const int* count_dev, int n_max, float stride, float* out, void* stream);
/* Quasi-dense association score (unicorn/tracker/quasi_dense_embed_tracker.py:166-175): scores = (softmax_rows(F) +
 * softmax_cols(F)) / 2 with F = E M^T, zeroed where labels differ (labels may be NULL).  workspace >= N*M+2N+2M floats. */
UC_API int uc_bisoftmax(const float* det_embeds, const float* memo_embeds, int N, int M, int C, const float* det_labels,
                        const float* memo_labels, float* workspace, float* scores, void* stream);
/* Greedy assignment of QuasiDenseEmbedTracker.match (unicorn/tracker/quasi_dense_embed_tracker.py:188-199) on the device: rows =
 * detections in descending score order, scores f32 [N,M] from uc_bisoftmax, memo_ids int64 [M] (-1 = backdrop), det_scores f32
 * (element stride ld_det: column 4 of the [N,5] box rows).  ids_out int64 [N]: the tracklet id, -2 (duplicate of a tracklet, dropped)
 * or -1 (unmatched).  taken_ws: M bytes of scratch.  One CTA; torch.max tie-breaking (first maximum). */
UC_API int uc_qd_assign(const float* scores, int N, int M, const long long* memo_ids, const float* det_scores, int ld_det, float match_thr,
                        float obj_thr, float nms_conf_thr, long long* ids_out, uint8_t* taken_ws, void* stream);
/* Pairwise IoU out[i,j] of xyxy f32 boxes with row strides.  plus_one = 0: torchvision.ops.box_iou
 * (quasi_dense_embed_tracker.py:80,146); plus_one = 1: cython_bbox.bbox_overlaps' inclusive-pixel convention
 * (unicorn/tracker/matching.py:65-68, ByteTrack). */
UC_API int uc_box_iou(const float* a, int lda, int N, const float* b, int ldb, int M, float* out, int plus_one, void* stream);

/* dst += aligned_bilinear(src, factor) on NHWC bf16 maps (condinst/comm.py:5-27; mask_branch.py:81-96). */
UC_API int uc_aligned_bilinear_add(const void* src, int lds, int hs, int ws, void* dst, int ldd, int C, int factor, void* stream);
/* Per-instance CondInst masks (condinst/dynamic_mask_head.py:61-87,159-225,284; utils/boxes.py:138-145) for the first
 * min(*count_dev, n_max) rows of the NMS output: mask_feats f32 [h,w,8], up_masks f32 [h,w,9*up_rate^2],
 * dyn_levels = HOST array of 3 device pointers to the controller outputs [h_k*w_k, ld_dyn] (169 used), level_hw /
 * level_strides / level_soi host arrays; anchors_dev = out_anchor of uc_postprocess; scratch >= n_max*h*w*(1+up^2)
 * floats; out_masks f32 [n_max, h*up*d, w*up*d] = sigmoid scores. */
UC_API int uc_dynamic_masks(const float* mask_feats, const float* up_masks, int h, int w, int up_rate, int d_rate,
                            const float* const* dyn_levels, int ld_dyn, const int* level_hw, const int* level_strides,
                            const float* level_soi, const int* anchors_dev, const int* count_dev, int n_max, float* scratch,
                            float* out_masks, void* stream);

/* VOS result assembly on the device (external/lib/test/tracker/unicorn_vos.py:129-155 mask resize to the original frame,
 * :105-121 soft aggregation + argmax): for every object either `mask` (f32 [Hin,Win] soft mask at network resolution, resized
 * with F.interpolate(scale_factor=1/r, bilinear, align_corners=False)[:H,:W]) or `init_mask` (uint8 [H,W] label map of the
 * frame the object first appears in; object = label == id) or neither (no detection: zeros).  objs is a HOST array in the
 * reference's list order (the float32 background product follows it).  soft_out (may be NULL) f32 [n,H,W]; seg_out uint8 [H,W]. */
typedef struct UcVosObject {
  const float* mask;
  const uint8_t* init_mask;
  int id;
} UcVosObject;
UC_API int uc_vos_aggregate(const UcVosObject* objs, int n, int Hin, int Win, int H, int W, float r, float* soft_out,
                            uint8_t* seg_out, void* stream);

/* MOTS mask tail on the device (unicorn/evaluators/mot_evaluator.py:804-805 resize + threshold, :858-866 overlap free, :882-888
 * area filter + COCO RLE): masks f32 [n_max, Hin, Win] (uc_dynamic_masks output); rows device int32 [K] = the mask rows in
 * output order (ascending track id); emit device int32 [K] = 1 for the rows that pass the area filter.  Every row is resized
 * with F.interpolate(scale_factor, bilinear, align_corners=False) — output floor(Hin * scale_factor) x floor(Win * scale_factor)
 * computed in double, source scale (float)(1 / scale_factor) —, cropped to [:img_h, :img_w], thresholded (value > thres) and
 * keeps only the pixels no earlier row of `rows` claimed (rows with emit = 0 claim too).  Each emitted row is encoded as the
 * COCO compressed RLE string of its column-major mask (byte-identical to unicorn_b200.results.rle_encode).
 * Outputs (device): out_len[k] = string length (0 when not emitted), out_off[k] = its offset in out_chars, *out_total = the sum
 * of the lengths.  Strings are written only where they fit in `capacity` bytes; when *out_total > capacity, run again with a
 * larger buffer.  workspace >= uc_mots_rle_workspace_bytes(K, Hin, Win, img_h, img_w, scale_factor) bytes (0 = bad sizes). */
UC_API long uc_mots_rle_workspace_bytes(int K, int Hin, int Win, int img_h, int img_w, double scale_factor);
UC_API int uc_mots_masks_rle(const float* masks, int n_max, int Hin, int Win, const int* rows, const int* emit, int K, int img_h,
                             int img_w, float thres, double scale_factor, void* workspace, long workspace_bytes, long long* out_len,
                             long long* out_off, long long* out_total, char* out_chars, long capacity, void* stream);

#ifdef __cplusplus
}
#endif
#endif
