/*
 * step_b200.h -- C ABI of libstep_b200.so: the sm_100a implementation of the STEP hot path.
 *
 * This is the drop-in boundary (SURVEY.md section 8b).  Every entry point takes raw device
 * pointers, plain sizes and an explicit cudaStream_t; none allocates, synchronises or touches
 * the default stream, so each is CUDA-graph capturable.  Every entry returns 0 on success or a
 * non-zero code (a cudaError_t, or STEP_E_* below); step_last_error() then describes it.
 *
 * Reference interface each group replaces (paths relative to the NVlabs/STEP tree):
 *   nms            external/maskrcnn_benchmark/csrc/vision.cpp:31  _C.nms  (nms.h:34-51,
 *                  cpu/nms_cpu.cpp:29-99, cuda/nms.cu:47-155)
 *   roi_align_*    vision.cpp:32-33  _C.roi_align_forward/backward  (ROIAlign.h:35-69,
 *                  cpu/ROIAlign_cpu.cpp:137-281, cuda/ROIAlign_cuda.cu:88-370)
 *   roi_pool_*     vision.cpp:34-35  _C.roi_pool_forward/backward   (ROIPool.h:35-71,
 *                  cuda/ROIPool_cuda.cu:40-226)
 *   tube_*         utils/tube_utils.py:10-27,59-92,127-189,214-266 and the per-step host loop of
 *                  utils/utils.py:61-129
 *   conv / pool / linear / head_*   the torch.nn calls of models/i3dpt.py:43-163,
 *                  models/networks.py:69-83, models/two_branch.py:60-111,132-138,223-274,337
 *   clip_*         the permute + (apex) cast at models/networks.py:77
 *   frames_*       data/augmentations.py:68-169,601-615; data/ava.py:330-338
 *
 * Tensor conventions: activations are channels-last -- [N, T, H, W, C] ("NDHWC") with an explicit
 * channel stride `ld` (elements) so a kernel can read or write a channel slice of a wider buffer
 * (this is how Mixed's concat, i3dpt.py:162, and the local-branch concat, two_branch.py:256,
 * disappear).  The *_nchw entry points take the reference's NCHW fp32 layout unchanged.
 */
#ifndef STEP_B200_H_
#define STEP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct CUstream_st* step_stream_t; /* == cudaStream_t */

enum { STEP_F32 = 0, STEP_F16 = 1 };
enum { STEP_OK = 0, STEP_E_ARG = 10001, STEP_E_UNSUPPORTED = 10002, STEP_E_WORKSPACE = 10003,
       STEP_E_DRIVER = 10004 };

int step_version(void);
const char* step_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
uint64_t step_launch_count(void);

/* ------------------------------------------------------------------ NMS ------------------ */
/* Greedy NMS, legacy "+1" areas, bit-exact with cpu/nms_cpu.cpp (ge=1: suppress when
 * IoU >= thr) or cuda/nms.cu (ge=0: IoU > thr).  Order: score descending, original index
 * ascending on ties.  keep_out receives the kept ORIGINAL indices in ascending order,
 * *n_keep (device int) their count.  Fully device-resident (no host scan, no D2H). */
size_t step_nms_workspace_bytes(int n);
int step_nms_f32(const float* boxes /*[n,4]*/, const float* scores /*[n]*/, int n, float thr, int ge,
                 int64_t* keep_out /*[n]*/, int* n_keep, void* workspace, size_t ws_bytes,
                 step_stream_t stream);
/* Many independent small problems in one launch (the per-clip x per-class loop of test.py:178-201):
 * segment s = rows [seg_offsets[s], seg_offsets[s+1]); at most 1024 rows per segment.
 * keep_mask[i] = 1 if row i survives NMS inside its segment.  Rows with score < min_score are
 * dropped before NMS (test.py:183 confidence threshold; pass -INF to disable). */
int step_nms_segmented_f32(const float* boxes, const float* scores, const int* seg_offsets, int n_seg,
                           float thr, int ge, float min_score, uint8_t* keep_mask, step_stream_t stream);
/* Rows one segment may hold (shared-memory resident problem); a longer segment traps instead of overrunning. */
int step_nms_segmented_max_rows(void);

/* Detection post-processing of the reference drivers (test.py:156-218, demo.py:121-198) in two launches, no host
 * round trip: for every (clip, class) keep the tubes whose class score > conf_thresh (scores.gt, test.py:183), clamp
 * their box with valid_tubes(valid_w, valid_h) (the drivers use its 400x400 defaults, test.py:191), greedy NMS with the
 * cpu/nms_cpu.cpp predicate, divide by (norm_w, norm_h) (test.py:197-198); then per clip either all survivors in file
 * order (class, tube) when topk <= 0, or the topk best in the order of the tuple sort of test.py:205-208.
 *   prob [n_rows, prob_ld >= ncls]  class scores of the centre frame;  loc: centre-frame box of row r at loc + r*loc_ld
 *   clip_offsets [n_clips+1] (device int32): rows of clip b = [clip_offsets[b], clip_offsets[b+1]), at most
 *   step_nms_segmented_max_rows() of them (max_per_clip is the caller's host-side bound, checked here).
 * Candidate arrays (index clip_start*ncls + class*n_clip + tube): keep [n_rows*ncls] u8, score [n_rows*ncls],
 * box [n_rows*ncls, 4] normalised.  Compact result: det [n_clips, cap, 8] = {x1, y1, x2, y2, score, class, tube, 0},
 * det_count [n_clips] (int32, <= cap). */
int step_detect_f32(const float* prob, int prob_ld, const float* loc, int loc_ld, const int* clip_offsets,
                    int n_clips, int n_rows, int max_per_clip, int ncls, float conf_thresh, float nms_thresh,
                    int ge, float valid_w, float valid_h, float norm_w, float norm_h, int topk, int cap,
                    uint8_t* keep, float* score, float* box, float* det, int* det_count, step_stream_t stream);

/* ------------------------------------------------------------------ ROI ops -------------- */
/* Reference layout (NCHW fp32 in, [R,C,ph,pw] fp32 out), arithmetic order of the reference. */
int step_roi_align_fwd_nchw_f32(const float* feat, int K, int C, int H, int W, const float* rois, int R,
                                float scale, int ph, int pw, int sampling_ratio, float* out,
                                step_stream_t stream);
int step_roi_align_bwd_nchw_f32(const float* grad_out, const float* rois, int R, float scale, int ph,
                                int pw, int K, int C, int H, int W, int sampling_ratio,
                                float* grad_in /* zero-filled by the call */, step_stream_t stream);
int step_roi_pool_fwd_nchw_f32(const float* feat, int K, int C, int H, int W, const float* rois, int R,
                               float scale, int ph, int pw, float* out, int32_t* argmax,
                               step_stream_t stream);
int step_roi_pool_bwd_nchw_f32(const float* grad_out, const int32_t* argmax, const float* rois, int R,
                               int ph, int pw, int K, int C, int H, int W,
                               float* grad_in /* zero-filled by the call */, step_stream_t stream);
/* Channels-last fast path: feat [K,H,W,C] (channel stride feat_ld), out [R,ph,pw,C] (channel
 * stride out_ld).  dtype STEP_F32 / STEP_F16 (fp32 accumulation, same operation order as the
 * reference; the fp32 variant is bit-identical to the NCHW one up to the permutation).
 * C must be a multiple of 8 (f16) / 4 (f32); feat_ld, out_ld likewise.
 * Frame map: ROI column 0 indexes frames of the slice conv_feat[:, t_start:t_start+roi_T]
 * (utils/utils.py:48); with roi_T > 0 the kernel reads frame (f / roi_T) * feat_T + t_start + f % roi_T
 * of the full map instead of needing the slice copied.  roi_T == 0: identity.
 * exact == 1: reference operation order, bit-identical (always used for f32).  f16 storage only: exact == 2:
 * 1/count folded into the tap weights, one fp32 FMA per tap (within one fp16 ulp of the exact result);
 * exact == 0: per-pixel merged weights + packed half2 FMAs (a convex combination: a few fp16 ulps). */
int step_roi_align_fwd_nhwc(const void* feat, int dtype, int K, int H, int W, int C, int feat_ld,
                            const float* rois, int R, float scale, int ph, int pw, int sampling_ratio,
                            void* out, int out_ld, int roi_T, int feat_T, int t_start, int exact,
                            step_stream_t stream);
int step_roi_pool_fwd_nhwc(const void* feat, int dtype, int K, int H, int W, int C, int feat_ld,
                           const float* rois, int R, float scale, int ph, int pw, void* out, int out_ld,
                           int roi_T, int feat_T, int t_start, step_stream_t stream);

/* ------------------------------------------------------------------ tube arithmetic ------ */
/* boxes are rows of 4 floats with a row stride (in floats) so the [.,5] flat-tube layout
 * (frame index first, tube_utils.py:238) can be addressed in place. */
int step_tube_decode_f32(const float* anchors, int anchor_stride, const float* deltas, int n, float* out,
                         step_stream_t stream);                         /* tube_utils.py:165-189 */
int step_tube_encode_f32(const float* gt, const float* anchors, int anchor_stride, int n, float* out,
                         step_stream_t stream);                         /* tube_utils.py:143-163 */
int step_tube_valid_f32(float* boxes /*in place, [n,4]*/, int n, float width, float height,
                        step_stream_t stream);                          /* tube_utils.py:59-92 */
int step_tube_extrapolate_f32(const float* tubes /*[n,L,4]*/, int n, int L, int T, float width,
                              float height, float* out /*[n,L+2T,4]*/, step_stream_t stream); /* :10-27 */
int step_tube_extend_f32(const float* tubes /*[n,5]*/, int n, float ratio, float width, float height,
                         float* out /*[n,5]*/, step_stream_t stream);   /* tube_utils.py:248-266 */
/* One launch for the whole between-steps host loop of utils/utils.py:61-129:
 * decode (local, and first/last when mode==PREDICT) -> optional temporal extension
 * (concat / extrapolate / mean) -> valid_tubes -> re-flatten with new frame indices.
 * flat_in [R,L,5]; loc/first/last [R,L,4]/[R,T,4]/[R,T,4]; clip_of_tube [R] int32;
 * pred_* are the history tensors; flat_out [R,L_out,5] with L_out = extend ? L+2T : L. */
enum { STEP_EXT_NONE = 0, STEP_EXT_PREDICT = 1, STEP_EXT_EXTRAPOLATE = 2, STEP_EXT_MEAN = 3 };
int step_tube_update_f32(const float* flat_in, const float* loc, const float* first, const float* last,
                         const int32_t* clip_of_tube, int R, int L, int T, int decode_neighbors,
                         int ext_mode, float width, float height, float* pred_loc, float* pred_first,
                         float* pred_last, float* flat_out, step_stream_t stream);

/* ------------------------------------------------------------------ layout --------------- */
/* clip [N,T,Cc,H,W] fp32 (the layout BaseNet.forward receives, networks.py:69-76) ->
 * channels-last [N,T,H,W,ld] in `dtype`, channels >= Cc zero-filled. */
int step_clip_to_ndhwc(const float* clip, int N, int T, int Cc, int H, int W, void* out, int dtype, int ld,
                       step_stream_t stream);
/* Same input, space-to-depth by 2 in (T,H,W) for the stride-2 stem (i3dpt.py:184-189):
 * out [N,T/2,H/2,W/2,ld] f16 with channel = ((rt*2+rh)*2+rw)*Cc + c. T,H,W must be even. */
int step_clip_to_s2d_f16(const float* clip, int N, int T, int Cc, int H, int W, void* out, int ld,
                         step_stream_t stream);
/* Test-time input transform from decoded frames (BaseTransform, augmentations.py:601-615, then the BGR -> RGB swap and
 * permute of ava.py:330-338): ConvertFromInts(scale) -> cv2.resize INTER_LINEAR on fp32 to (W, H) -> (v - mean) / std, in
 * the reference's fp32 order.  frames [N,T,Hmax,Wmax,3] uint8 BGR as cv2.imread returns them; clip n fills the top-left
 * H0 x W0 of each of its frame slots (row pitch Wmax*3 bytes), with sizes [N,2] = (H0, W0) a DEVICE int32 table, so one
 * captured graph serves any mix of source sizes up to (Hmax, Wmax).  The caller validates the table (1 <= H0 <= Hmax,
 * 1 <= W0 <= Wmax); the kernels clamp to the slot.  mean_* / std_* are in BGR order, as BaseTransform takes them;
 * scale is 0 ([0,255]), 1 ([0,1]) or 2 ([-1,1]).
 * step_frames_to_clip_f32: out [N,T,3,H,W] fp32 RGB, the clip BaseNet.forward receives.
 * step_frames_to_s2d_f16: out [N,T/2,H/2,W/2,32] f16 (32-byte aligned), bit-identical to step_clip_to_s2d_f16(ld = 32)
 * applied to the clip form.  T, H, W must be even. */
int step_frames_to_clip_f32(const uint8_t* frames, const int32_t* sizes, int N, int T, int Hmax, int Wmax, int H, int W,
                            int scale, float mean_b, float mean_g, float mean_r, float std_b, float std_g, float std_r,
                            float* out, step_stream_t stream);
int step_frames_to_s2d_f16(const uint8_t* frames, const int32_t* sizes, int N, int T, int Hmax, int Wmax, int H, int W,
                           int scale, float mean_b, float mean_g, float mean_r, float std_b, float std_g, float std_r,
                           void* out, step_stream_t stream);
/* channels-last [M, C] (stride ld) <-> planar [N, C, S] fp32, M = N*S (boundary conversions). */
int step_nhwc_to_nchw_f32(const void* in, int dtype, int N, int S, int C, int ld, float* out,
                          step_stream_t stream);
int step_nchw_to_nhwc(const float* in, int N, int S, int C, void* out, int dtype, int ld,
                      step_stream_t stream);

/* ------------------------------------------------------------------ conv / pool / linear - */
typedef struct {
  int dtype;                 /* STEP_F32: SIMT fp32 path.  STEP_F16: tcgen05 implicit GEMM, fp32 accumulate */
  int N, T, H, W;            /* input extent (pixels) */
  int Cin, in_ld;            /* input channels read, channel stride of x */
  int Cout, out_ld, out_coff;/* output channels, channel stride of y, first channel written in y */
  int KT, KH, KW;            /* filter taps */
  int ST, SH, SW;            /* strides (the f16 path supports stride 1 only; the stem uses s2d) */
  int PT, PH, PW;            /* low-side zero padding (TF "SAME": i3dpt.py:14-31) */
  int OT, OH, OW;            /* output extent */
  int relu;                  /* apply max(.,0) last */
  int w_ld;                  /* weight channel stride: w is [Cout, KT, KH, KW, w_ld] in `dtype` */
  const void* x;
  const void* w;
  const float* scale;        /* per-Cout multiplier (folded BatchNorm, i3dpt.py:107) or NULL (=1) */
  const float* shift;        /* per-Cout addend (folded BN shift / conv bias) or NULL (=0) */
  const void* residual;      /* optional tensor added before relu (two_branch.py:79-81), layout of y */
  int res_ld, res_coff;
  void* y;
  int a_mode;                /* f16 path: 0 auto, 1 linear (1x1x1 only), 2 box tiles, 3 TMA im2col,
                                4 input patch staged in shared memory (stride 1, Cin in {16,32,64}, Cout <= 256),
                                5 best of 3 / 4 per layer shape, 9 SIMT */
  /* Horizontally fused 1x1x1 layers that share an input (Mixed.branch_0 / branch_1[0] / branch_2[0],
   * i3dpt.py:133-147): output channels [0, split[0]) go to y, [split[0], split[1]) to y_extra[0],
   * [split[1], Cout) to y_extra[1], each with its own channel stride / offset.  n_splits = 0: plain conv.
   * f16 1x1x1 only; split points must be multiples of 16. */
  int n_splits;
  int split[2];
  void* y_extra[2];
  int ld_extra[2];
  int coff_extra[2];
  /* Structured zeros of the weights (a_mode 4 only): for the filter taps of the LAST t plane (kt == KT-1) the input
   * channels [zero_cin_last_kt, Cin) carry zero weights, so their 16-channel MMA steps are skipped.  0 = no such
   * structure.  The space-to-depth stem has it: tap plane qt = 2 only holds the rt = 0 sub-position (k = 2(q+1)+r <= 6),
   * engine.pack_stem_s2d. */
  int zero_cin_last_kt;
} step_conv_params;
int step_conv3d_fwd(const step_conv_params* p, step_stream_t stream);

/* MaxPool3dTFPadding (i3dpt.py:114-126): zero pad (low PT/PH/PW, high implied), ceil_mode. */
int step_maxpool3d_fwd(const void* x, int dtype, int N, int T, int H, int W, int C, int in_ld, int KT,
                       int KH, int KW, int ST, int SH, int SW, int PT, int PH, int PW, int pad_hi_t,
                       int pad_hi_h, int pad_hi_w, int OT, int OH, int OW, void* y, int out_ld,
                       step_stream_t stream);
/* mean over axis B: x [A, B, P, C] (C contiguous, pixel stride ld) -> y [A, P*C] fp32/f16
 * (the temporal mean of two_branch.py:249 taken before the classifier, which is linear). */
int step_mean_mid(const void* x, int dtype, int A, int B, int P, int C, int ld, void* y, int out_dtype,
                  step_stream_t stream);
/* y[m, n] = act(sum_k x[m,k] * w[n,k] + bias[n]); small-N GEMM (N <= 64) for global_cls,
 * local_reg, neighbor_reg (two_branch.py:246,261,269-270).  x [M,K] (row stride x_ld) in dtype,
 * w [N,K] in dtype, y fp32 [M, y_ld].  act: 0 none, 1 sigmoid (applied after accumulation).
 * accumulate != 0: y += result.  row_map (optional, device int32 [M]): x row read for output row m
 * (the per-tube context gather of utils/utils.py:54-57).
 * Split-K with a caller-provided fp32 workspace of step_linear_small_n_workspace_bytes(M,K,N). */
size_t step_linear_small_n_workspace_bytes(int M, int K, int N);
int step_linear_small_n(const void* x, int dtype, int M, int K, int x_ld, const void* w, const float* bias,
                        int N, float* y, int y_ld, int act, int accumulate, const int32_t* row_map,
                        void* workspace, size_t ws_bytes, step_stream_t stream);

/* local_reg + neighbor_reg1 + neighbor_reg2 of TwoBranchNet (two_branch.py:261-270) in one pass over the
 * [R*T, K] feature rows: w12 = [W_local | W_nb1 | W_nb2] (12 x K), bias12 likewise.  Writes
 * local_loc [R,T,4], first_loc [R,s1-s0,4] = (local + nb1)[:, s0:s1], last_loc [R,e1-e0,4] = (local + nb2)[:, e0:e1].
 * workspace: step_linear_small_n_workspace_bytes(R*T, K, 12). */
int step_head_regress(const void* x, int dtype, int R, int T, int K, int x_ld, const void* w12, const float* bias12,
                      int s0, int s1, int e0, int e1, float* local_loc, float* first, float* last, void* workspace,
                      size_t ws_bytes, step_stream_t stream);

/* Exit of a 2-D bottleneck of the local branch fused with the 1x1 convolution that consumes it, fp16, channels-last rows:
 *   y[M, inplanes] = relu(h[M, planes] * w3[inplanes, planes]^T + x[M, inplanes])      Bottleneck.forward, models/two_branch.py:79-83
 *                                                                                 (Bottleneck_resample.forward, :106-110)
 *   z[M, outplanes] = act(y * w1[outplanes, inplanes]^T + shift2)                   the next block's conv1 + ReLU (:68-69, relu2 = 1,
 *                                                                                 shift2 = NULL) or downsample2 (:259, relu2 = 0, bias)
 * in one launch; y may be NULL when nothing else reads it.  Bit-identical to step_conv3d_fwd called twice.  Built for the
 * reference's fixed head widths planes = 256, inplanes = 1024, outplanes = 256 (two_branch.py:190-192); other widths return
 * STEP_E_ARG and the caller launches the two convolutions.  Row pitches in elements. */
int step_bottleneck_exit_f16(const void* h, long long h_ld, const void* w3, const void* x, long long x_ld, const void* w1,
                             const float* shift2, int relu2, void* y, long long y_ld, void* z, long long z_ld, long long M,
                             int planes, int inplanes, int outplanes, step_stream_t stream);

/* ------------------------------------------------------------------ training (first pieces) ---- */
/* TwoBranchNet's losses (models/two_branch.py:276-333) and, when the d* pointers are given, the gradient of the training
 * objective mean(loss_cls) + w_loc * loss_loc + w_nb * loss_nb (train.py:323-347) with respect to the head outputs.
 *   logits [N,cls] (pre-sigmoid), local_loc [N,T_len,4], first_loc / last_loc [N,Tc,4], tubes [N,T_len,5],
 *   targets [N,3,6+cls] = (first, centre, last) x (box 4 | cls mask | loc mask | labels).
 * loss_cls [N*cls] holds the element-wise BCE (all zeros when no sample is positive: flags[0] = 0 and the reference then
 * returns the scalar 0), loss_loc / loss_nb [1]; flags [3] = {cls, loc, neighbour mask sums non-zero}.
 * dloc [N,T_len,4] already includes what flows back through the first / last slices.  scratch: N*12 floats. */
int step_head_losses_f32(const float* logits, const float* local_loc, const float* first_loc, const float* last_loc,
                         const float* tubes, const float* targets, int N, int cls, int T_len, int T, int Tc, float w_loc,
                         float w_nb, float* loss_cls, float* loss_loc, float* loss_nb, int* flags, float* dlogits,
                         float* dloc, float* dfirst, float* dlast, float* scratch, step_stream_t stream);
/* Channels-last ROIAlign backward without atomics (replaces _C.roi_align_backward, vision.cpp:33 /
 * cuda/ROIAlign_cuda.cu:201-278, whose atomicAdd scatter is not repeatable): grad_out [R,ph,pw,C] (channel stride
 * out_ld, STEP_F32 / STEP_F16) -> grad_in [K,H,W,C] fp32 (channel stride in_ld), written completely by the call. */
int step_roi_align_bwd_nhwc(const void* grad_out, int dtype, int out_ld, const float* rois, int R, float scale, int ph,
                            int pw, int K, int H, int W, int C, int sampling_ratio, float* grad_in, int in_ld,
                            step_stream_t stream);
/* Backward of y = x W^T + b for the small-N linears of the head (nn.Linear / global_cls, two_branch.py:246-270):
 * dx [M,K] (+)= dy W, dw [Nn,K] = dy^T x, db [Nn] = column sums of dy; any of dx / dw may be NULL.  Fixed summation order. */
int step_linear_small_n_bwd(const void* x, int dtype, int M, int K, int x_ld, const float* w, const float* dy, int Nn,
                            float* dx, int dx_accumulate, float* dw, float* db, step_stream_t stream);
/* Weight gradient of a 1x1(x1) convolution: dw[Cout,Cin] (+)= scale * sum_m dz[m,co] x[m,ci]; fp16 operands, fp32
 * tensor-core accumulation, pixel chunks reduced in a fixed order (deterministic). */
size_t step_conv1x1_wgrad_workspace_bytes(int M, int Cout, int Cin);
int step_conv1x1_wgrad_f16(const void* dz, int dz_ld, const void* x, int x_ld, int M, int Cout, int Cin, float scale,
                           float* dw, int dw_ld, int accumulate, void* workspace, size_t ws_bytes, step_stream_t stream);

/* Weight gradient of a stride-1 convolution with KT x KH x KW taps and low padding (PT, PH, PW) (zero outside the map):
 * dw[Cout, taps, dw_ld >= Cin] (+)= scale * sum_m dz[m, co] x[shift_tap(m), ci], x and dz on the same [N,T,H,W] pixel grid. */
size_t step_conv_wgrad_workspace_bytes(int M, int Cout, int Cin, int taps);
int step_conv_wgrad_f16(const void* dz, int dz_ld, const void* x, int x_ld, int N, int T, int H, int W, int Cout, int Cin,
                        int KT, int KH, int KW, int PT, int PH, int PW, float scale, float* dw, int dw_ld, int accumulate,
                        void* workspace, size_t ws_bytes, step_stream_t stream);
/* y = relu(scale * conv + shift (+ residual)): dz = dy * [y > 0] * scale (dense [M, C] at dz_ld), and, when dres is given,
 * dres += dy * [y > 0] (the residual input's gradient, accumulated in place).  fp16, channel slices via the ld arguments. */
int step_act_bwd_f16(const void* dy, int dy_ld, const void* y, int y_ld, const float* scale, int relu, long long M, int C,
                     void* dz, int dz_ld, void* dres, int dres_ld, step_stream_t stream);
/* out[c] = scale * sum_m x[m, c] (bias gradients); workspace >= 64 * C floats; fixed summation order. */
int step_colsum_f16(const void* x, int ld, long long M, int C, float scale, float* out, float* workspace, step_stream_t stream);
/* Backward of step_mean_mid: dx[a, b, p, c] += gscale * g[a, p*C + c] / B (fp16 dx, channel stride ld). */
int step_mean_mid_bwd(const float* g, int A, int B, int P, int C, float gscale, void* dx, int ld, step_stream_t stream);
/* dst[m, c] (fp16, channel stride ld) += gscale * src[m, c] (fp32 [M, C]). */
int step_f32_accum_f16(const float* src, long long M, int C, float gscale, void* dst, int ld, step_stream_t stream);
/* Backward of step_maxpool3d_fwd (zero padding takes part in the maximum, first maximum in scan order wins as in ATen):
 * dx += scatter(dy) without atomics; argmax_ws: N*OT*OH*OW*C bytes of scratch. */
int step_maxpool3d_bwd_f16(const void* x, int x_ld, const void* dy, int dy_ld, int N, int T, int H, int W, int C, int KT,
                           int KH, int KW, int ST, int SH, int SW, int PT, int PH, int PW, int pad_hi_t, int pad_hi_h,
                           int pad_hi_w, int OT, int OH, int OW, void* dx, int dx_ld, uint8_t* argmax_ws, step_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* STEP_B200_H_ */
