/*
 * s2a_b200.h -- C ABI of libs2a_b200.so: the S2ANet custom-op hot path for NVIDIA B200 (sm_100a).
 *
 * Plain C: device pointers, sizes and an explicit CUDA stream (a cudaStream_t passed as void*,
 * NULL = the legacy default stream).  No torch types.  Every function returns S2A_OK (0) or a
 * negative status; s2a_last_error() returns a thread-local message for the last failure.
 * All work is enqueued on `stream`; nothing synchronises the host unless stated.
 *
 * Each entry point names the reference (chongkuiqi/S2ANet) interface it replaces; the torch-side
 * binding that maps the reference's extension-module functions onto these symbols lives in
 * s2anet_b200/ (Python + ctypes) and is described in INTEGRATION.md.
 */
#ifndef S2A_B200_H_
#define S2A_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define S2A_EXPORT __attribute__((visibility("default")))
#else
#define S2A_EXPORT
#endif

enum {
  S2A_OK = 0,
  S2A_ERR_INVALID_ARGUMENT = -1,
  S2A_ERR_CUDA = -2,
  S2A_ERR_WORKSPACE = -3,
  S2A_ERR_UNSUPPORTED = -4
};

/* element types of activation / weight tensors */
enum { S2A_F32 = 0, S2A_BF16 = 1, S2A_F16 = 2 };

/* flags of s2a_box_iou_rotated */
enum {
  S2A_IOU_DEFAULT = 0,
  S2A_IOU_NO_REJECT = 1 /* run the polygon clipper on every pair (testing: must not change a bit) */
};

S2A_EXPORT int s2a_version(void);
S2A_EXPORT const char* s2a_last_error(void);
/* Measurement utility (bench.py): achieved FP32 FMA throughput of this GPU in TFLOP/s, the denominator of the
 * "pairs/s / FP32-bound" figure SURVEY.md 8d asks for next to the rotated-IoU numbers.  Blocking. */
S2A_EXPORT int s2a_measure_fp32_fma_tflops(double* tflops_out, int reps, void* stream);
/* Layout conversion between the reference's NCHW tensors (models/dcn/src/deform_conv_cuda.cpp:168-170 makes them
 * contiguous NCHW) and the NHWC operands of the tensor-core kernels: src [batch][rows][cols] -> dst [batch][cols][rows],
 * elements of 2 or 4 bytes.  NCHW -> NHWC: rows = C, cols = H*W; NHWC -> NCHW: rows = H*W, cols = C. */
S2A_EXPORT int s2a_transpose_planes(const void* src, void* dst, int64_t batch, int64_t rows, int64_t cols,
                                    int elem_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * box_iou_rotated -- replaces box_iou_rotated_cuda()
 *   reference: utils/box_iou_rotated/src/box_iou_rotated_cuda.cu:65-101 (host), :13-62 (kernel),
 *              utils/box_iou_rotated/src/box_iou_rotated.h:22-37 (dispatcher)
 * boxes1 [batch, n, 5], boxes2 [batch, m, 5] fp32 contiguous (x, y, w, h, theta[rad]);
 * out[b, i, j] = IoU(boxes1[b, i], boxes2[b, j]) written at out + b*n*ld_out + i*ld_out + j
 * (ld_out >= m, in elements).  batch = 1 is the reference's call; batch > 1 is the batched
 * anchor x GT assignment of BASELINE config 4.  n == 0 or m == 0 is a no-op.
 * row_begin/row_end restrict the computed rows to [row_begin, row_end) (anchor-row sharding across
 * GPUs); pass 0, n for everything.
 */
S2A_EXPORT int s2a_box_iou_rotated(const float* boxes1, int64_t n, const float* boxes2, int64_t m,
                                   int64_t batch, float* out, int64_t ld_out, int64_t row_begin,
                                   int64_t row_end, int flags, void* stream);
/* The same matrix, sharded by ROW TILES for several GPUs (SURVEY.md 8e: the anchor x GT matrix shards by anchor
 * rows): the n rows are cut into tiles of tile_rows (a multiple of 32, <= 256; 0 = 256) and this call computes the
 * tiles tile_first, tile_first + tile_step, tile_first + 2 tile_step, ... -- rank r of w ranks passes (r, w), which
 * deals the tiles out cyclically (contiguous row blocks would hand one rank all the large P5-P7 anchors, whose pairs
 * mostly reach the clipper).  compact = 0: rows are written at their global index of a [batch, n, ld_out] output;
 * compact != 0: out holds only this call's tiles, packed in order ([batch, ntiles_mine * tile_rows, ld_out]).
 * out_batch_stride (elements) = 0 selects the dense value of either layout. */
S2A_EXPORT int s2a_box_iou_rotated_tiles(const float* boxes1, int64_t n, const float* boxes2, int64_t m,
                                         int64_t batch, float* out, int64_t ld_out, int64_t out_batch_stride,
                                         int tile_rows, int tile_first, int tile_step, int compact, int flags,
                                         void* stream);

/* ---------------------------------------------------------------------------------------------
 * nms_rotated / ml_nms_rotated -- replace nms_rotated_cuda()
 *   reference: utils/nms_rotated/src/nms_rotated_cuda.cu:72-132 (host), :13-69 (kernel)
 *              utils/ml_nms_rotated/src/nms_rotated_cuda.cu:74-137, :13-71 (label-aware twin)
 * dets: n rows of 5 fp32 (x, y, w, h, theta), row stride det_stride elements (5 for a packed
 * tensor, 6 for the reference wrapper's dets[:, :5] view); scores: n fp32, stride score_stride;
 * labels: n fp32 or NULL (NULL = class-agnostic nms_rotated; non-NULL = ml_nms_rotated: boxes with
 * different labels never suppress each other).  Suppression predicate: IoU > iou_threshold, IoU
 * evaluated as IoU(earlier, later) in descending-score order (ties: lower index first).
 * keep_out: device int64[n]; the first *num_keep_out entries receive the ORIGINAL indices of the
 * kept boxes in descending-score order.  num_keep_out: device int32.  No host synchronisation
 * (the reference copies the whole mask to the host and sweeps it there).
 * workspace: device scratch of at least s2a_nms_rotated_workspace_bytes(n) bytes.
 */
S2A_EXPORT size_t s2a_nms_rotated_workspace_bytes(int64_t n);
S2A_EXPORT int s2a_nms_rotated(const float* dets, int64_t det_stride, const float* scores,
                               int64_t score_stride, const float* labels, int64_t n,
                               float iou_threshold, int64_t* keep_out, int32_t* num_keep_out,
                               void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * multiclass_nms_rotated -- replaces the Python routine of the same name
 *   reference: utils/bbox_nms_rotated.py:5-64
 * bboxes [n, 5] fp32, scores [n, num_classes] fp32 (post-sigmoid).  Candidates are the (box, class)
 * pairs with score > score_thr (strict) in row-major order; ml-NMS at iou_thr; if more than
 * max_per_img survive only the max_per_img best scores are kept.  Outputs (device):
 *   dets_out [max_out, 6] (x, y, w, h, theta, score) and labels_out [max_out] fp32, filled for the
 *   first *num_out rows in descending-score order; num_out int32; max_out = capacity of the output
 *   buffers (>= min(n*num_classes, max_per_img) to hold every possible result).
 * Sync-free and batched: `batch` images are processed by the same launches (image b reads
 * bboxes + b*n*5, scores + b*n*num_classes and writes row b of each output).
 * Sizes: n < 2^30 and n <= 819,200 boxes per image (the per-class sweep holds 16 bytes per 64 boxes
 * in shared memory, at most 200 KB), num_classes and batch <= 65535, and above 6,144 boxes per image
 * batch*num_classes*n < 2^31 - 256; larger sizes return S2A_ERR_UNSUPPORTED.  iou_thr must be >= 0
 * (S2A_ERR_UNSUPPORTED otherwise).
 * workspace: s2a_multiclass_nms_rotated_workspace_bytes(n, num_classes, batch) bytes, dominated by the
 * suppression mask of 8*batch*num_classes*n*ceil(n/64) bytes (for batch 8 and 15 classes: 0.68 GB
 * at n = 6,720, 7.1 GB at n = 21,824); the rest is 48*batch*num_classes*n + 32*batch*n bytes, plus
 * 16*batch*num_classes*n above 6,144 boxes per image (the sort keys).
 */
S2A_EXPORT size_t s2a_multiclass_nms_rotated_workspace_bytes(int64_t n, int64_t num_classes,
                                                             int64_t batch);
S2A_EXPORT int s2a_multiclass_nms_rotated(const float* bboxes, const float* scores, int64_t n,
                                          int64_t num_classes, int64_t batch, float score_thr,
                                          float iou_thr, int64_t max_per_img, float* dets_out,
                                          float* labels_out, int32_t* num_out, int64_t max_out,
                                          void* workspace, size_t workspace_bytes, void* stream);
/* The same NMS with the detection exchange of SURVEY.md 8e fused into its finaliser: instead of dets / labels /
 * counts, every kept detection is stored as an 8-float row (x, y, w, h, theta, score, label, 0: two 16-byte stores) into
 * the packed buffers dests[0 .. ndests-1], each [slots, max_out + 1, 8] fp32 and 16-byte aligned, at image slot slot0 + b; row max_out of a slot holds the
 * count in column 0.  With ndests = 1 this is the "pack" of the NCCL all-gather done by the kernel that produces the
 * detections; with ndests = world the destinations are the ranks' symmetric buffers (this rank's own and its peers'
 * NVLink-mapped pointers, <= 8) and the stores ARE the all-gather -- the caller only adds a barrier
 * (s2anet_b200/dist.py, DetectionExchange).  Rows past the count are unspecified.  Size limits and workspace as for
 * s2a_multiclass_nms_rotated. */
S2A_EXPORT int s2a_multiclass_nms_rotated_packed(const float* bboxes, const float* scores, int64_t n,
                                                 int64_t num_classes, int64_t batch, float score_thr,
                                                 float iou_thr, int64_t max_per_img, float* const* dests,
                                                 int ndests, int64_t slot0, int64_t max_out, void* workspace,
                                                 size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * ORN: active rotating filters and rotation-invariant pooling
 *   reference: models/orn/src/cuda/ActiveRotatingFilter_cuda.cu:19-46, 79-119 (arf_forward),
 *              :48-76, 122-163 (arf_backward); models/orn/src/vision.cpp:7-12 (exported names);
 *              models/orn/functions/rotation_invariant_pooling.py:19-27 (pooling)
 * weight [O, I, nOri, kH, kW]; indices uint8 [nOri*kH*kW, nRot] (1-based destination entry);
 * out [O*nRot, I*nOri, kH, kW].  dtype in {S2A_F32, S2A_BF16, S2A_F16} (pure data movement).
 */
S2A_EXPORT int s2a_arf_forward(const void* weight, const uint8_t* indices, void* out, int O, int I,
                               int nOri, int kH, int kW, int nRot, int dtype, void* stream);
S2A_EXPORT int s2a_arf_backward(const void* grad_out, const uint8_t* indices, void* grad_weight,
                                int O, int I, int nOri, int kH, int kW, int nRot, int dtype,
                                void* stream);
/* x [B, C, H, W] -> out [B, C/nOri, H, W]: max over each group of nOri consecutive channels. */
S2A_EXPORT int s2a_ri_pool_forward(const void* x, void* out, int64_t B, int64_t C, int64_t HW,
                                   int nOri, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Deformable convolution forward -- replaces deform_conv_forward_cuda()
 *   reference: models/dcn/src/deform_conv_cuda.cpp:152-260 (host), models/dcn/src/
 *              deform_conv_cuda_kernel.cu:189-242, 83-114 (im2col + bilinear)
 * x [B, C, H, W], offset [B, dgroups*2*kH*kW, Ho, Wo], weight [Co, C/groups, kH, kW],
 * out [B, Co, Ho, Wo]; all NCHW contiguous fp32.  One fused pass: sampling, contraction and the
 * NCHW store happen in a single kernel (no column buffer, no output transpose).
 * relu != 0 applies max(.,0) in the epilogue (AlignConv).
 */
S2A_EXPORT int s2a_deform_conv_forward_f32(const float* x, const float* offset,
                                           const float* weight, float* out, int B, int C, int H,
                                           int W, int Co, int kH, int kW, int strideH, int strideW,
                                           int padH, int padW, int dilH, int dilW, int groups,
                                           int dgroups, int relu, void* stream);

/* ---------------------------------------------------------------------------------------------
 * AlignConv forward -- replaces AlignConv.forward (offset generation + DeformConv + ReLU)
 *   reference: models/alignconv.py:29-98; models/dcn/deform_conv.py:15-71
 * x [B, C, H, W] NCHW fp32, anchors [B, H, W, 5] fp32 (image pixels, theta rad), weight
 * [Co, C, 3, 3] fp32, out [B, Co, H, W] fp32.  The 18-channel offset field is never materialised:
 * sample positions are derived from the anchors inside the kernel.
 */
S2A_EXPORT int s2a_alignconv_forward_f32(const float* x, const float* anchors, const float* weight,
                                         float* out, int B, int C, int H, int W, int Co,
                                         float stride, void* stream);

/* ORConv2d forward (3x3, pad 1, stride 1) -- replaces ORConv2d.forward = conv2d(x, ARF(w), bias)
 *   reference: models/orn/modules/ORConv.py:77-82
 * x [B, I*nOri, H, W] fp32; weight [O, I, nOri, 3, 3]; indices uint8 [nOri*9, nRot]; bias
 * [O*nRot] or NULL; out [B, O*nRot, H, W]; pooled (optional, may be NULL) [B, O*nRot/nRot... ]
 * = RotationInvariantPooling over groups of nRot consecutive output channels, produced by the
 * same kernel's epilogue. */
S2A_EXPORT int s2a_orconv_forward_f32(const float* x, const float* weight, const uint8_t* indices,
                                      const float* bias, float* out, float* pooled, int B, int H,
                                      int W, int O, int I, int nOri, int nRot, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core (tcgen05) path: bf16 / fp16 activations in channels-last (NHWC) layout, fp32
 * accumulation in TMEM.  Same reference interfaces as the _f32 entries above (AlignConv.forward,
 * models/alignconv.py:88-98; ORConv2d.forward + RotationInvariantPooling, models/orn/modules/
 * ORConv.py:77-82, models/orn/functions/rotation_invariant_pooling.py:19-27), for the half-precision
 * inference path of val.py (:126, :196, :246).
 *
 * s2a_conv_pack_weight: [Co, C, 3, 3] weights (f32/bf16/f16) -> packed [Co][9*C] 16-bit in
 * (64-channel block, tap, channel) K order.  With arf_indices != NULL the input is an ORConv bank
 * [O, I, nOri, 3, 3] (Co = O*nRot, C = I*nOri) and the ARF rotation (ActiveRotatingFilter_cuda.cu
 * :19-46) is applied while packing.  Needs C % 64 == 0.
 * x [B, H, W, C], anchors [B, H, W, 5] fp32, out [B, H, W, Co], pooled [B, H, W, Co/8] (may be NULL),
 * bias fp32 [Co] (may be NULL); dtype in {S2A_BF16, S2A_F16}; Co % 32 == 0, Co <= 256.
 */
S2A_EXPORT int s2a_conv_pack_weight(const void* weight, int in_dtype, const uint8_t* arf_indices,
                                    void* packed, int out_dtype, int Co, int C, int nOri, int nRot,
                                    void* stream);
S2A_EXPORT int s2a_alignconv_forward_tc(const void* x, const float* anchors,
                                        const void* packed_weight, void* out, int B, int C, int H,
                                        int W, int Co, float stride, int dtype, void* stream);
/* Generic deformable convolution on the same tcgen05 kernel: the 16-bit route of `deform_conv_forward_cuda`
 * (reference: models/dcn/src/deform_conv_cuda.cpp:152-260 with scalar_t = half, dispatched at
 * deform_conv_cuda_kernel.cu:258; models/dcn/deform_conv.py:45-70 casts offset and weight to the input dtype).
 * 3x3, stride 1, padding 1, dilation 1, groups 1, deformable_groups 1, C % 64 == 0, C_out % 32 == 0 <= 256.
 * x / out are NHWC 16-bit like s2a_alignconv_forward_tc; `offsets` is the reference's [B, 18, H, W] tensor
 * ((dy, dx) per tap, NCHW) in fp32 (offsets_dtype = S2A_F32) or in the activations' dtype; `packed_weight` comes
 * from s2a_conv_pack_weight (no ARF map).  round_positions != 0 rounds the sampling position and every bilinear
 * weight operation to the 16-bit type exactly as the reference's `scalar_t` arithmetic does (:94-110, :223-224);
 * 0 keeps them in fp32 (more accurate; what AlignConv's fused path does).  relu != 0 fuses a ReLU. */
S2A_EXPORT int s2a_deform_conv_forward_tc(const void* x, const void* offsets, int offsets_dtype,
                                          const void* packed_weight, void* out, int B, int C, int H, int W,
                                          int Co, int relu, int round_positions, int dtype, void* stream);
/* Deformable-conv backward w.r.t. the input (and, optionally, the offsets) on the tcgen05 kernel, 16-bit tensors:
 * replaces deform_conv_backward_input_cuda (models/dcn/src/deform_conv_cuda.cpp:262-373; kernels
 * deformable_col2im(_coord)_gpu_kernel, deform_conv_cuda_kernel.cu:278-435) for S2ANet's geometry (3x3, stride / pad /
 * dilation 1, one group).  Per tap: col_grad = grad_out x W_t^T as a 1x1 implicit GEMM (grad_out NHWC [B,H,W,Co],
 * wd [9][C][Co]: wd[t][c][co] = weight[co][c][t]) whose accumulator tile is scattered from tensor memory with the
 * bilinear weights of (pixel, tap) into grad_input (fp32 NHWC [B,H,W,C], ACCUMULATED -- zero it first, as the
 * reference's caller does, deform_conv.py:88-89) -- no column buffer, no library GEMM.  grad_offset (fp32
 * [B,18,H,W], accumulated; needs x NHWC 16-bit) may be NULL.  Nine launches. */
S2A_EXPORT int s2a_deform_conv_dgrad_tc(const void* grad_out, const void* offsets, int offsets_dtype,
                                        const void* wd, const void* x, float* grad_input,
                                        float* grad_offset, int B, int C, int H, int W, int Co, int dtype,
                                        void* stream);
/* Deformable-conv backward w.r.t. the weight on tcgen05, 16-bit tensors: replaces deform_conv_backward_parameters_cuda
 * (models/dcn/src/deform_conv_cuda.cpp:376-489: deformable_im2col into a column buffer + addmm_) for S2ANet's geometry
 * (3x3, stride / pad / dilation 1, one group; C and C_out in {128, 256}).  dW[co, c, tap] = sum over pixels of
 * grad_out[pixel, co] * sample[pixel, tap, c]: the contraction runs over pixels, both operands are MN-major
 * shared-memory tiles (grad_out NHWC via TMA; the bilinear samples built by the producer warps), the C_out x C fp32
 * accumulator of a tap lives in tensor memory across all pixel tiles of a CTA.  grad_weight_t is fp32 [9][C_out][C]
 * (tap-major; the caller permutes it to [C_out, C, 3, 3]) and is ACCUMULATED.  x, grad_out NHWC 16-bit. */
S2A_EXPORT int s2a_deform_conv_wgrad_tc(const void* x, const void* offsets, int offsets_dtype,
                                        const void* grad_out, float* grad_weight_t, int B, int C, int H, int W,
                                        int Co, int dtype, void* stream);
/* fp32 tensors on the tensor cores (3 x TF32 split, ~21 mantissa bits per product: inside the fp32 parity bar): the fast
 * route of the fp32 entries above for 3x3 / stride 1 / pad 1 / one group, C %% 32 == 0, C_out %% 32 == 0 <= 256.
 * s2a_conv_pack_weight_tf32: weight [Co][C][3][3] fp32 (or the ORConv bank through the ARF map, as
 * s2a_conv_pack_weight) -> two fp32 planes [Co][9*C], K order (tap, channel).  s2a_conv_forward_tf32x3: x NHWC fp32
 * [B,H,W,C]; mode 0: aux = anchors [B,H,W,5] (AlignConv, alignconv.py:29-98), mode 1: aux = offsets [B,18,H,W]
 * (deform_conv_forward_cuda), mode 2: regular grid (ORConv2d / conv2d, aux ignored); out NCHW fp32 [B,Co,H,W] (the
 * reference's layout), pooled [B,Co/8,H,W] or NULL; bias [Co] or NULL; relu != 0 fuses the ReLU. */
S2A_EXPORT int s2a_conv_pack_weight_tf32(const float* weight, const uint8_t* arf_indices, float* packed_hi,
                                         float* packed_lo, int Co, int C, int nOri, int nRot, void* stream);
S2A_EXPORT int s2a_conv_forward_tf32x3(const float* x, const float* aux, int mode, const float* packed_hi,
                                       const float* packed_lo, const float* bias, float* out, float* pooled,
                                       int B, int C, int H, int W, int Co, float stride, int relu, void* stream);
S2A_EXPORT int s2a_orconv_forward_tc(const void* x, const void* packed_weight, const float* bias,
                                     void* out, void* pooled, int B, int C, int H, int W, int Co,
                                     int dtype, void* stream);
/* Multi-level forms: all FPN levels of a batch in ONE persistent launch (the reference loops over
 * levels in Python, models/head.py:265).  Arrays have nlevels (<= 8) entries; every level shares
 * B, C, Co, the packed weights (and bias); xs[l] is [B, Hs[l], Ws[l], C] etc. */
S2A_EXPORT int s2a_alignconv_forward_tc_multi(int nlevels, const void* const* xs,
                                              const float* const* anchors, const void* packed_weight,
                                              void* const* outs, const int* Hs, const int* Ws,
                                              const float* strides, int B, int C, int Co, int dtype,
                                              void* stream);
S2A_EXPORT int s2a_orconv_forward_tc_multi(int nlevels, const void* const* xs,
                                           const void* packed_weight, const float* bias,
                                           void* const* outs, void* const* pooleds, const int* Hs,
                                           const int* Ws, int B, int C, int Co, int dtype, void* stream);

/* Stock convolution layers of the head on the same tcgen05 kernel (context, SURVEY 8 "callers": the FAM / ODM
 * towers and prediction convs of S2ANetHead.forward_single, models/head.py:296-348, are nn.Conv2d (+ReLU) in the
 * reference; routing them through conv_tc_kernel<PLAIN> removes the cuDNN launches between the custom ops).
 * Square kernels of size 1 or 3, stride 1, padding ks/2, dilation 1, groups 1.
 * s2a_conv2d_pack_weight: [Co, C, ks, ks] (f32/bf16/f16) -> packed [Co_pad][ks*ks*Cp] 16-bit with
 * Co_pad = round_up(Co, 32), Cp = round_up(C, 64) (zero padded).
 * s2a_conv2d_forward_tc_multi: xs[l] [B, H_l, W_l, C] (C % 8 == 0), outs[l] [B, H_l, W_l, Co_pad], bias fp32
 * [Co_pad] or NULL, relu != 0 applies max(., 0); one persistent launch for all levels. */
S2A_EXPORT int s2a_conv2d_pack_weight(const void* weight, int in_dtype, void* packed, int out_dtype,
                                      int Co, int C, int ks, void* stream);
S2A_EXPORT int s2a_conv2d_forward_tc_multi(int nlevels, const void* const* xs,
                                           const void* packed_weight, const float* bias,
                                           void* const* outs, const int* Hs, const int* Ws, int B,
                                           int C, int Co_pad, int ks, int relu, int dtype,
                                           void* stream);
/* Two such convolutions of one shape class (same C, Co_pad, ks, relu, dtype, B; own inputs / weights / biases /
 * outputs) in one persistent launch -- e.g. the classification and the regression tower layer of the head
 * (models/head.py:296-348 runs them one after the other): levels [0, split) use packed_weight0 / bias0, levels
 * [split, nlevels) packed_weight1 / bias1; nlevels <= 16.  Fills the 74 CTA pairs better than two launches. */
S2A_EXPORT int s2a_conv2d_forward_tc_multi2(int nlevels, int split, const void* const* xs,
                                            const void* packed_weight0, const void* packed_weight1,
                                            const float* bias0, const float* bias1, void* const* outs,
                                            const int* Hs, const int* Ws, int B, int C, int Co_pad, int ks,
                                            int relu, int dtype, void* stream);
/* The FAM regression head -- a 1x1 conv with 5 output channels padded to Co_pad = 32 (packed by
 * s2a_conv2d_pack_weight), + bias, no ReLU -- with the anchor decode of s2a_fam_decode in its epilogue:
 * refined[l] [B, H_l, W_l, 5] fp32 is bit-identical to s2a_fam_decode(strides, anchor_scale, anchor_angle,
 * wh_ratio_clip) of the head's stored output, which is never written.  One launch for all levels. */
S2A_EXPORT int s2a_conv2d_forward_tc_fam_decode(int nlevels, const void* const* xs,
                                                const void* packed_weight, const float* bias,
                                                float* const* refined, const int* Hs, const int* Ws,
                                                const float* strides, int B, int C, int Co_pad,
                                                float anchor_scale, float anchor_angle,
                                                double wh_ratio_clip, int dtype, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Box decode stages of the head (SURVEY.md 8(f) rows 2-3), batched over all FPN levels and images:
 * s2a_fam_decode is one launch, s2a_select_decode three (keys grid-wide, one CTA per (level, image) for the
 * exact top-k, gather + decode grid-wide).
 *
 * s2a_fam_decode -- replaces fam_bbox_decode + gen_grid_anchors
 *   reference: models/head.py:27-52 (fam_bbox_decode, wh_ratio_clip=1e-6), models/anchors.py:75-126
 *              (one square anchor per location: centre s*i + (s-1)/2, w = h = anchor_scale*s,
 *              theta = anchor_angle), models/boxes.py:82-162 (delta2bbox_rotated), utils/general.py:925-930.
 * deltas[l]: fam_bbox_pred of level l, logical shape [B, 5, H, W] with element strides
 * delta_strides[4*l .. 4*l+3] (NCHW or channels_last), dtype in {S2A_F32, S2A_BF16, S2A_F16};
 * refined[l]: [B, H, W, 5] fp32 contiguous (x, y, w, h, theta) = the rotated anchors AlignConv consumes.
 *
 * s2a_select_decode -- replaces get_bboxes_single_img up to the NMS call
 *   reference: models/head.py:684-717: sigmoid, per-level top-`topk` by best class score (only on
 *              levels with more than `topk` locations), gather, concatenation over levels, final
 *              delta2bbox_rotated with wh_ratio_clip (default 16/1000, models/boxes.py:226).
 * cls[l] [B, C, H, W] logits and reg[l] [B, 5, H, W] deltas (strided, dtype as above), anchors[l]
 * [B, H*W, 5] fp32 (the refined anchors).  Outputs: bboxes_out [B, n_total, 5] fp32, scores_out
 * [B, n_total, C] fp32 (post-sigmoid, rounded through the input dtype like the reference's half
 * tensors), n_total = sum_l min(H*W, topk); index_out (optional, may be NULL) [B, n_total] int32 =
 * location y*W + x of each candidate inside its level.  Candidates of a top-k level are ordered by
 * descending best score, ties by ascending location (torch.topk leaves ties unspecified).
 */
S2A_EXPORT int s2a_fam_decode(int nlevels, const void* const* deltas, const int64_t* delta_strides,
                              float* const* refined, const int* Hs, const int* Ws,
                              const float* strides, int B, float anchor_scale, float anchor_angle,
                              double wh_ratio_clip, int dtype, void* stream);
S2A_EXPORT size_t s2a_select_decode_workspace_bytes(int nlevels, const int* Hs, const int* Ws, int B);
S2A_EXPORT int s2a_select_decode(int nlevels, const void* const* cls, const int64_t* cls_strides,
                                 const void* const* reg, const int64_t* reg_strides,
                                 const float* const* anchors, const int* Hs, const int* Ws, int B,
                                 int num_classes, int topk, double wh_ratio_clip, int dtype,
                                 float* bboxes_out, float* scores_out, int32_t* index_out,
                                 int64_t n_total, void* workspace, size_t workspace_bytes,
                                 void* stream);

/* ---------------------------------------------------------------------------------------------
 * Deformable convolution backward, sampling side (SURVEY.md 8(f) row 1) -- replace deformable_im2col,
 * deformable_col2im and deformable_col2im_coord
 *   reference: models/dcn/src/deform_conv_cuda_kernel.cu:189-275, :278-351, :353-435 as called by
 *              deform_conv_backward_input_cuda / deform_conv_backward_parameters_cuda
 *              (models/dcn/src/deform_conv_cuda.cpp:262-489)
 * fp32, NCHW contiguous.  columns / grad_columns: [B, C*kH*kW, Ho*Wo] with K index c*kH*kW + i*kW + j (the order of
 * weight.flatten(1)).  s2a_deform_col2im_f32 ACCUMULATES into grad_input [B,C,H,W] and grad_offset
 * [B, dgroups*2*kH*kW, Ho, Wo] (the caller zeroes them, deform_conv.py:88-89); either may be NULL.  The two dense
 * contractions around these kernels are library GEMMs issued by the host binding (s2anet_b200/dcn.py).
 */
S2A_EXPORT int s2a_deform_im2col_f32(const float* x, const float* offset, float* columns, int B, int C,
                                     int H, int W, int kH, int kW, int strideH, int strideW, int padH,
                                     int padW, int dilH, int dilW, int dgroups, void* stream);
S2A_EXPORT int s2a_deform_col2im_f32(const float* grad_columns, const float* x, const float* offset,
                                     float* grad_input, float* grad_offset, int B, int C, int H, int W,
                                     int kH, int kW, int strideH, int strideW, int padH, int padW,
                                     int dilH, int dilW, int dgroups, void* stream);

/* ---------------------------------------------------------------------------------------------
 * assign_labels -- fused max-IoU label assignment (SURVEY.md 8(f) row 4), batched over images
 *   reference: models/utils.py:33-147 (assign_labels: bbox_iou_rotated + range / invalid-anchor filters + row
 *              max/argmax + negative / positive rules + the per-GT loop), utils/metrics.py:85-107
 * anchors [batch, num_anchors, 5], gts [batch, max_gts, 5] fp32 contiguous; gt_counts int32 [batch] (number of
 * real GT rows per image) or NULL (= max_gts everywhere).  assign_out int64 [batch, num_anchors]:
 * -2 ignored, -1 negative, >= 0 index of the assigned GT -- the reference's assign_gt_ids.  The IoU matrix is
 * never materialised (two passes over 64 x 256 tiles; IoU values bit-identical to s2a_box_iou_rotated).
 * img_h / img_w: imgs_size of the reference (anchors outside become ignored when filter_invalid_anchors != 0);
 * requires pos_iou_thr > 0 and min_pos_iou_thr >= 0 (the reference defaults are 0.5 / 0.4 / 0).
 */
S2A_EXPORT size_t s2a_assign_labels_workspace_bytes(int64_t batch, int64_t num_anchors, int64_t max_gts);
S2A_EXPORT int s2a_assign_labels(const float* anchors, const float* gts, const int32_t* gt_counts,
                                 int64_t batch, int64_t num_anchors, int64_t max_gts, float img_h,
                                 float img_w, float pos_iou_thr, float neg_iou_thr,
                                 float min_pos_iou_thr, int gt_max_assign_all,
                                 int filter_invalid_anchors, int64_t* assign_out, void* workspace,
                                 size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * poly_nms -- DOTA result-merging NMS on quadrilaterals, fp64 (SURVEY.md 8(f) row 4, second half)
 *   reference: DOTA_devkit/ResultMerge_multi_process.py:62-123 (py_cpu_nms_poly_fast),
 *              DOTA_devkit/polyiou/csrc/polyiou.cpp:9-126 (iou_poly and its helpers)
 * dets: rows of det_stride >= 9 doubles (x0 y0 x1 y1 x2 y2 x3 y3 score).  A later (lower-score) row is dropped
 * when its value against a kept row is not <= thresh, where value = overlap ratio of the two axis-aligned
 * bounding boxes (area (dx + 1)(dy + 1), overlap without the + 1) if that is not > 0, else the polygon IoU.
 * keep_out int64 [n]: kept row indices in descending-score order (equal scores: input order);
 * num_keep_out int32.  Every fp64 operation is individually rounded in the reference's order.
 * s2a_poly_iou_pairs: out[i] = iou_poly(p[i], q[i]) for 8-double polygons (parity probe).
 */
S2A_EXPORT size_t s2a_poly_nms_workspace_bytes(int64_t n);
S2A_EXPORT int s2a_poly_nms(const double* dets, int64_t det_stride, int64_t n, double thresh,
                            int64_t* keep_out, int32_t* num_keep_out, void* workspace,
                            size_t workspace_bytes, void* stream);
S2A_EXPORT int s2a_poly_iou_pairs(const double* p, const double* q, int64_t n, double* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* S2A_B200_H_ */
