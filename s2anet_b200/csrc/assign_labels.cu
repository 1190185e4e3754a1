// assign_labels.cu -- fused max-IoU label assignment for rotated anchors (SURVEY.md 8(f) row 4), batched.
//
// Replaces (reference): assign_labels, models/utils.py:33-147 -- bbox_iou_rotated (a [M, N] matrix per image),
// the range / invalid-anchor filters (:85-100), row max / argmax (:115), negative and positive rules (:116-123),
// and the per-GT Python loop that gives every GT its best anchor(s) (:128-144).  Here the IoU matrix never
// exists: two passes over 64 x 256 tiles, each evaluating the pairs with the same staged
// classify / compact / clip scheme as box_iou_rotated.cu (bit-identical IoU values, so the equality test of
// pass 2 against the column maxima of pass 1 is exact):
//   pass 1: per-anchor best (IoU, first GT index) and per-GT best (IoU, first anchor index) -- the latter
//           through one 64-bit atomicMax per (tile, GT) on a packed key;
//   pass 2: every anchor that reaches a GT's maximum (> min_pos_iou_thr) takes that GT, later GTs winning
//           (the reference loops GTs in ascending order, :130-144), then the positive / negative rules.
// Pairs proven disjoint have IoU exactly 0 and take part in neither maximum that matters (a row maximum of 0
// only tells "negative" from "ignored", which the count of valid pairs decides).
#include <climits>

#include "common.cuh"
#include "rbox_iou.cuh"

namespace s2a {

constexpr int kAsgR = 64, kAsgC = 256, kAsgThreads = 256;

struct AssignParams {
  const float* anchors;      // [B, M, 5]
  const float* gts;          // [B, Nmax, 5]
  const int32_t* gt_counts;  // [B] or null (= Nmax everywhere)
  unsigned long long* col_best;   // [B, Nmax] packed (IoU bits << 32 | ~anchor index), zeroed before pass 1; ~0 = a NaN IoU
  unsigned long long* row_best;   // [B, M] packed (IoU bits + 1 << 32 | ~gt index); 0 = no positive IoU
  int32_t* row_bad;          // [B, M] number of (valid-anchor) pairs whose IoU fell outside [0, 1]; sign bit: a NaN IoU
  int64_t* assign;           // [B, M]
  long long M, Nmax;
  float img_w, img_h, pos_thr, neg_thr, min_pos_thr;
  int gt_max_assign_all, filter_invalid_anchors;
};

// models/utils.py:71-77
__device__ __forceinline__ bool anchor_inside(const float* a, float img_w, float img_h) {
  return a[0] >= 0.0f && a[1] >= 0.0f && a[0] <= img_w && a[1] <= img_h && a[2] < img_w && a[3] < img_h;
}

// the general 24-point clipper (thread-local arrays), out of line: reached by degenerate pairs only
__device__ __noinline__ float asg_clip_general(const RBox& A, const RBox& B) { return rbox_iou_clip(A, B); }

template <int PASS>
__global__ void __launch_bounds__(kAsgThreads) assign_labels_kernel(const AssignParams p) {
  extern __shared__ float s_pts[];                   // 16 x kAsgThreads floats: candidate columns of the register clipper
  __shared__ RBox s_row[kAsgR];
  __shared__ RBox s_col[kAsgC];
  __shared__ __align__(16) uint16_t s_list[kAsgR * kAsgC];
  float* s_raw = reinterpret_cast<float*>(s_list);
  __shared__ unsigned long long s_rbest[kAsgR];      // pass 1: best (IoU, first GT) of each row over all column tiles
  __shared__ unsigned long long s_cbest[kAsgC];      // pass 1: best (IoU, first anchor) of each column inside this tile
  __shared__ int s_rbad[kAsgR];                      // pass 1: out-of-range pairs per row
  __shared__ int s_match[kAsgR];                     // pass 2: largest GT index whose maximum this anchor reaches
  __shared__ unsigned char s_rvalid[kAsgR];
  __shared__ int s_count;

  const int tid = threadIdx.x;
  const unsigned lane = tid & 31;
  const long long b = blockIdx.y;
  const long long row0 = (long long)blockIdx.x * kAsgR;
  const int nr = (int)min((long long)kAsgR, p.M - row0);
  const int ngt = p.gt_counts ? min(max(p.gt_counts[b], 0), (int)p.Nmax) : (int)p.Nmax;
  const float* g1 = p.anchors + (b * p.M + row0) * 5;

  for (int i = tid; i < kAsgR; i += kAsgThreads) { s_rbest[i] = 0ull; s_rbad[i] = 0; s_match[i] = -1; }
  for (int i = tid; i < nr * 5; i += kAsgThreads) s_raw[i] = g1[i];
  __syncthreads();
  if (tid < nr) {
    const float* r = s_raw + tid * 5;
    s_rvalid[tid] = !p.filter_invalid_anchors || anchor_inside(r, p.img_w, p.img_h);
    rbox_prep(r[0], r[1], r[2], r[3], r[4], s_row[tid]);
  }
  __syncthreads();

  for (int col0 = 0; col0 < ngt; col0 += kAsgC) {
    const int nc = min(kAsgC, ngt - col0);
    const float* g2 = p.gts + (b * p.Nmax + col0) * 5;
    __syncthreads();                                  // previous tile's list / column state fully consumed
    for (int i = tid; i < nc * 5; i += kAsgThreads) s_raw[i] = g2[i];
    if (tid == 0) s_count = 0;
    s_cbest[tid] = 0ull;
    __syncthreads();
    RBox cb;
    const bool col_ok = tid < nc;
    if (col_ok) {
      const float* r = s_raw + tid * 5;
      rbox_prep(r[0], r[1], r[2], r[3], r[4], cb);
      s_col[tid] = cb;
    }
    __syncthreads();                                  // s_raw (aliases s_list) is dead from here on

    // fast classification: thread = column, walking the rows; invalid anchors are skipped altogether
    // (their IoUs are overwritten with -0.5 in the reference, models/utils.py:100)
#pragma unroll 4
    for (int r = 0; r < nr; ++r) {
      const bool maybe = col_ok && s_rvalid[r] && rbox_classify_fast(s_row[r], cb) != RB_ZERO;
      const unsigned bal = __ballot_sync(0xffffffffu, maybe);
      if (bal) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_count, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (maybe) s_list[base + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)(r * kAsgC + tid);
      }
    }
    __syncthreads();
    // full classification, compacting in place (see box_iou_rotated.cu, phase 3)
    const int cnt_maybe = s_count;
    __syncthreads();
    if (tid == 0) s_count = 0;
    __syncthreads();
    for (int k0 = 0; k0 < cnt_maybe; k0 += kAsgThreads) {
      const int k = k0 + tid;
      bool clip = false;
      int pr = 0;
      if (k < cnt_maybe) {
        pr = s_list[k];
        clip = rbox_classify(s_row[pr >> 8], s_col[pr & (kAsgC - 1)]) != RB_ZERO;
      }
      __syncthreads();
      const unsigned bal = __ballot_sync(0xffffffffu, clip);
      if (bal) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_count, __popc(bal));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (clip) s_list[base + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)pr;
      }
    }
    __syncthreads();
    // clip the survivors and feed the reductions
    const int cnt = s_count;
    for (int k = tid; k < cnt; k += kAsgThreads) {
      const int pr = s_list[k];
      const int r = pr >> 8, c = pr & (kAsgC - 1);
      bool ok;
      float v = rbox_iou_clip_try(s_row[r], s_col[c], s_pts + tid, kAsgThreads, ok);
      if (!ok) v = asg_clip_general(s_row[r], s_col[c]);
      if (v != v) {
        // A NaN IoU passes the range filter (models/utils.py:89-96) and propagates through torch.max: the row maximum
        // is NaN (neither negative nor positive), and so is the GT's maximum (no anchor is forced onto it).  Marked by
        // the sign bit of the row's count, and by a column key above every IoU key.
        if (PASS == 1) { atomicOr(&s_rbad[r], INT_MIN); atomicMax(&s_cbest[c], ~0ull); }
        continue;
      }
      if (!(v >= 0.0f && v <= 1.0f)) {                  // models/utils.py:89-96: out-of-range IoUs become -0.5
        if (PASS == 1) atomicAdd(&s_rbad[r], 1);
        continue;
      }
      if (v == 0.0f) continue;                          // a zero takes part in no maximum that matters
      const unsigned bits = __float_as_uint(v);         // positive floats order like their bit patterns
      if (PASS == 1) {
        atomicMax(&s_rbest[r], ((unsigned long long)(bits + 1u) << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)(col0 + c)));
        atomicMax(&s_cbest[c], ((unsigned long long)bits << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)(row0 + r)));
      } else if (v > p.min_pos_thr) {
        const unsigned long long best = p.col_best[b * p.Nmax + col0 + c];
        const bool hit = p.gt_max_assign_all ? (unsigned)(best >> 32) == bits
                                             : best == (((unsigned long long)bits << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)(row0 + r)));
        if (hit) atomicMax(&s_match[r], col0 + c);      // GTs are visited in ascending order: the last one wins
      }
    }
    __syncthreads();
    if (PASS == 1 && tid < nc && s_cbest[tid] != 0ull) atomicMax(&p.col_best[b * p.Nmax + col0 + tid], s_cbest[tid]);
  }
  __syncthreads();

  if (tid < nr) {
    const long long a = b * p.M + row0 + tid;
    if (PASS == 1) {
      p.row_best[a] = s_rbest[tid];
      p.row_bad[a] = s_rbad[tid];
    } else {
      // models/utils.py:62-144 for one anchor
      long long res = -2;                                // ignored
      if (s_rvalid[tid]) {
        if (ngt == 0) {
          res = -1;                                      // :79-86: no GT at all -> every valid anchor is negative
        } else {
          const int bad = p.row_bad[a];
          if (bad >= 0) {                                // (< 0: a NaN IoU in the row, its maximum is NaN: ignored)
            const unsigned long long rb = p.row_best[a];
            const int nvalid = ngt - bad;                // pairs with an IoU in [0, 1]
            // row maximum: the best positive IoU, else 0 if any pair is valid, else -0.5
            const float mx = rb ? __uint_as_float((unsigned)(rb >> 32) - 1u) : (nvalid > 0 ? 0.0f : -0.5f);
            if (mx >= 0.0f && mx < p.neg_thr) res = -1;  // :116
            if (mx >= p.pos_thr) {                       // :122-123 (argmax = first index of the maximum)
              if (rb) res = (long long)(0xFFFFFFFFu - (unsigned)(rb & 0xFFFFFFFFull));
              else {                                     // maximum 0 reached the positive threshold (pos_thr <= 0): first valid pair
                res = 0;
              }
            }
          }
          if (s_match[tid] >= 0) res = s_match[tid];     // :130-144
        }
      }
      p.assign[a] = res;
    }
  }
}

}  // namespace s2a

extern "C" size_t s2a_assign_labels_workspace_bytes(int64_t batch, int64_t num_anchors, int64_t max_gts) {
  if (batch < 0 || num_anchors < 0 || max_gts < 0) return 0;
  return (size_t)batch * ((size_t)max_gts * 8 + (size_t)num_anchors * 12) + 256;
}

extern "C" int s2a_assign_labels(const float* anchors, const float* gts, const int32_t* gt_counts, int64_t batch,
                                 int64_t num_anchors, int64_t max_gts, float img_h, float img_w, float pos_iou_thr,
                                 float neg_iou_thr, float min_pos_iou_thr, int gt_max_assign_all,
                                 int filter_invalid_anchors, int64_t* assign_out, void* workspace, size_t workspace_bytes,
                                 void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(batch >= 0 && num_anchors >= 0 && max_gts >= 0, "assign_labels: negative size");
  S2A_CHECK_ARG(batch <= 65535, "assign_labels: batch must be <= 65535");
  S2A_CHECK_ARG(num_anchors < (1ll << 31) && max_gts < (1ll << 31), "assign_labels: too many boxes");
  S2A_CHECK_ARG(min_pos_iou_thr >= 0.0f, "assign_labels: min_pos_iou_thr must be >= 0 (got %g)", (double)min_pos_iou_thr);
  S2A_CHECK_ARG(pos_iou_thr > 0.0f, "assign_labels: pos_iou_thr must be > 0 (got %g)", (double)pos_iou_thr);
  if (batch == 0 || num_anchors == 0) return S2A_OK;
  S2A_CHECK_ARG(anchors && assign_out && (gts || max_gts == 0), "assign_labels: null pointer");
  if (!workspace || workspace_bytes < s2a_assign_labels_workspace_bytes(batch, num_anchors, max_gts)) {
    set_error("assign_labels: workspace too small");
    return S2A_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  AssignParams p{};
  p.anchors = anchors; p.gts = gts; p.gt_counts = gt_counts;
  uint8_t* w = reinterpret_cast<uint8_t*>(workspace);
  p.col_best = reinterpret_cast<unsigned long long*>(w);
  p.row_best = p.col_best + batch * max_gts;
  p.row_bad = reinterpret_cast<int32_t*>(p.row_best + batch * num_anchors);
  p.assign = assign_out;
  p.M = num_anchors; p.Nmax = max_gts;
  p.img_w = img_w; p.img_h = img_h; p.pos_thr = pos_iou_thr; p.neg_thr = neg_iou_thr; p.min_pos_thr = min_pos_iou_thr;
  p.gt_max_assign_all = gt_max_assign_all; p.filter_invalid_anchors = filter_invalid_anchors;
  if (max_gts > 0) S2A_CUDA_OK(cudaMemsetAsync(p.col_best, 0, (size_t)batch * max_gts * 8, st));
  dim3 grid((unsigned)ceil_div(num_anchors, kAsgR), (unsigned)batch);
  constexpr size_t kPtsBytes = sizeof(float) * 16 * kAsgThreads;     // dynamic, on top of ~45 KB of static shared memory
  S2A_CUDA_OK(cudaFuncSetAttribute(assign_labels_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPtsBytes));
  S2A_CUDA_OK(cudaFuncSetAttribute(assign_labels_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPtsBytes));
  assign_labels_kernel<1><<<grid, kAsgThreads, kPtsBytes, st>>>(p);
  S2A_LAUNCH_OK("assign_labels_kernel<1>");
  assign_labels_kernel<2><<<grid, kAsgThreads, kPtsBytes, st>>>(p);
  S2A_LAUNCH_OK("assign_labels_kernel<2>");
  return S2A_OK;
}
