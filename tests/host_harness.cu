// tests/host_harness.cu -- runs the product's __host__ __device__ IoU routines
// (s2anet_b200/csrc/rbox_iou.cuh) on the CPU so that the very source the sm_100a kernels
// compile can be checked against the oracle without a GPU.  Test infrastructure only.
#include <cstdint>
#include "../s2anet_b200/csrc/rbox_iou.cuh"
#include "../s2anet_b200/csrc/poly_iou.cuh"

extern "C" {

// mode 0: classify + clip (what the NMS kernels do); modes 3 / 4: the IoU kernel's path (see below); mode 1: clip for every pair that passes the
// reference's own area early-out (no disjointness shortcut); mode 2: returns the class (0/1).
void hh_pairwise(const float* b1, int64_t n, const float* b2, int64_t m, float* out, int mode) {
  s2a::RBox* A = new s2a::RBox[n > 0 ? n : 1];
  s2a::RBox* B = new s2a::RBox[m > 0 ? m : 1];
  for (int64_t i = 0; i < n; ++i) s2a::rbox_prep(b1[5*i], b1[5*i+1], b1[5*i+2], b1[5*i+3], b1[5*i+4], A[i]);
  for (int64_t j = 0; j < m; ++j) s2a::rbox_prep(b2[5*j], b2[5*j+1], b2[5*j+2], b2[5*j+3], b2[5*j+4], B[j]);
  for (int64_t i = 0; i < n; ++i)
    for (int64_t j = 0; j < m; ++j) {
      float v;
      float scratch[16];
      if (mode == 0) v = s2a::rbox_iou(A[i], B[j]);
      else if (mode == 2) v = (float)s2a::rbox_classify(A[i], B[j]);
      else if (mode == 3) {          // what box_iou_rotated_kernel does: fast test -> full classify -> register clipper
        s2a::RFast fa, fb; s2a::RAng aa, ab;
        s2a::rbox_fast_of(A[i], fa, aa); s2a::rbox_fast_of(B[j], fb, ab);
        if (s2a::rbox_fast_zero(fa, aa, fb, ab) || s2a::rbox_classify(A[i], B[j]) == s2a::RB_ZERO) v = 0.0f;
        else v = s2a::rbox_iou_clip_fast(A[i], B[j], scratch, 1);
      } else if (mode == 4) {        // register clipper for every pair that passes the area early-out
        float a1 = A[i].w * A[i].h, a2 = B[j].w * B[j].h;
        v = ((double)a1 < 1e-14 || (double)a2 < 1e-14) ? 0.0f : s2a::rbox_iou_clip_fast(A[i], B[j], scratch, 1);
      }
      else {
        float a1 = A[i].w * A[i].h, a2 = B[j].w * B[j].h;
        v = ((double)a1 < 1e-14 || (double)a2 < 1e-14) ? 0.0f : s2a::rbox_iou_clip(A[i], B[j]);
      }
      out[i * m + j] = v;
    }
  delete[] A; delete[] B;
}

// the product's fp64 polygon IoU (DOTA result merging), pair by pair
void hh_poly_iou_pairs(const double* p, const double* q, int64_t n, double* out) {
  for (int64_t i = 0; i < n; ++i) out[i] = s2a::poly_iou(p + 8 * i, q + 8 * i);
}

// the NMS kernels' upper bound of the intersection area (never used for an IoU value, only to skip clips)
void hh_inter_upper_bound(const float* b1, int64_t n, const float* b2, int64_t m, float* out) {
  for (int64_t i = 0; i < n; ++i) {
    s2a::RBox A;
    s2a::rbox_prep(b1[5*i], b1[5*i+1], b1[5*i+2], b1[5*i+3], b1[5*i+4], A);
    for (int64_t j = 0; j < m; ++j) {
      s2a::RBox B;
      s2a::rbox_prep(b2[5*j], b2[5*j+1], b2[5*j+2], b2[5*j+3], b2[5*j+4], B);
      out[i * m + j] = s2a::rbox_inter_upper_bound(A, B);
    }
  }
}

// the NMS kernels' clip skip: 1 where the pair's IoU provably cannot exceed thr[i * m + j] (one threshold per pair)
void hh_nms_cannot_exceed(const float* b1, int64_t n, const float* b2, int64_t m, const float* thr, uint8_t* out) {
  for (int64_t i = 0; i < n; ++i) {
    s2a::RBox A;
    s2a::rbox_prep(b1[5*i], b1[5*i+1], b1[5*i+2], b1[5*i+3], b1[5*i+4], A);
    for (int64_t j = 0; j < m; ++j) {
      s2a::RBox B;
      s2a::rbox_prep(b2[5*j], b2[5*j+1], b2[5*j+2], b2[5*j+3], b2[5*j+4], B);
      out[i * m + j] = s2a::rbox_nms_cannot_exceed(A, B, thr[i * m + j]) ? 1 : 0;
    }
  }
}

}
