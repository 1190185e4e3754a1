// rbox_iou.cuh -- rotated-box IoU device routines shared by box_iou_rotated, nms_rotated and
// ml_nms_rotated (sm_100a).
//
// Semantics follow the reference's CUDA build of single_box_iou_rotated
// (reference: utils/box_iou_rotated/src/box_iou_rotated_utils.h:55-375, __CUDACC__ branch of the
// hull sort at :209-226), re-organised for the GPU:
//   * per-box work (double-precision sin/cos, :62-64) is hoisted out of the pair loop ("RBox");
//   * a conservative circumscribed-circle test classifies most pairs as exactly-zero without
//     running the clipper (rbox_classify);
//   * the clipper keeps ONE 24-point array (the hull is built in place, squared distances are
//     recomputed instead of stored -- bit-identical because the reference permutes dist[] together
//     with the points);
//   * every multiply/add is an individually rounded IEEE fp32 operation (__fmul_rn & co., never
//     contracted into FMA), and every double-precision epsilon test of the reference is replaced
//     by the exactly equivalent fp32 comparison, so the result is bit-identical to the CPU oracle
//     (oracle/s2a_oracle.c, built with -ffp-contract=off) given the same per-box sin/cos.
//
// All functions are __host__ __device__ so that tests/host_harness.cu can run the very same
// source on the CPU against the oracle.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDA_ARCH__)
#define RB_MUL(a, b) __fmul_rn((a), (b))
#define RB_ADD(a, b) __fadd_rn((a), (b))
#define RB_SUB(a, b) __fsub_rn((a), (b))
#define RB_DIV(a, b) __fdiv_rn((a), (b))
#else   // host pass: compiled with -ffp-contract=off
#define RB_MUL(a, b) ((a) * (b))
#define RB_ADD(a, b) ((a) + (b))
#define RB_SUB(a, b) ((a) - (b))
#define RB_DIV(a, b) ((a) / (b))
#endif
#define RB_HD __host__ __device__ __forceinline__

namespace s2a {

// fp32 neighbours of the reference's double literals (none is representable in fp32, so
// "x < L" and "x <= L" are both "x <= lo(L)", and "x > L" is "x >= hi(L)").
#define RB_LO_1E14 __int_as_float_c(0x283424dc)
RB_HD float rb_bits(uint32_t u) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  union { uint32_t u; float f; } c; c.u = u; return c.f;
#endif
}
#undef RB_LO_1E14
#define RB_LO_1E14 rb_bits(0x283424dcu)   // largest fp32 < 1e-14
#define RB_LO_1E6  rb_bits(0x358637bdu)   // largest fp32 < 1e-6
#define RB_HI_1E6  rb_bits(0x358637beu)   // smallest fp32 > 1e-6
#define RB_HI_1E8  rb_bits(0x322bcc78u)   // smallest fp32 > 1e-8

// Per-box precomputation.  32 bytes -> two float4 loads.
struct __align__(16) RBox {
  float x, y, w, h;      // centre (unshifted), size
  float c2, s2;          // (float)cos(theta)*0.5f, (float)sin(theta)*0.5f   (reference :63-64)
  float r;               // >= half diagonal (circumscribed-circle radius), for the reject test
  float mn;              // min(|w|, |h|)
};

RB_HD void rbox_prep(float x, float y, float w, float h, float a, RBox& o) {
  o.x = x; o.y = y; o.w = w; o.h = h;
  double th = (double)a;
  o.c2 = RB_MUL((float)cos(th), 0.5f);
  o.s2 = RB_MUL((float)sin(th), 0.5f);
  o.r = 0.5f * sqrtf(w * w + h * h);
  o.mn = fminf(fabsf(w), fabsf(h));
}

// Pair classification.
//   RB_ZERO : the reference returns exactly +0.0f for this pair, either through its own area
//             early-out (:354-358) or because the boxes are provably disjoint (no candidate point
//             can be produced, so inter = 0 and iou = 0/(a1+a2) = 0).
//   RB_CLIP : run the clipper.
// Disjointness is established by a circumscribed-circle test (1 % margin) and, for the pairs that
// fail it, a separating-axis test over the four edge normals (margin 4e-3 of the pair's extent).
// The shortcut is only TAKEN when it is numerically safe to predict the reference's answer:
//   * no box side below 2e-3 of the extent (vertex rounding is ~2.4e-7 of the extent, so edge
//     directions are then accurate to ~1e-4 rad), and
//   * either no edge pair within ~0.6 degrees of parallel (|sin 2dT| > 0.02: every edge-pair
//     determinant is well conditioned), or -- for near-parallel / near-perpendicular boxes -- every
//     pair of parallel edges is at least 0.1 extent apart perpendicular to itself, which forces the
//     reference's |t1|, |t2| far above 1 whatever the noisy determinant is.  Near-parallel AND
//     near-collinear edges (boxes shifted along a shared edge line) are where the reference's t1/t2
//     are ill-conditioned; its answer there is reproduced by the clipper, never predicted.
// NaN/Inf inputs fail the comparisons and fall through to RB_CLIP.  See DESIGN.md "IoU reject test".

// Sliver guard (why a side may be as short as 2.5e-4 of the pair's extent).  Vertex coordinates carry an absolute
// rounding error eps_v <= 2^-22 * ext (ext = |dx| + |dy| + r1 + r2 bounds every coordinate after the centre shift), so
// an edge of length L has a direction error <= 5e-7 * ext / L: 2e-3 rad at L = 2.5e-4 * ext, a fifth of the 0.01 rad
// every edge pair keeps from parallel under the angle test -- the determinants stay well conditioned and a computed
// (t1, t2) in [0,1]^2 would put a common point within 3 * 2^-22 * ext / |sin phi| < 1e-4 * ext of both segments,
// impossible when they are `gap` apart.  The vertex-in-box test (:131-166) of a point at distance >= gap violates
// one of its four inequalities by >= (gap / sqrt 2) * L against an evaluation error <= 5e-7 * ext^2 + 7e-7 * ext * L;
// with a 4x safety factor that needs  gap * L > 3e-6 * ext^2.  The fast test's 10 % circle margin gives
// gap > 0.039 * ext, so L > 2.5e-4 * ext suffices there; the full test states the product rule explicitly.
// (Round 1 required L > 2e-3 * ext, which sent every far-away pair with a < 4 px box side -- 57 % of all clipped
// pairs of BASELINE config 4 -- through the clipper for a result of exactly zero.)
#define RB_SLIVER 2.5e-4f
#define RB_GAPRULE 3e-6f

// Stage 1 (every pair, ~25 flops, no divergence): the common case "circles clearly apart (10 %), edges clearly
// not parallel, no sliver" -> exactly zero.  Everything else is RB_MAYBE and goes to stage 2.
// `ext` over-estimates the pair's extent with the L1 norm (conservative: margins only grow).
enum { RB_ZERO = 0, RB_CLIP = 1, RB_MAYBE = 2 };

RB_HD int rbox_classify_fast(const RBox& A, const RBox& B) {
  const float dx = B.x - A.x, dy = B.y - A.y;
  const float rs = A.r + B.r;
  const float sd = B.s2 * A.c2 - B.c2 * A.s2;        // sin(tB - tA)/4
  const float cd = A.c2 * B.c2 + A.s2 * B.s2;        // cos(tB - tA)/4
  const float ext = fabsf(dx) + fabsf(dy) + rs;
  const bool ok = (dx * dx + dy * dy > 1.21f * rs * rs) && (fabsf(sd * cd) > 0.000625f) &&
                  (fminf(A.mn, B.mn) > RB_SLIVER * ext);
  return ok ? RB_ZERO : RB_MAYBE;
}

// The same test on the 24-byte per-box summary the IoU kernel keeps for its all-pairs pass: (x, y, r, mn) and
// (sin 2t, cos 2t).  |sin 2(tB - tA)| > 0.02 is the angle condition above (|sd * cd| = |sin 2 dT| / 32).
struct __align__(16) RFast { float x, y, r, mn; };
struct __align__(8) RAng { float s2t, c2t; };
RB_HD void rbox_fast_of(const RBox& b, RFast& f, RAng& a) {
  f.x = b.x; f.y = b.y; f.r = b.r; f.mn = b.mn;
  a.s2t = 8.0f * b.s2 * b.c2;                        // 2 sin cos
  a.c2t = 4.0f * (b.c2 * b.c2 - b.s2 * b.s2);        // cos^2 - sin^2
}
RB_HD bool rbox_fast_zero(const RFast& A, const RAng& aA, const RFast& B, const RAng& aB) {
  const float dx = B.x - A.x, dy = B.y - A.y;
  const float rs = A.r + B.r;
  const float ext = fabsf(dx) + fabsf(dy) + rs;
  const float s2d = aB.s2t * aA.c2t - aB.c2t * aA.s2t;
  return (dx * dx + dy * dy > 1.21f * rs * rs) && (fabsf(s2d) > 0.02f) && (fminf(A.mn, B.mn) > RB_SLIVER * ext);
}

// Near-parallel (C >= S) or near-perpendicular pairs: every pair of parallel edge lines is more than g apart,
// measured through the centres in A's frame (B's half extents along A's axes; duA, dvA: the centre offset there).
RB_HD bool rbox_parallel_edges_apart(const RBox& A, const RBox& B, float duA, float dvA, float S, float C, float g) {
  const float wB = fabsf(B.w), hB = fabsf(B.h);
  const float bu = 0.5f * (C >= S ? wB : hB), bv = 0.5f * (C >= S ? hB : wB);
  const float au = 0.5f * fabsf(A.w), av = 0.5f * fabsf(A.h);
  const float gv = fminf(fminf(fabsf(dvA + bv - av), fabsf(dvA + bv + av)),
                         fminf(fabsf(dvA - bv - av), fabsf(dvA - bv + av)));
  const float gu = fminf(fminf(fabsf(duA + bu - au), fabsf(duA + bu + au)),
                         fminf(fabsf(duA - bu - au), fabsf(duA - bu + au)));
  return gv > g && gu > g;
}

RB_HD int rbox_classify(const RBox& A, const RBox& B) {
  float a1 = RB_MUL(A.w, A.h), a2 = RB_MUL(B.w, B.h);
  if (a1 <= RB_LO_1E14 || a2 <= RB_LO_1E14) return RB_ZERO;     // (double)area < 1e-14
  const float dx = B.x - A.x, dy = B.y - A.y;
  const float d2 = dx * dx + dy * dy;
  const float rs = A.r + B.r;
  const float ext = fabsf(dx) + fabsf(dy) + rs;
  // sin(tB - tA)/4 and cos(tB - tA)/4 from the half-scaled sin/cos
  const float sd = B.s2 * A.c2 - B.c2 * A.s2;
  const float cd = A.c2 * B.c2 + A.s2 * B.s2;
  const float S = 4.0f * fabsf(sd), C = 4.0f * fabsf(cd);
  const float wA = fabsf(A.w), hA = fabsf(A.h), wB = fabsf(B.w), hB = fabsf(B.h);
  // centre offset in A's frame and in B's frame
  const float duA = 2.0f * (dx * A.c2 + dy * A.s2), dvA = 2.0f * (dy * A.c2 - dx * A.s2);
  bool sep = d2 > 1.0201f * rs * rs;
  // lower bound of the distance between the boxes: circles |d| - rs = (d2 - rs^2) / (|d| + rs) >= (d2 - rs^2) / ext;
  // separating axis: the margin itself
  float gap = (d2 - rs * rs) / ext;
  if (!sep) {
    const float mg = 4e-3f * ext;
    gap = mg;
    const float duB = 2.0f * (dx * B.c2 + dy * B.s2), dvB = 2.0f * (dy * B.c2 - dx * B.s2);
    sep = (fabsf(duA) > 0.5f * (wA + wB * C + hB * S) + mg) || (fabsf(dvA) > 0.5f * (hA + wB * S + hB * C) + mg) ||
          (fabsf(duB) > 0.5f * (wB + wA * C + hA * S) + mg) || (fabsf(dvB) > 0.5f * (hB + wA * S + hA * C) + mg);
  }
  const float mnp = fminf(A.mn, B.mn);
  if (sep && mnp > RB_SLIVER * ext && gap * mnp > RB_GAPRULE * ext * ext) {
    // |sd*cd| = |sin(2 dT)|/32
    if (fabsf(sd * cd) > 0.000625f) return RB_ZERO;
    if (rbox_parallel_edges_apart(A, B, duA, dvA, S, C, 0.1f * ext)) return RB_ZERO;
  }
  return RB_CLIP;
}

// Upper bound of the intersection AREA of two boxes with positive sizes (used by the NMS kernels only, to skip clips
// that cannot reach the threshold; never used for an IoU VALUE).  In A's frame B lies inside its axis-aligned extent
// (half sizes eu, ev around (du, dv)); the overlap of that rectangle with A bounds the intersection; same from B's
// side; and the intersection cannot exceed either area.
RB_HD float rbox_inter_upper_bound(const RBox& A, const RBox& B) {
  const float dx = B.x - A.x, dy = B.y - A.y;
  const float sd = B.s2 * A.c2 - B.c2 * A.s2, cd = A.c2 * B.c2 + A.s2 * B.s2;      // sin, cos of (tB - tA), / 4
  const float S = 4.0f * fabsf(sd), C = 4.0f * fabsf(cd);
  const float duA = 2.0f * (dx * A.c2 + dy * A.s2), dvA = 2.0f * (dy * A.c2 - dx * A.s2);
  const float duB = 2.0f * (dx * B.c2 + dy * B.s2), dvB = 2.0f * (dy * B.c2 - dx * B.s2);
  const float euA = 0.5f * (B.w * C + B.h * S), evA = 0.5f * (B.w * S + B.h * C);  // B's half extents on A's axes
  const float euB = 0.5f * (A.w * C + A.h * S), evB = 0.5f * (A.w * S + A.h * C);
  const float ouA = fmaxf(0.0f, fminf(0.5f * A.w, duA + euA) - fmaxf(-0.5f * A.w, duA - euA));
  const float ovA = fmaxf(0.0f, fminf(0.5f * A.h, dvA + evA) - fmaxf(-0.5f * A.h, dvA - evA));
  const float ouB = fmaxf(0.0f, fminf(0.5f * B.w, euB - duB) - fmaxf(-0.5f * B.w, -duB - euB));
  const float ovB = fmaxf(0.0f, fminf(0.5f * B.h, evB - dvB) - fmaxf(-0.5f * B.h, -dvB - evB));
  return fminf(fminf(ouA * ovA, ouB * ovB), fminf(A.w * A.h, B.w * B.h));
}

// NMS clip skip: true only if the reference's IoU of the pair cannot exceed thr, so the suppression bit is 0 without
// clipping.  Geometrically, inter <= min(area) and union >= max(area), and IoU <= ub / (a1 + a2 - ub) with ub the
// bound above; both tests keep 0.1 % slack on each side for the reference's fp32 arithmetic.  That slack only holds
// where the reference computes the polygon well, so the shortcut takes conditions of the kind rbox_classify takes:
//   * Sliver guard.  Vertex coordinates are off by eps_v <= 2^-22 * ext.  A polygon vertex that moves by d along its
//     own edge changes the area by <= d * L * sin(phi) / 2, and a crossing at angle phi is off by ~eps_v / sin(phi)
//     along the edge, so every vertex and every fan triangle adds ~eps_v * L.  The intersection error is then about
//     4 eps_v times the smaller box's perimeter 2 (a + b) <= 4 a (sides a >= b).  An intersection that can reach thr
//     is >= thr * max area >= thr * a * b, so the relative error is <= 16 eps_v / (thr * b) = 3.8e-6 * ext / (thr * b).
//     Under thr * mn > 4e-3 * ext that is below 1e-3: within the slack.
//   * Angle or band.  Edges at least ~0.6 degrees from parallel (|sin 2dT| > 0.02) have well-conditioned crossings.
//     Near-parallel or near-perpendicular pairs must keep every pair of parallel edge lines more than RB_NMS_BAND * ext
//     apart.  On (near-)parallel lines the reference's determinant is rounding noise of ~8 eps_v * L, and its t1, t2
//     are gap * L over that noise: > 500 for a gap of 1e-3 * ext, so no false crossing point appears.  Lines that do
//     cross inside the segments with a gap of 1e-3 * ext at the centre meet at an angle >= 2e-3 * ext / L, where the
//     determinant is well conditioned again.  Boxes that share an edge line (same angle, same height, one nested in the
//     other along the axis) are the failing case without this: the reference's clipper returns values up to 1.0 for a
//     true IoU of 0.5, and such a pair must be clipped to reproduce them.
// NaN or non-positive sizes fail the comparisons: no skip.
#define RB_NMS_SLIVER 4e-3f
#define RB_NMS_BAND 1e-3f
RB_HD bool rbox_nms_cannot_exceed(const RBox& A, const RBox& B, float thr) {
  if (!(thr > 0.0f && A.w > 0.0f && A.h > 0.0f && B.w > 0.0f && B.h > 0.0f)) return false;
  const float dx = B.x - A.x, dy = B.y - A.y;
  const float ext = fabsf(dx) + fabsf(dy) + A.r + B.r;
  if (!(thr * fminf(A.mn, B.mn) > RB_NMS_SLIVER * ext)) return false;
  const float sd = B.s2 * A.c2 - B.c2 * A.s2, cd = A.c2 * B.c2 + A.s2 * B.s2;
  if (!(fabsf(sd * cd) > 0.000625f)) {                     // |sin 2dT| <= 0.02
    const float S = 4.0f * fabsf(sd), C = 4.0f * fabsf(cd);
    const float duA = 2.0f * (dx * A.c2 + dy * A.s2), dvA = 2.0f * (dy * A.c2 - dx * A.s2);
    if (!rbox_parallel_edges_apart(A, B, duA, dvA, S, C, RB_NMS_BAND * ext)) return false;
  }
  const float ar = A.w * A.h, ac = B.w * B.h;
  if (fminf(ar, ac) < 0.999f * thr * fmaxf(ar, ac)) return true;
  const float ub = 1.001f * rbox_inter_upper_bound(A, B);
  return ub < 0.999f * thr * (ar + ac - ub);
}

struct RPt { float x, y; };
RB_HD float rb_cross(float ax, float ay, float bx, float by) {   // A.x*B.y - B.x*A.y  (:50-53)
  return RB_SUB(RB_MUL(ax, by), RB_MUL(bx, ay));
}
RB_HD float rb_dot(float ax, float ay, float bx, float by) {     // A.x*B.x + A.y*B.y  (:45-48)
  return RB_ADD(RB_MUL(ax, bx), RB_MUL(ay, by));
}

// Vertices of a box whose centre is already shifted (:55-75).
RB_HD void rbox_vertices(float xc, float yc, const RBox& b, float (&px)[4], float (&py)[4]) {
  float sh = RB_MUL(b.s2, b.h), cw = RB_MUL(b.c2, b.w);
  float ch = RB_MUL(b.c2, b.h), sw = RB_MUL(b.s2, b.w);
  px[0] = RB_SUB(RB_SUB(xc, sh), cw);
  py[0] = RB_SUB(RB_ADD(yc, ch), sw);
  px[1] = RB_SUB(RB_ADD(xc, sh), cw);
  py[1] = RB_SUB(RB_SUB(yc, ch), sw);
  float tx = RB_MUL(2.0f, xc), ty = RB_MUL(2.0f, yc);
  px[2] = RB_SUB(tx, px[0]);
  py[2] = RB_SUB(ty, py[0]);
  px[3] = RB_SUB(tx, px[1]);
  py[3] = RB_SUB(ty, py[1]);
}

// Candidate points of the intersection polygon (:77-167): the edge-edge crossings in (i, j) order, then the vertices
// of box 1 inside box 2, then the vertices of box 2 inside box 1 -- up to 24.  Every point goes to `sink.put(k, x, y)`
// (k = its ordinal); returns the count.  One source for all clippers below, so they see bit-identical points.
template <class Sink>
RB_HD int rbox_candidates(const RBox& A, const RBox& B, Sink& sink) {
  // centre shift (:340-349): fp32 sum, exact halving, subtraction that is exact in double and
  // rounds once -- identical to the fp32 expression below for all finite pixel-scale inputs.
  float shx = RB_MUL(RB_ADD(A.x, B.x), 0.5f);
  float shy = RB_MUL(RB_ADD(A.y, B.y), 0.5f);
  float p1x[4], p1y[4], p2x[4], p2y[4];
  rbox_vertices(RB_SUB(A.x, shx), RB_SUB(A.y, shy), A, p1x, p1y);
  rbox_vertices(RB_SUB(B.x, shx), RB_SUB(B.y, shy), B, p2x, p2y);

  float e2x[4], e2y[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    e2x[j] = RB_SUB(p2x[(j + 1) & 3], p2x[j]);
    e2y[j] = RB_SUB(p2y[(j + 1) & 3], p2y[j]);
  }

  int n = 0;
  // Edge i of box 1 against the four edges of box 2.  The i loop is ROLLED (one copy of the 4-edge body instead of
  // four: the unrolled form made the clipper ~1,000 instructions long and the kernel instruction-cache bound) and
  // box 1's vertices rotate through named registers instead of being indexed, so nothing goes to local memory.
#if defined(__CUDA_ARCH__)
#pragma unroll 1
#endif
  for (int i = 0; i < 4; ++i) {
    const float ax = p1x[0], ay = p1y[0];
    const float e1x = RB_SUB(p1x[1], ax), e1y = RB_SUB(p1y[1], ay);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float det = rb_cross(e2x[j], e2y[j], e1x, e1y);
      const float dx = RB_SUB(p2x[j], ax), dy = RB_SUB(p2y[j], ay);
      const float n1 = rb_cross(e2x[j], e2y[j], dx, dy), n2 = rb_cross(e1x, e1y, dx, dy);
      // Exact pre-test: parallel edges (fabs(det) <= 1e-14, :103) give no point; a quotient whose magnitude clearly
      // exceeds 1, or that is clearly negative, cannot pass "0 <= t <= 1" after IEEE division either (the 1e-4 /
      // 1e-30 margins dwarf the half-ulp of the division and exclude the underflow-to-(-0) case), so the two
      // divisions are skipped for the ~3 of 4 edge pairs that are nowhere near crossing.  Every test is written
      // as a negated comparison so that NaNs fall through to the exact path, and the tests are combined without
      // short-circuit evaluation: ONE (rarely taken, divergent) branch per edge pair instead of four.
      const float ad = fabsf(det), lim = 1.0001f * ad, tiny = 1e-30f * ad;
      const bool neg = det < 0.0f;
      const bool plausible = !(ad <= RB_LO_1E14) & !(fabsf(n1) > lim) & !(fabsf(n2) > lim) &
                             !(((n1 < 0.0f) != neg) & (fabsf(n1) > tiny)) & !(((n2 < 0.0f) != neg) & (fabsf(n2) > tiny));
      if (plausible) {
        const float t1 = RB_DIV(n1, det);
        // t2 is only tested, never used: strictly inside (0.0001 |det| < |n2| < 0.9999 |det|, same sign) the rounded
        // quotient is inside [0, 1] as well, and its division is skipped
        bool t2_ok = ((n2 < 0.0f) == neg) & (fabsf(n2) > 1e-4f * ad) & (fabsf(n2) < 0.9999f * ad);
        if (!t2_ok) {
          const float t2 = RB_DIV(n2, det);
          t2_ok = t2 >= 0.0f && t2 <= 1.0f;
        }
        if (t1 >= 0.0f && t1 <= 1.0f && t2_ok) {
          sink.put(n, RB_ADD(ax, RB_MUL(e1x, t1)), RB_ADD(ay, RB_MUL(e1y, t1)));
          ++n;
        }
      }
    }
    // rotate box 1's vertices: (0, 1, 2, 3) <- (1, 2, 3, 0); after four rounds they are back in place
    p1x[0] = p1x[1]; p1y[0] = p1y[1];
    p1x[1] = p1x[2]; p1y[1] = p1y[2];
    p1x[2] = p1x[3]; p1y[2] = p1y[3];
    p1x[3] = ax; p1y[3] = ay;
  }
  {
    float abab = rb_dot(e2x[0], e2y[0], e2x[0], e2y[0]);
    float adad = rb_dot(e2x[3], e2y[3], e2x[3], e2y[3]);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float apx = RB_SUB(p1x[i], p2x[0]), apy = RB_SUB(p1y[i], p2y[0]);
      float apab = rb_dot(apx, apy, e2x[0], e2y[0]);
      float apad = -rb_dot(apx, apy, e2x[3], e2y[3]);
      if (apab >= 0.0f && apad >= 0.0f && apab <= abab && apad <= adad) {
        sink.put(n, p1x[i], p1y[i]); ++n;
      }
    }
  }
  {
    const float e10x = RB_SUB(p1x[1], p1x[0]), e10y = RB_SUB(p1y[1], p1y[0]);      // edge 0 and edge 3 of box 1
    const float e13x = RB_SUB(p1x[0], p1x[3]), e13y = RB_SUB(p1y[0], p1y[3]);
    float abab = rb_dot(e10x, e10y, e10x, e10y);
    float adad = rb_dot(e13x, e13y, e13x, e13y);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float apx = RB_SUB(p2x[i], p1x[0]), apy = RB_SUB(p2y[i], p1y[0]);
      float apab = rb_dot(apx, apy, e10x, e10y);
      float apad = -rb_dot(apx, apy, e13x, e13y);
      if (apab >= 0.0f && apad >= 0.0f && apab <= abab && apad <= adad) {
        sink.put(n, p2x[i], p2y[i]); ++n;
      }
    }
  }
  return n;
}

// Hull + area on a 24-point array (the general path): in-place Graham hull in the CUDA build's exchange-sort order
// (:169-282), fan area (:284-296).  Returns the intersection area.
RB_HD float rbox_hull_area(float* qx, float* qy, int n) {
  float inter = 0.0f;
  if (n > 2) {
    // lowest point (min y, then min x), shift every point by it, move it to slot 0
    int t = 0;
    for (int i = 1; i < n; ++i)
      if (qy[i] < qy[t] || (qy[i] == qy[t] && qx[i] < qx[t])) t = i;
    float sx = qx[t], sy = qy[t];
    for (int i = 0; i < n; ++i) { qx[i] = RB_SUB(qx[i], sx); qy[i] = RB_SUB(qy[i], sy); }
    { float tx = qx[0], ty = qy[0]; qx[0] = qx[t]; qy[0] = qy[t]; qx[t] = tx; qy[t] = ty; }
    // exchange sort by polar angle; 1e-6 collinearity band, squared-distance tie break
    for (int i = 1; i < n - 1; ++i) {
      float ax = qx[i], ay = qy[i];
      float ad = rb_dot(ax, ay, ax, ay);
      for (int j = i + 1; j < n; ++j) {
        float bx = qx[j], by = qy[j];
        float cp = rb_cross(ax, ay, bx, by);
        bool sw = (cp <= -RB_HI_1E6);                               // cp < -1e-6
        if (!sw && fabsf(cp) <= RB_LO_1E6) sw = ad > rb_dot(bx, by, bx, by);   // |cp| < 1e-6 && di > dj
        if (sw) {
          qx[j] = ax; qy[j] = ay; ax = bx; ay = by;
          ad = rb_dot(ax, ay, ax, ay);
        }
      }
      qx[i] = ax; qy[i] = ay;
    }
    int k = 1;
    for (; k < n; ++k)
      if (rb_dot(qx[k], qy[k], qx[k], qy[k]) >= RB_HI_1E8) break;  // dist > 1e-8
    if (k < n) {
      qx[1] = qx[k]; qy[1] = qy[k];
      int m = 2;
      for (int i = k + 1; i < n; ++i) {
        float cx = qx[i], cy = qy[i];
        while (m > 1) {
          float ox = qx[m - 2], oy = qy[m - 2];
          float cr = rb_cross(RB_SUB(cx, ox), RB_SUB(cy, oy), RB_SUB(qx[m - 1], ox), RB_SUB(qy[m - 1], oy));
          if (!(cr >= 0.0f)) break;
          --m;
        }
        qx[m] = cx; qy[m] = cy; ++m;
      }
      if (m > 2) {
        float area = 0.0f;
        float ox = qx[0], oy = qy[0];
        for (int i = 1; i < m - 1; ++i)
          area = RB_ADD(area, fabsf(rb_cross(RB_SUB(qx[i], ox), RB_SUB(qy[i], oy),
                                             RB_SUB(qx[i + 1], ox), RB_SUB(qy[i + 1], oy))));
        inter = RB_MUL(area, 0.5f);                                  // area / 2.0
      }
    }
  }
  return inter;
}

struct RbArraySink {
  float* qx; float* qy;
  RB_HD void put(int k, float x, float y) { qx[k] = x; qy[k] = y; }
};

// The general clipper (thread-local 24-point arrays): iou = inter / (a1 + a2 - inter) (:361-362, unclamped).
// Precondition: both areas >= 1e-14 (rbox_classify handled the early-out).
RB_HD float rbox_iou_clip(const RBox& A, const RBox& B) {
  float qx[24], qy[24];
  RbArraySink sink{qx, qy};
  const int n = rbox_candidates(A, B, sink);
  const float inter = rbox_hull_area(qx, qy, n);
  const float a1 = RB_MUL(A.w, A.h), a2 = RB_MUL(B.w, B.h);
  return RB_DIV(inter, RB_SUB(RB_ADD(a1, a2), inter));
}

// ---- register-resident hull for 3 <= n <= 8 ------------------------------------------------------------------
// Two convex quadrilaterals in general position intersect in at most 8 points and every candidate is a vertex of the
// intersection polygon (21.8 M anchor x GT pairs of BASELINE config 4: n in {0, 3..8}, never more).  For those the
// reference's hull construction is a fixed sequence: the exchange sort (:209-226) is the comparator network
// (i, j), 1 <= i < j < n, whatever the data -- 21 compare-exchanges on 8 named registers, predicated on j < n -- and the
// Graham scan (:243-268) pops nothing when the sorted points are strictly convex.  This routine runs exactly the
// reference's operations in that case and REPORTS (returns false) instead of guessing in every other: the second
// point coincides with the first (:234-241 would skip it) or any scan step would pop (cr >= 0, :254).  The caller
// then runs the general clipper.  All indices are compile-time constants: no local memory.
RB_HD bool rbox_hull8(float (&qx)[8], float (&qy)[8], int n, float& inter) {
  // lowest point (min y, then min x)
  int t = 0;
  float sx = qx[0], sy = qy[0];
#pragma unroll
  for (int i = 1; i < 8; ++i)
    if (i < n && (qy[i] < sy || (qy[i] == sy && qx[i] < sx))) { t = i; sx = qx[i]; sy = qy[i]; }
#pragma unroll
  for (int i = 0; i < 8; ++i) { qx[i] = RB_SUB(qx[i], sx); qy[i] = RB_SUB(qy[i], sy); }
  {  // swap q[0] <-> q[t]
    const float t0x = qx[0], t0y = qy[0];
    float zx = t0x, zy = t0y;
#pragma unroll
    for (int i = 1; i < 8; ++i)
      if (i == t) { zx = qx[i]; zy = qy[i]; qx[i] = t0x; qy[i] = t0y; }
    qx[0] = zx; qy[0] = zy;
  }
  // exchange sort by polar angle; 1e-6 collinearity band, squared-distance tie break
#pragma unroll
  for (int i = 1; i < 7; ++i) {
    float ax = qx[i], ay = qy[i];
#pragma unroll
    for (int j = i + 1; j < 8; ++j) {
      // (selects, not branches: n differs from lane to lane)
      const float bx = qx[j], by = qy[j];
      const float cp = rb_cross(ax, ay, bx, by);
      bool sw = (cp <= -RB_HI_1E6);
      if (!sw && fabsf(cp) <= RB_LO_1E6) sw = rb_dot(ax, ay, ax, ay) > rb_dot(bx, by, bx, by);   // (rare: collinear)
      sw = sw & (j < n);
      qx[j] = sw ? ax : bx; qy[j] = sw ? ay : by;
      ax = sw ? bx : ax; ay = sw ? by : ay;
    }
    qx[i] = ax; qy[i] = ay;
  }
  bool ok = rb_dot(qx[1], qy[1], qx[1], qy[1]) >= RB_HI_1E8;      // k == 1: the second point is not a copy of the first
#pragma unroll
  for (int i = 2; i < 8; ++i) {
    const float ox = qx[i - 2], oy = qy[i - 2];
    const float cr = rb_cross(RB_SUB(qx[i], ox), RB_SUB(qy[i], oy), RB_SUB(qx[i - 1], ox), RB_SUB(qy[i - 1], oy));
    ok = ok & (!(cr >= 0.0f) | (i >= n));                         // the scan would not pop
  }
  float area = 0.0f;
  const float ox = qx[0], oy = qy[0];
#pragma unroll
  for (int i = 1; i < 7; ++i)
  {
    const float tri = fabsf(rb_cross(RB_SUB(qx[i], ox), RB_SUB(qy[i], oy), RB_SUB(qx[i + 1], ox), RB_SUB(qy[i + 1], oy)));
    area = (i < n - 1) ? RB_ADD(area, tri) : area;
  }
  inter = RB_MUL(area, 0.5f);
  return ok;
}

// Candidate points staged through a caller-provided scratch column (shared memory on the device: element k of this
// thread at scratch[k * stride], x in [0, 8), y in [8, 16)) -- dynamic indexing happens in the ADDRESS, the points
// then come back into 16 named registers for rbox_hull8.  Falls back to the general clipper when n > 8 or the hull is
// not the generic strictly convex one.  Bit-identical to rbox_iou_clip.
struct RbScratchSink {
  float* s; int stride;
  RB_HD void put(int k, float x, float y) {
    if (k < 8) { s[k * stride] = x; s[(8 + k) * stride] = y; }
  }
};

// `ok` = false: not the generic case, the value is meaningless and the caller must run rbox_iou_clip instead (kept
// out of line by the kernels: it is the only code that touches local memory).
RB_HD float rbox_iou_clip_try(const RBox& A, const RBox& B, float* scratch, int stride, bool& ok) {
  RbScratchSink sink{scratch, stride};
  const int n = rbox_candidates(A, B, sink);
  const float a1 = RB_MUL(A.w, A.h), a2 = RB_MUL(B.w, B.h);
  float inter = 0.0f;
  ok = n <= 8;
  if (n > 2 && ok) {
    float qx[8], qy[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      // (slots >= n hold stale values of earlier pairs: never read by a predicated step)
      qx[k] = scratch[k * stride];
      qy[k] = scratch[(8 + k) * stride];
    }
    ok = rbox_hull8(qx, qy, n, inter);
  }
  return RB_DIV(inter, RB_SUB(RB_ADD(a1, a2), inter));
}

RB_HD float rbox_iou_clip_fast(const RBox& A, const RBox& B, float* scratch, int stride) {
  bool ok;
  const float v = rbox_iou_clip_try(A, B, scratch, stride, ok);
  return ok ? v : rbox_iou_clip(A, B);
}

// Full semantic of single_box_iou_rotated on prepared boxes (:333-375).
RB_HD float rbox_iou(const RBox& A, const RBox& B) {
  return rbox_classify(A, B) == RB_ZERO ? 0.0f : rbox_iou_clip(A, B);
}

}  // namespace s2a
