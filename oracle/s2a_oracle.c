/*
 * s2a_oracle.c -- CPU oracle for the S2ANet custom-op hot path.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it,
 * and there only as the checker / the CPU baseline.  The product (s2anet_b200/) never
 * imports, links or falls back to this file.
 *
 * It is a from-scratch restatement, in plain C, of the algorithms of the reference
 * (chongkuiqi/S2ANet).  Every function cites the reference file:line it follows.  The
 * reference publishes no tests or golden vectors for this path (SURVEY.md section 4), so the
 * restatement is pinned against the reference's own sources compiled in place
 * (oracle/_ref, see oracle/build_ref.py) and the resulting vectors are committed under
 * tests/golden/ (generator: tests/golden/make_golden.py).
 *
 * Floating-point contract: compile with -ffp-contract=off and no fast-math.  All rotated-box
 * arithmetic is IEEE fp32 with individually rounded multiplies and adds, the few double
 * promotions of the reference kept where they matter, so that the sm_100a kernels (written
 * with __fmul_rn/__fadd_rn, i.e. also un-contracted) can be compared bit for bit.
 *
 * Semantics: where the reference's CPU and CUDA builds disagree (SURVEY.md A.4/A.5) the
 * CUDA build is followed, because the CUDA build is what val.py / train.py actually run:
 *   - hull ordering = the O(n^2) exchange sort that also permutes dist[]
 *   - NMS suppresses on  iou >  thr   (the CPU build uses >=; selectable here by a flag)
 */
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define S2A_API __attribute__((visibility("default")))

typedef struct { float x, y; } pt_t;

static inline float cross2(pt_t a, pt_t b) { return a.x * b.y - b.x * a.y; }
static inline float dot2(pt_t a, pt_t b) { return a.x * b.x + a.y * b.y; }
static inline pt_t sub2(pt_t a, pt_t b) { pt_t r = { a.x - b.x, a.y - b.y }; return r; }

/* utils/box_iou_rotated/src/box_iou_rotated_utils.h:55-75 (get_rotated_vertices).
 * theta is in RADIANS (the degree conversion is commented out at :59-62); cos/sin are
 * evaluated in double, narrowed to float and halved (:63-64). */
static void box_vertices(float xc, float yc, float w, float h, float a, pt_t p[4])
{
    double theta = (double)a;
    float c2 = (float)cos(theta) * 0.5f;
    float s2 = (float)sin(theta) * 0.5f;
    p[0].x = xc - s2 * h - c2 * w;
    p[0].y = yc + c2 * h - s2 * w;
    p[1].x = xc + s2 * h - c2 * w;
    p[1].y = yc - c2 * h - s2 * w;
    p[2].x = 2.0f * xc - p[0].x;
    p[2].y = 2.0f * yc - p[0].y;
    p[3].x = 2.0f * xc - p[1].x;
    p[3].y = 2.0f * yc - p[1].y;
}

/* box_iou_rotated_utils.h:77-167 (get_intersection_points): 16 edge/edge tests, then the
 * corners of box 1 inside box 2, then the corners of box 2 inside box 1.  Duplicates are
 * kept (up to 24 points). */
static int candidate_points(const pt_t p1[4], const pt_t p2[4], pt_t out[24])
{
    pt_t e1[4], e2[4];
    int n = 0;
    for (int i = 0; i < 4; ++i) {
        e1[i] = sub2(p1[(i + 1) & 3], p1[i]);
        e2[i] = sub2(p2[(i + 1) & 3], p2[i]);
    }
    for (int i = 0; i < 4; ++i) {
        for (int j = 0; j < 4; ++j) {
            float det = cross2(e2[j], e1[i]);
            if (fabs((double)det) <= 1e-14) continue;          /* :103, parallel edges */
            pt_t d = sub2(p2[j], p1[i]);
            float t1 = cross2(e2[j], d) / det;
            float t2 = cross2(e1[i], d) / det;
            if (t1 >= 0.0f && t1 <= 1.0f && t2 >= 0.0f && t2 <= 1.0f) {   /* :114 inclusive */
                out[n].x = p1[i].x + e1[i].x * t1;
                out[n].y = p1[i].y + e1[i].y * t1;
                ++n;
            }
        }
    }
    {   /* :121-142 corners of box 1 inside box 2, by projection on AB and AD */
        pt_t ab = e2[0], da = e2[3];
        float abab = dot2(ab, ab), adad = dot2(da, da);
        for (int i = 0; i < 4; ++i) {
            pt_t ap = sub2(p1[i], p2[0]);
            float apab = dot2(ap, ab);
            float apad = -dot2(ap, da);
            if (apab >= 0 && apad >= 0 && apab <= abab && apad <= adad) out[n++] = p1[i];
        }
    }
    {   /* :145-164 the mirror test */
        pt_t ab = e1[0], da = e1[3];
        float abab = dot2(ab, ab), adad = dot2(da, da);
        for (int i = 0; i < 4; ++i) {
            pt_t ap = sub2(p2[i], p1[0]);
            float apab = dot2(ap, ab);
            float apad = -dot2(ap, da);
            if (apab >= 0 && apad >= 0 && apab <= abab && apad <= adad) out[n++] = p2[i];
        }
    }
    return n;
}

/* box_iou_rotated_utils.h:169-282 (convex_hull_graham, shift_to_zero = true) in its
 * __CUDACC__ form (:209-226): exchange sort by polar angle around the lowest point with a
 * 1e-6 collinearity band and squared-distance tie break, dist[] permuted with q[]. */
static int hull_cuda_order(const pt_t *p, int n, pt_t *q)
{
    float dist[24];
    int t = 0;
    for (int i = 1; i < n; ++i)
        if (p[i].y < p[t].y || (p[i].y == p[t].y && p[i].x < p[t].x)) t = i;
    pt_t start = p[t];
    for (int i = 0; i < n; ++i) q[i] = sub2(p[i], start);
    { pt_t tmp = q[0]; q[0] = q[t]; q[t] = tmp; }
    for (int i = 0; i < n; ++i) dist[i] = dot2(q[i], q[i]);

    for (int i = 1; i < n - 1; ++i) {
        for (int j = i + 1; j < n; ++j) {
            float cp = cross2(q[i], q[j]);
            if (((double)cp < -1e-6) || (fabs((double)cp) < 1e-6 && dist[i] > dist[j])) {
                pt_t tq = q[i]; q[i] = q[j]; q[j] = tq;
                float td = dist[i]; dist[i] = dist[j]; dist[j] = td;
            }
        }
    }
    int k;
    for (k = 1; k < n; ++k)
        if ((double)dist[k] > 1e-8) break;                     /* :244-248 */
    if (k == n) return 1;                                       /* all points coincide */
    q[1] = q[k];
    int m = 2;
    for (int i = k + 1; i < n; ++i) {
        while (m > 1 && cross2(sub2(q[i], q[m - 2]), sub2(q[m - 1], q[m - 2])) >= 0) --m;
        q[m++] = q[i];
    }
    return m;
}

/* box_iou_rotated_utils.h:284-296 (polygon_area): fan of |cross| from q[0], halved. */
static float fan_area(const pt_t *q, int m)
{
    if (m <= 2) return 0.0f;
    float area = 0.0f;
    for (int i = 1; i < m - 1; ++i)
        area += fabsf(cross2(sub2(q[i], q[0]), sub2(q[i + 1], q[0])));
    return (float)((double)area / 2.0);
}

/* box_iou_rotated_utils.h:333-375 (single_box_iou_rotated).  The centre shift is an fp32
 * sum halved in double and subtracted in double, then narrowed (:340-349). */
S2A_API float s2a_oracle_single_iou(const float *b1, const float *b2)
{
    double shx = (double)(b1[0] + b2[0]) / 2.0;
    double shy = (double)(b1[1] + b2[1]) / 2.0;
    float x1 = (float)((double)b1[0] - shx), y1 = (float)((double)b1[1] - shy);
    float x2 = (float)((double)b2[0] - shx), y2 = (float)((double)b2[1] - shy);
    float area1 = b1[2] * b1[3];
    float area2 = b2[2] * b2[3];
    if ((double)area1 < 1e-14 || (double)area2 < 1e-14) return 0.0f;   /* :354-358 */

    pt_t p1[4], p2[4], cand[24], hull[24];
    box_vertices(x1, y1, b1[2], b1[3], b1[4], p1);
    box_vertices(x2, y2, b2[2], b2[3], b2[4], p2);
    float inter = 0.0f;
    int n = candidate_points(p1, p2, cand);
    if (n > 2) {                                                /* :316-318 */
        int m = hull_cuda_order(cand, n, hull);
        inter = fan_area(hull, m);
    }
    return inter / (area1 + area2 - inter);                     /* :361-362, unclamped */
}

/* utils/box_iou_rotated/src/box_iou_rotated_cuda.cu:13-62, 65-101: out[i*m + j] =
 * iou(boxes1[i], boxes2[j]); row-major [n, m] fp32. */
S2A_API void s2a_oracle_box_iou_rotated(const float *boxes1, int64_t n, const float *boxes2,
                                        int64_t m, float *out)
{
    for (int64_t i = 0; i < n; ++i)
        for (int64_t j = 0; j < m; ++j)
            out[i * m + j] = s2a_oracle_single_iou(boxes1 + 5 * i, boxes2 + 5 * j);
}

/* ---- rotated NMS ------------------------------------------------------------------- */

typedef struct { float score; int64_t idx; } sc_t;
static int by_score_desc(const void *a, const void *b)
{
    const sc_t *x = (const sc_t *)a, *y = (const sc_t *)b;
    if (x->score > y->score) return -1;
    if (x->score < y->score) return 1;
    return (x->idx > y->idx) - (x->idx < y->idx);   /* ties: lower index first (stable) */
}

/* utils/nms_rotated/src/nms_rotated_cuda.cu:72-132 and utils/ml_nms_rotated/src/
 * nms_rotated_cuda.cu:74-137: sort by score descending, greedy sweep over the suppression
 * relation iou(earlier, later) > thr, return ORIGINAL indices in descending-score order.
 * labels == NULL -> class-agnostic (nms_rotated); otherwise pairs with different labels
 * never suppress (ml_nms_rotated/src/box_iou_rotated_utils.h:317-322, float equality).
 * ge != 0 selects the CPU build's  >=  predicate (nms_rotated_cpu.cpp:52).
 * The reference sort is not stable; ties are broken here by index, lower first, which is
 * the order the library's stable sorts give (tests/test_gpu_postprocess_exact.py checks it
 * on tied 16-bit scores).  Returns the number of kept boxes. */
S2A_API int64_t s2a_oracle_nms_rotated(const float *dets, const float *scores,
                                       const float *labels, int64_t n, float thr, int ge,
                                       int64_t *keep)
{
    if (n <= 0) return 0;
    sc_t *ord = (sc_t *)malloc(sizeof(sc_t) * (size_t)n);
    uint8_t *dead = (uint8_t *)calloc((size_t)n, 1);
    for (int64_t i = 0; i < n; ++i) { ord[i].score = scores[i]; ord[i].idx = i; }
    qsort(ord, (size_t)n, sizeof(sc_t), by_score_desc);
    int64_t nk = 0;
    for (int64_t a = 0; a < n; ++a) {
        if (dead[a]) continue;
        int64_t i = ord[a].idx;
        keep[nk++] = i;
        for (int64_t b = a + 1; b < n; ++b) {
            if (dead[b]) continue;
            int64_t j = ord[b].idx;
            if (labels && labels[i] != labels[j]) continue;
            float v = s2a_oracle_single_iou(dets + 5 * i, dets + 5 * j);
            if (ge ? (v >= thr) : (v > thr)) dead[b] = 1;
        }
    }
    free(ord); free(dead);
    return nk;
}

/* ---- ORN: active rotating filters ------------------------------------------------- */

/* models/orn/src/cuda/ActiveRotatingFilter_cuda.cu:19-46 (ARF_forward_cuda_kernel):
 * weight [O, I, nOri, kH, kW], indices uint8 [nOri*kH*kW, nRot] (1-based destination
 * entry), out [O*nRot, I*nOri, kH, kW]:
 *   out[(o*nRot + k), i, idx[l][k]-1] = w[o, i, l]          (entry = nOri*kH*kW) */
S2A_API void s2a_oracle_arf_forward(const float *w, const uint8_t *indices, int O, int I,
                                    int nOri, int kH, int kW, int nRot, float *out)
{
    int nEntry = nOri * kH * kW;
    for (int o = 0; o < O; ++o)
        for (int i = 0; i < I; ++i)
            for (int l = 0; l < nEntry; ++l) {
                float v = w[((int64_t)o * I + i) * nEntry + l];
                for (int k = 0; k < nRot; ++k) {
                    int dst = (int)indices[l * nRot + k] - 1;
                    out[(((int64_t)o * nRot + k) * I + i) * nEntry + dst] = v;
                }
            }
}

/* ActiveRotatingFilter_cuda.cu:48-76 (ARF_backward_cuda_kernel): the gather-sum adjoint. */
S2A_API void s2a_oracle_arf_backward(const float *gout, const uint8_t *indices, int O, int I,
                                     int nOri, int kH, int kW, int nRot, float *gw)
{
    int nEntry = nOri * kH * kW;
    for (int o = 0; o < O; ++o)
        for (int i = 0; i < I; ++i)
            for (int l = 0; l < nEntry; ++l) {
                float acc = 0.0f;
                for (int k = 0; k < nRot; ++k) {
                    int src = (int)indices[l * nRot + k] - 1;
                    acc = acc + gout[(((int64_t)o * nRot + k) * I + i) * nEntry + src];
                }
                gw[((int64_t)o * I + i) * nEntry + l] = acc;
            }
}

/* models/orn/functions/rotation_invariant_pooling.py:19-27: max over each group of nOri
 * consecutive channels.  x [B, C, H, W] -> out [B, C/nOri, H, W]. */
S2A_API void s2a_oracle_ri_pool(const float *x, int B, int C, int H, int W, int nOri,
                                float *out)
{
    int64_t hw = (int64_t)H * W;
    int G = C / nOri;
    for (int b = 0; b < B; ++b)
        for (int g = 0; g < G; ++g)
            for (int64_t p = 0; p < hw; ++p) {
                float m = x[((int64_t)b * C + (int64_t)g * nOri) * hw + p];
                for (int o = 1; o < nOri; ++o) {
                    float v = x[((int64_t)b * C + (int64_t)g * nOri + o) * hw + p];
                    if (v > m) m = v;
                }
                out[((int64_t)b * G + g) * hw + p] = m;
            }
}

/* ---- deformable convolution ------------------------------------------------------- */

/* models/dcn/src/deform_conv_cuda_kernel.cu:83-114 (deformable_im2col_bilinear): floor,
 * fractional weights, corners outside the map read as 0. */
static float bilinear_fp32(const float *plane, int H, int W, float h, float w)
{
    int h_lo = (int)floorf(h), w_lo = (int)floorf(w);
    int h_hi = h_lo + 1, w_hi = w_lo + 1;
    float lh = h - (float)h_lo, lw = w - (float)w_lo;
    float hh = 1.0f - lh, hw = 1.0f - lw;
    float v1 = (h_lo >= 0 && w_lo >= 0) ? plane[h_lo * W + w_lo] : 0.0f;
    float v2 = (h_lo >= 0 && w_hi <= W - 1) ? plane[h_lo * W + w_hi] : 0.0f;
    float v3 = (h_hi <= H - 1 && w_lo >= 0) ? plane[h_hi * W + w_lo] : 0.0f;
    float v4 = (h_hi <= H - 1 && w_hi <= W - 1) ? plane[h_hi * W + w_hi] : 0.0f;
    float w1 = hh * hw, w2 = hh * lw, w3 = lh * hw, w4 = lh * lw;
    return w1 * v1 + w2 * v2 + w3 * v3 + w4 * v4;
}

/* models/dcn/src/deform_conv_cuda.cpp:152-260 (deform_conv_forward_cuda) with the im2col
 * of deform_conv_cuda_kernel.cu:189-242: for every output position the sampled column
 *   col[(c*kH + i)*kW + j] = bilinear(x[b, c], h_in + i*dil + off_y, w_in + j*dil + off_x)
 * (0 unless -1 < h < H and -1 < w < W, :228), then out = W[Co, C/g*kH*kW] . col per group
 * (:231-236).  Offsets: [B, dg*2*kH*kW, Ho, Wo], channel 2*(i*kW+j) = dy, +1 = dx (:218-221).
 * Sampling is fp32 like the reference; the contraction accumulates in double and rounds
 * once (the reference's cuBLAS summation order is unspecified, so parity on this op is a
 * tolerance, not bit equality).  x [B,C,H,W], w [Co, C/groups, kH, kW], out [B,Co,Ho,Wo]. */
S2A_API int s2a_oracle_deform_conv_forward(const float *x, const float *offset,
                                           const float *w, float *out, int B, int C, int H,
                                           int W, int Co, int kH, int kW, int sH, int sW,
                                           int pH, int pW, int dH, int dW, int groups,
                                           int dgroups, int relu)
{
    int Ho = (H + 2 * pH - (dH * (kH - 1) + 1)) / sH + 1;
    int Wo = (W + 2 * pW - (dW * (kW - 1) + 1)) / sW + 1;
    if (Ho < 1 || Wo < 1 || C % groups || Co % groups || C % dgroups) return -1;
    int Cg = C / groups, Cog = Co / groups, cpd = C / dgroups;
    int K = Cg * kH * kW;
    float *col = (float *)malloc(sizeof(float) * (size_t)C * kH * kW);
    int64_t ohw = (int64_t)Ho * Wo;
    for (int b = 0; b < B; ++b) {
        const float *offb = offset + (int64_t)b * dgroups * 2 * kH * kW * ohw;
        for (int ho = 0; ho < Ho; ++ho)
            for (int wo = 0; wo < Wo; ++wo) {
                int h_in = ho * sH - pH, w_in = wo * sW - pW;
                for (int c = 0; c < C; ++c) {
                    const float *plane = x + ((int64_t)b * C + c) * H * W;
                    const float *offg = offb + (int64_t)(c / cpd) * 2 * kH * kW * ohw;
                    for (int i = 0; i < kH; ++i)
                        for (int j = 0; j < kW; ++j) {
                            float oy = offg[(int64_t)(2 * (i * kW + j)) * ohw + (int64_t)ho * Wo + wo];
                            float ox = offg[(int64_t)(2 * (i * kW + j) + 1) * ohw + (int64_t)ho * Wo + wo];
                            float hs = (float)(h_in + i * dH) + oy;
                            float ws = (float)(w_in + j * dW) + ox;
                            float v = 0.0f;
                            if (hs > -1 && ws > -1 && hs < H && ws < W)
                                v = bilinear_fp32(plane, H, W, hs, ws);
                            col[(c * kH + i) * kW + j] = v;
                        }
                }
                for (int g = 0; g < groups; ++g)
                    for (int oc = 0; oc < Cog; ++oc) {
                        const float *wr = w + (int64_t)(g * Cog + oc) * K;
                        const float *cg = col + (int64_t)g * K;
                        double acc = 0.0;
                        for (int k = 0; k < K; ++k) acc += (double)wr[k] * (double)cg[k];
                        float r = (float)acc;
                        if (relu && r < 0.0f) r = 0.0f;
                        out[(((int64_t)b * Co + g * Cog + oc) * Ho + ho) * Wo + wo] = r;
                    }
            }
    }
    free(col);
    return 0;
}

/* models/alignconv.py:29-86 (AlignConv.get_offset), kernel 3x3: for location (yc, xc) with
 * anchor (x, y, w, h, a) in image pixels, tap (i, j) in {-1,0,1}^2:
 *   px = cos*(w/s/3*j) - sin*(h/s/3*i) + x/s ;  py = sin*(w/s/3*j) + cos*(h/s/3*i) + y/s
 *   offset = (py - (yc + i), px - (xc + j)), channels ordered [dy0, dx0, dy1, dx1, ...].
 * Operation order follows the torch expressions (fp32; cosf/sinf, so the last ulp can
 * differ from torch's vectorised cos/sin).  anchors [H*W, 5] -> out [18, H, W]. */
S2A_API void s2a_oracle_alignconv_offset(const float *anchors, int H, int W, float stride,
                                         float *out)
{
    int64_t hw = (int64_t)H * W;
    for (int yc = 0; yc < H; ++yc)
        for (int xc = 0; xc < W; ++xc) {
            const float *a = anchors + 5 * ((int64_t)yc * W + xc);
            float x = a[0] / stride, y = a[1] / stride, w = a[2] / stride, h = a[3] / stride;
            float cs = cosf(a[4]), sn = sinf(a[4]);
            float dw = w / 3.0f, dh = h / 3.0f;
            for (int i = -1; i <= 1; ++i)
                for (int j = -1; j <= 1; ++j) {
                    float tx = dw * (float)j, ty = dh * (float)i;
                    float xr = cs * tx - sn * ty;
                    float yr = sn * tx + cs * ty;
                    float xa = xr + x, ya = yr + y;
                    float offx = xa - ((float)xc + (float)j);
                    float offy = ya - ((float)yc + (float)i);
                    int t = (i + 1) * 3 + (j + 1);
                    out[(int64_t)(2 * t) * hw + (int64_t)yc * W + xc] = offy;
                    out[(int64_t)(2 * t + 1) * hw + (int64_t)yc * W + xc] = offx;
                }
        }
}

/* models/alignconv.py:88-98 (AlignConv.forward): per-image offsets, 3x3 / pad 1 / stride 1
 * deformable conv (groups = deformable_groups = 1, no bias), ReLU.
 * x [B,C,H,W], anchors [B,H,W,5], w [Co,C,3,3] -> out [B,Co,H,W]. */
S2A_API int s2a_oracle_alignconv_forward(const float *x, const float *anchors, const float *w,
                                         float *out, int B, int C, int H, int W, int Co,
                                         float stride)
{
    int64_t hw = (int64_t)H * W;
    float *off = (float *)malloc(sizeof(float) * (size_t)B * 18 * hw);
    for (int b = 0; b < B; ++b)
        s2a_oracle_alignconv_offset(anchors + (int64_t)b * hw * 5, H, W, stride,
                                    off + (int64_t)b * 18 * hw);
    int rc = s2a_oracle_deform_conv_forward(x, off, w, out, B, C, H, W, Co, 3, 3, 1, 1, 1, 1,
                                            1, 1, 1, 1, /*relu=*/1);
    free(off);
    return rc;
}

/* torch.nn.functional.conv2d as used by models/orn/modules/ORConv.py:80-82 (stride 1,
 * dilation 1, groups 1; zero padding).  x [B,C,H,W], w [Co,C,kH,kW], bias [Co] or NULL.
 * Double accumulation, one rounding. */
S2A_API void s2a_oracle_conv2d(const float *x, const float *w, const float *bias, float *out,
                               int B, int C, int H, int W, int Co, int kH, int kW, int pH,
                               int pW)
{
    int Ho = H + 2 * pH - kH + 1, Wo = W + 2 * pW - kW + 1;
    for (int b = 0; b < B; ++b)
        for (int oc = 0; oc < Co; ++oc)
            for (int ho = 0; ho < Ho; ++ho)
                for (int wo = 0; wo < Wo; ++wo) {
                    double acc = bias ? (double)bias[oc] : 0.0;
                    for (int c = 0; c < C; ++c)
                        for (int i = 0; i < kH; ++i) {
                            int hi = ho - pH + i;
                            if (hi < 0 || hi >= H) continue;
                            for (int j = 0; j < kW; ++j) {
                                int wi = wo - pW + j;
                                if (wi < 0 || wi >= W) continue;
                                acc += (double)x[(((int64_t)b * C + c) * H + hi) * W + wi] *
                                       (double)w[(((int64_t)oc * C + c) * kH + i) * kW + j];
                            }
                        }
                    out[(((int64_t)b * Co + oc) * Ho + ho) * Wo + wo] = (float)acc;
                }
}

/* models/orn/modules/ORConv.py:77-82 (ORConv2d.forward) = conv2d(x, ARF(weight), bias),
 * optionally followed by RotationInvariantPooling (rotation_invariant_pooling.py:19-27).
 * w [O, I, nOri, kH, kW]; x [B, I*nOri, H, W]; bias [O*nRot] or NULL;
 * out [B, O*nRot, H, W]; pooled [B, O*nRot/pool_group, H, W] or NULL. */
S2A_API void s2a_oracle_orconv_forward(const float *x, const float *w, const uint8_t *indices,
                                       const float *bias, float *out, float *pooled, int B,
                                       int H, int W, int O, int I, int nOri, int kH, int kW,
                                       int nRot, int pad, int pool_group)
{
    int Co = O * nRot, C = I * nOri;
    float *wr = (float *)malloc(sizeof(float) * (size_t)Co * C * kH * kW);
    s2a_oracle_arf_forward(w, indices, O, I, nOri, kH, kW, nRot, wr);
    s2a_oracle_conv2d(x, wr, bias, out, B, C, H, W, Co, kH, kW, pad, pad);
    if (pooled) {
        int Ho = H + 2 * pad - kH + 1, Wo = W + 2 * pad - kW + 1;
        s2a_oracle_ri_pool(out, B, Co, Ho, Wo, pool_group, pooled);
    }
    free(wr);
}
