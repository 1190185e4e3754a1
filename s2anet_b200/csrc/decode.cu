// decode.cu -- the two box-decode stages that sit either side of AlignConv/ORConv in the S2ANet head,
// each as ONE launch over all FPN levels and all images of the batch (SURVEY.md section 8(f) rows 2-3).
//
// Replaces (reference):
//   * fam_bbox_decode + gen_grid_anchors: models/head.py:27-52, models/anchors.py:75-126 --
//     `s2a_fam_decode` turns fam_bbox_pred [B,5,H,W] into the refined rotated anchors [B,H,W,5]
//     (the grid anchor is analytic: centre s*i + (s-1)/2, w = h = scale*s, theta = angle).
//   * get_bboxes_single_img up to (not including) the NMS: models/head.py:684-717 -- sigmoid,
//     per-level top-k by best class score, gather, concatenation over levels, final
//     delta2bbox_rotated; `s2a_select_decode` does all of it for the whole batch.
// Arithmetic: box_decode.cuh (shared with the FAM-decode epilogue of conv_tc.cu).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>
#include <type_traits>


#include "box_decode.cuh"
#include "common.cuh"

namespace s2a {

constexpr int DEC_MAX_LEVELS = 8;
constexpr int DEC_THREADS = 1024;

template <typename T> __device__ __forceinline__ float ld_as_float(const T* p);
template <> __device__ __forceinline__ float ld_as_float<float>(const float* p) { return *p; }
template <> __device__ __forceinline__ float ld_as_float<__nv_bfloat16>(const __nv_bfloat16* p) {
  return __bfloat162float(*p);
}
template <> __device__ __forceinline__ float ld_as_float<__half>(const __half* p) { return __half2float(*p); }

template <typename T> __device__ __forceinline__ float bits16_to_float(unsigned short b);
template <> __device__ __forceinline__ float bits16_to_float<float>(unsigned short) { return 0.0f; }   // (never used)
template <> __device__ __forceinline__ float bits16_to_float<__nv_bfloat16>(unsigned short b) {
  return __uint_as_float((uint32_t)b << 16);
}
template <> __device__ __forceinline__ float bits16_to_float<__half>(unsigned short b) { return __half2float(__ushort_as_half(b)); }

// The first `n` (<= 16) consecutive channels of one location as floats.  16-bit channels-last tensors whose
// locations are at least 16 (8) elements apart and 16-byte aligned are read with two (one) 16-byte loads --
// otherwise a warp would pull one 32-byte sector per 2-byte element.
template <typename T>
__device__ __forceinline__ void load_channels(const T* q, long long cstride, long long pstride, int n, float* out) {
  if (sizeof(T) == 2 && cstride == 1 && (reinterpret_cast<uintptr_t>(q) & 15) == 0 && pstride >= (n <= 8 ? 8 : 16) && n <= 16) {
    const uint4 v0 = __ldg(reinterpret_cast<const uint4*>(q));
    uint4 v1 = make_uint4(0u, 0u, 0u, 0u);
    if (n > 8) v1 = __ldg(reinterpret_cast<const uint4*>(q) + 1);
    const uint32_t w[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
#pragma unroll
    for (int c = 0; c < 16; ++c)
      if (c < n) out[c] = bits16_to_float<T>((unsigned short)(w[c >> 1] >> ((c & 1) * 16)));
  } else {
    for (int c = 0; c < n; ++c) out[c] = ld_as_float(q + c * cstride);
  }
}

// max that propagates NaN like torch.max (fmaxf drops it): a location with a NaN logit gets a NaN best score
__device__ __forceinline__ float nan_max(float a, float b) { return (b > a || b != b) ? b : a; }

// Top-k key of a best score: its bits (scores are >= 0, so they order like unsigned integers), NaN of either sign
// mapped to the largest key -- the reference's topk ranks NaN above every number
__device__ __forceinline__ uint32_t score_key(float s) { return s != s ? 0x7FFFFFFFu : __float_as_uint(s); }

// torch.sigmoid on a T tensor: T(1 / (1 + exp(-float(x)))) (ATen UnarySpecialOpsKernel)
template <typename T> __device__ __forceinline__ float sigmoid_t(float x) {
  return round_through<T>(__fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x))));
}

// ------------------------------------------------------------------------------------------------
// FAM decode
// ------------------------------------------------------------------------------------------------
struct FamLevel {
  const void* deltas;     // [B, 5, H, W], element strides s[4]
  float* out;             // [B, H, W, 5] fp32 contiguous
  long long s[4];
  int H, W;
  long long begin;        // first global position index of this level (positions = B*H*W per level)
  float stride;
};
struct FamParams {
  FamLevel lv[DEC_MAX_LEVELS];
  int nlevels, B;
  long long total;
  float scale, angle, lim;
};

template <typename T>
__global__ void __launch_bounds__(256) fam_decode_kernel(const __grid_constant__ FamParams p) {
  for (long long g = (long long)blockIdx.x * blockDim.x + threadIdx.x; g < p.total; g += (long long)gridDim.x * blockDim.x) {
    int l = 0;
    while (l + 1 < p.nlevels && g >= p.lv[l + 1].begin) ++l;
    const FamLevel& L = p.lv[l];
    long long r = g - L.begin;
    const int x = (int)(r % L.W);
    r /= L.W;
    const int y = (int)(r % L.H);
    const int b = (int)(r / L.H);
    float a[5];
    fam_grid_anchor(x, y, L.stride, p.scale, p.angle, a);
    const T* d = reinterpret_cast<const T*>(L.deltas) + b * L.s[0] + y * L.s[2] + x * L.s[3];
    float o[5];
    delta2bbox_rotated<T>(a, ld_as_float(d), ld_as_float(d + L.s[1]), ld_as_float(d + 2 * L.s[1]),
                          ld_as_float(d + 3 * L.s[1]), ld_as_float(d + 4 * L.s[1]), p.lim, o);
    float* dst = L.out + (((long long)b * L.H + y) * L.W + x) * 5;
#pragma unroll
    for (int i = 0; i < 5; ++i) dst[i] = o[i];
  }
}

// ------------------------------------------------------------------------------------------------
// select (per-level top-k) + decode
// ------------------------------------------------------------------------------------------------
struct SelLevel {
  const void* cls;        // [B, C, H, W] logits, element strides cs[4]
  const void* reg;        // [B, 5, H, W] deltas, element strides rs[4]
  const float* anchors;   // [B, H*W, 5] fp32 contiguous
  long long cs[4], rs[4];
  int H, W, n, k;         // n = H*W, k = min(n, topk)
  int out_off;            // first row of this level in the concatenated candidate list
  long long key_off;      // offset of this level inside one image's key scratch
};
struct SelParams {
  SelLevel lv[DEC_MAX_LEVELS];
  int nlevels, B, C, n_total;
  long long keys_per_image;
  uint32_t* keys;         // workspace [B][keys_per_image]
  float* bboxes;          // [B, n_total, 5]
  float* scores;          // [B, n_total, C]
  int32_t* index_out;     // optional [B, n_total]: position (y*W + x) of every candidate inside its level
  float lim;
  int debug;
  int smem_keys;          // keys of a level with at most this many locations live in shared memory
  int sort_bytes;         // offset of that key array inside the dynamic shared memory
  int split;              // 1: keys come from select_keys_kernel, the selection goes to sel_idx, gather_decode_kernel
                          //    writes the outputs (three launches, the two data-parallel ones grid-wide); 0: one launch
  int32_t* sel_idx;       // workspace [B][n_total]: selected location per output row (split mode)
};

__device__ __forceinline__ unsigned long long composite_key(uint32_t key, int i) {
  return ((unsigned long long)key << 32) | (unsigned long long)(0xFFFFFFFFu - (uint32_t)i);
}

// Best class score of every location of one (level, image) -> keys[i] (score_key of the T-rounded sigmoid), models/head.py:700-701.
// `t` of `NT` threads cooperate (a CTA, or the whole grid row of select_keys_kernel).
template <typename T>
__device__ __forceinline__ void compute_keys(const SelLevel& L, const T* cls, int C, int n, uint32_t* keys, int t, int NT) {
  constexpr int UNR = 4;                                  // locations in flight per thread (latency-bound loop)
  // 16-bit channels-last logits with at most 16 classes (the head's own layout): a PAIR of lanes reads one location
  // -- 16 bytes = 8 classes each -- so that a warp's load covers 16 consecutive pixels (8 cache lines) instead of
  // 32 pixels with every other 16-byte chunk skipped (32 sectors in 16 lines, and half the lanes' worth of loads)
  const bool paired = sizeof(T) == 2 && C <= 16 && L.cs[1] == 1 && (L.cs[3] & 7) == 0 && (L.cs[2] & 7) == 0 &&
                      (L.cs[0] & 7) == 0 && (reinterpret_cast<uintptr_t>(L.cls) & 15) == 0 && L.cs[3] >= (C <= 8 ? 8 : 16);
  if (paired) {
    const int HALF_T = NT / 2;
    const int half = t & 1, pr = t >> 1;
    for (int base = 0; base < n; base += UNR * HALF_T) {
      uint4 v[UNR];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int i = min(base + u * HALF_T + pr, n - 1);
        const int y = i / L.W, x = i - y * L.W;
        v[u] = make_uint4(0u, 0u, 0u, 0u);
        if (half * 8 < C) v[u] = __ldg(reinterpret_cast<const uint4*>(cls + y * L.cs[2] + x * L.cs[3]) + half);
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const uint32_t w[4] = {v[u].x, v[u].y, v[u].z, v[u].w};
        float m = -INFINITY;
#pragma unroll
        for (int e = 0; e < 8; ++e)
          if (half * 8 + e < C) m = nan_max(m, bits16_to_float<T>((unsigned short)(w[e >> 1] >> ((e & 1) * 16))));
        m = nan_max(m, __shfl_xor_sync(0xffffffffu, m, 1));
        const int i = base + u * HALF_T + pr;
        if (half == 0 && i < n) keys[i] = score_key(sigmoid_t<T>(m));
      }
    }
  } else
  for (int i0 = t; i0 < n; i0 += UNR * NT) {
    float m[UNR];
    if (C <= 16) {
      float v[UNR][16];
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int i = min(i0 + u * NT, n - 1);
        const int y = i / L.W, x = i - y * L.W;
        load_channels<T>(cls + y * L.cs[2] + x * L.cs[3], L.cs[1], L.cs[3], C, v[u]);
      }
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        m[u] = -INFINITY;
#pragma unroll
        for (int c = 0; c < 16; ++c)
          if (c < C) m[u] = nan_max(m[u], v[u][c]);
      }
    } else {
#pragma unroll
      for (int u = 0; u < UNR; ++u) {
        const int i = min(i0 + u * NT, n - 1);
        const int y = i / L.W, x = i - y * L.W;
        const T* q = cls + y * L.cs[2] + x * L.cs[3];
        m[u] = -INFINITY;
        for (int c = 0; c < C; ++c) m[u] = nan_max(m[u], ld_as_float(q + c * L.cs[1]));
      }
    }
    // sigmoid is monotone, so max_c sigmoid(x_c) == sigmoid(max_c x_c) bit for bit
#pragma unroll
    for (int u = 0; u < UNR; ++u)
      if (i0 + u * NT < n) keys[i0 + u * NT] = score_key(sigmoid_t<T>(m[u]));
  }
}

template <typename T, int ITEMS>
__global__ void __launch_bounds__(DEC_THREADS) select_decode_kernel(const __grid_constant__ SelParams p) {
  extern __shared__ __align__(16) uint8_t dsm[];
  __shared__ unsigned long long s_sel[DEC_THREADS * ITEMS];
  __shared__ unsigned int s_hist[256];
  __shared__ unsigned long long s_prefix;
  __shared__ int s_remaining, s_done, s_count;

  const SelLevel& L = p.lv[blockIdx.x];
  const int b = blockIdx.y, tid = threadIdx.x;
  const int n = L.n, k = L.k, C = p.C;
  const T* cls = reinterpret_cast<const T*>(L.cls) + b * L.cs[0];
  const T* reg = reinterpret_cast<const T*>(L.reg) + b * L.rs[0];
  const bool select = n > k;
  if (p.split && !select) return;                          // nothing to select: gather_decode_kernel takes row j = location j
  long long t0 = clock64(), t1 = t0, t2 = t0, t3 = t0;

  // composite sort key: (score bits, 16 significant bits for 16-bit inputs) . (index bits, lower location first)
  const int nb = 32 - __clz(max(n - 1, 1));                 // bits of a location index
  // a bf16 (fp16) score widened to fp32 has 16 (13) zero low bits
  const int kshift = std::is_same<T, __nv_bfloat16>::value ? 16 : (std::is_same<T, __half>::value ? 13 : 0);
  const int total_bits = 32 - kshift + nb;
  const unsigned idx_mask = (1u << nb) - 1u;
  auto composite = [&](uint32_t key, int i) -> unsigned long long {
    return ((unsigned long long)(key >> kshift) << nb) | (unsigned long long)(idx_mask - (unsigned)i);
  };
  if (select) {
    // ---- keys: best class score of every location (models/head.py:700-701); kept in shared memory when they fit
    uint32_t* keys = n <= p.smem_keys ? reinterpret_cast<uint32_t*>(dsm + p.sort_bytes)
                                      : p.keys + (long long)b * p.keys_per_image + L.key_off;
    if (p.split) {                                          // keys were produced grid-wide: bring them on chip
      const uint32_t* gk = p.keys + (long long)b * p.keys_per_image + L.key_off;
      if (keys != gk)
        for (int i = tid; i < n; i += DEC_THREADS) keys[i] = gk[i];
    } else {
      compute_keys<T>(L, cls, C, n, keys, tid, DEC_THREADS);
    }
    if (tid == 0) { s_prefix = 0ull; s_remaining = k; s_done = 0; s_count = 0; }
    __syncthreads();
    t1 = clock64();
    // ---- radix select of the k-th largest composite (score, lower index first): exact top-k with a
    // defined tie rule (torch.topk leaves ties unspecified) --------------------------------------
    for (int shift = ((total_bits - 1) / 8) * 8; shift >= 0; shift -= 8) {
      for (int i = tid; i < 256; i += DEC_THREADS) s_hist[i] = 0u;
      __syncthreads();
      const unsigned long long prefix = s_prefix;
      for (int base = 0; base < n; base += DEC_THREADS) {
        const int i = base + tid;
        unsigned bin = 0xFFFFFFFFu;                       // inactive lanes form their own group
        if (i < n) {
          const unsigned long long c = composite(keys[i], i);
          if (shift + 8 >= 64 || (c >> (shift + 8)) == (prefix >> (shift + 8))) bin = (unsigned)(c >> shift) & 255u;
        }
        // scores cluster in a handful of bins: one shared atomic per distinct bin per warp, not per key
        const unsigned peers = __match_any_sync(0xffffffffu, bin);
        if (bin != 0xFFFFFFFFu && (tid & 31) == __ffs(peers) - 1) atomicAdd(&s_hist[bin], (unsigned)__popc(peers));
      }
      __syncthreads();
      if (tid < 32) {
        // lane owns bins [8*lane, 8*lane+8); suffix sums from the top bin downwards
        unsigned int loc[8], sum = 0;
#pragma unroll
        for (int j = 0; j < 8; ++j) { loc[j] = s_hist[tid * 8 + j]; sum += loc[j]; }
        unsigned int incl = sum;              // inclusive suffix scan over lanes
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const unsigned int v = __shfl_down_sync(0xffffffffu, incl, o);
          if (tid + o < 32) incl += v;
        }
        const unsigned int above = incl - sum;   // elements in the bins of higher lanes
        const unsigned int rem = (unsigned int)s_remaining;
        if (above < rem && incl >= rem) {     // the crossing bin is in this lane
          unsigned int cum = above;
          for (int j = 7; j >= 0; --j) {
            if (cum + loc[j] >= rem) {
              s_prefix = prefix | ((unsigned long long)(tid * 8 + j) << shift);
              s_remaining = (int)(rem - cum);
              if (loc[j] == rem - cum) s_done = 1;      // the whole bin is selected: threshold found
              break;
            }
            cum += loc[j];
          }
        }
      }
      __syncthreads();
      if (s_done) break;
    }
    const unsigned long long thr = s_prefix;
    t2 = clock64();
    // ---- collect the k selected composites and sort them (descending score, ascending index) ----
    for (int i = tid; i < DEC_THREADS * ITEMS; i += DEC_THREADS) s_sel[i] = 0ull;
    __syncthreads();
    for (int base = 0; base < n; base += DEC_THREADS) {
      const int i = base + tid;
      const unsigned long long c = i < n ? composite(keys[i], i) : 0ull;
      const bool take = i < n && c >= thr;
      const unsigned bal = __ballot_sync(0xffffffffu, take);
      if (bal) {
        int pos = 0;
        if ((tid & 31) == 0) pos = atomicAdd(&s_count, __popc(bal));
        pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(bal & ((1u << (tid & 31)) - 1u));
        if (take && pos < DEC_THREADS * ITEMS) s_sel[pos] = c;
      }
    }
    // Bitonic sort of the DEC_THREADS * ITEMS slots in shared memory, descending (the zero padding ends up behind the
    // k survivors): 66 compare-exchange rounds for 2,048 slots, one barrier each -- a block radix sort of the same
    // keys (8 four-bit passes with their ranking scans) took 34 k cycles, six times longer.
    constexpr int NS = DEC_THREADS * ITEMS;
    static_assert((NS & (NS - 1)) == 0, "bitonic sort needs a power-of-two slot count");
    for (int size = 2; size <= NS; size <<= 1) {
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        __syncthreads();
#pragma unroll
        for (int t = tid; t < NS / 2; t += DEC_THREADS) {
          const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
          const unsigned long long a = s_sel[lo], c = s_sel[hi];
          const bool descending = (lo & size) == 0;            // (always true in the last merge: size == NS)
          if ((a < c) == descending) { s_sel[lo] = c; s_sel[hi] = a; }
        }
      }
    }
    __syncthreads();
  }

  t3 = clock64();
  if (p.split) {                                           // the selected locations, in output order
    int32_t* dst = p.sel_idx + (long long)b * p.n_total + L.out_off;
    for (int j = tid; j < k; j += DEC_THREADS) dst[j] = (int32_t)(idx_mask - (unsigned)(s_sel[j] & (unsigned long long)idx_mask));
    if (p.debug && tid == 0 && blockIdx.y == 0)
      printf("select_decode level %d (split): keys %lld, select %lld, collect+sort %lld cycles\n", (int)blockIdx.x, t1 - t0, t2 - t1,
             t3 - t2);
    return;
  }
  // ---- gather + sigmoid + final decode (models/head.py:703-717) ---------------------------------
  // Output rows of a level are contiguous ([k, C] scores, [k, 5] boxes), but a thread owns a whole row: written
  // directly that is 20 scattered 4-byte stores per location (32 sectors per warp instruction).  With at most 16
  // classes the rows of DEC_THREADS locations are staged in shared memory (the sort scratch and the keys are dead by
  // now; row strides C and 5 words are odd -> conflict-free) and copied out with coalesced stores.
  const bool staged = C <= 16;
  float* st_sc = reinterpret_cast<float*>(dsm);
  float* st_bb = st_sc + DEC_THREADS * C;
  for (int j0 = 0; j0 < k; j0 += DEC_THREADS) {
    const int j = j0 + tid;
    const int cnt = min(DEC_THREADS, k - j0);
    const long long row0 = (long long)b * p.n_total + L.out_off + j0;
    if (staged) __syncthreads();                     // (first round: everybody is done with the sort scratch / keys)
    if (j < k) {
      const int i = select ? (int)(idx_mask - (unsigned)(s_sel[j] & (unsigned long long)idx_mask)) : j;
      const int y = i / L.W, x = i - y * L.W;
      const long long row = row0 + tid;
      const T* q = cls + y * L.cs[2] + x * L.cs[3];
      float* so = staged ? st_sc + tid * C : p.scores + row * C;
      if (C <= 16) {
        float v[16];
        load_channels<T>(q, L.cs[1], L.cs[3], C, v);
#pragma unroll
        for (int c = 0; c < 16; ++c)
          if (c < C) so[c] = sigmoid_t<T>(v[c]);
      } else {
        for (int c = 0; c < C; ++c) so[c] = sigmoid_t<T>(ld_as_float(q + c * L.cs[1]));
      }
      float d[5];
      load_channels<T>(reg + y * L.rs[2] + x * L.rs[3], L.rs[1], L.rs[3], 5, d);
      const float* ap = L.anchors + ((long long)b * n + i) * 5;
      const float a[5] = {__ldg(ap), __ldg(ap + 1), __ldg(ap + 2), __ldg(ap + 3), __ldg(ap + 4)};
      float o[5];
      delta2bbox_rotated<T>(a, d[0], d[1], d[2], d[3], d[4], p.lim, o);
      float* bo = staged ? st_bb + tid * 5 : p.bboxes + row * 5;
#pragma unroll
      for (int e = 0; e < 5; ++e) bo[e] = o[e];
      if (p.index_out) p.index_out[row] = i;
    }
    if (staged) {
      __syncthreads();
      float* gs = p.scores + row0 * C;
      for (int e = tid; e < cnt * C; e += DEC_THREADS) gs[e] = st_sc[e];
      float* gb = p.bboxes + row0 * 5;
      for (int e = tid; e < cnt * 5; e += DEC_THREADS) gb[e] = st_bb[e];
    }
  }
  if (p.debug && tid == 0 && blockIdx.y == 0)
    printf("select_decode level %d: keys %lld, select %lld, collect+sort %lld, gather+decode %lld cycles\n", (int)blockIdx.x, t1 - t0, t2 - t1,
           t3 - t2, clock64() - t3);
}

// ---- split mode, launch 1: keys of every level that needs a selection, grid-wide ------------------------------
template <typename T>
__global__ void __launch_bounds__(256) select_keys_kernel(const __grid_constant__ SelParams p) {
  const SelLevel& L = p.lv[blockIdx.y];
  if (L.n <= L.k) return;
  const int b = blockIdx.z;
  const T* cls = reinterpret_cast<const T*>(L.cls) + b * L.cs[0];
  compute_keys<T>(L, cls, p.C, L.n, p.keys + (long long)b * p.keys_per_image + L.key_off,
                  (int)(blockIdx.x * blockDim.x + threadIdx.x), (int)(gridDim.x * blockDim.x));
}

// ---- split mode, launch 3: gather + sigmoid + final decode of every output row (models/head.py:703-717) ----------
// One thread per row of the concatenated candidate list; a block's 256 rows are contiguous in both outputs and go
// through shared memory so that the global stores are coalesced (row strides C and 5 words: conflict-free).
template <typename T>
__global__ void __launch_bounds__(256) gather_decode_kernel(const __grid_constant__ SelParams p) {
  extern __shared__ __align__(16) uint8_t dsm[];
  const int b = blockIdx.y, tid = threadIdx.x, C = p.C;
  const int r0 = blockIdx.x * 256, r = r0 + tid;
  const int cnt = min(256, p.n_total - r0);
  const bool staged = C <= 16;
  float* st_sc = reinterpret_cast<float*>(dsm);
  float* st_bb = st_sc + 256 * C;
  const long long row0 = (long long)b * p.n_total + r0;
  if (r < p.n_total) {
    int l = 0;
    while (l + 1 < p.nlevels && r >= p.lv[l + 1].out_off) ++l;
    const SelLevel& L = p.lv[l];
    const int j = r - L.out_off;
    const int i = L.n > L.k ? p.sel_idx[(long long)b * p.n_total + r] : j;
    const int y = i / L.W, x = i - y * L.W;
    const T* q = reinterpret_cast<const T*>(L.cls) + b * L.cs[0] + y * L.cs[2] + x * L.cs[3];
    const T* g = reinterpret_cast<const T*>(L.reg) + b * L.rs[0] + y * L.rs[2] + x * L.rs[3];
    float* so = staged ? st_sc + tid * C : p.scores + (row0 + tid) * C;
    if (C <= 16) {
      float v[16];
      load_channels<T>(q, L.cs[1], L.cs[3], C, v);
#pragma unroll
      for (int c = 0; c < 16; ++c)
        if (c < C) so[c] = sigmoid_t<T>(v[c]);
    } else {
      for (int c = 0; c < C; ++c) so[c] = sigmoid_t<T>(ld_as_float(q + c * L.cs[1]));
    }
    float d[5];
    load_channels<T>(g, L.rs[1], L.rs[3], 5, d);
    const float* ap = L.anchors + ((long long)b * L.n + i) * 5;
    const float a[5] = {__ldg(ap), __ldg(ap + 1), __ldg(ap + 2), __ldg(ap + 3), __ldg(ap + 4)};
    float o[5];
    delta2bbox_rotated<T>(a, d[0], d[1], d[2], d[3], d[4], p.lim, o);
    float* bo = staged ? st_bb + tid * 5 : p.bboxes + (row0 + tid) * 5;
#pragma unroll
    for (int e = 0; e < 5; ++e) bo[e] = o[e];
    if (p.index_out) p.index_out[row0 + tid] = i;
  }
  if (staged) {
    __syncthreads();
    float* gs = p.scores + row0 * C;
    for (int e = tid; e < cnt * C; e += 256) gs[e] = st_sc[e];
    float* gb = p.bboxes + row0 * 5;
    for (int e = tid; e < cnt * 5; e += 256) gb[e] = st_bb[e];
  }
}

template <typename T, int ITEMS>
static int launch_select(SelParams p, cudaStream_t st) {
  auto kern = select_decode_kernel<T, ITEMS>;
  p.sort_bytes = 0;                                              // (the keys start the dynamic shared memory)
  p.smem_keys = 16384;                                          // 64 KB: P3 of a 1024^2 image
  int need = 0;
  for (int l = 0; l < p.nlevels; ++l)
    if (p.lv[l].n > p.lv[l].k && p.lv[l].n <= p.smem_keys) need = std::max(need, p.lv[l].n);
  size_t smem = (size_t)p.sort_bytes + (size_t)need * sizeof(uint32_t);
  if (p.C <= 16) smem = std::max(smem, (size_t)DEC_THREADS * (p.C + 5) * sizeof(float));   // output staging (gather phase)
  S2A_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  if (p.split) {
    int nmax = 0;
    for (int l = 0; l < p.nlevels; ++l)
      if (p.lv[l].n > p.lv[l].k) nmax = std::max(nmax, p.lv[l].n);
    if (nmax > 0) {
      // pairs of threads, four locations in flight each: enough blocks to cover the largest level once
      const int bx = (int)std::min<long long>(ceil_div((long long)nmax * 2, 256 * 4), (long long)sm_count() * 4);
      select_keys_kernel<T><<<dim3(std::max(bx, 1), p.nlevels, p.B), 256, 0, st>>>(p);
      S2A_LAUNCH_OK("select_keys_kernel");
      kern<<<dim3(p.nlevels, p.B), DEC_THREADS, smem, st>>>(p);
      S2A_LAUNCH_OK("select_decode_kernel");
    }
    const size_t gsm = p.C <= 16 ? (size_t)256 * (p.C + 5) * sizeof(float) : 0;
    gather_decode_kernel<T><<<dim3((unsigned)ceil_div(p.n_total, 256), p.B), 256, gsm, st>>>(p);
    S2A_LAUNCH_OK("gather_decode_kernel");
    return S2A_OK;
  }
  kern<<<dim3(p.nlevels, p.B), DEC_THREADS, smem, st>>>(p);
  S2A_LAUNCH_OK("select_decode_kernel");
  return S2A_OK;
}

template <typename T>
static int launch_select_items(const SelParams& p, int kmax, cudaStream_t st) {
  if (kmax <= 2 * DEC_THREADS) return launch_select<T, 2>(p, st);
  return launch_select<T, 4>(p, st);
}

}  // namespace s2a

extern "C" int s2a_fam_decode(int nlevels, const void* const* deltas, const int64_t* delta_strides, float* const* refined,
                              const int* Hs, const int* Ws, const float* strides, int B, float anchor_scale,
                              float anchor_angle, double wh_ratio_clip, int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(nlevels >= 1 && nlevels <= DEC_MAX_LEVELS, "fam_decode: 1..%d levels per call", DEC_MAX_LEVELS);
  S2A_CHECK_ARG(B >= 0 && wh_ratio_clip > 0.0, "fam_decode: bad batch size or wh_ratio_clip");
  S2A_CHECK_ARG(dtype == S2A_F32 || dtype == S2A_BF16 || dtype == S2A_F16, "fam_decode: unknown dtype %d", dtype);
  if (B == 0) return S2A_OK;
  S2A_CHECK_ARG(deltas && delta_strides && refined && Hs && Ws && strides, "fam_decode: null pointer");
  FamParams p{};
  long long total = 0;
  for (int l = 0; l < nlevels; ++l) {
    S2A_CHECK_ARG(Hs[l] > 0 && Ws[l] > 0 && deltas[l] && refined[l] && strides[l] > 0.0f, "fam_decode: bad level %d", l);
    FamLevel& L = p.lv[l];
    L.deltas = deltas[l]; L.out = refined[l]; L.H = Hs[l]; L.W = Ws[l]; L.begin = total; L.stride = strides[l];
    for (int i = 0; i < 4; ++i) L.s[i] = delta_strides[4 * l + i];
    total += (long long)B * Hs[l] * Ws[l];
  }
  p.nlevels = nlevels; p.B = B; p.total = total; p.scale = anchor_scale; p.angle = anchor_angle;
  p.lim = clamp_limit(wh_ratio_clip, dtype);
  const int blocks = (int)std::min<long long>(ceil_div(total, 256), (long long)sm_count() * 8);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == S2A_F32) fam_decode_kernel<float><<<blocks, 256, 0, st>>>(p);
  else if (dtype == S2A_BF16) fam_decode_kernel<__nv_bfloat16><<<blocks, 256, 0, st>>>(p);
  else fam_decode_kernel<__half><<<blocks, 256, 0, st>>>(p);
  S2A_LAUNCH_OK("fam_decode_kernel");
  return S2A_OK;
}

extern "C" size_t s2a_select_decode_workspace_bytes(int nlevels, const int* Hs, const int* Ws, int B) {
  size_t keys = 0;
  for (int l = 0; l < nlevels; ++l) keys += (size_t)Hs[l] * Ws[l];
  // keys [B][sum H*W] uint32 + selected locations [B][n_total <= sum H*W] int32
  return 2 * keys * sizeof(uint32_t) * (size_t)(B > 0 ? B : 0) + 512;
}

extern "C" int s2a_select_decode(int nlevels, const void* const* cls, const int64_t* cls_strides, const void* const* reg,
                                 const int64_t* reg_strides, const float* const* anchors, const int* Hs, const int* Ws,
                                 int B, int num_classes, int topk, double wh_ratio_clip, int dtype, float* bboxes_out,
                                 float* scores_out, int32_t* index_out, int64_t n_total, void* workspace,
                                 size_t workspace_bytes, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(nlevels >= 1 && nlevels <= DEC_MAX_LEVELS, "select_decode: 1..%d levels per call", DEC_MAX_LEVELS);
  S2A_CHECK_ARG(B >= 0 && num_classes > 0 && wh_ratio_clip > 0.0, "select_decode: bad sizes");
  S2A_CHECK_ARG(dtype == S2A_F32 || dtype == S2A_BF16 || dtype == S2A_F16, "select_decode: unknown dtype %d", dtype);
  if (B == 0) return S2A_OK;
  S2A_CHECK_ARG(cls && cls_strides && reg && reg_strides && anchors && Hs && Ws && bboxes_out && scores_out,
                "select_decode: null pointer");
  SelParams p{};
  long long keys = 0;
  int off = 0, kmax = 0;
  for (int l = 0; l < nlevels; ++l) {
    S2A_CHECK_ARG(Hs[l] > 0 && Ws[l] > 0 && (long long)Hs[l] * Ws[l] < (1ll << 31) && cls[l] && reg[l] && anchors[l],
                  "select_decode: bad level %d", l);
    SelLevel& L = p.lv[l];
    L.cls = cls[l]; L.reg = reg[l]; L.anchors = anchors[l]; L.H = Hs[l]; L.W = Ws[l]; L.n = Hs[l] * Ws[l];
    L.k = (topk > 0 && L.n > topk) ? topk : L.n;          // models/head.py:699: only levels with more than topk locations
    for (int i = 0; i < 4; ++i) { L.cs[i] = cls_strides[4 * l + i]; L.rs[i] = reg_strides[4 * l + i]; }
    L.out_off = off; L.key_off = keys;
    off += L.k; keys += L.n;
    if (L.n > L.k) kmax = std::max(kmax, L.k);
  }
  S2A_CHECK_ARG(n_total == off, "select_decode: n_total must be sum_l min(H*W, topk) = %d (got %lld)", off, (long long)n_total);
  if (kmax > 4 * DEC_THREADS) {
    set_error("select_decode: topk up to %d is supported (got %d)", 4 * DEC_THREADS, kmax);
    return S2A_ERR_UNSUPPORTED;
  }
  if (workspace_bytes < s2a_select_decode_workspace_bytes(nlevels, Hs, Ws, B) || !workspace) {
    set_error("select_decode: workspace too small");
    return S2A_ERR_WORKSPACE;
  }
  p.nlevels = nlevels; p.B = B; p.C = num_classes; p.n_total = off; p.keys_per_image = keys;
  p.keys = reinterpret_cast<uint32_t*>(workspace); p.bboxes = bboxes_out; p.scores = scores_out; p.index_out = index_out;
  p.sel_idx = reinterpret_cast<int32_t*>(reinterpret_cast<uint8_t*>(workspace) + align_up((size_t)keys * sizeof(uint32_t) * B, 256));
  p.lim = clamp_limit(wh_ratio_clip, dtype);
  { const char* e = getenv("S2A_DEC_DEBUG"); p.debug = e ? atoi(e) : 0; }
  p.split = (p.debug & 2) ? 0 : 1;                          // S2A_DEC_DEBUG=2: the single-launch form (timing comparisons)
  p.debug &= 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == S2A_F32) return launch_select_items<float>(p, kmax, st);
  if (dtype == S2A_BF16) return launch_select_items<__nv_bfloat16>(p, kmax, st);
  return launch_select_items<__half>(p, kmax, st);
}
