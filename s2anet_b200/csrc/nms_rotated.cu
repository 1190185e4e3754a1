// nms_rotated.cu -- rotated NMS for sm_100a: nms_rotated, ml_nms_rotated (generic, score-ordered)
// and the fused, batched, class-segmented multiclass_nms_rotated.
//
// Replaces (reference): utils/nms_rotated/src/nms_rotated_cuda.cu:13-69 (mask kernel), :72-132
// (host: sort, mask, D2H copy, serial CPU sweep, H2D); utils/ml_nms_rotated/src/nms_rotated_cuda.cu
// :13-71, :74-137 (label-aware twin); utils/bbox_nms_rotated.py:5-64 (multiclass wrapper).
//
// What is different from the reference, and why:
//   * the suppression mask is computed for the upper triangle only (the reference computes both
//     triangles and never reads the lower one), 64x64 pairs per CTA, with the same
//     classify -> compact -> clip scheme as box_iou_rotated.cu so lanes are not parked on the
//     ~95 % of pairs that are trivially disjoint;
//   * the greedy sweep runs ON THE DEVICE in one CTA: each 64-box block is resolved by one warp with
//     register shuffles, then its kept rows are OR-ed into the running "removed" bitmap by the whole
//     CTA.  No device->host copy of the mask, no host sweep, no synchronisation;
//   * multiclass: (box, class) candidates never interact across classes, so the fused path sorts and
//     sweeps each (image, class) segment independently (15x fewer pair tests, 15 sweeps in parallel)
//     and merges the survivors by rank (binary searches), instead of sorting all candidates globally.
// Results are identical to the reference CUDA semantics: predicate IoU > thr, IoU(earlier, later).
#include <cub/cub.cuh>
#include <float.h>
#include <thrust/iterator/counting_iterator.h>
#include <thrust/iterator/transform_iterator.h>

#include "common.cuh"
#include "rbox_iou.cuh"

namespace s2a {

constexpr int kBlk = 64;            // boxes per mask word
constexpr int kMaskThreads = 256;   // (the polygon NMS tile: one CTA per tile)
constexpr int kSweepThreads = 1024;

// ------------------------------------------------------------------------------------------------
// tile body: 64 row boxes x 64 column boxes -> 64 suppression words, evaluated by ONE WARP
// ------------------------------------------------------------------------------------------------
// Same organisation as box_iou_rotated_kernel (round 2): the warp's lanes own two columns each and walk the rows;
// a ~20-flop test on 24-byte box summaries settles most pairs, the rest goes through warp-private queues -- full
// classification and the intersection bounds, then the register-resident clipper -- always with all lanes busy, and
// no barrier is wider than the warp.  (Round 1: one 256-thread CTA per tile, three CTA-wide phases, byte flags and a
// shuffle transpose to build the words: 89 G pairs/s at 10 k candidates against the IoU kernel's 300.)
constexpr int kTileWarps = 4;                        // warps (independent tiles in flight) per CTA
constexpr int kTileThreads = kTileWarps * 32;
constexpr int kTileQueue = 32 + 16 * kBlk;           // < 32 left over + one 16-row block of undecided pairs

struct WarpTileSmem {
  RBox row[kBlk];
  RBox col[kBlk];
  RFast rowf[kBlk];
  RAng rowa[kBlk];
  float lrow[kBlk];
  unsigned long long word[kBlk];
  uint16_t qm[kTileQueue];           // pairs the fast test could not decide: row << 6 | column
  uint16_t qc[kBlk];                 // pairs to clip
  float pts[16 * 32];                // per-lane candidate column of the register-resident clipper
};

// the general 24-point clipper (thread-local arrays), out of line: reached by degenerate pairs only
__device__ __noinline__ float nms_clip_general(const RBox& A, const RBox& B) { return rbox_iou_clip(A, B); }

// rows/cols: pointers to the first prepared box of the row/col block; nr/nc valid counts; diag: row block == col
// block (only c > r is evaluated); labels may be null (then every pair is a same-class pair).  On return (after a
// __syncwarp) s.word[r] bit c says "column box c is suppressed by row box r": same label and IoU > thr.
__device__ __forceinline__ void mask_tile_warp(WarpTileSmem& s, const RBox* __restrict__ rows,
                                               const RBox* __restrict__ cols, const float* __restrict__ lrows,
                                               const float* __restrict__ lcols, int nr, int nc, bool diag, float thr) {
  const unsigned lane = threadIdx.x & 31u, lt = (1u << lane) - 1u;
  // a zero IoU suppresses only under a negative threshold; then nothing may be settled by the zero test
  const bool use_fast = thr >= 0.0f;
  // ---- load: 2 x 64 prepared boxes (32 B each), summaries of the rows to shared memory, of this lane's two columns
  // to registers
  {
    const uint4* gr = reinterpret_cast<const uint4*>(rows);
    const uint4* gc = reinterpret_cast<const uint4*>(cols);
    uint4* sr = reinterpret_cast<uint4*>(s.row);
    uint4* sc = reinterpret_cast<uint4*>(s.col);
    for (int e = lane; e < nr * 2; e += 32) sr[e] = gr[e];
    for (int e = lane; e < nc * 2; e += 32) sc[e] = gc[e];
  }
  __syncwarp();
  RFast cf[2]; RAng ca[2];
  float lc[2];
  bool cok[2];
#pragma unroll
  for (int g = 0; g < 2; ++g) {
    const int c = 32 * g + (int)lane;
    cok[g] = c < nc;
    cf[g].x = cf[g].y = cf[g].r = cf[g].mn = 0.0f; ca[g].s2t = ca[g].c2t = 0.0f;
    lc[g] = 0.0f;
    if (cok[g]) { rbox_fast_of(s.col[c], cf[g], ca[g]); lc[g] = lcols ? lcols[c] : 0.0f; }
    const int r = c;
    if (r < nr) { rbox_fast_of(s.row[r], s.rowf[r], s.rowa[r]); s.lrow[r] = lrows ? lrows[r] : 0.0f; }
    s.word[c] = 0ull;
  }
  __syncwarp();

  int nm = 0, nq = 0, r = 0;
  while (true) {
    // ---- all pairs, 16 rows per block: one bit per undecided pair in a register, appended once per block
    for (; r < nr && nm < 32; r += 16) {
      unsigned mk = 0u;
#pragma unroll 1
      for (int h = 0; h < 2; ++h) {
        unsigned sub = 0u;
        const int r8 = r + 8 * h;
        const int nrow = min(8, nr - r8);
#pragma unroll
        for (int rr = 0; rr < 8; ++rr) {
          if (rr < nrow) {
            const RFast rf = s.rowf[r8 + rr];
            const RAng ra = s.rowa[r8 + rr];
            const float lr = s.lrow[r8 + rr];
#pragma unroll
            for (int g = 0; g < 2; ++g) {
              const int c = 32 * g + (int)lane;
              const bool valid = cok[g] && (!diag || c > r8 + rr) && lr == lc[g];       // labels differ -> IoU := 0
              const bool zero = use_fast && rbox_fast_zero(rf, ra, cf[g], ca[g]);
              if (valid && !zero) sub |= 1u << (g * 8 + rr);
            }
          }
        }
        mk |= ((sub & 0xffu) << (8 * h)) | ((sub >> 8) << (16 + 8 * h));
      }
      const int cntl = __popc(mk);
      int pos = cntl;
#pragma unroll
      for (int d = 1; d < 32; d <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, pos, d);
        if ((int)lane >= d) pos += up;
      }
      const int total = __shfl_sync(0xffffffffu, pos, 31);
      if (total) {
        pos += nm - cntl;
        while (mk) {
          const int bit = __ffs(mk) - 1;
          mk &= mk - 1u;
          s.qm[pos++] = (uint16_t)(((r + (bit & 15)) << 6) | ((bit >> 4) << 5) | lane);
        }
        nm += total;
        __syncwarp();
      }
    }
    const bool done = r >= nr;
    // ---- up to 32 undecided pairs: full classification, then the bounds that make a clip pointless
    if (nm >= 32 || (done && nm > 0)) {
      const int cnt = min(nm, 32);
      nm -= cnt;
      bool clip = false;
      int p = 0;
      if ((int)lane < cnt) {
        p = s.qm[nm + lane];
        const RBox& rb = s.row[p >> 6];
        const RBox& cb = s.col[p & (kBlk - 1)];
        if (rbox_classify(rb, cb) == RB_ZERO) {
          if (0.0f > thr) atomicOr(reinterpret_cast<unsigned*>(&s.word[p >> 6]) + ((p >> 5) & 1), 1u << (p & 31));
        } else {
          // the sweep only needs "IoU > thr": no clip for a pair whose IoU provably cannot exceed it
          clip = !rbox_nms_cannot_exceed(rb, cb, thr);
        }
      }
      const unsigned bal = __ballot_sync(0xffffffffu, clip);
      if (clip) s.qc[nq + __popc(bal & lt)] = (uint16_t)p;
      nq += __popc(bal);
      __syncwarp();
    }
    // ---- up to 32 pairs to clip, one per lane: candidate points in registers, general routine for degenerate pairs
    if (nq >= 32 || (done && nm == 0 && nq > 0)) {
      const int cnt = min(nq, 32);
      nq -= cnt;
      if ((int)lane < cnt) {
        const int p = s.qc[nq + lane];
        const RBox& rb = s.row[p >> 6];
        const RBox& cb = s.col[p & (kBlk - 1)];
        bool ok;
        float v = rbox_iou_clip_try(rb, cb, s.pts + lane, 32, ok);
        if (!ok) v = nms_clip_general(rb, cb);
        if (v > thr) atomicOr(reinterpret_cast<unsigned*>(&s.word[p >> 6]) + ((p >> 5) & 1), 1u << (p & 31));
      }
      __syncwarp();
    }
    if (done && nm == 0 && nq == 0) break;
  }
  __syncwarp();
}

// linear index over the upper triangle (row-major, diagonal included) of a cb x cb tile grid
__device__ __forceinline__ void decode_upper(long long t, int cb, int& rb, int& cbk) {
  // row r starts at r*cb - r(r-1)/2
  // (a float estimate; the two loops below make it exact)
  const float fcb = (float)cb + 0.5f;
  int r = (int)floorf(fcb - sqrtf(fmaxf(fcb * fcb - 2.0f * (float)t, 0.0f)));
  if (r < 0) r = 0;
  if (r > cb - 1) r = cb - 1;
  while (r > 0 && (long long)r * cb - (long long)r * (r - 1) / 2 > t) --r;
  while (r < cb - 1 && (long long)(r + 1) * cb - (long long)(r + 1) * r / 2 <= t) ++r;
  rb = r;
  cbk = r + (int)(t - ((long long)r * cb - (long long)r * (r - 1) / 2));
}

// ------------------------------------------------------------------------------------------------
// generic path
// ------------------------------------------------------------------------------------------------
__global__ void nms_gather_keys_kernel(const float* __restrict__ scores, int64_t stride, int n,
                                       float* __restrict__ keys, int* __restrict__ vals) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { keys[i] = scores[(int64_t)i * stride]; vals[i] = i; }
}

__global__ void nms_gather_prep_kernel(const float* __restrict__ dets, int64_t stride,
                                       const float* __restrict__ labels, const int* __restrict__ order,
                                       int n, RBox* __restrict__ boxes, float* __restrict__ lab_sorted) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const int src = order[i];
    const float* d = dets + (int64_t)src * stride;
    RBox b;
    rbox_prep(d[0], d[1], d[2], d[3], d[4], b);
    boxes[i] = b;
    if (labels) lab_sorted[i] = labels[src];
  }
}

__global__ void __launch_bounds__(kTileThreads)
nms_mask_kernel(const RBox* __restrict__ boxes, const float* __restrict__ labels, int n, int cb, long long tiles,
                float thr, unsigned long long* __restrict__ mask) {
  __shared__ WarpTileSmem sw[kTileWarps];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long t = (long long)blockIdx.x * kTileWarps + wid;        // one upper-triangle tile per warp
  if (t >= tiles) return;
  WarpTileSmem& s = sw[wid];
  int rb, cbk;
  decode_upper(t, cb, rb, cbk);
  const int nr = min(kBlk, n - rb * kBlk), nc = min(kBlk, n - cbk * kBlk);
  mask_tile_warp(s, boxes + (size_t)rb * kBlk, boxes + (size_t)cbk * kBlk,
                 labels ? labels + (size_t)rb * kBlk : nullptr, labels ? labels + (size_t)cbk * kBlk : nullptr,
                 nr, nc, rb == cbk, thr);
  for (int r = lane; r < nr; r += 32) mask[((size_t)rb * kBlk + r) * cb + cbk] = s.word[r];
}

// Greedy sweep of one score-ordered segment of n boxes.  mask row stride = ld words; only words
// j >= row/64 of a row are ever read.  Writes kept positions (0..n-1, ascending) through `emit`.
// s_remv, s_kw: cb words of shared memory each.  Must be called by all kSweepThreads threads of the CTA.
template <class Emit>
__device__ __forceinline__ int sweep_segment(const unsigned long long* __restrict__ mask, int n, int ld,
                                             unsigned long long* s_remv, unsigned long long* s_kw,
                                             Emit emit) {
  static_assert(kSweepThreads == 1024, "the column reduction below transposes a 32 x 32 block of words");
  __shared__ unsigned long long s_part[32][33];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int cb = (n + kBlk - 1) / kBlk;
  for (int j = tid; j < cb; j += kSweepThreads) s_remv[j] = 0ull;
  // The sweep is a chain of cb dependent steps, each of them two global-load latencies long if done naively
  // (diagonal words, then the kept rows).  Neither load depends on the outcome of the step: the diagonal words of
  // block b + 1 are requested before block b is resolved, and every warp requests the later words of ITS two rows
  // of block b while warp 0 resolves it, and only masks them with the keep bits afterwards.
  unsigned long long dlo = 0ull, dhi = 0ull;         // warp 0: diagonal words of the current block, rows lane / lane + 32
  if (warp == 0 && cb > 0) {
    if (lane < n) dlo = mask[(size_t)lane * ld];
    if (lane + 32 < n) dhi = mask[(size_t)(lane + 32) * ld];
  }
  __syncthreads();
  int total = 0;
  for (int b = 0; b < cb; ++b) {
    const int nb = min(kBlk, n - b * kBlk);
    const int ra = b * kBlk + 2 * warp, rbb = ra + 1;   // this warp's rows of block b
    const int j0 = b + 1 + lane, j1 = j0 + 32;
    unsigned long long va0 = 0ull, va1 = 0ull, vb0 = 0ull, vb1 = 0ull;
    if (ra < n) {
      const unsigned long long* pa = mask + (size_t)ra * ld;
      if (j0 < cb) va0 = pa[j0];
      if (j1 < cb) va1 = pa[j1];
    }
    if (rbb < n) {
      const unsigned long long* pb = mask + (size_t)rbb * ld;
      if (j0 < cb) vb0 = pb[j0];
      if (j1 < cb) vb1 = pb[j1];
    }
    if (warp == 0) {
      unsigned long long nlo = 0ull, nhi = 0ull;       // diagonal words of block b + 1
      const int rlo = (b + 1) * kBlk + lane, rhi = rlo + 32;
      if (rlo < n) nlo = mask[(size_t)rlo * ld + b + 1];
      if (rhi < n) nhi = mask[(size_t)rhi * ld + b + 1];
      unsigned long long rem = s_remv[b];
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const unsigned long long w = __shfl_sync(0xffffffffu, dlo, i);
        if (!((rem >> i) & 1ull)) rem |= w;
      }
#pragma unroll
      for (int i = 0; i < 32; ++i) {
        const unsigned long long w = __shfl_sync(0xffffffffu, dhi, i);
        if (!((rem >> (32 + i)) & 1ull)) rem |= w;
      }
      const unsigned long long valid = (nb == kBlk) ? ~0ull : ((1ull << nb) - 1ull);
      const unsigned long long kw = ~rem & valid;
      if (lane == 0) s_kw[b] = kw;                     // (the survivors are written out after the chain, in parallel)
      dlo = nlo; dhi = nhi;
    }
    __syncthreads();
    const unsigned long long kw = s_kw[b];
    total += __popcll(kw);
    // OR the kept rows of this block into the removed-bitmap of all later blocks.  Every warp holds, per lane, the
    // words of ITS two rows for columns b + 1 + lane (and + 32); the OR over the 32 warps goes through a padded
    // 32 x 32 transpose in shared memory and a warp reduction -- one writer per column, no atomics (32 warps
    // hammering the same 64-bit shared-memory words with atomicOr was most of the sweep's time).
    if (b + 1 < cb) {
      const bool ka = (kw >> (2 * warp)) & 1ull, kb2 = (kw >> (2 * warp + 1)) & 1ull;
      const unsigned long long a0 = (ka ? va0 : 0ull) | (kb2 ? vb0 : 0ull);
      const unsigned long long a1 = (ka ? va1 : 0ull) | (kb2 ? vb1 : 0ull);
      s_part[warp][lane] = a0;
      __syncthreads();
      {
        const unsigned long long v = s_part[lane][warp];
        const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)v), hi = __reduce_or_sync(0xffffffffu, (unsigned)(v >> 32));
        if (lane == 0 && b + 1 + warp < cb) s_remv[b + 1 + warp] |= ((unsigned long long)hi << 32) | lo;
      }
      if (b + 1 + 32 < cb) {
        __syncthreads();
        s_part[warp][lane] = a1;
        __syncthreads();
        const unsigned long long v = s_part[lane][warp];
        const unsigned lo = __reduce_or_sync(0xffffffffu, (unsigned)v), hi = __reduce_or_sync(0xffffffffu, (unsigned)(v >> 32));
        if (lane == 0 && b + 1 + 32 + warp < cb) s_remv[b + 1 + 32 + warp] |= ((unsigned long long)hi << 32) | lo;
      }
      if (b + 1 + 64 < cb && (ka || kb2)) {              // (segments of more than ~4,200 boxes: the far columns)
        const unsigned long long* pa = mask + (size_t)ra * ld;
        const unsigned long long* pb = mask + (size_t)rbb * ld;
        for (int j = j1 + 32; j < cb; j += 32) {
          unsigned long long acc = 0ull;
          if (ka) acc |= pa[j];
          if (kb2) acc |= pb[j];
          if (acc) atomicOr(&s_remv[j], acc);
        }
      }
    }
    __syncthreads();
  }
  // emission: warp w writes the survivors of blocks w, w + 32, ...; its first output position is the number of
  // survivors in the blocks before
  for (int b = warp; b < cb; b += kSweepThreads / 32) {
    int before = 0;
    for (int j = lane; j < b; j += 32) before += __popcll(s_kw[j]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) before += __shfl_xor_sync(0xffffffffu, before, o);
    const unsigned long long kw = s_kw[b];
    if ((kw >> lane) & 1ull) emit(before + __popcll(kw & ((1ull << lane) - 1ull)), b * kBlk + lane);
    if ((kw >> (lane + 32)) & 1ull)
      emit(before + __popcll(kw & ((1ull << (lane + 32)) - 1ull)), b * kBlk + 32 + lane);
  }
  return total;
}

__global__ void __launch_bounds__(kSweepThreads)
nms_sweep_kernel(const unsigned long long* __restrict__ mask, const int* __restrict__ order, int n,
                 int64_t* __restrict__ keep_out, int32_t* __restrict__ num_keep) {
  extern __shared__ unsigned long long s_dyn[];
  const int cb = (n + kBlk - 1) / kBlk;
  int total = sweep_segment(mask, n, cb, s_dyn, s_dyn + cb,
                            [&](int pos, int sorted_idx) { keep_out[pos] = (int64_t)order[sorted_idx]; });
  if (threadIdx.x == 0) *num_keep = total;
}

struct NmsWorkspace {
  float* keys_in; float* keys_out; int* vals_in; int* vals_out; RBox* boxes; float* labels;
  unsigned long long* mask; void* cub_tmp; size_t cub_bytes; size_t total;
};

static size_t cub_sort_bytes(int64_t n) {
  size_t bytes = 0;
  cub::DeviceRadixSort::SortPairsDescending(nullptr, bytes, (const float*)nullptr, (float*)nullptr,
                                            (const int*)nullptr, (int*)nullptr, (int)n);
  return bytes;
}

static NmsWorkspace carve_nms(void* base, int64_t n) {
  NmsWorkspace w;
  const int64_t cb = ceil_div(n, kBlk);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return (char*)base + o; };
  w.keys_in = (float*)take(sizeof(float) * n);
  w.keys_out = (float*)take(sizeof(float) * n);
  w.vals_in = (int*)take(sizeof(int) * n);
  w.vals_out = (int*)take(sizeof(int) * n);
  w.boxes = (RBox*)take(sizeof(RBox) * n);
  w.labels = (float*)take(sizeof(float) * n);
  w.mask = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)n * cb);
  w.cub_bytes = cub_sort_bytes(n);
  w.cub_tmp = take(w.cub_bytes);
  w.total = off;
  return w;
}

// ------------------------------------------------------------------------------------------------
// fused multiclass path
// ------------------------------------------------------------------------------------------------
constexpr int kSelThreads = 1024;
constexpr int kSelItems = 6;                       // 1024 * 6 = 6144 boxes per image at most
constexpr int kMcMaxBoxes = kSelThreads * kSelItems;  // above it, the selection is a device-wide segmented sort
constexpr int kMcSweepMaxSmem = 200 * 1024;               // the sweep's two bitmaps: 16 bytes per 64 boxes
constexpr int kMcMaxSweepBoxes = kMcSweepMaxSmem / 16 * kBlk;   // 819,200 boxes per image

__global__ void mc_prep_kernel(const float* __restrict__ bboxes, int64_t total, RBox* __restrict__ out) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < total) {
    const float* d = bboxes + i * 5;
    RBox b;
    rbox_prep(d[0], d[1], d[2], d[3], d[4], b);
    out[i] = b;
  }
}

// Rank key of candidate box i: descending key order is descending score, equal scores in ascending box order.
// Never 0 (the low word is >= 2^32 - 2^30), so 0 can pad a sort.
__device__ __forceinline__ unsigned long long mc_rank_key(float sv, int i) {
  // -0.0 and +0.0 are equal scores (ordered by box, like every other tie): one key for both
  const unsigned u = sv == 0.0f ? 0u : __float_as_uint(sv);
  const unsigned ord = (u & 0x80000000u) ? ~u : (u | 0x80000000u);       // unsigned order == float order
  return ((unsigned long long)ord << 32) | (unsigned long long)(0xFFFFFFFFu - (unsigned)i);
}

__device__ __forceinline__ int mc_key_box(unsigned long long k) {
  return (int)(0xFFFFFFFFu - (unsigned)(k & 0xFFFFFFFFull));
}

// One CTA per (class, image): ordered selection of the boxes whose class score exceeds the
// threshold, stable descending sort by score, gather of the prepared boxes into the segment.
template <int ITEMS>
__device__ __forceinline__ void mc_select_sort_body(const float* __restrict__ sc, int n, int C, int c,
                                                    float thr, const RBox* __restrict__ prepped,
                                                    float* __restrict__ seg_score, int* __restrict__ seg_box,
                                                    RBox* __restrict__ seg_rbox, int* __restrict__ seg_count,
                                                    void* smem) {
  // Only a fraction of the boxes passes the threshold for a given class (a few hundred of 5,344 on average), so the
  // candidates are compacted first -- in box order, as 64-bit keys (order-preserving score bits . ~box index) -- and
  // only the next power of two above their count is sorted (bitonic, shared memory): descending score, equal scores
  // in ascending box order, exactly what the stable radix sort of all 6,144 slots produced at twice the cost.
  using Scan = cub::BlockScan<int, kSelThreads>;
  __shared__ typename Scan::TempStorage s_scan;
  __shared__ int s_cnt;
  unsigned long long* s_keys = reinterpret_cast<unsigned long long*>(smem);     // [kSelThreads * ITEMS]
  unsigned long long key[ITEMS];
  int local = 0;
#pragma unroll
  for (int j = 0; j < ITEMS; ++j) {
    const int i = threadIdx.x * ITEMS + j;
    key[j] = 0ull;
    if (i < n) {
      const float sv = sc[(int64_t)i * C + c];
      if (sv > thr) {
        key[j] = mc_rank_key(sv, i);
        ++local;
      }
    }
  }
  int offset = 0, cnt = 0;
  Scan(s_scan).ExclusiveSum(local, offset, cnt);
  if (threadIdx.x == 0) s_cnt = cnt;
  __syncthreads();
  cnt = s_cnt;
  int ns = 2;
  while (ns < cnt) ns <<= 1;                              // slots to sort (<= kSelThreads * ITEMS rounded up to 2^k)
  for (int i = cnt + (int)threadIdx.x; i < ns; i += kSelThreads) s_keys[i] = 0ull;      // padding sorts last
#pragma unroll
  for (int j = 0; j < ITEMS; ++j)
    if (key[j]) s_keys[offset++] = key[j];
  for (int size = 2; size <= ns; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int t = threadIdx.x; t < ns / 2; t += kSelThreads) {
        const int lo = 2 * t - (t & (stride - 1)), hi = lo + stride;
        const unsigned long long a = s_keys[lo], d = s_keys[hi];
        if ((a < d) == ((lo & size) == 0)) { s_keys[lo] = d; s_keys[hi] = a; }
      }
    }
  }
  __syncthreads();
  for (int rank = threadIdx.x; rank < cnt; rank += kSelThreads) {
    const int box = mc_key_box(s_keys[rank]);
    seg_score[rank] = sc[(int64_t)box * C + c];           // (the input's bits: the key has no sign of zero)
    seg_box[rank] = box;
    seg_rbox[rank] = prepped[box];
  }
  if (threadIdx.x == 0) *seg_count = cnt;
}

template <int ITEMS>
__global__ void __launch_bounds__(kSelThreads)
mc_select_sort_kernel(const float* __restrict__ scores, int n, int C, float thr,
                      const RBox* __restrict__ prepped, float* __restrict__ seg_score,
                      int* __restrict__ seg_box, RBox* __restrict__ seg_rbox, int* __restrict__ seg_count) {
  extern __shared__ __align__(16) unsigned char s_sort[];
  const int c = blockIdx.x, b = blockIdx.y;
  const size_t seg = (size_t)b * C + c;
  mc_select_sort_body<ITEMS>(scores + (size_t)b * n * C, n, C, c, thr, prepped + (size_t)b * n,
                             seg_score + seg * n, seg_box + seg * n, seg_rbox + seg * n, seg_count + seg,
                             s_sort);
}

// Selection for n > kMcMaxBoxes, in three steps that produce what mc_select_sort_body produces:
//   mc_key_kernel      one thread per (image, box, class) score: the candidate's rank key is appended to its segment's
//                      slice [seg * n, seg * n + n) of `keys` (warp-aggregated atomics on seg_count, which must be
//                      zero on entry).  The append order varies from run to run; the keys of a segment are unique,
//                      so their sorted order does not.
//   cub::DeviceSegmentedRadixSort, descending, over [seg * n, seg * n + seg_count[seg]) (end offsets read on the
//                      device: no host round trip).
//   mc_gather_kernel   one thread per (segment, rank < count): the input's score bits, the box, the prepared box.
__global__ void mc_key_kernel(const float* __restrict__ scores, int n, int C, float thr,
                              unsigned long long* __restrict__ keys, int* __restrict__ seg_count) {
  const int b = blockIdx.y;
  const int e = blockIdx.x * blockDim.x + threadIdx.x;       // < n * C (< 2^31, checked by the host)
  const int i = e / C, c = e - i * C;
  const bool in = e < n * C;
  const float sv = in ? scores[((size_t)b * n + i) * C + c] : 0.0f;
  const bool cand = in && sv > thr;
  const unsigned cm = __ballot_sync(0xffffffffu, cand);
  if (!cand) return;
  const int seg = b * C + c;
  const unsigned peers = __match_any_sync(cm, seg);
  const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
  int base = 0;
  if (lane == leader) base = atomicAdd(&seg_count[seg], __popc(peers));
  base = __shfl_sync(peers, base, leader);
  keys[(size_t)seg * n + base + __popc(peers & ((1u << lane) - 1u))] = mc_rank_key(sv, i);
}

__global__ void mc_gather_kernel(const float* __restrict__ scores, int n, int C,
                                 const unsigned long long* __restrict__ keys, const int* __restrict__ seg_count,
                                 const RBox* __restrict__ prepped, float* __restrict__ seg_score,
                                 int* __restrict__ seg_box, RBox* __restrict__ seg_rbox) {
  const int c = blockIdx.y, b = blockIdx.z;
  const size_t seg = (size_t)b * C + c;
  const int rank = blockIdx.x * blockDim.x + threadIdx.x;
  if (rank >= seg_count[seg]) return;
  const size_t o = seg * n + rank;
  const int box = mc_key_box(keys[o]);
  seg_score[o] = scores[((size_t)b * n + box) * C + c];     // (the input's bits: the key has no sign of zero)
  seg_box[o] = box;
  seg_rbox[o] = prepped[(size_t)b * n + box];
}

struct McSegBegin {
  int n;
  __host__ __device__ int operator()(int s) const { return s * n; }
};
struct McSegEnd {
  int n;
  const int* count;
  __host__ __device__ int operator()(int s) const { return s * n + count[s]; }
};
using McBeginIt = thrust::transform_iterator<McSegBegin, thrust::counting_iterator<int>>;
using McEndIt = thrust::transform_iterator<McSegEnd, thrust::counting_iterator<int>>;

static cudaError_t mc_segmented_sort(void* tmp, size_t& tmp_bytes, cub::DoubleBuffer<unsigned long long>& keys, int n,
                                     int S, const int* seg_count, cudaStream_t st) {
  const thrust::counting_iterator<int> s0(0);
  return cub::DeviceSegmentedRadixSort::SortKeysDescending(tmp, tmp_bytes, keys, S * n, S,
                                                           McBeginIt(s0, McSegBegin{n}),
                                                           McEndIt(s0, McSegEnd{n, seg_count}), 0, 64, st);
}

// exclusive prefix of the per-segment tile counts (upper triangle incl. diagonal)
__global__ void mc_tile_scan_kernel(const int* __restrict__ seg_count, int S, long long* __restrict__ tile_off) {
  __shared__ long long s_part[1024];
  const int tid = threadIdx.x;
  const int per = (S + blockDim.x - 1) / blockDim.x;
  long long sum = 0;
  for (int k = 0; k < per; ++k) {
    const int s = tid * per + k;
    if (s < S) { const long long cb = (seg_count[s] + kBlk - 1) / kBlk; sum += cb * (cb + 1) / 2; }
  }
  s_part[tid] = sum;
  __syncthreads();
  if (tid == 0) {
    long long run = 0;
    for (int t = 0; t < (int)blockDim.x; ++t) { const long long v = s_part[t]; s_part[t] = run; run += v; }
    tile_off[S] = run;
  }
  __syncthreads();
  long long run = s_part[tid];
  for (int k = 0; k < per; ++k) {
    const int s = tid * per + k;
    if (s < S) {
      tile_off[s] = run;
      const long long cb = (seg_count[s] + kBlk - 1) / kBlk;
      run += cb * (cb + 1) / 2;
    }
  }
}

// Persistent: every WARP of the grid walks the global tile list (all segments' upper triangles) with a stride.
__global__ void __launch_bounds__(kTileThreads)
mc_mask_kernel(const RBox* __restrict__ seg_rbox, const int* __restrict__ seg_count,
               const long long* __restrict__ tile_off, int S, int n, int ld, float thr,
               unsigned long long* __restrict__ mask) {
  __shared__ WarpTileSmem sw[kTileWarps];
  const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
  WarpTileSmem& s = sw[wid];
  const long long total = tile_off[S];
  const long long nwarps = (long long)gridDim.x * kTileWarps;
  for (long long t = (long long)blockIdx.x * kTileWarps + wid; t < total; t += nwarps) {
    int lo = 0, hi = S - 1;                 // last segment whose offset <= t
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (tile_off[mid] <= t) lo = mid; else hi = mid - 1;
    }
    const int seg = lo;
    const int k = seg_count[seg];
    const int cb = (k + kBlk - 1) / kBlk;
    int rb, cbk;
    decode_upper(t - tile_off[seg], cb, rb, cbk);
    const RBox* boxes = seg_rbox + (size_t)seg * n;
    const int nr = min(kBlk, k - rb * kBlk), nc = min(kBlk, k - cbk * kBlk);
    mask_tile_warp(s, boxes + rb * kBlk, boxes + cbk * kBlk, nullptr, nullptr, nr, nc, rb == cbk, thr);
    for (int r = lane; r < nr; r += 32) mask[((size_t)seg * n + (size_t)rb * kBlk + r) * ld + cbk] = s.word[r];
    __syncwarp();
  }
}

// One CTA per segment: sweep, then compact the survivors (still in descending-score order).
__global__ void __launch_bounds__(kSweepThreads)
mc_sweep_kernel(const unsigned long long* __restrict__ mask, const int* __restrict__ seg_count, int n, int ld,
                const float* __restrict__ seg_score, const int* __restrict__ seg_box,
                float* __restrict__ kept_score, int* __restrict__ kept_box, int* __restrict__ kept_count) {
  extern __shared__ unsigned long long s_dyn[];
  const size_t seg = blockIdx.x;
  const int k = seg_count[seg];
  const float* sc = seg_score + seg * n;
  const int* bx = seg_box + seg * n;
  float* ks = kept_score + seg * n;
  int* kb = kept_box + seg * n;
  int total = sweep_segment(mask + seg * (size_t)n * ld, k, ld, s_dyn, s_dyn + ld,
                            [&](int pos, int sorted_idx) { ks[pos] = sc[sorted_idx]; kb[pos] = bx[sorted_idx]; });
  if (threadIdx.x == 0) kept_count[seg] = total;
}

// Merge by rank: a survivor's output row is the number of survivors of the same image that precede
// it in (score desc, box asc, class asc) order = its own position in its class + one binary search
// per other class.
// Destinations of the packed form: up to 8 buffers [slots, K + 1, 8] fp32 (one per rank of a node: this rank's own
// and its peers' over NVLink), row k < K = (x, y, w, h, theta, score, label, 0), row K = (count, 0, ...).  Rows are
// 32 bytes so that a detection is two 16-byte stores per destination (NVLink likes wide stores).
constexpr int kMcMaxPeers = 8;
struct McPush {
  float* dst[kMcMaxPeers];
  int npeers;          // 0: plain outputs (dets_out / labels_out / num_out)
  int slot0;           // image b of this call goes to slot slot0 + b of every destination
  int K;               // rows per image (max_out)
};

__global__ void mc_emit_kernel(const float* __restrict__ bboxes, const float* __restrict__ kept_score,
                               const int* __restrict__ kept_box, const int* __restrict__ kept_count, int n,
                               int C, int64_t max_per_img, int64_t max_out, float* __restrict__ dets_out,
                               float* __restrict__ labels_out, int32_t* __restrict__ num_out, const McPush push) {
  const int c = blockIdx.y, b = blockIdx.z;
  const size_t seg0 = (size_t)b * C;
  const int kc = kept_count[seg0 + c];
  if (blockIdx.x == 0 && c == 0 && threadIdx.x == 0) {
    long long tot = 0;
    for (int cc = 0; cc < C; ++cc) tot += kept_count[seg0 + cc];
    long long lim = max_per_img < max_out ? max_per_img : max_out;
    const int32_t cnt = (int32_t)(tot < lim ? tot : lim);
    if (num_out) num_out[b] = cnt;
    for (int p = 0; p < push.npeers; ++p) {
      float4* o = reinterpret_cast<float4*>(push.dst[p] + ((size_t)(push.slot0 + b) * (push.K + 1) + push.K) * 8);
      o[0] = make_float4((float)cnt, 0.0f, 0.0f, 0.0f);
      o[1] = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    }
  }
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= kc) return;
  const float sv = kept_score[(seg0 + c) * n + r];
  const int box = kept_box[(seg0 + c) * n + r];
  long long rank = r;
  for (int cc = 0; cc < C; ++cc) {
    if (cc == c) continue;
    const int kk = kept_count[seg0 + cc];
    const float* ks = kept_score + (seg0 + cc) * n;
    const int* kb = kept_box + (seg0 + cc) * n;
    int lo = 0, hi = kk;                                  // first index with score <= sv
    while (lo < hi) { const int mid = (lo + hi) >> 1; if (ks[mid] > sv) lo = mid + 1; else hi = mid; }
    int cnt = lo;
    for (int q = lo; q < kk && ks[q] == sv; ++q)          // exact score ties across classes
      if (kb[q] < box || (kb[q] == box && cc < c)) ++cnt;
    rank += cnt;
  }
  const long long lim = max_per_img < max_out ? max_per_img : max_out;
  if (rank < lim) {
    const float* d = bboxes + ((size_t)b * n + box) * 5;
    const float d0 = d[0], d1 = d[1], d2 = d[2], d3 = d[3], d4 = d[4];
    if (dets_out) {
      float* o = dets_out + ((size_t)b * max_out + rank) * 6;
      o[0] = d0; o[1] = d1; o[2] = d2; o[3] = d3; o[4] = d4; o[5] = sv;
      labels_out[(size_t)b * max_out + rank] = (float)c;
    }
    // the detection exchange fused into the finaliser: the row goes straight into the packed buffer of every rank
    // (plain stores through NVLink peer mappings; a kernel boundary + the exchange's barrier publish them)
    const float4 lo = make_float4(d0, d1, d2, d3), hi = make_float4(d4, sv, (float)c, 0.0f);
    for (int p = 0; p < push.npeers; ++p) {
      float4* o = reinterpret_cast<float4*>(push.dst[p] + ((size_t)(push.slot0 + b) * (push.K + 1) + rank) * 8);
      o[0] = lo;
      o[1] = hi;
    }
  }
}

struct McWorkspace {
  RBox* prepped; float* seg_score; int* seg_box; RBox* seg_rbox; int* seg_count; long long* tile_off;
  unsigned long long* mask; float* kept_score; int* kept_box; int* kept_count;
  unsigned long long* keys[2]; void* sort_tmp; size_t sort_bytes;       // n > kMcMaxBoxes only
  size_t total;
};

// The mask, [B * C][n][ceil(n / 64)] words, dominates: for B = 8 and C = 15, 0.68 GB at n = 6,720 and 7.1 GB at
// n = 21,824.  Above kMcMaxBoxes two [B * C][n] key buffers and the segmented sort's scratch are added.
static McWorkspace carve_mc(void* base, int64_t n, int64_t C, int64_t B) {
  McWorkspace w;
  const int64_t S = B * C, ld = ceil_div(n, kBlk);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return (char*)base + o; };
  w.prepped = (RBox*)take(sizeof(RBox) * B * n);
  w.seg_score = (float*)take(sizeof(float) * S * n);
  w.seg_box = (int*)take(sizeof(int) * S * n);
  w.seg_rbox = (RBox*)take(sizeof(RBox) * S * n);
  w.seg_count = (int*)take(sizeof(int) * S);
  w.tile_off = (long long*)take(sizeof(long long) * (S + 1));
  w.mask = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)S * n * ld);
  w.kept_score = (float*)take(sizeof(float) * S * n);
  w.kept_box = (int*)take(sizeof(int) * S * n);
  w.kept_count = (int*)take(sizeof(int) * S);
  w.keys[0] = w.keys[1] = nullptr;
  w.sort_tmp = nullptr;
  w.sort_bytes = 0;
  if (n > kMcMaxBoxes && S * n < (1ll << 31) - 256) {           // (larger S * n is refused by multiclass_impl)
    w.keys[0] = (unsigned long long*)take(sizeof(unsigned long long) * S * n);
    w.keys[1] = (unsigned long long*)take(sizeof(unsigned long long) * S * n);
    cub::DoubleBuffer<unsigned long long> db(nullptr, nullptr);
    mc_segmented_sort(nullptr, w.sort_bytes, db, (int)n, (int)S, nullptr, 0);
    w.sort_tmp = take(w.sort_bytes);
  }
  w.total = off;
  return w;
}

template <int ITEMS>
static cudaError_t launch_select_sort(dim3 grid, cudaStream_t st, const float* scores, int n, int C, float thr,
                                      const McWorkspace& w) {
  size_t slots = 2;                                      // (the bitonic network sorts a power-of-two slot count)
  while (slots < (size_t)kSelThreads * ITEMS) slots <<= 1;
  const size_t smem = sizeof(unsigned long long) * slots;
  auto kern = mc_select_sort_kernel<ITEMS>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  kern<<<grid, kSelThreads, smem, st>>>(scores, n, C, thr, w.prepped, w.seg_score, w.seg_box, w.seg_rbox,
                                        w.seg_count);
  return cudaGetLastError();
}

}  // namespace s2a

extern "C" size_t s2a_nms_rotated_workspace_bytes(int64_t n) {
  if (n <= 0) return 256;
  return s2a::carve_nms(nullptr, n).total;
}

extern "C" int s2a_nms_rotated(const float* dets, int64_t det_stride, const float* scores,
                               int64_t score_stride, const float* labels, int64_t n, float iou_threshold,
                               int64_t* keep_out, int32_t* num_keep_out, void* workspace,
                               size_t workspace_bytes, void* stream) {
  using namespace s2a;
  cudaStream_t st = (cudaStream_t)stream;
  S2A_CHECK_ARG(n >= 0 && n < (1ll << 30), "nms_rotated: n (%lld) out of range", (long long)n);
  S2A_CHECK_ARG(num_keep_out != nullptr, "nms_rotated: num_keep_out is null");
  if (n == 0) {
    S2A_CUDA_OK(cudaMemsetAsync(num_keep_out, 0, sizeof(int32_t), st));
    return S2A_OK;
  }
  S2A_CHECK_ARG(dets && scores && keep_out && workspace, "nms_rotated: null pointer");
  S2A_CHECK_ARG(det_stride >= 5 && score_stride >= 1, "nms_rotated: bad strides (%lld, %lld)",
                (long long)det_stride, (long long)score_stride);
  NmsWorkspace w = carve_nms(workspace, n);
  if (workspace_bytes < w.total) {
    set_error("nms_rotated: workspace too small (%zu < %zu bytes)", workspace_bytes, w.total);
    return S2A_ERR_WORKSPACE;
  }
  const int ni = (int)n;
  const int cb = (int)ceil_div(n, kBlk);
  const int tb = 256, gb = (int)ceil_div(n, tb);
  nms_gather_keys_kernel<<<gb, tb, 0, st>>>(scores, score_stride, ni, w.keys_in, w.vals_in);
  S2A_LAUNCH_OK("nms_gather_keys_kernel");
  size_t cub_bytes = w.cub_bytes;
  S2A_CUDA_OK(cub::DeviceRadixSort::SortPairsDescending(w.cub_tmp, cub_bytes, w.keys_in, w.keys_out, w.vals_in,
                                                        w.vals_out, ni, 0, 32, st));
  nms_gather_prep_kernel<<<gb, tb, 0, st>>>(dets, det_stride, labels, w.vals_out, ni, w.boxes, w.labels);
  S2A_LAUNCH_OK("nms_gather_prep_kernel");
  const long long tiles = (long long)cb * (cb + 1) / 2;
  S2A_CHECK_ARG(tiles < (1ll << 31), "nms_rotated: too many tiles");
  nms_mask_kernel<<<(unsigned)ceil_div(tiles, kTileWarps), kTileThreads, 0, st>>>(w.boxes, labels ? w.labels : nullptr, ni, cb,
                                                                                  (long long)tiles, iou_threshold, w.mask);
  S2A_LAUNCH_OK("nms_mask_kernel");
  const size_t smem = 2 * sizeof(unsigned long long) * (size_t)cb;
  S2A_CHECK_ARG(smem <= 200 * 1024, "nms_rotated: n too large for the single-CTA sweep");
  if (smem > 48 * 1024)
    S2A_CUDA_OK(cudaFuncSetAttribute(nms_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nms_sweep_kernel<<<1, kSweepThreads, smem, st>>>(w.mask, w.vals_out, ni, keep_out, num_keep_out);
  S2A_LAUNCH_OK("nms_sweep_kernel");
  return S2A_OK;
}

extern "C" size_t s2a_multiclass_nms_rotated_workspace_bytes(int64_t n, int64_t num_classes, int64_t batch) {
  if (n <= 0 || num_classes <= 0 || batch <= 0) return 256;
  return s2a::carve_mc(nullptr, n, num_classes, batch).total;
}

namespace s2a {
static int multiclass_impl(const float* bboxes, const float* scores, int64_t n, int64_t num_classes, int64_t batch,
                           float score_thr, float iou_thr, int64_t max_per_img, float* dets_out, float* labels_out,
                           int32_t* num_out, int64_t max_out, void* workspace, size_t workspace_bytes, void* stream,
                           const McPush& push);
}

extern "C" int s2a_multiclass_nms_rotated(const float* bboxes, const float* scores, int64_t n,
                                          int64_t num_classes, int64_t batch, float score_thr, float iou_thr,
                                          int64_t max_per_img, float* dets_out, float* labels_out,
                                          int32_t* num_out, int64_t max_out, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(num_out != nullptr || batch == 0, "multiclass_nms_rotated: num_out is null");
  S2A_CHECK_ARG((dets_out && labels_out) || batch == 0 || n == 0 || num_classes == 0 || max_out == 0 || max_per_img <= 0,
                "multiclass_nms_rotated: null pointer");
  McPush push{};
  return multiclass_impl(bboxes, scores, n, num_classes, batch, score_thr, iou_thr, max_per_img, dets_out, labels_out,
                         num_out, max_out, workspace, workspace_bytes, stream, push);
}

extern "C" int s2a_multiclass_nms_rotated_packed(const float* bboxes, const float* scores, int64_t n, int64_t num_classes,
                                                 int64_t batch, float score_thr, float iou_thr, int64_t max_per_img,
                                                 float* const* dests, int ndests, int64_t slot0, int64_t max_out,
                                                 void* workspace, size_t workspace_bytes, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(dests != nullptr && ndests >= 1 && ndests <= kMcMaxPeers, "multiclass_nms_rotated_packed: 1..%d destinations",
                kMcMaxPeers);
  S2A_CHECK_ARG(slot0 >= 0 && max_out > 0 && max_out < (1ll << 30), "multiclass_nms_rotated_packed: bad slot / max_out");
  McPush push{};
  push.npeers = ndests; push.slot0 = (int)slot0; push.K = (int)max_out;
  for (int p = 0; p < ndests; ++p) {
    S2A_CHECK_ARG(dests[p] != nullptr, "multiclass_nms_rotated_packed: null destination");
    push.dst[p] = dests[p];
  }
  return multiclass_impl(bboxes, scores, n, num_classes, batch, score_thr, iou_thr, max_per_img, nullptr, nullptr, nullptr,
                         max_out, workspace, workspace_bytes, stream, push);
}

namespace s2a {
__global__ void mc_zero_counts_kernel(int32_t* num_out, int batch, const McPush push) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  if (num_out) num_out[b] = 0;
  for (int p = 0; p < push.npeers; ++p) {
    float* o = push.dst[p] + ((size_t)(push.slot0 + b) * (push.K + 1) + push.K) * 8;
    for (int e = 0; e < 8; ++e) o[e] = 0.0f;
  }
}

static int multiclass_impl(const float* bboxes, const float* scores, int64_t n, int64_t num_classes, int64_t batch,
                           float score_thr, float iou_thr, int64_t max_per_img, float* dets_out, float* labels_out,
                           int32_t* num_out, int64_t max_out, void* workspace, size_t workspace_bytes, void* stream,
                           const McPush& push) {
  cudaStream_t st = (cudaStream_t)stream;
  S2A_CHECK_ARG(n >= 0 && num_classes >= 0 && batch >= 0, "multiclass_nms_rotated: negative size");
  if (batch == 0) return S2A_OK;
  if (n == 0 || num_classes == 0 || max_out == 0 || max_per_img <= 0) {
    mc_zero_counts_kernel<<<(unsigned)ceil_div(batch, 128), 128, 0, st>>>(num_out, (int)batch, push);
    S2A_LAUNCH_OK("mc_zero_counts_kernel");
    return S2A_OK;
  }
  S2A_CHECK_ARG(bboxes && scores && workspace, "multiclass_nms_rotated: null pointer");
  S2A_CHECK_ARG(max_out > 0, "multiclass_nms_rotated: max_out must be positive");
  S2A_CHECK_ARG(n < (1ll << 30), "multiclass_nms_rotated: n (%lld) out of range", (long long)n);
  if (!(iou_thr >= 0.0f)) {
    set_error("multiclass_nms_rotated: class-segmented path needs iou_thr >= 0 (got %g)", (double)iou_thr);
    return S2A_ERR_UNSUPPORTED;
  }
  S2A_CHECK_ARG(num_classes <= 65535 && batch <= 65535, "multiclass_nms_rotated: classes/batch must be <= 65535");
  // the per-segment sweep keeps two bitmaps of ceil(n / 64) words in shared memory
  const size_t smem = 2 * sizeof(unsigned long long) * (size_t)ceil_div(n, kBlk);
  if (smem > kMcSweepMaxSmem) {
    set_error("multiclass_nms_rotated: n (%lld) above %d boxes per image, the most the per-class sweep holds in "
              "shared memory", (long long)n, kMcMaxSweepBoxes);
    return S2A_ERR_UNSUPPORTED;
  }
  if (n > kMcMaxBoxes && batch * num_classes * n >= (1ll << 31) - 256) {
    set_error("multiclass_nms_rotated: batch * classes * n (%lld) must be below 2^31 - 256 above %d boxes per image",
              (long long)(batch * num_classes * n), kMcMaxBoxes);
    return S2A_ERR_UNSUPPORTED;
  }
  McWorkspace w = carve_mc(workspace, n, num_classes, batch);
  if (workspace_bytes < w.total) {
    set_error("multiclass_nms_rotated: workspace too small (%zu < %zu bytes)", workspace_bytes, w.total);
    return S2A_ERR_WORKSPACE;
  }
  const int ni = (int)n, C = (int)num_classes, B = (int)batch, S = B * C;
  const int ld = (int)ceil_div(n, kBlk);
  mc_prep_kernel<<<(unsigned)ceil_div(batch * n, 256), 256, 0, st>>>(bboxes, batch * n, w.prepped);
  S2A_LAUNCH_OK("mc_prep_kernel");
  if (ni <= kMcMaxBoxes) {
    dim3 gsel(C, B);
    cudaError_t e;
    if (ni <= kSelThreads) e = launch_select_sort<1>(gsel, st, scores, ni, C, score_thr, w);
    else if (ni <= 2 * kSelThreads) e = launch_select_sort<2>(gsel, st, scores, ni, C, score_thr, w);
    else e = launch_select_sort<kSelItems>(gsel, st, scores, ni, C, score_thr, w);
    S2A_CUDA_OK(e);
  } else {
    S2A_CUDA_OK(cudaMemsetAsync(w.seg_count, 0, sizeof(int) * S, st));
    mc_key_kernel<<<dim3((unsigned)ceil_div(n * C, 256), B), 256, 0, st>>>(scores, ni, C, score_thr, w.keys[0],
                                                                           w.seg_count);
    S2A_LAUNCH_OK("mc_key_kernel");
    cub::DoubleBuffer<unsigned long long> db(w.keys[0], w.keys[1]);
    size_t sort_bytes = w.sort_bytes;
    S2A_CUDA_OK(mc_segmented_sort(w.sort_tmp, sort_bytes, db, ni, S, w.seg_count, st));
    mc_gather_kernel<<<dim3((unsigned)ceil_div(n, 256), C, B), 256, 0, st>>>(scores, ni, C, db.Current(), w.seg_count,
                                                                             w.prepped, w.seg_score, w.seg_box,
                                                                             w.seg_rbox);
    S2A_LAUNCH_OK("mc_gather_kernel");
  }
  // (thread 0 walks the per-thread partial sums serially: no more threads than segments)
  const int scan_threads = (int)std::min<int64_t>(1024, align_up((size_t)S, 32));
  mc_tile_scan_kernel<<<1, scan_threads, 0, st>>>(w.seg_count, S, w.tile_off);
  S2A_LAUNCH_OK("mc_tile_scan_kernel");
  mc_mask_kernel<<<sm_count() * 5, kTileThreads, 0, st>>>(w.seg_rbox, w.seg_count, w.tile_off, S, ni, ld, iou_thr,
                                                          w.mask);
  S2A_LAUNCH_OK("mc_mask_kernel");
  if (smem > 48 * 1024)
    S2A_CUDA_OK(cudaFuncSetAttribute(mc_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  mc_sweep_kernel<<<S, kSweepThreads, smem, st>>>(w.mask, w.seg_count, ni, ld, w.seg_score, w.seg_box,
                                                  w.kept_score, w.kept_box, w.kept_count);
  S2A_LAUNCH_OK("mc_sweep_kernel");
  dim3 gemit((unsigned)ceil_div(n, 256), C, B);
  mc_emit_kernel<<<gemit, 256, 0, st>>>(bboxes, w.kept_score, w.kept_box, w.kept_count, ni, C, max_per_img,
                                        max_out, dets_out, labels_out, num_out, push);
  S2A_LAUNCH_OK("mc_emit_kernel");
  return S2A_OK;
}
}  // namespace s2a

// ================================================================================================
// DOTA result-merging NMS on polygons, fp64 (SURVEY.md 8(f) row 4, second half)
//
// Replaces (reference): py_cpu_nms_poly_fast (DOTA_devkit/ResultMerge_multi_process.py:62-123) and the polygon IoU
// it calls per pair (DOTA_devkit/polyiou/csrc/polyiou.cpp:108-126, restated in poly_iou.cuh).  Same device
// structure as nms_rotated: sort by score, upper-triangular 64 x 64 suppression tiles (axis-aligned prefilter for
// every pair, polygon IoU for the listed survivors), one-CTA sweep.  The reference keeps a later box iff
// `value <= thresh`, so a NaN value suppresses -- the predicate here is !(value <= thresh).
// ================================================================================================
#include "poly_iou.cuh"

namespace s2a {

struct PolyBox { double p[8]; double hb[5]; };      // polygon, (x1, y1, x2, y2, area) of its axis-aligned box

__global__ void poly_keys_kernel(const double* __restrict__ dets, int64_t stride, int n, double* __restrict__ keys,
                                 int* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { keys[i] = dets[(size_t)i * stride + 8]; vals[i] = i; }
}

__global__ void poly_prep_kernel(const double* __restrict__ dets, int64_t stride, const int* __restrict__ order, int n,
                                 PolyBox* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* d = dets + (size_t)order[i] * stride;
  PolyBox b;
#pragma unroll
  for (int e = 0; e < 8; ++e) b.p[e] = d[e];
  b.hb[0] = fmin(fmin(b.p[0], b.p[2]), fmin(b.p[4], b.p[6]));
  b.hb[1] = fmin(fmin(b.p[1], b.p[3]), fmin(b.p[5], b.p[7]));
  b.hb[2] = fmax(fmax(b.p[0], b.p[2]), fmax(b.p[4], b.p[6]));
  b.hb[3] = fmax(fmax(b.p[1], b.p[3]), fmax(b.p[5], b.p[7]));
  // areas = (x2 - x1 + 1) * (y2 - y1 + 1)   (ResultMerge_multi_process.py:69)
  b.hb[4] = __dmul_rn(__dadd_rn(__dsub_rn(b.hb[2], b.hb[0]), 1.0), __dadd_rn(__dsub_rn(b.hb[3], b.hb[1]), 1.0));
  out[i] = b;
}

struct PolyTileSmem {
  PolyBox row[kBlk];
  PolyBox col[kBlk];
  uint16_t list[kBlk * kBlk];
  __align__(16) uint8_t flag[kBlk * kBlk];
  int count;
};

__global__ void __launch_bounds__(kMaskThreads)
poly_mask_kernel(const PolyBox* __restrict__ boxes, int n, int cb, double thr, unsigned long long* __restrict__ mask) {
  __shared__ PolyTileSmem s;
  int rb, cbk;
  decode_upper((long long)blockIdx.x, cb, rb, cbk);
  const int nr = min(kBlk, n - rb * kBlk), nc = min(kBlk, n - cbk * kBlk);
  const bool diag = rb == cbk;
  const int tid = threadIdx.x;
  reinterpret_cast<uint4*>(s.flag)[tid] = make_uint4(0u, 0u, 0u, 0u);
  // 2 x 64 boxes of 13 doubles, copied word by word (coalesced)
  {
    const double* src_r = reinterpret_cast<const double*>(boxes + (size_t)rb * kBlk);
    const double* src_c = reinterpret_cast<const double*>(boxes + (size_t)cbk * kBlk);
    double* dst_r = reinterpret_cast<double*>(s.row);
    double* dst_c = reinterpret_cast<double*>(s.col);
    for (int e = tid; e < nr * 13; e += kMaskThreads) dst_r[e] = src_r[e];
    for (int e = tid; e < nc * 13; e += kMaskThreads) dst_c[e] = src_c[e];
  }
  if (tid == 0) s.count = 0;
  __syncthreads();
  const int c = tid & (kBlk - 1), r0 = tid >> 6;
  const unsigned lane = tid & 31;
  for (int k = 0; k < kBlk / 4; ++k) {
    const int r = r0 + 4 * k;
    bool clip = false;
    if (r < nr && c < nc && (!diag || c > r)) {
      const double* hi = s.row[r].hb;
      const double* hj = s.col[c].hb;
      const double w = fmax(0.0, __dsub_rn(fmin(hi[2], hj[2]), fmax(hi[0], hj[0])));
      const double h = fmax(0.0, __dsub_rn(fmin(hi[3], hj[3]), fmax(hi[1], hj[1])));
      const double inter = __dmul_rn(w, h);
      const double ovr = __ddiv_rn(inter, __dsub_rn(__dadd_rn(hi[4], hj[4]), inter));
      if (ovr > 0.0) clip = true;                       // polygon IoU replaces the value (below)
      else if (!(ovr <= thr)) s.flag[r * kBlk + c] = 1;  // NaN, or a negative threshold
    }
    const unsigned bal = __ballot_sync(0xffffffffu, clip);
    if (bal) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&s.count, __popc(bal));
      base = __shfl_sync(0xffffffffu, base, 0);
      if (clip) s.list[base + __popc(bal & ((1u << lane) - 1u))] = (uint16_t)(r * kBlk + c);
    }
  }
  __syncthreads();
  const int cnt = s.count;
  for (int k = tid; k < cnt; k += kMaskThreads) {
    const int p = s.list[k];
    const double v = poly_iou(s.row[p >> 6].p, s.col[p & (kBlk - 1)].p);
    if (!(v <= thr)) s.flag[p] = 1;
  }
  __syncthreads();
  if (tid < nr) {
    const uint4* f = reinterpret_cast<const uint4*>(s.flag + tid * kBlk);
    unsigned long long w = 0ull;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const uint4 v = f[q];
      const uint32_t x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const uint32_t nib = (x[e] & 1u) | ((x[e] >> 7) & 2u) | ((x[e] >> 14) & 4u) | ((x[e] >> 21) & 8u);
        w |= (unsigned long long)nib << (16 * q + 4 * e);
      }
    }
    mask[((size_t)rb * kBlk + tid) * cb + cbk] = w;
  }
}

__global__ void poly_iou_pairs_kernel(const double* __restrict__ p, const double* __restrict__ q, int64_t n,
                                      double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = poly_iou(p + 8 * i, q + 8 * i);
}

struct PolyWorkspace {
  double* keys_in; double* keys_out; int* vals_in; int* vals_out; PolyBox* boxes; unsigned long long* mask;
  void* cub_tmp; size_t cub_bytes; size_t total;
};

static PolyWorkspace carve_poly(void* base, int64_t n) {
  PolyWorkspace w;
  const int64_t cb = ceil_div(n, kBlk);
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off = align_up(off + bytes, 256); return (char*)base + o; };
  w.keys_in = (double*)take(sizeof(double) * n);
  w.keys_out = (double*)take(sizeof(double) * n);
  w.vals_in = (int*)take(sizeof(int) * n);
  w.vals_out = (int*)take(sizeof(int) * n);
  w.boxes = (PolyBox*)take(sizeof(PolyBox) * n);
  w.mask = (unsigned long long*)take(sizeof(unsigned long long) * (size_t)n * cb);
  w.cub_bytes = 0;
  cub::DeviceRadixSort::SortPairsDescending(nullptr, w.cub_bytes, (const double*)nullptr, (double*)nullptr,
                                            (const int*)nullptr, (int*)nullptr, (int)n);
  w.cub_tmp = take(w.cub_bytes);
  w.total = off;
  return w;
}

}  // namespace s2a

extern "C" size_t s2a_poly_nms_workspace_bytes(int64_t n) {
  if (n <= 0) return 256;
  return s2a::carve_poly(nullptr, n).total;
}

extern "C" int s2a_poly_nms(const double* dets, int64_t det_stride, int64_t n, double thresh, int64_t* keep_out,
                            int32_t* num_keep_out, void* workspace, size_t workspace_bytes, void* stream) {
  using namespace s2a;
  cudaStream_t st = (cudaStream_t)stream;
  S2A_CHECK_ARG(n >= 0 && n < (1ll << 30), "poly_nms: n (%lld) out of range", (long long)n);
  S2A_CHECK_ARG(num_keep_out != nullptr, "poly_nms: num_keep_out is null");
  if (n == 0) {
    S2A_CUDA_OK(cudaMemsetAsync(num_keep_out, 0, sizeof(int32_t), st));
    return S2A_OK;
  }
  S2A_CHECK_ARG(dets && keep_out && workspace, "poly_nms: null pointer");
  S2A_CHECK_ARG(det_stride >= 9, "poly_nms: rows are 8 polygon coordinates + score (stride %lld)", (long long)det_stride);
  PolyWorkspace w = carve_poly(workspace, n);
  if (workspace_bytes < w.total) {
    set_error("poly_nms: workspace too small (%zu < %zu bytes)", workspace_bytes, w.total);
    return S2A_ERR_WORKSPACE;
  }
  const int ni = (int)n;
  const int cb = (int)ceil_div(n, kBlk);
  const int tb = 256, gb = (int)ceil_div(n, tb);
  poly_keys_kernel<<<gb, tb, 0, st>>>(dets, det_stride, ni, w.keys_in, w.vals_in);
  S2A_LAUNCH_OK("poly_keys_kernel");
  size_t cub_bytes = w.cub_bytes;
  S2A_CUDA_OK(cub::DeviceRadixSort::SortPairsDescending(w.cub_tmp, cub_bytes, w.keys_in, w.keys_out, w.vals_in,
                                                        w.vals_out, ni, 0, 64, st));
  poly_prep_kernel<<<gb, tb, 0, st>>>(dets, det_stride, w.vals_out, ni, w.boxes);
  S2A_LAUNCH_OK("poly_prep_kernel");
  const long long tiles = (long long)cb * (cb + 1) / 2;
  S2A_CHECK_ARG(tiles < (1ll << 31), "poly_nms: too many tiles");
  poly_mask_kernel<<<(unsigned)tiles, kMaskThreads, 0, st>>>(w.boxes, ni, cb, thresh, w.mask);
  S2A_LAUNCH_OK("poly_mask_kernel");
  const size_t smem = 2 * sizeof(unsigned long long) * (size_t)cb;
  S2A_CHECK_ARG(smem <= 200 * 1024, "poly_nms: n too large for the single-CTA sweep");
  if (smem > 48 * 1024)
    S2A_CUDA_OK(cudaFuncSetAttribute(nms_sweep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  nms_sweep_kernel<<<1, kSweepThreads, smem, st>>>(w.mask, w.vals_out, ni, keep_out, num_keep_out);
  S2A_LAUNCH_OK("nms_sweep_kernel");
  return S2A_OK;
}

extern "C" int s2a_poly_iou_pairs(const double* p, const double* q, int64_t n, double* out, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(n >= 0, "poly_iou_pairs: negative n");
  if (n == 0) return S2A_OK;
  S2A_CHECK_ARG(p && q && out, "poly_iou_pairs: null pointer");
  poly_iou_pairs_kernel<<<(unsigned)ceil_div(n, 128), 128, 0, (cudaStream_t)stream>>>(p, q, n, out);
  S2A_LAUNCH_OK("poly_iou_pairs_kernel");
  return S2A_OK;
}
