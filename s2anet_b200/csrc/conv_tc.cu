// conv_tc.cu -- AlignConv and ORConv2d as a tcgen05 implicit GEMM for sm_100a (bf16 / fp16 in,
// fp32 accumulate in TMEM).
//
// Replaces (reference): AlignConv.forward = get_offset + DeformConv + ReLU (models/alignconv.py:29-98,
// models/dcn/src/deform_conv_cuda.cpp:152-260, deform_conv_cuda_kernel.cu:83-114, 189-242) and
// ORConv2d.forward + RotationInvariantPooling (models/orn/modules/ORConv.py:77-82,
// models/orn/src/cuda/ActiveRotatingFilter_cuda.cu:19-46, models/orn/functions/
// rotation_invariant_pooling.py:19-27).
//
// GEMM view:  D[m, n] = sum_k A[m, k] * Wp[n, k]
//   m : output position (a CTA owns a 128-pixel patch = 128 rows = one UMMA M: 8 rows x 16 pixels for AlignConv,
//       16 rows x 8 pixels for the plain convs)
//   n : output channel (N = C_out <= 256, the whole channel dimension in one UMMA N)
//   k : (64-channel block, tap, channel-in-block) -- 64-wide k-blocks, K' = 9*C_in
//   A : never exists in global memory.  For AlignConv a[m, (cb,t,c)] is the bilinear sample of x at
//       the position the m-th refined anchor assigns to tap t (alignconv.py:29-86 collapsed with
//       deform_conv_cuda_kernel.cu:210-228); for ORConv it is the plain shifted pixel.
//   Wp: weights pre-packed to [C_out][K'] 16-bit (ARF rotation folded into the packing for ORConv).
//
// Warp roles (persistent CTA pairs; AlignConv 24 warps, plain conv / ORConv 8): 16 producer warps (AlignConv only)
// build the A tiles -- per (row, tap) recipe -> 8 LDS.128 from a TMA-fed shared-memory halo of the feature map ->
// packed 16-bit blend -> tcgen05.st straight into the A stage in TENSOR MEMORY; 4 epilogue warps (tcgen05.ld ->
// bias / ReLU / 8-way orientation max -> staging -> TMA store; they also build the gather recipes two tiles
// ahead); one TMA warp (weight k-blocks, AlignConv halos); for ORConv / plain convs one more warp that loads the
// OPERAND HALO -- one SWIZZLE_128B box per (tile, channel block) that the tensor core reads for all nine taps
// through shifted shared-memory descriptors; one MMA warp that allocates TMEM and issues
// tcgen05.mma.cta_group::2 (M = 256 across the pair, N = C_out, K = 16, kind::f16; A from shared memory or from
// TMEM) under elect.sync.  Stages are recycled through one full/empty
// mbarrier pair each; tcgen05.commit (multicast to both CTAs) releases a stage when its MMAs retire.
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "box_decode.cuh"
#include "common.cuh"

namespace s2a {

// -DS2A_TC_TIMELINE: in-kernel clock probes of the MMA warp (printed under S2A_TC_DEBUG=8); off in normal builds
#ifdef S2A_TC_TIMELINE
#define S2A_TL(...) __VA_ARGS__
#else
#define S2A_TL(...)
#endif

constexpr int TC_M = 128;                 // rows per tile (8 x 16 patch) = one UMMA M
constexpr int TC_PH = 8, TC_PW = 16;       // AlignConv tile: 8 rows x 16 pixels
// Plain conv / ORConv tile: 16 rows x 8 pixels.  Its A operand is read by the tensor core straight out of a
// shared-memory HALO of the feature map (18 rows x 16 pixels x 64 channels, SWIZZLE_128B, written by ONE TMA box per
// (tile, 64-channel block)): tap (dy, dx) is the same halo seen through a descriptor whose start address is shifted
// by (dy * 16 + dx) pixels.  An 8-row core group of the UMMA operand = 8 x-consecutive pixels of one halo row
// (8 x 128 B), consecutive groups are one halo row (16 pixels = 2048 B = SBO) apart; a row pitch of 16 pixels keeps
// every group on the same swizzle phase, and the shift by dx 128-byte lines goes into the descriptor's base-offset
// field.  Every pixel travels L2 -> shared memory 2.25 times per 3 x 3 conv instead of 9 times (the convs were
// bound by the L2 -> SM fabric: 11.6 TB/s of TMA loads with one box per tap).
constexpr int TC_PPH = 16, TC_PPW = 8;
constexpr int TC_PHALO_PITCH = 16, TC_PHALO_ROWS = TC_PPH + 2;
constexpr int TC_PHALO_BYTES = TC_PHALO_ROWS * TC_PHALO_PITCH * 128;   // 36,864 B (a multiple of 1024)
constexpr int TC_KB = 64;                 // k-block (elements) = 128 bytes of 16-bit data
constexpr int TC_OUT_CH = 32;              // channels per epilogue TMA store (64-byte rows, SWIZZLE_64B)
constexpr int TC_OUT_BYTES = TC_M * TC_OUT_CH * 2;    // 8 KB
constexpr int TC_OUT_BUFS = 3;             // staging buffers: the TMA store of chunk i-1 may still be reading when chunk i is staged

enum { TC_ALIGN = 0, TC_PLAIN = 1, TC_PLAIN_S = 2 };

// Per-mode pipeline shape.
//  * ORConv2d (TC_PLAIN) is fed entirely by TMA and bound by the tensor pipe: a CTA PAIR (cta_group::2, one
//    TPC) shares every weight k-block -- each CTA stages half of the C_out rows -- in a ring of 4 stages of two
//    k-blocks with one full/empty barrier pair per stage; the A operand is the shared-memory halo (see TC_PPW).
//  * AlignConv (TC_ALIGN) is bound by the bilinear gather, i.e. by LSU wavefronts: 4 corners x 128 B per
//    (row, k-block) = 512 wavefronts per k-block next to 512 tensor-pipe cycles.  Its feature-map reads go
//    through a TMA-fed shared-memory halo (two 39 KB buffers) instead of L1, and the blended A operand never
//    touches shared memory: the producers write it straight into TENSOR MEMORY (tcgen05.st, 8 stages of 32
//    columns next to ONE 256-column accumulator) and the MMA takes A from TMEM.  That removes the A-stage
//    stores (128 + bank-conflict wavefronts per k-block) from the LSU pipe and the A reads from the
//    tensor core's shared-memory port.  The producers are the bottleneck, so a single accumulator is enough
//    (they keep filling the 8 A stages while the epilogue drains it).  A and B keep separate rings.
template <int MODE> struct TcCfg;
// GROUPS = producer groups of 4 warps (group g fills k-blocks g, g + GROUPS, ...): 16 producer warps for AlignConv
// (its gather is latency-bound), none for the TMA-fed plain conv (256 threads, registers to spare).
// KPS = k-blocks per stage: the MMA warp pays ~200 cycles of wait / commit / bookkeeping per STAGE and the tensor
// pipe only holds two MMAs ahead, so the tensor-bound plain conv moves two k-blocks (8 MMAs) per stage.
// BROWS = weight rows (output channels) one CTA stages per k-block.
// TC_PLAIN_S is the plain conv for C_out = 32 (the 15- and 5-channel prediction convs, padded): a tcgen05.mma takes
// >= 69 cycles however small N is and the MMA warp pays a fixed few hundred cycles of waits / commits / bookkeeping
// per STAGE, so with 2 KB of weights per k-block a stage carries all NINE taps of a channel block (36 MMAs).
// NHALO = halo buffers (a power of two).  A halo is requested when the buffer it goes to is released, NHALO - 1
// channel blocks ahead of its first use: 2 buffers give the 512-cycle k-blocks of the wide conv 4,600 cycles for
// the load; the narrow conv runs a channel block in ~2,500 cycles -- less than the load takes -- and keeps 4.
template <> struct TcCfg<TC_ALIGN> { static constexpr int CG = 2, SA = 6, SB = 6, GROUPS = 4, KPS = 1, BROWS = 128, NHALO = 2; static constexpr bool UNIFIED = true; };
template <> struct TcCfg<TC_PLAIN> { static constexpr int CG = 2, SA = 4, SB = 4, GROUPS = 0, KPS = 2, BROWS = 128, NHALO = 2; static constexpr bool UNIFIED = true; };
template <> struct TcCfg<TC_PLAIN_S> { static constexpr int CG = 2, SA = 3, SB = 3, GROUPS = 0, KPS = 9, BROWS = 16, NHALO = 4; static constexpr bool UNIFIED = true; };
template <int MODE> constexpr int tc_threads() { return (TcCfg<MODE>::GROUPS * 4 + 8) * 32; }
constexpr int TC_MAX_STAGES = 8;
constexpr int TC_EPI_THREADS = 128;                   // 4 epilogue warps, one per TMEM lane quadrant
// warps: GROUPS x 4 producers | 4 epilogue | TMA | MMA | 2 idle (pad to a multiple of 4 warps)
constexpr int TC_ACC_STAGES = 2;                      // double-buffered accumulator: 2 x 256 TMEM columns
constexpr int TC_TMEM_COLS = 512;
constexpr int TC_MAX_HALOS = 4;
constexpr int TC_NBAR = 4 * TC_MAX_STAGES + 2 * TC_ACC_STAGES + 2 + 2 * TC_MAX_HALOS;   // + table full x 2, halo full/empty
constexpr int TC_MAX_LEVELS = 16;         // (two 8-level problems in one launch, see wsplit)
constexpr uint32_t kSpinLimit = 1u << 26;            // watchdog: trap instead of hanging the GPU

// AlignConv reads the feature map through a shared-memory HALO: for every (tile, 64-channel block) TMA loads
// the (8 + 2*3) x (16 + 2*3) pixel window around the tile once (39 KB, zero-filled outside the map, two
// buffers), and the nine taps of that channel block gather their bilinear corners from it with LDS.128 --
// fixed latency, no L1 tags, no misses.  Corners outside the window (large or far-shifted anchors) are read
// from global memory instead, per sample.
constexpr int TC_HALO = 3;
constexpr int TC_HW = TC_PW + 2 * TC_HALO, TC_HH = TC_PH + 2 * TC_HALO;      // 22 x 14 pixels
constexpr int TC_HALO_BYTES = TC_HW * TC_HH * TC_KB * 2;                      // 39,424 B per buffer

// One (row, tap) gather recipe, 12 bytes: the four bilinear weights already rounded to the 16-bit type, and
// `base`: bit 31 = "all corners are inside the halo window", bits 2..30 = index of the (clamped) top-left
// corner pixel -- inside the halo window if bit 31 is set, inside the image otherwise -- bit 0 = "right
// corners are one pixel further", bit 1 = "bottom corners are one row further".  Corners that fall outside
// the map keep a valid (clamped) address and get weight 0, which is the reference's rule
// (deform_conv_cuda_kernel.cu:97-108, :228).
struct __align__(4) TapSample { uint32_t base; uint32_t w01; uint32_t w23; };
constexpr uint32_t TC_IN_HALO = 0x80000000u;

struct TcLevel {
  const void* x;          // [B, H, W, C] 16-bit (channels_last)
  const float* anchors;   // [B, H, W, 5] (TC_ALIGN)
  const void* offsets;    // TC_ALIGN, generic deformable conv: [B, 18, H, W] offsets (dy, dx per tap) instead of anchors
  void* out;              // [B, H, W, Co] 16-bit
  void* pooled;           // [B, H, W, Co/8] 16-bit or null
  int H, W, tiles_x, tiles_y;
  int tile_begin;         // first global tile index of this level
  float stride;
  float* refine;          // FAM decode (conv_tc_kernel<TC_PLAIN, T, true>): [B, H, W, 5] fp32 refined anchors
};

struct TcParams {
  TcLevel lv[TC_MAX_LEVELS];
  const float* bias;      // [Co] fp32 or null
  // Two convolutions of the same shape class (C, C_out, kernel, ReLU) may share a launch: levels >= wsplit use the
  // second packed weight / bias.  One launch of 2 x 682 tile groups fills 74 CTA pairs to 97 % (19 rounds for 18.4),
  // two launches of 682 only to 92 % (10 rounds for 9.2 each).  The second problem starts at an even tile index, so a
  // CTA pair never mixes weights.
  const float* bias2;
  int wsplit;
  int nlevels, total_tiles;
  int B, C, Co;
  int ks;                 // TC_PLAIN: square kernel size, 1 or 3 (pad ks/2, stride 1); TC_ALIGN: 3
  int relu;
  int off_f32;            // generic deformable conv: the offsets are fp32 (else the activations' 16-bit type)
  int pos_round;          // ... and sampling positions / bilinear weights are rounded like the reference's scalar_t = half path
  int debug;              // timing experiments only (S2A_TC_DEBUG): 1 = no weight TMA after warm-up, 2 = no gather loads
  // TC_PLAIN, 1 x 1, "dgrad" epilogue (sc_tap >= 0): the accumulator tile is the column gradient of ONE tap,
  // col_grad[pixel, c] = sum_co grad_out[pixel, co] * W[co, c, tap]; instead of being stored it is scattered with the
  // bilinear weights of (pixel, tap) into grad_input (fp32 NHWC, red.global.add.v4.f32) and, optionally, contracted with
  // the corner differences of x into the offset gradient (deform_conv_cuda_kernel.cu:278-435).  Level 0 only.
  float* sc_gi;           // [B, H, W, Co] fp32, accumulated
  float* sc_goff;         // [B, 18, H, W] fp32, accumulated (+=), or null
  const void* sc_x;       // [B, H, W, Co] 16-bit (needed for sc_goff)
  const void* sc_off;     // [B, 18, H, W] offsets, fp32 or the 16-bit type
  int sc_off_f32;
  int sc_tap;             // -1: ordinary epilogue
  // TC_PLAIN, 1 x 1, FAM-decode epilogue (conv_tc_kernel<TC_PLAIN, T, true>): the first 5 output channels are the FAM
  // regression deltas; they are rounded to T exactly as the ordinary epilogue stores them and decoded against the grid
  // anchor (models/head.py:27-52) instead of being stored.
  float fd_scale, fd_angle, fd_lim;   // anchor scale, anchor angle, dw / dh clamp bound (rounded to T)
};

struct TileCoord { int lvl, b, ty0, tx0; };

// TMA descriptors: the packed weights, and (TC_PLAIN only) one 4-D NHWC map per level
struct TcMaps {
  CUtensorMap w[2];               // packed weights (second: levels >= wsplit)
  CUtensorMap x[TC_MAX_LEVELS];   // TC_PLAIN: A tiles are loaded from these
  CUtensorMap y[TC_MAX_LEVELS];   // outputs: the epilogue stores 8 x 16 x 32-channel boxes through these
};

template <int MODE> __host__ __device__ constexpr int tc_pw() { return MODE != 0 ? TC_PPW : TC_PW; }
template <int MODE> __host__ __device__ constexpr int tc_ph() { return MODE != 0 ? TC_PPH : TC_PH; }

template <int MODE>
__device__ __forceinline__ TileCoord decode_tile(const TcParams& p, int tile) {
  int l = 0;
#pragma unroll 1
  while (l + 1 < p.nlevels && tile >= p.lv[l + 1].tile_begin) ++l;
  const TcLevel& L = p.lv[l];
  int t = tile - L.tile_begin;
  const int tpi = L.tiles_x * L.tiles_y;
  TileCoord c;
  c.lvl = l;
  c.b = t / tpi;
  t -= c.b * tpi;
  c.ty0 = (t / L.tiles_x) * tc_ph<MODE>();
  c.tx0 = (t % L.tiles_x) * tc_pw<MODE>();
  return c;
}

// ---------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.shared::cta.b64 st, [%0];\n\t}" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("{\n\t.reg .b64 st;\n\tmbarrier.arrive.expect_tx.shared::cta.b64 st, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// non-blocking probe of a phase (mbarrier.test_wait never suspends the thread)
__device__ __forceinline__ bool mbar_test(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > kSpinLimit) {
      printf("s2a conv_tc: mbarrier wait timed out (block %d thread %d)\n", (int)blockIdx.x, (int)threadIdx.x);
      __trap();
    }
  }
}
// A try_wait costs the issuing thread ~150 cycles even when the phase is already complete, a test_wait ~40
// (tools/umma_bench2.cu): on the MMA warp's critical path, where the awaited phase is nearly always complete, probe
// first and fall back to the suspending wait only if it is not.
__device__ __forceinline__ void mbar_wait_likely_ready(uint32_t bar, uint32_t parity) {
  if (!mbar_test(bar, parity)) mbar_wait(bar, parity);
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// one lane of a fully converged warp (the compiler keeps warp-uniform operands of the tcgen05 / TMA instructions
// issued under it in uniform registers; issuing them from an `if (lane == 0)` region instead costs a
// per-instruction ELECT/R2UR "waterfall" loop)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
  return pred != 0;
}

// cluster helpers (CTA pair)
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_id_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%clusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_count_x() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%nclusterid.x;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `addr` (a shared::cta address of this CTA) inside CTA `rank` of the cluster
__device__ __forceinline__ uint32_t map_to_cta(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
// arrive on an mbarrier that may live in the peer CTA (shared::cluster address).  Default semantics
// (.release at CTA scope, as CUTLASS's ClusterBarrier::arrive(cta_id) does): the `.release.cluster` form
// compiles to MEMBAR.ALL.GPU + ERRBAR in front of the arrive, which cost the AlignConv producers ~15 % of
// their issue samples (ncu source view, profiles/r1_conv_tc_v8).  The data this arrive publishes is only ever
// read by the tensor core of the WRITING CTA (each SM reads its own A tile), after fence.proxy.async.
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}

// TMA loads.  `bar` is a shared::cluster address: with cta_group::2 the completion may be signalled on
// the leader CTA's barrier while the data lands in this CTA's shared memory.
template <int CG>
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  if (CG == 2)
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
            "r"(dst), "l"((uint64_t)map), "r"(c0), "r"(c1), "r"(bar)
        : "memory");
  else
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(dst),
                 "l"((uint64_t)map), "r"(c0), "r"(c1), "r"(bar)
                 : "memory");
}
template <int CG>
__device__ __forceinline__ void tma_load_4d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2, int c3,
                                            uint32_t bar) {
  if (CG == 2)
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], "
        "[%6];" ::"r"(dst), "l"((uint64_t)map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
        : "memory");
  else
    asm volatile(
        "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4, %5}], [%6];" ::"r"(dst),
        "l"((uint64_t)map), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(bar)
        : "memory");
}
// TMA store of a 4-D box from shared memory (bulk async-group completion)
__device__ __forceinline__ void tma_store_4d(const CUtensorMap* map, uint32_t src, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5}], [%1];" ::"l"((uint64_t)map),
               "r"(src), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
// all but the most recent store have finished READING their shared-memory source (two staging buffers)
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
// all but the two most recent stores have finished reading (three staging buffers used round-robin)
__device__ __forceinline__ void tma_store_wait_read2() { asm volatile("cp.async.bulk.wait_group.read 2;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_THREADS) : "memory"); }

// TMEM allocation; for a CTA pair one warp of EACH CTA executes it (both get the same base)
template <int CG> __device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t cols) {
  if (CG == 2) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
}
template <int CG> __device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  if (CG == 2) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
  else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
// D[tmem, (128*CG) x N] (+)= A[smem, 128 rows per CTA] * B[smem, N/CG rows per CTA]; issued by the leader CTA only
template <int CG>
__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  if (CG == 2)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
        "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
// D[tmem] (+)= A[TMEM, 128 lanes per CTA x 8 columns (K = 16 packed 16-bit)] * B[smem]
template <int CG>
__device__ __forceinline__ void umma_f16_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  if (CG == 2)
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
  else
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}" ::"r"(d_tmem),
        "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(acc)
        : "memory");
}
// registers -> TMEM, shape 16x256b.x4: 16 lanes x 32 columns.  Thread T holds, for every 8-column group g,
// columns 8g + 2(T%4) + {0,1} of lane T/4 in r[4g], r[4g+1] and of lane T/4 + 8 in r[4g+2], r[4g+3].
__device__ __forceinline__ void tmem_st_16x256b_x4(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.16x256b.x4.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};" ::"r"(taddr),
      "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]),
      "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// arrive (once the MMAs issued so far have completed) on the barrier at the same offset in every CTA of the group
template <int CG> __device__ __forceinline__ void umma_commit(uint32_t bar) {
  if (CG == 2)
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"((uint16_t)3)
                 : "memory");
  else
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// the same load without the wait: several can be in flight, tmem_ld_wait() completes all of them
__device__ __forceinline__ void tmem_ld32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Warpgroup register reallocation (all four warps of a warpgroup execute it together).  AlignConv's 768 threads
// start with 80 registers each; the TMA / MMA warpgroup gives registers back and the epilogue warpgroup takes them,
// so that it can keep TWO 32-column accumulator chunks (64 fp32 registers) in flight per tensor-memory wait.
template <int N> __device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N> __device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// two fp32 -> one packed 16-bit pair (lo in the low half) with the ReLU folded into the conversion
template <typename T> __device__ __forceinline__ uint32_t pack2_relu(float lo, float hi);
template <> __device__ __forceinline__ uint32_t pack2_relu<__nv_bfloat16>(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
template <> __device__ __forceinline__ uint32_t pack2_relu<__half>(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.f16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}

__device__ __forceinline__ void red_add_v4(float* addr, float a, float b, float c, float d) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// K-major, SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor layout):
// start address >> 4 | LBO (unused for swizzled K-major, 1) << 16 | SBO (8 rows * 128 B = 1024 B) >> 4
// << 32 | version 1 << 46 | layout SWIZZLE_128B (2) << 61.
// Bits 49-51 (base offset) are added by the caller when the start address is not 1024-byte aligned.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr, uint32_t sbo_bytes = 1024) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46) |
         (2ull << 61);
}

// 16-bit element helpers
template <typename T> struct Half2Of;
template <> struct Half2Of<__nv_bfloat16> { using type = __nv_bfloat162; };
template <> struct Half2Of<__half> { using type = __half2; };
__device__ __forceinline__ float2 to_f2(__nv_bfloat162 v) { return __bfloat1622float2(v); }
__device__ __forceinline__ float2 to_f2(__half2 v) { return __half22float2(v); }
template <typename T> __device__ __forceinline__ typename Half2Of<T>::type from_f2(float a, float b);
template <> __device__ __forceinline__ __nv_bfloat162 from_f2<__nv_bfloat16>(float a, float b) {
  return __floats2bfloat162_rn(a, b);
}
template <> __device__ __forceinline__ __half2 from_f2<__half>(float a, float b) { return __floats2half2_rn(a, b); }

__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
  uint4 r;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "r"(addr));
  return r;
}
// 16-byte store through a 32-bit shared-space address.  A store through a generic pointer into dynamic shared memory
// makes the compiler rebuild the shared window from SR_CgaCtaId (an S2R -- XU pipe) next to EVERY store of a loop: ncu
// showed the XU pipe 98 % busy in conv_tf32x3_kernel's producers before its stores went through this.
__device__ __forceinline__ void sts_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}

// Packed 16-bit bilinear blend of one 16-byte chunk (8 channels): o = w0*v0 + w1*v1 + w2*v2 + w3*v3 with
// HMUL2/HFMA2 on bf16x2 / f16x2 pairs.  The reference's half-precision path evaluates the same
// expression in scalar_t = half (deformable_im2col_bilinear, deform_conv_cuda_kernel.cu:110-113), and
// the value is rounded to 16 bits for the tensor core either way; doing the four-term sum in packed
// 16-bit math quarters the producer warps' instruction count, which is what bounds this kernel.
template <typename T>
__device__ __forceinline__ uint4 blend4(const uint4& v0, const uint4& v1, const uint4& v2, const uint4& v3, uint32_t w01,
                                        uint32_t w23) {
  using H2 = typename Half2Of<T>::type;
  // broadcast each 16-bit weight to both halves of a pair
  const uint32_t u0 = __byte_perm(w01, 0, 0x1010), u1 = __byte_perm(w01, 0, 0x3232);
  const uint32_t u2 = __byte_perm(w23, 0, 0x1010), u3 = __byte_perm(w23, 0, 0x3232);
  const H2 w0 = *reinterpret_cast<const H2*>(&u0), w1 = *reinterpret_cast<const H2*>(&u1),
           w2 = *reinterpret_cast<const H2*>(&u2), w3 = *reinterpret_cast<const H2*>(&u3);
  const H2* a = reinterpret_cast<const H2*>(&v0);
  const H2* b = reinterpret_cast<const H2*>(&v1);
  const H2* c = reinterpret_cast<const H2*>(&v2);
  const H2* d = reinterpret_cast<const H2*>(&v3);
  uint4 o;
  H2* oh = reinterpret_cast<H2*>(&o);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    H2 t = __hmul2(w0, a[i]);
    t = __hfma2(w1, b[i], t);
    t = __hfma2(w2, c[i], t);
    t = __hfma2(w3, d[i], t);
    oh[i] = t;
  }
  return o;
}

// ---------------------------------------------------------------------------------------------
// the kernel: persistent, one CTA per SM, tiles of all levels handed out round-robin
// ---------------------------------------------------------------------------------------------
// sample table of one tile: (row, tap) -> top-left pixel + fractional weights.  Position formula:
// models/alignconv.py:29-86 with the offset added back as the deformable im2col does
// (deform_conv_cuda_kernel.cu:223-227); same operation order as csrc/conv_f32.cu.
template <typename T>
__device__ __forceinline__ void build_tap_table(const TcParams& p, const TileCoord& tc, TapSample* tab, int t0, int nt) {
  const TcLevel& L = p.lv[tc.lvl];
  const int H = L.H, W = L.W;
  for (int e = t0; e < TC_M * 9; e += nt) {
    const int r = e / 9, t = e - 9 * r;
    const int y = tc.ty0 + r / TC_PW, x = tc.tx0 + r % TC_PW;
    TapSample s;
    s.base = TC_IN_HALO; s.w01 = 0u; s.w23 = 0u;          // weight-0 sample: reads halo pixel 0
    if (y < H && x < W) {
      const int ti = t / 3, tj = t - 3 * ti;
      float h, w;
      if (L.offsets) {
        // generic deformable conv (deform_conv_cuda_kernel.cu:218-227): h_im = h_in + i + offset_h, pad 1 / stride 1
        const size_t oi = (((size_t)tc.b * 18 + 2 * t) * H + y) * W + x, plane = (size_t)H * W;
        float offy, offx;
        if (p.off_f32) {
          offy = reinterpret_cast<const float*>(L.offsets)[oi];
          offx = reinterpret_cast<const float*>(L.offsets)[oi + plane];
        } else {
          offy = (float)reinterpret_cast<const T*>(L.offsets)[oi];
          offx = (float)reinterpret_cast<const T*>(L.offsets)[oi + plane];
        }
        h = __fadd_rn((float)(y - 1 + ti), offy);
        w = __fadd_rn((float)(x - 1 + tj), offx);
        if (p.pos_round) { h = (float)(T)h; w = (float)(T)w; }     // `scalar_t h_im` of the reference's 16-bit kernel
      } else {
        const float* a = L.anchors + ((size_t)(tc.b * H + y) * W + x) * 5;
        const float ax = a[0] / L.stride, ay = a[1] / L.stride, aw = a[2] / L.stride, ah = a[3] / L.stride;
        const float cs = cosf(a[4]), sn = sinf(a[4]);
        const float dw = aw / 3.0f, dh = ah / 3.0f;
        const float fi = (float)(ti - 1), fj = (float)(tj - 1);
        const float txx = __fmul_rn(dw, fj), tyy = __fmul_rn(dh, fi);
        const float xr = __fsub_rn(__fmul_rn(cs, txx), __fmul_rn(sn, tyy));
        const float yr = __fadd_rn(__fmul_rn(sn, txx), __fmul_rn(cs, tyy));
        const float xa = __fadd_rn(xr, ax), ya = __fadd_rn(yr, ay);
        const float offx = __fsub_rn(xa, __fadd_rn((float)x, fj));
        const float offy = __fsub_rn(ya, __fadd_rn((float)y, fi));
        h = __fadd_rn((float)(y - 1 + ti), offy);
        w = __fadd_rn((float)(x - 1 + tj), offx);
      }
      if (h > -1.0f && w > -1.0f && h < (float)H && w < (float)W) {
        const float hf = floorf(h), wf = floorf(w);
        const int y0 = (int)hf, x0 = (int)wf;
        const float ly = h - hf, lx = w - wf;
        float hy = 1.0f - ly, hx = 1.0f - lx;
        float w00 = hy * hx, w01_ = hy * lx, w10 = ly * hx, w11 = ly * lx;
        if (p.pos_round && L.offsets) {       // every operation of deformable_im2col_bilinear rounded to scalar_t (:94-110)
          hy = (float)(T)hy; hx = (float)(T)hx;
          w00 = (float)(T)(hy * hx); w01_ = (float)(T)(hy * lx); w10 = (float)(T)(ly * hx); w11 = (float)(T)(ly * lx);
        }
        const bool t_ok = y0 >= 0, b_ok = y0 + 1 <= H - 1, l_ok = x0 >= 0, r_ok = x0 + 1 <= W - 1;
        const int yt = max(y0, 0), yb = min(y0 + 1, H - 1), xl = max(x0, 0), xrr = min(x0 + 1, W - 1);
        using H2 = typename Half2Of<T>::type;
        const H2 p01 = from_f2<T>((t_ok && l_ok) ? w00 : 0.0f, (t_ok && r_ok) ? w01_ : 0.0f);
        const H2 p23 = from_f2<T>((b_ok && l_ok) ? w10 : 0.0f, (b_ok && r_ok) ? w11 : 0.0f);
        s.w01 = *reinterpret_cast<const uint32_t*>(&p01);
        s.w23 = *reinterpret_cast<const uint32_t*>(&p23);
        const int hy0 = yt - (tc.ty0 - TC_HALO), hx0 = xl - (tc.tx0 - TC_HALO);     // top-left corner inside the halo window?
        const bool in_halo = hy0 >= 0 && hx0 >= 0 && yb - (tc.ty0 - TC_HALO) < TC_HH && xrr - (tc.tx0 - TC_HALO) < TC_HW;
        const uint32_t pix = in_halo ? (uint32_t)(hy0 * TC_HW + hx0) : (uint32_t)(yt * W + xl);
        s.base = (in_halo ? TC_IN_HALO : 0u) | (pix << 2) | (xrr > xl ? 1u : 0u) | (yb > yt ? 2u : 0u);
      }
    }
    tab[e] = s;
  }
}

// Work assignment: the launch is a grid of CTA groups (clusters of CG CTAs; CG = 2 is a CTA pair = one TPC).
// Group q owns the tiles CG*q .. CG*q + CG - 1: each CTA produces its own 128-row A tile and stages its own
// 1/CG of the weight k-block (C_out/CG rows); the leader CTA (rank 0) issues ONE tcgen05.mma per K=16 step
// for the whole group (M = 128*CG, N = C_out), and each CTA drains its own 128 accumulator lanes.  When the
// number of tiles is not a multiple of CG the last group's spare CTA runs a "ghost" copy of the last tile
// and stores nothing.
template <int MODE, typename T, bool FD = false>
__global__ void __launch_bounds__(tc_threads<MODE>(), 1)
conv_tc_kernel(const __grid_constant__ TcMaps maps, const __grid_constant__ TcParams p) {
  static_assert(!FD || MODE == TC_PLAIN, "the FAM-decode epilogue belongs to the plain conv");
  using Cfg = TcCfg<MODE>;
  constexpr int CG = Cfg::CG, SA = Cfg::SA, SB = Cfg::SB;
  constexpr bool UNI = Cfg::UNIFIED;                   // B shares A's stage index and barriers
  static_assert(!UNI || SA == SB, "a unified ring needs equally many A and B stages");
  constexpr int GROUPS = Cfg::GROUPS, KPS = Cfg::KPS;
  static_assert(GROUPS < SA && SA <= TC_MAX_STAGES && SB <= TC_MAX_STAGES, "stage rings");
  static_assert(MODE != TC_ALIGN || 256 + SA * 32 <= TC_TMEM_COLS, "AlignConv: accumulator + A stages must fit tensor memory");
  constexpr bool IS_PLAIN = MODE != TC_ALIGN;                   // TC_PLAIN or TC_PLAIN_S
  constexpr int B_KB_BYTES = Cfg::BROWS * TC_KB * 2;            // one k-block of this CTA's weight rows
  constexpr int B_STAGE_BYTES = KPS * B_KB_BYTES;
  extern __shared__ uint8_t smem_raw[];
  // SWIZZLE_128B operands need 1024-byte aligned tiles: align the dynamic window by hand (the offset is
  // the same in both CTAs of a pair, which the paired MMA and the multicast commits rely on)
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  // carve: B stages | 3 output staging buffers | 2 halo buffers | ALIGN: 2 sample tables | barriers | tmem pointer
  constexpr int ACC = MODE == TC_ALIGN ? 1 : 2;        // accumulators: PLAIN 2 x 256 TMEM columns; ALIGN 1 (+ 8 A stages x 32 columns)
  constexpr uint32_t A_TMEM_COL0 = 256;                // ALIGN: first TMEM column of the A stages
  constexpr int HALO_BYTES = MODE == TC_ALIGN ? TC_HALO_BYTES : TC_PHALO_BYTES;
  uint8_t* sB = smem;
  uint8_t* s_out = sB + SB * B_STAGE_BYTES;                              // 3 x 8 KB, 1024-byte aligned (SWIZZLE_64B)
  uint8_t* s_halo = s_out + TC_OUT_BUFS * TC_OUT_BYTES;                  // 1024-byte aligned (PLAIN: SWIZZLE_128B operand)
  constexpr int NH = Cfg::NHALO, NHL = NH == 4 ? 2 : 1;
  static_assert((NH == 2 || NH == 4) && NH <= TC_MAX_HALOS && (MODE != TC_ALIGN || NH == 2), "halo buffers");
  TapSample* s_tab = reinterpret_cast<TapSample*>(s_halo + NH * HALO_BYTES);          // ALIGN only
  static_assert(TC_HALO_BYTES % 128 == 0 && TC_PHALO_BYTES % 1024 == 0 && (TC_OUT_BUFS * TC_OUT_BYTES) % 1024 == 0 &&
                B_STAGE_BYTES % 1024 == 0, "TMA source / destination alignment");
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(
      s_halo + NH * HALO_BYTES + (MODE == TC_ALIGN ? 2 * sizeof(TapSample) * TC_M * 9 : (size_t)0));
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + TC_NBAR);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t bar_full_a = smem_u32(s_bar), bar_empty_a = bar_full_a + 8 * TC_MAX_STAGES,
                 bar_full_b = bar_empty_a + 8 * TC_MAX_STAGES, bar_empty_b = bar_full_b + 8 * TC_MAX_STAGES,
                 bar_acc_full = bar_empty_b + 8 * TC_MAX_STAGES, bar_acc_empty = bar_acc_full + 8 * TC_ACC_STAGES,
                 bar_tab_full = bar_acc_empty + 8 * TC_ACC_STAGES,       // 2 barriers
                 bar_halo_full = bar_tab_full + 16, bar_halo_empty = bar_halo_full + 8 * TC_MAX_HALOS;   // 4 + 4 barriers
  // warps 0-15 producers | 16-19 epilogue (one warpgroup) | 20 TMA, 21 MMA, 22-23 idle (one warpgroup)
  constexpr int kProdWarps = GROUPS * 4, kEpiWarp0 = kProdWarps, kTmaWarp = kEpiWarp0 + TC_EPI_THREADS / 32,
                kMmaWarp = kTmaWarp + 1;

  const uint32_t cta_rank = CG == 2 ? cluster_ctarank() : 0u;     // 0 = leader (issues the MMAs, owns the "full" barriers)
  const bool leader = cta_rank == 0;
  // "full" barriers and the accumulator-empty barrier live in the leader CTA; everybody signals them there
  const uint32_t ld_full_a = CG == 2 ? map_to_cta(bar_full_a, 0) : bar_full_a,
                 ld_full_b = UNI ? ld_full_a : (CG == 2 ? map_to_cta(bar_full_b, 0) : bar_full_b),
                 ld_acc_empty = CG == 2 ? map_to_cta(bar_acc_empty, 0) : bar_acc_empty;

  const int ncb = (p.C + TC_KB - 1) / TC_KB;         // 64-channel blocks (TC_PLAIN: a partial block is zero-filled by TMA)
  const int ntap = p.ks * p.ks;
  const int nkb = ncb * ntap;
  const int co_part = p.Co / CG;                     // weight rows (output channels) staged by this CTA
  const uint32_t b_bytes_group = (uint32_t)p.Co * TC_KB * 2;
  const int ngroups = (p.total_tiles + CG - 1) / CG;
  const int first_q = CG == 2 ? (int)cluster_id_x() : (int)blockIdx.x;
  const int q_step = CG == 2 ? (int)cluster_count_x() : (int)gridDim.x;
  // tile of this CTA in group q; ghost = duplicate of the last tile, nothing stored
#define S2A_TILE_OF(q) min((q) * CG + (int)cta_rank, p.total_tiles - 1)
#define S2A_IS_GHOST(q) ((q) * CG + (int)cta_rank >= p.total_tiles)

  if (tid == 0) {
    for (int s = 0; s < SA; ++s) {
      // full_a: ALIGN -- one elected arrive per producer warp of the owning group, from every CTA of the group;
      //         PLAIN -- the leader TMA thread's expect_tx arrive (+ the TMA bytes of A and B from every CTA)
      mbar_init(bar_full_a + 8 * s, MODE == TC_ALIGN ? 1 + 4 * CG : 1);
      mbar_init(bar_empty_a + 8 * s, 1);        // one (multicast) tcgen05.commit
    }
    for (int s = 0; s < SB && !UNI; ++s) {
      mbar_init(bar_full_b + 8 * s, 1);         // the leader TMA thread's expect_tx arrive (+ bytes)
      mbar_init(bar_empty_b + 8 * s, 1);
    }
    for (int s = 0; s < TC_ACC_STAGES; ++s) {
      mbar_init(bar_acc_full + 8 * s, 1);       // tcgen05.commit after the last k-block of a tile group
      mbar_init(bar_acc_empty + 8 * s, CG * (TC_EPI_THREADS / 32));   // one elected arrive per epilogue warp of the group
      mbar_init(bar_tab_full + 8 * s, TC_EPI_THREADS);
    }
    for (int s = 0; s < TC_MAX_HALOS; ++s) {
      mbar_init(bar_halo_full + 8 * s, 1);                   // the TMA thread's expect_tx arrive (+ bytes)
      // ALIGN: one elected arrive per producer warp; plain conv: one (multicast) tcgen05.commit
      mbar_init(bar_halo_empty + 8 * s, kProdWarps > 0 ? kProdWarps : 1);
    }
    fence_barrier_init();
  }
  if (warp == kMmaWarp) tmem_alloc<CG>(smem_u32(s_tmem), TC_TMEM_COLS);
  tc_fence_before();
  if (CG == 2) cluster_sync_all();              // barriers of both CTAs initialised before anybody signals them
  else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  S2A_TL(long long dbg_c0 = 0; unsigned long long dbg_t0 = 0;
         if ((p.debug & 8) && blockIdx.x == 0) {
           dbg_c0 = clock64();
           asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(dbg_t0));
         })

  auto role_producer = [&]() {
    // ===================== A producers (AlignConv: bilinear gather through the LSU) =====================
    // In TC_PLAIN mode (ORConv2d) the A tile is a shifted patch of the NHWC map, which TMA fetches
    // directly (zero-filled outside the map), so these warps have nothing to do.
    const int group = warp >> 2;               // producer group: owns global k-blocks group, group + G, ...
    // Thread mapping = the tcgen05.st 16x256b fragment: warp w of a group owns TMEM lanes (tile rows)
    // 32*(w%4) .. +31; thread T handles rows T/4 + 8k (k = 0..3) and, of each row's 128-byte k-block line, the
    // 16-byte chunks q = T%4 and q + 4.  In TMEM column order those 32 bytes sit at 32g + 8q (+8) for g = 0..3;
    // the weight packer applies the same channel permutation inside every 64-channel block (tc_kperm).
    const int wq = warp & 3;
    const int q4 = lane & 3, r8 = lane >> 2;
    // even rows read chunk q first, odd rows chunk q + 4: one LDS.128 of a warp then spreads over all 32 banks
    const int c_first = (r8 & 1) ? q4 + 4 : q4, c_second = (r8 & 1) ? q4 : q4 + 4;
    // Group g produces the global k-blocks g, g + G, g + 2G, ... (the sequence runs on across tiles).  Stage
    // index and phase bit advance incrementally: no 64-bit div/mod on these latency-critical paths.
    int kb = group;                            // k-block inside the current tile
    int s = group % SA;                        // A stage of that k-block
    uint32_t ph = (uint32_t)(group / SA) & 1u;
    uint32_t hseq = 0;                         // running (tile, channel block) counter: halo buffer = hseq & 1
    const uint32_t halo_u32 = smem_u32(s_halo);
    constexpr int GSTEP = GROUPS > 0 ? GROUPS : 1;      // (GROUPS == 0: this branch is dead code)
    int it = 0;
    for (int q = first_q; MODE == TC_ALIGN && q < ngroups; q += q_step, ++it) {
      const int tile = S2A_TILE_OF(q);
      const TileCoord tc = decode_tile<MODE>(p, tile);
      const TcLevel& L = p.lv[tc.lvl];
      const int H = L.H, W = L.W;
      const uint32_t pix_stride = (uint32_t)p.C * 2u, row_stride = (uint32_t)W * pix_stride;
      const uint8_t* xb = reinterpret_cast<const uint8_t*>(L.x) + (size_t)tc.b * H * W * p.C * 2;
      const TapSample* tab = s_tab + (it & 1) * (TC_M * 9);
      mbar_wait(bar_tab_full + 8 * (it & 1), (uint32_t)(it >> 1) & 1u);
      int cb = kb / 9, tap = kb - 9 * cb;
      for (; kb < nkb; kb += GSTEP, tap += GSTEP, s += GSTEP) {
        if (tap >= 9) { tap -= 9; ++cb; }
        if (s >= SA) { s -= SA; ph ^= 1u; }
        const uint32_t hcur = hseq + (uint32_t)cb;                  // this k-block's (tile, channel block)
        mbar_wait(bar_halo_full + 8 * (hcur & 1u), (hcur >> 1) & 1u);
        mbar_wait(bar_empty_a + 8 * s, ph ^ 1u);
        tc_fence_after();
        if (!(p.debug & 2)) {
          const uint8_t* src = xb + (size_t)cb * TC_KB * 2;                    // channel block inside a pixel (global fallback)
          const uint32_t hsrc = halo_u32 + (hcur & 1u) * TC_HALO_BYTES;
          const TapSample* trow = tab + (wq * 32 + r8) * 9 + tap;
#pragma unroll
          for (int half = 0; half < 2; ++half) {                               // TMEM lanes 32*wq + 16*half .. +15
            uint32_t frag[16];
#pragma unroll
            for (int i = 0; i < 2; ++i) {                                      // rows r8 and r8 + 8 of this half
              const TapSample sm = trow[(half * 16 + i * 8) * 9];
              uint4 va[4], vb[4];                                              // [corner]: first / second chunk
              const uint32_t pix = (sm.base & ~TC_IN_HALO) >> 2;
              const uint32_t o1 = (uint32_t)c_first * 16u, o2 = (uint32_t)c_second * 16u;
              if (__all_sync(0xffffffffu, (sm.base & TC_IN_HALO) != 0u)) {     // warp-uniform: no dependent divergence
                const uint32_t q0 = hsrc + pix * (TC_KB * 2);
                const uint32_t dx = (sm.base & 1u) ? (uint32_t)(TC_KB * 2) : 0u;
                const uint32_t dy = (sm.base & 2u) ? (uint32_t)(TC_HW * TC_KB * 2) : 0u;
                va[0] = lds_v4(q0 + o1); va[1] = lds_v4(q0 + dx + o1);
                va[2] = lds_v4(q0 + dy + o1); va[3] = lds_v4(q0 + dy + dx + o1);
                vb[0] = lds_v4(q0 + o2); vb[1] = lds_v4(q0 + dx + o2);
                vb[2] = lds_v4(q0 + dy + o2); vb[3] = lds_v4(q0 + dy + dx + o2);
              } else if (sm.base & TC_IN_HALO) {
                const uint32_t q0 = hsrc + pix * (TC_KB * 2);
                const uint32_t dx = (sm.base & 1u) ? (uint32_t)(TC_KB * 2) : 0u;
                const uint32_t dy = (sm.base & 2u) ? (uint32_t)(TC_HW * TC_KB * 2) : 0u;
                va[0] = lds_v4(q0 + o1); va[1] = lds_v4(q0 + dx + o1);
                va[2] = lds_v4(q0 + dy + o1); va[3] = lds_v4(q0 + dy + dx + o1);
                vb[0] = lds_v4(q0 + o2); vb[1] = lds_v4(q0 + dx + o2);
                vb[2] = lds_v4(q0 + dy + o2); vb[3] = lds_v4(q0 + dy + dx + o2);
              } else {                               // a corner outside the halo window: straight from global memory
                const uint8_t* q0 = src + (size_t)pix * pix_stride;
                const uint32_t dx = (sm.base & 1u) ? pix_stride : 0u, dy = (sm.base & 2u) ? row_stride : 0u;
                va[0] = ldg_nc_v4(q0 + o1); va[1] = ldg_nc_v4(q0 + dx + o1);
                va[2] = ldg_nc_v4(q0 + dy + o1); va[3] = ldg_nc_v4(q0 + dy + dx + o1);
                vb[0] = ldg_nc_v4(q0 + o2); vb[1] = ldg_nc_v4(q0 + dx + o2);
                vb[2] = ldg_nc_v4(q0 + dy + o2); vb[3] = ldg_nc_v4(q0 + dy + dx + o2);
              }
              const uint4 b1 = blend4<T>(va[0], va[1], va[2], va[3], sm.w01, sm.w23);
              const uint4 b2 = blend4<T>(vb[0], vb[1], vb[2], vb[3], sm.w01, sm.w23);
              const uint4 lo = (r8 & 1) ? b2 : b1, hi = (r8 & 1) ? b1 : b2;     // chunk q / chunk q + 4
              frag[0 + 2 * i] = lo.x; frag[1 + 2 * i] = lo.y;                   // column group 0
              frag[4 + 2 * i] = lo.z; frag[5 + 2 * i] = lo.w;                   // group 1
              frag[8 + 2 * i] = hi.x; frag[9 + 2 * i] = hi.y;                   // group 2
              frag[12 + 2 * i] = hi.z; frag[13 + 2 * i] = hi.w;                 // group 3
            }
            tmem_st_16x256b_x4(tmem_base + ((uint32_t)(wq * 32 + half * 16) << 16) + A_TMEM_COL0 + (uint32_t)s * 32u, frag);
          }
          tmem_st_wait();
        }
        tc_fence_before();                 // tensor-memory stores ordered before the arrive the MMA thread waits on
        __syncwarp();
        if (lane == 0) {
          mbar_arrive_cluster(ld_full_a + 8 * s);                  // on the leader CTA's barrier
          if (tap >= 9 - GSTEP) mbar_arrive(bar_halo_empty + 8 * (hcur & 1u));   // this warp's last tap of the channel block
        }
      }
      kb -= nkb;                           // first k-block of this group in the next tile
      hseq += (uint32_t)ncb;
    }
  };
  auto role_tma = [&]() {
    // ===================== TMA: this CTA's C_out/CG weight rows (and, PLAIN, its A tile) =====================
    // (the whole warp walks the loop and waits; one elected lane arms the barrier and issues the copies)
    {
      int sa = 0, sb = 0;
      uint32_t pa = 0, pb = 0;                   // phase bits of the stage rings
      uint32_t hseq = 0;                         // running (tile, channel block) counter of the halo buffers
      bool warm = false;
      // AlignConv: halo of one (tile, channel block) = the 14 x 22 pixel window around the tile as one 4-D box
      // {64, 22, 14, 1}, zero-filled outside the map, into buffer (sequence number & 1)
      auto load_halo = [&](const TileCoord& t, int cblk) {
        const uint32_t hb = hseq & 1u;
        mbar_wait(bar_halo_empty + 8 * hb, ((hseq >> 1) & 1u) ^ 1u);
        if (elect_one()) {
          mbar_arrive_expect_tx(bar_halo_full + 8 * hb, TC_HALO_BYTES);
          tma_load_4d<1>(smem_u32(s_halo + hb * TC_HALO_BYTES), &maps.x[t.lvl], cblk * TC_KB, t.tx0 - TC_HALO, t.ty0 - TC_HALO,
                         t.b, bar_halo_full + 8 * hb);
        }
        __syncwarp();
        ++hseq;
      };
      if (MODE == TC_ALIGN && first_q < ngroups) load_halo(decode_tile<MODE>(p, S2A_TILE_OF(first_q)), 0);
      for (int q = first_q; IS_PLAIN && q < ngroups; q += q_step) {
        // plain conv / ORConv: a stage carries KPS weight k-blocks (this CTA's C_out/CG rows of each); the A operand
        // is the halo the halo warp loads
        const CUtensorMap* wmap = &maps.w[decode_tile<MODE>(p, S2A_TILE_OF(q)).lvl >= p.wsplit ? 1 : 0];
        for (int kb = 0; kb < nkb; kb += KPS) {
          const int nk = min(KPS, nkb - kb);
          mbar_wait(bar_empty_a + 8 * sa, pa ^ 1u);
          if (elect_one()) {
            if ((p.debug & 1) && warm) {
              if (leader) mbar_arrive(bar_full_a + 8 * sa);
            } else {
              if (leader) mbar_arrive_expect_tx(bar_full_a + 8 * sa, (uint32_t)nk * b_bytes_group);
#pragma unroll
              for (int j = 0; j < KPS; ++j) {
                if (j < nk)
                  tma_load_2d<CG>(smem_u32(sB + sa * B_STAGE_BYTES + j * B_KB_BYTES), wmap, (kb + j) * TC_KB,
                                  (int)cta_rank * co_part, ld_full_a + 8 * sa);
              }
            }
          }
          __syncwarp();
          if (++sa == SA) { sa = 0; pa ^= 1u; }
        }
        warm = true;
      }
      for (int q = first_q; MODE == TC_ALIGN && q < ngroups; q += q_step) {
        const TileCoord tc = decode_tile<MODE>(p, S2A_TILE_OF(q));
        int cb = 0, tap = 0;
        for (int kb = 0; kb < nkb; ++kb) {
          if (UNI) {
            // one ring: the weight k-block and the A operand of a k-block complete the same "full" barrier (the
            // producer warps arrive on it after their tcgen05.st)
            if (MODE == TC_ALIGN && tap == 3) {
              // halo of the NEXT (tile, channel block), requested six k-blocks before its first use
              if (cb + 1 < ncb) load_halo(tc, cb + 1);
              else if (q + q_step < ngroups) load_halo(decode_tile<MODE>(p, S2A_TILE_OF(q + q_step)), 0);
            }
            mbar_wait(bar_empty_a + 8 * sa, pa ^ 1u);
            if (elect_one()) {
              if ((p.debug & 1) && warm) {
                if (leader) mbar_arrive(bar_full_a + 8 * sa);
              } else {
                if (leader) mbar_arrive_expect_tx(bar_full_a + 8 * sa, b_bytes_group);
                tma_load_2d<CG>(smem_u32(sB + sa * B_STAGE_BYTES), &maps.w[0], kb * TC_KB, (int)cta_rank * co_part, ld_full_a + 8 * sa);
              }
            }
            __syncwarp();
            if (++sa == SA) { sa = 0; pa ^= 1u; }
          } else {
            if (MODE == TC_ALIGN && tap == 3) {
              // halo of the NEXT (tile, channel block), requested six k-blocks before its first use
              if (cb + 1 < ncb) load_halo(tc, cb + 1);
              else if (q + q_step < ngroups) load_halo(decode_tile<MODE>(p, S2A_TILE_OF(q + q_step)), 0);
            }
            mbar_wait(bar_empty_b + 8 * sb, pb ^ 1u);
            if (elect_one()) {
              if ((p.debug & 1) && warm) {
                if (leader) mbar_arrive(bar_full_b + 8 * sb);
              } else {
                if (leader) mbar_arrive_expect_tx(bar_full_b + 8 * sb, b_bytes_group);
                tma_load_2d<CG>(smem_u32(sB + sb * B_STAGE_BYTES), &maps.w[0], kb * TC_KB, (int)cta_rank * co_part, ld_full_b + 8 * sb);
              }
            }
            __syncwarp();
            if (++sb == SB) { sb = 0; pb ^= 1u; }
          }
          if (++tap == ntap) { tap = 0; ++cb; }
        }
        warm = true;
      }
    }
  };
  auto role_halo = [&]() {
    // ===================== plain conv: halo loads (the A operand) =====================
    // One box {64 ch, 16, 18, 1} per (tile, 64-channel block) at (tx0 - 1, ty0 - 1), zero-filled outside the map and
    // beyond C, into buffer (sequence number & 1).  A buffer is recycled when the last tap's MMAs of its channel
    // block have retired (tcgen05.commit, multicast to both CTAs); both CTAs' boxes complete the leader's barrier.
    const uint32_t ld_halo_full = CG == 2 ? map_to_cta(bar_halo_full, 0) : bar_halo_full;
    // ring depth / buffer size: a 1 x 1 conv's "halo" is the bare 16 KB tile and lives one k-block only, so the
    // same shared memory holds a ring of four of them (its loads are latency-, not bandwidth-bound)
    const int nhl = (p.ks == 3) ? NHL : 2;
    const uint32_t nh_mask = (1u << nhl) - 1u, hstride = p.ks == 3 ? (uint32_t)TC_PHALO_BYTES : (uint32_t)(TC_M * 128);
    uint32_t hseq = 0;
    for (int q = first_q; q < ngroups; q += q_step) {
      const TileCoord tc = decode_tile<MODE>(p, S2A_TILE_OF(q));
      for (int cb = 0; cb < ncb; ++cb, ++hseq) {
        const uint32_t hb = hseq & nh_mask;
        mbar_wait(bar_halo_empty + 8 * hb, ((hseq >> nhl) & 1u) ^ 1u);
        if (elect_one()) {
          // (a 1 x 1 conv needs no border: its box is the 8 x 16 tile itself, pitch 8 pixels)
          if (leader) mbar_arrive_expect_tx(bar_halo_full + 8 * hb, (uint32_t)CG * hstride);
          tma_load_4d<CG>(smem_u32(s_halo + hb * hstride), &maps.x[tc.lvl], cb * TC_KB, tc.tx0 - (p.ks >> 1),
                          tc.ty0 - (p.ks >> 1), tc.b, ld_halo_full + 8 * hb);
        }
        __syncwarp();
      }
    }
  };
  auto role_mma = [&]() {
    // ===================== MMA issuer (leader CTA only) =====================
    if (leader) {                                    // the whole warp runs the loop; one elected lane issues
      // instruction descriptor (cute::UMMA::InstrDescriptor): D=f32 (1<<4), A/B format (bf16=1, f16=0)
      // at bits 7 / 10, K-major A and B, N>>3 at bit 17, M>>4 at bit 24 (M = 128 per CTA of the group)
      const uint32_t fmt = std::is_same<T, __nv_bfloat16>::value ? 1u : 0u;
      const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(p.Co >> 3) << 17) |
                             ((uint32_t)((TC_M * CG) >> 4) << 24);
      // tcgen05.mma issue blocks this thread while the tensor pipe is busy (measured: no deep issue queue),
      // so everything else this thread does per k-block must overlap with MMAs that are already queued:
      // the wait for the NEXT stage (and, at a tile boundary, for the next accumulator) sits between the
      // second and the third MMA of the current k-block.  tools/umma_bench2.cu: 634 -> 528 cycles per
      // k-block (ideal 512) for exactly this change.
      static_assert(UNI, "the MMA thread handles one barrier pair per stage");
      // Everything this thread touches per k-block advances incrementally (stage barrier addresses, operand
      // descriptors, TMEM column of the A stage): the instructions between two MMAs are on the critical path.
      // plain conv: the A operand of tap (ti, tj) is the halo buffer seen from pixel (ti, tj) on: start address
      // + (ti * 16 + tj) 128-byte lines, SBO = one halo row (2048 B), base offset = tj (the swizzle phase of the
      // first line; rows are a multiple of 8 lines apart and do not change it)
      const int hpitch = p.ks == 3 ? TC_PHALO_PITCH : TC_PPW;      // halo row pitch in pixels (1 x 1: the bare tile)
      const int nhl = (p.ks == 3) ? NHL : 2;                       // log2(halo ring depth), see the halo warp
      const uint32_t nh_mask = (1u << nhl) - 1u, hstride16 = (p.ks == 3 ? (uint32_t)TC_PHALO_BYTES : (uint32_t)(TC_M * 128)) >> 4;
      const uint64_t hdesc0 = umma_desc_sw128(smem_u32(s_halo), (uint32_t)hpitch * 128u);
      const uint64_t bdesc0 = umma_desc_sw128(smem_u32(sB));
      const uint32_t atm0 = tmem_base + A_TMEM_COL0;
      uint64_t bdesc = bdesc0;
      int tap = 0;                                   // plain conv: tap of the next k-block, and the running
      uint32_t hseq = 0;                             // (tile, channel block) counter: halo buffer = hseq % NHALO
      uint32_t atm = atm0, full_bar = bar_full_a, empty_bar = bar_empty_a;
      int sa = 0, it = 0;
      uint32_t pa = 0;
      S2A_TL(long long tl[10]; long long tw_acc = 0, tw_a = 0, tw_halo = 0; int n_block = 0;)
      mbar_wait(bar_acc_empty, 1u);
      mbar_wait(bar_full_a, 0u);
      tc_fence_after();
      for (int q = first_q; q < ngroups; q += q_step, ++it) {
        const int as = it % ACC;
        S2A_TL(if ((p.debug & 8) && it < 9) tl[it] = clock64();)
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * 256);
        const bool last_tile = q + q_step >= ngroups;
        // the accumulator tile group it + 1 will use, and the phase of its "drained" barrier
        const uint32_t acc_bar = bar_acc_empty + 8 * ((it + 1) % ACC), acc_par = ((uint32_t)((it + 1) / ACC) & 1u) ^ 1u;
        const uint32_t acc_full_bar = bar_acc_full + 8 * as;
        for (int kb = 0; kb < nkb; kb += KPS) {
          const int nk = KPS == 1 ? 1 : min(KPS, nkb - kb);          // k-blocks in this stage
          // +32 bytes (>>4 = 2) per K=16 step inside the swizzle atom; A in TMEM: +8 columns per K=16 step.
          // Every MMA of the stage but the last two is issued first ...
          uint64_t a_last = 0ull;                    // plain conv: A descriptor of the stage's last k-block, and the
          uint32_t rel_last = 0u;                    // halo barrier to release after it (if it is a block's last tap)
          if (IS_PLAIN) {
            // (all lanes) the halo of every channel block that starts inside this stage -- requested nine k-blocks ago
            int t = tap;
            uint32_t h = hseq;
#pragma unroll
            for (int j = 0; j < KPS; ++j) {
              if (j < nk) {
                if (t == 0) {
                  S2A_TL(long long w0 = (p.debug & 8) ? clock64() : 0;)
                  mbar_wait_likely_ready(bar_halo_full + 8 * (h & nh_mask), (h >> nhl) & 1u);
                  tc_fence_after();
                  S2A_TL(if (p.debug & 8) tw_halo += clock64() - w0;)
                }
                if (++t == ntap) { t = 0; ++h; }
              }
            }
          }
          const bool issuer = elect_one();
          if (issuer) {
            if (MODE == TC_ALIGN) {
              umma_f16_ts<CG>(d_tmem, atm, bdesc, idesc, kb != 0 ? 1u : 0u);
              umma_f16_ts<CG>(d_tmem, atm + 8u, bdesc + 2, idesc, 1u);
            } else {
              int t = tap;
              uint32_t h = hseq;
#pragma unroll
              for (int j = 0; j < KPS; ++j) {
                if (j < nk) {
                  const int ti = (t * 11) >> 5, tj = t - 3 * ti;         // (1 x 1: t = 0)
                  const uint64_t aj = hdesc0 + (uint64_t)((h & nh_mask) * hstride16) +
                                      (uint64_t)((ti * hpitch + tj) * (128 >> 4));
                  const uint64_t bj = bdesc + (uint64_t)(j * (B_KB_BYTES >> 4));
                  uint32_t rel = 0u;
                  if (++t == ntap) { t = 0; rel = bar_halo_empty + 8 * (h & nh_mask); ++h; }
                  umma_f16<CG>(d_tmem, aj, bj, idesc, (kb | j) != 0 ? 1u : 0u);
                  umma_f16<CG>(d_tmem, aj + 2, bj + 2, idesc, 1u);
                  if (j + 1 < nk) {
                    umma_f16<CG>(d_tmem, aj + 4, bj + 4, idesc, 1u);
                    umma_f16<CG>(d_tmem, aj + 6, bj + 6, idesc, 1u);
                    if (rel) umma_commit<CG>(rel);
                  } else {                           // (the last k-block's second half follows the wait below)
                    a_last = aj; rel_last = rel;
                  }
                }
              }
            }
          }
          if (IS_PLAIN) {                            // (all lanes) advance the tap / halo counters past this stage
#pragma unroll
            for (int j = 0; j < KPS; ++j)
              if (j < nk && ++tap == ntap) { tap = 0; ++hseq; }
          }
          __syncwarp();
          // ... then the next stage is awaited in the shadow of the MMAs just queued ...
          uint32_t nfull = full_bar + 8, npa = pa;
          const bool wrap = sa + 1 == SA;
          if (wrap) { nfull = bar_full_a; npa ^= 1u; }
          const bool new_acc = kb + KPS >= nkb;
          const bool more = !new_acc || !last_tile;
          bool ready = false;
          if (IS_PLAIN) {
            // tensor-bound: the next stage is (nearly) always there (and, at a tile boundary, the next accumulator
            // has to be drained)
            if (more) {
              S2A_TL(long long w0 = (p.debug & 8) ? clock64() : 0;)
              if (new_acc) mbar_wait_likely_ready(acc_bar, acc_par);
              S2A_TL(long long w1 = (p.debug & 8) ? clock64() : 0;)
              mbar_wait_likely_ready(nfull, npa);
              tc_fence_after();
              S2A_TL(if (p.debug & 8) { if (new_acc) tw_acc += w1 - w0; tw_a += clock64() - w1; ++n_block; })
              ready = true;
            }
          } else {
            // AlignConv: probe without blocking; if the next stage is not there yet, release this k-block's stage
            // FIRST -- blocking here with two MMAs unissued would hold a stage the producers need.  With a single
            // accumulator the next tile always has to wait for the epilogue: never "ready" across tiles.
            ready = __all_sync(0xffffffffu, more && !new_acc && mbar_test(nfull, npa));
            if (ready) tc_fence_after();
          }
          // ... and the last two MMAs and the commit follow
          if (issuer) {
            if (MODE == TC_ALIGN) {
              umma_f16_ts<CG>(d_tmem, atm + 16u, bdesc + 4, idesc, 1u);
              umma_f16_ts<CG>(d_tmem, atm + 24u, bdesc + 6, idesc, 1u);
            } else {
              const uint64_t bj = bdesc + (uint64_t)((nk - 1) * (B_KB_BYTES >> 4));
              umma_f16<CG>(d_tmem, a_last + 4, bj + 4, idesc, 1u);
              umma_f16<CG>(d_tmem, a_last + 6, bj + 6, idesc, 1u);
              if (rel_last) umma_commit<CG>(rel_last);   // halo buffer (of both CTAs) reusable
            }
            umma_commit<CG>(empty_bar);             // stage (of every CTA of the group) reusable once these MMAs have read it
            if (new_acc) umma_commit<CG>(acc_full_bar);   // accumulators of this tile group complete
          }
          __syncwarp();
          if (more && !ready) {
            S2A_TL(long long w0 = (p.debug & 8) ? clock64() : 0;)
            if (new_acc) mbar_wait(acc_bar, acc_par);
            S2A_TL(long long w1 = (p.debug & 8) ? clock64() : 0;)
            mbar_wait(nfull, npa);
            tc_fence_after();
            S2A_TL(if (p.debug & 8) { tw_acc += w1 - w0; tw_a += clock64() - w1; ++n_block; })
          }
          if (wrap) { sa = 0; bdesc = bdesc0; atm = atm0; empty_bar = bar_empty_a; }
          else { ++sa; bdesc += B_STAGE_BYTES >> 4; atm += 32u; empty_bar += 8; }
          full_bar = nfull; pa = npa;
        }
      }
#ifdef S2A_TC_TIMELINE
      if ((p.debug & 8) && blockIdx.x == 0 && lane == 0) {
        tl[min(it, 9)] = clock64();
        printf("s2a conv_tc MMA thread: blocked %d times: acc %lld, full %lld, halo %lld cycles; start +%lld;", n_block, tw_acc, tw_a, tw_halo, tl[0] - dbg_c0);
        for (int i = 0; i < min(it, 9); ++i) printf(" tile%d %lld", i, tl[i + 1] - tl[i]);
        printf("\n");
      }
#endif
    }
  };
  auto role_epilogue = [&]() {
    // ===================== epilogue warps (also build the sample tables) =====================
    const int et = tid - kEpiWarp0 * 32;          // 0..127
    const int quad = warp & 3;                    // TMEM lane quadrant this warp may read (warp id % 4)
    using H2 = typename Half2Of<T>::type;
    if (MODE == TC_ALIGN) {
      // tables of the first two tiles
      for (int j = 0; j < 2; ++j) {
        const int q = first_q + j * q_step;
        if (q < ngroups) {
          build_tap_table<T>(p, decode_tile<MODE>(p, S2A_TILE_OF(q)), s_tab + j * (TC_M * 9), et, TC_EPI_THREADS);
          mbar_arrive(bar_tab_full + 8 * j);
        }
      }
    }
    int it = 0;
    for (int q = first_q; q < ngroups; q += q_step, ++it) {
      const int as = it % ACC, tb = it & 1;         // accumulator / sample-table buffer of this tile
      const bool ghost = S2A_IS_GHOST(q);
      const TileCoord tc = decode_tile<MODE>(p, S2A_TILE_OF(q));
      const TcLevel& L = p.lv[tc.lvl];
      mbar_wait(bar_acc_full + 8 * as, (uint32_t)(it / ACC) & 1u);
      tc_fence_after();
      const int r = quad * 32 + lane;
      const int y = tc.ty0 + r / tc_pw<MODE>(), x = tc.tx0 + r % tc_pw<MODE>();
      const bool valid = (y < L.H && x < L.W) && !ghost && tc.b < p.B;       // (b == B: the padding tile before wsplit)
      const float* bias = tc.lvl >= p.wsplit ? p.bias2 : p.bias;
      const size_t pos = (size_t)(tc.b * L.H + y) * L.W + x;
      // Staging + store of one packed 32-channel chunk.  Each epilogue warp stores its own 32 tile rows (2 spatial
      // rows x 16 pixels) -- no barrier across the four warps.  Three 2 KB staging buffers per warp, used round-robin:
      // when the elected lane's wait returns, every store of this warp but the two most recent ones has finished
      // reading its buffer; __syncwarp publishes that.
      // (scalars, not the struct: a by-reference capture of `tc` kept it in local memory)
      const int tc_lvl = tc.lvl, tc_b = tc.b, tc_tx0 = tc.tx0, tc_ty0 = tc.ty0;
      void* const pooled_ptr = L.pooled;
      auto emit_chunk = [&](const uint32_t (&pk)[16], float m0_, float m1_, float m2_, float m3_, int c0, int ci) {
        const bool issuer = elect_one();
        if (issuer) tma_store_wait_read2();
        __syncwarp();
        uint8_t* sbuf = s_out + (ci % TC_OUT_BUFS) * TC_OUT_BYTES + quad * (32 * TC_OUT_CH * 2);
        uint8_t* row = sbuf + lane * (TC_OUT_CH * 2);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          *reinterpret_cast<uint4*>(row + ((j ^ ((lane >> 1) & 3)) << 4)) =
              make_uint4(pk[4 * j], pk[4 * j + 1], pk[4 * j + 2], pk[4 * j + 3]);
        fence_proxy_async_smem();
        __syncwarp();
        if (issuer && !ghost && !(p.debug & 64))
          tma_store_4d(&maps.y[tc_lvl], smem_u32(sbuf), c0, tc_tx0, tc_ty0 + (32 / tc_pw<MODE>()) * quad, tc_b);
        if (IS_PLAIN && valid && pooled_ptr) {
          uint2 o;
          H2* oh = reinterpret_cast<H2*>(&o);
          oh[0] = from_f2<T>(m0_, m1_);
          oh[1] = from_f2<T>(m2_, m3_);
          *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(pooled_ptr) + (pos * (p.Co / 8) + c0 / 8) * 2) = o;
        }
      };
      const uint32_t acc_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(as * 256);
      // (one arrive per warp: 128 per-thread arrives on the leader's barrier -- half of them remote -- took ~3,000
      // cycles to get through, on the critical path of the accumulator hand-off)
      auto release_acc = [&]() {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(ld_acc_empty + 8 * as);
      };
      if (MODE == TC_ALIGN) {
        // AlignConv has ONE accumulator: the MMA warp waits for this drain between tiles, so it is organised for
        // latency.  Two 32-column chunks are loaded per tensor-memory wait (the second load's latency hides behind the
        // first), ReLU is folded into the conversion (cvt.rn.relu), and a pair's stores are issued without waiting for
        // the previous pair's (three staging buffers).  No bias, no pooling (alignconv.py:97).
        for (int c0 = 0, ci = 0; c0 < p.Co && !(p.debug & 32); c0 += 2 * TC_OUT_CH, ci += 2) {
          const bool two = c0 + TC_OUT_CH < p.Co;
          uint32_t va[32], vb[32];
          tmem_ld32_nowait(acc_addr + (uint32_t)c0, va);
          if (two) tmem_ld32_nowait(acc_addr + (uint32_t)(c0 + TC_OUT_CH), vb);
          tmem_ld_wait();
          if (c0 + 2 * TC_OUT_CH >= p.Co) release_acc();      // last columns are in registers: the accumulator is free
          uint32_t pk[16];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            if (p.relu) pk[i >> 1] = pack2_relu<T>(__uint_as_float(va[i]), __uint_as_float(va[i + 1]));
            else { const H2 h = from_f2<T>(__uint_as_float(va[i]), __uint_as_float(va[i + 1])); pk[i >> 1] = *reinterpret_cast<const uint32_t*>(&h); }
          }
          emit_chunk(pk, 0.0f, 0.0f, 0.0f, 0.0f, c0, ci);
          if (two) {
#pragma unroll
            for (int i = 0; i < 32; i += 2) {
              if (p.relu) pk[i >> 1] = pack2_relu<T>(__uint_as_float(vb[i]), __uint_as_float(vb[i + 1]));
              else { const H2 h = from_f2<T>(__uint_as_float(vb[i]), __uint_as_float(vb[i + 1])); pk[i >> 1] = *reinterpret_cast<const uint32_t*>(&h); }
            }
            emit_chunk(pk, 0.0f, 0.0f, 0.0f, 0.0f, c0 + TC_OUT_CH, ci + 1);
          }
        }
      } else if (FD) {
        // ---- FAM decode: this thread owns one pixel.  d_k = T(acc_k + bias_k) is bit for bit what the ordinary epilogue
        // stores for channel k (and fam_decode_kernel reads back), and the decode is fam_decode_kernel's own code. ----
        uint32_t v[32];
        tmem_ld32(acc_addr, v);
        release_acc();                                    // the deltas are in registers: the accumulator is free
        if (valid) {
          float d[5], a[5], o[5];
#pragma unroll
          for (int k = 0; k < 5; ++k) d[k] = round_through<T>(__uint_as_float(v[k]) + __ldg(bias + k));
          fam_grid_anchor(x, y, L.stride, p.fd_scale, p.fd_angle, a);
          delta2bbox_rotated<T>(a, d[0], d[1], d[2], d[3], d[4], p.fd_lim, o);
          float* dst = L.refine + pos * 5;
#pragma unroll
          for (int k = 0; k < 5; ++k) dst[k] = o[k];
        }
      } else if (IS_PLAIN && p.sc_tap >= 0) {
        // ---- dgrad: scatter the column gradient of tap sc_tap (this thread: one pixel, 32 channels at a time) ----
        const int H = L.H, W = L.W, t = p.sc_tap;
        const int ti = t / 3, tj = t - 3 * ti;
        bool inb = false, c_t = false, c_b = false, c_l = false, c_r = false;
        float hy = 0.f, hx = 0.f, ly = 0.f, lx = 0.f;
        int yt = 0, xl = 0;
        if (valid) {
          const size_t oi = (((size_t)tc.b * 18 + 2 * t) * H + y) * W + x, plane = (size_t)H * W;
          float offy, offx;
          if (p.sc_off_f32) {
            offy = reinterpret_cast<const float*>(p.sc_off)[oi];
            offx = reinterpret_cast<const float*>(p.sc_off)[oi + plane];
          } else {
            offy = (float)reinterpret_cast<const T*>(p.sc_off)[oi];
            offx = (float)reinterpret_cast<const T*>(p.sc_off)[oi + plane];
          }
          const float h = (float)(y - 1 + ti) + offy, w = (float)(x - 1 + tj) + offx;
          if (h > -1.0f && w > -1.0f && h < (float)H && w < (float)W) {
            inb = true;
            const float hf = floorf(h), wf = floorf(w);
            const int y0 = (int)hf, x0 = (int)wf;
            ly = h - hf; lx = w - wf; hy = 1.0f - ly; hx = 1.0f - lx;
            c_t = y0 >= 0; c_b = y0 + 1 <= H - 1; c_l = x0 >= 0; c_r = x0 + 1 <= W - 1;
            yt = y0; xl = x0;
          }
        }
        const float w1 = (c_t && c_l) ? hy * hx : 0.f, w2 = (c_t && c_r) ? hy * lx : 0.f;
        const float w3 = (c_b && c_l) ? ly * hx : 0.f, w4 = (c_b && c_r) ? ly * lx : 0.f;
        const int Cg = p.Co;                                   // channels of x / grad_input (the GEMM's N)
        // clamped corner addresses (a corner outside the map has weight 0 and is never touched)
        const size_t rowp = (size_t)W * Cg;
        // per-corner element offsets: top-left (yt, xl), top-right (yt, xl + 1), bottom-left (yt + 1, xl), bottom-right
        const size_t a_tl = ((size_t)tc.b * H + max(yt, 0)) * rowp + (size_t)max(xl, 0) * Cg;
        const size_t a_tr = ((size_t)tc.b * H + max(yt, 0)) * rowp + (size_t)min(xl + 1, W - 1) * Cg;
        const size_t a_bl = ((size_t)tc.b * H + min(yt + 1, H - 1)) * rowp + (size_t)max(xl, 0) * Cg;
        const size_t a_br = ((size_t)tc.b * H + min(yt + 1, H - 1)) * rowp + (size_t)min(xl + 1, W - 1) * Cg;
        float gy = 0.f, gx = 0.f;
        // The reductions are issued COALESCED: a warp's 32 x 32-channel chunk goes through a 4 KB shared-memory
        // transpose (16-byte chunks XOR-swizzled by the pixel), then for every pixel of the warp lanes 8c .. 8c+7 add
        // the 128 contiguous bytes of corner c -- one instruction = four full 128-byte segments of grad_input.  (Round-2
        // first version: every lane reduced into its own pixel's row, 32 half-used sectors per instruction; the L2
        // reduction rate, not the tensor core, is what bounds this kernel.)
        float* s_tile = reinterpret_cast<float*>(s_out) + quad * 1024;                  // [32 px][32 ch] fp32
        uint32_t* s_corner = reinterpret_cast<uint32_t*>(s_out + 16384) + quad * 256;   // [32 px][4 weights | 4 offsets / 4]
        __syncwarp();
        s_corner[lane * 8 + 0] = __float_as_uint(w1); s_corner[lane * 8 + 1] = __float_as_uint(w2);
        s_corner[lane * 8 + 2] = __float_as_uint(w3); s_corner[lane * 8 + 3] = __float_as_uint(w4);
        // (offsets are multiples of C / 4 >= 8: bit 0 carries "this corner lies inside the map")
        s_corner[lane * 8 + 4] = (uint32_t)(a_tl >> 2) | ((inb && c_t && c_l) ? 1u : 0u);
        s_corner[lane * 8 + 5] = (uint32_t)(a_tr >> 2) | ((inb && c_t && c_r) ? 1u : 0u);
        s_corner[lane * 8 + 6] = (uint32_t)(a_bl >> 2) | ((inb && c_b && c_l) ? 1u : 0u);
        s_corner[lane * 8 + 7] = (uint32_t)(a_br >> 2) | ((inb && c_b && c_r) ? 1u : 0u);
        const int cn = lane >> 3, sub = lane & 7;
        // offset gradient (get_coordinate_weight, deform_conv_cuda_kernel.cu:147-187): needs D_c = <column gradient of
        // the pixel, x at corner c> for the four corners (a corner outside the map counts as zeros).  The lanes that
        // reduce corner c of pixel r into grad_input also load the matching 4 channels of x there (8 bytes each, 64
        // contiguous bytes per corner) and keep a partial D_c per pixel; the partials are combined after the channel loop.
        const bool want_goff = p.sc_goff != nullptr;
        float dacc[32];
#pragma unroll
        for (int r = 0; r < 32; ++r) dacc[r] = 0.f;
        for (int c0 = 0; c0 < p.Co; c0 += TC_OUT_CH) {
          uint32_t v[32];
          tmem_ld32(acc_addr + (uint32_t)c0, v);
          if (c0 + TC_OUT_CH >= p.Co) release_acc();
          __syncwarp();                                   // the previous chunk has been read by every lane
#pragma unroll
          for (int j = 0; j < 8; ++j)
            *reinterpret_cast<uint4*>(s_tile + lane * 32 + ((j ^ (lane & 7)) << 2)) =
                make_uint4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
          __syncwarp();
          // the x loads of the offset gradient are issued first: their latency hides behind the reduction loop (the
          // reductions are volatile asm statements no load can be scheduled across)
          uint2 xv[32];
          if (want_goff) {
            const T* xs = reinterpret_cast<const T*>(p.sc_x) + c0 + 4 * sub;
#pragma unroll
            for (int r = 0; r < 32; ++r) {
              const uint32_t ow = s_corner[r * 8 + 4 + cn];
              xv[r] = (ow & 1u) ? __ldg(reinterpret_cast<const uint2*>(xs + ((size_t)(ow & ~7u) << 2))) : make_uint2(0u, 0u);
            }
          }
          float* gi = p.sc_gi + c0 + 4 * sub;
#pragma unroll 4
          for (int r = 0; r < 32; ++r) {
            const float wq = __uint_as_float(s_corner[r * 8 + cn]);
            if (wq != 0.f) {
              const float4 q = *reinterpret_cast<const float4*>(s_tile + r * 32 + ((sub ^ (r & 7)) << 2));
              red_add_v4(gi + ((size_t)(s_corner[r * 8 + 4 + cn] & ~7u) << 2), wq * q.x, wq * q.y, wq * q.z, wq * q.w);
            }
          }
          if (want_goff) {
#pragma unroll
            for (int r = 0; r < 32; ++r) {
              const float4 q = *reinterpret_cast<const float4*>(s_tile + r * 32 + ((sub ^ (r & 7)) << 2));
              const float2 xa = to_f2(*reinterpret_cast<const H2*>(&xv[r].x)), xb = to_f2(*reinterpret_cast<const H2*>(&xv[r].y));
              dacc[r] += q.x * xa.x + q.y * xa.y + q.z * xb.x + q.w * xb.y;
            }
          }
        }
        if (want_goff) {
#pragma unroll
          for (int r = 0; r < 32; ++r) {
            float d = dacc[r];
            d += __shfl_xor_sync(0xffffffffu, d, 1);
            d += __shfl_xor_sync(0xffffffffu, d, 2);
            d += __shfl_xor_sync(0xffffffffu, d, 4);
            const float D1 = __shfl_sync(0xffffffffu, d, 0), D2 = __shfl_sync(0xffffffffu, d, 8);
            const float D3 = __shfl_sync(0xffffffffu, d, 16), D4 = __shfl_sync(0xffffffffu, d, 24);
            if (lane == r) {
              gy = hx * (D3 - D1) + lx * (D4 - D2);
              gx = hy * (D2 - D1) + ly * (D4 - D3);
            }
          }
        }
        if (p.sc_goff && valid) {       // one thread per (pixel, tap) and one tap per launch: plain read-modify-write
          float* go = p.sc_goff + (((size_t)tc.b * 18 + 2 * t) * H + y) * W + x;
          go[0] += gy;
          go[(size_t)H * W] += gx;
        }
      } else {
        // 32 channels at a time: TMEM -> registers -> bias / ReLU / 8-way orientation max -> 16-bit -> a 64-byte row
        // of the staging buffer (SWIZZLE_64B, conflict-free) -> one TMA store of the 8 x 16 x 32-channel box.  The
        // stores never touch the LSU global path, and partial tiles are clipped by TMA.
        for (int c0 = 0, ci = 0; c0 < p.Co && !(p.debug & 32); c0 += TC_OUT_CH, ++ci) {
          uint32_t v[32];
          tmem_ld32(acc_addr + (uint32_t)c0, v);
          if (c0 + TC_OUT_CH >= p.Co) release_acc();          // last columns are in registers: the accumulator is free
          uint32_t pk[16];
          float m[4];
#pragma unroll
          for (int i = 0; i < 32; i += 2) {
            float t0 = __uint_as_float(v[i]), t1 = __uint_as_float(v[i + 1]);
            if (bias) { t0 += __ldg(bias + c0 + i); t1 += __ldg(bias + c0 + i + 1); }
            if (p.relu) { t0 = fmaxf(t0, 0.0f); t1 = fmaxf(t1, 0.0f); }
            const H2 h = from_f2<T>(t0, t1);
            pk[i >> 1] = *reinterpret_cast<const uint32_t*>(&h);
            const float mx = fmaxf(t0, t1);
            m[i >> 3] = (i & 7) == 0 ? mx : fmaxf(m[i >> 3], mx);
          }
          emit_chunk(pk, m[0], m[1], m[2], m[3], c0, ci);
        }
      }
      if (p.debug & 32) { tc_fence_before(); __syncwarp(); if (lane == 0) mbar_arrive_cluster(ld_acc_empty + 8 * as); }
      if (MODE == TC_ALIGN) {
        // every A k-block of tile `it` has been produced (its MMAs completed), so table (it & 1) is free:
        // build the table of tile it + 2 into it
        const int nxt = q + 2 * q_step;
        if (nxt < ngroups) {
          build_tap_table<T>(p, decode_tile<MODE>(p, S2A_TILE_OF(nxt)), s_tab + tb * (TC_M * 9), et, TC_EPI_THREADS);
          mbar_arrive(bar_tab_full + 8 * tb);
        }
      }
    }
  };
  if (MODE == TC_ALIGN) {
    // Warpgroups 0-3: producers (80 registers, the launch value), 4: epilogue, 5: TMA / MMA / two idle warps.  The
    // last one gives registers back and the epilogue takes them (setmaxnreg is a warpgroup-wide instruction, so each
    // role's code sits under the branch of its warpgroup and ptxas allocates per branch).
    if (warp < kProdWarps) {
      role_producer();
    } else if (warp < kTmaWarp) {
      reg_alloc<104>();
      role_epilogue();
    } else {
      reg_dealloc<56>();
      if (warp == kTmaWarp) role_tma();
      else if (warp == kMmaWarp) role_mma();
    }
  } else {
    if (warp == kTmaWarp) role_tma();
    else if (warp == kMmaWarp + 1) role_halo();
    else if (warp == kMmaWarp) role_mma();
    else if (warp >= kEpiWarp0 && warp < kTmaWarp) role_epilogue();
  }
#undef S2A_TILE_OF
#undef S2A_IS_GHOST
  if (warp >= kEpiWarp0 && warp < kTmaWarp) tma_store_wait_all();   // (the lanes that issued output stores wait for them)
  tc_fence_before();
  if (CG == 2) cluster_sync_all();   // no CTA may exit (or free TMEM) while its partner can still signal / read it
  else __syncthreads();
#ifdef S2A_TC_TIMELINE
  if ((p.debug & 8) && blockIdx.x == 0 && tid == 0) {
    unsigned long long t1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
    const long long c1 = clock64();
    printf("s2a conv_tc clock probe: %lld cycles in %llu ns = %.0f MHz\n", c1 - dbg_c0, t1 - dbg_t0,
           (double)(c1 - dbg_c0) * 1e3 / (double)(t1 - dbg_t0));
  }
#endif
  if (warp == kMmaWarp) {
    tc_fence_after();
    tmem_dealloc<CG>(tmem_base, TC_TMEM_COLS);
  }
}

// ---------------------------------------------------------------------------------------------
// weight packing: [Co][C][3][3] (any of f32/bf16/f16) -> [Co][(cb, tap, c64)] 16-bit, optionally
// through the ARF map (ORConv: w [O, I, nOri, 3, 3], indices [nOri*9, nRot])
// ---------------------------------------------------------------------------------------------
// AlignConv keeps its A operand in tensor memory, written with tcgen05.st 16x256b fragments: thread q = T%4 of a
// row holds the row's 16-byte chunks q and q + 4, which land at TMEM K-byte offsets 32g + 8q (g = 0..3).  This is
// the channel (inside a 64-channel block) that sits at K position p of the A operand; the packed AlignConv
// weights use the same order.
__host__ __device__ inline int tc_kperm(int p) {
  const int b = 2 * p, g = b >> 5, q = (b & 31) >> 3, t = b & 7;
  const int pix_byte = g < 2 ? 16 * q + 8 * g + t : 64 + 16 * q + 8 * (g - 2) + t;
  return pix_byte >> 1;
}

template <typename TIn, typename TOut>
__global__ void pack_weight_kernel(const TIn* __restrict__ w, const uint8_t* __restrict__ arf_idx, TOut* __restrict__ wp,
                                   int Co, int C, int nOri, int nRot, int arfI) {
  __shared__ uint8_t s_inv[8 * 72];
  const int nEntry = nOri * 9;
  if (arf_idx) {
    for (int i = threadIdx.x; i < nEntry * nRot; i += blockDim.x) {
      const int l = i / nRot, k = i % nRot;
      s_inv[k * nEntry + ((int)arf_idx[i] - 1)] = (uint8_t)l;
    }
    __syncthreads();
  }
  const int64_t total = (int64_t)Co * C * 9;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    // destination order: n, cb, tap, c
    const int c = (int)(e % 64);
    int64_t r = e / 64;
    const int tap = (int)(r % 9);
    r /= 9;
    const int cb = (int)(r % (C / 64));
    const int n = (int)(r / (C / 64));
    const int cin = cb * 64 + (arf_idx ? c : tc_kperm(c));   // no ARF map = AlignConv weights: TMEM A operand order
    float v;
    if (arf_idx) {
      const int o = n / nRot, k = n % nRot;
      const int ii = cin / nOri, lay = cin % nOri;
      const int l = s_inv[k * nEntry + lay * 9 + tap];
      v = (float)w[((int64_t)o * arfI + ii) * nEntry + l];
    } else {
      v = (float)w[((int64_t)n * C + cin) * 9 + tap];
    }
    wp[e] = (TOut)v;
  }
}

// plain conv weights [Co][C][ks][ks] -> [Co_pad][(cb, tap, c64)] with C padded to a multiple of 64 and Co to
// Co_pad (zero rows / zero channels), for the stock conv layers of the head routed through conv_tc_kernel<PLAIN>
template <typename TIn, typename TOut>
__global__ void pack_conv2d_kernel(const TIn* __restrict__ w, TOut* __restrict__ wp, int Co, int Co_pad, int C, int ncb,
                                   int ntap) {
  const int64_t total = (int64_t)Co_pad * ncb * ntap * 64;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int c = (int)(e % 64);
    int64_t r = e / 64;
    const int tap = (int)(r % ntap);
    r /= ntap;
    const int cb = (int)(r % ncb);
    const int n = (int)(r / ncb);
    const int cin = cb * 64 + c;
    const float v = (n < Co && cin < C) ? (float)w[((int64_t)n * C + cin) * ntap + tap] : 0.0f;
    wp[e] = (TOut)v;
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

template <int MODE>
constexpr size_t tc_smem_bytes() {
  using Cfg = TcCfg<MODE>;
  return 1024 /*alignment slack*/ + (size_t)Cfg::SB * Cfg::KPS * (Cfg::BROWS * TC_KB * 2) +
         (size_t)TC_OUT_BUFS * TC_OUT_BYTES +
         (MODE == TC_ALIGN ? 2 * (size_t)TC_HALO_BYTES + 2 * sizeof(TapSample) * TC_M * 9
                           : (size_t)Cfg::NHALO * TC_PHALO_BYTES) +
         8 * TC_NBAR + 16;
}

template <int MODE, typename T, bool FD = false>
static int launch_tc(const TcMaps& tmap, const TcParams& p, cudaStream_t st) {
  constexpr int CG = TcCfg<MODE>::CG;
  auto kern = conv_tc_kernel<MODE, T, FD>;
  constexpr size_t smem = tc_smem_bytes<MODE>();
  static_assert(smem <= 227 * 1024, "shared memory budget");
  S2A_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // persistent: at most one CTA per SM, launched as clusters of CG CTAs (CG = 2: a CTA pair = one TPC)
  const int ngroups = (p.total_tiles + CG - 1) / CG;
  const int nclusters = std::max(1, std::min(ngroups, sm_count() / CG));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3((unsigned)(nclusters * CG));
  cfg.blockDim = dim3(tc_threads<MODE>());
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  S2A_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, tmap, p));
  S2A_LAUNCH_OK("conv_tc_kernel");
  return S2A_OK;
}

struct TcScatter { float* gi; float* goff; const void* x; const void* off; int off_f32; int tap; };
struct TcFamDecode { float* const* refined; float scale, angle, lim; };

static int conv_tc_common(int mode, int nlevels, const void* const* xs, const float* const* anchors, const void* wp,
                          const float* bias, void* const* outs, void* const* pooleds, const int* Hs, const int* Ws,
                          const float* strides, int B, int C, int Co, int relu, int dtype, cudaStream_t st, int ks = 3,
                          int wsplit = -1, const void* wp2 = nullptr, const float* bias2 = nullptr,
                          const void* const* offsets = nullptr, int off_f32 = 0, int pos_round = 0,
                          const TcScatter* sc = nullptr, const TcFamDecode* fd = nullptr) {
  if (wsplit < 0) wsplit = nlevels;              // one problem: every level uses the first weights
  S2A_CHECK_ARG(nlevels >= 1 && nlevels <= TC_MAX_LEVELS, "conv_tc: 1..%d levels per launch", TC_MAX_LEVELS);
  S2A_CHECK_ARG(B >= 0 && C > 0 && Co > 0, "conv_tc: bad tensor sizes");
  S2A_CHECK_ARG(dtype == S2A_BF16 || dtype == S2A_F16, "conv_tc: dtype must be bf16 or f16");
  S2A_CHECK_ARG(ks == 3 || (ks == 1 && mode == TC_PLAIN), "conv_tc: kernel size must be 3 (or 1 for the plain conv)");
  if ((mode == TC_ALIGN ? C % 64 != 0 : C % 8 != 0) || Co % 32 != 0 || Co > 256) {
    set_error("conv_tc: needs C %% 64 == 0 (plain conv: C %% 8 == 0) and C_out a multiple of 32 up to 256 (got C=%d, C_out=%d)",
              C, Co);
    return S2A_ERR_UNSUPPORTED;
  }
  const int Kp = ((C + TC_KB - 1) / TC_KB) * TC_KB * ks * ks;      // packed K' (C padded to 64-channel blocks)
  if (B == 0) return S2A_OK;
  S2A_CHECK_ARG(xs && wp && (fd ? fd->refined != nullptr : outs != nullptr) && Hs && Ws, "conv_tc: null pointer");
  TcParams p{};
  long long tiles = 0;
  for (int l = 0; l < nlevels; ++l) {
    S2A_CHECK_ARG(Hs[l] > 0 && Ws[l] > 0 && Hs[l] < 32768 && Ws[l] < 32768, "conv_tc: bad feature map size");
    S2A_CHECK_ARG((long long)Hs[l] * Ws[l] * C * 2 < (1ll << 32), "conv_tc: one image of a level must be < 4 GiB");
    S2A_CHECK_ARG(xs[l] && (fd ? fd->refined[l] != nullptr : outs[l] != nullptr) &&
                  (mode == TC_PLAIN || (anchors && anchors[l]) || (offsets && offsets[l])), "conv_tc: null level pointer");
    TcLevel& L = p.lv[l];
    L.x = xs[l]; L.anchors = anchors ? anchors[l] : nullptr; L.out = outs ? outs[l] : nullptr;
    L.pooled = pooleds ? pooleds[l] : nullptr; L.refine = fd ? fd->refined[l] : nullptr;
    L.offsets = offsets ? offsets[l] : nullptr;
    L.H = Hs[l]; L.W = Ws[l];
    const int pw = mode == TC_PLAIN ? TC_PPW : TC_PW, ph = mode == TC_PLAIN ? TC_PPH : TC_PH;
    L.tiles_x = (Ws[l] + pw - 1) / pw; L.tiles_y = (Hs[l] + ph - 1) / ph;
    if (l == wsplit) tiles += tiles & 1;         // the second problem starts at an even tile: pairs never mix weights
    L.tile_begin = (int)tiles;
    L.stride = strides ? strides[l] : 1.0f;
    S2A_CHECK_ARG((mode == TC_PLAIN && !fd) || L.stride > 0.0f, "conv_tc: stride must be positive");
    tiles += (long long)B * L.tiles_x * L.tiles_y;
  }
  S2A_CHECK_ARG(tiles < (1ll << 31), "conv_tc: too many tiles");
  S2A_CHECK_ARG(!(pooleds && pooleds[0]) || Co % 8 == 0, "conv_tc: pooling needs C_out %% 8 == 0");
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_error("conv_tc: cuTensorMapEncodeTiled is not available from the driver"); return S2A_ERR_CUDA; }
  TcMaps tmap;
  memset(&tmap, 0, sizeof(tmap));
  const CUtensorMapDataType tdt = dtype == S2A_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  for (int l = 0; l < nlevels; ++l) {
    // TC_PLAIN: halo windows {64 ch, 16, 18, 1} (SWIZZLE_128B, read by the tensor core as the A operand of every
    // tap; a 1 x 1 conv loads the bare tile {64 ch, 8, 16, 1}); TC_ALIGN: halo windows {64 ch, 22, 14, 1}, plain layout (one 128-byte line per pixel, gathered by
    // LDS); both zero-filled outside the map
    const cuuint64_t xd[4] = {(cuuint64_t)C, (cuuint64_t)Ws[l], (cuuint64_t)Hs[l], (cuuint64_t)B};
    const cuuint64_t xs_[3] = {(cuuint64_t)C * 2, (cuuint64_t)Ws[l] * C * 2, (cuuint64_t)Hs[l] * Ws[l] * C * 2};
    const cuuint32_t xb[4] = {(cuuint32_t)TC_KB, (cuuint32_t)(mode == TC_PLAIN ? (ks == 3 ? TC_PHALO_PITCH : TC_PPW) : TC_HW),
                              (cuuint32_t)(mode == TC_PLAIN ? (ks == 3 ? TC_PHALO_ROWS : TC_PPH) : TC_HH), 1};
    const cuuint32_t xe[4] = {1, 1, 1, 1};
    CUresult xr = enc(&tmap.x[l], tdt, 4, const_cast<void*>(xs[l]), xd, xs_, xb, xe, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      mode == TC_PLAIN ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (xr != CUDA_SUCCESS) { set_error("conv_tc: cuTensorMapEncodeTiled (x, level %d) failed (%d)", l, (int)xr); return S2A_ERR_CUDA; }
  }
  for (int l = 0; l < nlevels && !fd; ++l) {         // (the FAM decode stores no feature map)
    const cuuint64_t yd[4] = {(cuuint64_t)Co, (cuuint64_t)Ws[l], (cuuint64_t)Hs[l], (cuuint64_t)B};
    const cuuint64_t ys_[3] = {(cuuint64_t)Co * 2, (cuuint64_t)Ws[l] * Co * 2, (cuuint64_t)Hs[l] * Ws[l] * Co * 2};
    const int pw = mode == TC_PLAIN ? TC_PPW : TC_PW;
    const cuuint32_t yb[4] = {(cuuint32_t)TC_OUT_CH, (cuuint32_t)pw, (cuuint32_t)(32 / pw), 1};      // one epilogue warp's 32 tile rows
    const cuuint32_t ye[4] = {1, 1, 1, 1};
    CUresult yr = enc(&tmap.y[l], tdt, 4, outs[l], yd, ys_, yb, ye, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (yr != CUDA_SUCCESS) { set_error("conv_tc: cuTensorMapEncodeTiled (out, level %d) failed (%d)", l, (int)yr); return S2A_ERR_CUDA; }
  }
  const cuuint64_t gdim[2] = {(cuuint64_t)Kp, (cuuint64_t)Co};
  const cuuint64_t gstr[1] = {(cuuint64_t)Kp * 2};
  const int cg = mode == TC_PLAIN ? TcCfg<TC_PLAIN>::CG : TcCfg<TC_ALIGN>::CG;
  const cuuint32_t box[2] = {(cuuint32_t)TC_KB, (cuuint32_t)(Co / cg)};   // each CTA of a group stages 1/CG of the rows
  const cuuint32_t estr[2] = {1, 1};
  for (int wi = 0; wi < 2; ++wi) {
    const void* wsrc = wi == 0 ? wp : (wp2 ? wp2 : wp);
    CUresult cr = enc(&tmap.w[wi], tdt, 2,
                      const_cast<void*>(wsrc), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("conv_tc: cuTensorMapEncodeTiled failed (%d)", (int)cr); return S2A_ERR_CUDA; }
  }
  p.bias = bias; p.bias2 = bias2; p.wsplit = wsplit; p.nlevels = nlevels; p.total_tiles = (int)tiles;
  p.B = B; p.C = C; p.Co = Co; p.relu = relu; p.ks = ks; p.off_f32 = off_f32; p.pos_round = pos_round;
  p.sc_tap = -1;
  if (sc) {
    S2A_CHECK_ARG(mode == TC_PLAIN && ks == 1 && nlevels == 1 && sc->tap >= 0 && sc->tap < 9 && sc->gi && sc->off &&
                  (!sc->goff || sc->x), "conv_tc: bad dgrad (scatter) arguments");
    p.sc_gi = sc->gi; p.sc_goff = sc->goff; p.sc_x = sc->x; p.sc_off = sc->off; p.sc_off_f32 = sc->off_f32; p.sc_tap = sc->tap;
  }
  { const char* e = getenv("S2A_TC_DEBUG"); p.debug = e ? atoi(e) : 0; }
  if (fd) {
    S2A_CHECK_ARG(mode == TC_PLAIN && ks == 1 && Co == TC_OUT_CH && !relu && bias && !sc && !(pooleds && pooleds[0]),
                  "conv_tc: bad FAM-decode arguments");
    p.fd_scale = fd->scale; p.fd_angle = fd->angle; p.fd_lim = fd->lim;
    return dtype == S2A_BF16 ? launch_tc<TC_PLAIN, __nv_bfloat16, true>(tmap, p, st)
                             : launch_tc<TC_PLAIN, __half, true>(tmap, p, st);
  }
  if (mode == TC_ALIGN) {
    return dtype == S2A_BF16 ? launch_tc<TC_ALIGN, __nv_bfloat16>(tmap, p, st) : launch_tc<TC_ALIGN, __half>(tmap, p, st);
  }
  if (Co == 2 * TcCfg<TC_PLAIN_S>::BROWS && ks == 3)          // the narrow prediction convs: nine taps per stage
    return dtype == S2A_BF16 ? launch_tc<TC_PLAIN_S, __nv_bfloat16>(tmap, p, st) : launch_tc<TC_PLAIN_S, __half>(tmap, p, st);
  return dtype == S2A_BF16 ? launch_tc<TC_PLAIN, __nv_bfloat16>(tmap, p, st) : launch_tc<TC_PLAIN, __half>(tmap, p, st);
}

// =================================================================================================
// wgrad: dW[co, c, tap] = sum_pixels grad_out[pixel, co] * S[pixel, tap, c]   (S = the bilinear samples of the forward)
//
// Replaces deform_conv_backward_parameters_cuda for S2ANet's geometry (models/dcn/src/deform_conv_cuda.cpp:376-489:
// deformable_im2col into a [C*9, H*W] column buffer + addmm_).  The contraction runs over PIXELS, so both operands
// arrive "MN-major" for the tensor core: grad_out is NHWC ([pixel][co], co contiguous) and a tile of samples is
// [pixel][channel].  Both are 128-byte rows in SWIZZLE_128B shared memory -- exactly the tiles the forward kernels
// already build -- read through MN-major descriptors (canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units:
// 64 M/N elements per 128-byte row, K rows 128 B apart, 8-row groups SBO = 1024 B apart, the next 64 M/N elements LBO
// away; instruction-descriptor bits 15 / 16 select MN-major A / B).  No column buffer, no library GEMM.
//
// One CTA (no pairs) owns ONE TAP and every `ngroups`-th 8 x 16-pixel tile: its accumulator dW[:, :, tap] -- Co x C fp32 =
// 2 x 128 lanes x 256 columns -- stays in tensor memory (all 512 columns) across its tiles and is added to global memory
// once at the end (red.global.add.v4.f32 into a [9][Co][C] buffer).  Per tile: a TMA warp loads the grad_out tile
// (Co/64 boxes {64 co, 16, 8, 1}, two buffers); 16 producer warps compute their pixel's sampling position from the
// offsets, gather the four corners straight from global memory (L2), blend in packed 16-bit math like the forward and
// store 128-byte sample rows, swizzled, into the two 32 KB stages (128 channels each); the MMA warp issues, per stage,
// Co/128 x 8 tcgen05.mma (M = 128 co, N = 128 channels, K = 16 pixels).
// =================================================================================================
constexpr int WG_PROD_WARPS = 16;
constexpr int WG_THREADS = (WG_PROD_WARPS + 2) * 32;          // + TMA warp + MMA warp
constexpr int WG_BLOCK_BYTES = TC_M * 128;                    // one [128 pixels x 64 channels] sub-tile: 16 KB
constexpr int WG_STAGE_BYTES = 2 * WG_BLOCK_BYTES;            // a stage: 128 channels
constexpr int WG_G_BYTES = 4 * WG_BLOCK_BYTES;                // a grad_out tile: up to 256 co
constexpr size_t WG_SMEM = 1024 + 2 * WG_STAGE_BYTES + 2 * WG_G_BYTES + 16 * 8 + 16;

struct WgParams {
  const void* x;          // [B, H, W, C] 16-bit
  const void* off;        // [B, 18, H, W]
  float* dwt;             // [9, Co, C] fp32, accumulated
  int off_f32;
  int B, C, Co, H, W, tiles_x, tiles_y, total_tiles;
};

// MN-major, SWIZZLE_128B shared-memory matrix descriptor (see the header comment)
__device__ __forceinline__ uint64_t umma_desc_mn_sw128(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes = 1024) {
  return (uint64_t)((smem_addr & 0x3FFFFu) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFFu) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFFu) << 32) | (1ull << 46) | (2ull << 61);
}

template <typename T>
__global__ void __launch_bounds__(WG_THREADS, 1)
wgrad_tc_kernel(const __grid_constant__ CUtensorMap gmap, const WgParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sS = smem;                                   // 2 stages x 32 KB
  uint8_t* sG = sS + 2 * WG_STAGE_BYTES;                // 2 grad_out tiles x 64 KB
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(sG + 2 * WG_G_BYTES);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 16);
  const uint32_t bar_s_full = smem_u32(s_bar), bar_s_empty = bar_s_full + 16, bar_g_full = bar_s_full + 32,
                 bar_g_empty = bar_s_full + 48, bar_acc = bar_s_full + 64;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int tap = blockIdx.x % 9, grp = blockIdx.x / 9, ngrp = gridDim.x / 9;
  const int nh = p.Co / 128;                            // output-channel halves (MMA M = 128)
  const int nf = p.C / 128;                             // stage fills per tile (128 channels each)

  if (tid == 0) {
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_s_full + 8 * s, WG_PROD_WARPS / 2);  // one elected arrive per producer warp of the stage
      mbar_init(bar_s_empty + 8 * s, 1);                 // tcgen05.commit
      mbar_init(bar_g_full + 8 * s, 1);                  // expect_tx arrive (+ bytes)
      mbar_init(bar_g_empty + 8 * s, 1);                 // tcgen05.commit
    }
    mbar_init(bar_acc, 1);
    fence_barrier_init();
  }
  if (warp == WG_PROD_WARPS + 1) tmem_alloc<1>(smem_u32(s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  const int my_tiles = grp < p.total_tiles ? (p.total_tiles - grp + ngrp - 1) / ngrp : 0;

  if (warp < WG_PROD_WARPS) {
    // ===================== producers: sample rows into the stages =====================
    // group = 4 warps = the 128 pixels of a tile for ONE 64-channel block; groups 2f, 2f + 1 fill stage f
    const int group = warp >> 2, f = group >> 1, sub = group & 1;
    const int r = (warp & 3) * 32 + lane;               // tile row = pixel (y = r / 16, x = r % 16)
    const int ti = tap / 3, tj = tap - 3 * ti;
    const uint32_t dst_tile = smem_u32(sS) + (uint32_t)(f * WG_STAGE_BYTES + sub * WG_BLOCK_BYTES + (warp & 3) * (32 * 128));   // this warp's 32 rows
    const int cb = 2 * f + sub;                         // 64-channel block of x this thread samples
    // lane = the pixel whose parameters it computes; the loads are issued with eight lanes per pixel (four full 128-byte
    // lines per warp instruction, parameters by shuffle) -- see conv_tf32x3_kernel
    const int src0 = lane >> 3, jch = lane & 7;
    for (int it = 0; it < my_tiles && f < nf; ++it) {
      int tile = grp + it * ngrp;
      const int tpi = p.tiles_x * p.tiles_y;
      const int b = tile / tpi;
      tile -= b * tpi;
      const int ty0 = (tile / p.tiles_x) * TC_PH, tx0 = (tile % p.tiles_x) * TC_PW;
      const int y = ty0 + r / TC_PW, x = tx0 + r % TC_PW;
      // this pixel's sampling position for the CTA's tap (deform_conv_cuda_kernel.cu:218-227) -> corners + weights
      uint32_t w01 = 0u, w23 = 0u;
      uint32_t base = 0;      // (element offset of the clamped top-left corner) / 8, bit 0: right neighbour, bit 1: lower one
      const size_t rowp = (size_t)p.W * p.C;
      if (y < p.H && x < p.W) {
        const size_t oi = (((size_t)b * 18 + 2 * tap) * p.H + y) * p.W + x, plane = (size_t)p.H * p.W;
        float offy, offx;
        if (p.off_f32) {
          offy = reinterpret_cast<const float*>(p.off)[oi];
          offx = reinterpret_cast<const float*>(p.off)[oi + plane];
        } else {
          offy = (float)reinterpret_cast<const T*>(p.off)[oi];
          offx = (float)reinterpret_cast<const T*>(p.off)[oi + plane];
        }
        const float h = (float)(y - 1 + ti) + offy, w = (float)(x - 1 + tj) + offx;
        if (h > -1.0f && w > -1.0f && h < (float)p.H && w < (float)p.W) {
          const float hf = floorf(h), wf = floorf(w);
          const int y0 = (int)hf, x0 = (int)wf;
          const float ly = h - hf, lx = w - wf, hy = 1.0f - ly, hx = 1.0f - lx;
          const bool t_ok = y0 >= 0, b_ok = y0 + 1 <= p.H - 1, l_ok = x0 >= 0, r_ok = x0 + 1 <= p.W - 1;
          using H2 = typename Half2Of<T>::type;
          const H2 p01 = from_f2<T>((t_ok && l_ok) ? hy * hx : 0.0f, (t_ok && r_ok) ? hy * lx : 0.0f);
          const H2 p23 = from_f2<T>((b_ok && l_ok) ? ly * hx : 0.0f, (b_ok && r_ok) ? ly * lx : 0.0f);
          w01 = *reinterpret_cast<const uint32_t*>(&p01);
          w23 = *reinterpret_cast<const uint32_t*>(&p23);
          const size_t img = (size_t)b * p.H * rowp;
          const int yt = max(y0, 0), xl = max(x0, 0);
          const bool has_r = min(x0 + 1, p.W - 1) > xl, has_b = min(y0 + 1, p.H - 1) > yt;
          // (C is a multiple of 64: the offset / 8 has its low three bits free)
          base = (uint32_t)((img + yt * rowp + (size_t)xl * p.C) >> 3) | (has_r ? 1u : 0u) | (has_b ? 2u : 0u);
        }
      }
      const T* xp = reinterpret_cast<const T*>(p.x) + cb * 64 + 8 * jch;
      // batches of two iterations: shuffles + eight corner loads first, then the blends and stores (volatile asm keeps
      // loads and stores in program order: interleaved, every iteration paid its own L2 round trip); no branch around
      // the loads (base 0 is a valid address, zero weights give a zero row); the first batch flies while the stage drains
#pragma unroll 1
      for (int i0 = 0; i0 < 8; i0 += 2) {               // four pixels x eight 16-byte chunks (8 channels) per instruction
        uint4 q[2][4];
        uint32_t s01[2], s23[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int src = 4 * (i0 + u) + src0;
          s01[u] = __shfl_sync(0xffffffffu, w01, src);
          s23[u] = __shfl_sync(0xffffffffu, w23, src);
          const uint32_t sb = __shfl_sync(0xffffffffu, base, src);
          const T* q0 = xp + ((size_t)(sb & ~7u) << 3);
          const size_t dx = (sb & 1u) ? (size_t)p.C : 0, dy = (sb & 2u) ? rowp : 0;
          q[u][0] = ldg_nc_v4(q0); q[u][1] = ldg_nc_v4(q0 + dx);
          q[u][2] = ldg_nc_v4(q0 + dy); q[u][3] = ldg_nc_v4(q0 + dy + dx);
        }
        if (i0 == 0) mbar_wait(bar_s_empty + 8 * f, (uint32_t)(it & 1) ^ 1u);
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int src = 4 * (i0 + u) + src0;
          uint4 o = blend4<T>(q[u][0], q[u][1], q[u][2], q[u][3], s01[u], s23[u]);
          if ((s01[u] | s23[u]) == 0u) o = make_uint4(0u, 0u, 0u, 0u);          // (0 x NaN of an unrelated pixel)
          sts_v4(dst_tile + (uint32_t)(src * 128 + ((jch ^ (src & 7)) << 4)), o.x, o.y, o.z, o.w);          // SWIZZLE_128B
        }
      }
      fence_proxy_async_smem();                          // generic-proxy stores -> visible to the tensor core
      __syncwarp();
      if (lane == 0) mbar_arrive(bar_s_full + 8 * f);
    }
  } else if (warp == WG_PROD_WARPS) {
    // ===================== TMA: grad_out tiles =====================
    for (int it = 0; it < my_tiles; ++it) {
      int tile = grp + it * ngrp;
      const int tpi = p.tiles_x * p.tiles_y;
      const int b = tile / tpi;
      tile -= b * tpi;
      const int ty0 = (tile / p.tiles_x) * TC_PH, tx0 = (tile % p.tiles_x) * TC_PW;
      const int buf = it & 1;
      mbar_wait(bar_g_empty + 8 * buf, ((uint32_t)(it >> 1) & 1u) ^ 1u);
      if (elect_one()) {
        mbar_arrive_expect_tx(bar_g_full + 8 * buf, (uint32_t)(p.Co / 64) * WG_BLOCK_BYTES);
        for (int j = 0; j < p.Co / 64; ++j)
          tma_load_4d<1>(smem_u32(sG + buf * WG_G_BYTES + j * WG_BLOCK_BYTES), &gmap, j * 64, tx0, ty0, b, bar_g_full + 8 * buf);
      }
      __syncwarp();
    }
  } else {
    // ===================== MMA issuer =====================
    const uint32_t fmt = std::is_same<T, __nv_bfloat16>::value ? 1u : 0u;
    // D = f32, A / B format, A and B MN-major (bits 15, 16), N = 128, M = 128
    const uint32_t idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | (1u << 15) | (1u << 16) | ((uint32_t)(128 >> 3) << 17) |
                           ((uint32_t)(128 >> 4) << 24);
    for (int it = 0; it < my_tiles; ++it) {
      const int buf = it & 1;
      mbar_wait(bar_g_full + 8 * buf, (uint32_t)(it >> 1) & 1u);
      for (int f = 0; f < nf; ++f) {
        mbar_wait(bar_s_full + 8 * f, (uint32_t)(it & 1));
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sbase = smem_u32(sS + f * WG_STAGE_BYTES);
          for (int h = 0; h < nh; ++h) {
            const uint32_t gbase = smem_u32(sG + buf * WG_G_BYTES + 2 * h * WG_BLOCK_BYTES);
            const uint32_t d_tmem = tmem_base + (uint32_t)(h * 256 + f * 128);
#pragma unroll
            for (int k = 0; k < 8; ++k) {               // K = 16 pixels per MMA: two 8-row groups = 2048 bytes
              const uint64_t adesc = umma_desc_mn_sw128(gbase + k * 2048, WG_BLOCK_BYTES);
              const uint64_t bdesc = umma_desc_mn_sw128(sbase + k * 2048, WG_BLOCK_BYTES);
              umma_f16<1>(d_tmem, adesc, bdesc, idesc, (it | k) != 0 ? 1u : 0u);
            }
          }
          umma_commit<1>(bar_s_empty + 8 * f);           // the stage may be refilled once these MMAs have read it
          if (f == nf - 1) umma_commit<1>(bar_g_empty + 8 * buf);
          if (f == nf - 1 && it == my_tiles - 1) umma_commit<1>(bar_acc);
        }
        __syncwarp();
      }
    }
  }

  // ===================== epilogue: tensor memory -> dWt[tap] (fp32, atomics; once per CTA) =====================
  if (my_tiles > 0 && warp < 4) {
    mbar_wait(bar_acc, 0u);
    tc_fence_after();
    for (int h = 0; h < nh; ++h) {
      float* orow = p.dwt + ((size_t)tap * p.Co + h * 128 + warp * 32 + lane) * p.C;
      for (int c0 = 0; c0 < p.C; c0 += 32) {
        uint32_t v[32];
        tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(h * 256 + c0), v);
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          red_add_v4(orow + c0 + j, __uint_as_float(v[j]), __uint_as_float(v[j + 1]), __uint_as_float(v[j + 2]),
                     __uint_as_float(v[j + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == WG_PROD_WARPS + 1) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

static int launch_wgrad(const void* x, const void* off, int off_f32, const void* grad_out, float* dwt, int B, int C, int H,
                        int W, int Co, int dtype, cudaStream_t st) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_error("wgrad_tc: cuTensorMapEncodeTiled is not available from the driver"); return S2A_ERR_CUDA; }
  CUtensorMap gmap;
  memset(&gmap, 0, sizeof(gmap));
  const CUtensorMapDataType tdt = dtype == S2A_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const cuuint64_t gd[4] = {(cuuint64_t)Co, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
  const cuuint64_t gs[3] = {(cuuint64_t)Co * 2, (cuuint64_t)W * Co * 2, (cuuint64_t)H * W * Co * 2};
  const cuuint32_t gb[4] = {64, (cuuint32_t)TC_PW, (cuuint32_t)TC_PH, 1};
  const cuuint32_t ge[4] = {1, 1, 1, 1};
  CUresult cr = enc(&gmap, tdt, 4, const_cast<void*>(grad_out), gd, gs, gb, ge, CU_TENSOR_MAP_INTERLEAVE_NONE,
                    CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (cr != CUDA_SUCCESS) { set_error("wgrad_tc: cuTensorMapEncodeTiled failed (%d)", (int)cr); return S2A_ERR_CUDA; }
  WgParams p{};
  p.x = x; p.off = off; p.dwt = dwt; p.off_f32 = off_f32; p.B = B; p.C = C; p.Co = Co; p.H = H; p.W = W;
  p.tiles_x = (W + TC_PW - 1) / TC_PW; p.tiles_y = (H + TC_PH - 1) / TC_PH;
  const long long tiles = (long long)B * p.tiles_x * p.tiles_y;
  S2A_CHECK_ARG(tiles < (1ll << 31), "wgrad_tc: too many tiles");
  p.total_tiles = (int)tiles;
  const int groups = std::max(1, std::min((int)std::min<long long>(tiles, 1 << 20), sm_count() / 9));
  if (dtype == S2A_BF16) {
    S2A_CUDA_OK(cudaFuncSetAttribute(wgrad_tc_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG_SMEM));
    wgrad_tc_kernel<__nv_bfloat16><<<9 * groups, WG_THREADS, WG_SMEM, st>>>(gmap, p);
  } else {
    S2A_CUDA_OK(cudaFuncSetAttribute(wgrad_tc_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)WG_SMEM));
    wgrad_tc_kernel<__half><<<9 * groups, WG_THREADS, WG_SMEM, st>>>(gmap, p);
  }
  S2A_LAUNCH_OK("wgrad_tc_kernel");
  return S2A_OK;
}

// =================================================================================================
// fp32 AlignConv / DeformConv / ORConv2d on the tensor cores: 3 x TF32 split (round 2)
//
// The exact-order fp32 path of round 1 (conv_f32.cu, SIMT FMAs fed by a scalar NCHW gather) ran AlignConv at P3 in
// 0.98 ms where the reference's im2col + cuBLAS SGEMM takes 0.59 ms.  Here the same contraction runs on
// tcgen05.mma.kind::tf32 with both operands split into two TF32 terms, a = a_hi + a_lo (a_hi = a rounded to the nearest
// TF32 value, a_lo = a - a_hi, exact in fp32, rounded likewise: the residual is below 2^-24 |a|), and three MMAs per K
// step: a_hi*w_hi + a_lo*w_hi + a_hi*w_lo (the dropped a_lo*w_lo term is 2^-22 relative).  Products of TF32 values are
// exact in fp32; what is left is the accumulation, which the tensor core does with truncation -- hence the second
// accumulator below.  Measured against fp64: rel-L2 5.5e-6 (the SIMT kernel 1.4e-6, the reference binary 8.6e-7).
//
// One CTA (no pairs) per 8 x 16-pixel tile, persistent, 18 warps.  12 producer warps in 3 groups of 128 threads; a group
// fills one A stage (the hi and lo [128 pixels x 32 channels] tiles of one k-block = 32 channels of one tap).  A lane
// computes the sampling position of ITS pixel for the tap -- from the anchors (AlignConv, alignconv.py:29-86), an explicit
// offset tensor (deform_conv_cuda_kernel.cu:218-227) or the regular grid (ORConv2d) -- but the gather is issued with
// eight lanes per (pixel, corner): a warp instruction reads four full 128-byte lines of the NHWC fp32 map, the pixel's
// weights and packed corner offset arrive by shuffle, the loads of two such iterations are in flight before either is
// blended (fp32), split and stored (swizzled 16-byte chunks).  A TMA warp streams the hi / lo planes of the packed
// weights (32 KB each per k-block, two stages); the MMA warp issues 12 tcgen05.mma (M = 128, N = C_out, K = 8) per
// k-block into two tensor-memory accumulators (a_hi*w_hi | the two correction products); 4 epilogue warps add the two,
// the bias, apply ReLU / the 8-way orientation max and store NCHW fp32 (a warp writes 2 x 64 contiguous bytes per channel).
// =================================================================================================
constexpr int TF_KB = 32;                                   // channels per k-block: 128 bytes of fp32
constexpr int TF_PROD_GROUPS = 3, TF_PROD_WARPS = 4 * TF_PROD_GROUPS;
constexpr int TF_NB = 2;                                    // gather iterations whose loads are in flight together
constexpr int TF_THREADS = (TF_PROD_WARPS + 4 + 2) * 32;    // + 4 epilogue warps + TMA warp + MMA warp
constexpr int TF_A_BYTES = TC_M * 128;                      // one [128 pixels x 32 channels] fp32 tile: 16 KB
constexpr int TF_B_BYTES = 256 * 128;                       // one [256 co x 32 channels] fp32 tile: 32 KB
// Stages: one A stage (hi + lo, 32 KB) PER PRODUCER GROUP -- k-block n is always produced by group n % 3 into A stage
// n % 3 (9 * C/32 is a multiple of 3), so a group only ever waits on the next phase of its own barrier (with two shared
// stages a group could run two phases ahead of the barrier it polls, which a parity wait cannot tell apart) -- and two B
// stages (hi + lo, 64 KB) filled in order by the TMA warp.
constexpr int TF_A_STAGE = 2 * TF_A_BYTES, TF_B_STAGE = 2 * TF_B_BYTES;
constexpr int TF_A_STAGES = TF_PROD_GROUPS, TF_B_STAGES = 2;
constexpr int TF_B_OFF = TF_A_STAGES * TF_A_STAGE;
constexpr size_t TF_SMEM = 1024 + TF_A_STAGES * TF_A_STAGE + TF_B_STAGES * TF_B_STAGE + 16 * 8 + 16;
enum { TF_ANCHORS = 0, TF_OFFSETS = 1, TF_GRID = 2 };

struct TfParams {
  const float* x;         // [B, H, W, C] fp32 (channels_last)
  const float* aux;       // anchors [B, H, W, 5] (TF_ANCHORS) or offsets [B, 18, H, W] (TF_OFFSETS)
  const float* bias;      // [Co] or null
  float* out;             // [B, Co, H, W] fp32 (NCHW, the reference's layout)
  float* pooled;          // [B, Co/8, H, W] or null
  int mode, relu;
  float stride;
  int B, C, Co, H, W, tiles_x, tiles_y, total_tiles;
};

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc)
      : "memory");
}
// nearest TF32 value (ties away from zero), low 13 mantissa bits zero: with hi = rna(v), lo = rna(v - hi) the residual
// v - hi - lo is below 2^-24 |v| and unbiased (a mask would truncate: twice the residual, and always towards zero)
__device__ __forceinline__ float tf32_hi(float v) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(v));
  return __uint_as_float(r);
}
__device__ __forceinline__ uint4 ldg_nc_f4(const float* p) { return ldg_nc_v4(p); }

__global__ void __launch_bounds__(TF_THREADS, 1)
conv_tf32x3_kernel(const __grid_constant__ CUtensorMap map_hi, const __grid_constant__ CUtensorMap map_lo, const TfParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint64_t* s_bar = reinterpret_cast<uint64_t*>(smem + TF_B_OFF + TF_B_STAGES * TF_B_STAGE);
  uint32_t* s_tmem = reinterpret_cast<uint32_t*>(s_bar + 16);
  const uint32_t bar_a_full = smem_u32(s_bar), bar_a_empty = bar_a_full + 24, bar_b_full = bar_a_full + 48,
                 bar_b_empty = bar_a_full + 64, bar_acc_full = bar_a_full + 80, bar_acc_empty = bar_a_full + 96;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr int kEpi0 = TF_PROD_WARPS, kTma = TF_PROD_WARPS + 4, kMma = TF_PROD_WARPS + 5;
  const int ncb = p.C / TF_KB, nkb = 9 * ncb;
  const int my_tiles = (int)blockIdx.x < p.total_tiles ? (p.total_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  const uint32_t b_bytes = (uint32_t)p.Co * 128u;

  if (tid == 0) {
    for (int s = 0; s < TF_A_STAGES; ++s) {
      mbar_init(bar_a_full + 8 * s, 4);                 // the four producer warps of the owning group
      mbar_init(bar_a_empty + 8 * s, 1);                // tcgen05.commit
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(bar_b_full + 8 * s, 1);                 // the TMA thread's expect_tx
      mbar_init(bar_b_empty + 8 * s, 1);                // tcgen05.commit
    }
    mbar_init(bar_acc_full, 1);                         // tcgen05.commit after the last k-block of a tile
    mbar_init(bar_acc_empty, 4);                        // one elected arrive per epilogue warp
    fence_barrier_init();
  }
  if (warp == kMma) tmem_alloc<1>(smem_u32(s_tmem), 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;

  auto tile_coords = [&](int it, int& b, int& ty0, int& tx0) {
    int tile = (int)blockIdx.x + it * (int)gridDim.x;
    const int tpi = p.tiles_x * p.tiles_y;
    b = tile / tpi;
    tile -= b * tpi;
    ty0 = (tile / p.tiles_x) * TC_PH;
    tx0 = (tile % p.tiles_x) * TC_PW;
  };

  if (warp < TF_PROD_WARPS) {
    // ===================== producers: fp32 samples, split into TF32 hi / lo rows =====================
    const int group = warp >> 2;
    const int wq = warp & 3;
    const int r = wq * 32 + lane;                       // the tile row (pixel) whose sampling parameters this lane computes
    // The gather itself is issued with eight lanes per (pixel, corner): a warp instruction reads four full 128-byte lines
    // (pixels 4 i .. 4 i + 3 of the warp's 32, i = 0..7) instead of 32 sectors in 32 lines -- ncu of the first version
    // (a lane = a pixel, looping over the eight chunks): L1TEX at 83 %, everything else below 31 %.  The parameters of
    // a pixel travel from the lane that computed them by shuffle.
    const int src0 = lane >> 3, jch = lane & 7;
    const uint32_t tile_hi = smem_u32(smem) + (uint32_t)(group * TF_A_STAGE + wq * (32 * 128));   // this warp's 32 rows
    for (int it = 0; it < my_tiles; ++it) {
      int b, ty0, tx0;
      tile_coords(it, b, ty0, tx0);
      const int y = ty0 + r / TC_PW, x = tx0 + r % TC_PW;
      const bool inside = y < p.H && x < p.W;
      float ax = 0.f, ay = 0.f, dw = 0.f, dh = 0.f, cs = 1.f, sn = 0.f;
      if (p.mode == TF_ANCHORS && inside) {
        const float* a = p.aux + ((size_t)(b * p.H + y) * p.W + x) * 5;
        ax = a[0] / p.stride; ay = a[1] / p.stride;
        dw = (a[2] / p.stride) / 3.0f; dh = (a[3] / p.stride) / 3.0f;
        cs = cosf(a[4]); sn = sinf(a[4]);
      }
      const size_t rowp = (size_t)p.W * p.C, img = (size_t)b * p.H * rowp;
      int last_tap = -1;
      float w1 = 0.f, w2 = 0.f, w3 = 0.f, w4 = 0.f;
      uint32_t base = 0;      // (element offset of the clamped top-left corner) / 4, bit 0: a right neighbour exists, bit 1: a lower one
      for (int kb = group; kb < nkb; kb += TF_PROD_GROUPS) {
        const int use = it * (nkb / TF_PROD_GROUPS) + kb / TF_PROD_GROUPS;     // how often this group's stage was filled
        const int tap = kb / ncb, cb = kb - tap * ncb;
        if (tap != last_tap) {
          // sampling position of (pixel, tap) and its bilinear corners / weights (deform_conv_cuda_kernel.cu:83-114, :228)
          last_tap = tap;
          w1 = w2 = w3 = w4 = 0.f;
          base = 0;
          if (inside) {
            const int ti = tap / 3, tj = tap - 3 * ti;
            float h, w;
            if (p.mode == TF_ANCHORS) {               // models/alignconv.py:29-86, operation order preserved
              const float fi = (float)(ti - 1), fj = (float)(tj - 1);
              const float txx = __fmul_rn(dw, fj), tyy = __fmul_rn(dh, fi);
              const float xr = __fsub_rn(__fmul_rn(cs, txx), __fmul_rn(sn, tyy));
              const float yr = __fadd_rn(__fmul_rn(sn, txx), __fmul_rn(cs, tyy));
              const float xa = __fadd_rn(xr, ax), ya = __fadd_rn(yr, ay);
              const float offx = __fsub_rn(xa, __fadd_rn((float)x, fj));
              const float offy = __fsub_rn(ya, __fadd_rn((float)y, fi));
              h = __fadd_rn((float)(y - 1 + ti), offy);
              w = __fadd_rn((float)(x - 1 + tj), offx);
            } else if (p.mode == TF_OFFSETS) {
              const size_t oi = (((size_t)b * 18 + 2 * tap) * p.H + y) * p.W + x;
              h = (float)(y - 1 + ti) + p.aux[oi];
              w = (float)(x - 1 + tj) + p.aux[oi + (size_t)p.H * p.W];
            } else {
              h = (float)(y - 1 + ti);
              w = (float)(x - 1 + tj);
            }
            if (h > -1.0f && w > -1.0f && h < (float)p.H && w < (float)p.W) {
              const float hf = floorf(h), wf = floorf(w);
              const int y0 = (int)hf, x0 = (int)wf;
              const float ly = h - hf, lx = w - wf, hy = 1.0f - ly, hx = 1.0f - lx;
              const bool t_ok = y0 >= 0, b_ok = y0 + 1 <= p.H - 1, l_ok = x0 >= 0, r_ok = x0 + 1 <= p.W - 1;
              w1 = (t_ok && l_ok) ? hy * hx : 0.f; w2 = (t_ok && r_ok) ? hy * lx : 0.f;
              w3 = (b_ok && l_ok) ? ly * hx : 0.f; w4 = (b_ok && r_ok) ? ly * lx : 0.f;
              // clamped corners (a corner outside the map has weight 0): top-left (yt, xl); the right / lower neighbours
              // are one pixel / one row further unless the clamp folds them onto the same pixel
              const int yt = max(y0, 0), xl = max(x0, 0);
              const bool has_r = min(x0 + 1, p.W - 1) > xl, has_b = min(y0 + 1, p.H - 1) > yt;
              base = (uint32_t)((img + yt * rowp + (size_t)xl * p.C) >> 2) | (has_r ? 1u : 0u) | (has_b ? 2u : 0u);
            }
          }
        }
        const float* xp = p.x + cb * TF_KB + 4 * jch;
        // Batches of TF_NB iterations (four pixels x eight 16-byte chunks per warp instruction each): all shuffles and
        // corner loads of a batch are issued before any of its stores -- the loads and stores are volatile asm
        // statements the compiler keeps in program order, so interleaving them (first version) meant one L2 round trip
        // per iteration.  There is no branch around the loads either: a pixel without a sample has base 0, a valid
        // address, and its row is zeroed by a select.  The first batch is in flight while the stage drains.
#pragma unroll 1
        for (int i0 = 0; i0 < 8; i0 += TF_NB) {
          uint4 q[TF_NB][4];
          float sw[TF_NB][4];
#pragma unroll
          for (int u = 0; u < TF_NB; ++u) {
            const int src = 4 * (i0 + u) + src0;
            sw[u][0] = __shfl_sync(0xffffffffu, w1, src); sw[u][1] = __shfl_sync(0xffffffffu, w2, src);
            sw[u][2] = __shfl_sync(0xffffffffu, w3, src); sw[u][3] = __shfl_sync(0xffffffffu, w4, src);
            const uint32_t sb = __shfl_sync(0xffffffffu, base, src);
            const float* q0 = xp + ((size_t)(sb & ~7u) << 2);
            const size_t dx = (sb & 1u) ? (size_t)p.C : 0, dy = (sb & 2u) ? rowp : 0;
            q[u][0] = ldg_nc_f4(q0); q[u][1] = ldg_nc_f4(q0 + dx);
            q[u][2] = ldg_nc_f4(q0 + dy); q[u][3] = ldg_nc_f4(q0 + dy + dx);
          }
          if (i0 == 0) mbar_wait(bar_a_empty + 8 * group, ((uint32_t)use & 1u) ^ 1u);
#pragma unroll
          for (int u = 0; u < TF_NB; ++u) {
            const int src = 4 * (i0 + u) + src0;
            const float s1 = sw[u][0], s2 = sw[u][1], s3 = sw[u][2], s4 = sw[u][3];
            const bool any = (s1 != 0.f) | (s2 != 0.f) | (s3 != 0.f) | (s4 != 0.f);
            const uint32_t u1[4] = {q[u][0].x, q[u][0].y, q[u][0].z, q[u][0].w}, u2[4] = {q[u][1].x, q[u][1].y, q[u][1].z, q[u][1].w};
            const uint32_t u3[4] = {q[u][2].x, q[u][2].y, q[u][2].z, q[u][2].w}, u4[4] = {q[u][3].x, q[u][3].y, q[u][3].z, q[u][3].w};
            float hi[4], lo[4];
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float t = s1 * __uint_as_float(u1[e]) + s2 * __uint_as_float(u2[e]) + s3 * __uint_as_float(u3[e]) +
                              s4 * __uint_as_float(u4[e]);
              const float v = any ? t : 0.f;
              hi[e] = tf32_hi(v);
              lo[e] = tf32_hi(v - hi[e]);
            }
            const uint32_t row_hi = tile_hi + (uint32_t)(src * 128 + ((jch ^ (src & 7)) << 4));           // SWIZZLE_128B
            sts_v4(row_hi, __float_as_uint(hi[0]), __float_as_uint(hi[1]), __float_as_uint(hi[2]), __float_as_uint(hi[3]));
            sts_v4(row_hi + TF_A_BYTES, __float_as_uint(lo[0]), __float_as_uint(lo[1]), __float_as_uint(lo[2]),
                   __float_as_uint(lo[3]));
          }
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_a_full + 8 * group);
      }
    }
  } else if (warp >= kTma) {
   if (warp == kTma) {
    // ===================== TMA: hi / lo halves of the packed weights, one k-block per stage =====================
    for (int it = 0; it < my_tiles; ++it) {
      for (int kb = 0; kb < nkb; ++kb) {
        const int n = it * nkb + kb, s = n & 1;
        mbar_wait(bar_b_empty + 8 * s, ((uint32_t)(n >> 1) & 1u) ^ 1u);
        if (elect_one()) {
          uint8_t* sb = smem + TF_B_OFF + s * TF_B_STAGE;
          mbar_arrive_expect_tx(bar_b_full + 8 * s, 2u * b_bytes);
          tma_load_2d<1>(smem_u32(sb), &map_hi, kb * TF_KB, 0, bar_b_full + 8 * s);
          tma_load_2d<1>(smem_u32(sb + TF_B_BYTES), &map_lo, kb * TF_KB, 0, bar_b_full + 8 * s);
        }
        __syncwarp();
      }
    }
   } else {
    // ===================== MMA issuer =====================
    // D = f32, A / B = TF32 (format 2), K-major, N = C_out, M = 128
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(p.Co >> 3) << 17) | ((uint32_t)(TC_M >> 4) << 24);
    // Two accumulators per tile: the hi*hi products in columns [0, 256), the two correction products (2^-11 of the
    // former) in [256, 512).  The tensor core TRUNCATES when it adds into the fp32 accumulator (measured: all 864 MMAs of
    // an output into one accumulator leave rel-L2 1.6e-5 against fp64, the SIMT kernel 1.4e-6); keeping the small terms
    // apart takes two thirds of the additions out of the large sum, and the epilogue adds the two in round-to-nearest.
    for (int it = 0; it < my_tiles; ++it) {
      mbar_wait(bar_acc_empty, ((uint32_t)it & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t d_main = tmem_base, d_corr = tmem_base + 256u;
      for (int kb = 0; kb < nkb; ++kb) {
        const int n = it * nkb + kb, s = n & 1, g = kb % TF_PROD_GROUPS;
        const int use = it * (nkb / TF_PROD_GROUPS) + kb / TF_PROD_GROUPS;
        mbar_wait(bar_a_full + 8 * g, (uint32_t)use & 1u);
        mbar_wait(bar_b_full + 8 * s, (uint32_t)(n >> 1) & 1u);
        tc_fence_after();
        if (elect_one()) {
          const uint32_t sa = smem_u32(smem + g * TF_A_STAGE), sb = smem_u32(smem + TF_B_OFF + s * TF_B_STAGE);
          const uint64_t a_hi = umma_desc_sw128(sa), a_lo = umma_desc_sw128(sa + TF_A_BYTES);
          const uint64_t b_hi = umma_desc_sw128(sb), b_lo = umma_desc_sw128(sb + TF_B_BYTES);
#pragma unroll
          for (int k = 0; k < 4; ++k) {                 // K = 8 fp32 = 32 bytes per step inside the 128-byte swizzle atom
            umma_tf32(d_main, a_hi + 2 * k, b_hi + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_tf32(d_corr, a_lo + 2 * k, b_hi + 2 * k, idesc, (kb | k) != 0 ? 1u : 0u);
            umma_tf32(d_corr, a_hi + 2 * k, b_lo + 2 * k, idesc, 1u);
          }
          umma_commit<1>(bar_a_empty + 8 * g);
          umma_commit<1>(bar_b_empty + 8 * s);
          if (kb == nkb - 1) umma_commit<1>(bar_acc_full);
        }
        __syncwarp();
      }
    }
   }
  } else {
    // ===================== epilogue: bias / ReLU / orientation max, NCHW fp32 stores =====================
    const int quad = warp & 3;                          // warps 12..15: warp % 4 = the TMEM lane quadrant
    const int r = quad * 32 + lane;
    for (int it = 0; it < my_tiles; ++it) {
      int b, ty0, tx0;
      tile_coords(it, b, ty0, tx0);
      const int y = ty0 + r / TC_PW, x = tx0 + r % TC_PW;
      const bool valid = y < p.H && x < p.W;
      mbar_wait(bar_acc_full, (uint32_t)it & 1u);
      tc_fence_after();
      const size_t plane = (size_t)p.H * p.W, pix = (size_t)y * p.W + x;
      for (int c0 = 0; c0 < p.Co; c0 += 32) {
        uint32_t v[32], vc[32];
        tmem_ld32_nowait(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)c0, v);
        tmem_ld32_nowait(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(256 + c0), vc);
        tmem_ld_wait();
        if (c0 + 32 >= p.Co) {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(bar_acc_empty);
        }
        if (valid) {
          float* o = p.out + ((size_t)b * p.Co + c0) * plane + pix;
          float m[4];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            float t = __uint_as_float(v[j]) + __uint_as_float(vc[j]);
            if (p.bias) t += __ldg(p.bias + c0 + j);
            if (p.relu) t = fmaxf(t, 0.0f);
            o[(size_t)j * plane] = t;
            m[j >> 3] = (j & 7) == 0 ? t : fmaxf(m[j >> 3], t);
          }
          if (p.pooled) {
            float* po = p.pooled + ((size_t)b * (p.Co / 8) + c0 / 8) * plane + pix;
#pragma unroll
            for (int g = 0; g < 4; ++g) po[(size_t)g * plane] = m[g];
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kMma) {
    tc_fence_after();
    tmem_dealloc<1>(tmem_base, 512);
  }
}

// weights [Co][C][3][3] fp32 (optionally through the ARF map: w [O, I, nOri, 3, 3], indices [nOri*9, nRot]) ->
// hi / lo TF32 planes [Co][(tap, c)] (K' = 9 C, k-block = 32 channels of one tap)
__global__ void pack_weight_tf32_kernel(const float* __restrict__ w, const uint8_t* __restrict__ arf_idx, float* __restrict__ hi,
                                        float* __restrict__ lo, int Co, int C, int nOri, int nRot, int arfI) {
  __shared__ uint8_t s_inv[8 * 72];
  const int nEntry = nOri * 9;
  if (arf_idx) {
    for (int i = threadIdx.x; i < nEntry * nRot; i += blockDim.x) {
      const int l = i / nRot, k = i % nRot;
      s_inv[k * nEntry + ((int)arf_idx[i] - 1)] = (uint8_t)l;
    }
    __syncthreads();
  }
  const int64_t total = (int64_t)Co * C * 9;
  for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
    const int cin = (int)(e % C);
    int64_t rr = e / C;
    const int tap = (int)(rr % 9);
    const int n = (int)(rr / 9);
    float v;
    if (arf_idx) {
      const int o = n / nRot, k = n % nRot;
      const int ii = cin / nOri, lay = cin % nOri;
      const int l = s_inv[k * nEntry + lay * 9 + tap];
      v = w[((int64_t)o * arfI + ii) * nEntry + l];
    } else {
      v = w[((int64_t)n * C + cin) * 9 + tap];
    }
    const float h = tf32_hi(v);
    hi[e] = h;
    lo[e] = tf32_hi(v - h);
  }
}

static int launch_tf32x3(const TfParams& p0, const float* w_hi, const float* w_lo, cudaStream_t st) {
  TfParams p = p0;
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) { set_error("conv_tf32x3: cuTensorMapEncodeTiled is not available from the driver"); return S2A_ERR_CUDA; }
  CUtensorMap maps[2];
  memset(maps, 0, sizeof(maps));
  const int Kp = 9 * p.C;
  const cuuint64_t gd[2] = {(cuuint64_t)Kp, (cuuint64_t)p.Co};
  const cuuint64_t gs[1] = {(cuuint64_t)Kp * 4};
  const cuuint32_t box[2] = {(cuuint32_t)TF_KB, (cuuint32_t)p.Co};
  const cuuint32_t es[2] = {1, 1};
  for (int i = 0; i < 2; ++i) {
    CUresult cr = enc(&maps[i], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(i == 0 ? w_hi : w_lo), gd, gs, box, es,
                      CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                      CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (cr != CUDA_SUCCESS) { set_error("conv_tf32x3: cuTensorMapEncodeTiled failed (%d)", (int)cr); return S2A_ERR_CUDA; }
  }
  p.tiles_x = (p.W + TC_PW - 1) / TC_PW; p.tiles_y = (p.H + TC_PH - 1) / TC_PH;
  const long long tiles = (long long)p.B * p.tiles_x * p.tiles_y;
  S2A_CHECK_ARG(tiles < (1ll << 31), "conv_tf32x3: too many tiles");
  p.total_tiles = (int)tiles;
  S2A_CUDA_OK(cudaFuncSetAttribute(conv_tf32x3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)TF_SMEM));
  const int grid = (int)std::max<long long>(1, std::min<long long>(tiles, sm_count()));
  conv_tf32x3_kernel<<<grid, TF_THREADS, TF_SMEM, st>>>(maps[0], maps[1], p);
  S2A_LAUNCH_OK("conv_tf32x3_kernel");
  return S2A_OK;
}

template <typename TIn>
static int pack_dispatch(const void* w, const uint8_t* idx, void* wp, int Co, int C, int nOri, int nRot, int arfI,
                         int out_dtype, cudaStream_t st) {
  const int64_t total = (int64_t)Co * C * 9;
  const int blocks = (int)std::min<int64_t>(ceil_div(total, 256), (int64_t)sm_count() * 8);
  if (out_dtype == S2A_BF16)
    pack_weight_kernel<TIn, __nv_bfloat16><<<blocks, 256, 0, st>>>((const TIn*)w, idx, (__nv_bfloat16*)wp, Co, C, nOri, nRot, arfI);
  else
    pack_weight_kernel<TIn, __half><<<blocks, 256, 0, st>>>((const TIn*)w, idx, (__half*)wp, Co, C, nOri, nRot, arfI);
  S2A_LAUNCH_OK("pack_weight_kernel");
  return S2A_OK;
}

}  // namespace s2a

extern "C" int s2a_conv_pack_weight(const void* weight, int in_dtype, const uint8_t* arf_indices, void* packed,
                                    int out_dtype, int Co, int C, int nOri, int nRot, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(Co > 0 && C > 0 && C % 64 == 0, "conv_pack_weight: C must be a positive multiple of 64");
  S2A_CHECK_ARG(out_dtype == S2A_BF16 || out_dtype == S2A_F16, "conv_pack_weight: packed dtype must be bf16 or f16");
  S2A_CHECK_ARG(weight && packed, "conv_pack_weight: null pointer");
  int arfI = 0;
  if (arf_indices) {
    S2A_CHECK_ARG(nOri >= 1 && nOri <= 8 && nRot >= 1 && nRot <= 8 && C % nOri == 0 && Co % nRot == 0,
                  "conv_pack_weight: bad ARF configuration");
    arfI = C / nOri;
  }
  cudaStream_t st = (cudaStream_t)stream;
  switch (in_dtype) {
    case S2A_F32: return pack_dispatch<float>(weight, arf_indices, packed, Co, C, nOri, nRot, arfI, out_dtype, st);
    case S2A_BF16: return pack_dispatch<__nv_bfloat16>(weight, arf_indices, packed, Co, C, nOri, nRot, arfI, out_dtype, st);
    case S2A_F16: return pack_dispatch<__half>(weight, arf_indices, packed, Co, C, nOri, nRot, arfI, out_dtype, st);
  }
  set_error("conv_pack_weight: unknown input dtype %d", in_dtype);
  return S2A_ERR_INVALID_ARGUMENT;
}

extern "C" int s2a_alignconv_forward_tc(const void* x, const float* anchors, const void* packed_weight, void* out, int B,
                                        int C, int H, int W, int Co, float stride, int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(H > 0 && W > 0, "alignconv_tc: bad feature map size");
  return conv_tc_common(TC_ALIGN, 1, &x, &anchors, packed_weight, nullptr, &out, nullptr, &H, &W, &stride, B, C, Co, 1,
                        dtype, (cudaStream_t)stream);
}

extern "C" int s2a_deform_conv_forward_tc(const void* x, const void* offsets, int offsets_dtype, const void* packed_weight,
                                          void* out, int B, int C, int H, int W, int Co, int relu, int round_positions,
                                          int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(H > 0 && W > 0, "deform_conv_tc: bad feature map size");
  S2A_CHECK_ARG(offsets != nullptr || B == 0, "deform_conv_tc: null offsets");
  S2A_CHECK_ARG(offsets_dtype == S2A_F32 || offsets_dtype == dtype, "deform_conv_tc: offsets must be fp32 or the activations' dtype");
  const float one = 1.0f;
  return conv_tc_common(TC_ALIGN, 1, &x, nullptr, packed_weight, nullptr, &out, nullptr, &H, &W, &one, B, C, Co, relu ? 1 : 0,
                        dtype, (cudaStream_t)stream, 3, -1, nullptr, nullptr, &offsets, offsets_dtype == S2A_F32 ? 1 : 0,
                        round_positions ? 1 : 0);
}

extern "C" int s2a_deform_conv_dgrad_tc(const void* grad_out, const void* offsets, int offsets_dtype, const void* wd,
                                        const void* x, float* grad_input, float* grad_offset, int B, int C, int H, int W,
                                        int Co, int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(H > 0 && W > 0 && B >= 0, "deform_conv_dgrad_tc: bad sizes");
  S2A_CHECK_ARG(C % 32 == 0 && C <= 256 && Co % 64 == 0,
                "deform_conv_dgrad_tc: needs C %% 32 == 0 <= 256 and C_out %% 64 == 0 (got C=%d, C_out=%d)", C, Co);
  S2A_CHECK_ARG(offsets_dtype == S2A_F32 || offsets_dtype == dtype, "deform_conv_dgrad_tc: offsets must be fp32 or the tensors' dtype");
  if (B == 0) return S2A_OK;
  S2A_CHECK_ARG(grad_out && offsets && wd && grad_input && (!grad_offset || x), "deform_conv_dgrad_tc: null pointer");
  // nine 1 x 1 convolutions grad_out [pixels, Co] x W_t^T [C, Co] on the plain-conv mainloop, each with the scatter
  // epilogue of its tap; wd = [9][C][Co] 16-bit is already the packed layout of a 1 x 1 weight (Co %% 64 == 0)
  void* fake_out = grad_input;             // (only to build an output tensor map the scatter epilogue never uses)
  for (int t = 0; t < 9; ++t) {
    TcScatter sc{grad_input, grad_offset, x, offsets, offsets_dtype == S2A_F32 ? 1 : 0, t};
    const void* wt = reinterpret_cast<const uint8_t*>(wd) + (size_t)t * C * Co * 2;
    const int rc = conv_tc_common(TC_PLAIN, 1, &grad_out, nullptr, wt, nullptr, &fake_out, nullptr, &H, &W, nullptr, B,
                                  /*C_in=*/Co, /*C_out=*/C, 0, dtype, (cudaStream_t)stream, 1, -1, nullptr, nullptr, nullptr, 0, 0,
                                  &sc);
    if (rc != S2A_OK) return rc;
  }
  return S2A_OK;
}

extern "C" int s2a_deform_conv_wgrad_tc(const void* x, const void* offsets, int offsets_dtype, const void* grad_out,
                                        float* grad_weight_t, int B, int C, int H, int W, int Co, int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(H > 0 && W > 0 && B >= 0, "deform_conv_wgrad_tc: bad sizes");
  S2A_CHECK_ARG(dtype == S2A_BF16 || dtype == S2A_F16, "deform_conv_wgrad_tc: dtype must be bf16 or f16");
  if ((C != 128 && C != 256) || (Co != 128 && Co != 256)) {
    set_error("deform_conv_wgrad_tc: needs C and C_out in {128, 256} (the accumulator is C_out x C fp32 in tensor memory; got C=%d, C_out=%d)", C, Co);
    return S2A_ERR_UNSUPPORTED;
  }
  S2A_CHECK_ARG(offsets_dtype == S2A_F32 || offsets_dtype == dtype, "deform_conv_wgrad_tc: offsets must be fp32 or the tensors' dtype");
  if (B == 0) return S2A_OK;
  S2A_CHECK_ARG(x && offsets && grad_out && grad_weight_t, "deform_conv_wgrad_tc: null pointer");
  return launch_wgrad(x, offsets, offsets_dtype == S2A_F32 ? 1 : 0, grad_out, grad_weight_t, B, C, H, W, Co, dtype,
                      (cudaStream_t)stream);
}

extern "C" int s2a_conv_pack_weight_tf32(const float* weight, const uint8_t* arf_indices, float* packed_hi, float* packed_lo,
                                         int Co, int C, int nOri, int nRot, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(Co > 0 && C > 0 && weight && packed_hi && packed_lo, "conv_pack_weight_tf32: bad arguments");
  int arfI = 0;
  if (arf_indices) {
    S2A_CHECK_ARG(nOri >= 1 && nOri <= 8 && nRot >= 1 && nRot <= 8 && C % nOri == 0 && Co % nRot == 0,
                  "conv_pack_weight_tf32: bad ARF configuration");
    arfI = C / nOri;
  }
  const int64_t total = (int64_t)Co * C * 9;
  const int blocks = (int)std::min<int64_t>(ceil_div(total, 256), (int64_t)sm_count() * 8);
  pack_weight_tf32_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(weight, arf_indices, packed_hi, packed_lo, Co, C, nOri, nRot, arfI);
  S2A_LAUNCH_OK("pack_weight_tf32_kernel");
  return S2A_OK;
}

extern "C" int s2a_conv_forward_tf32x3(const float* x, const float* aux, int mode, const float* packed_hi, const float* packed_lo,
                                       const float* bias, float* out, float* pooled, int B, int C, int H, int W, int Co,
                                       float stride, int relu, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(B >= 0 && H > 0 && W > 0, "conv_forward_tf32x3: bad tensor sizes");
  S2A_CHECK_ARG(mode == TF_ANCHORS || mode == TF_OFFSETS || mode == TF_GRID, "conv_forward_tf32x3: mode must be 0, 1 or 2");
  if (C % 32 != 0 || Co % 32 != 0 || Co > 256 || C <= 0) {
    set_error("conv_forward_tf32x3: needs C %% 32 == 0 and C_out a multiple of 32 up to 256 (got C=%d, C_out=%d)", C, Co);
    return S2A_ERR_UNSUPPORTED;
  }
  S2A_CHECK_ARG(mode != TF_ANCHORS || stride > 0.0f, "conv_forward_tf32x3: stride must be positive");
  S2A_CHECK_ARG(!pooled || Co % 8 == 0, "conv_forward_tf32x3: pooling needs C_out %% 8 == 0");
  if (B == 0) return S2A_OK;
  S2A_CHECK_ARG(x && packed_hi && packed_lo && out && (mode == TF_GRID || aux), "conv_forward_tf32x3: null pointer");
  TfParams p{};
  p.x = x; p.aux = aux; p.bias = bias; p.out = out; p.pooled = pooled; p.mode = mode; p.relu = relu; p.stride = stride;
  p.B = B; p.C = C; p.Co = Co; p.H = H; p.W = W;
  return launch_tf32x3(p, packed_hi, packed_lo, (cudaStream_t)stream);
}

extern "C" int s2a_orconv_forward_tc(const void* x, const void* packed_weight, const float* bias, void* out, void* pooled,
                                     int B, int C, int H, int W, int Co, int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(H > 0 && W > 0, "orconv_tc: bad feature map size");
  return conv_tc_common(TC_PLAIN, 1, &x, nullptr, packed_weight, bias, &out, &pooled, &H, &W, nullptr, B, C, Co, 0, dtype,
                        (cudaStream_t)stream);
}

extern "C" int s2a_alignconv_forward_tc_multi(int nlevels, const void* const* xs, const float* const* anchors,
                                              const void* packed_weight, void* const* outs, const int* Hs, const int* Ws,
                                              const float* strides, int B, int C, int Co, int dtype, void* stream) {
  using namespace s2a;
  return conv_tc_common(TC_ALIGN, nlevels, xs, anchors, packed_weight, nullptr, outs, nullptr, Hs, Ws, strides, B, C, Co,
                        1, dtype, (cudaStream_t)stream);
}

extern "C" int s2a_orconv_forward_tc_multi(int nlevels, const void* const* xs, const void* packed_weight,
                                           const float* bias, void* const* outs, void* const* pooleds, const int* Hs,
                                           const int* Ws, int B, int C, int Co, int dtype, void* stream) {
  using namespace s2a;
  return conv_tc_common(TC_PLAIN, nlevels, xs, nullptr, packed_weight, bias, outs, pooleds, Hs, Ws, nullptr, B, C, Co, 0,
                        dtype, (cudaStream_t)stream);
}

extern "C" int s2a_conv2d_pack_weight(const void* weight, int in_dtype, void* packed, int out_dtype, int Co, int C, int ks,
                                      void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(Co > 0 && C > 0 && (ks == 1 || ks == 3), "conv2d_pack_weight: bad sizes (kernel size 1 or 3)");
  S2A_CHECK_ARG(out_dtype == S2A_BF16 || out_dtype == S2A_F16, "conv2d_pack_weight: packed dtype must be bf16 or f16");
  S2A_CHECK_ARG(weight && packed, "conv2d_pack_weight: null pointer");
  const int ncb = (C + TC_KB - 1) / TC_KB, ntap = ks * ks, Co_pad = (Co + 31) / 32 * 32;
  const int64_t total = (int64_t)Co_pad * ncb * ntap * 64;
  const int blocks = (int)std::min<int64_t>(ceil_div(total, 256), (int64_t)sm_count() * 8);
  cudaStream_t st = (cudaStream_t)stream;
#define S2A_PACK2D(TIN)                                                                                                     \
  if (out_dtype == S2A_BF16)                                                                                                \
    pack_conv2d_kernel<TIN, __nv_bfloat16><<<blocks, 256, 0, st>>>((const TIN*)weight, (__nv_bfloat16*)packed, Co, Co_pad, C, ncb, ntap); \
  else                                                                                                                      \
    pack_conv2d_kernel<TIN, __half><<<blocks, 256, 0, st>>>((const TIN*)weight, (__half*)packed, Co, Co_pad, C, ncb, ntap);
  switch (in_dtype) {
    case S2A_F32: S2A_PACK2D(float) break;
    case S2A_BF16: S2A_PACK2D(__nv_bfloat16) break;
    case S2A_F16: S2A_PACK2D(__half) break;
    default: set_error("conv2d_pack_weight: unknown input dtype %d", in_dtype); return S2A_ERR_INVALID_ARGUMENT;
  }
#undef S2A_PACK2D
  S2A_LAUNCH_OK("pack_conv2d_kernel");
  return S2A_OK;
}

extern "C" int s2a_conv2d_forward_tc_multi(int nlevels, const void* const* xs, const void* packed_weight, const float* bias,
                                           void* const* outs, const int* Hs, const int* Ws, int B, int C, int Co_pad, int ks,
                                           int relu, int dtype, void* stream) {
  using namespace s2a;
  return conv_tc_common(TC_PLAIN, nlevels, xs, nullptr, packed_weight, bias, outs, nullptr, Hs, Ws, nullptr, B, C, Co_pad, relu,
                        dtype, (cudaStream_t)stream, ks);
}

// Two convolutions of one shape class (same C, C_out, kernel size, ReLU, dtype and batch; their own inputs, weights,
// biases and outputs) in ONE persistent launch: levels [0, split) belong to the first, [split, nlevels) to the second.
extern "C" int s2a_conv2d_forward_tc_multi2(int nlevels, int split, const void* const* xs, const void* packed_weight0,
                                            const void* packed_weight1, const float* bias0, const float* bias1,
                                            void* const* outs, const int* Hs, const int* Ws, int B, int C, int Co_pad,
                                            int ks, int relu, int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(split >= 1 && split < nlevels, "conv2d_forward_tc_multi2: split must separate two non-empty level lists");
  S2A_CHECK_ARG(packed_weight1 != nullptr, "conv2d_forward_tc_multi2: null pointer");
  return conv_tc_common(TC_PLAIN, nlevels, xs, nullptr, packed_weight0, bias0, outs, nullptr, Hs, Ws, nullptr, B, C, Co_pad,
                        relu, dtype, (cudaStream_t)stream, ks, split, packed_weight1, bias1);
}

// The FAM regression head (1 x 1, 5 output channels padded to 32, + bias; packed by s2a_conv2d_pack_weight) with the
// anchor decode of s2a_fam_decode in its epilogue: refined[l] [B, H_l, W_l, 5] fp32, bit-identical to s2a_fam_decode of
// the head's stored output; the deltas themselves are never written.
extern "C" int s2a_conv2d_forward_tc_fam_decode(int nlevels, const void* const* xs, const void* packed_weight,
                                                const float* bias, float* const* refined, const int* Hs, const int* Ws,
                                                const float* strides, int B, int C, int Co_pad, float anchor_scale,
                                                float anchor_angle, double wh_ratio_clip, int dtype, void* stream) {
  using namespace s2a;
  S2A_CHECK_ARG(Co_pad == TC_OUT_CH, "conv2d_forward_tc_fam_decode: the head must be padded to %d channels (got %d)",
                TC_OUT_CH, Co_pad);
  S2A_CHECK_ARG(bias && refined && strides, "conv2d_forward_tc_fam_decode: null pointer");
  S2A_CHECK_ARG(wh_ratio_clip > 0.0, "conv2d_forward_tc_fam_decode: wh_ratio_clip must be positive");
  const TcFamDecode fd{refined, anchor_scale, anchor_angle, clamp_limit(wh_ratio_clip, dtype)};
  return conv_tc_common(TC_PLAIN, nlevels, xs, nullptr, packed_weight, bias, nullptr, nullptr, Hs, Ws, strides, B, C, Co_pad, 0,
                        dtype, (cudaStream_t)stream, 1, -1, nullptr, nullptr, nullptr, 0, 0, nullptr, &fd);
}
