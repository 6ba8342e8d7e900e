// 3x3 "same" convolution of an NHWC half-precision board tensor on a CTA PAIR (tcgen05 cta_group::2).
//
//   out[b*64 + y*8 + x][n] = sum_{dy,dx,c} act[b][y+dy][x+dx][c] * W[n][((dy+1)*3 + dx+1)*Cin + c]
//
// Why a second kernel next to tc_gemm.cuh: the single-CTA kernel is bound by what feeds the tensor pipe (its
// 128 x 320 tile needs 56 KB of operands per 64-deep k-block) and by an epilogue that cannot overlap the next
// tile (320 of the 512 TMEM columns hold one accumulator).  Here
//   * two CTAs (one TPC) issue ONE 256 x N/2 x 16 MMA: each CTA stages only ITS 128 rows of A and a QUARTER of
//     the W rows (the pair reads each other's half of B), which halves the W bytes per flop;
//   * one A box {64 ch, 10 x, 8 y, 2 boards} per (k-chunk, dy) serves the three dx taps: the box starts at
//     x = -1 and is 10 wide, so TMA zero-fills both borders, and tap dx is the SAME shared-memory box read
//     through a descriptor that starts (dx + 1) rows later with a 10-row (1280 B) stride between 8-row groups
//     -- A traffic drops 3x against one box per tap;
//   * the N output channels are processed as two halves of N/2 columns in two TMEM accumulators (columns
//     0.. and 256..), so the epilogue of one half overlaps the main loop of the next.
//
// Work item = (group of 4 boards, channel half).  CTA r of the pair owns boards 4t + 2r, 4t + 2r + 1 (TMEM lanes
// 0..127 of its own tensor memory).  Warp 0 = TMA producer (both CTAs; every load signals the LEADER's full
// barrier), warp 1 = MMA issuer (leader CTA only) and TMEM allocator, warps 4..19 = epilogue: four warps per TMEM lane quarter, each
// holding its share of the accumulator (every fourth 16-column chunk) in registers -- the epilogue is latency bound, and four warps
// per scheduler hide what two could not (setmaxnreg moves registers from the control warpgroup to the four epilogue warpgroups).
//
// Epilogues (an epilogue warp owns 32 rows = half a board and every other 16-column chunk of the work item; one chunk = one
// GroupNorm group):
//   plain          out_f32 / out_half (+ SE squeeze sums by warp reduce-scatter); the tile leaves through a TMA bulk store
//   GroupNorm      act(GN(acc)) -> out_half (conv1 of a residual block); statistics exchanged between the four warps of a board
//   FUSE kernels   conv2 of a residual block: x_new = x + gate * acc with the x tiles arriving AND leaving by TMA (64-byte swizzled,
//                  double buffered per warp), then the next block's GroupNorm + activation -> out_half; conv1 additionally writes
//                  the half-board sums from which the SE gate of conv2 is computed ahead of conv2 (ConvPairParams::prims)
// A plain GEMM mode (conv = 0, K <= 320) keeps the A tile of a group of boards resident across its (slice, half) work items.
//
// F8 (3x3 mode only): the operands are e4m3 and a k-block is 128 channels -- still one 128-byte row, so the A box, CP_A_SLOT, the
// swizzle and the dx-shifted descriptors are the 16-bit ones byte for byte.  Each k-block issues 4 x kind::f8f6f4 MMAs of K = 32
// (32 bytes each, like the 4 x K = 16 of the 16-bit kernel).  The epilogue first multiplies the accumulator by ConvPairParams::w_dq
// (the inverse of the power-of-two weight scale, exact), and writes its GroupNorm'ed output as e4m3 (rounded in registers first, so
// that the SE half-board sums describe exactly what conv2 reads).
#pragma once
#include "tc_gemm.cuh"
#include <cuda_fp8.h>

namespace m0 {
namespace tc {

struct ConvPairParams {
  int boards;       // valid boards; rows b*64.. of the output are stored only for b < boards
  int N;            // output channels: N % 32 == 0, 64 <= N <= 512
  int kb_per_tap;   // Cin / 64
  int conv;         // 1: 3x3 convolution (A = x-padded NHWC boxes); 0: plain GEMM out = A[boards*64][64*kb_per_tap] W^T (A box {64, 128})
  int n_slices;     // >= 1: consecutive groups of N output channels handled by this launch (W rows / output columns advance by N)
  int stages;
  int fp16;         // operands are IEEE fp16 instead of bf16
  float* out_f32;   // [boards*64][ldc] or null
  __nv_bfloat16* out_half;   // same shape, 16-bit storage in the operand format, or null
  int ldc;
  int out_tma;      // 1: the output goes out through tma_out (box {16 columns, 32 rows} of the out_f32 / out_half tensor, row-major) -- the
                    // epilogue warps only fill a shared-memory tile; 0: direct stores from the smem transposer
  // fused epilogues (tc_gemm.cuh GemmParams): GroupNorm(16-channel groups over a board) + activation -> out_half,
  // or the SE squeeze partial sums pool_part[(board*2 + half board)][n]
  int act;
  const float* gn_gamma;
  const float* gn_beta;
  float* pool_part;
  // SE + residual fusion (conv2 of a residual block):
  //   resid_x != null: x_new = resid_x + gate[board][n] * acc (gate null -> 1), written back to resid_x (fp32, same ldc); then
  //                    gn_gamma != null -> out_half = half(act(GroupNorm(x_new))) (bn1 + activation of the NEXT block),
  //                    else out_half (if any) = half(x_new)
  //   prims != null  : (on the GroupNorm'ed output of conv1 = the input of conv2) prims[(board*2 + half)][6][N], half precision:
  //                    per half board and channel {sum of the 32 squares, sum of the board-edge rank, sum of file a, sum of file h,
  //                    corner on file a, corner on file h}.  The mean over the board of the NEXT 3x3 convolution's output is a
  //                    linear function of these (zero padding only removes edge ranks / files), which lets the SE gate of
  //                    conv2 be computed BEFORE conv2 runs (nn_tc_kernels.cu: se_fold_kernel).
  float* resid_x;
  const float* gate;
  __nv_bfloat16* prims;
  const float* w_dq;   // F8: per output channel factor applied to the accumulator before anything else (1 / weight scale)
};

static constexpr int CP_EPI_WARP0 = 4;    // warpgroup 0: TMA producer, MMA issuer, two idle warps
static constexpr int CP_EPI_WARPS = 16;   // warpgroups 1-4: epilogue, four warps per TMEM lane quarter (the epilogue is latency bound:
                                          // four warps per scheduler hide what two could not)
static constexpr int CP_CSETS = CP_EPI_WARPS / 4;   // the warps of a lane quarter take every CP_CSETS-th 16-column chunk
static constexpr int CP_THREADS = (CP_EPI_WARP0 + CP_EPI_WARPS) * 32;
// setmaxnreg: the kernel launches with 65536 / 640 -> 96 registers per thread; the control warpgroup gives back 128 * (96 - 40) = 7168,
// of which the four epilogue warpgroups take 512 * (104 - 96) = 4096.  An increase can only draw on what the CTA's own decrease released
// (asking for more blocks forever).
static constexpr int CP_REGS_CTRL = 40, CP_REGS_EPI = 104;
static constexpr int CP_A_SLOT = 160 * 128;   // 2 boards x 8 y x 10 x rows of 64 channels
static constexpr int CP_EPI_BYTES = CP_EPI_WARPS * 2048 + 2 * 512 * 4 + 2 * 4 * 16 * 2 * 4 + CP_EPI_WARPS * 64 * 4;   // tiles + gamma/beta + GN sums + SE gates
static constexpr int CP_EPI_BYTES_FUSE = CP_EPI_BYTES + CP_EPI_WARPS * 2048;   // FUSE = 2: 4 KB of tiles per epilogue warp instead of 2 KB

__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// loads issued by either CTA of the pair; the transaction bytes are credited to the barrier at cluster address bar
__device__ __forceinline__ void tma_load_4d_pair(void* dst, const CUtensorMap* map, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
                   smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
               : "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
                   smem_u32(dst)),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(bar), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* dst_smem, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() { asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}
// D (128 lanes in EACH CTA of the pair) (+)= A (128 rows from each CTA) * B^T (N/2 rows from each CTA); leader CTA only
__device__ __forceinline__ void umma_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same with e4m3 operands (the instruction descriptor's A / B format 0 = E4M3 under kind::f8f6f4, K = 32 per instruction)
__device__ __forceinline__ void umma_pair_f8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f8f6f4 [%0], %1, %2, %3, p;\n\t"
      "}\n" ::"r"(tmem_d),
      "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// four floats -> four e4m3 bytes (round to nearest even, saturating to +-448), the first in the lowest byte
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
  const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
  const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
  return lo | (hi << 16);
}
// x rounded to the nearest e4m3 value (saturating), as a float
__device__ __forceinline__ float round_e4m3(float x) {
  return __half2float(__half(__nv_cvt_fp8_to_halfraw(__nv_cvt_float_to_fp8(x, __NV_SATFINITE, __NV_E4M3), __NV_E4M3)));
}
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
}
// K-major 128-byte-swizzled operand whose 8-row groups are sbo_bytes apart (1024 for a dense tile)
// bulk tensor store of a row-major shared-memory tile (box of the map) to global memory; rows / columns past the tensor are clipped
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* smem_src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(reinterpret_cast<uint64_t>(map)),
               "r"(smem_u32(smem_src)), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
// The swizzle phase follows the absolute shared-memory address bits [7,10) (measured: a start that is a multiple of 128 B but not
// of 1024 B reads the rows TMA wrote there correctly with base_offset = 0), which is what lets one x-padded box serve three taps.
__device__ __forceinline__ uint64_t make_smem_desc_sbo(uint32_t smem_addr, uint32_t sbo_bytes) {
  return (uint64_t)((smem_addr >> 4) & 0x3FFFu) | (1ull << 16) | ((uint64_t)(sbo_bytes >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

// FUSE compiles the extra epilogues in (kept out of the plain kernels: code size costs instruction fetch):
//   0 = plain / GroupNorm, 1 = + half-board sums (conv1 of a fused block), 2 = SE gate + residual + next GroupNorm (conv2; 8 KB of
//   tiles per epilogue warp, which leaves room for 3 pipeline stages instead of 4)
template <int NCH, int FUSE, bool F8 = false>
__global__ void __launch_bounds__(CP_THREADS, 1)
conv_pair_kernel(const __grid_constant__ CUtensorMap tma_a, const __grid_constant__ CUtensorMap tma_w, const __grid_constant__ CUtensorMap tma_out,
                 const __grid_constant__ CUtensorMap tma_x, const ConvPairParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  const int nh = p.N >> 1, nq = p.N >> 2;
  const int wq_bytes = nq * 128;
  // 3x3 mode: ring stage = x-padded A box + the three W tiles of its dx taps.
  // plain mode (K <= 320): the whole A tile of a group of boards (kb_per_tap x 16 KB) is RESIDENT and double buffered across groups
  // -- every (slice, half) work item of the group reuses it -- and the ring carries only the W tiles.
  const int a_res_bytes = p.conv ? 0 : p.kb_per_tap * A_TILE_BYTES;
  const int stage_bytes = p.conv ? CP_A_SLOT + 3 * wq_bytes : wq_bytes;
  uint8_t* a_res = smem;                        // [2][kb_per_tap][16 KB]   (plain mode)
  smem += 2 * (size_t)a_res_bytes;              // ring base
  const int ns2 = 2 * (p.n_slices > 1 ? p.n_slices : 1);   // work items per group of 4 boards: (slice, channel half)
  float* epi_stage = reinterpret_cast<float*>(smem + (size_t)p.stages * stage_bytes);
  float* s_gamma = epi_stage + CP_EPI_WARPS * (FUSE == 2 ? 1024 : 512);   // [512]
  float* s_beta = s_gamma + 512;          // [512]
  float* s_stats = s_beta + 512;          // [2 accumulators][4 quarters][16 groups][sum, sumsq]
  float* s_gate = s_stats + 256;          // [epilogue warps][NCH * 16 <= 64]
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(s_gate + CP_EPI_WARPS * 64);
  uint64_t* empty_bar = full_bar + p.stages;
  uint64_t* tmem_full_bar = empty_bar + p.stages;   // [2]
  uint64_t* tmem_empty_bar = tmem_full_bar + 2;     // [2], only the leader's are used
  uint64_t* a_full_bar = tmem_empty_bar + 2;        // [2] resident A tile landed (leader's are used)
  uint64_t* a_empty_bar = a_full_bar + 2;           // [2] every MMA reading the resident A tile has completed
  uint64_t* x_bar = a_empty_bar + 2;                // [epilogue warps][2] residual tiles landed (FUSE = 2)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(x_bar + 2 * CP_EPI_WARPS);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank();
  const int num_tiles = (p.boards + 3) >> 2;
  const int num_clusters = gridDim.x >> 1;
  const int cluster_id = blockIdx.x >> 1;
  const int steps = p.conv ? p.kb_per_tap * 3 : p.kb_per_tap;
  constexpr int KE = F8 ? 128 : BK;   // operand elements per k-block (one 128-byte row either way)

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tma_a);
    tma_prefetch_desc(&tma_w);
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&tmem_full_bar[b], 1);
      mbar_init(&tmem_empty_bar[b], 2 * CP_EPI_WARPS);   // one arrival per epilogue warp of both CTAs
      mbar_init(&a_full_bar[b], 1);
      mbar_init(&a_empty_bar[b], 1);
    }
    for (int i = 0; i < 2 * CP_EPI_WARPS; ++i) mbar_init(&x_bar[i], 1);
    fence_barrier_init();
  }
  if (warp == 1) {
    tmem_alloc_pair(tmem_slot, 512);
    tmem_relinquish_pair();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < CP_EPI_WARP0) {
   asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(CP_REGS_CTRL));
   if (warp == 0) {
    // ===== TMA producer (both CTAs) =====
    if (lane == 0) {
      const uint32_t lead_full = mapa_u32(smem_u32(full_bar), 0);
      int stage = 0;
      uint32_t phase = 0;
      const uint32_t lead_afull = mapa_u32(smem_u32(a_full_bar), 0);
      // plain mode: the resident A tile of a group, all k-blocks, into buffer it & 1 (signals the leader's a_full barrier)
      auto load_a_tile = [&](int t, int it) {
        const int ab = it & 1;
        mbar_wait(&a_empty_bar[ab], (uint32_t)((it >> 1) & 1) ^ 1u);
        if (rank == 0) mbar_expect_tx(&a_full_bar[ab], (uint32_t)(2 * a_res_bytes));
        for (int kb = 0; kb < p.kb_per_tap; ++kb)
          tma_load_2d_pair(a_res + (size_t)ab * a_res_bytes + (size_t)kb * A_TILE_BYTES, &tma_a, lead_afull + (uint32_t)ab * 8u, kb * BK,
                           (t * 4 + rank * 2) * 64);
      };
      int it = 0;
      if (!p.conv && cluster_id < num_tiles) load_a_tile(cluster_id, 0);
      for (int t = cluster_id; t < num_tiles; t += num_clusters, ++it) {
        const int board0 = t * 4 + rank * 2;   // boards past the end are zero-filled by TMA
        if (!p.conv && t + num_clusters < num_tiles) load_a_tile(t + num_clusters, it + 1);   // one group ahead
        for (int u2 = 0; u2 < ns2; ++u2) {
          const int w_row = (u2 >> 1) * p.N + (u2 & 1) * nh + rank * nq;
          if (p.conv) {
            for (int kc = 0; kc < p.kb_per_tap; ++kc) {
              for (int dyi = 0; dyi < 3; ++dyi) {
                mbar_wait(&empty_bar[stage], phase ^ 1);
                if (rank == 0) mbar_expect_tx(&full_bar[stage], (uint32_t)(2 * stage_bytes));
                const uint32_t bar = lead_full + (uint32_t)stage * 8u;
                uint8_t* a_dst = smem + (size_t)stage * stage_bytes;
                tma_load_4d_pair(a_dst, &tma_a, bar, kc * KE, -1, dyi - 1, board0);
#pragma unroll
                for (int dxi = 0; dxi < 3; ++dxi)
                  tma_load_2d_pair(a_dst + CP_A_SLOT + dxi * wq_bytes, &tma_w, bar, ((dyi * 3 + dxi) * p.kb_per_tap + kc) * KE, w_row);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
              }
            }
          } else {
            for (int kb = 0; kb < p.kb_per_tap; ++kb) {
              mbar_wait(&empty_bar[stage], phase ^ 1);
              if (rank == 0) mbar_expect_tx(&full_bar[stage], (uint32_t)(2 * stage_bytes));
              tma_load_2d_pair(smem + (size_t)stage * stage_bytes, &tma_w, lead_full + (uint32_t)stage * 8u, kb * BK, w_row);
              if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issuer (leader CTA) =====
    if (rank == 0) {
      const uint32_t idesc = make_idesc_bf16(256, nh, F8 ? 1 : p.fp16);   // F8: format 0 = E4M3 (1 would be E5M2)
      const uint32_t smem_base = smem_u32(smem);
      int stage = 0;
      uint32_t phase = 0, unit = 0;
      int it = 0;
      for (int t = cluster_id; t < num_tiles; t += num_clusters, ++it) {
        const uint32_t a_tile = smem_u32(a_res) + (uint32_t)(it & 1) * (uint32_t)a_res_bytes;
        if (!p.conv) {
          mbar_wait(&a_full_bar[it & 1], (uint32_t)(it >> 1) & 1u);   // the group's resident A tile has landed in both CTAs
          tc_fence_after();
        }
        for (int u2 = 0; u2 < ns2; ++u2, ++unit) {
          const uint32_t buf = unit & 1u;
          mbar_wait(&tmem_empty_bar[buf], ((unit >> 1) & 1u) ^ 1u);   // both CTAs' epilogues have drained this accumulator
          tc_fence_after();
          const uint32_t d = tmem_base + buf * 256u;
          for (int step = 0; step < steps; ++step) {
            mbar_wait(&full_bar[stage], phase);
            tc_fence_after();
            const uint32_t a_addr = smem_base + (uint32_t)stage * (uint32_t)stage_bytes;
            if (elect_one()) {
              if (p.conv) {
#pragma unroll
                for (int dxi = 0; dxi < 3; ++dxi) {
                  const uint64_t adesc = make_smem_desc_sbo(a_addr + dxi * 128, 1280);
                  const uint64_t bdesc = make_smem_desc_sbo(a_addr + CP_A_SLOT + dxi * wq_bytes, 1024);
                  if constexpr (F8) {   // 4 x K = 32 e4m3: 32 bytes of K per instruction, as 4 x K = 16 at 16 bits
#pragma unroll
                    for (int k = 0; k < 4; ++k) umma_pair_f8(d, adesc + 2 * k, bdesc + 2 * k, idesc, (step > 0 || dxi > 0 || k > 0) ? 1u : 0u);
                  } else {
#pragma unroll
                    for (int k = 0; k < BK / 16; ++k) umma_pair(d, adesc + 2 * k, bdesc + 2 * k, idesc, (step > 0 || dxi > 0 || k > 0) ? 1u : 0u);
                  }
                }
              } else {
                const uint64_t adesc = make_smem_desc_sbo(a_tile + (uint32_t)step * A_TILE_BYTES, 1024);
                const uint64_t bdesc = make_smem_desc_sbo(a_addr, 1024);
#pragma unroll
                for (int k = 0; k < BK / 16; ++k) umma_pair(d, adesc + 2 * k, bdesc + 2 * k, idesc, (step > 0 || k > 0) ? 1u : 0u);
              }
              umma_commit_pair(&empty_bar[stage], 3);   // frees the stage in both CTAs
            }
            __syncwarp();
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
          if (elect_one()) {
            umma_commit_pair(&tmem_full_bar[buf], 3);
            if (!p.conv && u2 == ns2 - 1) umma_commit_pair(&a_empty_bar[it & 1], 3);   // the resident A buffer may be refilled
          }
          __syncwarp();
        }
      }
    }
   }
  } else {
    asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(CP_REGS_EPI));
    // ===== epilogue (both CTAs): TMEM -> registers (whole share of the warp, then the accumulator is released at once)
    //       -> GroupNorm / activation in registers -> smem transpose -> coalesced stores, 16 columns at a time =====
    const int quarter = warp & 3;
    const int cset = (warp - CP_EPI_WARP0) >> 2;        // the CP_CSETS warps of a lane quarter interleave their 16-column chunks
    // per-warp staging: 2 KB (transposer / two 1 KB output tiles / one fp32 tile), or 4 KB with FUSE = 2 (two 2 KB residual tiles, updated in
    // place and stored from where they landed)
    uint8_t* wtile = reinterpret_cast<uint8_t*>(epi_stage) + (size_t)(warp - CP_EPI_WARP0) * (FUSE == 2 ? 4096 : 2048);
    float* stg = reinterpret_cast<float*>(wtile);
    uint8_t* xin = wtile;                          // FUSE: residual tiles by TMA
    uint8_t* xout = wtile;                         // output tiles of the bulk stores
    uint64_t* xbar = x_bar + (warp - CP_EPI_WARP0) * 2;
    uint32_t xuse[2] = {0, 0};                     // completed uses of each residual tile buffer (mbarrier phase)
    float* wgate = s_gate + (warp - CP_EPI_WARP0) * (NCH * 16);   // this warp's SE gates of the current work item
    const bool fused_gn = p.gn_gamma != nullptr;
    const bool resid = FUSE == 2 && p.resid_x != nullptr;
    const bool want_prims = FUSE == 1 && p.prims != nullptr;
    const bool out8 = F8 && fused_gn;   // the GroupNorm'ed output is the e4m3 operand of the next convolution
    const int epi_tid = ((warp - CP_EPI_WARP0) << 5) | lane;
    const uint32_t lead_empty = mapa_u32(smem_u32(tmem_empty_bar), 0);
    const int nchunks = nh >> 4;
    const int M = p.boards * 64;
    const int act = p.act;
    if (fused_gn) {
      for (int c = epi_tid; c < p.N; c += CP_EPI_WARPS * 32) { s_gamma[c] = p.gn_gamma[c]; s_beta[c] = p.gn_beta[c]; }
      asm volatile("bar.sync 1, %0;" ::"n"(CP_EPI_WARPS * 32) : "memory");
    }
    uint32_t unit = 0, nstore = 0;   // nstore: bulk stores issued by this warp (selects the output tile buffer)
    for (int t = cluster_id; t < num_tiles; t += num_clusters) {
      for (int u2 = 0; u2 < ns2; ++u2, ++unit) {
        const int h = u2 & 1, cbase = (u2 >> 1) * p.N + h * nh;   // first output column of this work item
        const uint32_t buf = unit & 1u;
        const int row0 = t * 256 + rank * 128 + quarter * 32;
        const int m_lane = row0 + lane;
        // residual tiles of this warp's first two chunks (TMA -> shared memory) and the SE gates of its board: requested before
        // the accumulator is ready
        if (resid) {
          if (lane == 0) {
            tma_store_wait_read<0>();      // the tiles of the previous work item have been read by their bulk stores
#pragma unroll
            for (int k = 0; k < 2; ++k)
              if (k < NCH && cset + CP_CSETS * k < nchunks) {
                mbar_expect_tx(&xbar[k], 2048);
                tma_load_2d(xin + k * 2048, &tma_x, &xbar[k], cbase + (cset + CP_CSETS * k) * 16, row0);
              }
          }
          if (p.gate) {
            const int bq = row0 >> 6;
            const int k = lane >> 2, q = lane & 3, ci = cset + CP_CSETS * k;
            if (k < NCH && ci < nchunks && row0 < M)
              *reinterpret_cast<float4*>(wgate + k * 16 + 4 * q) = __ldg(reinterpret_cast<const float4*>(p.gate + (size_t)bq * p.N + h * nh + ci * 16 + 4 * q));
          }
        }
        mbar_wait(&tmem_full_bar[buf], (unit >> 1) & 1u);
        tc_fence_after();
        const uint32_t tmem_row = tmem_base + buf * 256u + ((uint32_t)(quarter * 32) << 16);
        float* stats = s_stats + buf * 128;
        uint32_t r[NCH][16];
#pragma unroll
        for (int k = 0; k < NCH; ++k)
          if (cset + CP_CSETS * k < nchunks) tmem_ld_32x16(tmem_row + (uint32_t)((cset + CP_CSETS * k) * 16), r[k]);
        tmem_ld_wait();
        // the accumulator is free again: the MMAs of the work item after next may overwrite it while this one is stored
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(lead_empty + buf * 8u);
        if constexpr (F8) {
          // undo the weight scale first: GroupNorm statistics, SE sums and the residual add all see the true convolution
#pragma unroll
          for (int k = 0; k < NCH; ++k) {
            const int ci = cset + CP_CSETS * k;
            if (ci >= nchunks) break;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 d4 = __ldg(reinterpret_cast<const float4*>(p.w_dq + cbase + ci * 16 + 4 * q));
              r[k][4 * q + 0] = __float_as_uint(__uint_as_float(r[k][4 * q + 0]) * d4.x);
              r[k][4 * q + 1] = __float_as_uint(__uint_as_float(r[k][4 * q + 1]) * d4.y);
              r[k][4 * q + 2] = __float_as_uint(__uint_as_float(r[k][4 * q + 2]) * d4.z);
              r[k][4 * q + 3] = __float_as_uint(__uint_as_float(r[k][4 * q + 3]) * d4.w);
            }
          }
        }
        if (resid) {
          // x_new = x + gate * conv  (SE excitation + residual add, resnet.py:68-80): the x tile arrives by TMA (64-byte swizzle: 16-byte
          // chunk c of row i sits at c ^ ((i >> 1) & 3)), x_new leaves the same way; nothing here touches global memory directly
          const int sw = (lane >> 1) & 3;
#pragma unroll
          for (int k = 0; k < NCH; ++k) {
            const int ci = cset + CP_CSETS * k;
            if (ci >= nchunks) break;
            const int col = cbase + ci * 16;
            const int xb = k & 1;
            mbar_wait(&xbar[xb], (xuse[xb]++) & 1u);
            uint8_t* xt = xin + xb * 2048 + lane * 64;   // this lane's row: read, updated and written back in place
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              float4* px = reinterpret_cast<float4*>(xt + ((q ^ sw) << 4));
              const float4 x4 = *px;
              float4 g4 = make_float4(1.f, 1.f, 1.f, 1.f);
              if (p.gate) g4 = *reinterpret_cast<const float4*>(wgate + k * 16 + 4 * q);
              const float4 y4 = make_float4(fmaf(__uint_as_float(r[k][4 * q + 0]), g4.x, x4.x), fmaf(__uint_as_float(r[k][4 * q + 1]), g4.y, x4.y),
                                            fmaf(__uint_as_float(r[k][4 * q + 2]), g4.z, x4.z), fmaf(__uint_as_float(r[k][4 * q + 3]), g4.w, x4.w));
              *px = y4;
              r[k][4 * q + 0] = __float_as_uint(y4.x); r[k][4 * q + 1] = __float_as_uint(y4.y);
              r[k][4 * q + 2] = __float_as_uint(y4.z); r[k][4 * q + 3] = __float_as_uint(y4.w);
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) {
              tma_store_2d(&tma_x, xin + xb * 2048, col, row0);
              tma_store_commit();
              if (k + 2 < NCH && ci + 2 * CP_CSETS < nchunks) {   // refill this buffer with the chunk after next once the store has read it
                tma_store_wait_read<0>();
                mbar_expect_tx(&xbar[xb], 2048);
                tma_load_2d(xin + xb * 2048, &tma_x, &xbar[xb], col + 2 * CP_CSETS * 16, row0);
              }
            }
          }
          if (!fused_gn && !p.out_half) continue;   // (half(x_new) for the attention qkv GEMM goes out through the tile loop below)
          if (lane == 0) tma_store_wait_read<0>();  // the residual tiles double as output tiles from here on
          __syncwarp();
        }
        if (fused_gn) {
          // per (half board = this warp, group of 16 channels = one chunk) sum and sum of squares
#pragma unroll
          for (int k = 0; k < NCH; ++k) {
            if (cset + CP_CSETS * k < nchunks) {
              float s0 = 0.f, q0 = 0.f;
#pragma unroll
              for (int j = 0; j < 16; ++j) {
                const float a = __uint_as_float(r[k][j]);
                s0 += a;
                q0 = fmaf(a, a, q0);
              }
#pragma unroll
              for (int off = 16; off > 0; off >>= 1) {
                s0 += __shfl_xor_sync(0xFFFFFFFFu, s0, off);
                q0 += __shfl_xor_sync(0xFFFFFFFFu, q0, off);
              }
              if (lane == 0) *reinterpret_cast<float2*>(stats + (quarter * 16 + cset + CP_CSETS * k) * 2) = make_float2(s0, q0);
            }
          }
          // the warps that hold one board (two lane quarters x CP_CSETS) exchange their partial sums
          if (quarter < 2) asm volatile("bar.sync 2, %0;" ::"n"(CP_EPI_WARPS * 16) : "memory");
          else asm volatile("bar.sync 3, %0;" ::"n"(CP_EPI_WARPS * 16) : "memory");
        }
#pragma unroll
        for (int k = 0; k < NCH; ++k) {
          const int ci = cset + CP_CSETS * k;
          if (ci >= nchunks) break;
          const int col = cbase + ci * 16;
          if (fused_gn) {
            const float2 sa = *reinterpret_cast<const float2*>(stats + ((quarter & 2) * 16 + ci) * 2);
            const float2 sb = *reinterpret_cast<const float2*>(stats + ((quarter | 1) * 16 + ci) * 2);
            const float mean = (sa.x + sb.x) * (1.0f / 1024.0f);
            const float var = fmaxf((sa.y + sb.y) * (1.0f / 1024.0f) - mean * mean, 0.0f);
            const float rstd = rsqrtf(var + 1e-5f);
            float y[16];
#pragma unroll
            for (int q = 0; q < 4; ++q) {
              const float4 g4 = *reinterpret_cast<const float4*>(s_gamma + col + 4 * q);
              const float4 b4 = *reinterpret_cast<const float4*>(s_beta + col + 4 * q);
              y[4 * q + 0] = fmaf(__uint_as_float(r[k][4 * q + 0]) - mean, g4.x * rstd, b4.x);
              y[4 * q + 1] = fmaf(__uint_as_float(r[k][4 * q + 1]) - mean, g4.y * rstd, b4.y);
              y[4 * q + 2] = fmaf(__uint_as_float(r[k][4 * q + 2]) - mean, g4.z * rstd, b4.z);
              y[4 * q + 3] = fmaf(__uint_as_float(r[k][4 * q + 3]) - mean, g4.w * rstd, b4.w);
            }
            if (act == ACT_SILU) {
#pragma unroll
              for (int j = 0; j < 16; ++j) y[j] = __fdividef(y[j], 1.0f + __expf(-y[j]));
            } else if (act == ACT_RELU) {
#pragma unroll
              for (int j = 0; j < 16; ++j) y[j] = fmaxf(y[j], 0.0f);
            }
            if constexpr (F8) {
#pragma unroll
              for (int j = 0; j < 16; ++j) y[j] = round_e4m3(y[j]);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) r[k][j] = __float_as_uint(y[j]);
          }
          if (p.out_tma && !want_prims) {
            // ---- output through TMA: this lane's row of the chunk goes into a row-major tile, one bulk store per chunk ----
            if (p.pool_part && row0 < M) {
              // column sums over the 32 rows (lanes) of this half board: reduce-scatter over lane bits 4..1, then bit 0
              float a8[8], a4[4], a2[2];
              const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4, b1 = lane & 2;
#pragma unroll
              for (int j = 0; j < 8; ++j) {
                const float send = __uint_as_float(b4 ? r[k][j] : r[k][8 + j]), keep = __uint_as_float(b4 ? r[k][8 + j] : r[k][j]);
                a8[j] = keep + __shfl_xor_sync(0xFFFFFFFFu, send, 16);
              }
#pragma unroll
              for (int j = 0; j < 4; ++j) a4[j] = (b3 ? a8[4 + j] : a8[j]) + __shfl_xor_sync(0xFFFFFFFFu, b3 ? a8[j] : a8[4 + j], 8);
#pragma unroll
              for (int j = 0; j < 2; ++j) a2[j] = (b2 ? a4[2 + j] : a4[j]) + __shfl_xor_sync(0xFFFFFFFFu, b2 ? a4[j] : a4[2 + j], 4);
              float a1 = (b1 ? a2[1] : a2[0]) + __shfl_xor_sync(0xFFFFFFFFu, b1 ? a2[0] : a2[1], 2);
              a1 += __shfl_xor_sync(0xFFFFFFFFu, a1, 1);
              if (!(lane & 1)) p.pool_part[(size_t)(row0 >> 5) * p.N + col + (b4 ? 8 : 0) + (b3 ? 4 : 0) + (b2 ? 2 : 0) + (b1 ? 1 : 0)] = a1;
            }
            if (p.out_half && out8) {
              uint8_t* tile = xout + (nstore & 1) * (FUSE == 2 ? 2048 : 1024);   // 32 rows x 16 e4m3 bytes
              if (lane == 0) tma_store_wait_read<1>();
              __syncwarp();
              const float* f = reinterpret_cast<const float*>(r[k]);
              *reinterpret_cast<uint4*>(tile + lane * 16) = make_uint4(pack_e4m3x4(f[0], f[1], f[2], f[3]), pack_e4m3x4(f[4], f[5], f[6], f[7]),
                                                                      pack_e4m3x4(f[8], f[9], f[10], f[11]), pack_e4m3x4(f[12], f[13], f[14], f[15]));
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) { tma_store_2d(&tma_out, tile, col, row0); tma_store_commit(); }
              ++nstore;
            } else if (p.out_half) {
              uint8_t* tile = xout + (nstore & 1) * (FUSE == 2 ? 2048 : 1024);   // two tiles alternate
              if (lane == 0) tma_store_wait_read<1>();                                 // the store that last read this tile is done
              __syncwarp();
              uint4 lo, hi;
              lo.x = pack_half2(__uint_as_float(r[k][0]), __uint_as_float(r[k][1]), p.fp16);
              lo.y = pack_half2(__uint_as_float(r[k][2]), __uint_as_float(r[k][3]), p.fp16);
              lo.z = pack_half2(__uint_as_float(r[k][4]), __uint_as_float(r[k][5]), p.fp16);
              lo.w = pack_half2(__uint_as_float(r[k][6]), __uint_as_float(r[k][7]), p.fp16);
              hi.x = pack_half2(__uint_as_float(r[k][8]), __uint_as_float(r[k][9]), p.fp16);
              hi.y = pack_half2(__uint_as_float(r[k][10]), __uint_as_float(r[k][11]), p.fp16);
              hi.z = pack_half2(__uint_as_float(r[k][12]), __uint_as_float(r[k][13]), p.fp16);
              hi.w = pack_half2(__uint_as_float(r[k][14]), __uint_as_float(r[k][15]), p.fp16);
              *reinterpret_cast<uint4*>(tile + lane * 32) = lo;
              *reinterpret_cast<uint4*>(tile + lane * 32 + 16) = hi;
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) { tma_store_2d(&tma_out, tile, col, row0); tma_store_commit(); }
              ++nstore;
            } else {
              uint8_t* tile = xout;                                                     // one 32 x 64 B tile
              if (lane == 0) tma_store_wait_read<0>();
              __syncwarp();
#pragma unroll
              for (int q = 0; q < 4; ++q)
                *reinterpret_cast<uint4*>(tile + lane * 64 + q * 16) = make_uint4(r[k][4 * q], r[k][4 * q + 1], r[k][4 * q + 2], r[k][4 * q + 3]);
              fence_proxy_async();
              __syncwarp();
              if (lane == 0) { tma_store_2d(&tma_out, tile, col, row0); tma_store_commit(); }
            }
            continue;
          }
          // lane = row; 16-byte chunk q of row i sits at chunk position q ^ ((i >> 1) & 3) (conflict-free both ways)
          const int sw = (lane >> 1) & 3;
#pragma unroll
          for (int q = 0; q < 4; ++q)
            *reinterpret_cast<uint4*>(stg + lane * 16 + ((q ^ sw) << 2)) = make_uint4(r[k][4 * q], r[k][4 * q + 1], r[k][4 * q + 2], r[k][4 * q + 3]);
          __syncwarp();
          if (p.pool_part && row0 < M) {
            // column sums of this half board: lane = (row parity, column)
            const int c = lane & 15, par = lane >> 4;
            float cs_sum = 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int rr = 2 * i + par;
              cs_sum += stg[rr * 16 + ((((c >> 2) ^ ((rr >> 1) & 3)) << 2) | (c & 3))];
            }
            cs_sum += __shfl_xor_sync(0xFFFFFFFFu, cs_sum, 16);
            if (par == 0) p.pool_part[(size_t)(row0 >> 5) * p.N + col + c] = cs_sum;
          }
          if (want_prims && row0 < M) {
            // sums of this half board that determine the SE squeeze of the NEXT convolution's output (see ConvPairParams::prims):
            // lane = (row parity, column); row rr = 2i + par is square (y = rr >> 3, x = rr & 7) of the half board
            const int c = lane & 15, par = lane >> 4, hb = quarter & 1;
            const int edge = hb ? 3 : 0;   // the board's first / last rank inside this half
            float tsum = 0.f, rsum = 0.f, c0 = 0.f, c7 = 0.f, k0 = 0.f, k7 = 0.f;
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              const int rr = 2 * i + par;
              const float v = stg[rr * 16 + ((((c >> 2) ^ ((rr >> 1) & 3)) << 2) | (c & 3))];
              tsum += v;
              const bool on_edge = (i >> 2) == edge;
              rsum += on_edge ? v : 0.f;
              if ((i & 3) == 0) { c0 += par == 0 ? v : 0.f; k0 += (on_edge && par == 0) ? v : 0.f; }
              if ((i & 3) == 3) { c7 += par == 1 ? v : 0.f; k7 += (on_edge && par == 1) ? v : 0.f; }
            }
            tsum += __shfl_xor_sync(0xFFFFFFFFu, tsum, 16); rsum += __shfl_xor_sync(0xFFFFFFFFu, rsum, 16);
            c0 += __shfl_xor_sync(0xFFFFFFFFu, c0, 16); c7 += __shfl_xor_sync(0xFFFFFFFFu, c7, 16);
            k0 += __shfl_xor_sync(0xFFFFFFFFu, k0, 16); k7 += __shfl_xor_sync(0xFFFFFFFFu, k7, 16);
            __nv_bfloat16* pp = p.prims + (size_t)(row0 >> 5) * 6 * p.N + col + c;
            const float v0 = par ? c7 : tsum, v1 = par ? k0 : rsum, v2 = par ? k7 : c0;
            const int j0 = par ? 3 : 0, j1 = par ? 4 : 1, j2 = par ? 5 : 2;
            const uint32_t h01 = pack_half2(v0, v1, p.fp16), h2 = pack_half2(v2, 0.f, p.fp16);
            reinterpret_cast<uint16_t*>(pp)[(size_t)j0 * p.N] = (uint16_t)(h01 & 0xFFFFu);
            reinterpret_cast<uint16_t*>(pp)[(size_t)j1 * p.N] = (uint16_t)(h01 >> 16);
            reinterpret_cast<uint16_t*>(pp)[(size_t)j2 * p.N] = (uint16_t)(h2 & 0xFFFFu);
          }
          if (p.out_f32) {
            const int q = lane & 3;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const int rr = (lane >> 2) + 8 * i;
              const int m = row0 + rr;
              if (m < M) {
                uint4 v = *reinterpret_cast<const uint4*>(stg + rr * 16 + ((q ^ ((rr >> 1) & 3)) << 2));
                *reinterpret_cast<uint4*>(p.out_f32 + (size_t)m * p.ldc + col + 4 * q) = v;
              }
            }
          }
          if (p.out_half && out8) {
            const int hq = lane & 1;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int rr = (lane >> 1) + 16 * i;
              const int m = row0 + rr;
              if (m < M) {
                const int sw2 = (rr >> 1) & 3;
                float4 lo = *reinterpret_cast<const float4*>(stg + rr * 16 + (((2 * hq) ^ sw2) << 2));
                float4 hi = *reinterpret_cast<const float4*>(stg + rr * 16 + (((2 * hq + 1) ^ sw2) << 2));
                *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(p.out_half) + (size_t)m * p.ldc + col + 8 * hq) =
                    make_uint2(pack_e4m3x4(lo.x, lo.y, lo.z, lo.w), pack_e4m3x4(hi.x, hi.y, hi.z, hi.w));
              }
            }
          } else if (p.out_half) {
            const int hq = lane & 1;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const int rr = (lane >> 1) + 16 * i;
              const int m = row0 + rr;
              if (m < M) {
                const int sw2 = (rr >> 1) & 3;
                float4 lo = *reinterpret_cast<const float4*>(stg + rr * 16 + (((2 * hq) ^ sw2) << 2));
                float4 hi = *reinterpret_cast<const float4*>(stg + rr * 16 + (((2 * hq + 1) ^ sw2) << 2));
                uint4 pk;
                pk.x = pack_half2(lo.x, lo.y, p.fp16); pk.y = pack_half2(lo.z, lo.w, p.fp16);
                pk.z = pack_half2(hi.x, hi.y, p.fp16); pk.w = pack_half2(hi.z, hi.w, p.fp16);
                *reinterpret_cast<uint4*>(p.out_half + (size_t)m * p.ldc + col + 8 * hq) = pk;
              }
            }
          }
          __syncwarp();
        }
      }
    }
    if (lane == 0) tma_store_wait_read<0>();   // the tile buffers must outlive the bulk stores that read them
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();   // no CTA leaves while its peer may still signal its barriers or read its shared memory
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc_pair(tmem_base, 512);
  }
}

}  // namespace tc
}  // namespace m0
