// Tensor-core path of PolicyValueNet.forward (precision fp16 = default, or bf16): the 3x3 convolutions of the trunk run on the CTA-pair
// tcgen05 kernel of tc_conv_pair.cuh, the 1x1 convolutions / linear layers on the single-CTA tcgen05 GEMM of tc_gemm.cuh (16-bit operands,
// fp32 accumulation in tensor memory); normalisation statistics, the SE gate, softmax and the last value layers stay in fp32.
// This file owns the per-network device state (16-bit weights, TMA tensor maps, activation buffers) and issues the launches.
// Environment switches (measurement / A-B comparison): M0_TC_PAIR=0 single-CTA kernel for the 3x3 convolutions, M0_TC_FUSE_SE=0 separate SE /
// residual kernels instead of the fused conv2 epilogue, M0_TC_PAIR_GEMM=1 pair kernel for the K = 320 GEMMs, M0_TC_CLUSTER / M0_TC_STAGES cluster
// size / pipeline-depth caps, M0_TC_PROFILE=1 per-launch-site event timing printed at exit.
#include "net_host.cuh"
#include "tc_gemm.cuh"
#include "tc_conv_pair.cuh"
#include <new>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <string>
#include <utility>
#include <vector>

using namespace m0;

namespace m0 {
int nn_se_apply_gn(const __nv_bfloat16* conv_out, const float* gate, float* x, const float* gamma, const float* beta, __nv_bfloat16* a_out, int B,
                   int C, int act, cudaStream_t s);
int nn_planes_to_nhwc_half(const float* planes, __nv_bfloat16* out, int B, int P, cudaStream_t s);
int nn_se_hidden(const float* part, int splits, long long split_stride, const float* b1, __nv_bfloat16* hidden, int B, int hid, int ld, int act,
                 cudaStream_t s);
int nn_gn_act_res(const float* x, const float* gamma, const float* beta, const float* residual, long long residual_bstride, float* out,
                  __nv_bfloat16* out_half, int B, int C, int act, cudaStream_t s);
int nn_attention_tc(const void* qkv_half, const float* rel_bias, void* out_half, int B, int C, int heads, float mix, cudaStream_t s);
int nn_se_tail(const float* part, int splits, long long split_stride, int ld, const float* b1, const float* w2t, const float* b2, float* gate, int B,
               int C, int hid, int act, cudaStream_t s);
int nn_value_tail(const float* gate, const float* h, const float* w3, const float* b3, float* values, int B, int C, cudaStream_t s);
int nn_se_gate(const float* pool, const float* w1t, const float* b1, const float* w2t, const float* b2, float* gate, int B, int C, int hid, int act,
               cudaStream_t s);
}  // namespace m0

namespace m0 {
// out[c][r] = in[r][c]  (SE weights are read coalesced by the gate kernel)
__global__ void transpose_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int cols) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  int r = i / cols, c = i % cols;
  out[c * rows + r] = in[i];
}
// SE squeeze folded through conv2 (tc_conv_pair.cuh, ConvPairParams::prims).  With P = the 12 x C half-board sums of conv2's INPUT
// (k = (half*6 + j)*C + ci), the board mean of conv2's output channel c is (1/64) sum_k Wcomb[c][k] P[k], where zero padding turns
// each tap (dy, dx) into "all squares minus an edge rank minus an edge file plus their corner":
//   j = 0 total: + all 9 taps | j = 1 edge rank (rank 1 in half 0, rank 8 in half 1): - the taps that look past it
//   j = 2 file a: - taps dx=+1 | j = 3 file h: - taps dx=-1 | j = 4, 5 corners on file a / h: + the one diagonal tap.
// The first SE layer is linear in the mean, so it is folded in as well: out[u][k] = (1/64) sum_c W1[u][c] Wcomb[c][k].
__global__ void se_fold_kernel(const float* __restrict__ conv_w, const float* __restrict__ w1, float* __restrict__ out, int C, int hid) {
  const int K = 12 * C;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= hid * K) return;
  const int u = i / K, k = i - u * K;
  const int ci = k % C, j = (k / C) % 6, hb = k / (6 * C);
  // signed tap set of this (half, j): bit t of plus / minus
  unsigned plus = 0, minus = 0;
  switch (j) {
    case 0: plus = 0x1FF; break;
    case 1: minus = hb ? 0x007 : 0x1C0; break;          // rank 8 is lost by dy = -1 (taps 0..2), rank 1 by dy = +1 (taps 6..8)
    case 2: minus = 0x124; break;                       // file a is lost by dx = +1 (taps 2, 5, 8)
    case 3: minus = 0x049; break;                       // file h is lost by dx = -1 (taps 0, 3, 6)
    case 4: plus = hb ? (1u << 2) : (1u << 8); break;   // a8 comes back for (dy -1, dx +1), a1 for (dy +1, dx +1)
    default: plus = hb ? (1u << 0) : (1u << 6); break;  // h8 for (dy -1, dx -1), h1 for (dy +1, dx -1)
  }
  float acc = 0.f;
  for (int c = 0; c < C; ++c) {
    const float* wr = conv_w + (size_t)c * 9 * C + ci;
    float wsum = 0.f;
#pragma unroll
    for (int t = 0; t < 9; ++t) {
      if (plus & (1u << t)) wsum += wr[t * C];
      if (minus & (1u << t)) wsum -= wr[t * C];
    }
    acc = fmaf(w1[u * C + c], wsum, acc);
  }
  out[i] = acc * (1.0f / 64.0f);
}
// in [rows][cols] -> out [rows][cols_pad] with zero padding columns (T = float, or uint16_t for 16-bit values: zero bits are +0)
template <typename T>
__global__ void pad_cols_kernel(const T* __restrict__ in, T* __restrict__ out, int rows, int cols, int cols_pad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols_pad) return;
  const int r = i / cols_pad, c = i - r * cols_pad;
  out[i] = c < cols ? in[r * cols + c] : T(0);
}
}  // namespace m0

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

// 2-D bf16 row-major matrix [rows][cols], box {64 cols, box_rows}, 128-byte swizzle, zero fill outside
int make_map_2d(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { m0_set_error("cuTensorMapEncodeTiled is not available from the driver"); return M0_ERR_CUDA; }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * 2};
  cuuint32_t box[2] = {64, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { m0_set_error("cuTensorMapEncodeTiled(2d %llu x %llu) failed: %d", (unsigned long long)rows, (unsigned long long)cols, (int)r); return M0_ERR_CUDA; }
  return M0_OK;
}

// 4-D view of NHWC activations [boards][8][8][C] bf16: dims {C, 8, 8, boards}, box {64, 8, 8, 2}
int make_map_nhwc(CUtensorMap* m, const void* ptr, uint64_t boards, uint64_t C, uint32_t box_x = 8) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { m0_set_error("cuTensorMapEncodeTiled is not available from the driver"); return M0_ERR_CUDA; }
  cuuint64_t dims[4] = {C, 8, 8, boards};
  cuuint64_t strides[3] = {C * 2, C * 2 * 8, C * 2 * 64};
  cuuint32_t box[4] = {64, box_x, 8, 2};   // box_x = 10: the CTA-pair kernel's x-padded box (tc_conv_pair.cuh)
  cuuint32_t estr[4] = {1, 1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 4, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { m0_set_error("cuTensorMapEncodeTiled(nhwc boards=%llu C=%llu) failed: %d", (unsigned long long)boards, (unsigned long long)C, (int)r); return M0_ERR_CUDA; }
  return M0_OK;
}

// row-major output tensor [rows][cols] (16-bit or fp32) written by the pair kernel's bulk stores: box {16 columns, 32 rows}, no swizzle
int make_map_out(CUtensorMap* m, const void* ptr, uint64_t rows, uint64_t cols, bool fp32, bool swizzle64 = false) {
  EncodeTiledFn enc = get_encode();
  if (!enc) { m0_set_error("cuTensorMapEncodeTiled is not available from the driver"); return M0_ERR_CUDA; }
  cuuint64_t dims[2] = {cols, rows};
  cuuint64_t strides[1] = {cols * (fp32 ? 4 : 2)};
  cuuint32_t box[2] = {16, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, fp32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { m0_set_error("cuTensorMapEncodeTiled(out %llu x %llu) failed: %d", (unsigned long long)rows, (unsigned long long)cols, (int)r); return M0_ERR_CUDA; }
  return M0_OK;
}

struct TcWeight {
  __nv_bfloat16* w = nullptr;  // [n][k] bf16
  CUtensorMap map;             // box {64, n_part / cluster}
  CUtensorMap map_pair;        // box {64, n / 4}: a quarter of the output channels per CTA and accumulator (tc_conv_pair.cuh)
  bool pair = false;
  int n = 0, k = 0, n_part = 0, cluster = 1;
  int n_launch = 0;            // output channels per launch / slice
};

// CTAs per cluster for a launch: the W tile is multicast within the cluster (M0_TC_CLUSTER overrides)
int pick_cluster(int n_part) {
  static int forced = -1;
  if (forced < 0) {
    const char* e = getenv("M0_TC_CLUSTER");
    forced = e ? atoi(e) : 0;
  }
  int cs = forced > 0 ? forced : 2;
  while (cs > 1 && ((n_part / cs) % 8 != 0 || n_part % cs != 0)) cs >>= 1;  // slices are whole 8-row swizzle atoms
  return cs;
}

struct TcBlock {
  TcWeight conv1, conv2, qkv, proj;
  TcWeight se_fold, se_w2;   // [hid][12C] first SE layer folded through conv2, [C][hid padded to 64] second SE layer
};

struct TcState {
  int sm_count = 148;
  int max_smem = 0;
  // dynamic shared memory already granted to the kernels ON THIS STATE'S DEVICE (cudaFuncSetAttribute is per device: a process-wide
  // record would leave the kernels of a second device at the 48 KB default)
  size_t smem_pair[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  size_t smem_gemm = 0;
  TcWeight pst, inter;
  std::vector<TcBlock> blocks;
  // SE: pooled half-board sums [cap][2][C], hidden [cap][hid], gate [cap][C]; W1 duplicated over the two halves and scaled by 1/64
  float *pool = nullptr, *se_hid = nullptr, *se_gate = nullptr;
  std::vector<float*> se_w1t, se_w2t;   // per block [C][hid], [hid][C]
  // fused SE path: half-board sums of conv2's input [cap][12C] and the hidden layer [cap][hid_pad] in half precision
  bool se_fused = false;
  int hid_pad = 0;
  __nv_bfloat16 *prims = nullptr, *se_hid_h = nullptr;
  float* se_part = nullptr;     // split-K partial sums of the first SE layer [k_splits][rows][hid_pad]
  int se_splits = 1;
  size_t se_rows = 0;
  CUtensorMap prims_mat, se_hid_mat;
  // stem on tensor cores: planes as NHWC half with 64 channels, weights [C][9*64]
  __nv_bfloat16* planes_h = nullptr;
  __nv_bfloat16* qkv_h = nullptr;   // [cap][64][3C] half (attention input)
  // heads on tensor cores
  bool heads_tc = false;
  TcWeight pol_conv, pol_fc1, pol_fc2, val_conv1, val_conv2, val_fc1, val_fc2, val_gate;
  bool val_tail_tc = false;      // value_fc2 and value_gate on tensor cores as well (M0_TC_VALUE_TAIL=0: fp32 SIMT GEMMs)
  int pol_rank_pad = 0;
  __nv_bfloat16 *ph_h = nullptr, *pf_h = nullptr, *vh_h = nullptr;   // [cap][4096], [cap][rank_pad], [cap][64][128]
  __nv_bfloat16 *vf1_h = nullptr, *vf2_h = nullptr;                  // [cap][2C], [cap][C]: operands of value_fc2 / value_gate
  CUtensorMap ph_mat, pf_mat, vh_conv_mat, vh_fc_mat, vf1_mat, vf2_mat;
  CUtensorMap planes_conv;
  TcWeight stem;
  // bf16 activation buffers [cap][64][C] and their maps
  int cap = 0;
  __nv_bfloat16 *a1 = nullptr, *a2 = nullptr;
  CUtensorMap a1_conv, a2_conv, a1_mat, a2_mat;
  CUtensorMap a1_convp, a2_convp, planes_convp;   // x-padded boxes of the CTA-pair kernel
  CUtensorMap x_io;                               // residual stream n->x (fp32, 64-byte swizzled tiles) for the fused conv2 epilogue
  const void* x_ptr = nullptr;
  CUtensorMap qkv_out, t2f_out;                   // qkv (half, 3C columns) and n->t2 as fp32 (attention projection)
  CUtensorMap a1_out, a2_out, t1_out, t2h_out;    // output maps of the pair kernel's bulk stores (a1, a2 half; n->t1 fp32; n->t2 as half)
  const void *t1_ptr = nullptr, *t2_ptr = nullptr;
  int out_rows = 0;
  std::vector<void*> allocs;
};

// CUDA-event timing of every launch of the tensor-core forward, by launch site: M0_TC_PROFILE=1 prints the table at exit,
// m0_profile_enable / m0_profile_get expose it to bench.py (per-kernel durations inside the running pipeline)
struct TcProfiler {
  struct Rec { const char* name; cudaEvent_t a, b; };
  std::vector<Rec> pending;
  std::vector<std::pair<std::string, std::pair<double, long>>> acc;
  int on = -1;
  bool enabled() {
    if (on < 0) {
      const char* e = getenv("M0_TC_PROFILE");
      on = (e && atoi(e)) ? 1 : 0;
      if (on) atexit(&TcProfiler::dump_static);
    }
    return on >= 1;
  }
  void set(int enable) { enabled(); on = enable ? 2 : 0; }   // programmatic switch (m0_profile_enable): no dump at exit
  void reset() { collect(); acc.clear(); }
  static TcProfiler& get() { static TcProfiler p; return p; }
  void begin(const char* name, cudaStream_t s) {
    Rec r; r.name = name;
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, s);
    pending.push_back(r);
  }
  void end(cudaStream_t s) { cudaEventRecord(pending.back().b, s); }
  void collect() {
    for (Rec& r : pending) {
      cudaEventSynchronize(r.b);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, r.a, r.b);
      bool found = false;
      for (auto& kv : acc) if (kv.first == r.name) { kv.second.first += ms; kv.second.second++; found = true; break; }
      if (!found) acc.push_back({r.name, {ms, 1}});
      cudaEventDestroy(r.a); cudaEventDestroy(r.b);
    }
    pending.clear();
  }
  static void dump_static() {
    TcProfiler& p = get();
    double tot = 0;
    for (auto& kv : p.acc) tot += kv.second.first;
    fprintf(stderr, "[m0 tc profile] total %.3f ms\n", tot);
    for (auto& kv : p.acc)
      fprintf(stderr, "[m0 tc profile] %5.1f%%  n=%5ld  avg=%9.1f us  %s\n", 100.0 * kv.second.first / tot, kv.second.second,
              1e3 * kv.second.first / kv.second.second, kv.first.c_str());
  }
};
#define PROF(name, call)                                   \
  do {                                                     \
    TcProfiler& _p = TcProfiler::get();                    \
    if (_p.enabled()) {                                    \
      _p.begin(name, s);                                   \
      int _r = (call);                                     \
      _p.end(s);                                           \
      if (_r != M0_OK) return _r;                          \
    } else {                                               \
      int _r = (call);                                     \
      if (_r != M0_OK) return _r;                          \
    }                                                      \
  } while (0)

#define TRY(x)            \
  do {                    \
    int _r = (x);         \
    if (_r != M0_OK) return _r; \
  } while (0)

int n_part_for(int n) { return n <= 256 ? n : n / 2; }

// 64-deep k-blocks per tap of cin input channels.  A tail block (cin % 64 == 32) reads channels past cin, which the activation maps
// zero-fill (their channel extent is cin); 3x3 weights are stored with each tap padded to whole k-blocks (make_weight), 1x1 weights
// [n][cin] are zero-filled by their map as well.
int kblocks_for(int cin) { return (cin + 63) / 64; }

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
// columns per launch slice of a wide K <= 320 GEMM: the widest divisor of n that leaves room for two accumulators in tensor memory
// (<= 256 columns, multiple of 16 so that a 2-CTA cluster splits the W tile into whole swizzle atoms); M0_TC_SLICE overrides
int slice_width_for(int n, int dflt) {
  static int forced = -1;
  if (forced < 0) forced = env_int("M0_TC_SLICE", 0);
  if (forced > 0) return (n % forced == 0) ? forced : dflt;
  if (!env_int("M0_TC_ACC2", 1)) return dflt;
  for (int w = 256; w >= 64; w -= 16)
    if (n % w == 0) return w;
  return dflt;
}
// 3x3 convolutions whose output width suits the CTA-pair kernel (M0_TC_PAIR=0 keeps the single-CTA kernel)
bool pair_ok(int n) {
  static int on = -1;
  if (on < 0) on = env_int("M0_TC_PAIR", 1);
  return on && n % 32 == 0 && n >= 64 && n <= 512;
}

struct ConvFusion {   // optional fused epilogue inputs / outputs of the CTA-pair convolution (tc_conv_pair.cuh)
  float* resid_x = nullptr;
  const float* gate = nullptr;
  __nv_bfloat16* prims = nullptr;
  const CUtensorMap* x_map = nullptr;   // resid_x as a [rows][C] fp32 tensor, box {16, 32}, 64-byte swizzle (tiles in and out by TMA)
};

int launch_conv_pair(TcState* st, const CUtensorMap& a_map, const TcWeight& w, int boards, int cin, float* out_f32, __nv_bfloat16* out_half,
                     int ldc, int act, cudaStream_t s, const float* gn_gamma = nullptr, const float* gn_beta = nullptr, float* pool_part = nullptr,
                     const ConvFusion* fuse = nullptr, int conv = 1, int n_slices = 1, const CUtensorMap* out_map = nullptr) {
  tc::ConvPairParams p;
  memset(&p, 0, sizeof(p));
  p.boards = boards;
  p.N = w.n_launch;
  p.kb_per_tap = kblocks_for(cin);
  p.conv = conv;
  p.n_slices = n_slices;
  if (n_slices > 1 && (gn_gamma || pool_part || fuse)) { m0_set_error("pair kernel: fused epilogues need a single slice"); return M0_ERR_ARG; }
  p.fp16 = nn_half_format();
  p.out_f32 = out_f32;
  p.out_half = out_half;
  p.ldc = ldc;
  p.act = act;
  p.gn_gamma = gn_gamma;
  p.gn_beta = gn_beta;
  p.pool_part = pool_part;
  if (fuse) { p.resid_x = fuse->resid_x; p.gate = fuse->gate; p.prims = fuse->prims; }
  static int cap = -1;
  if (cap < 0) cap = env_int("M0_TC_STAGES", 0);   // pipeline-depth experiments
  const int stage_bytes = conv ? tc::CP_A_SLOT + 3 * (w.n_launch / 4) * 128 : (w.n_launch / 4) * 128;
  const int a_res = conv ? 0 : 2 * kblocks_for(cin) * tc::A_TILE_BYTES;   // plain mode keeps two resident A tiles (K <= 320)
  const int fz = !fuse ? 0 : fuse->resid_x ? 2 : fuse->prims ? 1 : 0;   // tc_conv_pair.cuh FUSE variants
  const int epi_bytes = fz == 2 ? tc::CP_EPI_BYTES_FUSE : tc::CP_EPI_BYTES;
  int stages = (st->max_smem - 2048 - epi_bytes - a_res) / stage_bytes;
  if (stages > 8) stages = 8;
  if (cap > 0 && stages > cap) stages = cap;
  if (stages < 2) { m0_set_error("pair convolution: stage does not fit in shared memory (N=%d)", w.n_launch); return M0_ERR_ARG; }
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + a_res + epi_bytes + 1024 + 512;
  // epilogue register tile: 16-column chunks per warp = ceil((N / 2 / 16) / CP_CSETS)
  const int nch = (w.n_launch / 32 + tc::CP_CSETS - 1) / tc::CP_CSETS;
  if (nch > 4) { m0_set_error("pair kernel: N = %d is too wide", w.n_launch); return M0_ERR_ARG; }
  auto kernel = fz == 2 ? (nch <= 1 ? tc::conv_pair_kernel<1, 2> : nch <= 3 ? tc::conv_pair_kernel<3, 2> : tc::conv_pair_kernel<4, 2>)
                : fz == 1 ? (nch <= 1 ? tc::conv_pair_kernel<1, 1> : nch <= 3 ? tc::conv_pair_kernel<3, 1> : tc::conv_pair_kernel<4, 1>)
                          : (nch <= 1 ? tc::conv_pair_kernel<1, 0> : nch <= 3 ? tc::conv_pair_kernel<3, 0> : tc::conv_pair_kernel<4, 0>);
  const int kidx = (nch <= 1 ? 0 : nch <= 3 ? 1 : 2) + 3 * fz;
  if (smem > st->smem_pair[kidx]) {
    M0_CUDA_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    st->smem_pair[kidx] = smem;
  }
  const int tiles = (boards + 3) / 4;
  int clusters = st->sm_count / 2;
  if (clusters > tiles) clusters = tiles;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(clusters * 2));
  cfg.blockDim = dim3(tc::CP_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  if (fuse && fuse->resid_x && (!fuse->x_map || (out_half && !out_map))) { m0_set_error("pair kernel: the residual epilogue needs the x and output tensor maps"); return M0_ERR_ARG; }
  p.out_tma = (out_map && !(fuse && fuse->prims)) ? 1 : 0;   // the epilogue fills shared-memory tiles and TMA writes them out
  M0_CUDA_TRY(cudaLaunchKernelEx(&cfg, kernel, a_map, w.map_pair, out_map ? *out_map : a_map, (fuse && fuse->x_map) ? *fuse->x_map : a_map, p));
  return m0_check_launch("conv_pair_kernel");
}

// n_launch: output channels per kernel launch (N <= 320 -> <= 512 TMEM columns); wider layers are split by rows.
// taps = 9: w_f32 is [n][9][k / 9]; each tap is stored in whole 64-channel k-blocks, zero columns after its k / 9 channels, so that the
// tail k-block of a tap never reads the next tap's weights.
int make_weight(TcState* st, TcWeight* out, const float* w_f32, int n, int k, int n_launch, cudaStream_t s, int taps = 1) {
  const int cin = k / taps, cin_pad = taps > 1 ? kblocks_for(cin) * 64 : cin;
  k = taps * cin_pad;
  out->n = n;
  out->k = k;
  out->n_part = n_part_for(n_launch);
  out->cluster = pick_cluster(out->n_part);
  void* p = nullptr;
  M0_CUDA_TRY(cudaMalloc(&p, (size_t)n * k * 2));
  st->allocs.push_back(p);
  out->w = (__nv_bfloat16*)p;
  if (cin_pad != cin) {
    float* padded = nullptr;
    M0_CUDA_TRY(cudaMallocAsync((void**)&padded, (size_t)n * k * 4, s));
    pad_cols_kernel<float><<<(n * k + 255) / 256, 256, 0, s>>>(w_f32, padded, n * taps, cin, cin_pad);
    int rc = m0_check_launch("pad_taps");
    if (rc == M0_OK) rc = nn_f32_to_bf16(padded, out->w, (size_t)n * k, s);
    cudaFreeAsync(padded, s);
    TRY(rc);
  } else {
    TRY(nn_f32_to_bf16(w_f32, out->w, (size_t)n * k, s));
  }
  out->n_launch = n_launch;
  out->pair = pair_ok(n_launch) && n % n_launch == 0;
  if (out->pair) TRY(make_map_2d(&out->map_pair, out->w, (uint64_t)n, (uint64_t)k, (uint32_t)(n_launch / 4)));
  return make_map_2d(&out->map, out->w, (uint64_t)n, (uint64_t)k, (uint32_t)(out->n_part / out->cluster));
}

int pow2_cols(int n) {
  int c = 32;
  while (c < n) c <<= 1;
  return c;
}

// one launch of the tensor-core GEMM: rows [0, M), output columns [w_row0, w_row0 + N) of the layer
int launch_gemm(TcState* st, const CUtensorMap& a_map, const TcWeight& w, int M, int conv, int taps, int cin, int w_row0, int N, float* out_f32,
                __nv_bfloat16* out_bf16, int ldc, int col0, const float* bias, int act, float scale, cudaStream_t s,
                const float* gn_gamma = nullptr, const float* gn_beta = nullptr, float* pool_part = nullptr, int n_store = -1, int n_slices = 1,
                int k_splits = 1, long long split_stride = 0) {
  tc::GemmParams p;
  memset(&p, 0, sizeof(p));
  p.M = M;
  p.N = N;
  p.n_slices = n_slices;
  p.k_splits = k_splits;
  p.split_stride = split_stride;
  if (k_splits > 1 && (out_bf16 || bias || act != ACT_NONE || gn_gamma || pool_part || (taps * kblocks_for(cin)) % k_splits != 0 || !out_f32)) {
    m0_set_error("tensor-core GEMM: split-K needs a plain fp32 output and a K range divisible into whole k-blocks");
    return M0_ERR_ARG;
  }
  p.n_store = n_store >= 0 ? n_store : N * n_slices;
  if (w.n_part > N || N % w.n_part != 0) { m0_set_error("tensor-core GEMM: launch width %d does not match the weight map box %d", N, w.n_part); return M0_ERR_ARG; }
  p.n_part = w.n_part;
  p.taps = taps;
  p.kb_per_tap = kblocks_for(cin);
  p.conv = conv;
  p.w_row0 = w_row0;
  // two accumulators when they fit into the 512 columns of tensor memory (M0_TC_ACC2=0: single accumulator, for A-B comparison)
  {
    static int acc2 = -1;
    if (acc2 < 0) acc2 = env_int("M0_TC_ACC2", 1);
    const int stride = (N + 31) / 32 * 32;
    p.acc_stages = (acc2 && 2 * stride <= 512 && !gn_gamma) ? 2 : 1;
    p.acc_stride = stride;
    p.tmem_cols = pow2_cols(p.acc_stages * stride);
  }
  p.out_f32 = out_f32;
  p.out_bf16 = out_bf16;
  p.ldc = ldc;
  p.col0 = col0;
  p.bias = bias;
  p.act = act;
  p.scale = scale;
  p.gn_gamma = gn_gamma;
  p.gn_beta = gn_beta;
  p.pool_part = pool_part;
  if ((gn_gamma || pool_part) && (w_row0 != 0 || N % 32 != 0)) { m0_set_error("fused epilogue needs the full channel range"); return M0_ERR_ARG; }
  p.cluster = w.cluster;
  p.fp16 = nn_half_format();
  const int stage_bytes = tc::A_TILE_BYTES + N * tc::BK * 2;
  int stages = (st->max_smem - 2048 - tc::EPI_STAGE_BYTES) / stage_bytes;
  if (stages > 6) stages = 6;
  {
    static int cap = -1;
    if (cap < 0) { const char* e = getenv("M0_TC_STAGES"); cap = e ? atoi(e) : 0; }
    if (cap > 0 && stages > cap) stages = cap;
  }
  if (stages < 2) { m0_set_error("tensor-core GEMM: tile does not fit in shared memory (N=%d)", N); return M0_ERR_ARG; }
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + tc::EPI_STAGE_BYTES + 1024 + 256;
  if (smem > st->smem_gemm) {
    M0_CUDA_TRY(cudaFuncSetAttribute(tc::gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    st->smem_gemm = smem;
  }
  const int tiles = (M + tc::BM - 1) / tc::BM;
  const int cs = w.cluster;
  const int groups = (tiles + cs - 1) / cs;
  int clusters = st->sm_count / cs;
  if (clusters > groups * n_slices * k_splits) clusters = groups * n_slices * k_splits;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)(clusters * cs));
  cfg.blockDim = dim3(tc::NUM_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = (unsigned)cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  M0_CUDA_TRY(cudaLaunchKernelEx(&cfg, tc::gemm_tc_kernel, a_map, w.map, p));
  return m0_check_launch("gemm_tc_kernel");
}

// 3x3 convolution of B boards with all C_out channels in one launch: CTA-pair kernel when the weight supports it
int conv3x3(TcState* st, const CUtensorMap& a_map, const CUtensorMap& a_map_pair, const TcWeight& w, int B, int cin, float* out_f32,
            __nv_bfloat16* out_half, int act, cudaStream_t s, const float* gn_gamma = nullptr, const float* gn_beta = nullptr,
            float* pool_part = nullptr, const ConvFusion* fuse = nullptr, const CUtensorMap* out_map = nullptr) {
  if (w.pair) return launch_conv_pair(st, a_map_pair, w, B, cin, out_f32, out_half, w.n, act, s, gn_gamma, gn_beta, pool_part, fuse, 1, 1, out_map);
  if (fuse) { m0_set_error("fused SE / residual epilogue needs the CTA-pair convolution"); return M0_ERR_ARG; }
  return launch_gemm(st, a_map, w, B * 64, 1, 9, cin, 0, w.n, out_f32, out_half, w.n, 0, nullptr, act, 1.0f, s, gn_gamma, gn_beta, pool_part);
}

// out = A[B*64][cin] W^T for all n_slices * n_launch output channels in one launch (1x1 convolutions over the board tensor)
int gemm_rows64(TcState* st, const CUtensorMap& a_mat, const TcWeight& w, int B, int cin, float* out_f32, __nv_bfloat16* out_half, int ldc,
                cudaStream_t s, const CUtensorMap* out_map = nullptr) {
  const int n_slices = w.n / w.n_launch;
  // M0_TC_PAIR_GEMM=1: CTA-pair kernel with the A tile resident across the (slice, half) work items of a group of boards; measured
  // slower than the single-CTA kernel for K = 320 (both are bound by their epilogues there), so it is opt-in
  static int pg = -1;
  if (pg < 0) pg = env_int("M0_TC_PAIR_GEMM", 0);
  if (pg && w.pair && cin <= 320)
    return launch_conv_pair(st, a_mat, w, B, cin, out_f32, out_half, ldc, ACT_NONE, s, nullptr, nullptr, nullptr, nullptr, 0, n_slices, out_map);
  return launch_gemm(st, a_mat, w, B * 64, 0, 1, cin, 0, w.n_launch, out_f32, out_half, ldc, 0, nullptr, ACT_NONE, 1.0f, s, nullptr, nullptr, nullptr, -1,
                     n_slices);
}

int tc_reserve(m0_net* n, TcState* st, int B) {
  const int need = (B + 1) & ~1;  // tiles hold two boards
  if (need <= st->cap) return M0_OK;
  const size_t C = n->cfg.channels;
  if (st->a1) cudaFree(st->a1);
  if (st->a2) cudaFree(st->a2);
  if (st->pool) cudaFree(st->pool);
  if (st->se_hid) cudaFree(st->se_hid);
  if (st->se_gate) cudaFree(st->se_gate);
  if (st->planes_h) cudaFree(st->planes_h);
  if (st->qkv_h) cudaFree(st->qkv_h);
  if (st->ph_h) cudaFree(st->ph_h);
  if (st->pf_h) cudaFree(st->pf_h);
  if (st->vh_h) cudaFree(st->vh_h);
  if (st->vf1_h) cudaFree(st->vf1_h);
  if (st->vf2_h) cudaFree(st->vf2_h);
  st->vf1_h = st->vf2_h = nullptr;
  if (st->prims) cudaFree(st->prims);
  if (st->se_hid_h) cudaFree(st->se_hid_h);
  if (st->se_part) cudaFree(st->se_part);
  st->se_part = nullptr;
  st->prims = st->se_hid_h = nullptr;
  st->qkv_h = st->ph_h = st->pf_h = st->vh_h = nullptr;
  st->a1 = st->a2 = nullptr;
  st->pool = st->se_hid = st->se_gate = nullptr;
  st->planes_h = nullptr;
  st->cap = 0;
  M0_CUDA_TRY(cudaMalloc((void**)&st->pool, (size_t)need * 2 * C * 4));
  M0_CUDA_TRY(cudaMalloc((void**)&st->se_hid, (size_t)need * (n->cfg.se_hidden > 0 ? n->cfg.se_hidden : 1) * 4));
  M0_CUDA_TRY(cudaMalloc((void**)&st->se_gate, (size_t)need * C * 4));
  M0_CUDA_TRY(cudaMalloc((void**)&st->planes_h, (size_t)need * 64 * 64 * 2));
  M0_CUDA_TRY(cudaMalloc((void**)&st->qkv_h, (size_t)need * 64 * 3 * C * 2));
  if (st->heads_tc) {
    const size_t rp = (size_t)st->pol_rank_pad;
    M0_CUDA_TRY(cudaMalloc((void**)&st->ph_h, (size_t)need * 4096 * 2));
    M0_CUDA_TRY(cudaMalloc((void**)&st->pf_h, (size_t)need * rp * 2));
    M0_CUDA_TRY(cudaMalloc((void**)&st->vh_h, (size_t)need * 8192 * 2));
    M0_CUDA_TRY(cudaMemset(st->pf_h, 0, (size_t)need * rp * 2));   // padding columns stay zero
    TRY(make_map_2d(&st->ph_mat, st->ph_h, (uint64_t)need, 4096, 128));
    TRY(make_map_2d(&st->pf_mat, st->pf_h, (uint64_t)need, rp, 128));
    TRY(make_map_2d(&st->vh_conv_mat, st->vh_h, (uint64_t)need * 64, 128, 128));
    TRY(make_map_2d(&st->vh_fc_mat, st->vh_h, (uint64_t)need, 8192, 128));
    if (st->val_tail_tc) {
      M0_CUDA_TRY(cudaMalloc((void**)&st->vf1_h, (size_t)need * 2 * C * 2));
      M0_CUDA_TRY(cudaMalloc((void**)&st->vf2_h, (size_t)need * C * 2));
      TRY(make_map_2d(&st->vf1_mat, st->vf1_h, (uint64_t)need, 2 * C, 128));
      TRY(make_map_2d(&st->vf2_mat, st->vf2_h, (uint64_t)need, C, 128));
    }
  }
  if (st->se_fused && n->cfg.se) {
    // rows are padded to whole 128-row GEMM tiles; the padding columns of the hidden layer stay zero
    const size_t rows = ((size_t)need + 127) / 128 * 128;
    M0_CUDA_TRY(cudaMalloc((void**)&st->prims, rows * 12 * C * 2));
    M0_CUDA_TRY(cudaMalloc((void**)&st->se_hid_h, rows * st->hid_pad * 2));
    M0_CUDA_TRY(cudaMemset(st->prims, 0, rows * 12 * C * 2));
    M0_CUDA_TRY(cudaMemset(st->se_hid_h, 0, rows * st->hid_pad * 2));
    const int kblocks = 12 * (int)C / 64;
    st->se_splits = kblocks % 4 == 0 ? 4 : kblocks % 3 == 0 ? 3 : kblocks % 2 == 0 ? 2 : 1;
    st->se_rows = rows;
    M0_CUDA_TRY(cudaMalloc((void**)&st->se_part, (size_t)st->se_splits * rows * st->hid_pad * 4));
    TRY(make_map_2d(&st->prims_mat, st->prims, rows, 12 * C, 128));
    TRY(make_map_2d(&st->se_hid_mat, st->se_hid_h, rows, (uint64_t)st->hid_pad, 128));
  }
  M0_CUDA_TRY(cudaMemset(st->planes_h, 0, (size_t)need * 64 * 64 * 2));
  TRY(make_map_nhwc(&st->planes_conv, st->planes_h, need, 64));
  TRY(make_map_nhwc(&st->planes_convp, st->planes_h, need, 64, 10));
  M0_CUDA_TRY(cudaMalloc((void**)&st->a1, (size_t)need * 64 * C * 2));
  M0_CUDA_TRY(cudaMalloc((void**)&st->a2, (size_t)need * 64 * C * 2));
  M0_CUDA_TRY(cudaMemset(st->a1, 0, (size_t)need * 64 * C * 2));
  M0_CUDA_TRY(cudaMemset(st->a2, 0, (size_t)need * 64 * C * 2));
  TRY(make_map_nhwc(&st->a1_conv, st->a1, need, C));
  TRY(make_map_nhwc(&st->a2_conv, st->a2, need, C));
  TRY(make_map_nhwc(&st->a1_convp, st->a1, need, C, 10));
  TRY(make_map_nhwc(&st->a2_convp, st->a2, need, C, 10));
  st->t1_ptr = st->t2_ptr = nullptr;   // the output maps are rebuilt on the next forward
  TRY(make_map_2d(&st->a1_mat, st->a1, (uint64_t)need * 64, C, 128));
  TRY(make_map_2d(&st->a2_mat, st->a2, (uint64_t)need * 64, C, 128));
  st->cap = need;
  return M0_OK;
}

}  // namespace

namespace m0 {

struct TcStates {
  TcState* st[2] = {nullptr, nullptr};
};

int tc_net_prepare(::m0_net* n, cudaStream_t s) {
  if (!n->tc) n->tc = new (std::nothrow) TcStates();
  TcStates* all = (TcStates*)n->tc;
  if (!all) { m0_set_error("out of host memory"); return M0_ERR_ARG; }
  const int fmt = nn_half_format();
  if (all->st[fmt]) return M0_OK;
  const m0_net_config& c = n->cfg;
  if (c.channels % 32 != 0 || c.channels < 64 || c.channels > 320) {
    m0_set_error("16-bit tensor-core path needs channels %% 32 == 0 and 64 <= channels <= 320 (got %d)", c.channels);
    return M0_ERR_ARG;
  }
  TcState* st = new (std::nothrow) TcState();
  if (!st) { m0_set_error("out of host memory"); return M0_ERR_ARG; }
  cudaDeviceGetAttribute(&st->sm_count, cudaDevAttrMultiProcessorCount, n->device);
  cudaDeviceGetAttribute(&st->max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, n->device);
  const int C = c.channels;
  int rc = M0_OK;
  do {
    // stem on tensor cores: input channels zero-padded to 64
    if ((rc = make_weight(st, &st->stem, n->w.stem_w, C, 9 * c.planes, C, s, 9)) != M0_OK) break;
    if (c.se) {
      st->se_w1t.resize(c.blocks, nullptr);
      st->se_w2t.resize(c.blocks, nullptr);
      const int hc = c.se_hidden * C;
      for (int i = 0; i < c.blocks && rc == M0_OK; ++i) {
        float *w1t = nullptr, *w2t = nullptr;
        if ((rc = m0_check_cuda(cudaMalloc((void**)&w1t, (size_t)hc * 4), "cudaMalloc se")) != M0_OK) break;
        st->allocs.push_back(w1t);
        if ((rc = m0_check_cuda(cudaMalloc((void**)&w2t, (size_t)hc * 4), "cudaMalloc se")) != M0_OK) break;
        st->allocs.push_back(w2t);
        st->se_w1t[i] = w1t;
        st->se_w2t[i] = w2t;
        transpose_f32_kernel<<<(hc + 255) / 256, 256, 0, s>>>(n->w.blocks[i].se_w1, w1t, c.se_hidden, C);   // [hid][C] -> [C][hid]
        transpose_f32_kernel<<<(hc + 255) / 256, 256, 0, s>>>(n->w.blocks[i].se_w2, w2t, C, c.se_hidden);   // [C][hid] -> [hid][C]
        rc = m0_check_launch("transpose_se");
      }
      if (rc != M0_OK) break;
    }
    if (c.policy_factor_rank > 0 && c.policy_factor_rank % 16 == 0 && c.policy_factor_rank <= 320) {
      // heads: 1x1 convolutions and the wide fully connected layers as tensor-core GEMMs
      const int r = c.policy_factor_rank, rp = (r + 63) / 64 * 64;
      st->pol_rank_pad = rp;
      float* w2p = nullptr;   // policy_fc2 weights with the K dimension zero-padded to a multiple of 64
      const int ps_pad = (c.policy_size + 319) / 320 * 320;   // whole 320-column launches; the padding rows are zero
      if ((rc = m0_check_cuda(cudaMalloc((void**)&w2p, (size_t)ps_pad * rp * 4), "cudaMalloc pol_fc2")) != M0_OK) break;
      st->allocs.push_back(w2p);
      if ((rc = m0_check_cuda(cudaMemsetAsync(w2p, 0, (size_t)ps_pad * rp * 4, s), "memset")) != M0_OK) break;
      if ((rc = m0_check_cuda(cudaMemcpy2DAsync(w2p, (size_t)rp * 4, n->w.pol_fc2_w, (size_t)r * 4, (size_t)r * 4, c.policy_size,
                                                cudaMemcpyDeviceToDevice, s), "pad pol_fc2")) != M0_OK) break;
      if ((rc = make_weight(st, &st->pol_conv, n->w.pol_conv_w, 64, C, 64, s)) != M0_OK) break;
      if ((rc = make_weight(st, &st->pol_fc1, n->w.pol_fc1_w, r, 4096, r, s)) != M0_OK) break;
      if ((rc = make_weight(st, &st->pol_fc2, w2p, ps_pad, rp, 320, s)) != M0_OK) break;
      if ((rc = make_weight(st, &st->val_conv1, n->w.val_conv1_w, 128, C, 128, s)) != M0_OK) break;
      if ((rc = make_weight(st, &st->val_conv2, n->w.val_conv2_w, 128, 128, 128, s)) != M0_OK) break;
      // C > 256 runs as two MMAs of C / 2 columns side by side in tensor memory; 288 is cut into 144-column launches instead, which
      // keeps every accumulator at a 32-column boundary
      const int fc1_launch = n_part_for(C) % 32 == 0 ? C : slice_width_for(C, C);
      if ((rc = make_weight(st, &st->val_fc1, n->w.val_fc1_w, 2 * C, 8192, fc1_launch, s)) != M0_OK) break;
      if (env_int("M0_TC_VALUE_TAIL", 1)) {
        if ((rc = make_weight(st, &st->val_fc2, n->w.val_fc2_w, C, 2 * C, slice_width_for(C, C), s)) != M0_OK) break;
        if ((rc = make_weight(st, &st->val_gate, n->w.val_gate_w, C, C, slice_width_for(C, C), s)) != M0_OK) break;
        st->val_tail_tc = true;
      }
      st->heads_tc = true;
    }
    if (c.chess_features) {
      if (c.piece_square_tables && (rc = make_weight(st, &st->pst, n->w.pst_w, C, C, env_int("M0_TC_SLICE_PROJ", 1) ? slice_width_for(C, C) : C, s)) != M0_OK) break;
      if ((rc = make_weight(st, &st->inter, n->w.inter_w, C, 9 * C, C, s, 9)) != M0_OK) break;
    }
    // fused SE + residual epilogue of conv2 (M0_TC_FUSE_SE=0 keeps the separate SE / residual kernels)
    st->hid_pad = (c.se_hidden + 63) / 64 * 64;
    st->se_fused = env_int("M0_TC_FUSE_SE", 1) != 0 && pair_ok(C) && (!c.se || c.se_hidden <= 256);
    st->blocks.resize(c.blocks);
    for (int i = 0; i < c.blocks && rc == M0_OK; ++i) {
      const m0_block_weights& b = n->w.blocks[i];
      if ((rc = make_weight(st, &st->blocks[i].conv1, b.conv1_w, C, 9 * C, C, s, 9)) != M0_OK) break;
      if ((rc = make_weight(st, &st->blocks[i].conv2, b.conv2_w, C, 9 * C, C, s, 9)) != M0_OK) break;
      if (st->se_fused && c.se) {
        // the first SE GEMM runs hid16 = hid rounded up to 16 output columns (the MMA width granule); the extra rows of the folded
        // weight are zero and their columns are not stored
        const int hid = c.se_hidden, hid16 = (hid + 15) / 16 * 16, K = 12 * C, hp = st->hid_pad;
        float *fold = nullptr, *w2p = nullptr;
        if ((rc = m0_check_cuda(cudaMalloc((void**)&fold, (size_t)hid16 * K * 4), "cudaMalloc se_fold")) != M0_OK) break;
        st->allocs.push_back(fold);
        if ((rc = m0_check_cuda(cudaMemsetAsync(fold, 0, (size_t)hid16 * K * 4, s), "memset se_fold")) != M0_OK) break;
        if ((rc = m0_check_cuda(cudaMalloc((void**)&w2p, (size_t)C * hp * 4), "cudaMalloc se_w2")) != M0_OK) break;
        st->allocs.push_back(w2p);
        se_fold_kernel<<<(hid * K + 255) / 256, 256, 0, s>>>(b.conv2_w, b.se_w1, fold, C, hid);
        pad_cols_kernel<float><<<(C * hp + 255) / 256, 256, 0, s>>>(b.se_w2, w2p, C, hid, hp);
        if ((rc = m0_check_launch("se_fold")) != M0_OK) break;
        if ((rc = make_weight(st, &st->blocks[i].se_fold, fold, hid16, K, hid16, s)) != M0_OK) break;
        if ((rc = make_weight(st, &st->blocks[i].se_w2, w2p, C, hp, C, s)) != M0_OK) break;
      }
      if (b.has_attention) {
        if ((rc = make_weight(st, &st->blocks[i].qkv, b.att_qkv_w, 3 * C, C, slice_width_for(3 * C, C), s)) != M0_OK) break;
        if ((rc = make_weight(st, &st->blocks[i].proj, b.att_proj_w, C, C, env_int("M0_TC_SLICE_PROJ", 1) ? slice_width_for(C, C) : C, s)) != M0_OK) break;
      }
    }
  } while (0);
  if (rc != M0_OK) {
    for (void* p : st->allocs) cudaFree(p);
    delete st;
    return rc;
  }
  all->st[fmt] = st;
  return M0_OK;
}

void tc_net_release(::m0_net* n) {
  TcStates* all = (TcStates*)n->tc;
  if (!all) return;
  for (int f = 0; f < 2; ++f) {
    TcState* st = all->st[f];
    if (!st) continue;
    for (void* p : st->allocs) cudaFree(p);
    if (st->a1) cudaFree(st->a1);
    if (st->a2) cudaFree(st->a2);
    if (st->pool) cudaFree(st->pool);
    if (st->se_hid) cudaFree(st->se_hid);
    if (st->se_gate) cudaFree(st->se_gate);
    if (st->planes_h) cudaFree(st->planes_h);
    if (st->qkv_h) cudaFree(st->qkv_h);
    if (st->ph_h) cudaFree(st->ph_h);
    if (st->pf_h) cudaFree(st->pf_h);
    if (st->vh_h) cudaFree(st->vh_h);
    if (st->vf1_h) cudaFree(st->vf1_h);
    if (st->vf2_h) cudaFree(st->vf2_h);
    if (st->prims) cudaFree(st->prims);
    if (st->se_hid_h) cudaFree(st->se_hid_h);
    if (st->se_part) cudaFree(st->se_part);
    delete st;
  }
  delete all;
  n->tc = nullptr;
}

int tc_net_forward(::m0_net* n, const float* planes, int B, float* logits, float* values, cudaStream_t s) {
  TcState* st = ((TcStates*)n->tc)->st[nn_half_format()];
  TRY(net_ws_reserve(n, B));
  TRY(tc_reserve(n, st, B));
  const m0_net_config& c = n->cfg;
  const m0_net_weights& w = n->w;
  const int C = c.channels, M = B * 64, act = c.activation;
  const float* none = nullptr;
  if (st->t1_ptr != n->t1 || st->t2_ptr != n->t2 || st->x_ptr != n->x || st->out_rows != M) {
    // output maps of the bulk stores: their row extent is exactly this batch (rows of padding boards are clipped by TMA)
    TRY(make_map_out(&st->a1_out, st->a1, (uint64_t)M, C, false));
    TRY(make_map_out(&st->a2_out, st->a2, (uint64_t)M, C, false));
    TRY(make_map_out(&st->t1_out, n->t1, (uint64_t)M, C, true));
    TRY(make_map_out(&st->t2h_out, n->t2, (uint64_t)M, C, false));
    TRY(make_map_out(&st->t2f_out, n->t2, (uint64_t)M, C, true));
    TRY(make_map_out(&st->qkv_out, st->qkv_h, (uint64_t)M, 3 * (uint64_t)C, false));
    TRY(make_map_out(&st->x_io, n->x, (uint64_t)M, C, true, true));
    st->x_ptr = n->x;
    st->t1_ptr = n->t1;
    st->t2_ptr = n->t2;
    st->out_rows = M;
  }
  // stem: planes -> NHWC half (64 channels, zero padded) -> tensor-core conv3x3 -> GN + act (+ position encoding)
  PROF("planes_to_nhwc_half", nn_planes_to_nhwc_half(planes, st->planes_h, B, c.planes, s));
  PROF("conv_other", conv3x3(st, st->planes_conv, st->planes_convp, st->stem, B, 64, n->t1, nullptr, ACT_NONE, s, nullptr, nullptr, nullptr, nullptr, &st->t1_out));
  if (c.chess_features) {
    PROF("gn_act_res", nn_gn_act_res(n->t1, w.stem_gn_w, w.stem_gn_b, w.pos_enc, 0, n->x, st->a1, B, C, act, s));
    float* cur = n->x;
    if (c.piece_square_tables) {
      PROF("gemm_pst", gemm_rows64(st, st->a1_mat, st->pst, B, C, n->t1, nullptr, C, s, &st->t1_out));
      PROF("gn_act_res", nn_gn_act_res(n->t1, w.pst_gn_w, w.pst_gn_b, n->x, (long long)64 * C, n->t2, st->a1, B, C, act, s));
      cur = n->t2;
    }
    PROF("conv_other", conv3x3(st, st->a1_conv, st->a1_convp, st->inter, B, C, n->t1, nullptr, ACT_NONE, s, nullptr, nullptr, nullptr, nullptr, &st->t1_out));
    PROF("gn_act_res", nn_gn_act_res(n->t1, w.inter_gn_w, w.inter_gn_b, cur, (long long)64 * C, n->x, nullptr, B, C, act, s));
  } else {
    PROF("groupnorm_f32", nn_groupnorm_f32(n->t1, w.stem_gn_w, w.stem_gn_b, nullptr, 0, n->x, B, C, act, s));
  }
  // a1 = act(GN1(x)) of the first block; later blocks get it from the fused SE / residual kernel of their predecessor
  if (c.blocks > 0) PROF("se_apply_gn", nn_se_apply_gn(nullptr, nullptr, n->x, w.blocks[0].gn1_w, w.blocks[0].gn1_b, st->a1, B, C, act, s));
  int att_seen = 0;
  bool heads_input_ready = false;   // a1 already holds half(x) of the final residual stream
  const int stride = c.infer_attention_stride > 1 ? c.infer_attention_stride : 1;
  for (int i = 0; i < c.blocks; ++i) {
    const m0_block_weights& b = w.blocks[i];
    const TcBlock& tb = st->blocks[i];
    bool run_att = false;
    if (b.has_attention) {
      att_seen++;
      run_att = (att_seen % stride) == 0;
    }
    const bool last = (i + 1 == c.blocks);
    const bool fuse_next = !last && !run_att;
    const bool tc_att = run_att && C == c.attention_heads * 16;
    __nv_bfloat16* next_a = (fuse_next || run_att) ? st->a1 : nullptr;
    if (st->se_fused) {
      // conv1: a2 = act(GN2(conv1(a1))) and, for SE, the half-board sums of a2 that determine conv2's pooled output
      ConvFusion f1;
      f1.prims = c.se ? st->prims : nullptr;
      PROF("conv1+gn", conv3x3(st, st->a1_conv, st->a1_convp, tb.conv1, B, C, nullptr, st->a2, act, s, b.gn2_w, b.gn2_b, nullptr, &f1));
      if (c.se) {
        // SE excitation before conv2 runs: hidden = act(fold * sums + b1), gate = sigmoid(W2 hidden + b2)  (resnet.py:61-64)
        // first layer split over K (60 k-blocks on only B/128 tiles otherwise), partial sums reduced with the bias + activation
        static int se_nosplit = -1;
        if (se_nosplit < 0) se_nosplit = env_int("M0_SE_NOSPLIT", 0);
        if (se_nosplit) {
          // one launch: bias + activation in the GEMM epilogue, hidden layer written in the operand format (no split-K, no reduction kernel)
          PROF("se_fc1", launch_gemm(st, st->prims_mat, tb.se_fold, B, 0, 1, 12 * C, 0, tb.se_fold.n, nullptr, st->se_hid_h, st->hid_pad, 0, b.se_b1, act, 1.0f, s,
                                     nullptr, nullptr, nullptr, c.se_hidden));
        } else {
          PROF("se_fc1", launch_gemm(st, st->prims_mat, tb.se_fold, B, 0, 1, 12 * C, 0, tb.se_fold.n, st->se_part, nullptr, st->hid_pad, 0, none, ACT_NONE, 1.0f, s,
                                     nullptr, nullptr, nullptr, c.se_hidden, 1, st->se_splits, (long long)st->se_rows * st->hid_pad));
          static int se_tail = -1;
          if (se_tail < 0) se_tail = env_int("M0_SE_TAIL", 1);
          if (se_tail) {
            // reduction of the partial sums + bias + activation + second SE layer + sigmoid in one small SIMT launch
            PROF("se_tail", nn_se_tail(st->se_part, st->se_splits, (long long)st->se_rows * st->hid_pad, st->hid_pad, b.se_b1, st->se_w2t[i], b.se_b2,
                                       st->se_gate, B, C, c.se_hidden, act, s));
            goto se_done;
          }
          PROF("se_hidden", nn_se_hidden(st->se_part, st->se_splits, (long long)st->se_rows * st->hid_pad, b.se_b1, st->se_hid_h, B, c.se_hidden, st->hid_pad, act, s));
        }
        PROF("se_fc2", launch_gemm(st, st->se_hid_mat, tb.se_w2, B, 0, 1, st->hid_pad, 0, C, st->se_gate, nullptr, C, 0, b.se_b2, ACT_SIGMOID, 1.0f, s));
      se_done:;
      }
      // conv2 with the whole block tail in its epilogue: x += gate * conv2 ; a1 = act(GN1_{i+1}(x)) (or half(x) before attention)
      ConvFusion f2;
      f2.resid_x = n->x;
      f2.gate = c.se ? st->se_gate : nullptr;
      f2.x_map = &st->x_io;
      PROF("conv2+se+res+gn", conv3x3(st, st->a2_conv, st->a2_convp, tb.conv2, B, C, nullptr, next_a, act, s, fuse_next ? w.blocks[i + 1].gn1_w : nullptr,
                                      fuse_next ? w.blocks[i + 1].gn1_b : nullptr, nullptr, &f2, next_a ? &st->a1_out : nullptr));
    } else {
      // conv1 with GN2 + activation fused into the epilogue: a2 = act(GN2(conv1(a1)))
      PROF("conv1+gn", conv3x3(st, st->a1_conv, st->a1_convp, tb.conv1, B, C, nullptr, st->a2, act, s, b.gn2_w, b.gn2_b, nullptr, nullptr, &st->a2_out));
      // conv2 with the SE squeeze (half-board column sums) fused into the epilogue
      // (conv2's output is kept in the 16-bit operand format, as under the reference's autocast; the fp32 buffer t2 is reused for it)
      __nv_bfloat16* t2h = reinterpret_cast<__nv_bfloat16*>(n->t2);
      PROF("conv2+pool", conv3x3(st, st->a2_conv, st->a2_convp, tb.conv2, B, C, nullptr, t2h, ACT_NONE, s, nullptr, nullptr, c.se ? st->pool : nullptr, nullptr,
                                 &st->t2h_out));
      const float* gate = nullptr;
      if (c.se) {
        PROF("se_gate", nn_se_gate(st->pool, st->se_w1t[i], b.se_b1, st->se_w2t[i], b.se_b2, st->se_gate, B, C, c.se_hidden, act, s));
        gate = st->se_gate;
      }
      // x += conv2 * gate ; a1 = act(GN1_{i+1}(x)), or half(x) when the attention qkv GEMM consumes x next
      PROF("se_apply_gn", nn_se_apply_gn(t2h, gate, n->x, fuse_next ? w.blocks[i + 1].gn1_w : nullptr, fuse_next ? w.blocks[i + 1].gn1_b : nullptr,
                                         next_a, B, C, act, s));
    }
    if (run_att) {
      const float* rb = c.attention_relbias ? b.att_rel_bias : nullptr;
      if (tc_att) {
        PROF("gemm_qkv", gemm_rows64(st, st->a1_mat, tb.qkv, B, C, nullptr, st->qkv_h, 3 * C, s, &st->qkv_out));
        PROF("attention_tc", nn_attention_tc(st->qkv_h, rb, st->a2, B, C, c.attention_heads, c.attention_unmasked_mix, s));
      } else {
        PROF("gemm_qkv", gemm_rows64(st, st->a1_mat, tb.qkv, B, C, n->qkv, nullptr, 3 * C, s));
        PROF("attention_f32", nn_attention_f32(n->qkv, rb, n->t1, B, C, c.attention_heads, c.attention_unmasked_mix, s));
        PROF("f32_to_bf16", nn_f32_to_bf16(n->t1, st->a2, (size_t)M * C, s));
      }
      // the projection leaves the GEMM in the 16-bit operand format, as under the reference's autocast (M0_TC_PROJ_F32=1: fp32 hand-off)
      static int proj_f32 = -1;
      if (proj_f32 < 0) proj_f32 = env_int("M0_TC_PROJ_F32", 0);
      const bool fused_ln = C % 32 == 0 && C <= 320;
      const bool proj_half = fused_ln && !proj_f32;
      if (proj_half) PROF("gemm_proj", gemm_rows64(st, st->a2_mat, tb.proj, B, C, nullptr, reinterpret_cast<__nv_bfloat16*>(n->t2), C, s, &st->t2h_out));
      else PROF("gemm_proj", gemm_rows64(st, st->a2_mat, tb.proj, B, C, n->t2, nullptr, C, s, &st->t2f_out));
      // x = LN(proj + x) and, in the same pass, a1 = act(GN1_{i+1}(x)) for the next block (after the last block: a1 = half(x) for the heads)
      if (fused_ln) {
        heads_input_ready = last && st->heads_tc;
        PROF("ln_res_gn", nn_ln_res_gn(n->t2, proj_half ? 1 : 0, n->x, b.att_ln_w, b.att_ln_b, last ? nullptr : w.blocks[i + 1].gn1_w,
                                       last ? nullptr : w.blocks[i + 1].gn1_b, (last && !st->heads_tc) ? nullptr : st->a1, B, C, act, s));
      } else {
        PROF("layernorm_residual_f32", nn_layernorm_residual_f32(n->t2, n->x, b.att_ln_w, b.att_ln_b, n->x, M, C, s));
        if (!last) PROF("se_apply_gn", nn_se_apply_gn(nullptr, nullptr, n->x, w.blocks[i + 1].gn1_w, w.blocks[i + 1].gn1_b, st->a1, B, C, act, s));
      }
    }
  }
  if (!st->heads_tc) return net_forward_heads_f32(n, B, logits, values, s);
  // ---- heads (resnet.py:697-753) on tensor cores; the three small value layers after fc1 stay in fp32 ----
  const int vact = c.value_activation, r = c.policy_factor_rank, rp = st->pol_rank_pad;
  if (!heads_input_ready) PROF("f32_to_bf16", nn_f32_to_bf16(n->x, st->a1, (size_t)M * C, s));
  // policy: conv1x1 C->64, GN, act, fc1 + ReLU, fc2 * logit scale
  PROF("gemm_pol_conv", launch_gemm(st, st->a1_mat, st->pol_conv, M, 0, 1, C, 0, 64, n->t1, nullptr, 64, 0, none, ACT_NONE, 1.0f, s));
  PROF("gn_act_res", nn_gn_act_res(n->t1, w.pol_gn_w, w.pol_gn_b, nullptr, 0, nullptr, st->ph_h, B, 64, act, s));
  PROF("gemm_pol_fc1", launch_gemm(st, st->ph_mat, st->pol_fc1, B, 0, 1, 4096, 0, r, nullptr, st->pf_h, rp, 0, w.pol_fc1_b, ACT_RELU, 1.0f, s));
  // one launch over all 320-column slices of the (zero-padded) policy_fc2 weight; the padding columns are not stored
  PROF("gemm_pol_fc2", launch_gemm(st, st->pf_mat, st->pol_fc2, B, 0, 1, rp, 0, 320, logits, nullptr, c.policy_size, 0, w.pol_fc2_b, ACT_NONE,
                                   w.policy_logit_scale, s, nullptr, nullptr, nullptr, c.policy_size, (c.policy_size + 319) / 320));
  // value: conv1x1 C->128, GN, act, conv1x1 128->128, GN, act, fc1 (+ activation) on tensor cores
  PROF("gemm_val_conv1", launch_gemm(st, st->a1_mat, st->val_conv1, M, 0, 1, C, 0, 128, n->vh1, nullptr, 128, 0, none, ACT_NONE, 1.0f, s));
  PROF("gn_act_res", nn_gn_act_res(n->vh1, w.val_gn1_w, w.val_gn1_b, nullptr, 0, nullptr, st->vh_h, B, 128, act, s));
  PROF("gemm_val_conv2", launch_gemm(st, st->vh_conv_mat, st->val_conv2, M, 0, 1, 128, 0, 128, n->vh1, nullptr, 128, 0, none, ACT_NONE, 1.0f, s));
  PROF("gn_act_res", nn_gn_act_res(n->vh1, w.val_gn2_w, w.val_gn2_b, nullptr, 0, nullptr, st->vh_h, B, 128, act, s));
  if (st->val_tail_tc) {
    // fc1 (+ activation) -> 16-bit, fc2 (+ activation) and the gate's linear layer + sigmoid on tensor cores (resnet.py:747-752);
    // value = tanh(fc3(fc2_out * gate)) in one small reduction kernel
    PROF("gemm_val_fc1", launch_gemm(st, st->vh_fc_mat, st->val_fc1, B, 0, 1, 8192, 0, st->val_fc1.n_launch, nullptr, st->vf1_h, 2 * C, 0, w.val_fc1_b, vact,
                                     1.0f, s, nullptr, nullptr, nullptr, -1, 2 * C / st->val_fc1.n_launch));
    PROF("gemm_val_fc2", launch_gemm(st, st->vf1_mat, st->val_fc2, B, 0, 1, 2 * C, 0, st->val_fc2.n_launch, n->vf2, st->vf2_h, C, 0, w.val_fc2_b, vact, 1.0f, s,
                                     nullptr, nullptr, nullptr, -1, C / st->val_fc2.n_launch));
    PROF("gemm_val_gate", launch_gemm(st, st->vf2_mat, st->val_gate, B, 0, 1, C, 0, st->val_gate.n_launch, n->vg, nullptr, C, 0, w.val_gate_b, ACT_SIGMOID, 1.0f,
                                      s, nullptr, nullptr, nullptr, -1, C / st->val_gate.n_launch));
    PROF("value_tail", nn_value_tail(n->vg, n->vf2, w.val_fc3_w, w.val_fc3_b, values, B, C, s));
  } else {
    PROF("gemm_val_fc1", launch_gemm(st, st->vh_fc_mat, st->val_fc1, B, 0, 1, 8192, 0, st->val_fc1.n_launch, n->vf1, nullptr, 2 * C, 0, w.val_fc1_b, vact, 1.0f,
                                     s, nullptr, nullptr, nullptr, -1, 2 * C / st->val_fc1.n_launch));
    PROF("gemm_f32", nn_gemm_f32(A_DIRECT, n->vf1, w.val_fc2_w, w.val_fc2_b, nullptr, n->vf2, B, C, 2 * C, 2 * C, C, 0, vact, 1.0f, s));
    PROF("gemm_f32", nn_gemm_f32(A_DIRECT, n->vf2, w.val_gate_w, w.val_gate_b, n->vf2, n->vg, B, C, C, C, C, 0, ACT_SIGMOID, 1.0f, s));
    PROF("gemm_f32", nn_gemm_f32(A_DIRECT, n->vg, w.val_fc3_w, w.val_fc3_b, nullptr, values, B, 1, C, C, 1, 0, ACT_TANH, 1.0f, s));
  }
  if (TcProfiler::get().enabled()) TcProfiler::get().collect();
  return M0_OK;
}

}  // namespace m0

// Stand-alone entry point of the tensor-core convolution / GEMM (tests and the roofline micro-benchmark):
//   taps = 9: out[b*64+sq][n] = conv3x3(act NHWC bf16 [boards][8][8][cin], w [n][9*cin]) ; taps = 1: plain GEMM act[boards*64][cin] x w[n][cin]^T
extern "C" int m0_tc_conv(const uint16_t* d_act_bf16, const uint16_t* d_w_bf16, int boards, int cin, int n, int taps, float* d_out_f32,
                          void* stream) {
  if (!d_act_bf16 || !d_w_bf16 || !d_out_f32 || boards <= 0 || (boards & 1) || cin <= 0 || cin % 32 != 0 || n % 16 != 0 || n > 320 ||
      (taps != 1 && taps != 9)) {
    m0_set_error("m0_tc_conv: invalid argument (boards even, cin %% 32 == 0, n %% 16 == 0, n <= 320, taps in {1, 9})");
    return M0_ERR_ARG;
  }
  // the operands of this entry point are bf16 by contract, whatever 16-bit format the last forward of the process selected
  struct FormatGuard {
    int saved;
    FormatGuard() : saved(nn_half_format()) { nn_set_half_format(0); }
    ~FormatGuard() { nn_set_half_format(saved); }
  } format_guard;
  static TcState st;
  static int st_dev = -1;
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev != st_dev) {   // shared-memory grants are per device
    for (size_t& v : st.smem_pair) v = 0;
    st.smem_gemm = 0;
    st_dev = dev;
  }
  cudaDeviceGetAttribute(&st.sm_count, cudaDevAttrMultiProcessorCount, dev);
  cudaDeviceGetAttribute(&st.max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  const cudaStream_t s = (cudaStream_t)stream;
  // 3x3 weights with cin % 64 == 32 are copied with every tap padded to whole k-blocks (the layout make_weight gives the network's
  // weights); the copy is stream-ordered and freed after the launch
  const int kw = taps * kblocks_for(cin) * 64;
  void* w_pad = nullptr;
  if (taps == 9 && kw != taps * cin) {
    M0_CUDA_TRY(cudaMallocAsync(&w_pad, (size_t)n * kw * 2, s));
    pad_cols_kernel<uint16_t><<<(n * kw + 255) / 256, 256, 0, s>>>(d_w_bf16, (uint16_t*)w_pad, n * taps, cin, kw / taps);
    const int rc = m0_check_launch("pad_taps");
    if (rc != M0_OK) { cudaFreeAsync(w_pad, s); return rc; }
  }
  auto run = [&](const void* wp, int k) -> int {
    TcWeight w;
    w.w = (__nv_bfloat16*)wp;
    w.n = n;
    w.k = k;
    w.n_part = n_part_for(n);
    w.cluster = pick_cluster(w.n_part);
    TRY(make_map_2d(&w.map, wp, (uint64_t)n, (uint64_t)k, (uint32_t)(w.n_part / w.cluster)));
    CUtensorMap a;
    w.n_launch = n;
    if (taps == 9 && pair_ok(n)) {
      w.pair = true;
      TRY(make_map_2d(&w.map_pair, wp, (uint64_t)n, (uint64_t)k, (uint32_t)(n / 4)));
      TRY(make_map_nhwc(&a, d_act_bf16, (uint64_t)boards, (uint64_t)cin, 10));
      CUtensorMap om;
      TRY(make_map_out(&om, d_out_f32, (uint64_t)boards * 64, (uint64_t)n, true));
      return launch_conv_pair(&st, a, w, boards, cin, d_out_f32, nullptr, n, ACT_NONE, s, nullptr, nullptr, nullptr, nullptr, 1, 1, &om);
    }
    if (taps == 1 && pair_ok(n) && cin <= 320) {   // plain GEMM over whole boards on the CTA-pair kernel (qkv / proj / piece-square projections)
      w.pair = true;
      TRY(make_map_2d(&w.map_pair, wp, (uint64_t)n, (uint64_t)cin, (uint32_t)(n / 4)));
      TRY(make_map_2d(&a, d_act_bf16, (uint64_t)boards * 64, (uint64_t)cin, 128));
      return launch_conv_pair(&st, a, w, boards, cin, d_out_f32, nullptr, n, ACT_NONE, s, nullptr, nullptr, nullptr, nullptr, 0, 1);
    }
    if (taps == 9) TRY(make_map_nhwc(&a, d_act_bf16, (uint64_t)boards, (uint64_t)cin));
    else TRY(make_map_2d(&a, d_act_bf16, (uint64_t)boards * 64, (uint64_t)cin, 128));
    return launch_gemm(&st, a, w, boards * 64, taps == 9 ? 1 : 0, taps, cin, 0, n, d_out_f32, nullptr, n, 0, nullptr, ACT_NONE, 1.0f, s);
  };
  const int rc = w_pad ? run(w_pad, kw) : run(d_w_bf16, taps * cin);
  if (w_pad) cudaFreeAsync(w_pad, s);
  return rc;
}

// ---- per-launch-site timing of the tensor-core forward (bench.py roofline; diagnostics) -------------------------------------------
extern "C" int m0_profile_enable(int enable) {
  TcProfiler& p = TcProfiler::get();
  p.reset();
  p.set(enable);
  return M0_OK;
}
// accumulated milliseconds and launch count of one launch site ("conv1+gn", "conv2+pool", "se_apply_gn", ...); name == NULL sums all
extern "C" int m0_profile_get(const char* name, double* total_ms, long long* launches) {
  TcProfiler& p = TcProfiler::get();
  p.collect();
  double ms = 0;
  long long cnt = 0;
  for (auto& kv : p.acc)
    if (!name || kv.first == name) { ms += kv.second.first; cnt += kv.second.second; }
  if (total_ms) *total_ms = ms;
  if (launches) *launches = cnt;
  return M0_OK;
}
