// FP32 kernels of the PolicyValueNet inference forward (azchess/model/resnet.py:656-760).
//
// This is the exactness-oriented path (BASELINE north_star: "fp32 NN path within 1e-4 relative"):
// plain SIMT kernels with fp32 accumulation, no tensor cores.  The throughput path is the bf16
// tcgen05 implicit-GEMM pipeline in nn_tc_kernels.cu; both share the activation layout
// (NHWC: [board][square = row*8 + col][channel]) and the weight layout (GEMM "B" operand
// W[n][k], k = (ky*3 + kx)*Cin + ci for 3x3 convolutions).
#include "nn.cuh"
#include <cuda_fp16.h>
#include <cuda_fp8.h>

namespace m0 {

// 16-bit operand format of the tensor-core path: bf16 (default) or IEEE fp16, selected per forward call
static int g_half_fp16 = 0;
void nn_set_half_format(int fp16) { g_half_fp16 = fp16 ? 1 : 0; }
int nn_half_format() { return g_half_fp16; }

__device__ __forceinline__ __nv_bfloat16 to_half16(float x, int fp16) {
  if (fp16) {
    __half h = __float2half_rn(x);
    return *reinterpret_cast<__nv_bfloat16*>(&h);  // storage is an opaque 16-bit word
  }
  return __float2bfloat16(x);
}

__device__ __forceinline__ float act_apply(float x, int act) {
  switch (act) {
    case ACT_RELU: return x > 0.0f ? x : 0.0f;
    case ACT_SILU: return x / (1.0f + expf(-x));
    case ACT_LEAKY: return x > 0.0f ? x : 0.05f * x;  // F.leaky_relu(negative_slope=0.05), resnet.py:588
    case ACT_TANH: return tanhf(x);
    case ACT_SIGMOID: return 1.0f / (1.0f + expf(-x));
    default: return x;
  }
}

// ---- generic GEMM: C[m][n] = act(sum_k A(m,k) * W[n][k] + bias[n]) * scale (* mul[m][n]) ------------------
// A(m,k) comes from one of three loaders: a row-major matrix, the 3x3 im2col view of NHWC
// activations (zero padding), or the 3x3 im2col view of the NCHW input planes.
template <int MODE>
__device__ __forceinline__ float gemm_load_a(const float* __restrict__ A, int m, int k, int K, int lda, int cin) {
  if (MODE == A_DIRECT) return A[(size_t)m * lda + k];
  const int b = m >> 6, sq = m & 63;
  const int tap = k / cin, ci = k - tap * cin;
  const int y = (sq >> 3) + tap / 3 - 1, x = (sq & 7) + tap % 3 - 1;
  if ((unsigned)y >= 8u || (unsigned)x >= 8u) return 0.0f;
  if (MODE == A_IM2COL_NHWC) return A[((size_t)b * 64 + y * 8 + x) * cin + ci];
  return A[((size_t)b * cin + ci) * 64 + y * 8 + x];  // A_IM2COL_NCHW
}

template <int MODE>
__global__ void __launch_bounds__(256)
gemm_f32_kernel(const float* __restrict__ A, const float* __restrict__ W, const float* __restrict__ bias,
                const float* __restrict__ mul, float* __restrict__ C, int M, int N, int K, int lda, int ldc, int cin,
                int act, float scale) {
  constexpr int BM = 64, BN = 64, BK = 16;
  __shared__ float sA[BK][BM + 4];
  __shared__ float sW[BK][BN + 4];
  const int tid = threadIdx.x;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tm = (tid >> 4) * 4, tn = (tid & 15) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
  for (int k0 = 0; k0 < K; k0 += BK) {
    // 64x16 tiles: 1024 elements, 4 per thread; consecutive threads walk k (contiguous in memory)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      int idx = tid + e * 256;
      int kk = idx & 15, r = idx >> 4;
      int k = k0 + kk;
      float va = 0.0f, vw = 0.0f;
      if (k < K) {
        if (m0 + r < M) va = gemm_load_a<MODE>(A, m0 + r, k, K, lda, cin);
        if (n0 + r < N) vw = W[(size_t)(n0 + r) * K + k];
      }
      sA[kk][r] = va;
      sW[kk][r] = vw;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < BK; ++kk) {
      float a[4], w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sA[kk][tm + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) w[j] = sW[kk][tn + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int m = m0 + tm + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      int n = n0 + tn + j;
      if (n >= N) continue;
      float v = acc[i][j];
      if (bias) v += bias[n];
      v = act_apply(v, act) * scale;
      if (mul) v *= mul[(size_t)m * ldc + n];
      C[(size_t)m * ldc + n] = v;
    }
  }
}

// ---- GroupNorm (+activation, +residual): nn.GroupNorm(C/16, C), eps 1e-5 (resnet.py:18-24) ----------------
// x, out: NHWC [B][64][C]; one block per board, one thread per channel; groups of 16 channels are
// half-warps.  out = act(GN(x)) + residual  (residual optional, batch stride may be 0 = broadcast)
__global__ void groupnorm_f32_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta,
                                     const float* __restrict__ residual, long long residual_bstride, float* __restrict__ out,
                                     __nv_bfloat16* __restrict__ out_bf16, int C, int act, int fp16) {
  const int b = blockIdx.x, c = threadIdx.x;
  const float* xb = x + (size_t)b * 64 * C;
  float s = 0.0f;
  for (int sq = 0; sq < 64; ++sq) s += xb[sq * C + c];
#pragma unroll
  for (int off = 8; off > 0; off >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, off);
  const float mean = s * (1.0f / 1024.0f);
  float v = 0.0f;
  for (int sq = 0; sq < 64; ++sq) {
    float d = xb[sq * C + c] - mean;
    v = fmaf(d, d, v);
  }
#pragma unroll
  for (int off = 8; off > 0; off >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, off);
  const float rstd = rsqrtf(v * (1.0f / 1024.0f) + 1e-5f);
  const float g = gamma[c] * rstd, bb = beta[c] - mean * g;
  float* ob = out ? out + (size_t)b * 64 * C : nullptr;
  __nv_bfloat16* hb = out_bf16 ? out_bf16 + (size_t)b * 64 * C : nullptr;
  const float* rb = residual ? residual + (size_t)b * residual_bstride : nullptr;
  for (int sq = 0; sq < 64; ++sq) {
    float y = act_apply(fmaf(xb[sq * C + c], g, bb), act);
    if (rb) y += rb[sq * C + c];
    if (ob) ob[sq * C + c] = y;
    if (hb) hb[sq * C + c] = to_half16(y, fp16);
  }
}

// fp32 -> bf16 copy (weights at prepare time; activations that feed a tensor-core GEMM)
__global__ void f32_to_bf16_kernel(const float* __restrict__ in, __nv_bfloat16* __restrict__ out, size_t n, int fp16) {
  size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i + 3 < n) {
    float4 v = *reinterpret_cast<const float4*>(in + i);
    out[i] = to_half16(v.x, fp16);
    out[i + 1] = to_half16(v.y, fp16);
    out[i + 2] = to_half16(v.z, fp16);
    out[i + 3] = to_half16(v.w, fp16);
  } else {
    for (; i < n; ++i) out[i] = to_half16(in[i], fp16);
  }
}

// ---- squeeze-excitation + residual: resnet.py:59-80 ---------------------------------------------------------
// x_out = x + conv_out * sigmoid(W2 * act(W1 * avgpool(conv_out) + b1) + b2); one block per board, C threads
__global__ void se_residual_f32_kernel(const float* __restrict__ conv_out, const float* __restrict__ x,
                                       const float* __restrict__ w1, const float* __restrict__ b1,
                                       const float* __restrict__ w2, const float* __restrict__ b2,
                                       float* __restrict__ x_out, int C, int hidden, int act, int use_se) {
  extern __shared__ float sm[];
  float* s_pool = sm;          // [C]
  float* s_hid = sm + C;       // [hidden]
  const int b = blockIdx.x, c = threadIdx.x;
  const float* ob = conv_out + (size_t)b * 64 * C;
  float e = 1.0f;
  if (use_se) {
    float s = 0.0f;
    for (int sq = 0; sq < 64; ++sq) s += ob[sq * C + c];
    s_pool[c] = s * (1.0f / 64.0f);
    __syncthreads();
    if (c < hidden) {
      float h = b1[c];
      for (int i = 0; i < C; ++i) h = fmaf(w1[(size_t)c * C + i], s_pool[i], h);
      s_hid[c] = act_apply(h, act);
    }
    __syncthreads();
    float z = b2[c];
    for (int j = 0; j < hidden; ++j) z = fmaf(w2[(size_t)c * hidden + j], s_hid[j], z);
    e = 1.0f / (1.0f + expf(-z));
  }
  const float* xb = x + (size_t)b * 64 * C;
  float* yb = x_out + (size_t)b * 64 * C;
  for (int sq = 0; sq < 64; ++sq) yb[sq * C + c] = xb[sq * C + c] + ob[sq * C + c] * e;
}

// ---- ChessAttention core: resnet.py:141-174 --------------------------------------------------------------------
// qkv NHWC [B][64][3C] with channel = which*C + head*D + d (resnet.py:142-144); out [B][64][C], channel = head*D + d.
// One block per (board, head), one thread per query square.
__device__ __forceinline__ bool chess_attn_mask(int i, int j) {  // resnet.py:105-129
  int ri = i >> 3, ci = i & 7, rj = j >> 3, cj = j & 7;
  int dr = ri - rj, dc = ci - cj;
  int adr = dr < 0 ? -dr : dr, adc = dc < 0 ? -dc : dc;
  return dr == 0 || dc == 0 || adr == adc || (adr == 2 && adc == 1) || (adr == 1 && adc == 2) || (adr <= 1 && adc <= 1);
}

template <int D>
__global__ void __launch_bounds__(64)
attention_f32_kernel(const float* __restrict__ qkv, const float* __restrict__ rel_bias, float* __restrict__ out, int C, int heads,
                     float unmasked_mix) {
  __shared__ float sk[64][D + 1];
  __shared__ float sv[64][D + 1];
  const int b = blockIdx.x / heads, h = blockIdx.x % heads, i = threadIdx.x;
  const float* base = qkv + ((size_t)b * 64 + i) * 3 * C + h * D;
  float q[D];
#pragma unroll
  for (int d = 0; d < D; ++d) {
    q[d] = base[d];
    sk[i][d] = base[C + d];
    sv[i][d] = base[2 * C + d];
  }
  __syncthreads();
  const float inv_sqrt = 1.0f / sqrtf((float)D);
  float sc[64];
  float mx_u = -INFINITY, mx_m = -INFINITY;
  const float* rb = rel_bias ? rel_bias + ((size_t)h * 64 + i) * 64 : nullptr;
#pragma unroll 4
  for (int j = 0; j < 64; ++j) {
    float s = 0.0f;
#pragma unroll
    for (int d = 0; d < D; ++d) s = fmaf(q[d], sk[j][d], s);
    s *= inv_sqrt;
    if (rb) s += rb[j];
    s = fminf(fmaxf(s, -50.0f), 50.0f);
    sc[j] = s;
    mx_u = fmaxf(mx_u, s);
    mx_m = fmaxf(mx_m, chess_attn_mask(i, j) ? s : -1e4f);
  }
  float sum_u = 0.0f, sum_m = 0.0f;
  float ou[D], om[D];
#pragma unroll
  for (int d = 0; d < D; ++d) ou[d] = om[d] = 0.0f;
#pragma unroll 4
  for (int j = 0; j < 64; ++j) {
    float eu = expf(sc[j] - mx_u);
    float em = expf((chess_attn_mask(i, j) ? sc[j] : -1e4f) - mx_m);
    sum_u += eu;
    sum_m += em;
#pragma unroll
    for (int d = 0; d < D; ++d) {
      ou[d] = fmaf(eu, sv[j][d], ou[d]);
      om[d] = fmaf(em, sv[j][d], om[d]);
    }
  }
  const float blend = 1.0f - unmasked_mix;
  float* o = out + ((size_t)b * 64 + i) * C + h * D;
#pragma unroll
  for (int d = 0; d < D; ++d) {
    float vm = om[d] / sum_m, vu = ou[d] / sum_u;
    float r;
    if (unmasked_mix > 0.0f && unmasked_mix < 1.0f) r = blend * vm + (1.0f - blend) * vu;  // resnet.py:160-167
    else if (unmasked_mix >= 1.0f) r = vm;
    else r = vu;
    o[d] = r;
  }
}

// ---- residual + LayerNorm over channels: resnet.py:182-188 ------------------------------------------------------------
// out[t][:] = LN(proj[t][:] + x[t][:]) for every token t = (board, square); one warp per token
__global__ void layernorm_residual_f32_kernel(const float* __restrict__ proj, const float* __restrict__ x,
                                              const float* __restrict__ gamma, const float* __restrict__ beta,
                                              float* __restrict__ out, int tokens, int C) {
  const int t = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (t >= tokens) return;
  const float* p = proj + (size_t)t * C;
  const float* xr = x + (size_t)t * C;
  float s = 0.0f;
  for (int c = lane; c < C; c += 32) s += p[c] + xr[c];
  for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xFFFFFFFFu, s, off);
  const float mean = s / (float)C;
  float v = 0.0f;
  for (int c = lane; c < C; c += 32) {
    float d = p[c] + xr[c] - mean;
    v = fmaf(d, d, v);
  }
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, off);
  const float rstd = rsqrtf(v / (float)C + 1e-5f);
  float* o = out + (size_t)t * C;
  for (int c = lane; c < C; c += 32) o[c] = (p[c] + xr[c] - mean) * rstd * gamma[c] + beta[c];
}

// Tensor-core path: x_new = LN(proj + x) (resnet.py:182-188) and, fused, a_out = half(act(GroupNorm_16ch(x_new))) = the bn1 +
// activation of the next residual block (resnet.py:46-47).  One block (8 warps) per board; warp w owns tokens 8w..8w+7, lane l
// owns channels 2l + 64j (j < NJ = ceil(C / 64)): proj and x are read once, the sums live in registers for both normalisations.
// C % 64 == 32: the last j holds channels for lanes 0..15 only (two GroupNorm groups); the other lanes' values there are zero and
// take no part in the LayerNorm statistics or the stores.
// HALF_IN: proj is the 16-bit output of the projection GEMM (the reference's proj convolution runs under autocast, resnet.py:676-677);
// gn_g == nullptr with a_out != nullptr: a_out = half(x_new) without the GroupNorm (the operand of the head GEMMs after the last block)
// fp16 = 2 (precision fp8): 16-bit values are fp16 and the GroupNorm'ed a_out is e4m3 (the operand of the next e4m3 conv1)
template <int C, bool HALF_IN>
__global__ void __launch_bounds__(256, 2)
ln_res_gn_kernel(const float* __restrict__ proj, float* __restrict__ x, const float* __restrict__ ln_g, const float* __restrict__ ln_b,
                 const float* __restrict__ gn_g, const float* __restrict__ gn_b, __nv_bfloat16* __restrict__ a_out, int act, int fp16) {
  constexpr int NJ = (C + 63) / 64;
  __shared__ float s_part[8][NJ][4][2];
  const int b = blockIdx.x, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const size_t base = ((size_t)b * 64 + warp * 8) * C + 2 * lane;
  // channels 2 lane + 64 j exist (always, unless C % 64 == 32 and j is the last k-block)
  auto has = [lane](int j) { return C % 64 == 0 || j < NJ - 1 || lane < 16; };
  float v[8][2 * NJ];
#pragma unroll
  for (int t = 0; t < 8; ++t)
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      if (!has(j)) { v[t][2 * j] = v[t][2 * j + 1] = 0.f; continue; }
      float2 p2;
      if (HALF_IN) {
        const uint32_t h = __ldg(reinterpret_cast<const uint32_t*>(reinterpret_cast<const uint16_t*>(proj) + base + (size_t)t * C + 64 * j));
        if (fp16) p2 = __half22float2(*reinterpret_cast<const __half2*>(&h));
        else p2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&h));
      } else {
        p2 = __ldg(reinterpret_cast<const float2*>(proj + base + (size_t)t * C + 64 * j));
      }
      const float2 x2 = *reinterpret_cast<const float2*>(x + base + (size_t)t * C + 64 * j);
      v[t][2 * j] = p2.x + x2.x;
      v[t][2 * j + 1] = p2.y + x2.y;
    }
  float lg[2 * NJ], lb[2 * NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    if (!has(j)) { lg[2 * j] = lg[2 * j + 1] = lb[2 * j] = lb[2 * j + 1] = 0.f; continue; }
    const float2 g2 = *reinterpret_cast<const float2*>(ln_g + 2 * lane + 64 * j), b2 = *reinterpret_cast<const float2*>(ln_b + 2 * lane + 64 * j);
    lg[2 * j] = g2.x; lg[2 * j + 1] = g2.y; lb[2 * j] = b2.x; lb[2 * j + 1] = b2.y;
  }
  // LayerNorm over the C channels of each token (two-pass, from registers)
  float mean[8], rstd[8];
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 2 * NJ; ++k) s += v[t][k];
    mean[t] = s;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1)
#pragma unroll
    for (int t = 0; t < 8; ++t) mean[t] += __shfl_xor_sync(0xFFFFFFFFu, mean[t], off);
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    mean[t] *= (1.0f / C);
    float d2 = 0.f;
#pragma unroll
    for (int k = 0; k < 2 * NJ; ++k) {
      if (!has(k >> 1)) continue;
      const float d = v[t][k] - mean[t];
      d2 = fmaf(d, d, d2);
    }
    rstd[t] = d2;
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1)
#pragma unroll
    for (int t = 0; t < 8; ++t) rstd[t] += __shfl_xor_sync(0xFFFFFFFFu, rstd[t], off);
#pragma unroll
  for (int t = 0; t < 8; ++t) {
    rstd[t] = rsqrtf(rstd[t] * (1.0f / C) + 1e-5f);
#pragma unroll
    for (int k = 0; k < 2 * NJ; ++k) v[t][k] = (v[t][k] - mean[t]) * rstd[t] * lg[k] + lb[k];
#pragma unroll
    for (int j = 0; j < NJ; ++j)
      if (has(j)) *reinterpret_cast<float2*>(x + base + (size_t)t * C + 64 * j) = make_float2(v[t][2 * j], v[t][2 * j + 1]);
  }
  if (!a_out) return;
  if (!gn_g) {   // plain 16-bit copy of the new residual stream
#pragma unroll
    for (int t = 0; t < 8; ++t)
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        if (!has(j)) continue;
        uint32_t pk;
        if (fp16) { __half2 h = __floats2half2_rn(v[t][2 * j], v[t][2 * j + 1]); pk = *reinterpret_cast<uint32_t*>(&h); }
        else { __nv_bfloat162 h = __floats2bfloat162_rn(v[t][2 * j], v[t][2 * j + 1]); pk = *reinterpret_cast<uint32_t*>(&h); }
        *reinterpret_cast<uint32_t*>(a_out + base + (size_t)t * C + 64 * j) = pk;
      }
    return;
  }
  // GroupNorm over (board, 16 channels): channel 2l + 64j belongs to group 4j + l / 8 -> 8 lanes x 8 tokens x 8 warps
  const int sub = lane >> 3;
  float gm[NJ], gr[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < 8; ++t) s += v[t][2 * j] + v[t][2 * j + 1];
    s += __shfl_xor_sync(0xFFFFFFFFu, s, 1); s += __shfl_xor_sync(0xFFFFFFFFu, s, 2); s += __shfl_xor_sync(0xFFFFFFFFu, s, 4);
    if ((lane & 7) == 0) s_part[warp][j][sub][0] = s;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += s_part[w][j][sub][0];
    gm[j] = tot * (1.0f / 1024.0f);
    float d2 = 0.f;
#pragma unroll
    for (int t = 0; t < 8; ++t) {
      const float a0 = v[t][2 * j] - gm[j], a1 = v[t][2 * j + 1] - gm[j];
      d2 = fmaf(a0, a0, d2);
      d2 = fmaf(a1, a1, d2);
    }
    d2 += __shfl_xor_sync(0xFFFFFFFFu, d2, 1); d2 += __shfl_xor_sync(0xFFFFFFFFu, d2, 2); d2 += __shfl_xor_sync(0xFFFFFFFFu, d2, 4);
    if ((lane & 7) == 0) s_part[warp][j][sub][1] = d2;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += s_part[w][j][sub][1];
    gr[j] = rsqrtf(tot * (1.0f / 1024.0f) + 1e-5f);
  }
  if (gn_g) {
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
      if (!has(j)) continue;
      const float2 g2 = *reinterpret_cast<const float2*>(gn_g + 2 * lane + 64 * j), b2 = *reinterpret_cast<const float2*>(gn_b + 2 * lane + 64 * j);
      const float g0 = g2.x * gr[j], g1 = g2.y * gr[j];
      const float b0 = b2.x - gm[j] * g0, b1 = b2.y - gm[j] * g1;
#pragma unroll
      for (int t = 0; t < 8; ++t) {
        float y0 = fmaf(v[t][2 * j], g0, b0), y1 = fmaf(v[t][2 * j + 1], g1, b1);
        if (act == ACT_SILU) { y0 = __fdividef(y0, 1.0f + __expf(-y0)); y1 = __fdividef(y1, 1.0f + __expf(-y1)); }
        else if (act == ACT_RELU) { y0 = fmaxf(y0, 0.f); y1 = fmaxf(y1, 0.f); }
        if (fp16 == 2) {
          *reinterpret_cast<uint16_t*>(reinterpret_cast<uint8_t*>(a_out) + base + (size_t)t * C + 64 * j) =
              __nv_cvt_float2_to_fp8x2(make_float2(y0, y1), __NV_SATFINITE, __NV_E4M3);
          continue;
        }
        uint32_t pk;
        if (fp16) { __half2 h = __floats2half2_rn(y0, y1); pk = *reinterpret_cast<uint32_t*>(&h); }
        else { __nv_bfloat162 h = __floats2bfloat162_rn(y0, y1); pk = *reinterpret_cast<uint32_t*>(&h); }
        *reinterpret_cast<uint32_t*>(a_out + base + (size_t)t * C + 64 * j) = pk;
      }
    }
  }
}

// NHWC [B][64][C] -> NCHW [B][C][8][8] (SSL head outputs are returned in the reference's layout)
__global__ void nhwc_to_nchw_f32_kernel(const float* __restrict__ in, float* __restrict__ out, int B, int C) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t total = (size_t)B * 64 * C;
  if (i >= total) return;
  int sq = (int)(i & 63);
  size_t bc = i >> 6;
  int c = (int)(bc % C);
  size_t b = bc / C;
  out[i] = in[(b * 64 + sq) * C + c];
}

// ---- launch helpers (host) -----------------------------------------------------------------------------------------------------
int nn_gemm_f32(int mode, const float* A, const float* W, const float* bias, const float* mul, float* C, int M, int N, int K,
                int lda, int ldc, int cin, int act, float scale, cudaStream_t s) {
  dim3 grid((N + 63) / 64, (M + 63) / 64);
  if (mode == A_DIRECT) gemm_f32_kernel<A_DIRECT><<<grid, 256, 0, s>>>(A, W, bias, mul, C, M, N, K, lda, ldc, cin, act, scale);
  else if (mode == A_IM2COL_NHWC) gemm_f32_kernel<A_IM2COL_NHWC><<<grid, 256, 0, s>>>(A, W, bias, mul, C, M, N, K, lda, ldc, cin, act, scale);
  else gemm_f32_kernel<A_IM2COL_NCHW><<<grid, 256, 0, s>>>(A, W, bias, mul, C, M, N, K, lda, ldc, cin, act, scale);
  return m0_check_launch("gemm_f32");
}
int nn_groupnorm_f32(const float* x, const float* gamma, const float* beta, const float* residual, long long residual_bstride,
                     float* out, int B, int C, int act, cudaStream_t s) {
  groupnorm_f32_kernel<<<B, C, 0, s>>>(x, gamma, beta, residual, residual_bstride, out, nullptr, C, act, 0);
  return m0_check_launch("groupnorm_f32");
}
int nn_groupnorm_mixed(const float* x, const float* gamma, const float* beta, const float* residual, long long residual_bstride,
                       float* out, __nv_bfloat16* out_bf16, int B, int C, int act, cudaStream_t s) {
  groupnorm_f32_kernel<<<B, C, 0, s>>>(x, gamma, beta, residual, residual_bstride, out, out_bf16, C, act, g_half_fp16);
  return m0_check_launch("groupnorm_mixed");
}
int nn_f32_to_bf16(const float* in, __nv_bfloat16* out, size_t n, cudaStream_t s) {
  if (n == 0) return M0_OK;
  size_t threads = (n + 3) / 4;
  f32_to_bf16_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, s>>>(in, out, n, g_half_fp16);
  return m0_check_launch("f32_to_bf16");
}
int nn_se_residual_f32(const float* conv_out, const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                       float* x_out, int B, int C, int hidden, int act, int use_se, cudaStream_t s) {
  se_residual_f32_kernel<<<B, C, (C + hidden) * sizeof(float), s>>>(conv_out, x, w1, b1, w2, b2, x_out, C, hidden, act, use_se);
  return m0_check_launch("se_residual_f32");
}
int nn_attention_f32(const float* qkv, const float* rel_bias, float* out, int B, int C, int heads, float unmasked_mix, cudaStream_t s) {
  const int D = C / heads;
  if (D == 16) attention_f32_kernel<16><<<B * heads, 64, 0, s>>>(qkv, rel_bias, out, C, heads, unmasked_mix);
  else if (D == 8) attention_f32_kernel<8><<<B * heads, 64, 0, s>>>(qkv, rel_bias, out, C, heads, unmasked_mix);
  else if (D == 32) attention_f32_kernel<32><<<B * heads, 64, 0, s>>>(qkv, rel_bias, out, C, heads, unmasked_mix);
  else { m0_set_error("attention: unsupported head_dim %d", D); return M0_ERR_ARG; }
  return m0_check_launch("attention_f32");
}
int nn_layernorm_residual_f32(const float* proj, const float* x, const float* gamma, const float* beta, float* out, int tokens, int C,
                              cudaStream_t s) {
  layernorm_residual_f32_kernel<<<(tokens + 7) / 8, 256, 0, s>>>(proj, x, gamma, beta, out, tokens, C);
  return m0_check_launch("layernorm_residual_f32");
}
// x <- LN(proj + x) in place; a_out (optional) = half(act(GroupNorm(x))) with the next block's bn1 parameters
int nn_ln_res_gn(const void* proj, int proj_half, float* x, const float* ln_g, const float* ln_b, const float* gn_g, const float* gn_b,
                 __nv_bfloat16* a_out, int B, int C, int act, cudaStream_t s, bool a_e4m3) {
  const int fp16 = a_e4m3 ? 2 : g_half_fp16;
  const float* p = reinterpret_cast<const float*>(proj);
#define M0_LN_CASE(C)                                                                                                     \
  if (proj_half) ln_res_gn_kernel<C, true><<<B, 256, 0, s>>>(p, x, ln_g, ln_b, gn_g, gn_b, a_out, act, fp16);             \
  else ln_res_gn_kernel<C, false><<<B, 256, 0, s>>>(p, x, ln_g, ln_b, gn_g, gn_b, a_out, act, fp16);                      \
  break;
  switch (C) {
    case 64: M0_LN_CASE(64)
    case 96: M0_LN_CASE(96)
    case 128: M0_LN_CASE(128)
    case 160: M0_LN_CASE(160)
    case 192: M0_LN_CASE(192)
    case 224: M0_LN_CASE(224)
    case 256: M0_LN_CASE(256)
    case 288: M0_LN_CASE(288)
    case 320: M0_LN_CASE(320)
    default: m0_set_error("ln_res_gn: unsupported channel count %d", C); return M0_ERR_ARG;
  }
#undef M0_LN_CASE
  return m0_check_launch("ln_res_gn");
}
int nn_nhwc_to_nchw_f32(const float* in, float* out, int B, int C, cudaStream_t s) {
  size_t total = (size_t)B * 64 * C;
  nhwc_to_nchw_f32_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(in, out, B, C);
  return m0_check_launch("nhwc_to_nchw_f32");
}

}  // namespace m0
