// Memory-bound glue kernels of the tensor-core forward, fused so that the residual stream is read and
// written once per residual block.
#include "nn.cuh"
#include <cuda_fp16.h>
#include <cuda_fp8.h>

namespace m0 {

__device__ __forceinline__ float fk_act(float x, int act) {
  switch (act) {
    case ACT_RELU: return x > 0.0f ? x : 0.0f;
    case ACT_SILU: return __fdividef(x, 1.0f + __expf(-x));
    default: return x;
  }
}
__device__ __forceinline__ __nv_bfloat16 fk_half(float x, int fp16) {
  if (fp16) {
    __half h = __float2half_rn(x);
    return *reinterpret_cast<__nv_bfloat16*>(&h);
  }
  return __float2bfloat16(x);
}

// x_new = x + conv_out * gate   (SE excitation + residual add, resnet.py:68-80)
// a_out = half(act(GroupNorm(x_new)))   (bn1 + activation of the NEXT pre-activation block, resnet.py:46-47), or half(x_new) when
// gamma is null, or nothing when a_out is null.  conv_out is the 16-bit output of conv2 (operand format).  fp16 = 2 (precision fp8):
// 16-bit values are fp16 and the GroupNorm'ed a_out is e4m3 (the operand of the next e4m3 conv1).
// One block per board, C threads.  Thread (rg, q) owns 8 consecutive channels of 8 rows: every access is 16 bytes wide (8 halves or
// one of two float4), x and conv_out are read once, x_new / a_out written once.  GroupNorm statistics: 2 adjacent threads (= 16
// channels) x 8 row groups per group.
__device__ __forceinline__ void unpack_half8(const uint4& u, int fp16, float (&f)[8]) {
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    if (fp16) {
      const float2 t = __half22float2(*reinterpret_cast<const __half2*>(&w[i]));
      f[2 * i] = t.x; f[2 * i + 1] = t.y;
    } else {
      const float2 t = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&w[i]));
      f[2 * i] = t.x; f[2 * i + 1] = t.y;
    }
  }
}
__device__ __forceinline__ uint32_t fk_pack2(float a, float b, int fp16) {
  if (fp16) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}

__device__ __forceinline__ uint32_t fk_e4m3x4(float a, float b, float c, float d) {
  const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
  const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
  return lo | (hi << 16);
}

__global__ void __launch_bounds__(320, 2)
se_apply_gn_kernel(const __nv_bfloat16* __restrict__ conv_out, const float* __restrict__ gate, float* __restrict__ x,
                   const float* __restrict__ gamma, const float* __restrict__ beta, __nv_bfloat16* __restrict__ a_out, int C, int act, int fp16) {
  __shared__ float s_part[8][40][2];
  const int b = blockIdx.x;
  const int nq = C >> 3;                       // 8-channel columns (<= 40)
  const int q = threadIdx.x % nq, rg = threadIdx.x / nq;   // rg < 8 when blockDim == C
  const size_t base = (size_t)b * 64 * C + (size_t)rg * 8 * C + 8 * q;
  float v[8][8];
  if (conv_out) {
    float e[8];
    if (gate) {
      const float4 e0 = *reinterpret_cast<const float4*>(gate + (size_t)b * C + 8 * q);
      const float4 e1 = *reinterpret_cast<const float4*>(gate + (size_t)b * C + 8 * q + 4);
      e[0] = e0.x; e[1] = e0.y; e[2] = e0.z; e[3] = e0.w; e[4] = e1.x; e[5] = e1.y; e[6] = e1.z; e[7] = e1.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) e[j] = 1.0f;
    }
    uint4 cv[8];
#pragma unroll
    for (int r = 0; r < 8; ++r) cv[r] = __ldg(reinterpret_cast<const uint4*>(conv_out + base + (size_t)r * C));
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const float4 x0 = *reinterpret_cast<const float4*>(x + base + (size_t)r * C);
      const float4 x1 = *reinterpret_cast<const float4*>(x + base + (size_t)r * C + 4);
      float c[8];
      unpack_half8(cv[r], fp16, c);
      v[r][0] = fmaf(c[0], e[0], x0.x); v[r][1] = fmaf(c[1], e[1], x0.y); v[r][2] = fmaf(c[2], e[2], x0.z); v[r][3] = fmaf(c[3], e[3], x0.w);
      v[r][4] = fmaf(c[4], e[4], x1.x); v[r][5] = fmaf(c[5], e[5], x1.y); v[r][6] = fmaf(c[6], e[6], x1.z); v[r][7] = fmaf(c[7], e[7], x1.w);
    }
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      *reinterpret_cast<float4*>(x + base + (size_t)r * C) = make_float4(v[r][0], v[r][1], v[r][2], v[r][3]);
      *reinterpret_cast<float4*>(x + base + (size_t)r * C + 4) = make_float4(v[r][4], v[r][5], v[r][6], v[r][7]);
    }
  } else {   // plain GroupNorm of x: nothing to add, nothing to write back
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      const float4 x0 = *reinterpret_cast<const float4*>(x + base + (size_t)r * C);
      const float4 x1 = *reinterpret_cast<const float4*>(x + base + (size_t)r * C + 4);
      v[r][0] = x0.x; v[r][1] = x0.y; v[r][2] = x0.z; v[r][3] = x0.w; v[r][4] = x1.x; v[r][5] = x1.y; v[r][6] = x1.z; v[r][7] = x1.w;
    }
  }
  if (!a_out) return;
  __nv_bfloat16* ao = a_out + base;
  if (!gamma) {  // the next consumer is the attention qkv GEMM: it takes the raw residual stream in half precision
#pragma unroll
    for (int r = 0; r < 8; ++r)
      *reinterpret_cast<uint4*>(ao + (size_t)r * C) = make_uint4(fk_pack2(v[r][0], v[r][1], fp16), fk_pack2(v[r][2], v[r][3], fp16),
                                                                 fk_pack2(v[r][4], v[r][5], fp16), fk_pack2(v[r][6], v[r][7], fp16));
    return;
  }
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < 8; ++r) s += ((v[r][0] + v[r][1]) + (v[r][2] + v[r][3])) + ((v[r][4] + v[r][5]) + (v[r][6] + v[r][7]));
  s += __shfl_xor_sync(0xFFFFFFFFu, s, 1);   // 2 adjacent threads = one group of 16 channels (C/8 is even: pairs never straddle a warp)
  s_part[rg][q][0] = s;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int g = 0; g < 8; ++g) tot += s_part[g][q][0];
  const float mean = tot * (1.0f / 1024.0f);
  float d2 = 0.f;
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float a = v[r][j] - mean;
      d2 = fmaf(a, a, d2);
    }
  d2 += __shfl_xor_sync(0xFFFFFFFFu, d2, 1);
  s_part[rg][q][1] = d2;
  __syncthreads();
  float vs = 0.f;
#pragma unroll
  for (int g = 0; g < 8; ++g) vs += s_part[g][q][1];
  const float rstd = rsqrtf(vs * (1.0f / 1024.0f) + 1e-5f);
  float gsc[8], bsh[8];
  {
    const float4 g0 = *reinterpret_cast<const float4*>(gamma + 8 * q), g1 = *reinterpret_cast<const float4*>(gamma + 8 * q + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(beta + 8 * q), b1 = *reinterpret_cast<const float4*>(beta + 8 * q + 4);
    const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) { gsc[j] = gg[j] * rstd; bsh[j] = bb[j] - mean * gsc[j]; }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    float y[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) y[j] = fk_act(fmaf(v[r][j], gsc[j], bsh[j]), act);
    if (fp16 == 2) {
      *reinterpret_cast<uint2*>(reinterpret_cast<uint8_t*>(a_out) + base + (size_t)r * C) = make_uint2(fk_e4m3x4(y[0], y[1], y[2], y[3]), fk_e4m3x4(y[4], y[5], y[6], y[7]));
      continue;
    }
    *reinterpret_cast<uint4*>(ao + (size_t)r * C) =
        make_uint4(fk_pack2(y[0], y[1], fp16), fk_pack2(y[2], y[3], fp16), fk_pack2(y[4], y[5], fp16), fk_pack2(y[6], y[7], fp16));
  }
}

// out = act(GroupNorm_16ch(x)) + residual (residual optional; residual_bstride = 0 broadcasts one board, e.g. the positional
// encoding), written as fp32 and / or 16-bit.  Same thread layout as se_apply_gn_kernel: one block per board, C threads, thread
// (rg, q) owns 8 channels x 8 rows in registers, so x is read once with 16-byte loads (stem / piece-square / interaction / head
// normalisations of the tensor-core forward, resnet.py:18-24).
__global__ void __launch_bounds__(320, 2)
gn_act_res_kernel(const float* __restrict__ x, const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ residual,
                  long long residual_bstride, float* __restrict__ out, __nv_bfloat16* __restrict__ out_half, int C, int act, int fp16) {
  __shared__ float s_part[8][40][2];
  const int b = blockIdx.x;
  const int nq = C >> 3;
  const int q = threadIdx.x % nq, rg = threadIdx.x / nq;
  const size_t off = (size_t)rg * 8 * C + 8 * q;
  const size_t base = (size_t)b * 64 * C + off;
  float v[8][8];
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const float4 x0 = *reinterpret_cast<const float4*>(x + base + (size_t)r * C);
    const float4 x1 = *reinterpret_cast<const float4*>(x + base + (size_t)r * C + 4);
    v[r][0] = x0.x; v[r][1] = x0.y; v[r][2] = x0.z; v[r][3] = x0.w; v[r][4] = x1.x; v[r][5] = x1.y; v[r][6] = x1.z; v[r][7] = x1.w;
  }
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < 8; ++r) s += ((v[r][0] + v[r][1]) + (v[r][2] + v[r][3])) + ((v[r][4] + v[r][5]) + (v[r][6] + v[r][7]));
  s += __shfl_xor_sync(0xFFFFFFFFu, s, 1);
  s_part[rg][q][0] = s;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int g = 0; g < 8; ++g) tot += s_part[g][q][0];
  const float mean = tot * (1.0f / 1024.0f);
  float d2 = 0.f;
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float a = v[r][j] - mean;
      d2 = fmaf(a, a, d2);
    }
  d2 += __shfl_xor_sync(0xFFFFFFFFu, d2, 1);
  s_part[rg][q][1] = d2;
  __syncthreads();
  float vs = 0.f;
#pragma unroll
  for (int g = 0; g < 8; ++g) vs += s_part[g][q][1];
  const float rstd = rsqrtf(vs * (1.0f / 1024.0f) + 1e-5f);
  float gsc[8], bsh[8];
  {
    const float4 g0 = *reinterpret_cast<const float4*>(gamma + 8 * q), g1 = *reinterpret_cast<const float4*>(gamma + 8 * q + 4);
    const float4 b0 = *reinterpret_cast<const float4*>(beta + 8 * q), b1 = *reinterpret_cast<const float4*>(beta + 8 * q + 4);
    const float gg[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
    const float bb[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
    for (int j = 0; j < 8; ++j) { gsc[j] = gg[j] * rstd; bsh[j] = bb[j] - mean * gsc[j]; }
  }
  const float* rb = residual ? residual + (size_t)b * residual_bstride + off : nullptr;
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    float y[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) y[j] = fk_act(fmaf(v[r][j], gsc[j], bsh[j]), act);
    if (rb) {
      const float4 r0 = *reinterpret_cast<const float4*>(rb + (size_t)r * C), r1 = *reinterpret_cast<const float4*>(rb + (size_t)r * C + 4);
      y[0] += r0.x; y[1] += r0.y; y[2] += r0.z; y[3] += r0.w; y[4] += r1.x; y[5] += r1.y; y[6] += r1.z; y[7] += r1.w;
    }
    if (out) {
      *reinterpret_cast<float4*>(out + base + (size_t)r * C) = make_float4(y[0], y[1], y[2], y[3]);
      *reinterpret_cast<float4*>(out + base + (size_t)r * C + 4) = make_float4(y[4], y[5], y[6], y[7]);
    }
    if (out_half)
      *reinterpret_cast<uint4*>(out_half + base + (size_t)r * C) =
          make_uint4(fk_pack2(y[0], y[1], fp16), fk_pack2(y[2], y[3], fp16), fk_pack2(y[4], y[5], fp16), fk_pack2(y[6], y[7], fp16));
  }
}

// NCHW float32 planes [B][P][8][8] -> NHWC half [B][64][64] with channels P..63 zero (stem input of the tensor-core path)
__global__ void planes_to_nhwc_half_kernel(const float* __restrict__ planes, __nv_bfloat16* __restrict__ out, int B, int P, int fp16) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // over B*64*64
  if (i >= (size_t)B * 64 * 64) return;
  const int c = (int)(i & 63);
  const int sq = (int)((i >> 6) & 63);
  const size_t b = i >> 12;
  out[i] = c < P ? fk_half(planes[(b * P + c) * 64 + sq], fp16) : fk_half(0.0f, fp16);
}

// SE excitation for 16 boards per block (resnet.py:61-64): s = avgpool, h = act(W1 s + b1), gate = sigmoid(W2 h + b2).
// pool: half-board column sums [B][2][C]; w1t [C][hid] and w2t [hid][C] are transposed so that threads read them coalesced.
// Both layers keep 16 board accumulators per thread, so every weight is loaded once per block and the loads of consecutive
// iterations are independent (unrolled: the kernel is latency-bound, not bandwidth-bound).
__global__ void __launch_bounds__(320)
se_gate_kernel(const float* __restrict__ pool, const float* __restrict__ w1t, const float* __restrict__ b1, const float* __restrict__ w2t,
               const float* __restrict__ b2, float* __restrict__ gate, int B, int C, int hid, int act) {
  extern __shared__ float sm[];
  float* s_pool = sm;                      // [C][16]   (board index fastest: one 64-byte broadcast row per channel)
  float* s_hid = sm + 16 * C;              // [hid][16]
  float* s_red = s_hid + 16 * hid;         // [4][hid][16] partial sums of layer 1
  const int b0 = blockIdx.x * 16, t = threadIdx.x;
  const int nb = min(16, B - b0);
  for (int i = t; i < 16 * C; i += blockDim.x) {
    const int j = i / C, c = i - j * C;
    float v = 0.f;
    if (j < nb) {
      const float* pp = pool + (size_t)(b0 + j) * 2 * C;
      v = (pp[c] + pp[C + c]) * (1.0f / 64.0f);
    }
    s_pool[c * 16 + j] = v;
  }
  __syncthreads();
  // layer 1: thread (part, u) accumulates channels [part*C/4, (part+1)*C/4) of hidden unit u for the 16 boards
  {
    const int parts = blockDim.x / hid;        // 4 when blockDim = 320, hid = 80
    const int part = t / hid, u = t - part * hid;
    if (part < parts) {
      float h[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) h[j] = 0.f;
      const int c0 = part * (C / parts), c1 = (part + 1 == parts) ? C : c0 + C / parts;
#pragma unroll 16
      for (int c = c0; c < c1; ++c) {   // 16 independent weight loads in flight: the loop is bound by L2 latency
        const float w = __ldg(w1t + c * hid + u);
        const float4* sp = reinterpret_cast<const float4*>(s_pool + c * 16);
        const float4 p0 = sp[0], p1 = sp[1], p2 = sp[2], p3 = sp[3];
        h[0] = fmaf(w, p0.x, h[0]); h[1] = fmaf(w, p0.y, h[1]); h[2] = fmaf(w, p0.z, h[2]); h[3] = fmaf(w, p0.w, h[3]);
        h[4] = fmaf(w, p1.x, h[4]); h[5] = fmaf(w, p1.y, h[5]); h[6] = fmaf(w, p1.z, h[6]); h[7] = fmaf(w, p1.w, h[7]);
        h[8] = fmaf(w, p2.x, h[8]); h[9] = fmaf(w, p2.y, h[9]); h[10] = fmaf(w, p2.z, h[10]); h[11] = fmaf(w, p2.w, h[11]);
        h[12] = fmaf(w, p3.x, h[12]); h[13] = fmaf(w, p3.y, h[13]); h[14] = fmaf(w, p3.z, h[14]); h[15] = fmaf(w, p3.w, h[15]);
      }
      float4* dst = reinterpret_cast<float4*>(s_red + (part * hid + u) * 16);
      dst[0] = make_float4(h[0], h[1], h[2], h[3]); dst[1] = make_float4(h[4], h[5], h[6], h[7]);
      dst[2] = make_float4(h[8], h[9], h[10], h[11]); dst[3] = make_float4(h[12], h[13], h[14], h[15]);
    }
    __syncthreads();
    for (int o = t; o < hid * 16; o += blockDim.x) {
      const int u2 = o >> 4;
      float a = b1[u2];
      for (int pp = 0; pp < parts; ++pp) a += s_red[pp * hid * 16 + o];
      s_hid[o] = fk_act(a, act);
    }
    __syncthreads();
  }
  for (int c = t; c < C; c += blockDim.x) {
    float z[16];
    const float bias = b2[c];
#pragma unroll
    for (int j = 0; j < 16; ++j) z[j] = bias;
#pragma unroll 16
    for (int u = 0; u < hid; ++u) {
      const float w = __ldg(w2t + u * C + c);
      const float4* sh = reinterpret_cast<const float4*>(s_hid + u * 16);
      const float4 p0 = sh[0], p1 = sh[1], p2 = sh[2], p3 = sh[3];
      z[0] = fmaf(w, p0.x, z[0]); z[1] = fmaf(w, p0.y, z[1]); z[2] = fmaf(w, p0.z, z[2]); z[3] = fmaf(w, p0.w, z[3]);
      z[4] = fmaf(w, p1.x, z[4]); z[5] = fmaf(w, p1.y, z[5]); z[6] = fmaf(w, p1.z, z[6]); z[7] = fmaf(w, p1.w, z[7]);
      z[8] = fmaf(w, p2.x, z[8]); z[9] = fmaf(w, p2.y, z[9]); z[10] = fmaf(w, p2.z, z[10]); z[11] = fmaf(w, p2.w, z[11]);
      z[12] = fmaf(w, p3.x, z[12]); z[13] = fmaf(w, p3.y, z[13]); z[14] = fmaf(w, p3.z, z[14]); z[15] = fmaf(w, p3.w, z[15]);
    }
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (j < nb) gate[(size_t)(b0 + j) * C + c] = __fdividef(1.0f, 1.0f + __expf(-z[j]));
  }
}

int nn_se_gate(const float* pool, const float* w1t, const float* b1, const float* w2t, const float* b2, float* gate, int B, int C, int hid, int act,
               cudaStream_t s) {
  if (hid <= 0 || hid > 320 || C > 320) { m0_set_error("se_gate: unsupported shape C = %d, hidden width %d", C, hid); return M0_ERR_ARG; }
  const int parts = 320 / hid;
  const size_t smem = (size_t)16 * (C + hid + (size_t)parts * hid) * sizeof(float);
  if (smem > 48 * 1024) {
    // past the 48 KB default (C = 320 with hid > 256 needs up to 60 KB): grant the largest need of any supported shape, once per device,
    // so that no net lowers the limit under another
    static unsigned long long granted = 0;   // bit d: device d's kernel has the grant
    int dev = 0;
    cudaGetDevice(&dev);
    if (dev >= 64 || !((granted >> dev) & 1ull)) {
      const int most = 16 * (320 + 320 + 320) * (int)sizeof(float);
      cudaError_t e = cudaFuncSetAttribute(se_gate_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, most);
      if (e != cudaSuccess) { m0_set_error("se_gate: cannot reserve %d bytes of shared memory (%s)", most, cudaGetErrorString(e)); return M0_ERR_CUDA; }
      if (dev < 64) granted |= 1ull << dev;
    }
  }
  se_gate_kernel<<<(B + 15) / 16, 320, smem, s>>>(pool, w1t, b1, w2t, b2, gate, B, C, hid, act);
  return m0_check_launch("se_gate");
}

int nn_se_apply_gn(const __nv_bfloat16* conv_out, const float* gate, float* x, const float* gamma, const float* beta, __nv_bfloat16* a_out, int B,
                   int C, int act, cudaStream_t s, bool a_e4m3) {
  if (C > 320 || C % 32 != 0) { m0_set_error("se_apply_gn: unsupported channel count %d", C); return M0_ERR_ARG; }
  if (C % 16 != 0) { m0_set_error("se_apply_gn: channels must be a multiple of 16"); return M0_ERR_ARG; }
  se_apply_gn_kernel<<<B, C, 0, s>>>(conv_out, gate, x, gamma, beta, a_out, C, act, a_e4m3 ? 2 : nn_half_format());
  return m0_check_launch("se_apply_gn");
}
int nn_gn_act_res(const float* x, const float* gamma, const float* beta, const float* residual, long long residual_bstride, float* out,
                  __nv_bfloat16* out_half, int B, int C, int act, cudaStream_t s) {
  if (C > 320 || C % 16 != 0) { m0_set_error("gn_act_res: unsupported channel count %d", C); return M0_ERR_ARG; }
  if (act != ACT_NONE && act != ACT_RELU && act != ACT_SILU) { m0_set_error("gn_act_res: unsupported activation %d", act); return M0_ERR_ARG; }
  gn_act_res_kernel<<<B, C, 0, s>>>(x, gamma, beta, residual, residual_bstride, out, out_half, C, act, nn_half_format());
  return m0_check_launch("gn_act_res");
}
// hidden[b][u] = half(act(sum_ks part[ks][b][u] + b1[u])) for u < hid: reduction of the split-K partial sums of the first SE layer
__global__ void se_hidden_kernel(const float* __restrict__ part, int splits, long long split_stride, const float* __restrict__ b1,
                                 __nv_bfloat16* __restrict__ hidden, int B, int hid, int ld, int act, int fp16) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= B * hid) return;
  const int b = i / hid, u = i - b * hid;
  float a = b1[u];
  for (int ks = 0; ks < splits; ++ks) a += part[(size_t)ks * split_stride + (size_t)b * ld + u];
  hidden[(size_t)b * ld + u] = fk_half(fk_act(a, act), fp16);
}
int nn_se_hidden(const float* part, int splits, long long split_stride, const float* b1, __nv_bfloat16* hidden, int B, int hid, int ld, int act,
                 cudaStream_t s) {
  se_hidden_kernel<<<(B * hid + 255) / 256, 256, 0, s>>>(part, splits, split_stride, b1, hidden, B, hid, ld, act, nn_half_format());
  return m0_check_launch("se_hidden");
}
// The tail of the SE excitation in one launch (resnet.py:62-64): hidden = act(sum of the split-K partial sums of the first layer + b1),
// gate = sigmoid(W2 hidden + b2).  Eight boards per block; the hidden vectors live in shared memory, thread = output channel, W2 is read
// transposed ([hid][C]: coalesced across the threads, L1 / L2 resident: 102 KB).  The two tiny tensor-core launches it replaces
// (reduction kernel + a [B x 128] x [128 x 320] GEMM) cost 9 + 25 us of mostly fixed overhead per block.
static constexpr int SE_TAIL_BOARDS = 8;
__global__ void __launch_bounds__(320, 4)   // 4 blocks of 320 threads per SM: the 512 blocks of a 4096-board batch are one wave on 148 SMs
se_tail_kernel(const float* __restrict__ part, int splits, long long split_stride, int ld, const float* __restrict__ b1,
                               const float* __restrict__ w2t, const float* __restrict__ b2, float* __restrict__ gate, int B, int C, int hid, int act) {
  extern __shared__ __align__(16) float s_hid[];   // [hid][SE_TAIL_BOARDS]: the eight boards' values of one hidden unit are two 16-byte reads
  const int b0 = blockIdx.x * SE_TAIL_BOARDS;
  const int nb = min(SE_TAIL_BOARDS, B - b0);
  for (int i = threadIdx.x; i < SE_TAIL_BOARDS * hid; i += blockDim.x) {
    const int b = i / hid, u = i - b * hid;
    float a = 0.f;
    if (b < nb) {
      a = b1[u];
      for (int ks = 0; ks < splits; ++ks) a += part[(size_t)ks * split_stride + (size_t)(b0 + b) * ld + u];
      a = fk_act(a, act);
    }
    s_hid[u * SE_TAIL_BOARDS + b] = a;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    float acc[SE_TAIL_BOARDS];
#pragma unroll
    for (int b = 0; b < SE_TAIL_BOARDS; ++b) acc[b] = 0.f;
    for (int u0 = 0; u0 < hid; u0 += 16) {     // sixteen weight loads in flight per thread, then the arithmetic
      float w[16];
#pragma unroll
      for (int k = 0; k < 16; ++k) w[k] = (u0 + k < hid) ? __ldg(w2t + (size_t)(u0 + k) * C + c) : 0.f;
#pragma unroll
      for (int k = 0; k < 16; ++k) {
        if (u0 + k >= hid) break;
        const float4 h0 = *reinterpret_cast<const float4*>(s_hid + (u0 + k) * SE_TAIL_BOARDS);
        const float4 h1 = *reinterpret_cast<const float4*>(s_hid + (u0 + k) * SE_TAIL_BOARDS + 4);
        acc[0] = fmaf(w[k], h0.x, acc[0]); acc[1] = fmaf(w[k], h0.y, acc[1]); acc[2] = fmaf(w[k], h0.z, acc[2]); acc[3] = fmaf(w[k], h0.w, acc[3]);
        acc[4] = fmaf(w[k], h1.x, acc[4]); acc[5] = fmaf(w[k], h1.y, acc[5]); acc[6] = fmaf(w[k], h1.z, acc[6]); acc[7] = fmaf(w[k], h1.w, acc[7]);
      }
    }
    const float bias = b2[c];
#pragma unroll
    for (int b = 0; b < SE_TAIL_BOARDS; ++b)
      if (b < nb) gate[(size_t)(b0 + b) * C + c] = __fdividef(1.0f, 1.0f + __expf(-(acc[b] + bias)));
  }
}
int nn_se_tail(const float* part, int splits, long long split_stride, int ld, const float* b1, const float* w2t, const float* b2, float* gate, int B,
               int C, int hid, int act, cudaStream_t s) {
  const int threads = C >= 320 ? 320 : ((C + 31) / 32 * 32);
  se_tail_kernel<<<(B + SE_TAIL_BOARDS - 1) / SE_TAIL_BOARDS, threads, (size_t)SE_TAIL_BOARDS * hid * sizeof(float), s>>>(
      part, splits, split_stride, ld, b1, w2t, b2, gate, B, C, hid, act);
  return m0_check_launch("se_tail");
}
// value = tanh(value_fc3(h * gate)) (resnet.py:750-753): one warp per board, h = value_fc2 output, gate = sigmoid(value_gate(h))
__global__ void value_tail_kernel(const float* __restrict__ gate, const float* __restrict__ h, const float* __restrict__ w3, const float* __restrict__ b3,
                                  float* __restrict__ values, int B, int C) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  float acc = 0.f;
  for (int c = lane; c < C; c += 32) acc = fmaf(w3[c], h[(size_t)b * C + c] * gate[(size_t)b * C + c], acc);
  for (int off = 16; off > 0; off >>= 1) acc += __shfl_xor_sync(0xFFFFFFFFu, acc, off);
  if (lane == 0) values[b] = tanhf(acc + b3[0]);
}
int nn_value_tail(const float* gate, const float* h, const float* w3, const float* b3, float* values, int B, int C, cudaStream_t s) {
  value_tail_kernel<<<(B + 7) / 8, 256, 0, s>>>(gate, h, w3, b3, values, B, C);
  return m0_check_launch("value_tail");
}
int nn_planes_to_nhwc_half(const float* planes, __nv_bfloat16* out, int B, int P, cudaStream_t s) {
  const size_t total = (size_t)B * 64 * 64;
  planes_to_nhwc_half_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(planes, out, B, P, nn_half_format());
  return m0_check_launch("planes_to_nhwc_half");
}

}  // namespace m0
