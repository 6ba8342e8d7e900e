// Host-side evaluator object shared by net_capi.cu (fp32 path, C ABI) and nn_tc_kernels.cu (bf16 path).
#pragma once
#include "nn.cuh"

struct m0_net {
  int device;
  m0_net_config cfg;
  m0_net_weights w;
  // workspace (fp32 activations, NHWC), grown on demand
  int ws_batch;
  float *x, *t1, *t2, *qkv;          // [B][64][C] x3, [B][64][3C]
  float *ph, *pf, *vh1, *vh2, *vf1, *vf2, *vg;  // head temporaries
  float *ssl_a, *ssl_b, *ssl_c;
  void* tc;                          // bf16 path state (nn_tc_kernels.cu)
};

namespace m0 {
int net_ws_reserve(::m0_net* n, int B);
int net_forward_heads_f32(::m0_net* n, int B, float* logits, float* values, cudaStream_t s);
// slot: 0 = bf16, 1 = fp16, 2 = fp8 (e4m3 tower convolutions, fp16 elsewhere)
int tc_net_prepare(::m0_net* net, int slot, cudaStream_t s);
int tc_net_forward(::m0_net* net, int slot, const float* d_planes, int B, float* d_logits, float* d_values, cudaStream_t s);
void tc_net_release(::m0_net* net);
}  // namespace m0
