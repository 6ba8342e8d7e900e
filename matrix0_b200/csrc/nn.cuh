// PolicyValueNet inference (azchess/model/resnet.py) -- shared declarations of the CUDA evaluator.
#pragma once
#include <cuda_bf16.h>
#include "m0_common.cuh"

namespace m0 {
int nn_groupnorm_mixed(const float* x, const float* gamma, const float* beta, const float* residual, long long residual_bstride,
                       float* out, __nv_bfloat16* out_bf16, int B, int C, int act, cudaStream_t s);
int nn_f32_to_bf16(const float* in, __nv_bfloat16* out, size_t n, cudaStream_t s);
void nn_set_half_format(int fp16);  // 0 = bf16, 1 = fp16 storage for the 16-bit tensor-core operands
int nn_half_format();

enum { ACT_NONE = 0, ACT_RELU = 1, ACT_SILU = 2, ACT_LEAKY = 3, ACT_TANH = 4, ACT_SIGMOID = 5 };
enum { A_DIRECT = 0, A_IM2COL_NHWC = 1, A_IM2COL_NCHW = 2 };

// fp32 path (nn_f32_kernels.cu)
int nn_gemm_f32(int mode, const float* A, const float* W, const float* bias, const float* mul, float* C, int M, int N, int K,
                int lda, int ldc, int cin, int act, float scale, cudaStream_t s);
int nn_groupnorm_f32(const float* x, const float* gamma, const float* beta, const float* residual, long long residual_bstride,
                     float* out, int B, int C, int act, cudaStream_t s);
int nn_se_residual_f32(const float* conv_out, const float* x, const float* w1, const float* b1, const float* w2, const float* b2,
                       float* x_out, int B, int C, int hidden, int act, int use_se, cudaStream_t s);
int nn_attention_f32(const float* qkv, const float* rel_bias, float* out, int B, int C, int heads, float unmasked_mix, cudaStream_t s);
int nn_layernorm_residual_f32(const float* proj, const float* x, const float* gamma, const float* beta, float* out, int tokens, int C,
                              cudaStream_t s);
int nn_nhwc_to_nchw_f32(const float* in, float* out, int B, int C, cudaStream_t s);
int nn_ln_res_gn(const void* proj, int proj_half, float* x, const float* ln_g, const float* ln_b, const float* gn_g, const float* gn_b,
                 __nv_bfloat16* a_out, int B, int C, int act, cudaStream_t s, bool a_e4m3 = false);

}  // namespace m0

// ---- C-ABI structs (include/matrix0_b200.h) ------------------------------------------------------------------
#define M0_MAX_BLOCKS 64
#define M0_MAX_SSL_HEADS 8

// NetConfig subset (resnet.py:247-282) that shapes the inference forward
struct m0_net_config {
  int planes, channels, blocks, policy_size;
  int se, se_hidden;
  int attention, attention_heads, attention_every_k, attention_relbias, infer_attention_stride;
  float attention_unmasked_mix;
  int policy_factor_rank;
  int activation;        // ACT_RELU | ACT_SILU          (cfg.activation)
  int value_activation;  // ACT_RELU | ACT_SILU | ACT_LEAKY (cfg.value_activation)
  int chess_features, piece_square_tables;
  int n_ssl_heads;
  int ssl_out_channels[M0_MAX_SSL_HEADS];
};

// All pointers are DEVICE pointers to contiguous float32 tensors owned by the caller, already in
// the kernel layouts: conv / linear weights as W[n][k] with k = (ky*3+kx)*Cin + ci for 3x3
// kernels; fc weights that consume a flattened NCHW map have their columns permuted to NHWC order.
struct m0_block_weights {
  const float *gn1_w, *gn1_b, *conv1_w, *gn2_w, *gn2_b, *conv2_w;
  const float *se_w1, *se_b1, *se_w2, *se_b2;
  int has_attention;  // a ChessAttention module follows this block in the tower
  const float *att_qkv_w, *att_proj_w, *att_ln_w, *att_ln_b, *att_rel_bias;
};

struct m0_net_weights {
  const float *stem_w, *stem_gn_w, *stem_gn_b;
  const float *pos_enc, *pst_w, *pst_gn_w, *pst_gn_b, *inter_w, *inter_gn_w, *inter_gn_b;
  m0_block_weights blocks[M0_MAX_BLOCKS];
  const float *pol_conv_w, *pol_gn_w, *pol_gn_b, *pol_fc1_w, *pol_fc1_b, *pol_fc2_w, *pol_fc2_b;
  float policy_logit_scale;  // clamp(softplus(raw) + 1e-3, max=5), resnet.py:709-710 (evaluated by the caller)
  const float *val_conv1_w, *val_gn1_w, *val_gn1_b, *val_conv2_w, *val_gn2_w, *val_gn2_b;
  const float *val_fc1_w, *val_fc1_b, *val_fc2_w, *val_fc2_b, *val_gate_w, *val_gate_b, *val_fc3_w, *val_fc3_b;
  const float *ssl_conv1_w[M0_MAX_SSL_HEADS], *ssl_gn_w[M0_MAX_SSL_HEADS], *ssl_gn_b[M0_MAX_SSL_HEADS], *ssl_conv2_w[M0_MAX_SSL_HEADS];
};
