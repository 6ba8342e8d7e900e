// C-ABI of the evaluator: PolicyValueNet.forward (azchess/model/resnet.py:755-760) as a sequence of
// CUDA kernel launches on the caller's stream.  precision 0 = fp32 SIMT path (parity within 1e-4),
// precision 1 / 2 = bf16 / fp16 tensor-core path, 3 = fp8 (fp16 with e4m3 tower convolutions) (nn_tc_kernels.cu).
#include "net_host.cuh"
#include <new>
#include <string.h>

using namespace m0;

#define TRY(x)            \
  do {                    \
    int _r = (x);         \
    if (_r != M0_OK) return _r; \
  } while (0)

static void ws_free(m0_net* n) {
  float** ptrs[] = {&n->x, &n->t1, &n->t2, &n->qkv, &n->ph, &n->pf, &n->vh1, &n->vh2, &n->vf1, &n->vf2, &n->vg, &n->ssl_a, &n->ssl_b, &n->ssl_c};
  for (float** p : ptrs) {
    if (*p) cudaFree(*p);
    *p = nullptr;
  }
  n->ws_batch = 0;
}

static int ws_reserve(m0_net* n, int B) {
  if (B <= n->ws_batch) return M0_OK;
  ws_free(n);
  const size_t C = n->cfg.channels, T = (size_t)B * 64;
  int rank = n->cfg.policy_factor_rank > 0 ? n->cfg.policy_factor_rank : 1;
  M0_CUDA_TRY(cudaMalloc(&n->x, T * C * 4));
  M0_CUDA_TRY(cudaMalloc(&n->t1, T * C * 4));
  M0_CUDA_TRY(cudaMalloc(&n->t2, T * C * 4));
  M0_CUDA_TRY(cudaMalloc(&n->qkv, T * 3 * C * 4));
  M0_CUDA_TRY(cudaMalloc(&n->ph, T * 64 * 4));
  M0_CUDA_TRY(cudaMalloc(&n->pf, (size_t)B * rank * 4));
  M0_CUDA_TRY(cudaMalloc(&n->vh1, T * 128 * 4));
  M0_CUDA_TRY(cudaMalloc(&n->vh2, T * 128 * 4));
  M0_CUDA_TRY(cudaMalloc(&n->vf1, (size_t)B * 2 * C * 4));
  M0_CUDA_TRY(cudaMalloc(&n->vf2, (size_t)B * C * 4));
  M0_CUDA_TRY(cudaMalloc(&n->vg, (size_t)B * C * 4));
  M0_CUDA_TRY(cudaMalloc(&n->ssl_a, T * (C / 2) * 4));
  M0_CUDA_TRY(cudaMalloc(&n->ssl_b, T * (C / 2) * 4));
  M0_CUDA_TRY(cudaMalloc(&n->ssl_c, T * 16 * 4));
  n->ws_batch = B;
  return M0_OK;
}

// x <- tower(features(stem(planes)))  (resnet.py:656-695, fp32)
static int forward_features_f32(m0_net* n, const float* planes, int B, cudaStream_t s) {
  const m0_net_config& c = n->cfg;
  const m0_net_weights& w = n->w;
  const int C = c.channels, M = B * 64, act = c.activation;
  // stem: conv3x3(planes -> C), GN, act ; chess features: + position encoding (resnet.py:229-231)
  TRY(nn_gemm_f32(A_IM2COL_NCHW, planes, w.stem_w, nullptr, nullptr, n->t1, M, C, 9 * c.planes, 0, C, c.planes, ACT_NONE, 1.0f, s));
  if (c.chess_features) {
    TRY(nn_groupnorm_f32(n->t1, w.stem_gn_w, w.stem_gn_b, w.pos_enc, 0, n->x, B, C, act, s));
    if (c.piece_square_tables) {  // x = x + act(GN(conv1x1(x)))  (resnet.py:233-236)
      TRY(nn_gemm_f32(A_DIRECT, n->x, w.pst_w, nullptr, nullptr, n->t1, M, C, C, C, C, C, ACT_NONE, 1.0f, s));
      TRY(nn_groupnorm_f32(n->t1, w.pst_gn_w, w.pst_gn_b, n->x, (long long)64 * C, n->t2, B, C, act, s));
    } else {
      M0_CUDA_TRY(cudaMemcpyAsync(n->t2, n->x, (size_t)M * C * 4, cudaMemcpyDeviceToDevice, s));
    }
    // x = x + act(GN(conv3x3(x)))  (resnet.py:238-242)
    TRY(nn_gemm_f32(A_IM2COL_NHWC, n->t2, w.inter_w, nullptr, nullptr, n->t1, M, C, 9 * C, 0, C, C, ACT_NONE, 1.0f, s));
    TRY(nn_groupnorm_f32(n->t1, w.inter_gn_w, w.inter_gn_b, n->t2, (long long)64 * C, n->x, B, C, act, s));
  } else {
    TRY(nn_groupnorm_f32(n->t1, w.stem_gn_w, w.stem_gn_b, nullptr, 0, n->x, B, C, act, s));
  }
  // tower (pre-activation residual blocks, resnet.py:44-51; attention stride at inference, :678-687)
  int att_seen = 0;
  const int stride = c.infer_attention_stride > 1 ? c.infer_attention_stride : 1;
  for (int i = 0; i < c.blocks; ++i) {
    const m0_block_weights& b = w.blocks[i];
    TRY(nn_groupnorm_f32(n->x, b.gn1_w, b.gn1_b, nullptr, 0, n->t1, B, C, act, s));
    TRY(nn_gemm_f32(A_IM2COL_NHWC, n->t1, b.conv1_w, nullptr, nullptr, n->t2, M, C, 9 * C, 0, C, C, ACT_NONE, 1.0f, s));
    TRY(nn_groupnorm_f32(n->t2, b.gn2_w, b.gn2_b, nullptr, 0, n->t1, B, C, act, s));
    TRY(nn_gemm_f32(A_IM2COL_NHWC, n->t1, b.conv2_w, nullptr, nullptr, n->t2, M, C, 9 * C, 0, C, C, ACT_NONE, 1.0f, s));
    TRY(nn_se_residual_f32(n->t2, n->x, b.se_w1, b.se_b1, b.se_w2, b.se_b2, n->x, B, C, c.se_hidden, act, c.se, s));
    if (b.has_attention) {
      att_seen++;
      if (att_seen % stride == 0) {
        TRY(nn_gemm_f32(A_DIRECT, n->x, b.att_qkv_w, nullptr, nullptr, n->qkv, M, 3 * C, C, C, 3 * C, C, ACT_NONE, 1.0f, s));
        TRY(nn_attention_f32(n->qkv, c.attention_relbias ? b.att_rel_bias : nullptr, n->t1, B, C, c.attention_heads, c.attention_unmasked_mix, s));
        TRY(nn_gemm_f32(A_DIRECT, n->t1, b.att_proj_w, nullptr, nullptr, n->t2, M, C, C, C, C, C, ACT_NONE, 1.0f, s));
        TRY(nn_layernorm_residual_f32(n->t2, n->x, b.att_ln_w, b.att_ln_b, n->x, M, C, s));
      }
    }
  }
  return M0_OK;
}

// policy / value heads (resnet.py:697-753)
static int forward_heads_f32(m0_net* n, int B, float* logits, float* values, cudaStream_t s) {
  const m0_net_config& c = n->cfg;
  const m0_net_weights& w = n->w;
  const int C = c.channels, M = B * 64, act = c.activation, vact = c.value_activation;
  // policy: conv1x1 C->64, GN, act, flatten, fc (factorised or dense), * logit scale
  TRY(nn_gemm_f32(A_DIRECT, n->x, w.pol_conv_w, nullptr, nullptr, n->t1, M, 64, C, C, 64, C, ACT_NONE, 1.0f, s));
  TRY(nn_groupnorm_f32(n->t1, w.pol_gn_w, w.pol_gn_b, nullptr, 0, n->ph, B, 64, act, s));
  if (c.policy_factor_rank > 0) {
    TRY(nn_gemm_f32(A_DIRECT, n->ph, w.pol_fc1_w, w.pol_fc1_b, nullptr, n->pf, B, c.policy_factor_rank, 4096, 4096, c.policy_factor_rank, 0, ACT_RELU, 1.0f, s));
    TRY(nn_gemm_f32(A_DIRECT, n->pf, w.pol_fc2_w, w.pol_fc2_b, nullptr, logits, B, c.policy_size, c.policy_factor_rank, c.policy_factor_rank, c.policy_size, 0, ACT_NONE, w.policy_logit_scale, s));
  } else {
    TRY(nn_gemm_f32(A_DIRECT, n->ph, w.pol_fc1_w, w.pol_fc1_b, nullptr, logits, B, c.policy_size, 4096, 4096, c.policy_size, 0, ACT_NONE, w.policy_logit_scale, s));
  }
  // value: conv1x1 C->128, GN, act, conv1x1 128->128, GN, act, flatten, fc1, fc2, gate, fc3, tanh
  TRY(nn_gemm_f32(A_DIRECT, n->x, w.val_conv1_w, nullptr, nullptr, n->vh1, M, 128, C, C, 128, C, ACT_NONE, 1.0f, s));
  TRY(nn_groupnorm_f32(n->vh1, w.val_gn1_w, w.val_gn1_b, nullptr, 0, n->vh2, B, 128, act, s));
  TRY(nn_gemm_f32(A_DIRECT, n->vh2, w.val_conv2_w, nullptr, nullptr, n->vh1, M, 128, 128, 128, 128, 128, ACT_NONE, 1.0f, s));
  TRY(nn_groupnorm_f32(n->vh1, w.val_gn2_w, w.val_gn2_b, nullptr, 0, n->vh2, B, 128, act, s));
  TRY(nn_gemm_f32(A_DIRECT, n->vh2, w.val_fc1_w, w.val_fc1_b, nullptr, n->vf1, B, 2 * C, 8192, 8192, 2 * C, 0, vact, 1.0f, s));
  TRY(nn_gemm_f32(A_DIRECT, n->vf1, w.val_fc2_w, w.val_fc2_b, nullptr, n->vf2, B, C, 2 * C, 2 * C, C, 0, vact, 1.0f, s));
  TRY(nn_gemm_f32(A_DIRECT, n->vf2, w.val_gate_w, w.val_gate_b, n->vf2, n->vg, B, C, C, C, C, 0, ACT_SIGMOID, 1.0f, s));
  TRY(nn_gemm_f32(A_DIRECT, n->vg, w.val_fc3_w, w.val_fc3_b, nullptr, values, B, 1, C, C, 1, 0, ACT_TANH, 1.0f, s));
  return M0_OK;
}

extern "C" {

int m0_net_destroy(m0_net* n);

int m0_net_create(int device, const m0_net_config* cfg, const m0_net_weights* weights, m0_net** out) {
  if (!cfg || !weights || !out) { m0_set_error("m0_net_create: null argument"); return M0_ERR_ARG; }
  if (cfg->blocks <= 0 || cfg->blocks > M0_MAX_BLOCKS || cfg->channels % 32 != 0 || cfg->channels > 1024 || cfg->policy_size != 4672 ||
      cfg->n_ssl_heads > M0_MAX_SSL_HEADS) {
    m0_set_error("m0_net_create: unsupported configuration (blocks=%d channels=%d policy=%d)", cfg->blocks, cfg->channels, cfg->policy_size);
    return M0_ERR_ARG;
  }
  m0::DeviceGuard device_guard(device);
  M0_CUDA_TRY(device_guard.err);
  m0_net* n = new (std::nothrow) m0_net();
  if (!n) { m0_set_error("m0_net_create: out of host memory"); return M0_ERR_ARG; }
  memset(n, 0, sizeof(*n));
  n->device = device;
  n->cfg = *cfg;
  n->w = *weights;
  *out = n;
  return M0_OK;
}

int m0_net_destroy(m0_net* n) {
  if (!n) return M0_OK;
  m0::DeviceGuard device_guard(n->device);
  ws_free(n);
  tc_net_release(n);
  delete n;
  return M0_OK;
}

// PolicyValueNet.forward(x) (resnet.py:755-760): d_planes float32[B][planes][8][8] -> d_logits float32[B][4672],
// d_values float32[B].  precision: 0 = fp32, 1 = bf16, 2 = fp16, 3 = fp8 tensor cores.
int m0_net_forward(m0_net* n, const float* d_planes, int B, float* d_logits, float* d_values, int precision, void* stream) {
  if (!n || !d_planes || !d_logits || !d_values || B < 0) { m0_set_error("m0_net_forward: invalid argument"); return M0_ERR_ARG; }
  if (B == 0) return M0_OK;
  cudaStream_t s = (cudaStream_t)stream;
  if (precision >= 1 && precision <= 3) {  // 1 = bf16, 2 = fp16 operands, 3 = fp16 with e4m3 tower convolutions (fp32 accumulate)
    nn_set_half_format(precision >= 2);
    TRY(tc_net_prepare(n, precision - 1, s));
    return tc_net_forward(n, precision - 1, d_planes, B, d_logits, d_values, s);
  }
  TRY(ws_reserve(n, B));
  TRY(forward_features_f32(n, d_planes, B, s));
  return forward_heads_f32(n, B, d_logits, d_values, s);
}

// forward(x, return_ssl=True) (resnet.py:736-745): additionally writes head h's output float32[B][k_h][8][8] (NCHW)
// to d_ssl_out[h] for every h with a non-null pointer.  fp32 path only (never used during search).
int m0_net_forward_ssl(m0_net* n, const float* d_planes, int B, float* d_logits, float* d_values, float* const* d_ssl_out, void* stream) {
  if (!n || !d_planes || !d_logits || !d_values || !d_ssl_out || B < 0) { m0_set_error("m0_net_forward_ssl: invalid argument"); return M0_ERR_ARG; }
  if (B == 0) return M0_OK;
  cudaStream_t s = (cudaStream_t)stream;
  TRY(ws_reserve(n, B));
  TRY(forward_features_f32(n, d_planes, B, s));
  TRY(forward_heads_f32(n, B, d_logits, d_values, s));
  const int C = n->cfg.channels, H = C / 2, M = B * 64;
  for (int h = 0; h < n->cfg.n_ssl_heads; ++h) {
    if (!d_ssl_out[h]) continue;
    const int k = n->cfg.ssl_out_channels[h];
    if (k > 16) { m0_set_error("m0_net_forward_ssl: head %d has %d > 16 channels", h, k); return M0_ERR_ARG; }
    TRY(nn_gemm_f32(A_DIRECT, n->x, n->w.ssl_conv1_w[h], nullptr, nullptr, n->ssl_a, M, H, C, C, H, C, ACT_NONE, 1.0f, s));
    TRY(nn_groupnorm_f32(n->ssl_a, n->w.ssl_gn_w[h], n->w.ssl_gn_b[h], nullptr, 0, n->ssl_b, B, H, n->cfg.activation, s));
    TRY(nn_gemm_f32(A_DIRECT, n->ssl_b, n->w.ssl_conv2_w[h], nullptr, nullptr, n->ssl_c, M, k, H, H, k, H, ACT_NONE, 1.0f, s));
    TRY(nn_nhwc_to_nchw_f32(n->ssl_c, d_ssl_out[h], B, k, s));
  }
  return M0_OK;
}

}  // extern "C"

// shared with the tensor-core path (nn_tc_kernels.cu)
namespace m0 {
int net_ws_reserve(::m0_net* n, int B) { return ws_reserve(n, B); }
int net_forward_heads_f32(::m0_net* n, int B, float* logits, float* values, cudaStream_t s) { return forward_heads_f32(n, B, logits, values, s); }
}  // namespace m0
