// C-ABI of the search engine: creation / destruction of the device-resident game trees and the
// launch wrappers around the warp-per-game tree kernels (tree_kernels.cu).
#include "engine.cuh"
#include <new>
#include <string.h>

namespace m0 {
// kernels (tree_kernels.cu)
__global__ void reset_games_kernel(EngineView E, const int* games, int n_games);
__global__ void set_positions_kernel(EngineView E, const int* games, int n_games, const u64* root_pos, const u64* hist_pos,
                                     const u16* hist_moves, const int* hist_lens, int hist_stride);
__global__ void search_begin_kernel(EngineView E, float* planes, int* out_info, double* out_value);
__global__ void search_select_kernel(EngineView E, int batch_cap, int* sims_left, float* planes, unsigned long long rng_step);
__global__ void search_expand_backup_kernel(EngineView E, const float* logits, int logits_stride, const float* values);
__global__ void search_result_kernel(EngineView E, u16* out_moves, int* out_visits, double* out_child_q, double* out_prior,
                                     int* out_count, float* out_pi, double* out_root_q, int* out_root_n);
__global__ void search_add_dirichlet_kernel(EngineView E, const double* noise, const int* apply, unsigned long long rng_step);
// kernels (tree_multi_kernels.cu)
__global__ void search_select_multi_kernel(EngineView E, int batch_cap, int* sims_left);
__global__ void multi_scan_kernel(EngineView E);
__global__ void multi_encode_kernel(EngineView E, int g0, int g1, int row0, int mode, float* planes, int row_cap);
__global__ void search_expand_backup_multi_kernel(EngineView E, int g0, int g1, const float* logits, int logits_stride, const float* values,
                                                  int row0, int per_sample, int row_cap);
}  // namespace m0

using namespace m0;

#include "engine_host.cuh"

#define TRY(x)            \
  do {                    \
    int _r = (x);         \
    if (_r != M0_OK) return _r; \
  } while (0)

static int engine_alloc(m0_engine* e) {
  EngineView& v = e->v;
  const size_t G = v.G, N = (size_t)v.G * v.max_nodes, T = (size_t)v.G * v.tt_cap, D = (size_t)v.G * v.max_depth,
               H = (size_t)v.G * v.hist_cap;
  TRY(dev_alloc(e, &v.root_pos, G * POSITION_WORDS));
  TRY(dev_alloc(e, &v.root_key, G));
  TRY(dev_alloc(e, &v.root_ep_legal, G));
  TRY(dev_alloc(e, &v.root_node, G));
  TRY(dev_alloc(e, &v.active, G));
  TRY(dev_alloc(e, &v.hist_key, H));
  TRY(dev_alloc(e, &v.hist_irrev, H));
  TRY(dev_alloc(e, &v.hist_len, G));
  TRY(dev_alloc(e, &v.node_prior, N, false));
  TRY(dev_alloc(e, &v.node_w, N, false));
  TRY(dev_alloc(e, &v.node_q, N, false));
  TRY(dev_alloc(e, &v.node_n, N, false));
  TRY(dev_alloc(e, &v.node_first, N, false));
  TRY(dev_alloc(e, &v.node_creator, N, false));
  TRY(dev_alloc(e, &v.node_mv, N, false));
  TRY(dev_alloc(e, &v.node_nchild, N, false));
  TRY(dev_alloc(e, &v.node_count, G));
  TRY(dev_alloc(e, &v.tt_lo, T));
  TRY(dev_alloc(e, &v.tt_hi, T));
  TRY(dev_alloc(e, &v.tt_val, T, false));
  TRY(dev_alloc(e, &v.tt_count, G));
  TRY(dev_alloc(e, &v.path_node, D));
  TRY(dev_alloc(e, &v.path_key, D));
  TRY(dev_alloc(e, &v.path_irrev, D));
  TRY(dev_alloc(e, &v.path_len, G));
  TRY(dev_alloc(e, &v.leaf_pos, G * POSITION_WORDS));
  TRY(dev_alloc(e, &v.leaf_moves, G * MAX_MOVES));
  TRY(dev_alloc(e, &v.leaf_idx, G * MAX_MOVES));
  TRY(dev_alloc(e, &v.leaf_n, G));
  TRY(dev_alloc(e, &v.pend_node, G));
  TRY(dev_alloc(e, &v.pend_count, G));
  TRY(dev_alloc(e, &v.pend_flags, G));
  TRY(dev_alloc(e, &v.status, G));
  TRY(dev_alloc(e, &v.counters, (size_t)CTR_COUNT));
  TRY(dev_alloc(e, &v.jit_cursor, G));
  TRY(dev_alloc(e, &v.nrm_cursor, G));
  TRY(dev_alloc(e, &e->d_params, 1));
  e->cpuct_cap = v.max_depth + 1;
  TRY(dev_alloc(e, &e->d_cpuct, (size_t)e->cpuct_cap));
  v.params = e->d_params;
  v.cpuct = e->d_cpuct;
  return M0_OK;
}

extern "C" {

int m0_engine_destroy(m0_engine* e);

// One engine per GPU (not thread-safe; one host thread drives it).
// max_nodes: node slots per game; tt_capacity: transposition slots per game (rounded up to 2^k,
// 0 = 2 * max_nodes); max_depth: selection path cap; hist_cap: game-history entries kept per game.
int m0_engine_create(int device, int max_games, int max_nodes, int tt_capacity, int max_depth, int hist_cap, m0_engine** out) {
  if (!out || max_games <= 0 || max_nodes < 64 || max_depth < 8 || hist_cap < 0) {
    m0_set_error("m0_engine_create: invalid argument");
    return M0_ERR_ARG;
  }
  m0::DeviceGuard device_guard(device);
  M0_CUDA_TRY(device_guard.err);
  m0_engine* e = new (std::nothrow) m0_engine();
  if (!e) { m0_set_error("m0_engine_create: out of host memory"); return M0_ERR_ARG; }
  e->device = device;
  e->bytes = 0;
  e->rng_step = 0;
  memset(&e->v, 0, sizeof(e->v));
  memset(&e->sp, 0, sizeof(e->sp));
  e->d_sp_params = nullptr;
  e->sp_step = 0;
  e->finished_read = 0;
  e->v.G = max_games;
  e->v.max_nodes = max_nodes;
  e->v.tt_cap = next_pow2(tt_capacity > 0 ? tt_capacity : 2 * max_nodes);
  e->v.max_depth = max_depth;
  e->v.hist_cap = hist_cap > 0 ? hist_cap : 1;
  int rc = engine_alloc(e);
  if (rc != M0_OK) { m0_engine_destroy(e); return rc; }
  *out = e;
  return M0_OK;
}

int m0_engine_destroy(m0_engine* e) {
  if (!e) return M0_OK;
  m0::DeviceGuard device_guard(e->device);
  for (void* p : e->allocs) cudaFree(p);
  delete e;
  return M0_OK;
}

long long m0_engine_bytes(const m0_engine* e) { return e ? (long long)e->bytes : 0; }

int m0_engine_configure(m0_engine* e, const m0_search_config* c, void* stream) {
  if (!e || !c || c->cpuct_len <= 0 || !c->cpuct_by_depth) { m0_set_error("m0_engine_configure: invalid argument"); return M0_ERR_ARG; }
  m0::DeviceGuard device_guard(e->device);
  M0_CUDA_TRY(device_guard.err);
  SearchParams p;
  memset(&p, 0, sizeof(p));
  p.fpu_reduction = c->fpu_reduction;
  p.draw_penalty = c->draw_penalty;
  p.jitter = c->selection_jitter > 0 ? c->selection_jitter : 0.001;  // mcts.py:893-897
  p.dirichlet_alpha = c->dirichlet_alpha;
  p.dirichlet_frac = c->dirichlet_frac;
  p.jitter_on = c->deterministic ? 0 : 1;
  p.no_instant_backtrack = c->no_instant_backtrack;
  p.legal_softmax = c->legal_softmax;
  p.entropy_noise = c->deterministic ? 0 : c->enable_entropy_noise;
  p.value_from_white = c->value_from_white;
  int len = c->cpuct_len < e->cpuct_cap ? c->cpuct_len : e->cpuct_cap;
  p.cpuct_len = len;
  p.seed = c->seed;
  p.max_children = c->max_children > 0 ? c->max_children : 0;
  p.min_child_prior = c->min_child_prior > 0.0 ? c->min_child_prior : 0.0;
  p.raw_logit_priors = c->raw_logit_priors ? 1 : 0;
  p.virtual_loss = c->virtual_loss;
  p.virtual_loss_on = (c->virtual_loss_on && c->virtual_loss > 0.0) ? 1 : 0;
  if (p.entropy_noise && !p.legal_softmax && !e->v.full_scratch) {
    // noise over all 4672 entries of the full softmax (mcts.py:164-186): one float64 row of scratch per game
    TRY(dev_alloc(e, &e->v.full_scratch, (size_t)e->v.G * POLICY_SIZE, false));
  }
  cudaStream_t s = (cudaStream_t)stream;
  M0_CUDA_TRY(cudaMemcpyAsync(e->d_params, &p, sizeof(p), cudaMemcpyHostToDevice, s));
  M0_CUDA_TRY(cudaMemcpyAsync(e->d_cpuct, c->cpuct_by_depth, sizeof(double) * len, cudaMemcpyHostToDevice, s));
  M0_CUDA_TRY(cudaStreamSynchronize(s));  // the host struct may go away after return
  return M0_OK;
}

// MCTS.reset() (mcts.py:1477-1488) for a list of game slots (d_games == NULL: the first n slots)
int m0_games_reset(m0_engine* e, const int* d_games, int n, void* stream) {
  if (!e || n < 0 || n > e->v.G) { m0_set_error("m0_games_reset: invalid argument"); return M0_ERR_ARG; }
  if (n == 0) return M0_OK;
  int bx = (e->v.tt_cap + 1023) / 1024;
  if (bx > 64) bx = 64;
  dim3 grid(bx, n);
  reset_games_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(e->v, d_games, n);
  return m0_check_launch("m0_games_reset");
}

// Set root positions (packed uint64[n][9]) and optionally the move-stack history that precedes each
// root (positions uint64[n][hist_stride][9], moves uint16[n][hist_stride], lengths int32[n]); replaces the
// `board` argument of MCTS.run (mcts.py:318): board.copy() carries the move stack into the search (:558).
int m0_games_set_positions(m0_engine* e, const int* d_games, int n, const uint64_t* d_root_pos, const uint64_t* d_hist_pos,
                           const uint16_t* d_hist_moves, const int32_t* d_hist_lens, int hist_stride, void* stream) {
  if (!e || n < 0 || n > e->v.G || !d_root_pos) { m0_set_error("m0_games_set_positions: invalid argument"); return M0_ERR_ARG; }
  if (n == 0) return M0_OK;
  set_positions_kernel<<<n, 64, 0, (cudaStream_t)stream>>>(e->v, d_games, n, d_root_pos, d_hist_pos, d_hist_moves, d_hist_lens, hist_stride);
  return m0_check_launch("m0_games_set_positions");
}

// Current root position of every game (packed records uint64[G][9]): what selfplay_worker encodes as the training state
// before each search (internal.py:447) -- read back by the self-play recorder.
int m0_games_get_positions(m0_engine* e, uint64_t* d_out_pos, void* stream) {
  if (!e || !d_out_pos) { m0_set_error("m0_games_get_positions: invalid argument"); return M0_ERR_ARG; }
  return m0_check_cuda(cudaMemcpyAsync(d_out_pos, e->v.root_pos, (size_t)e->v.G * 9 * sizeof(uint64_t), cudaMemcpyDeviceToDevice, (cudaStream_t)stream),
                       "m0_games_get_positions");
}

static inline int tree_blocks(const m0_engine* e) { return (e->v.G + TREE_WARPS - 1) / TREE_WARPS; }

// MCTS.run prologue (mcts.py:336-371): d_info int32[G] (bit0 terminal root, bit1 needs evaluation),
// d_value float64[G] terminal value; d_planes float32[G][19][8][8] receives the roots to evaluate.
// With the store of m0_search_reuse_enable, a root found among the stored entries is expanded from that entry and the other roots
// are also written, in compact rows, to the miss buffer (the miss counter gives the row count).
int m0_search_begin(m0_engine* e, float* d_planes, int32_t* d_info, double* d_value, void* stream) {
  if (!e || !d_info || !d_value) { m0_set_error("m0_search_begin: invalid argument"); return M0_ERR_ARG; }
  if (e->v.rc_slots) M0_CUDA_TRY(cudaMemsetAsync(e->v.rc_miss_count, 0, sizeof(int), (cudaStream_t)stream));
  search_begin_kernel<<<tree_blocks(e), TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(e->v, d_planes, d_info, d_value);
  return m0_check_launch("m0_search_begin");
}

// One mini-batch of `batch_n` simulations per game (mcts.py:535-558): selection + immediate terminal backups;
// leaves needing the network are left pending and their planes written to d_planes[g].
int m0_search_select(m0_engine* e, int batch_n, float* d_planes, void* stream) {
  if (!e || batch_n <= 0) { m0_set_error("m0_search_select: invalid argument"); return M0_ERR_ARG; }
  e->rng_step += 1;
  search_select_kernel<<<tree_blocks(e), TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(e->v, batch_n, nullptr, d_planes, e->rng_step);
  return m0_check_launch("m0_search_select");
}

// Same with a per-game simulation budget: game g runs min(batch_cap, d_sims_left[g]) simulations and its budget is
// decremented (playout-cap randomisation gives every MCTS.run its own count, mcts.py:380-385).
int m0_search_select_var(m0_engine* e, int batch_cap, int32_t* d_sims_left, float* d_planes, void* stream) {
  if (!e || batch_cap <= 0 || !d_sims_left) { m0_set_error("m0_search_select_var: invalid argument"); return M0_ERR_ARG; }
  e->rng_step += 1;
  search_select_kernel<<<tree_blocks(e), TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(e->v, batch_cap, d_sims_left, d_planes, e->rng_step);
  return m0_check_launch("m0_search_select_var");
}

// Expansion (Node._expand, mcts.py:135-225), child registration (:1330-1346) and the owed backups
// (:946-953) for every pending leaf; d_logits float32[G][stride], d_values float32[G].
int m0_search_expand_backup(m0_engine* e, const float* d_logits, int logits_stride, const float* d_values, void* stream) {
  if (!e || !d_logits || !d_values || logits_stride < POLICY_SIZE) { m0_set_error("m0_search_expand_backup: invalid argument"); return M0_ERR_ARG; }
  search_expand_backup_kernel<<<tree_blocks(e), TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(e->v, d_logits, logits_stride, d_values);
  return m0_check_launch("m0_search_expand_backup");
}

// Root Dirichlet noise (mcts.py:955-992).  d_noise float64[G][256] or NULL (device RNG); d_apply int32[G] or NULL (all).
int m0_search_add_dirichlet(m0_engine* e, const double* d_noise, const int32_t* d_apply, void* stream) {
  if (!e) { m0_set_error("m0_search_add_dirichlet: invalid argument"); return M0_ERR_ARG; }
  e->rng_step += 1;
  search_add_dirichlet_kernel<<<tree_blocks(e), TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(e->v, d_noise, d_apply, e->rng_step);
  return m0_check_launch("m0_search_add_dirichlet");
}

// Pending-evaluation table of the current step: int32[G] multiplicities (0 = nothing pending)
int m0_search_pending(m0_engine* e, int32_t* d_counts_out, void* stream) {
  if (!e || !d_counts_out) { m0_set_error("m0_search_pending: invalid argument"); return M0_ERR_ARG; }
  M0_CUDA_TRY(cudaMemcpyAsync(d_counts_out, e->v.pend_flags, sizeof(int) * e->v.G, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return M0_OK;
}
int m0_search_pending_counts(m0_engine* e, int32_t* d_counts_out, void* stream) {
  if (!e || !d_counts_out) { m0_set_error("m0_search_pending_counts: invalid argument"); return M0_ERR_ARG; }
  M0_CUDA_TRY(cudaMemcpyAsync(d_counts_out, e->v.pend_count, sizeof(int) * e->v.G, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return M0_OK;
}

// visit_counts / policy / root value of MCTS.run (mcts.py:431, :465, :504-507)
int m0_search_result(m0_engine* e, uint16_t* d_moves, int32_t* d_visits, double* d_child_q, double* d_prior, int32_t* d_count,
                     float* d_pi, double* d_root_q, int32_t* d_root_n, void* stream) {
  if (!e || !d_moves || !d_visits || !d_count || !d_root_q || !d_root_n) { m0_set_error("m0_search_result: invalid argument"); return M0_ERR_ARG; }
  search_result_kernel<<<tree_blocks(e), TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(e->v, d_moves, d_visits, d_child_q, d_prior, d_count, d_pi, d_root_q, d_root_n);
  return m0_check_launch("m0_search_result");
}

// ---- the reference's mini-batch as shipped: per-simulation jitter, distinct leaves (tree_multi_kernels.cu) ---------------------
// Allocates the per-game sample / leaf tables for mini-batches of up to `samples_per_batch` simulations (inference_batch_size);
// virtual_loss != 0 also allocates the per-node in-flight counters of the virtual-loss mode (m0_search_config.virtual_loss_on).
int m0_search_multi_enable(m0_engine* e, int samples_per_batch, int virtual_loss) {
  if (!e || samples_per_batch <= 0 || samples_per_batch > 4096) { m0_set_error("m0_search_multi_enable: invalid argument"); return M0_ERR_ARG; }
  if (virtual_loss && !e->v.node_inflight) {
    m0::DeviceGuard device_guard(e->device);
    M0_CUDA_TRY(device_guard.err);
    TRY(dev_alloc(e, &e->v.node_inflight, (size_t)e->v.G * e->v.max_nodes));
  }
  if (e->v.ml_cap >= samples_per_batch) return M0_OK;
  if (e->v.ml_cap > 0) { m0_set_error("m0_search_multi_enable: already enabled with a smaller batch (%d)", e->v.ml_cap); return M0_ERR_STATE; }
  m0::DeviceGuard device_guard(e->device);
  M0_CUDA_TRY(device_guard.err);
  EngineView& v = e->v;
  const size_t G = v.G, S = G * (size_t)samples_per_batch;
  TRY(dev_alloc(e, &v.ml_n_samples, G));
  TRY(dev_alloc(e, &v.ml_n_leaves, G));
  TRY(dev_alloc(e, &v.ml_smp_leaf, S, false));
  TRY(dev_alloc(e, &v.ml_smp_len, S, false));
  TRY(dev_alloc(e, &v.ml_smp_path, S * (size_t)v.max_depth, false));
  TRY(dev_alloc(e, &v.ml_leaf_node, S, false));
  TRY(dev_alloc(e, &v.ml_leaf_first, S, false));
  TRY(dev_alloc(e, &v.ml_leaf_pos, S * POSITION_WORDS, false));
  TRY(dev_alloc(e, &v.ml_row_base, G + 1));
  v.ml_cap = samples_per_batch;
  return M0_OK;
}

// Random draws of the stochastic search.  d_jitter float64[G][jitter_stride]: the values random.random() returns, consumed one per
// child per visited node in selection order (mcts.py:893-897); d_normal float64[G][normal_stride]: the N(0, 0.1) variates of the
// entropy noise, k per noisy expansion in expansion order (mcts.py:181).  NULL selects the counter-based device generator.  Resets the
// per-game cursors; a game that runs past its stream sets status bit 16 and continues on the device generator.
int m0_search_set_streams(m0_engine* e, const double* d_jitter, long long jitter_stride, const double* d_normal, long long normal_stride, void* stream) {
  if (!e || (d_jitter && jitter_stride <= 0) || (d_normal && normal_stride <= 0)) { m0_set_error("m0_search_set_streams: invalid argument"); return M0_ERR_ARG; }
  e->v.jit_stream = d_jitter;
  e->v.jit_stride = d_jitter ? jitter_stride : 0;
  e->v.nrm_stream = d_normal;
  e->v.nrm_stride = d_normal ? normal_stride : 0;
  M0_CUDA_TRY(cudaMemsetAsync(e->v.jit_cursor, 0, sizeof(unsigned long long) * e->v.G, (cudaStream_t)stream));
  M0_CUDA_TRY(cudaMemsetAsync(e->v.nrm_cursor, 0, sizeof(unsigned long long) * e->v.G, (cudaStream_t)stream));
  return M0_OK;
}

// Collection of one mini-batch per game (mcts.py:535-558 + _collect_leaf_position :742-769): batch_n selections with per-simulation
// jitter, terminal leaves backed up immediately, the other samples recorded.  d_sims_left int32[G] (or NULL) as in m0_search_select_var.
// Afterwards the compact row numbering is computed; d_row_base int32[G + 1] (row_base[G] = total rows) and d_n_samples int32[G] receive
// copies when not NULL.
int m0_search_select_multi(m0_engine* e, int batch_n, int32_t* d_sims_left, int32_t* d_row_base, int32_t* d_n_samples, void* stream) {
  if (!e || batch_n <= 0) { m0_set_error("m0_search_select_multi: invalid argument"); return M0_ERR_ARG; }
  if (e->v.ml_cap < batch_n) { m0_set_error("m0_search_select_multi: call m0_search_multi_enable(%d) first", batch_n); return M0_ERR_STATE; }
  cudaStream_t s = (cudaStream_t)stream;
  search_select_multi_kernel<<<tree_blocks(e), TREE_WARPS * 32, 0, s>>>(e->v, batch_n, d_sims_left);
  TRY(m0_check_launch("m0_search_select_multi"));
  multi_scan_kernel<<<1, 1024, 0, s>>>(e->v);
  TRY(m0_check_launch("m0_search_select_multi(scan)"));
  if (d_row_base) M0_CUDA_TRY(cudaMemcpyAsync(d_row_base, e->v.ml_row_base, sizeof(int) * (e->v.G + 1), cudaMemcpyDeviceToDevice, s));
  if (d_n_samples) M0_CUDA_TRY(cudaMemcpyAsync(d_n_samples, e->v.ml_n_samples, sizeof(int) * e->v.G, cudaMemcpyDeviceToDevice, s));
  return M0_OK;
}

// row_cap > 0 (compact rows only): games whose rows do not end within row_cap rows of row0 are skipped by BOTH calls and keep their
// samples -- the host can launch an evaluator batch for "as many leading games as fit" before it has read the row numbering.
// encode_board of the collected leaves of games [g0, g1) (mcts.py:571-583).  mode 0: compact rows, row = row_base[g] + slot - row0;
// mode 1: dense per leaf, row = (g - g0) * samples_per_batch + slot; mode 2: one row per SAMPLE in collection order (duplicates
// repeated, as the reference's batch tensor holds them), row = (g - g0) * samples_per_batch + sample.
int m0_search_multi_encode(m0_engine* e, int g0, int g1, int row0, int mode, float* d_planes, int row_cap, void* stream) {
  if (!e || !d_planes || g0 < 0 || g1 > e->v.G || g0 >= g1 || e->v.ml_cap <= 0 || mode < 0 || mode > 2) { m0_set_error("m0_search_multi_encode: invalid argument"); return M0_ERR_ARG; }
  const long long warps = (long long)(g1 - g0) * e->v.ml_cap;
  multi_encode_kernel<<<(unsigned)((warps + TREE_WARPS - 1) / TREE_WARPS), TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(e->v, g0, g1, row0, mode, d_planes, mode == 0 ? row_cap : 0);
  return m0_check_launch("m0_search_multi_encode");
}

// Node._expand + _prune_children + _register_children_in_tt + _backpropagate for the samples of games [g0, g1) in collection order
// (mcts.py:654-670).  per_sample = 0: d_logits / d_values rows are the compact rows starting at row0 (one row per distinct leaf);
// per_sample = 1: one row per sample, game g's rows start at (g - g0) * samples_per_batch (mode 2 of m0_search_multi_encode).
int m0_search_expand_backup_multi(m0_engine* e, int g0, int g1, const float* d_logits, int logits_stride, const float* d_values, int row0,
                                  int per_sample, int row_cap, void* stream) {
  if (!e || !d_logits || !d_values || logits_stride < POLICY_SIZE || g0 < 0 || g1 > e->v.G || g0 >= g1 || e->v.ml_cap <= 0) {
    m0_set_error("m0_search_expand_backup_multi: invalid argument");
    return M0_ERR_ARG;
  }
  search_expand_backup_multi_kernel<<<(g1 - g0 + TREE_WARPS - 1) / TREE_WARPS, TREE_WARPS * 32, 0, (cudaStream_t)stream>>>(
      e->v, g0, g1, d_logits, logits_stride, d_values, row0, per_sample, per_sample ? 0 : row_cap);
  return m0_check_launch("m0_search_expand_backup_multi");
}

// ---- reuse of the root's evaluation across moves ------------------------------------------------------------------------------------
// Allocates a store of `slots` (1..64) entries per game: the expansion kernels keep the network output of every evaluated child of the
// root, and the next m0_search_begin expands a root whose packed position equals a stored one from that entry instead of asking for an
// evaluation.  Roots without an entry go to d_miss_planes float32[G][19][8][8] in compact rows, counted in d_miss_count int32[1]; the
// expansion then reads the evaluator's row r for the root written to row r.  The two caller buffers must stay alive.  The entries are
// the outputs of the network that produced them: m0_search_reuse_clear must be called when the evaluator changes.
int m0_search_reuse_enable(m0_engine* e, int slots, float* d_miss_planes, int32_t* d_miss_count) {
  if (!e || slots <= 0 || slots > REUSE_MAX_SLOTS || !d_miss_planes || !d_miss_count) { m0_set_error("m0_search_reuse_enable: invalid argument"); return M0_ERR_ARG; }
  if (e->v.rc_slots && e->v.rc_slots != slots) { m0_set_error("m0_search_reuse_enable: already enabled with %d slots", e->v.rc_slots); return M0_ERR_STATE; }
  EngineView& v = e->v;
  if (!v.rc_slots) {
    m0::DeviceGuard device_guard(e->device);
    M0_CUDA_TRY(device_guard.err);
    const size_t G = v.G, S = G * (size_t)slots;
    TRY(dev_alloc(e, &v.rc_fill, G));
    TRY(dev_alloc(e, &v.rc_pos, S * POSITION_WORDS, false));
    TRY(dev_alloc(e, &v.rc_logits, S * POLICY_SIZE, false));
    TRY(dev_alloc(e, &v.rc_value, S, false));
    TRY(dev_alloc(e, &v.rc_src, G, false));
    v.rc_slots = slots;
  }
  v.rc_miss_planes = d_miss_planes;
  v.rc_miss_count = d_miss_count;
  return M0_OK;
}

// Forgets every stored entry (the evaluator's weights changed, or a caller wants every root evaluated again).
int m0_search_reuse_clear(m0_engine* e, void* stream) {
  if (!e || !e->v.rc_slots) { m0_set_error("m0_search_reuse_clear: invalid argument (store not enabled)"); return M0_ERR_ARG; }
  return m0_check_cuda(cudaMemsetAsync(e->v.rc_fill, 0, sizeof(int) * e->v.G, (cudaStream_t)stream), "m0_search_reuse_clear");
}

// Engine counters (uint64[16], see engine.cuh CTR_*) and sticky per-game status bits (int32[G])
int m0_engine_counters(m0_engine* e, unsigned long long* h_out16) {
  if (!e || !h_out16) { m0_set_error("m0_engine_counters: invalid argument"); return M0_ERR_ARG; }
  M0_CUDA_TRY(cudaMemcpy(h_out16, e->v.counters, sizeof(unsigned long long) * CTR_COUNT, cudaMemcpyDeviceToHost));
  return M0_OK;
}
int m0_engine_status(m0_engine* e, int32_t* d_status_out, int32_t* d_node_count_out, void* stream) {
  if (!e) { m0_set_error("m0_engine_status: invalid argument"); return M0_ERR_ARG; }
  if (d_status_out) M0_CUDA_TRY(cudaMemcpyAsync(d_status_out, e->v.status, sizeof(int) * e->v.G, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  if (d_node_count_out) M0_CUDA_TRY(cudaMemcpyAsync(d_node_count_out, e->v.node_count, sizeof(int) * e->v.G, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return M0_OK;
}

}  // extern "C"
