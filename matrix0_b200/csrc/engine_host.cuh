// Host-side engine object shared by the C-ABI translation units.
#pragma once
#include "engine.cuh"
#include "selfplay.cuh"
#include <vector>

using namespace m0;

// Host-side mirror of MCTSConfig fields the device needs (include/matrix0_b200.h: m0_search_config)
struct m0_search_config {
  double fpu_reduction, draw_penalty, selection_jitter, dirichlet_alpha, dirichlet_frac;
  int deterministic;  // 1 = parity mode: jitter term is exactly zero, no noise
  int no_instant_backtrack, legal_softmax, enable_entropy_noise, value_from_white;
  int cpuct_len;
  unsigned long long seed;
  const double* cpuct_by_depth;  // host pointer, cpuct_len entries (mcts.py:927-944 evaluated per depth)
  int max_children;              // _prune_children (mcts.py:806-826), 0 = off
  int raw_logit_priors;          // SURVEY Q3 switch: the direct-model path's _expand_with_legal_priors(logits[idx]) for non-root leaves
  double min_child_prior;        // 0 = off
  double virtual_loss;           // MCTSConfig.virtual_loss (mcts.py:75)
  int virtual_loss_on;           // 1 = apply the reference's in-flight marking inside a mini-batch (its own callers never do, SURVEY Q2b)
  int reserved;
};

struct m0_engine {
  int device;
  EngineView v;
  std::vector<void*> allocs;
  SearchParams* d_params;
  double* d_cpuct;
  int cpuct_cap;
  unsigned long long rng_step;
  size_t bytes;
  m0::SelfPlayState sp;        // self-play game-loop state (selfplay_kernels.cu)
  m0::SelfPlayParams* d_sp_params;
  unsigned long long sp_step;
  unsigned finished_read;
  m0::GumbelView gb;           // Gumbel search state (gumbel_kernels.cu); gb.logit == NULL until m0_gumbel_configure
  unsigned long long gb_step;  // expansion calls so far: keys the device Gumbel draws
};

static constexpr int TREE_WARPS = 4;

template <typename T>
static int dev_alloc(m0_engine* e, T** p, size_t count, bool zero = true) {
  void* q = nullptr;
  size_t bytes = count * sizeof(T);
  if (bytes == 0) bytes = sizeof(T);
  M0_CUDA_TRY(cudaMalloc(&q, bytes));
  if (zero) M0_CUDA_TRY(cudaMemset(q, 0, bytes));
  e->allocs.push_back(q);
  e->bytes += bytes;
  *p = (T*)q;
  return M0_OK;
}

static int next_pow2(int x) {
  int p = 1;
  while (p < x) p <<= 1;
  return p;
}

