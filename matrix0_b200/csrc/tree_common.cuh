// Warp-cooperative building blocks shared by the tree kernels (tree_kernels.cu: one pending leaf per game and
// mini-batch; tree_multi_kernels.cu: the as-shipped stochastic mini-batches): sequential fp64 backups, the
// repetition test of a leaf, the random draws, and Node._expand with entropy noise and child pruning.
#pragma once
#include "engine.cuh"
#include "movegen_warp.cuh"

namespace m0 {

static constexpr int TREE_WARPS = 4;
static constexpr int TREE_THREADS = TREE_WARPS * 32;
static constexpr unsigned FULL = 0xFFFFFFFFu;

__device__ __forceinline__ double uniform01(u64 x) { return (double)(x >> 11) * (1.0 / 9007199254740992.0); }

// ---- random draws --------------------------------------------------------------------------------------
// random.random() of mcts.py:893-897 for child `j` of the node being scanned; `cur` = draws this game consumed so far
__device__ __forceinline__ double draw_jitter_uniform(const EngineView& E, const SearchParams& P, int g, unsigned long long cur, int j) {
  const unsigned long long at = cur + (unsigned long long)j;
  if (E.jit_stream && at < (unsigned long long)E.jit_stride) return E.jit_stream[(size_t)g * E.jit_stride + at];
  return uniform01(mix64(P.seed ^ mix64(0xA24BAED4963EE407ull * (u64)(g + 1)) ^ mix64(at + 0x9E3779B97F4A7C15ull)));
}
// np.random.normal(0, 0.1) of mcts.py:181 for entry `j` of the expansion that starts at draw `cur`
__device__ __forceinline__ double draw_noise_normal(const EngineView& E, const SearchParams& P, int g, unsigned long long cur, int j) {
  const unsigned long long at = cur + (unsigned long long)j;
  if (E.nrm_stream && at < (unsigned long long)E.nrm_stride) return E.nrm_stream[(size_t)g * E.nrm_stride + at];
  u64 a = mix64(P.seed ^ mix64(0x9FB21C651E98DF25ull * (u64)(g + 1)) ^ mix64(2 * at + 0x632BE59BD9B4E019ull));
  u64 b = mix64(a + 0x9E3779B97F4A7C15ull);
  // Box-Muller in single precision (the variates only have to be N(0, 0.1)-distributed: 24-bit uniforms, fast intrinsics)
  const float u1 = ((float)(a >> 40) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)(b >> 40) * (1.0f / 16777216.0f);
  return (double)(0.1f * (sqrtf(-2.0f * __logf(u1)) * __cosf(6.2831853f * u2)));
}

// ---- backup: azchess/mcts.py:946-953, `times` identical backprops of value v_leaf along `path` -------------
__device__ __forceinline__ void warp_backup_path(const EngineView& E, int g, const int* path, int len, double v_leaf, int times, int lane) {
  const size_t nb = (size_t)g * E.max_nodes;
  // a node can occur twice in a path (transposition back to an ancestor): then the sequential
  // interleaving of the reference matters and one lane replays it literally
  bool dup = false;
  for (int i = lane; i < len; i += 32) {
    int a = path[i];
    for (int j = 0; j < i; ++j) dup |= (path[j] == a);
  }
  dup = __any_sync(FULL, dup);
  if (!dup) {
    for (int i = lane; i < len; i += 32) {
      int node = path[i];
      double v = ((len - 1 - i) & 1) ? -v_leaf : v_leaf;
      int n = E.node_n[nb + node];
      double w = E.node_w[nb + node], q;
      backup_repeated(n, w, q, v, times);
      E.node_n[nb + node] = n;
      E.node_w[nb + node] = w;
      E.node_q[nb + node] = q;
    }
  } else if (lane == 0) {
    for (int t = 0; t < times; ++t) {
      double v = v_leaf;
      for (int i = len - 1; i >= 0; --i) {
        int node = path[i];
        int n = E.node_n[nb + node] + 1;
        double w = d_add(E.node_w[nb + node], v);
        E.node_n[nb + node] = n;
        E.node_w[nb + node] = w;
        E.node_q[nb + node] = d_div(w, (double)n);
        v = -v;
      }
    }
  }
  __syncwarp();
}
__device__ __forceinline__ void warp_backup(const EngineView& E, int g, int len, double v_leaf, int times, int lane) {
  warp_backup_path(E, g, E.path_node + (size_t)g * E.max_depth, len, v_leaf, times, lane);
}

// chess.Board.is_repetition(5) for the leaf: occurrences of the leaf key among the positions since
// the last irreversible move, walking the search path and then the game history backwards
__device__ __forceinline__ bool leaf_is_fivefold(const EngineView& E, int g, int depth, const Key128& cur) {
  int count = 0;
  const Key128* pk = E.path_key + (size_t)g * E.max_depth;
  const u8* pi = E.path_irrev + (size_t)g * E.max_depth;
  for (int d = depth - 1; d >= 0; --d) {
    if (pi[d]) return false;
    if (key_eq(pk[d], cur) && ++count >= 4) return true;
  }
  const Key128* hk = E.hist_key + (size_t)g * E.hist_cap;
  const u8* hi = E.hist_irrev + (size_t)g * E.hist_cap;
  for (int i = E.hist_len[g] - 1; i >= 0; --i) {
    if (hi[i]) return false;
    if (key_eq(hk[i], cur) && ++count >= 4) return true;
  }
  return false;
}

// board.is_game_over() of a position reached by the search (mcts.py:747 / :336) and, for a live one, its legal moves in
// python-chess order in `s_moves`.  Returns the move count; *terminal_value is set when the position is terminal
// (_terminal_value, mcts.py:1223-1229).  depth / key: place on the search path for the repetition test.
__device__ __forceinline__ int warp_leaf_moves(const EngineView& E, const SearchParams& P, int g, const Position& pos, int depth, const Key128& key,
                                               u16* s_moves, bool* terminal, double* terminal_value, int lane) {
  int in_check = 0;
  int n_moves = warp_generate_legal_moves(pos, s_moves, &in_check, lane);   // one own piece per lane, python-chess order
  if (n_moves > MAX_MOVES) n_moves = MAX_MOVES;
  bool term = n_moves == 0 || is_insufficient_material(pos) || (pos_halfmove(pos) >= 150 && n_moves > 0);
  if (!term && pos_halfmove(pos) >= 8) {
    int rep = 0;
    if (lane == 0) rep = leaf_is_fivefold(E, g, depth, key) ? 1 : 0;
    term = __shfl_sync(FULL, rep, 0) != 0;
  }
  *terminal = term;
  *terminal_value = (n_moves == 0 && in_check) ? -1.0 : P.draw_penalty;
  __syncwarp();
  return n_moves;
}

// ---- Node._expand (mcts.py:135-225) + _prune_children (:806-826) + _register_children_in_tt (:1330-1346) ----
struct ExpandSmem {
  float p[MAX_MOVES];      // priors
  Key128 key[MAX_MOVES];   // child keys; before that: scratch for the entropy terms (float) and the noisy distribution (double)
  u16 ord[MAX_MOVES];      // child order after pruning
};

// Expands `node` (not expanded yet) at `pos` with legal moves mvs[0..k) / policy indices idx[0..k) from the logits row `lg`.
// reg: register the children in the transposition table; is_root: the expansion MCTS.run does itself (never the Q3 shortcut).
__device__ __forceinline__ void warp_expand(const EngineView& E, const SearchParams& P, int g, int node, const Position& pos, const u16* mvs,
                                            const u16* idx, int k, const float* __restrict__ lg, bool reg, bool is_root, ExpandSmem& S, int lane) {
  const size_t nb = (size_t)g * E.max_nodes;
  float* s_p = S.p;
  const float uniform = (float)(1.0 / (double)k);
  if (P.raw_logit_priors && !is_root && P.legal_softmax) {
    // SURVEY Q3, the direct-model path: pri = p_logits[idxs]; pri / float(pri.sum()) unless the sum is non-finite or <= 0
    for (int j = lane; j < k; j += 32) s_p[j] = lg[idx[j]];
    __syncwarp();
    float total = 0.0f;
    if (lane == 0) total = np_pairwise_sum_f32(s_p, k);
    total = __shfl_sync(FULL, total, 0);
    if (isfinite(total) && total > 0.0f) {
      for (int j = lane; j < k; j += 32) s_p[j] = f_div(s_p[j], total);
    } else {
      for (int j = lane; j < k; j += 32) s_p[j] = uniform;
    }
  } else {
    // np.any(np.isnan(logits)) or np.any(np.isinf(logits)) over the whole vector (mcts.py:147)
    // (an exponent field of all ones; 16-byte loads, four in flight per lane: the row is 18.7 KB of streaming reads)
    bool bad = false;
    if ((reinterpret_cast<uintptr_t>(lg) & 15) == 0) {
      const uint4* lg4 = reinterpret_cast<const uint4*>(lg);
      u32 acc = 0;
#pragma unroll 4
      for (int i = lane; i < POLICY_SIZE / 4; i += 32) {
        const uint4 v = __ldg(lg4 + i);
        acc |= (u32)((v.x & 0x7F800000u) == 0x7F800000u) | (u32)((v.y & 0x7F800000u) == 0x7F800000u) |
               (u32)((v.z & 0x7F800000u) == 0x7F800000u) | (u32)((v.w & 0x7F800000u) == 0x7F800000u);
      }
      bad = acc != 0;
    } else {
      for (int i = lane; i < POLICY_SIZE; i += 32) bad |= !isfinite(lg[i]);
    }
    bad = __any_sync(FULL, bad);
    if (bad) {
      for (int j = lane; j < k; j += 32) s_p[j] = uniform;
    } else {
      float mx = -INFINITY;
      if (P.legal_softmax) {
        for (int j = lane; j < k; j += 32) mx = fmaxf(mx, lg[idx[j]]);
      } else {
        for (int i = lane; i < POLICY_SIZE; i += 32) mx = fmaxf(mx, lg[i]);
      }
      for (int off = 16; off > 0; off >>= 1) mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, off));
      float sum = 0.0f;
      if (P.legal_softmax) {
        for (int j = lane; j < k; j += 32) {
          float e = expf(f_sub(lg[idx[j]], mx));
          s_p[j] = e;
          sum = f_add(sum, e);
        }
      } else {
        for (int i = lane; i < POLICY_SIZE; i += 32) sum = f_add(sum, expf(f_sub(lg[i], mx)));
        for (int j = lane; j < k; j += 32) s_p[j] = expf(f_sub(lg[idx[j]], mx));
      }
      for (int off = 16; off > 0; off >>= 1) sum = f_add(sum, __shfl_xor_sync(FULL, sum, off));
      __syncwarp();
      for (int j = lane; j < k; j += 32) s_p[j] = f_div(s_p[j], sum);   // dist (legal_only) / dist[idx] (full softmax)
      __syncwarp();
      if (P.entropy_noise && !P.legal_softmax && E.full_scratch) {
        // mcts.py:164-186 on the FULL distribution: entropy over all 4672 entries against log(k), N(0, 0.1) on every entry, floor,
        // renormalise over all 4672; the priors are then read at the legal indices.  Scratch: one float64 row per game in global memory.
        double* d = E.full_scratch + (size_t)g * POLICY_SIZE;
        float* t = reinterpret_cast<float*>(d);
        for (int i = lane; i < POLICY_SIZE; i += 32) {
          const float pi = f_div(expf(f_sub(lg[i], mx)), sum);
          t[i] = f_mul(pi, logf(f_add(pi, 1e-8f)));
        }
        __syncwarp();
        int noisy = 0;
        if (lane == 0) {
          const float ent = -np_pairwise_sum_f32_big(t, POLICY_SIZE);
          const double hmax = log((double)(k > 1 ? k : 1));
          noisy = d_div((double)ent, hmax > 1e-9 ? hmax : 1e-9) > 0.9 ? 1 : 0;
        }
        noisy = __shfl_sync(FULL, noisy, 0);
        __syncwarp();
        if (noisy) {
          const unsigned long long cur = E.nrm_cursor[g];
          if (E.nrm_stream && cur + (unsigned long long)POLICY_SIZE > (unsigned long long)E.nrm_stride && lane == 0) E.status[g] |= ST_STREAM_EXHAUSTED;
          for (int i = POLICY_SIZE - 1 - lane; i >= 0; i -= 32) {   // descending: the float32 terms in the low half of the row are dead by now
            const float pi = f_div(expf(f_sub(lg[i], mx)), sum);
            const double x = d_add((double)pi, draw_noise_normal(E, P, g, cur, i));
            d[i] = x > 1e-8 ? x : (x != x ? x : 1e-8);
          }
          __syncwarp();
          double tot = 0.0;
          if (lane == 0) {
            tot = np_pairwise_sum_f64_big(d, POLICY_SIZE);
            E.nrm_cursor[g] = cur + (unsigned long long)POLICY_SIZE;
            atomicAdd(&E.counters[CTR_NOISY_EXPANSIONS], 1ull);
          }
          tot = __shfl_sync(FULL, tot, 0);
          for (int j = lane; j < k; j += 32) s_p[j] = (float)d_div(d[idx[j]], tot);
          __syncwarp();
        }
      }
      if (P.entropy_noise && P.legal_softmax) {
        // mcts.py:170-186 on the active (legal-only) distribution: H = -sum(dist * log(dist + 1e-8)) in float32,
        // ratio = H / max(1e-9, log(k)) in float64; above 0.9: dist + N(0, 0.1) in float64, floor 1e-8, renormalise
        float* t = reinterpret_cast<float*>(S.key);
        for (int j = lane; j < k; j += 32) t[j] = f_mul(s_p[j], logf(f_add(s_p[j], 1e-8f)));
        __syncwarp();
        int noisy = 0;
        if (lane == 0) {
          const float ent = -np_pairwise_sum_f32(t, k);
          const double hmax = log((double)(k > 1 ? k : 1));
          noisy = d_div((double)ent, hmax > 1e-9 ? hmax : 1e-9) > 0.9 ? 1 : 0;
        }
        noisy = __shfl_sync(FULL, noisy, 0);
        __syncwarp();
        if (noisy) {
          double* d = reinterpret_cast<double*>(S.key);
          const unsigned long long cur = E.nrm_cursor[g];
          if (E.nrm_stream && cur + (unsigned long long)k > (unsigned long long)E.nrm_stride && lane == 0) E.status[g] |= ST_STREAM_EXHAUSTED;
          for (int j = lane; j < k; j += 32) {
            double x = d_add((double)s_p[j], draw_noise_normal(E, P, g, cur, j));
            d[j] = x > 1e-8 ? x : (x != x ? x : 1e-8);   // np.maximum propagates NaN
          }
          __syncwarp();
          double tot = 0.0;
          if (lane == 0) {
            tot = np_pairwise_sum_f64(d, k);
            E.nrm_cursor[g] = cur + (unsigned long long)k;
            atomicAdd(&E.counters[CTR_NOISY_EXPANSIONS], 1ull);
          }
          tot = __shfl_sync(FULL, tot, 0);
          for (int j = lane; j < k; j += 32) s_p[j] = (float)d_div(d[j], tot);   // float(dist[i]) -> np.float32 array
          __syncwarp();
        }
      }
      for (int j = lane; j < k; j += 32) {
        float p = s_p[j];
        if (!(p >= 0.0f) || isinf(p)) p = 0.0f;  // mcts.py:198-199
        s_p[j] = p;
      }
      __syncwarp();
      float total = 0.0f;
      if (lane == 0) total = np_pairwise_sum_f32(s_p, k);  // lp.sum(), mcts.py:206
      total = __shfl_sync(FULL, total, 0);
      if (total > 0.0f && isfinite(total)) {
        for (int j = lane; j < k; j += 32) s_p[j] = f_div(s_p[j], total);  // mcts.py:210
      } else {
        for (int j = lane; j < k; j += 32) s_p[j] = uniform;
      }
    }
  }
  __syncwarp();
  // _prune_children (mcts.py:806-826): drop priors below min_child_prior, then keep the max_children largest priors
  // (stable descending sort, so the kept children are re-ordered by prior when the cut applies); no renormalisation
  int kk = k;
  const bool prune = P.min_child_prior > 0.0 || (P.max_children > 0 && k > P.max_children);
  if (prune) {
    if (lane == 0) {
      int m = 0;
      for (int j = 0; j < k; ++j)
        if (!(P.min_child_prior > 0.0) || (double)s_p[j] >= P.min_child_prior) S.ord[m++] = (u16)j;
      if (P.max_children > 0 && m > P.max_children) {
        for (int a = 1; a < m; ++a) {   // stable insertion sort, descending prior
          const u16 x = S.ord[a];
          const float px = s_p[x];
          int b = a - 1;
          while (b >= 0 && s_p[S.ord[b]] < px) { S.ord[b + 1] = S.ord[b]; --b; }
          S.ord[b + 1] = x;
        }
        m = P.max_children;
      }
      kk = m;
    }
    kk = __shfl_sync(FULL, kk, 0);
    __syncwarp();
  }
  int first = 0;
  if (lane == 0) {
    first = E.node_count[g];
    if (first + kk > E.max_nodes) {
      E.status[g] |= ST_NODE_OVERFLOW;
      first = -1;
    } else {
      E.node_count[g] = first + kk;
    }
  }
  first = __shfl_sync(FULL, first, 0);
  if (first < 0) return;
  // child.q = -self.parent.q when the expanding node's creator has q != 0 (mcts.py:221-222)
  const int creator = E.node_creator[nb + node];
  double q0 = 0.0;
  if (creator >= 0) {
    double cq = E.node_q[nb + creator];
    if (cq != 0.0) q0 = -cq;
  }
  // the priors leave shared memory before the key scratch (which aliases the noise scratch) is written
  float pr[MAX_MOVES / 32];
  int src[MAX_MOVES / 32];
#pragma unroll
  for (int t = 0; t < MAX_MOVES / 32; ++t) {
    const int j = lane + 32 * t;
    src[t] = j < kk ? (prune ? (int)S.ord[j] : j) : 0;
    pr[t] = j < kk ? s_p[src[t]] : 0.0f;
  }
  __syncwarp();
#pragma unroll
  for (int t = 0; t < MAX_MOVES / 32; ++t) {
    const int j = lane + 32 * t;
    if (j >= kk) continue;
    const size_t c = nb + first + j;
    const u16 mv = mvs[src[t]];
    E.node_prior[c] = (double)pr[t];
    E.node_w[c] = 0.0;
    E.node_q[c] = q0;
    E.node_n[c] = 0;
    E.node_first[c] = -1;
    E.node_creator[c] = node;
    E.node_mv[c] = (u32)mv | ((u32)idx[src[t]] << 16);
    E.node_nchild[c] = 0;
    if (reg) {
      // self.tt[key] = child for every child (mcts.py:1330-1346).  The children of one node are different positions, so the
      // lanes insert concurrently; "last writer wins" only orders EQUAL keys, i.e. this expansion against earlier ones
      Position cp = pos;
      push_move(cp, mv);
      tt_put_concurrent(E, g, position_key(cp), first + j);
    }
  }
  __syncwarp();
  if (lane == 0) {
    E.node_first[nb + node] = first;
    E.node_nchild[nb + node] = (u16)kk;
    atomicAdd(&E.counters[CTR_EXPANSIONS], 1ull);
    atomicAdd(&E.counters[CTR_CHILDREN_CREATED], (unsigned long long)kk);
  }
  __syncwarp();
}

// Keeps the network output of a child of the root (a leaf at path length 2) for the next move's root (EngineView::rc_*): the
// logits row, the value as the network returned it and the packed position.  A full store records nothing more; the next root is
// then evaluated again, which gives the same result.
__device__ __forceinline__ void warp_record_root_child(const EngineView& E, int g, const u64* pos_words, const float* __restrict__ lg,
                                                       float value, int lane) {
  const int n = E.rc_fill[g];
  if (n >= E.rc_slots) return;
  const size_t e = (size_t)g * E.rc_slots + n;
  float* dst = E.rc_logits + e * POLICY_SIZE;
  if ((reinterpret_cast<uintptr_t>(lg) & 15) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(lg);
    float4* d4 = reinterpret_cast<float4*>(dst);
#pragma unroll 4
    for (int i = lane; i < POLICY_SIZE / 4; i += 32) d4[i] = __ldg(s4 + i);
  } else {
    for (int i = lane; i < POLICY_SIZE; i += 32) dst[i] = lg[i];
  }
  if (lane < POSITION_WORDS) E.rc_pos[e * POSITION_WORDS + lane] = pos_words[lane];
  __syncwarp();
  if (lane == 0) {
    E.rc_value[e] = value;
    E.rc_fill[g] = n + 1;
  }
  __syncwarp();
}

}  // namespace m0
