// Gumbel AlphaZero search for batched self-play (Danihelka et al., "Policy improvement by planning with Gumbel", ICLR 2022), one
// warp per game as in tree_kernels.cu.  DESIGN.md §9 states the algorithm; oracle/gumbel_ref.py restates it in float64 for the tests.
//
// A move: m0_search_begin (root planes) -> evaluator -> gumbel_expand_backup (root: children, r, Gumbel draws, N = 1, W = r)
//         -> n x [gumbel_select (one leaf per game) -> evaluator -> gumbel_expand_backup] -> gumbel_result.
// The tree is plain: children occupy consecutive node slots and are reached only through their parent (no transposition hops).
// Every node keeps N and W (EngineView::node_n / node_w) from the view of its side to move; the value of child a for its parent
// is q(a) = -W(a) / N(a).  Terminal leaves are never expanded: every visit re-derives their value and backs it up at once.
#include "tree_common.cuh"

namespace m0 {

static constexpr int GB_T = MAX_MOVES / 32;   // children per lane

__device__ __forceinline__ double warp_max_d(double x) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) x = fmax(x, __shfl_xor_sync(FULL, x, off));
  return x;
}
__device__ __forceinline__ double warp_min_d(double x) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) x = fmin(x, __shfl_xor_sync(FULL, x, off));
  return x;
}
__device__ __forceinline__ double warp_sum_d(double x) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) x += __shfl_xor_sync(FULL, x, off);
  return x;
}
// first maximum in child order: (score, child) of the lane whose child wins
__device__ __forceinline__ void warp_argmax_first(double& s, int& j) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double os = __shfl_xor_sync(FULL, s, off);
    const int oj = __shfl_xor_sync(FULL, j, off);
    if (oj >= 0 && (j < 0 || os > s || (os == s && oj < j))) { s = os; j = oj; }
  }
}

// Children of `node` (first child fc, nc children), lane-strided: child j = lane + 32 t sits in entry t.
struct GbChildren {
  double l[GB_T];    // logits l(a) in float64
  int n[GB_T];       // N(a)
  double sg[GB_T];   // sigma(completed Q)(a)
  double lmax;       // max l over the node's children
  int nsum;          // Nc = sum of N(a)
  int nmax;          // max N(a)
};

// sigma at a node: p = softmax(l); v_mix = (r + Nc * sum_{N>0} p q / sum_{N>0} p) / (1 + Nc) (r when Nc = 0);
// Q^ = q where N > 0, else v_mix; Q~ = (Q^ - min) / max(max - min, 1e-8); sigma = (c_visit + max N) * c_scale * Q~
__device__ __forceinline__ void warp_children_sigma(const EngineView& E, const GumbelView& GB, size_t nb, int node, int fc, int nc, int lane,
                                                    GbChildren& C) {
  double w[GB_T];
  double mx = -INFINITY;
  int ns = 0, nm = 0;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    const int j = lane + 32 * t;
    C.l[t] = -INFINITY;
    C.n[t] = 0;
    w[t] = 0.0;
    if (j < nc) {
      const size_t c = nb + fc + j;
      C.l[t] = (double)GB.logit[c];
      C.n[t] = E.node_n[c];
      w[t] = E.node_w[c];
      mx = fmax(mx, C.l[t]);
      ns += C.n[t];
      nm = max(nm, C.n[t]);
    }
  }
  mx = warp_max_d(mx);
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    ns += __shfl_xor_sync(FULL, ns, off);
    nm = max(nm, __shfl_xor_sync(FULL, nm, off));
  }
  double e[GB_T], se = 0.0;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    e[t] = lane + 32 * t < nc ? exp(C.l[t] - mx) : 0.0;
    se += e[t];
  }
  se = warp_sum_d(se);
  double spq = 0.0, sp = 0.0;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    if (C.n[t] > 0) {
      const double p = e[t] / se;
      spq += p * (-w[t] / (double)C.n[t]);
      sp += p;
    }
  }
  spq = warp_sum_d(spq);
  sp = warp_sum_d(sp);
  const double r = (double)GB.r[nb + node];
  const double vmix = ns == 0 ? r : (r + (double)ns * spq / sp) / (double)(1 + ns);
  double qh[GB_T], lo = INFINITY, hi = -INFINITY;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    qh[t] = C.n[t] > 0 ? -w[t] / (double)C.n[t] : vmix;
    if (lane + 32 * t < nc) { lo = fmin(lo, qh[t]); hi = fmax(hi, qh[t]); }
  }
  lo = warp_min_d(lo);
  hi = warp_max_d(hi);
  const double scale = (GB.c_visit + (double)nm) * GB.c_scale, den = fmax(hi - lo, 1e-8);
#pragma unroll
  for (int t = 0; t < GB_T; ++t) C.sg[t] = scale * ((qh[t] - lo) / den);
  C.lmax = mx;
  C.nsum = ns;
  C.nmax = nm;
}

// T(m, n)[k]: the visit count a root candidate must have at simulation k -- sequential halving written as a visit schedule
// (DESIGN.md §9).  In every phase the k candidates still in play have equal visits, so a round appends k copies of one value.
__device__ __forceinline__ int halving_schedule_at(int m, int n, int k) {
  if (m <= 1) return k;
  int L = 0;
  while ((1 << L) < m) ++L;   // ceil(log2(m))
  int len = 0, v = 0, kk = m;
  while (true) {
    const int d = L * kk, reps = n / d > 1 ? n / d : 1;
    for (int i = 0; i < reps; ++i) {
      if (k < len + kk) return v;
      len += kk;
      ++v;
    }
    kk = kk / 2 > 2 ? kk / 2 : 2;
  }
}

// root score g(a) + l(a) - max l + sigma(a) over the children with N(a) == target
__device__ __forceinline__ void root_argmax(const GumbelView& GB, int g, int nc, int target, const GbChildren& C, int lane, double& best_s, int& best_j) {
  best_s = -INFINITY;
  best_j = -1;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    const int j = lane + 32 * t;
    if (j < nc && C.n[t] == target) {
      const double s = GB.draw[(size_t)g * MAX_MOVES + j] + C.l[t] - C.lmax + C.sg[t];
      if (best_j < 0 || s > best_s) { best_s = s; best_j = j; }
    }
  }
  warp_argmax_first(best_s, best_j);
}

// One leaf per game: the root rule at the root, argmax softmax(l + sigma) - N / (1 + Nc) below it.  A live leaf's planes go to row g
// of `planes` and the game is left pending (pend_flags: PEND_ACTIVE); a terminal leaf is backed up here and writes no row, as does a
// game that has run its n simulations or holds no search.
__global__ void __launch_bounds__(TREE_THREADS)
gumbel_select_kernel(EngineView E, GumbelView GB, float* __restrict__ planes) {
  __shared__ u16 s_moves[TREE_WARPS][MAX_MOVES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  const int root = E.root_node[g];
  const size_t nb = (size_t)g * E.max_nodes;
  const int k = root >= 0 ? E.node_n[nb + root] - 1 : GB.n;   // simulations done: the root starts at N = 1
  if (root < 0 || k >= GB.n || E.node_first[nb + root] < 0) {
    if (lane == 0) { E.pend_flags[g] = 0; E.pend_count[g] = 0; }
    return;
  }
  const SearchParams& P = *E.params;
  int* path = E.path_node + (size_t)g * E.max_depth;
  Key128* pkey = E.path_key + (size_t)g * E.max_depth;
  u8* pirrev = E.path_irrev + (size_t)g * E.max_depth;
  Position pos = load_position(E.root_pos + (size_t)g * POSITION_WORDS);
  bool cur_epl = E.root_ep_legal[g] != 0;
  Key128 cur_key = E.root_key[g];
  int node = root, depth = 0;
  if (lane == 0) path[0] = root;
  while (true) {
    const int fc = E.node_first[nb + node];
    const int nc = fc < 0 ? 0 : E.node_nchild[nb + node];
    if (nc == 0) break;
    if (depth >= E.max_depth - 1) {
      if (lane == 0) E.status[g] |= ST_DEPTH_CAP;
      break;
    }
    GbChildren C;
    warp_children_sigma(E, GB, nb, node, fc, nc, lane, C);
    double best_s;
    int best_j;
    if (depth == 0) {
      const int mp = GB.m < nc ? GB.m : nc;
      root_argmax(GB, g, nc, halving_schedule_at(mp, GB.n, k), C, lane, best_s, best_j);
    } else {
      double z[GB_T], mz = -INFINITY;
#pragma unroll
      for (int t = 0; t < GB_T; ++t) {
        z[t] = C.l[t] + C.sg[t];
        if (lane + 32 * t < nc) mz = fmax(mz, z[t]);
      }
      mz = warp_max_d(mz);
      double ez[GB_T], se = 0.0;
#pragma unroll
      for (int t = 0; t < GB_T; ++t) {
        ez[t] = lane + 32 * t < nc ? exp(z[t] - mz) : 0.0;
        se += ez[t];
      }
      se = warp_sum_d(se);
      const double inv_n = 1.0 + (double)C.nsum;
      best_s = -INFINITY;
      best_j = -1;
#pragma unroll
      for (int t = 0; t < GB_T; ++t) {
        const int j = lane + 32 * t;
        if (j < nc) {
          const double s = ez[t] / se - (double)C.n[t] / inv_n;
          if (best_j < 0 || s > best_s) { best_s = s; best_j = j; }
        }
      }
      warp_argmax_first(best_s, best_j);
    }
    if (best_j < 0) best_j = 0;   // no root candidate holds the scheduled count: cannot happen while m' <= the legal moves
    const int child = fc + best_j;
    const Move mv = (Move)(E.node_mv[nb + child] & 0xFFFFu);
    PushInfo info = push_move(pos, mv);
    const bool irrev = info.zeroing || info.reduced_castling || cur_epl;
    bool epl;
    cur_key = position_key(pos, &epl);
    cur_epl = epl;
    if (lane == 0) {
      pirrev[depth] = irrev ? 1 : 0;
      pkey[depth + 1] = cur_key;
      path[depth + 1] = child;
    }
    depth++;
    node = child;
  }
  __syncwarp();
  bool terminal;
  double tv;
  const int n_moves = warp_leaf_moves(E, P, g, pos, depth, cur_key, s_moves[wib], &terminal, &tv, lane);
  if (terminal) {
    warp_backup(E, g, depth + 1, py_clip_unit(tv), 1, lane);
    if (lane == 0) {
      E.pend_flags[g] = 0;
      E.pend_count[g] = 0;
      atomicAdd(&E.counters[CTR_SIMS], 1ull);
      atomicAdd(&E.counters[CTR_TERMINAL_SIMS], 1ull);
    }
    return;
  }
  const int wtm = pos_turn(pos);
  for (int j = lane; j < n_moves; j += 32) {
    const Move m = s_moves[wib][j];
    E.leaf_moves[(size_t)g * MAX_MOVES + j] = m;
    E.leaf_idx[(size_t)g * MAX_MOVES + j] = (u16)policy_index(m, wtm);
  }
  if (lane == 0) {
    E.leaf_n[g] = n_moves;
    store_position(E.leaf_pos + (size_t)g * POSITION_WORDS, pos);
    E.path_len[g] = depth + 1;
    E.pend_node[g] = node;
    E.pend_count[g] = 1;
    E.pend_flags[g] = PEND_ACTIVE | PEND_EXPAND;
    atomicAdd(&E.counters[CTR_SIMS], 1ull);
    atomicAdd(&E.counters[CTR_NN_EVALS], 1ull);
  }
  planes += (size_t)g * (19 * 64);
  warp_write_planes(pos, planes, lane);
}

// Expansion of every pending node from row g of the evaluator's output, then the backup of its value r along the path (leaf
// included: a fresh node holds N = 1, W = r).  The root pending after m0_search_begin (path length 1) also gets its Gumbel draws.
__global__ void __launch_bounds__(TREE_THREADS)
gumbel_expand_backup_kernel(EngineView E, GumbelView GB, const float* __restrict__ logits, int logits_stride, const float* __restrict__ values,
                            unsigned long long rng_step) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  const int flags = E.pend_flags[g];
  if (!(flags & PEND_ACTIVE)) return;
  const size_t nb = (size_t)g * E.max_nodes;
  const int node = E.pend_node[g];
  const float* lg = logits + (size_t)g * logits_stride;
  const float r = fminf(fmaxf(values[g], -1.0f), 1.0f);
  const int k = E.leaf_n[g];
  if (E.node_first[nb + node] < 0 && k > 0) {
    int first = 0;
    if (lane == 0) {
      first = E.node_count[g];
      if (first + k > E.max_nodes) {
        E.status[g] |= ST_NODE_OVERFLOW;
        first = -1;
      } else {
        E.node_count[g] = first + k;
      }
    }
    first = __shfl_sync(FULL, first, 0);
    if (first >= 0) {
      const u16* mvs = E.leaf_moves + (size_t)g * MAX_MOVES;
      const u16* idx = E.leaf_idx + (size_t)g * MAX_MOVES;
      for (int j = lane; j < k; j += 32) {
        const size_t c = nb + first + j;
        E.node_w[c] = 0.0;
        E.node_q[c] = 0.0;
        E.node_n[c] = 0;
        E.node_first[c] = -1;
        E.node_creator[c] = node;
        E.node_mv[c] = (u32)mvs[j] | ((u32)idx[j] << 16);
        E.node_nchild[c] = 0;
        GB.logit[c] = lg[idx[j]];
      }
      __syncwarp();
      if (lane == 0) {
        E.node_first[nb + node] = first;
        E.node_nchild[nb + node] = (u16)k;
        atomicAdd(&E.counters[CTR_EXPANSIONS], 1ull);
        atomicAdd(&E.counters[CTR_CHILDREN_CREATED], (unsigned long long)k);
      }
    }
  }
  if (lane == 0) GB.r[nb + node] = r;
  if (flags & PEND_ROOT) {
    // g(a) ~ Gumbel(0, 1) once per legal move and move played: caller-supplied, or keyed by (seed, game, call, move slot)
    const u64 seed = E.params->seed;
    for (int j = lane; j < k; j += 32) {
      double d;
      if (GB.user_draw) {
        d = GB.user_draw[(size_t)g * MAX_MOVES + j];
      } else {
        double u = uniform01(mix64(seed ^ mix64(rng_step * 0xA0761D6478BD642Full + (u64)(g + 1)) ^ mix64((u64)(j + 1) * 0xE7037ED1A0B428DBull)));
        u = u > 0.0 ? u : 1.0 / 9007199254740992.0;
        d = -log(-log(u));
      }
      GB.draw[(size_t)g * MAX_MOVES + j] = d;
    }
    if (lane == 0) GB.choice[g] = -1;
  }
  __syncwarp();
  warp_backup(E, g, E.path_len[g], py_clip_unit((double)r), 1, lane);
  if (lane == 0) {
    E.pend_flags[g] = 0;
    E.pend_count[g] = 0;
  }
}

// After the n simulations: the move played (argmax of the root score over the most visited children), the policy target
// pi' = softmax(l + sigma) at the root (float64, stored as float32 at its policy index, 0 elsewhere), the search value
// W(root) / N(root), and per root child its visits, q and pi'.  Every output except d_move / d_value may be NULL.
__global__ void __launch_bounds__(TREE_THREADS)
gumbel_result_kernel(EngineView E, GumbelView GB, u16* __restrict__ out_move, float* __restrict__ out_pi, double* __restrict__ out_value,
                     int* __restrict__ out_visits, double* __restrict__ out_q, double* __restrict__ out_pi_children, int* __restrict__ out_count) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G) return;
  const size_t nb = (size_t)g * E.max_nodes;
  const int root = E.active[g] ? E.root_node[g] : -1;
  const int fc = root >= 0 ? E.node_first[nb + root] : -1;
  const int nc = fc < 0 ? 0 : E.node_nchild[nb + root];
  float* pi = out_pi ? out_pi + (size_t)g * POLICY_SIZE : nullptr;
  if (pi) {
    float4* p4 = reinterpret_cast<float4*>(pi);
    for (int i = lane; i < POLICY_SIZE / 4; i += 32) p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncwarp();
  if (nc == 0) {
    if (lane == 0) {
      GB.choice[g] = -1;
      GB.value[g] = 0.0;
      GB.entropy[g] = 0.0;
      out_move[g] = (u16)MOVE_NONE;
      out_value[g] = 0.0;
      if (out_count) out_count[g] = 0;
    }
    return;
  }
  GbChildren C;
  warp_children_sigma(E, GB, nb, root, fc, nc, lane, C);
  double z[GB_T], mz = -INFINITY;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    z[t] = C.l[t] + C.sg[t];
    if (lane + 32 * t < nc) mz = fmax(mz, z[t]);
  }
  mz = warp_max_d(mz);
  double ez[GB_T], se = 0.0;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    ez[t] = lane + 32 * t < nc ? exp(z[t] - mz) : 0.0;
    se += ez[t];
  }
  se = warp_sum_d(se);
  // entropy of pi' as the visit-count modes take it (internal.py:433-441): float32 entries clipped to [1e-12, 1] over all 4672
  double ent = 0.0;
#pragma unroll
  for (int t = 0; t < GB_T; ++t) {
    const int j = lane + 32 * t;
    if (j >= nc) continue;
    const size_t c = nb + fc + j;
    const float p = (float)(ez[t] / se);
    double pd = (double)p;
    if (pd < 1e-12) pd = 1e-12;
    ent -= pd * log(pd);
    if (pi) pi[E.node_mv[c] >> 16] = p;
    if (out_pi_children) out_pi_children[(size_t)g * MAX_MOVES + j] = ez[t] / se;
    if (out_visits) out_visits[(size_t)g * MAX_MOVES + j] = C.n[t];
    if (out_q) out_q[(size_t)g * MAX_MOVES + j] = C.n[t] > 0 ? -E.node_w[c] / (double)C.n[t] : 0.0;
  }
  ent = warp_sum_d(ent) - (double)(POLICY_SIZE - nc) * (1e-12 * log(1e-12));
  double best_s;
  int best_j;
  root_argmax(GB, g, nc, C.nmax, C, lane, best_s, best_j);
  if (lane == 0) {
    const double v = E.node_w[nb + root] / (double)E.node_n[nb + root];
    GB.choice[g] = best_j;
    GB.value[g] = v;
    GB.entropy[g] = ent;
    out_move[g] = (u16)(E.node_mv[nb + fc + best_j] & 0xFFFFu);
    out_value[g] = v;
    if (out_count) out_count[g] = nc;
  }
}

}  // namespace m0
