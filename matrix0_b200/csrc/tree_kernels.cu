// Warp-per-game MCTS tree kernels: root lookup, PUCT selection, leaf expansion, backup, result
// extraction.  Reference-exact mode reproduces azchess/mcts.py with the deterministic harness of
// SURVEY section 7-0c (jitter neutralised, noise off): the batch-collision semantics of
// _run_simulations_parallel_batched (:514-740, SURVEY Q1), edge-child vs TT-node statistics
// (:865-881 vs :918-920, Q4), fp64 sequential backups (:946-953, Q7) and last-writer-wins
// transposition registration (:1330-1346).
//
// Memory behaviour: one warp per game; the children of a node occupy consecutive slots of the
// per-game node arrays, so the PUCT scan reads prior/n/q/move with fully coalesced lane-strided
// loads (24 B per child); the leaf position lives in registers of every lane (no broadcast
// traffic) and the leaf move list is staged in shared memory.
#include "tree_common.cuh"

namespace m0 {

// ---- game bookkeeping -------------------------------------------------------------------------------
__global__ void reset_games_kernel(EngineView E, const int* __restrict__ games, int n_games) {
  // grid.y = game slot in the list, threads clear that game's transposition table
  int gi = blockIdx.y;
  if (gi >= n_games) return;
  int g = games ? games[gi] : gi;
  size_t base = (size_t)g * E.tt_cap;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < E.tt_cap; i += gridDim.x * blockDim.x) {
    E.tt_lo[base + i] = 0;
    E.tt_hi[base + i] = 0;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    E.node_count[g] = 0;
    E.tt_count[g] = 0;
    E.hist_len[g] = 0;
    E.root_node[g] = -1;
    E.pend_flags[g] = 0;
    E.pend_count[g] = 0;
    E.status[g] = 0;
    E.active[g] = 0;
  }
}

// Set the root position of games and (optionally) the game history that precedes it.
// hist_pos [n_games][hist_stride][9] / hist_moves [n_games][hist_stride]: positions P_0..P_{L-1} before the
// root and the moves played from them (board.move_stack); thread i of a game computes key(P_i) and
// Board.is_irreversible(m_i).
__global__ void set_positions_kernel(EngineView E, const int* __restrict__ games, int n_games, const u64* __restrict__ root_pos,
                                     const u64* __restrict__ hist_pos, const u16* __restrict__ hist_moves,
                                     const int* __restrict__ hist_lens, int hist_stride) {
  int gi = blockIdx.x;
  if (gi >= n_games) return;
  int g = games ? games[gi] : gi;
  int L = hist_lens ? hist_lens[gi] : 0;
  if (L > E.hist_cap) L = E.hist_cap;  // host keeps only the tail
  for (int i = threadIdx.x; i < L; i += blockDim.x) {
    Position p = load_position(hist_pos + ((size_t)gi * hist_stride + i) * POSITION_WORDS);
    bool epl;
    Key128 k = position_key(p, &epl);
    PushInfo info = push_move(p, hist_moves[(size_t)gi * hist_stride + i]);
    E.hist_key[(size_t)g * E.hist_cap + i] = k;
    E.hist_irrev[(size_t)g * E.hist_cap + i] = (info.zeroing || info.reduced_castling || epl) ? 1 : 0;
  }
  if (threadIdx.x == 0) {
    Position p = load_position(root_pos + (size_t)gi * POSITION_WORDS);
    store_position(E.root_pos + (size_t)g * POSITION_WORDS, p);
    E.hist_len[g] = L;
    E.active[g] = 1;
    E.root_node[g] = -1;
    E.pend_flags[g] = 0;
    E.pend_count[g] = 0;
  }
}

// ---- MCTS.run prologue: azchess/mcts.py:336-371, 398-416 -----------------------------------------------
// Per game: terminal root? -> flag; root = tt.get(key) or a fresh Node that needs an evaluation.
// out_info[g]: bit0 terminal root, bit1 evaluation requested; out_value[g] = terminal value.
__global__ void __launch_bounds__(TREE_THREADS)
search_begin_kernel(EngineView E, float* __restrict__ planes, int* __restrict__ out_info, double* __restrict__ out_value) {
  __shared__ u16 s_moves[TREE_WARPS][MAX_MOVES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  const size_t nb = (size_t)g * E.max_nodes;
  Position pos = load_position(E.root_pos + (size_t)g * POSITION_WORDS);
  bool epl;
  Key128 key = position_key(pos, &epl);
  int in_check = 0;
  int n_moves = warp_generate_legal_moves(pos, s_moves[wib], &in_check, lane);
  if (n_moves > MAX_MOVES) n_moves = MAX_MOVES;
  // board.is_game_over(): the search path is empty, so only the game history can repeat
  if (lane == 0) {
    E.root_key[g] = key;
    E.root_ep_legal[g] = epl ? 1 : 0;
    E.path_key[(size_t)g * E.max_depth] = key;
  }
  __syncwarp();
  bool terminal = n_moves == 0 || is_insufficient_material(pos) || (pos_halfmove(pos) >= 150 && n_moves > 0);
  if (!terminal && pos_halfmove(pos) >= 8) {
    int rep = 0;
    if (lane == 0) rep = leaf_is_fivefold(E, g, 0, key) ? 1 : 0;
    terminal = __shfl_sync(FULL, rep, 0) != 0;
  }
  if (terminal) {
    if (lane == 0) {
      out_info[g] = 1;
      out_value[g] = (n_moves == 0 && in_check) ? -1.0 : E.params->draw_penalty;
      E.pend_flags[g] = 0;
      E.pend_count[g] = 0;
      E.root_node[g] = -1;
      if (E.rc_slots) E.rc_fill[g] = 0;
    }
    return;
  }
  int root = 0, flags = 0;
  if (lane == 0) {
    root = tt_get(E, g, key);
    if (root < 0) {
      // root = Node(); expand after inference (children NOT registered, mcts.py:350-358); tt[key] = root
      int cnt = E.node_count[g];
      if (cnt >= E.max_nodes) {
        E.status[g] |= ST_NODE_OVERFLOW;
        root = 0;
      } else {
        root = cnt;
        E.node_count[g] = cnt + 1;
        E.node_prior[nb + root] = 0.0;
        E.node_w[nb + root] = 0.0;
        E.node_q[nb + root] = 0.0;
        E.node_n[nb + root] = 0;
        E.node_first[nb + root] = -1;
        E.node_creator[nb + root] = -1;
        E.node_mv[nb + root] = MOVE_NONE;
        E.node_nchild[nb + root] = 0;
        tt_put(E, g, key, root);
        flags = PEND_ACTIVE | PEND_EXPAND | PEND_ROOT;
      }
    } else if (E.node_first[nb + root] < 0) {
      // TT hit on a never-expanded node: expand, register children, root.q = v (mcts.py:399-413)
      flags = PEND_ACTIVE | PEND_EXPAND | PEND_REGISTER | PEND_SET_Q | PEND_ROOT;
    }
    E.root_node[g] = root;
    E.path_node[(size_t)g * E.max_depth] = root;
    E.path_len[g] = 1;
    E.pend_node[g] = root;
    E.pend_count[g] = 0;
    E.pend_flags[g] = flags;
    out_info[g] = flags ? 2 : 0;
    out_value[g] = 0.0;
  }
  flags = __shfl_sync(FULL, flags, 0);
  if (flags) {
    const int wtm = pos_turn(pos);
    for (int k = lane; k < n_moves; k += 32) {
      Move mv = s_moves[wib][k];
      E.leaf_moves[(size_t)g * MAX_MOVES + k] = mv;
      E.leaf_idx[(size_t)g * MAX_MOVES + k] = (u16)policy_index(mv, wtm);
    }
    if (lane == 0) {
      E.leaf_n[g] = n_moves;
      store_position(E.leaf_pos + (size_t)g * POSITION_WORDS, pos);
    }
    if (planes) warp_write_planes(pos, planes + (size_t)g * (19 * 64), lane);
    if (E.rc_slots) {
      // the root among the children evaluated during the previous move (all 9 words: pieces, side to move, castling, clocks)?
      // hit: the expansion reads that entry; miss: the root's planes go to the next compact row of the caller's miss buffer
      const u64* rw = E.root_pos + (size_t)g * POSITION_WORDS;
      const int fill = E.rc_fill[g];
      int src = 0;
      bool hit = false;
      for (int e0 = 0; e0 < fill && !hit; e0 += 32) {   // one entry per lane
        const u64* ew = E.rc_pos + ((size_t)g * E.rc_slots + e0 + lane) * POSITION_WORDS;
        bool eq = e0 + lane < fill;
        for (int w = 0; w < POSITION_WORDS && eq; ++w) eq = ew[w] == rw[w];
        const unsigned hits = __ballot_sync(FULL, eq);
        if (hits) {
          hit = true;
          src = -1 - (e0 + __ffs(hits) - 1);
        }
      }
      if (hit) {
        if (lane == 0) atomicAdd(&E.counters[CTR_ROOT_REUSED], 1ull);
      } else {
        int row = 0;
        if (lane == 0) row = atomicAdd(E.rc_miss_count, 1);
        src = __shfl_sync(FULL, row, 0);
        warp_write_planes(pos, E.rc_miss_planes + (size_t)src * (19 * 64), lane);
      }
      if (lane == 0) E.rc_src[g] = src;
    }
  }
  if (E.rc_slots && lane == 0) E.rc_fill[g] = 0;   // this move records its own root children
}

// ---- selection: azchess/mcts.py:742-769 (_collect_leaf_position) + :851-925 (_select) ----------------------
// Runs up to batch_n simulations for the game.  Terminal leaves are backed up immediately
// (:747-751); the first non-terminal leaf becomes the game's pending evaluation with multiplicity
// (remaining simulations of the batch), which is exactly what the reference's collected batch
// contains when nothing can change between its selections (SURVEY Q1).
__global__ void __launch_bounds__(TREE_THREADS)
search_select_kernel(EngineView E, int batch_cap, int* __restrict__ sims_left, float* __restrict__ planes, unsigned long long rng_step) {
  __shared__ u16 s_moves[TREE_WARPS][MAX_MOVES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  const int root = E.root_node[g];
  if (root < 0) {
    if (lane == 0) { E.pend_flags[g] = 0; E.pend_count[g] = 0; }
    return;
  }
  const SearchParams& P = *E.params;
  const size_t nb = (size_t)g * E.max_nodes;
  int* path = E.path_node + (size_t)g * E.max_depth;
  Key128* pkey = E.path_key + (size_t)g * E.max_depth;
  u8* pirrev = E.path_irrev + (size_t)g * E.max_depth;
  const Position root_pos = load_position(E.root_pos + (size_t)g * POSITION_WORDS);
  const bool root_epl = E.root_ep_legal[g] != 0;
  unsigned long long c_scanned = 0, c_path = 0, c_term = 0, c_hops = 0;

  int batch_n = batch_cap;
  if (sims_left) {  // per-game simulation budgets (playout cap randomisation, mcts.py:380-385)
    int left = sims_left[g];
    batch_n = left < batch_cap ? left : batch_cap;
    __syncwarp();
    if (lane == 0) sims_left[g] = left - batch_n;
  }
  int remaining = batch_n;
  int pend_m = 0;
  while (remaining > 0) {
    Position pos = root_pos;
    int node = root, depth = 0;
    bool cur_epl = root_epl;
    Key128 cur_key = E.root_key[g];
    while (true) {
      const int fc = E.node_first[nb + node];
      if (fc < 0) break;
      const int nc = E.node_nchild[nb + node];
      if (nc == 0) break;
      if (depth >= E.max_depth - 1) {
        if (lane == 0) E.status[g] |= ST_DEPTH_CAP;
        break;
      }
      const int pn = E.node_n[nb + node];
      const double sqrt_pv = d_sqrt((double)(pn > 1 ? pn : 1));
      const double fpu_q = d_sub(E.node_q[nb + node], P.fpu_reduction);
      const double cp = E.cpuct[depth < P.cpuct_len ? depth : P.cpuct_len - 1];
      const u32 prev_mv = E.node_mv[nb + node] & 0xFFFFu;
      const bool backtrack_check = P.no_instant_backtrack && depth >= 1 && prev_mv != MOVE_NONE;
      double best_s = -1e9;
      int best_j = -1;
      for (int j = lane; j < nc; j += 32) {
        const size_t c = nb + fc + j;
        const int cn = E.node_n[c];
        const double q = cn == 0 ? fpu_q : E.node_q[c];
        double s = puct_score(q, cp, E.node_prior[c], sqrt_pv, cn);
        if (backtrack_check) {
          u32 mv = E.node_mv[c] & 0xFFFFu;
          if ((mv & 63u) == ((prev_mv >> 6) & 63u) && ((mv >> 6) & 63u) == (prev_mv & 63u)) s = d_sub(s, 0.01);
        }
        if (P.jitter_on) {
          u64 r = mix64(P.seed ^ mix64(rng_step + 0x9E3779B97F4A7C15ull * (u64)(g + 1)) ^ ((u64)(fc + j) << 20) ^ (u64)(batch_n - remaining));
          s = d_add(s, d_mul(d_sub(uniform01(r), 0.5), P.jitter));
        }
        if (s > best_s) { best_s = s; best_j = j; }
      }
      c_scanned += nc;
      // first maximum in child order (strict '>' scan, mcts.py:901)
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        double os = __shfl_xor_sync(FULL, best_s, off);
        int oj = __shfl_xor_sync(FULL, best_j, off);
        bool take = oj >= 0 && (best_j < 0 || os > best_s || (os == best_s && oj < best_j));
        if (take) { best_s = os; best_j = oj; }
      }
      if (best_j < 0) best_j = 0;  // "Fallback: selected first child" (mcts.py:911-914)
      const int child = fc + best_j;
      const Move mv = (Move)(E.node_mv[nb + child] & 0xFFFFu);
      PushInfo info = push_move(pos, mv);
      const bool irrev = info.zeroing || info.reduced_castling || cur_epl;
      bool epl;
      cur_key = position_key(pos, &epl);
      cur_epl = epl;
      int hop = 0;
      if (lane == 0) hop = tt_get(E, g, cur_key);
      hop = __shfl_sync(FULL, hop, 0);
      const int nxt = hop >= 0 ? hop : child;  // node = self._tt_get(key) or best_child (mcts.py:919)
      if (hop >= 0 && hop != child) c_hops++;
      if (lane == 0) {
        pirrev[depth] = irrev ? 1 : 0;
        pkey[depth + 1] = cur_key;
        path[depth + 1] = nxt;
      }
      depth++;
      node = nxt;
    }
    __syncwarp();
    c_path += depth + 1;
    // leaf: terminal? (board.is_game_over(), mcts.py:747)
    int in_check = 0;
    int n_moves = warp_generate_legal_moves(pos, s_moves[wib], &in_check, lane);
    if (n_moves > MAX_MOVES) n_moves = MAX_MOVES;
    bool terminal = n_moves == 0 || is_insufficient_material(pos) || (pos_halfmove(pos) >= 150 && n_moves > 0);
    if (!terminal && pos_halfmove(pos) >= 8) {
      int rep = 0;
      if (lane == 0) rep = leaf_is_fivefold(E, g, depth, cur_key) ? 1 : 0;
      terminal = __shfl_sync(FULL, rep, 0) != 0;
    }
    if (terminal) {
      const double v = (n_moves == 0 && in_check) ? -1.0 : P.draw_penalty;  // _terminal_value, mcts.py:1223-1229
      warp_backup(E, g, depth + 1, py_clip_unit(v), 1, lane);
      remaining--;
      c_term++;
      continue;
    }
    // pending leaf shared by all remaining simulations of this batch
    const int wtm = pos_turn(pos);
    for (int k = lane; k < n_moves; k += 32) {
      Move mv = s_moves[wib][k];
      E.leaf_moves[(size_t)g * MAX_MOVES + k] = mv;
      E.leaf_idx[(size_t)g * MAX_MOVES + k] = (u16)policy_index(mv, wtm);
    }
    if (lane == 0) {
      E.leaf_n[g] = n_moves;
      store_position(E.leaf_pos + (size_t)g * POSITION_WORDS, pos);
      E.path_len[g] = depth + 1;
      E.pend_node[g] = node;
    }
    if (planes) warp_write_planes(pos, planes + (size_t)g * (19 * 64), lane);
    pend_m = remaining;
    remaining = 0;
  }
  if (lane == 0) {
    E.pend_count[g] = pend_m;
    E.pend_flags[g] = pend_m > 0 ? (PEND_ACTIVE | PEND_EXPAND | PEND_REGISTER) : 0;
    atomicAdd(&E.counters[CTR_SIMS], (unsigned long long)batch_n);
    atomicAdd(&E.counters[CTR_TERMINAL_SIMS], c_term);
    atomicAdd(&E.counters[CTR_CHILDREN_SCANNED], c_scanned);
    atomicAdd(&E.counters[CTR_PATH_NODES], c_path);
    atomicAdd(&E.counters[CTR_TT_HOPS], c_hops);
    if (pend_m > 0) atomicAdd(&E.counters[CTR_NN_EVALS], 1ull);
  }
}

// ---- expansion + backup: azchess/mcts.py:135-225 (Node._expand), :1330-1346, :654-670 ---------------------
__global__ void __launch_bounds__(TREE_THREADS)
search_expand_backup_kernel(EngineView E, const float* __restrict__ logits, int logits_stride, const float* __restrict__ values) {
  __shared__ ExpandSmem s_x[TREE_WARPS];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  const int flags = E.pend_flags[g];
  if (!(flags & PEND_ACTIVE)) return;
  const SearchParams& P = *E.params;
  const size_t nb = (size_t)g * E.max_nodes;
  const int node = E.pend_node[g];
  const int times = E.pend_count[g];
  const Position pos = load_position(E.leaf_pos + (size_t)g * POSITION_WORDS);
  // the game's network row: row g, or for a root evaluation with the store enabled, the entry or compact row search_begin chose.
  // Row g is read only in the branch that uses it: the root evaluation's buffers hold just the compact rows (or none at all).
  const float* lg;
  float vf;
  if ((flags & PEND_ROOT) && E.rc_slots) {
    const int src = E.rc_src[g];
    if (src < 0) {
      const size_t e = (size_t)g * E.rc_slots + (-1 - src);
      lg = E.rc_logits + e * POLICY_SIZE;
      vf = E.rc_value[e];
    } else {
      lg = logits + (size_t)src * logits_stride;
      vf = values[src];
    }
  } else {
    lg = logits + (size_t)g * logits_stride;
    vf = values[g];
    if (E.rc_slots && E.path_len[g] == 2) warp_record_root_child(E, g, E.leaf_pos + (size_t)g * POSITION_WORDS, lg, vf, lane);
  }
  // value: float(np.clip(value, -1, 1)) (mcts.py:668) ; _infer clips the same way (:1180)
  vf = fminf(fmaxf(vf, -1.0f), 1.0f);
  double v = (double)vf;
  if ((flags & PEND_ROOT) && P.value_from_white && !pos_turn(pos)) v = -v;  // mcts.py:1184-1186

  const int k = E.leaf_n[g];
  if ((flags & PEND_EXPAND) && E.node_first[nb + node] < 0 && k > 0)
    warp_expand(E, P, g, node, pos, E.leaf_moves + (size_t)g * MAX_MOVES, E.leaf_idx + (size_t)g * MAX_MOVES, k,
                lg, (flags & PEND_REGISTER) != 0, (flags & PEND_ROOT) != 0, s_x[wib], lane);
  if ((flags & PEND_SET_Q) && lane == 0) E.node_q[nb + node] = v;  // root.q = v (mcts.py:412-413)
  __syncwarp();
  if (times > 0) warp_backup(E, g, E.path_len[g], py_clip_unit(v), times, lane);
  if (lane == 0) {
    E.pend_flags[g] = 0;
    E.pend_count[g] = 0;
  }
}


// ---- root Dirichlet noise: azchess/mcts.py:955-992 ---------------------------------------------------------
// p <- p*(1-frac) + noise*frac, clamped to [1e-8, 1-1e-8], no renormalisation.  noise == NULL: the
// kernel draws Dirichlet(alpha) itself (Marsaglia-Tsang gamma variates from a counter-based hash RNG);
// otherwise noise float64[G][256] comes from the caller (the single-game drop-in passes
// np.random.dirichlet so that it consumes the reference's RNG stream).  apply int32[G] gates per game.
__device__ double gamma_variate(double alpha, u64& rng) {
  double boost = 1.0;
  if (alpha < 1.0) {
    rng = mix64(rng + 0x9E3779B97F4A7C15ull);
    double u = uniform01(rng);
    if (u <= 0.0) u = 1e-300;
    boost = pow(u, 1.0 / alpha);
    alpha += 1.0;
  }
  const double d = alpha - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
  for (int it = 0; it < 64; ++it) {
    rng = mix64(rng + 0x9E3779B97F4A7C15ull);
    double u1 = uniform01(rng);
    rng = mix64(rng + 0x9E3779B97F4A7C15ull);
    double u2 = uniform01(rng);
    if (u1 <= 0.0) u1 = 1e-300;
    double x = sqrt(-2.0 * log(u1)) * cos(6.283185307179586 * u2);
    double v = 1.0 + c * x;
    if (v <= 0.0) continue;
    v = v * v * v;
    rng = mix64(rng + 0x9E3779B97F4A7C15ull);
    double u = uniform01(rng);
    if (u <= 0.0) u = 1e-300;
    if (log(u) < 0.5 * x * x + d - d * v + d * log(v)) return d * v * boost;
  }
  return d * boost;
}

__global__ void __launch_bounds__(TREE_THREADS)
search_add_dirichlet_kernel(EngineView E, const double* __restrict__ noise, const int* __restrict__ apply, unsigned long long rng_step) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  if (apply && !apply[g]) return;
  const SearchParams& P = *E.params;
  const int root = E.root_node[g];
  if (root < 0 || P.dirichlet_frac <= 0.0) return;
  const size_t nb = (size_t)g * E.max_nodes;
  const int fc = E.node_first[nb + root];
  if (fc < 0) return;
  const int nc = E.node_nchild[nb + root];
  const double frac = P.dirichlet_frac, keep = d_sub(1.0, frac);
  double gam[MAX_MOVES / 32];
  double sum = 0.0;
  if (!noise) {
    for (int t = 0, j = lane; j < nc; j += 32, ++t) {
      u64 rng = mix64(P.seed ^ mix64(rng_step * 0xD6E8FEB86659FD93ull + (u64)(g + 1)) ^ ((u64)(j + 1) << 32));
      gam[t] = gamma_variate(P.dirichlet_alpha, rng);
      sum += gam[t];
    }
    for (int off = 16; off > 0; off >>= 1) sum += __shfl_xor_sync(FULL, sum, off);
    if (!(sum > 0.0)) sum = 1.0;
  }
  for (int t = 0, j = lane; j < nc; j += 32, ++t) {
    const double eta = noise ? noise[(size_t)g * MAX_MOVES + j] : gam[t] / sum;
    double p = d_add(d_mul(E.node_prior[nb + fc + j], keep), d_mul(eta, frac));
    p = (p < 1.0 - 1e-8) ? p : 1.0 - 1e-8;  // max(1e-8, min(1 - 1e-8, p))
    p = (p > 1e-8) ? p : 1e-8;
    E.node_prior[nb + fc + j] = p;
  }
}

// ---- results: azchess/mcts.py:431 (visit counts), :828-849 (_policy_from_root), :504 (root_q) ----------------
__global__ void __launch_bounds__(TREE_THREADS)
search_result_kernel(EngineView E, u16* __restrict__ out_moves, int* __restrict__ out_visits, double* __restrict__ out_child_q,
                     double* __restrict__ out_prior, int* __restrict__ out_count, float* __restrict__ out_pi,
                     double* __restrict__ out_root_q, int* __restrict__ out_root_n) {
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  const size_t nb = (size_t)g * E.max_nodes;
  const int root = E.root_node[g];
  float* pi = out_pi ? out_pi + (size_t)g * POLICY_SIZE : nullptr;
  if (pi) {
    float4* p4 = reinterpret_cast<float4*>(pi);
    for (int i = lane; i < POLICY_SIZE / 4; i += 32) p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  }
  __syncwarp();
  if (root < 0) {
    if (lane == 0) { out_count[g] = 0; out_root_q[g] = 0.0; out_root_n[g] = 0; }
    return;
  }
  const int fc = E.node_first[nb + root];
  const int nc = fc < 0 ? 0 : E.node_nchild[nb + root];
  long long total = 0;
  for (int j = lane; j < nc; j += 32) total += E.node_n[nb + fc + j];
  for (int off = 16; off > 0; off >>= 1) total += __shfl_xor_sync(FULL, total, off);
  for (int j = lane; j < nc; j += 32) {
    const size_t c = nb + fc + j;
    const int n = E.node_n[c];
    const u32 mv = E.node_mv[c];
    out_moves[(size_t)g * MAX_MOVES + j] = (u16)(mv & 0xFFFFu);
    out_visits[(size_t)g * MAX_MOVES + j] = n;
    if (out_child_q) out_child_q[(size_t)g * MAX_MOVES + j] = E.node_q[c];
    if (out_prior) out_prior[(size_t)g * MAX_MOVES + j] = E.node_prior[c];
    if (pi) {
      // pi[idx] = child.n / total (Python float division, stored to float32); uniform when total == 0
      float val = total > 0 ? (float)d_div((double)n, (double)total) : (float)d_div(1.0, (double)nc);
      if ((mv >> 16) < (u32)POLICY_SIZE) pi[mv >> 16] = val;
    }
  }
  if (lane == 0) {
    out_count[g] = nc;
    out_root_q[g] = E.node_q[nb + root];
    out_root_n[g] = E.node_n[nb + root];
  }
}

}  // namespace m0
