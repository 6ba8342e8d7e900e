// The reference's mini-batch AS SHIPPED (azchess/mcts.py:535-740 with selection_jitter in force, SURVEY Q2b): every one of
// the batch_n simulations of a mini-batch walks the tree with its OWN jitter draws -- random.random() per child per
// visited node, mcts.py:893-897 -- so a batch collects up to batch_n different leaves.  Nothing but terminal backups
// (:747-751) changes the statistics during collection; after inference the samples are processed in collection order:
// expand the leaf if it still is one (+ entropy noise, pruning, TT registration), then back the sample's own path up
// (:654-670).  Samples that reached the same node with the same board share one network row (identical planes give identical
// rows), all others get their own; the rows of all games are compacted into one evaluator batch.
//
// One warp owns one game.  Kernels:
//   search_select_multi_kernel        collection of one mini-batch per game (selection, terminal backups, leaf table)
//   multi_scan_kernel                 exclusive prefix sum of the per-game leaf counts -> compact row numbers
//   multi_encode_kernel               planes of the compact rows of a range of games
//   search_expand_backup_multi_kernel expansion + backup of the samples of a range of games, in sample order
#include "tree_common.cuh"

namespace m0 {

// Most simulations of a mini-batch repeat the path of the one before them (nothing but terminal backups changes the tree during
// collection): the move made at each depth, the position it leads to, its key and the transposition-table hop are remembered per
// depth and reused while the path prefix stays the same -- only the PUCT scan with its fresh jitter draws is repeated.
static constexpr int WALK_CACHE_DEPTH = 12;
struct WalkCache {
  u64 pos[WALK_CACHE_DEPTH][POSITION_WORDS];
  Key128 key[WALK_CACHE_DEPTH];
  int child[WALK_CACHE_DEPTH], nxt[WALK_CACHE_DEPTH];
  u8 epl[WALK_CACHE_DEPTH], irrev[WALK_CACHE_DEPTH];
};

__global__ void __launch_bounds__(TREE_THREADS)
search_select_multi_kernel(EngineView E, int batch_cap, int* __restrict__ sims_left) {
  __shared__ u16 s_moves[TREE_WARPS][MAX_MOVES];
  __shared__ WalkCache s_cache[TREE_WARPS];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * TREE_WARPS + wib;
  if (g >= E.G) return;
  if (!E.active[g] || E.root_node[g] < 0) {
    if (lane == 0) { E.ml_n_samples[g] = 0; E.ml_n_leaves[g] = 0; }
    return;
  }
  const int root = E.root_node[g];
  const SearchParams& P = *E.params;
  const size_t nb = (size_t)g * E.max_nodes;
  int* path = E.path_node + (size_t)g * E.max_depth;
  Key128* pkey = E.path_key + (size_t)g * E.max_depth;
  u8* pirrev = E.path_irrev + (size_t)g * E.max_depth;
  int* smp_leaf = E.ml_smp_leaf + (size_t)g * E.ml_cap;
  int* smp_len = E.ml_smp_len + (size_t)g * E.ml_cap;
  int* leaf_node = E.ml_leaf_node + (size_t)g * E.ml_cap;
  int* leaf_first = E.ml_leaf_first + (size_t)g * E.ml_cap;
  const Position root_pos = load_position(E.root_pos + (size_t)g * POSITION_WORDS);
  const bool root_epl = E.root_ep_legal[g] != 0;
  unsigned long long c_scanned = 0, c_path = 0, c_term = 0, c_hops = 0;
  unsigned long long jcur = E.jit_cursor[g];

  int batch_n = batch_cap < E.ml_cap ? batch_cap : E.ml_cap;
  if (sims_left) {  // per-game simulation budgets (playout cap randomisation, mcts.py:380-385)
    int left = sims_left[g];
    batch_n = left < batch_n ? left : batch_n;
    __syncwarp();
    if (lane == 0) sims_left[g] = left - batch_n;
  }
  int n_samples = 0, n_leaves = 0;
  if (lane == 0) path[0] = root;
  const bool vl = P.virtual_loss_on && E.node_inflight != nullptr && P.virtual_loss > 0.0;
  u16* inflight = vl ? E.node_inflight + nb : nullptr;
  if (vl) {   // inflight_counts = {} for this mini-batch
    const int cnt = E.node_count[g];
    for (int i = lane; i < cnt; i += 32) inflight[i] = 0;
    __syncwarp();
  }
  WalkCache& wc = s_cache[wib];
  int cached = 0;   // depths 0 .. cached-1 of the cache describe the previous walk
  for (int sim = 0; sim < batch_n; ++sim) {
    Position pos = root_pos;
    int node = root, depth = 0;
    bool cur_epl = root_epl;
    Key128 cur_key = E.root_key[g];
    bool same_prefix = true;
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
        if (vl) s = d_sub(s, d_mul((double)inflight[fc + j], P.virtual_loss));                                   // mcts.py:889-890
        if (P.jitter_on) s = d_add(s, d_mul(d_sub(draw_jitter_uniform(E, P, g, jcur, j), 0.5), P.jitter));   // mcts.py:893-897
        if (s > best_s) { best_s = s; best_j = j; }
      }
      if (P.jitter_on) {
        if (E.jit_stream && jcur + (unsigned long long)nc > (unsigned long long)E.jit_stride && lane == 0) E.status[g] |= ST_STREAM_EXHAUSTED;
        jcur += (unsigned long long)nc;   // one random.random() per child, in child order
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
      int nxt;
      if (same_prefix && depth < cached && wc.child[depth] == child) {
        // the same move as in the previous walk, from the same position: position, key, hop and the path entries are already there
        pos = load_position(wc.pos[depth]);
        cur_key = wc.key[depth];
        cur_epl = wc.epl[depth] != 0;
        nxt = wc.nxt[depth];
        if (nxt != child) c_hops++;
        if (vl && lane == 0) inflight[child] += 1;
      } else {
        same_prefix = false;
        const Move mv = (Move)(E.node_mv[nb + child] & 0xFFFFu);
        PushInfo info = push_move(pos, mv);
        const bool irrev = info.zeroing || info.reduced_castling || cur_epl;
        bool epl;
        cur_key = position_key(pos, &epl);
        cur_epl = epl;
        int hop = 0;
        if (lane == 0) hop = tt_get(E, g, cur_key);
        hop = __shfl_sync(FULL, hop, 0);
        nxt = hop >= 0 ? hop : child;  // node = self._tt_get(key) or best_child (mcts.py:919)
        if (hop >= 0 && hop != child) c_hops++;
        __syncwarp();
        if (lane == 0) {
          pirrev[depth] = irrev ? 1 : 0;
          pkey[depth + 1] = cur_key;
          path[depth + 1] = nxt;
          if (vl) inflight[child] += 1;   // inflight_counts[best_child] += 1 (the EDGE child, mcts.py:922-923)
          if (depth < WALK_CACHE_DEPTH) {
            store_position(wc.pos[depth], pos);
            wc.key[depth] = cur_key;
            wc.child[depth] = child;
            wc.nxt[depth] = nxt;
            wc.epl[depth] = epl ? 1 : 0;
            wc.irrev[depth] = irrev ? 1 : 0;
          }
        }
        cached = depth < WALK_CACHE_DEPTH ? depth + 1 : WALK_CACHE_DEPTH;   // deeper entries belong to another path now
        __syncwarp();
      }
      depth++;
      node = nxt;
      if (vl) __syncwarp();
    }
    __syncwarp();
    c_path += depth + 1;
    // Is this leaf already in the game's leaf table (same node, same board)?  Then an earlier simulation of this mini-batch found it
    // alive -- legal moves exist, material and the 75-move clock are properties of the board -- and only the repetition test, which
    // looks at THIS path, has to be repeated.  Otherwise generate the moves and test the position (board.is_game_over(), mcts.py:747).
    int slot = -1;
    const u64* lp = E.ml_leaf_pos + (size_t)g * E.ml_cap * POSITION_WORDS;
    for (int r = lane; r < n_leaves; r += 32)
      if (leaf_node[r] == node && lp[(size_t)r * POSITION_WORDS + 8] == pos.state) slot = r;
    for (int off = 16; off > 0; off >>= 1) slot = max(slot, __shfl_xor_sync(FULL, slot, off));
    bool terminal = false;
    double tv = P.draw_penalty;
    if (slot >= 0) {
      if (pos_halfmove(pos) >= 8) {
        int rep = 0;
        if (lane == 0) rep = leaf_is_fivefold(E, g, depth, cur_key) ? 1 : 0;
        terminal = __shfl_sync(FULL, rep, 0) != 0;
      }
    } else {
      warp_leaf_moves(E, P, g, pos, depth, cur_key, s_moves[wib], &terminal, &tv, lane);
    }
    if (terminal) {
      warp_backup(E, g, depth + 1, py_clip_unit(tv), 1, lane);   // mcts.py:747-751: immediately, visible to the rest of the batch
      c_term++;
      continue;
    }
    // sample {board, node, path}.  A row is shared only by samples with the same node AND the same board: a transposition-table node
    // can be reached with different clocks (not part of the key, but part of the planes), and the reference evaluates every sample's
    // own board (mcts.py:571-583)
    if (slot < 0) {
      slot = n_leaves++;
      if (lane == 0) {
        leaf_node[slot] = node;
        leaf_first[slot] = n_samples;
        store_position(E.ml_leaf_pos + ((size_t)g * E.ml_cap + slot) * POSITION_WORDS, pos);
      }
    }
    int* sp = E.ml_smp_path + ((size_t)g * E.ml_cap + n_samples) * E.max_depth;
    for (int i = lane; i <= depth; i += 32) sp[i] = path[i];
    if (lane == 0) {
      smp_leaf[n_samples] = slot;
      smp_len[n_samples] = depth + 1;
    }
    n_samples++;
    __syncwarp();
  }
  if (lane == 0) {
    E.ml_n_samples[g] = n_samples;
    E.ml_n_leaves[g] = n_leaves;
    E.jit_cursor[g] = jcur;
    E.pend_flags[g] = 0;
    E.pend_count[g] = 0;
    atomicAdd(&E.counters[CTR_SIMS], (unsigned long long)batch_n);
    atomicAdd(&E.counters[CTR_TERMINAL_SIMS], c_term);
    atomicAdd(&E.counters[CTR_CHILDREN_SCANNED], c_scanned);
    atomicAdd(&E.counters[CTR_PATH_NODES], c_path);
    atomicAdd(&E.counters[CTR_TT_HOPS], c_hops);
    atomicAdd(&E.counters[CTR_NN_EVALS], (unsigned long long)n_leaves);
    atomicAdd(&E.counters[CTR_LEAF_SAMPLES], (unsigned long long)n_samples);
  }
}

// row_base[g] = sum of ml_n_leaves[0..g), row_base[G] = total: one block, G up to a few 10^4
__global__ void __launch_bounds__(1024) multi_scan_kernel(EngineView E) {
  __shared__ int s_part[1024];
  const int t = threadIdx.x, per = (E.G + 1023) / 1024;
  const int lo = t * per, hi = min(E.G, lo + per);
  int sum = 0;
  for (int g = lo; g < hi; ++g) sum += E.ml_n_leaves[g];
  s_part[t] = sum;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    int v = t >= off ? s_part[t - off] : 0;
    __syncthreads();
    s_part[t] += v;
    __syncthreads();
  }
  int run = s_part[t] - sum;
  for (int g = lo; g < hi; ++g) {
    E.ml_row_base[g] = run;
    run += E.ml_n_leaves[g];
  }
  if (t == 1023) E.ml_row_base[E.G] = s_part[1023];
}

// encode_board of the collected leaves of games [g0, g1): one warp per (game, slot).  mode 0: compact rows, row = row_base[g] + leaf slot
// - row0; mode 1: dense per leaf, row = (g - g0) * ml_cap + leaf slot; mode 2: one row per SAMPLE, row = (g - g0) * ml_cap + sample
__global__ void __launch_bounds__(TREE_THREADS)
multi_encode_kernel(EngineView E, int g0, int g1, int row0, int mode, float* __restrict__ planes, int row_cap) {
  const int lane = threadIdx.x & 31;
  const long long w = (long long)blockIdx.x * TREE_WARPS + (threadIdx.x >> 5);
  const int g = g0 + (int)(w / E.ml_cap), r = (int)(w % E.ml_cap);
  if (g >= g1 || r >= (mode == 2 ? E.ml_n_samples[g] : E.ml_n_leaves[g])) return;
  if (row_cap > 0 && E.ml_row_base[g + 1] - row0 > row_cap) return;   // this game's rows do not fit the evaluator batch: a later chunk
  const int leaf = mode == 2 ? E.ml_smp_leaf[(size_t)g * E.ml_cap + r] : r;
  const Position pos = load_position(E.ml_leaf_pos + ((size_t)g * E.ml_cap + leaf) * POSITION_WORDS);
  const size_t row = mode == 0 ? (size_t)(E.ml_row_base[g] + r - row0) : (size_t)(g - g0) * E.ml_cap + r;
  warp_write_planes(pos, planes + row * (19 * 64), lane);
}

// Samples of games [g0, g1) in collection order (mcts.py:654-670): expand + register if the node is still a leaf, back up.
// Row addressing: per_sample == 0: logits / values row of leaf slot r of game g = ml_row_base[g] + r - row0 (compact rows);
//                 per_sample == 1: one row per SAMPLE, game g's rows start at (g - g0) * ml_cap: the expansion reads the row of the
//                 first sample that reached the leaf, every sample backs up the value of its own row (what the reference's zip over
//                 (sample, policy, value) does with an arbitrary backend).
__global__ void __launch_bounds__(TREE_THREADS)
search_expand_backup_multi_kernel(EngineView E, int g0, int g1, const float* __restrict__ logits, int logits_stride, const float* __restrict__ values,
                                  int row0, int per_sample, int row_cap) {
  __shared__ ExpandSmem s_x[TREE_WARPS];
  __shared__ u16 s_moves[TREE_WARPS][MAX_MOVES];
  __shared__ u16 s_idx[TREE_WARPS][MAX_MOVES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = g0 + blockIdx.x * TREE_WARPS + wib;
  if (g >= g1 || !E.active[g]) return;
  const int n_samples = E.ml_n_samples[g];
  if (n_samples <= 0) return;
  if (row_cap > 0 && E.ml_row_base[g + 1] - row0 > row_cap) return;   // not part of this evaluator batch (samples stay pending)
  const SearchParams& P = *E.params;
  const size_t nb = (size_t)g * E.max_nodes;
  const int* smp_leaf = E.ml_smp_leaf + (size_t)g * E.ml_cap;
  const int* smp_len = E.ml_smp_len + (size_t)g * E.ml_cap;
  const int* leaf_node = E.ml_leaf_node + (size_t)g * E.ml_cap;
  const int* leaf_first = E.ml_leaf_first + (size_t)g * E.ml_cap;
  const long long base = per_sample ? (long long)(g - g0) * E.ml_cap : (long long)E.ml_row_base[g] - row0;
  for (int s = 0; s < n_samples;) {
    const int r = smp_leaf[s];
    const int node = leaf_node[r];
    if (E.node_first[nb + node] < 0) {   // `not node.is_expanded()` (mcts.py:657)
      const Position pos = load_position(E.ml_leaf_pos + ((size_t)g * E.ml_cap + r) * POSITION_WORDS);
      int chk = 0;
      int k = warp_generate_legal_moves(pos, s_moves[wib], &chk, lane);
      if (k > MAX_MOVES) k = MAX_MOVES;
      const int wtm = pos_turn(pos);
      for (int j = lane; j < k; j += 32) s_idx[wib][j] = (u16)policy_index(s_moves[wib][j], wtm);
      __syncwarp();
      const long long lrow = base + (per_sample ? leaf_first[r] : r);
      if (k > 0) warp_expand(E, P, g, node, pos, s_moves[wib], s_idx[wib], k, logits + (size_t)lrow * logits_stride, true, false, s_x[wib], lane);
      if (E.rc_slots && smp_len[s] == 2)
        warp_record_root_child(E, g, E.ml_leaf_pos + ((size_t)g * E.ml_cap + r) * POSITION_WORDS, logits + (size_t)lrow * logits_stride,
                               values[lrow], lane);
    }
    // Consecutive samples with the same leaf row and the same path (the common case: a mini-batch mostly repeats one path) back the same
    // value up the same nodes: `run` sequential backups collapse into one pass that performs the same `run` additions per node in the same
    // order (backup_repeated), since nothing else touches those nodes in between.  Rows per sample may carry different values: no grouping.
    const int len = smp_len[s];
    const int* ps = E.ml_smp_path + ((size_t)g * E.ml_cap + s) * E.max_depth;
    int run = 1;
    if (!per_sample) {
      while (s + run < n_samples && smp_leaf[s + run] == r && smp_len[s + run] == len) {
        const int* pn = E.ml_smp_path + ((size_t)g * E.ml_cap + s + run) * E.max_depth;
        bool diff = false;
        for (int i = lane; i < len; i += 32) diff |= ps[i] != pn[i];
        if (__any_sync(FULL, diff)) break;
        ++run;
      }
    }
    float vf = values[base + (per_sample ? s : r)];
    vf = fminf(fmaxf(vf, -1.0f), 1.0f);   // float(np.clip(value, -1, 1)), mcts.py:668
    warp_backup_path(E, g, ps, len, py_clip_unit((double)vf), run, lane);
    s += run;
  }
  if (lane == 0) {
    E.ml_n_samples[g] = 0;
    E.ml_n_leaves[g] = 0;
  }
}

}  // namespace m0
