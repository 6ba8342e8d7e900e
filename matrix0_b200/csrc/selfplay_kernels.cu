// Device-resident self-play game loop: the per-ply part of azchess/selfplay/internal.py:382-600 for
// thousands of games at once (one warp per game).  After a search finishes, one launch samples the
// move from the visit counts (sample_move_from_counts, :690-735), applies the resign rule (:507-536),
// pushes the move, decides whether the game continues (board.is_game_over() / should_adjudicate_draw,
// draw.py:31-41 / max_game_len, :382-384), records finished games and restarts their slots from the
// start position with `opening_random_plies` uniformly random legal moves (:371-379).
#include "engine.cuh"
#include "selfplay.cuh"
#include "movegen_warp.cuh"

namespace m0 {

static constexpr int SP_WARPS = 4;
static constexpr unsigned FULLM = 0xFFFFFFFFu;

__device__ __forceinline__ double sp_uniform(u64& rng) {
  rng = mix64(rng + 0x9E3779B97F4A7C15ull);
  return (double)(rng >> 11) * (1.0 / 9007199254740992.0);
}

__device__ __forceinline__ Position start_position() {
  Position p;
  p.pawns = 0x00FF00000000FF00ull; p.knights = 0x4200000000000042ull; p.bishops = 0x2400000000000024ull;
  p.rooks = 0x8100000000000081ull; p.queens = 0x0800000000000008ull; p.kings = 0x1000000000000010ull;
  p.occ_w = 0x000000000000FFFFull; p.occ_b = 0xFFFF000000000000ull;
  p.state = pack_state(1, CR_WK | CR_WQ | CR_BK | CR_BQ, EP_NONE, 0, 1);
  return p;
}

// occurrences of `key` among the positions since the last irreversible move (game history only)
__device__ int hist_occurrences(const EngineView& E, int g, const Key128& key) {
  const Key128* hk = E.hist_key + (size_t)g * E.hist_cap;
  const u8* hi = E.hist_irrev + (size_t)g * E.hist_cap;
  int c = 0;
  for (int i = E.hist_len[g] - 1; i >= 0; --i) {
    if (hi[i]) break;
    if (key_eq(hk[i], key)) ++c;
  }
  return c;
}

enum { END_NONE = 0, END_CHECKMATE = 1, END_STALEMATE = 2, END_INSUFFICIENT = 3, END_FIFTY = 4, END_REPETITION = 5,
       END_MAX_LEN = 6, END_RESIGN = 7, END_ADJUDICATED = 8 };

// The heuristic half of should_adjudicate_draw (draw.py:43-82; the standard rules above it are game_end_reason): after min_plies
// moves, fewer than min_unique different moves among the last `window`, a halfmove clock at the cap, or little material left.
__device__ bool draw_heuristics(const EngineView& E, const SelfPlayState& S, int g, const Position& pos, int lane) {
  const SelfPlayParams& P = *S.params;
  if (!P.draw_enabled) return false;
  const int L = E.hist_len[g];                       // len(moves)
  if (L < P.draw_min_plies) return false;
  if (P.draw_window > 0 && P.draw_min_unique > 0 && L >= P.draw_window) {
    const u16* mv = S.hist_move + (size_t)g * E.hist_cap + (L - P.draw_window);
    int unique = 0;
    for (int i = lane; i < P.draw_window; i += 32) {  // len(set(str(m) for m in recent)): a move is new if no earlier one equals it
      bool seen = false;
      for (int j = 0; j < i; ++j) seen |= (mv[j] == mv[i]);
      unique += seen ? 0 : 1;
    }
    for (int off = 16; off > 0; off >>= 1) unique += __shfl_xor_sync(FULLM, unique, off);
    if (unique < P.draw_min_unique) return true;
  }
  if (P.draw_halfmove_cap && pos_halfmove(pos) >= P.draw_halfmove_cap) return true;
  if (P.draw_material_threshold > 0) {
    const u64 occ = pos.occ_w | pos.occ_b;
    const int material = popcnt(pos.pawns & occ) + 3 * popcnt(pos.knights & occ) + 3 * popcnt(pos.bishops & occ) +
                         5 * popcnt(pos.rooks & occ) + 9 * popcnt(pos.queens & occ);
    if (material <= P.draw_material_threshold) return true;
  }
  return false;
}

// Does the game end at `pos` before another search?  (warp-cooperative; s_moves = this warp's scratch)
//   board.is_game_over()                                      internal.py:382
//   should_adjudicate_draw (heuristics disabled by default)   draw.py:31-41
// which together equal board.is_game_over(claim_draw=True) plus stalemate.
__device__ int game_end_reason(const EngineView& E, int g, const Position& pos, u16* s_moves, int lane) {
  int in_check = 0;
  int n_moves = warp_generate_legal_moves(pos, s_moves, &in_check, lane);
  if (n_moves > MAX_MOVES) n_moves = MAX_MOVES;
  if (n_moves == 0) return in_check ? END_CHECKMATE : END_STALEMATE;
  if (is_insufficient_material(pos)) return END_INSUFFICIENT;
  const int hm = pos_halfmove(pos);
  if (hm >= 100) return END_FIFTY;  // is_fifty_moves() (and is_seventyfive_moves at 150)
  bool epl;
  const Key128 key = position_key(pos, &epl);
  // is_repetition(3) / first half of can_claim_threefold_repetition: the position occurred twice before
  int prev = 0;
  if (hm >= 4) {
    if (lane == 0) prev = hist_occurrences(E, g, key);
    prev = __shfl_sync(FULLM, prev, 0);
    if (prev >= 2) return END_REPETITION;
  }
  // claims that need a look at the replies: a legal move after which the fifty-move rule or a
  // third occurrence holds (can_claim_fifty_moves at clock 99, second half of can_claim_threefold)
  const bool check_fifty = hm >= 99, check_rep = hm >= 3;
  if (check_fifty || check_rep) {
    int hit = 0;
    for (int j = lane; j < n_moves; j += 32) {
      Position c = pos;
      PushInfo info = push_move(c, s_moves[j]);
      const bool irreversible = info.zeroing || info.reduced_castling || epl;
      if (check_rep && !irreversible) {
        Key128 ck = position_key(c);
        // transpositions = {current position} + history since the last irreversible move
        int occ = hist_occurrences(E, g, ck) + (key_eq(ck, key) ? 1 : 0);
        if (occ >= 2) hit |= 1;
      }
      if (check_fifty && !info.zeroing) {
        Move tmp[MAX_MOVES];
        if (generate_legal_moves(c, tmp) > 0) hit |= 2;
      }
    }
    hit = __reduce_or_sync(FULLM, hit);
    if (hit & 2) return END_FIFTY;
    if (hit & 1) return END_REPETITION;
  }
  return END_NONE;
}

__device__ void append_history(const EngineView& E, const SelfPlayState& S, int g, const Key128& key, bool irrev, Move mv) {
  int L = E.hist_len[g];
  if (L >= E.hist_cap) {
    E.status[g] |= ST_HIST_OVERFLOW;
    return;
  }
  S.hist_move[(size_t)g * E.hist_cap + L] = mv;
  E.hist_key[(size_t)g * E.hist_cap + L] = key;
  E.hist_irrev[(size_t)g * E.hist_cap + L] = irrev ? 1 : 0;
  E.hist_len[g] = L + 1;
}

// take one game from the start budget (selfplay_worker plays exactly `games` games, internal.py:326): false -> the slot goes idle
__device__ bool take_start_budget(const EngineView& E, const SelfPlayState& S, int g, int lane) {
  int ok = 1;
  if (lane == 0) {
    if (*S.start_budget < (1 << 30)) {
      int old = atomicSub(S.start_budget, 1);
      if (old <= 0) { atomicAdd(S.start_budget, 1); ok = 0; }
    }
    if (!ok) {
      E.active[g] = 0;
      E.root_node[g] = -1;
      E.pend_flags[g] = 0;
      E.pend_count[g] = 0;
    }
  }
  return __shfl_sync(FULLM, ok, 0) != 0;
}

// start a fresh game in slot g: start position + opening_random_plies uniformly random legal moves
__device__ void start_game(const EngineView& E, const SelfPlayState& S, int g, u16* s_moves, int lane, u64& rng) {
  Position pos = start_position();
  if (lane == 0) {
    E.hist_len[g] = 0;
    S.ply[g] = 0;
    S.consec_bad[g] = 0;
    S.recent_n[g] = 0;
    S.ent_n[g] = 0;
    S.ent_sum[g] = 0.0;
    S.last_value[g] = 0.0;
  }
  __syncwarp();
  for (int k = 0; k < S.params->opening_random_plies; ++k) {
    int chk = 0;
    int n = warp_generate_legal_moves(pos, s_moves, &chk, lane);
    if (n == 0 || is_insufficient_material(pos)) break;  // board.is_game_over() (no repetition possible this early)
    if (n > MAX_MOVES) n = MAX_MOVES;
    int pick = 0;
    if (lane == 0) pick = (int)(sp_uniform(rng) * n);
    pick = __shfl_sync(FULLM, pick, 0);
    if (pick >= n) pick = n - 1;
    const Move mv = s_moves[pick];
    bool epl;
    const Key128 key = position_key(pos, &epl);
    PushInfo info = push_move(pos, mv);
    if (lane == 0) append_history(E, S, g, key, info.zeroing || info.reduced_castling || epl, mv);
    __syncwarp();
  }
  if (lane == 0) {
    store_position(E.root_pos + (size_t)g * POSITION_WORDS, pos);
    E.active[g] = 1;
    E.root_node[g] = -1;
    E.pend_flags[g] = 0;
    E.pend_count[g] = 0;
    S.games_started[g] += 1;
  }
  __syncwarp();
}

// (re)start every game slot flagged in S.need_start (or all of them when `all` != 0)
__global__ void __launch_bounds__(SP_WARPS * 32)
selfplay_start_kernel(EngineView E, SelfPlayState S, int all, unsigned long long step) {
  __shared__ u16 s_moves[SP_WARPS][MAX_MOVES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * SP_WARPS + wib;
  if (g >= E.G) return;
  if (!all && !S.need_start[g]) return;
  u64 rng = mix64(S.params->seed ^ mix64(step * 0xA0761D6478BD642Full + (u64)(g + 1)));
  if (take_start_budget(E, S, g, lane)) start_game(E, S, g, s_moves[wib], lane, rng);
  if (lane == 0) S.need_start[g] = 0;
}

// does the current root end the game before any search?  (loop condition of internal.py:382-384)
// Finished games are recorded and restarted in place.  Returns through S.need_search[g] whether slot g
// holds a position to search next.
__device__ void settle_game(const EngineView& E, const SelfPlayState& S, int g, u16* s_moves, int lane, u64& rng) {
  for (int guard = 0; guard < 4; ++guard) {
    Position pos = load_position(E.root_pos + (size_t)g * POSITION_WORDS);
    int reason = game_end_reason(E, g, pos, s_moves, lane);
    const int ply = S.ply[g];
    if (reason == END_NONE && ply >= S.params->max_game_len) reason = END_MAX_LEN;
    if (reason == END_NONE && draw_heuristics(E, S, g, pos, lane)) reason = END_ADJUDICATED;
    if (reason == END_NONE) return;
    // z from White's point of view: game_result() (internal.py:738-750) or, where no formal result exists (length cap, heuristic
    // adjudication), the last search value -- 0.0 before the first search (:587-599)
    double z = 0.0;
    if (reason == END_CHECKMATE) z = pos_turn(pos) ? -1.0 : 1.0;
    else if (reason == END_MAX_LEN || reason == END_ADJUDICATED) z = ply > 0 ? S.last_value[g] : 0.0;
    if (lane == 0) {
      unsigned slot = atomicAdd(S.finished_count, 1u);
      FinishedGame* f = S.finished + (slot % S.finished_cap);
      f->game = g;
      f->plies = ply;
      f->z = (float)z;
      f->reason = reason;
      f->avg_entropy = (float)(S.ent_sum[g] / (double)(S.ent_total[g] > 0 ? S.ent_total[g] : 1));
      atomicAdd(&E.counters[CTR_GAMES_FINISHED], 1ull);
      S.ent_total[g] = 0;
    }
    __syncwarp();
    if (!take_start_budget(E, S, g, lane)) return;
    start_game(E, S, g, s_moves, lane, rng);
  }
}

// one ply for every game: sample the move from the finished search, resign rule, push, settle.
// GUMBEL: the move, the search value and the policy entropy come from gumbel_result_kernel (GB) instead of the visit counts; the
// temperature schedule and the visit sampling do not apply (the Gumbel draw is the sampling).
template <bool GUMBEL>
__global__ void __launch_bounds__(SP_WARPS * 32)
selfplay_advance_kernel(EngineView E, SelfPlayState S, unsigned long long step, u16* __restrict__ out_move, GumbelView GB) {
  __shared__ u16 s_moves[SP_WARPS][MAX_MOVES];
  __shared__ float s_w[SP_WARPS][MAX_MOVES];
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int g = blockIdx.x * SP_WARPS + wib;
  if (g >= E.G || !E.active[g]) return;
  const SelfPlayParams& P = *S.params;
  const size_t nb = (size_t)g * E.max_nodes;
  u64 rng = mix64(P.seed ^ mix64(step * 0xD6E8FEB86659FD93ull + (u64)(g + 1) * 0x9E3779B97F4A7C15ull));
  const int root = E.root_node[g];
  Position pos = load_position(E.root_pos + (size_t)g * POSITION_WORDS);
  if (root < 0) {  // nothing was searched (terminal root): settle and return
    settle_game(E, S, g, s_moves[wib], lane, rng);
    return;
  }
  const int fc = E.node_first[nb + root];
  const int nc = fc < 0 ? 0 : E.node_nchild[nb + root];
  int pick = 0;
  double entropy = 0.0, v = 0.0;
  if constexpr (GUMBEL) {
    pick = GB.choice[g];
    entropy = GB.entropy[g];
    v = GB.value[g];
    if (pick < 0 || pick >= nc) {   // no result for this search
      settle_game(E, S, g, s_moves[wib], lane, rng);
      return;
    }
  } else {
    // temperature schedule by full-move number (internal.py:386-394)
    double temperature = P.temperature_end;
    if (P.temperature_moves > 0) {
      int mn = pos_fullmove(pos);
      double t = (double)(mn < P.temperature_moves ? mn : P.temperature_moves) / (double)P.temperature_moves;
      temperature = P.temperature_start + (P.temperature_end - P.temperature_start) * t;
    }
    if (P.argmax_after_plies >= 0) temperature = S.ply[g] < P.argmax_after_plies ? P.temperature_start : 0.0;   // arena.py:75-91
    // visit counts -> move (internal.py:690-735)
    long long total = 0;
    int best_n = -1, best_j = 0;
    for (int j = lane; j < nc; j += 32) {
      int n = E.node_n[nb + fc + j];
      total += n;
      if (n > best_n) { best_n = n; best_j = j; }
    }
    for (int off = 16; off > 0; off >>= 1) {
      total += __shfl_xor_sync(FULLM, total, off);
      int on = __shfl_xor_sync(FULLM, best_n, off), oj = __shfl_xor_sync(FULLM, best_j, off);
      if (on > best_n || (on == best_n && oj < best_j)) { best_n = on; best_j = oj; }
    }
    pick = best_j;
    // the one np.random draw sample_move_from_counts makes (np.random.choice): supplied by the caller or from the device generator
    const double u01 = S.uniforms ? S.uniforms[g] : sp_uniform(rng);
    if (P.low_visit_threshold > 0 && best_n < P.low_visit_threshold && temperature < 0.8) temperature = 0.8;   // internal.py:419-425
    if (total > 0) {
      // policy entropy of pi = n / total, pi clipped to [1e-12, 1] over all 4672 entries (internal.py:433-441)
      double e = 0.0;
      for (int j = lane; j < nc; j += 32) {
        double p = (double)(float)((double)E.node_n[nb + fc + j] / (double)total);
        if (p < 1e-12) p = 1e-12;
        e -= p * log(p);
      }
      for (int off = 16; off > 0; off >>= 1) e += __shfl_xor_sync(FULLM, e, off);
      entropy = e - (double)(POLICY_SIZE - nc) * (1e-12 * log(1e-12));
      if (temperature >= 1e-3) {
        // visits.astype(float32) ** (1 / T), float32 pairwise sum, float32 divide; np.random.choice(k, p): p as float64, cdf = cumsum(p),
        // cdf /= cdf[-1], index = searchsorted(cdf, u, 'right') (internal.py:713-734)
        const float inv_t = (float)(1.0 / temperature);
        for (int j = lane; j < nc; j += 32) s_w[wib][j] = powf((float)E.node_n[nb + fc + j], inv_t);
        __syncwarp();
        if (lane == 0) {
          const float sum = np_pairwise_sum_f32(s_w[wib], nc);
          if (sum > 0.0f && isfinite(sum)) {
            double last = 0.0;
            for (int j = 0; j < nc; ++j) last = d_add(last, (double)f_div(s_w[wib][j], sum));
            double acc = 0.0;
            int sel = nc - 1;
            for (int j = 0; j < nc; ++j) {
              acc = d_add(acc, (double)f_div(s_w[wib][j], sum));
              if (d_div(acc, last) > u01) { sel = j; break; }
            }
            pick = sel;
          } else if (!(sum <= 0.0f)) {
            // the float32 sum overflowed: visit_dist /= inf leaves NaNs and the reference falls back to np.random.choice(legal_moves)
            pick = (int)(u01 * nc);
            if (pick >= nc) pick = nc - 1;
          } else {
            pick = (int)(u01 * nc);   // visit_sum <= 0: uniform over the legal moves (:717-722)
            if (pick >= nc) pick = nc - 1;
          }
        }
        pick = __shfl_sync(FULLM, pick, 0);
      }
    } else if (nc > 0) {
      if (lane == 0) pick = (int)(u01 * nc);  // uniform over legal moves (internal.py:701-707)
      pick = __shfl_sync(FULLM, pick, 0);
      if (pick >= nc) pick = nc - 1;
    }
    if (nc == 0) {  // cannot happen for a searched root; be safe
      settle_game(E, S, g, s_moves[wib], lane, rng);
      return;
    }
    const int rn = E.node_n[nb + root];
    v = rn > 0 ? E.node_q[nb + root] : 0.0;  // value returned by MCTS.run (mcts.py:504)
  }
  const Move mv = (Move)(E.node_mv[nb + fc + pick] & 0xFFFFu);
  int ply = S.ply[g] + 1;                               // len(states) after the append (internal.py:447)
  bool resigned = false;
  if (lane == 0) {
    S.ply[g] = ply;
    S.last_value[g] = v;
    S.ent_sum[g] += entropy;
    S.ent_total[g] += 1;
    // sliding windows for the resign rule (internal.py:437-441, :507-536)
    const int W = P.resign_window > 0 ? (P.resign_window < SP_WINDOW ? P.resign_window : SP_WINDOW) : 1;
    float* re = S.recent_ent + (size_t)g * SP_WINDOW;
    int en = S.ent_n[g];
    if (en == W) { for (int i = 1; i < W; ++i) re[i - 1] = re[i]; en = W - 1; }
    re[en++] = (float)entropy;
    S.ent_n[g] = en;
    if (P.resign_threshold > -1.0 && ply >= P.min_resign_plies) {
      float* rv = S.recent_val + (size_t)g * SP_WINDOW;
      int vn = S.recent_n[g];
      if (vn == W) { for (int i = 1; i < W; ++i) rv[i - 1] = rv[i]; vn = W - 1; }
      rv[vn++] = (float)v;
      S.recent_n[g] = vn;
      int cb = (v < P.resign_threshold) ? S.consec_bad[g] + 1 : 0;
      S.consec_bad[g] = cb;
      const int need = (W / 2) > 2 ? (W / 2) : 2;
      bool stable_bad = false, low_unc = false;
      if (vn >= need) {
        double s = 0.0;
        for (int i = 0; i < vn; ++i) s += rv[i];
        stable_bad = (s / vn) < (P.resign_threshold + P.resign_value_margin);
      }
      if (en >= need) {
        double s = 0.0;
        for (int i = 0; i < en; ++i) s += re[i];
        low_unc = (s / en) < P.resign_min_entropy;
      }
      resigned = cb >= P.resign_consecutive_bad && (stable_bad || low_unc);
    }
    atomicAdd(&E.counters[CTR_POSITIONS_PLAYED], 1ull);
    if (out_move) out_move[g] = mv;
  }
  resigned = __shfl_sync(FULLM, resigned ? 1 : 0, 0) != 0;
  if (resigned) {
    if (lane == 0) {
      unsigned slot = atomicAdd(S.finished_count, 1u);
      FinishedGame* f = S.finished + (slot % S.finished_cap);
      f->game = g;
      f->plies = ply;
      f->z = pos_turn(pos) ? -1.0f : 1.0f;  // internal.py:530
      f->reason = END_RESIGN;
      f->avg_entropy = (float)(S.ent_sum[g] / (double)(S.ent_total[g] > 0 ? S.ent_total[g] : 1));
      atomicAdd(&E.counters[CTR_GAMES_FINISHED], 1ull);
      S.ent_total[g] = 0;
    }
    __syncwarp();
    if (!take_start_budget(E, S, g, lane)) return;
    start_game(E, S, g, s_moves[wib], lane, rng);
    settle_game(E, S, g, s_moves[wib], lane, rng);
    return;
  }
  // board.push(move) with the move-stack bookkeeping (internal.py:538-539)
  bool epl;
  const Key128 key = position_key(pos, &epl);
  PushInfo info = push_move(pos, mv);
  if (lane == 0) {
    append_history(E, S, g, key, info.zeroing || info.reduced_castling || epl, mv);
    store_position(E.root_pos + (size_t)g * POSITION_WORDS, pos);
    E.root_node[g] = -1;
  }
  __syncwarp();
  settle_game(E, S, g, s_moves[wib], lane, rng);
}

template __global__ void selfplay_advance_kernel<false>(EngineView, SelfPlayState, unsigned long long, u16*, GumbelView);
template __global__ void selfplay_advance_kernel<true>(EngineView, SelfPlayState, unsigned long long, u16*, GumbelView);

// drop every game's tree (nodes + transposition table) but keep positions and history: the
// per-move equivalent of constructing a fresh MCTS (see DESIGN.md, reference quirk Q12)
__global__ void clear_trees_kernel(EngineView E) {
  const int g = blockIdx.y;
  if (g >= E.G) return;
  const size_t base = (size_t)g * E.tt_cap;
  uint4* lo = reinterpret_cast<uint4*>(E.tt_lo + base);
  uint4* hi = reinterpret_cast<uint4*>(E.tt_hi + base);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < E.tt_cap / 2; i += gridDim.x * blockDim.x) {
    lo[i] = make_uint4(0, 0, 0, 0);
    hi[i] = make_uint4(0, 0, 0, 0);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    E.node_count[g] = 0;
    E.tt_count[g] = 0;
    E.root_node[g] = -1;
    E.pend_flags[g] = 0;
    E.pend_count[g] = 0;
  }
}

}  // namespace m0
