// Device-resident search engine state: thousands of concurrent games, each a structure-of-arrays
// MCTS tree (one node per slot), a per-game transposition table and the position-key history
// needed for repetition detection.  One warp owns one game in every tree kernel.
//
// Reference objects mirrored (azchess/mcts.py): Node (:120-133) -> the node_* arrays,
// MCTS.tt (:302, OrderedDict key -> Node, last writer wins :1255) -> the tt_* arrays,
// MCTSConfig (:61-117) -> SearchParams, board.move_stack/_stack -> hist_* (+ path_* while searching).
#pragma once
#include "m0_common.cuh"
#include "search_math.cuh"

namespace m0 {

// pend_flags bits
enum { PEND_ACTIVE = 1, PEND_EXPAND = 2, PEND_REGISTER = 4, PEND_SET_Q = 8, PEND_ROOT = 16 };
// status bits (sticky, per game)
enum { ST_NODE_OVERFLOW = 1, ST_TT_OVERFLOW = 2, ST_DEPTH_CAP = 4, ST_HIST_OVERFLOW = 8, ST_STREAM_EXHAUSTED = 16 };
// counters
enum { CTR_SIMS = 0, CTR_TERMINAL_SIMS, CTR_NN_EVALS, CTR_EXPANSIONS, CTR_TT_HOPS, CTR_CHILDREN_SCANNED,
       CTR_PATH_NODES, CTR_CHILDREN_CREATED, CTR_GAMES_FINISHED, CTR_POSITIONS_PLAYED, CTR_NOISY_EXPANSIONS, CTR_LEAF_SAMPLES,
       CTR_ROOT_REUSED, CTR_COUNT = 16 };
static constexpr int REUSE_MAX_SLOTS = 64;   // stored root children per game (the root's warp compares 32 at a time)

struct SearchParams {
  double fpu_reduction;     // mcts.py:868-869
  double draw_penalty;      // mcts.py:1227-1228
  double jitter;            // selection_jitter, or 0.001 when configured 0 (mcts.py:893-897)
  double dirichlet_alpha;   // mcts.py:960
  double dirichlet_frac;    // mcts.py:961
  int jitter_on;            // 0 = deterministic parity mode (equivalent to random.random() == 0.5)
  int no_instant_backtrack; // mcts.py:883
  int legal_softmax;        // mcts.py:158
  int entropy_noise;        // mcts.py:179
  int value_from_white;     // mcts.py:1184 (root evaluation only, SURVEY Q10)
  int cpuct_len;            // entries of the per-depth cpuct table (mcts.py:927-944)
  unsigned long long seed;
  int max_children;         // _prune_children, mcts.py:806-826 (0 = off)
  int raw_logit_priors;     // SURVEY Q3: non-root leaves get logits[idx] / sum(logits[idx]) (_expand_with_legal_priors, mcts.py:227-256, :697-703)
  double min_child_prior;   // mcts.py:817-818 (0 = off)
  double virtual_loss;      // mcts.py:889-890, applied per in-flight selection of an edge when virtual_loss_on
  int virtual_loss_on;      // the reference's in-flight marking (_select's inflight_counts, :889-890 / :922-923), which no caller of the
                            // reference passes (SURVEY Q2b): switched on it spreads the simulations of a mini-batch over distinct leaves
  int pad_;
};

struct EngineView {
  int G, max_nodes, tt_cap, max_depth, hist_cap;
  // game state
  u64* root_pos;          // [G][9]
  Key128* root_key;       // [G]
  u8* root_ep_legal;      // [G]
  int* root_node;         // [G]
  u8* active;             // [G]
  Key128* hist_key;       // [G][hist_cap]  key of the position BEFORE game ply i
  u8* hist_irrev;         // [G][hist_cap]  Board.is_irreversible(move i) evaluated on that position
  int* hist_len;          // [G]
  // nodes [G][max_nodes]
  double* node_prior;
  double* node_w;
  double* node_q;
  int* node_n;
  int* node_first;        // first child index, -1 = not expanded
  int* node_creator;      // Node.parent (the node that created it), -1 = None
  u32* node_mv;           // move | policy_idx << 16 ; move 0xFFFF = None
  u16* node_nchild;
  int* node_count;        // [G]
  // transposition table [G][tt_cap], open addressing, (0,0) = empty
  u64* tt_lo;
  u64* tt_hi;
  int* tt_val;
  int* tt_count;          // [G]
  // per-step scratch
  int* path_node;         // [G][max_depth]
  Key128* path_key;       // [G][max_depth]
  u8* path_irrev;         // [G][max_depth]  irreversibility of the move path[d] -> path[d+1]
  int* path_len;          // [G]
  u64* leaf_pos;          // [G][9]
  u16* leaf_moves;        // [G][256]
  u16* leaf_idx;          // [G][256]
  int* leaf_n;            // [G]
  int* pend_node;         // [G]
  int* pend_count;        // [G] number of backups owed to the pending leaf
  int* pend_flags;        // [G]
  int* status;            // [G]
  unsigned long long* counters;  // [CTR_COUNT]
  const SearchParams* params;
  const double* cpuct;    // [cpuct_len]
  // random draws of the stochastic mode: caller-supplied streams (parity: the values random.random() / np.random.normal
  // would have returned, consumed in the reference's order) or, when NULL, a counter-based device generator
  const double* jit_stream;       // [G][jit_stride] uniforms in [0,1)   (mcts.py:893-897)
  const double* nrm_stream;       // [G][nrm_stride] N(0, 0.1) variates  (mcts.py:181)
  long long jit_stride, nrm_stride;
  unsigned long long* jit_cursor; // [G] draws consumed so far
  unsigned long long* nrm_cursor; // [G]
  // as-shipped mini-batches (tree_multi_kernels.cu): every simulation of a batch selects with its own jitter and the
  // distinct leaves each get a network row; allocated by m0_search_multi_enable (ml_cap = 0: not enabled)
  int ml_cap;             // samples per game and batch (>= inference_batch_size)
  int* ml_n_samples;      // [G] non-terminal samples collected by the last select
  int* ml_n_leaves;       // [G] distinct leaf nodes among them
  int* ml_smp_leaf;       // [G][ml_cap] sample -> leaf slot
  int* ml_smp_len;        // [G][ml_cap] path length of the sample
  int* ml_smp_path;       // [G][ml_cap][max_depth] path nodes (root first)
  int* ml_leaf_node;      // [G][ml_cap] leaf slot -> node
  int* ml_leaf_first;     // [G][ml_cap] leaf slot -> first sample that reached it
  u64* ml_leaf_pos;       // [G][ml_cap][9]
  int* ml_row_base;       // [G + 1] exclusive prefix of ml_n_leaves: compact network rows
  u16* node_inflight;     // [G][max_nodes] in-flight selections of an edge child within the current mini-batch (virtual loss)
  double* full_scratch;   // [G][4672] entropy noise over the FULL policy vector (legal_softmax = false, mcts.py:164-186); else NULL
  // network outputs of the root's children, kept for the next move (m0_search_reuse_enable; rc_slots = 0: not enabled).  The next
  // root is the child that was played, and a row's output is a function of its packed position alone, so a stored entry whose
  // position equals the new root is exactly what a second evaluation would return.
  int rc_slots;           // entries per game (<= REUSE_MAX_SLOTS)
  int* rc_fill;           // [G] entries recorded since the last search_begin
  u64* rc_pos;            // [G][rc_slots][9]
  float* rc_logits;       // [G][rc_slots][4672]
  float* rc_value;        // [G][rc_slots] value as the network returned it (before clipping)
  int* rc_src;            // [G] where the root expansion reads its row: entry s -> -1 - s, compact miss row r -> r
  float* rc_miss_planes;  // [G][19][8][8] caller's buffer: planes of the roots found in no entry, in compact rows
  int* rc_miss_count;     // [1] caller's counter: rows written to rc_miss_planes by the last search_begin
};

static constexpr u32 MOVE_NONE = 0xFFFFu;

// ---- transposition table -----------------------------------------------------------------------
__device__ __forceinline__ int tt_get(const EngineView& E, int g, const Key128& k) {
  const size_t base = (size_t)g * E.tt_cap;
  u32 mask = (u32)E.tt_cap - 1;
  u32 h = (u32)k.lo & mask;
  for (int probe = 0; probe < E.tt_cap; ++probe) {
    u64 lo = E.tt_lo[base + h];
    u64 hi = E.tt_hi[base + h];
    if (lo == 0 && hi == 0) return -1;
    if (lo == k.lo && hi == k.hi) return E.tt_val[base + h];
    h = (h + 1) & mask;
  }
  return -1;
}
// self.tt[key] = node : overwrite when present (last writer wins), insert otherwise
__device__ __forceinline__ void tt_put(const EngineView& E, int g, const Key128& k, int node) {
  const size_t base = (size_t)g * E.tt_cap;
  u32 mask = (u32)E.tt_cap - 1;
  u32 h = (u32)k.lo & mask;
  for (int probe = 0; probe < E.tt_cap; ++probe) {
    u64 lo = E.tt_lo[base + h];
    u64 hi = E.tt_hi[base + h];
    if (lo == k.lo && hi == k.hi) { E.tt_val[base + h] = node; return; }
    if (lo == 0 && hi == 0) {
      if (E.tt_count[g] >= E.tt_cap - E.tt_cap / 8) { E.status[g] |= ST_TT_OVERFLOW; return; }
      E.tt_lo[base + h] = k.lo;
      E.tt_hi[base + h] = k.hi;
      E.tt_val[base + h] = node;
      E.tt_count[g] += 1;
      return;
    }
    h = (h + 1) & mask;
  }
  E.status[g] |= ST_TT_OVERFLOW;
}

// The same for many lanes of the game's warp at once, each with a DIFFERENT key (the children of one node are different positions):
// an empty slot is claimed with a compare-and-swap on its low word, so two lanes probing into the same slot cannot both take it.
// A lane that meets a foreign low word just probes on; complete entries are all that later kernels see.
__device__ __forceinline__ void tt_put_concurrent(const EngineView& E, int g, const Key128& k, int node) {
  const size_t base = (size_t)g * E.tt_cap;
  const u32 mask = (u32)E.tt_cap - 1;
  u32 h = (u32)k.lo & mask;
  for (int probe = 0; probe < E.tt_cap; ++probe) {
    const u64 lo = E.tt_lo[base + h];
    if (lo == k.lo && E.tt_hi[base + h] == k.hi) { E.tt_val[base + h] = node; return; }
    if (lo == 0 && E.tt_hi[base + h] == 0) {
      if (atomicAdd(&E.tt_count[g], 0) >= E.tt_cap - E.tt_cap / 8) { atomicOr(&E.status[g], ST_TT_OVERFLOW); return; }
      const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long*>(&E.tt_lo[base + h]), 0ull, (unsigned long long)k.lo);
      if (old == 0ull) {
        E.tt_hi[base + h] = k.hi;
        E.tt_val[base + h] = node;
        atomicAdd(&E.tt_count[g], 1);
        return;
      }
    }
    h = (h + 1) & mask;
  }
  atomicOr(&E.status[g], ST_TT_OVERFLOW);
}

}  // namespace m0
