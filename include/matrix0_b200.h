/* matrix0_b200 -- C ABI of the B200-native self-play search engine.
 *
 * The reference (lukifer23/Matrix0) is pure Python and has no FFI; its seams for this path are the
 * Python duck-types listed in SURVEY.md section 8b.  This header is the boundary a binding for
 * those seams links against: plain pointers and sizes, no torch / C++ types.  Every function
 * returns 0 on success or a negative M0_ERR_* code; m0_last_error() then returns a thread-local,
 * library-owned message.  Unless stated otherwise all buffer pointers are DEVICE pointers supplied
 * by the caller (e.g. torch tensor.data_ptr()); the library never allocates memory the caller
 * sees, never synchronises the host unless the function name ends in _host or _sync, and launches
 * on the `stream` argument (a cudaStream_t passed as void*).  There is no CPU implementation
 * behind any entry point.
 *
 * Devices: a handle (m0_engine, m0_net) lives on the device passed to its *_create.  The entry
 * points that allocate or free (create / destroy / configure / multi_enable) switch to that
 * device themselves and restore the caller's current device before they return; every other
 * entry point launches on the CALLER'S current device and `stream`, which must be the handle's
 * (cudaSetDevice(handle's device) or torch.cuda.device(...) around the call).  Handles of several
 * devices may coexist in one process.
 *
 * Each entry point cites the reference interface it replaces (paths relative to the reference).
 */
#ifndef MATRIX0_B200_H
#define MATRIX0_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define M0_OK 0
#define M0_ERR_CUDA (-1)     /* a CUDA runtime call or launch failed */
#define M0_ERR_ARG (-2)      /* invalid argument */
#define M0_ERR_STATE (-3)    /* call sequence error (e.g. search step without begin) */
#define M0_ERR_CAPACITY (-4) /* node pool / table capacity exhausted */

#define M0_POSITION_WORDS 9  /* packed position: 8 bitboards + state word (csrc/chess_core.cuh) */
#define M0_RAW_WORDS 10      /* raw python-chess record, see m0_positions_pack */
#define M0_MAX_MOVES 256     /* row stride of move / index lists */
#define M0_POLICY_SIZE 4672  /* azchess/encoding.py:51 POLICY_SHAPE = (8, 8, 73) */
#define M0_PLANES 19         /* azchess/encoding.py:11 */

/* ---- library ------------------------------------------------------------------------------ */
const char* m0_last_error(void);
int m0_version(void);
int m0_device_count(void);            /* <= 0: the product cannot run (no CPU path) */
int m0_device_sm_count(int device);
unsigned long long m0_launch_count(void); /* kernel launches issued by the library so far */

/* ---- positions ------------------------------------------------------------------------------
 * Raw record per position (uint64[10]), the public fields of python-chess's chess.Board that the
 * reference reads (encoding.py:22-33, mcts.py:342):
 *   [0..5] pawns, knights, bishops, rooks, queens, kings   [6] occupied_co[WHITE]  [7] occupied_co[BLACK]
 *   [8] castling_rights (rook-square mask)   [9] turn | ep_square<<8 (255 = None) | halfmove_clock<<16 | fullmove_number<<32
 * m0_positions_pack applies Board.clean_castling_rights() and writes packed positions uint64[n][9]. */
int m0_positions_pack(const uint64_t* d_raw, int n, uint64_t* d_pos, void* stream);
/* Synthetic positions for benches/tests: position i = plies_i (hash(seed,i) % (max_plies+1)) uniformly
 * random legal moves from the start position -- batch form of azchess/utils/board.py:7-38. */
int m0_random_playouts(uint64_t* d_pos, int n, uint64_t seed, int max_plies, void* stream);

/* ---- encoding: azchess/encoding.py ------------------------------------------------------------
 * m0_encode_positions is the fused entry point; any output pointer may be NULL.  Planes and / or mask alone run the
 * half-warp-per-position kernel (legal moves as a set, HBM-roofline); a call that asks for the ORDERED lists
 * (d_moves / d_idx / d_counts) runs the thread-per-position kernel with the python-chess ordered generator for all outputs.
 * Both produce identical planes and masks (tests/test_encoding_gpu.py::test_config2_full_size_against_oracle_digests compares them on the
 * bench's 1 Mi synthetic positions, 1,019,010 of them distinct, and 131,072 of those against SHA-256 digests of the oracle's outputs).
 *   d_planes float32[n][19][8][8]   = encode_board          (encoding.py:11-37, row = 7 - rank)
 *   d_mask   uint8[n][4672]         = MoveEncoder.get_legal_actions (encoding.py:243-253)
 *   d_moves  uint16[n][256]         = list(board.legal_moves) in python-chess generation order,
 *                                     packed from | to<<6 | promotion<<12 (mcts.py:140)
 *   d_idx    uint16[n][256]         = move_to_index of each move (encoding.py:113-150)
 *   d_counts int32[n]               = number of legal moves */
int m0_encode_positions(const uint64_t* d_pos, int n, float* d_planes, uint8_t* d_mask, uint16_t* d_moves,
                        uint16_t* d_idx, int32_t* d_counts, void* stream);
int m0_encode_planes(const uint64_t* d_pos, int n, float* d_planes, void* stream);
int m0_legal_mask(const uint64_t* d_pos, int n, uint8_t* d_mask, void* stream);
int m0_legal_moves(const uint64_t* d_pos, int n, uint16_t* d_moves, uint16_t* d_idx, int32_t* d_counts, void* stream);

/* SSL target maps of azchess/ssl_algorithms.py create_enhanced_ssl_targets (:502-535), one position per row as selfplay_worker
 * calls it (internal.py:460-466); float32, plane coordinates (row = 7 - rank); any output may be NULL:
 *   d_piece[n][13][8][8] (_create_piece_targets :537-557)   d_threat[n][8][8] (detect_threats_batch :51-143)
 *   d_pin[n][8][8] (detect_pins_batch :256-346)   d_fork[n][8][8] (detect_forks_batch :348-421)
 *   d_control[n][8][8] in {-1, 0, 1} (calculate_square_control_batch :423-500) */
int m0_ssl_targets(const uint64_t* d_pos, int n, float* d_piece, float* d_threat, float* d_pin, float* d_fork, float* d_control, void* stream);

/* ---- search engine: azchess/mcts.py ------------------------------------------------------------
 * One engine per GPU holds up to max_games concurrent games as GPU-resident structure-of-arrays
 * trees (Node, mcts.py:120-133), a per-game transposition table (MCTS.tt, :302) and the move-stack
 * key history used for repetition detection.  One host thread drives an engine. */
typedef struct m0_engine m0_engine;

/* Device-relevant subset of MCTSConfig (mcts.py:61-117).  cpuct_by_depth[d] = MCTS._cpuct_at(d)
 * (:927-944) evaluated by the caller for d = 0..cpuct_len-1 (deeper plies reuse the last entry).
 * deterministic = 1 reproduces the reference with random.random() == 0.5 and noise off. */
typedef struct m0_search_config {
  double fpu_reduction, draw_penalty, selection_jitter, dirichlet_alpha, dirichlet_frac;
  int deterministic;
  int no_instant_backtrack, legal_softmax, enable_entropy_noise, value_from_white;
  int cpuct_len;
  unsigned long long seed;
  const double* cpuct_by_depth; /* HOST pointer */
  int max_children;        /* MCTS._prune_children (mcts.py:806-826): keep the max_children largest priors; 0 = off */
  int raw_logit_priors;    /* 1 = the reference's direct-model path (no inference backend, legal_softmax): non-root leaves are expanded by
                              Node._expand_with_legal_priors on the RAW logits of the legal moves (mcts.py:697-703, :227-256; SURVEY Q3) */
  double min_child_prior;  /* drop children whose prior is below this (mcts.py:817-818); 0 = off */
  double virtual_loss;     /* MCTSConfig.virtual_loss (mcts.py:75) */
  int virtual_loss_on;     /* 1 = throughput mode: the in-flight marking of MCTS._select (inflight_counts, mcts.py:889-890, :922-923) is applied
                              within every mini-batch of m0_search_select_multi, so its simulations spread over distinct leaves.  The reference
                              ships this code but none of its callers passes inflight_counts (SURVEY Q2b): 0 reproduces the reference. */
  int reserved;
} m0_search_config;

int m0_engine_create(int device, int max_games, int max_nodes, int tt_capacity, int max_depth, int hist_cap, m0_engine** out);
int m0_engine_destroy(m0_engine* e);
long long m0_engine_bytes(const m0_engine* e);
int m0_engine_configure(m0_engine* e, const m0_search_config* cfg, void* stream); /* MCTS.__init__ (mcts.py:270-315) */
int m0_games_reset(m0_engine* e, const int* d_games, int n, void* stream);         /* MCTS.reset (mcts.py:1477-1488) */
/* `board` argument of MCTS.run (mcts.py:318): root positions uint64[n][9] plus, optionally, the move-stack
 * history before each root: positions uint64[n][hist_stride][9], moves uint16[n][hist_stride], lengths int32[n]. */
int m0_games_set_positions(m0_engine* e, const int* d_games, int n, const uint64_t* d_root_pos, const uint64_t* d_hist_pos,
                           const uint16_t* d_hist_moves, const int32_t* d_hist_lens, int hist_stride, void* stream);
/* root position of every game, packed records uint64[G][9] (the state selfplay_worker records before a search, internal.py:447) */
int m0_games_get_positions(m0_engine* e, uint64_t* d_out_pos, void* stream);
/* MCTS.run prologue (mcts.py:336-371): d_info int32[G] bit0 = terminal root (d_value float64[G] = _terminal_value),
 * bit1 = root needs an evaluation (its planes are written to d_planes float32[G][19][8][8]). */
int m0_search_begin(m0_engine* e, float* d_planes, int32_t* d_info, double* d_value, void* stream);
/* one mini-batch of batch_n simulations per game: _collect_leaf_position / _select (mcts.py:742-769, :851-925) */
int m0_search_select(m0_engine* e, int batch_n, float* d_planes, void* stream);
/* Node._expand + _register_children_in_tt + _backpropagate for the pending leaves (mcts.py:135-225, :1330-1346, :946-953);
 * d_logits float32[G][logits_stride >= 4672], d_values float32[G] are the evaluator outputs (infer_np, inference.py:585). */
/* the same with per-game simulation budgets d_sims_left int32[G] (playout-cap randomisation, mcts.py:380-385) */
int m0_search_select_var(m0_engine* e, int batch_cap, int32_t* d_sims_left, float* d_planes, void* stream);
int m0_search_expand_backup(m0_engine* e, const float* d_logits, int logits_stride, const float* d_values, void* stream);
/* MCTS._add_dirichlet (mcts.py:955-992): d_noise float64[G][256] supplied by the caller, or NULL to draw
 * Dirichlet(alpha) on the device; d_apply int32[G] gates games (NULL = all). */
int m0_search_add_dirichlet(m0_engine* e, const double* d_noise, const int32_t* d_apply, void* stream);
int m0_search_pending(m0_engine* e, int32_t* d_flags_out, void* stream);         /* int32[G], 0 = nothing pending */
int m0_search_pending_counts(m0_engine* e, int32_t* d_counts_out, void* stream); /* int32[G] backups owed per pending leaf */
/* MCTS.run results (mcts.py:431, :465, :504-507) in child (= legal move) order; d_child_q/d_prior/d_pi may be NULL */
int m0_search_result(m0_engine* e, uint16_t* d_moves, int32_t* d_visits, double* d_child_q, double* d_prior, int32_t* d_count,
                     float* d_pi, double* d_root_q, int32_t* d_root_n, void* stream);
/* ---- the mini-batch as shipped (selection_jitter in force, config.yaml:138): every simulation of a batch selects with its own
 * random.random() draws (mcts.py:893-897), so a batch holds up to batch_n different leaves; duplicated leaves share a network row.
 * Sequence per mini-batch: m0_search_select_multi -> m0_search_multi_encode -> evaluator -> m0_search_expand_backup_multi. */
int m0_search_multi_enable(m0_engine* e, int samples_per_batch, int virtual_loss);
/* caller-supplied draws (parity with the reference under a seeded RNG): d_jitter float64[G][jitter_stride] = random.random() values in
 * consumption order, d_normal float64[G][normal_stride] = np.random.normal(0, 0.1) values of the entropy noise (mcts.py:181);
 * NULL = device generator.  Status bit 16 is set for a game that exhausts a stream. */
int m0_search_set_streams(m0_engine* e, const double* d_jitter, long long jitter_stride, const double* d_normal, long long normal_stride, void* stream);
/* _collect_leaf_position x batch_n (mcts.py:535-558, :742-769); d_row_base int32[G+1] / d_n_samples int32[G] (either may be NULL) receive
 * the compact row numbering (row_base[G] = number of rows to evaluate) and the samples collected per game */
int m0_search_select_multi(m0_engine* e, int batch_n, int32_t* d_sims_left, int32_t* d_row_base, int32_t* d_n_samples, void* stream);
/* encode_board of the collected leaves of games [g0, g1) into d_planes float32[rows][19][8][8]; mode 0 compact rows (row_base[g] + slot
 * - row0), 1 dense per leaf ((g - g0) * samples_per_batch + slot), 2 one row per sample in collection order */
int m0_search_multi_encode(m0_engine* e, int g0, int g1, int row0, int mode, float* d_planes, int row_cap, void* stream);
/* expansion (+ entropy noise, pruning, TT registration) and backup of the samples of games [g0, g1) in collection order (mcts.py:654-670) */
/* row_cap > 0 (compact rows): games whose rows end beyond row0 + row_cap are skipped by m0_search_multi_encode AND by this call and keep
 * their samples, so an evaluator batch of row_cap rows can be launched before the host has read the row numbering */
int m0_search_expand_backup_multi(m0_engine* e, int g0, int g1, const float* d_logits, int logits_stride, const float* d_values, int row0,
                                  int per_sample, int row_cap, void* stream);
/* ---- reuse of the root's evaluation across moves: a store of `slots` (1..64) entries per game keeps the network output of every
 * evaluated child of the root; the next m0_search_begin expands a root whose packed position (all 9 words) equals a stored one from
 * that entry.  The other roots needing an evaluation are ALSO written in compact rows to d_miss_planes float32[G][19][8][8], their
 * count to d_miss_count int32[1], and m0_search_expand_backup reads their outputs from the evaluator rows 0..count-1 of d_logits /
 * d_values.  Both buffers are the caller's and must stay alive.  Entries belong to the network that produced them: clear the store
 * when the evaluator changes.  Counter 12 counts the roots expanded from the store. */
int m0_search_reuse_enable(m0_engine* e, int slots, float* d_miss_planes, int32_t* d_miss_count);
int m0_search_reuse_clear(m0_engine* e, void* stream);
int m0_engine_counters(m0_engine* e, unsigned long long* h_out16); /* host buffer; synchronises */
int m0_engine_status(m0_engine* e, int32_t* d_status_out, int32_t* d_node_count_out, void* stream);

/* ---- self-play game loop: azchess/selfplay/internal.py:326-600 for all game slots of an engine -------------- */
typedef struct m0_selfplay_config { /* selfplay: section of the reference config, internal.py:347-381 */
  double temperature_start, temperature_end, resign_threshold, resign_min_entropy, resign_value_margin;
  int temperature_moves, max_game_len, min_resign_plies, resign_window, resign_consecutive_bad, opening_random_plies;
  unsigned long long seed;
  int argmax_after_plies; /* >= 0: arena move rule (arena.py:75-91): sample at temperature_start while plies < this, then argmax;
                             < 0: the self-play temperature schedule (internal.py:386-394) */
  int low_visit_threshold; /* internal.py:419-425: max visit count below this -> temperature at least 0.8; 0 = off */
  /* heuristic half of should_adjudicate_draw (draw.py:43-82), the merged `draw:` / `selfplay.draw:` sections (config.py:37-49) */
  int draw_enabled, draw_min_plies, draw_window, draw_min_unique, draw_halfmove_cap, draw_material_threshold;
} m0_selfplay_config;
typedef struct m0_finished_game {
  int game, plies; /* slot, len(states) */
  float z;         /* result from White's point of view (internal.py:587-599) */
  int reason;      /* 1 checkmate 2 stalemate 3 insufficient material 4 fifty-move claim 5 repetition claim 6 max_game_len 7 resignation
                      8 heuristic draw adjudication (draw.py:43-82; z = last search value, internal.py:587-599) */
  float avg_entropy;
} m0_finished_game;
int m0_selfplay_configure(m0_engine* e, const m0_selfplay_config* cfg, void* stream);
int m0_selfplay_start(m0_engine* e, void* stream);                      /* new game in every slot, internal.py:326-379 */
int m0_selfplay_advance(m0_engine* e, uint16_t* d_out_move, void* stream); /* one ply: sample, resign, push, finish/restart */
/* `games` argument of selfplay_worker (internal.py:94, :326): at most `games` more games are started (initial start + restarts), idle
 * slots afterwards, so every started game is played to its end; < 0 = unlimited (default) */
int m0_selfplay_set_start_budget(m0_engine* e, long long games, void* stream);
int m0_selfplay_active_games(m0_engine* e, int* h_out, void* stream);       /* slots holding a game; host int; synchronises */
/* d_uniforms float64[G]: the np.random.choice draw of sample_move_from_counts (internal.py:734) for the next advances; NULL = device RNG */
int m0_selfplay_set_uniforms(m0_engine* e, const double* d_uniforms);
int m0_selfplay_plies(m0_engine* e, int32_t* d_out, void* stream);        /* len(states) per slot, int32[G] */
int m0_trees_clear(m0_engine* e, void* stream);                         /* fresh MCTS per move (keeps positions + histories) */
int m0_selfplay_finished(m0_engine* e, m0_finished_game* h_out, int max_records, int* n_out, void* stream); /* host buffer; syncs */

/* ---- evaluator: azchess/model/resnet.py PolicyValueNet (inference forward) ------------------------------
 * Activations are NHWC ([board][square = row*8+col][channel]) inside the library; the API keeps the
 * reference's NCHW planes in and (B,4672)/(B,) out. */
#define M0_MAX_BLOCKS 64
#define M0_MAX_SSL_HEADS 8
enum { M0_ACT_NONE = 0, M0_ACT_RELU = 1, M0_ACT_SILU = 2, M0_ACT_LEAKY = 3 };

typedef struct m0_net_config { /* NetConfig, resnet.py:247-282 */
  int planes, channels, blocks, policy_size;
  int se, se_hidden;
  int attention, attention_heads, attention_every_k, attention_relbias, infer_attention_stride;
  float attention_unmasked_mix;
  int policy_factor_rank;
  int activation, value_activation; /* M0_ACT_* */
  int chess_features, piece_square_tables;
  int n_ssl_heads;
  int ssl_out_channels[M0_MAX_SSL_HEADS];
} m0_net_config;

/* Device pointers to contiguous float32 parameters owned by the caller (state_dict tensors re-laid-out):
 * convolution / linear weights as W[n][k], k = (ky*3+kx)*Cin + ci for 3x3 kernels; fc weights that consume a
 * flattened NCHW feature map have their columns permuted to NHWC order (sq*channels + c). */
typedef struct m0_block_weights {
  const float *gn1_w, *gn1_b, *conv1_w, *gn2_w, *gn2_b, *conv2_w; /* ResidualBlock, resnet.py:27-84 */
  const float *se_w1, *se_b1, *se_w2, *se_b2;
  int has_attention;                                                  /* ChessAttention follows, resnet.py:87-190 */
  const float *att_qkv_w, *att_proj_w, *att_ln_w, *att_ln_b, *att_rel_bias;
} m0_block_weights;

typedef struct m0_net_weights {
  const float *stem_w, *stem_gn_w, *stem_gn_b;                        /* resnet.py:314-318 */
  const float *pos_enc, *pst_w, *pst_gn_w, *pst_gn_b, *inter_w, *inter_gn_w, *inter_gn_b; /* ChessSpecificFeatures :197-244 */
  m0_block_weights blocks[M0_MAX_BLOCKS];
  const float *pol_conv_w, *pol_gn_w, *pol_gn_b, *pol_fc1_w, *pol_fc1_b, *pol_fc2_w, *pol_fc2_b; /* :447-452, :483-491 */
  float policy_logit_scale;                                           /* clamp(softplus(raw)+1e-3, max 5), :709-710 */
  const float *val_conv1_w, *val_gn1_w, *val_gn1_b, *val_conv2_w, *val_gn2_w, *val_gn2_b;         /* :494-502 */
  const float *val_fc1_w, *val_fc1_b, *val_fc2_w, *val_fc2_b, *val_gate_w, *val_gate_b, *val_fc3_w, *val_fc3_b; /* :503-509 */
  const float *ssl_conv1_w[M0_MAX_SSL_HEADS], *ssl_gn_w[M0_MAX_SSL_HEADS], *ssl_gn_b[M0_MAX_SSL_HEADS], *ssl_conv2_w[M0_MAX_SSL_HEADS];
} m0_net_weights;

typedef struct m0_net m0_net;
int m0_net_create(int device, const m0_net_config* cfg, const m0_net_weights* weights, m0_net** out);
int m0_net_destroy(m0_net* net);
/* PolicyValueNet.forward (resnet.py:755-760): d_planes float32[B][planes][8][8] -> d_logits float32[B][4672], d_values
 * float32[B].  precision 0 = fp32 SIMT kernels (parity <= 1e-4), 1 = bf16 and 2 = fp16 operands on the tcgen05 tensor-core pipeline
 * (fp32 accumulation; fp16 is the reference's autocast dtype and the default of the Python layer). */
int m0_net_forward(m0_net* net, const float* d_planes, int B, float* d_logits, float* d_values, int precision, void* stream);
/* The dominant kernel on its own (tests, roofline micro-benchmark): tcgen05/TMA implicit GEMM over bf16 operands.
 * taps = 9: 3x3 "same" convolution of NHWC activations d_act_bf16[boards][8][8][cin] with d_w_bf16[n][9*cin]
 * (k = (ky*3+kx)*cin + ci, nn.Conv2d of resnet.py:32-34); taps = 1: d_act_bf16[boards*64][cin] x d_w_bf16[n][cin]^T.
 * d_out_f32[boards*64][n].  boards even, cin % 32 == 0, n % 16 == 0, n <= 320.  With cin % 64 == 32 the last 64-deep k-block
 * of each tap is half empty: the activations are zero-filled past cin, and 3x3 weights are copied with each tap padded to whole
 * k-blocks (stream-ordered allocation, freed after the launch). */
int m0_tc_conv(const uint16_t* d_act_bf16, const uint16_t* d_w_bf16, int boards, int cin, int n, int taps, float* d_out_f32, void* stream);
/* Per-launch-site CUDA-event timing of the tensor-core forward (measurement aid, no reference counterpart): after
 * m0_profile_enable(1) every kernel launch of m0_net_forward (precision 1, 2) is bracketed by events on its stream;
 * m0_profile_get returns the accumulated milliseconds and launch count of one site ("conv1+gn", "conv2+pool",
 * "se_apply_gn", "attention_tc", ... ; NULL = all sites).  m0_profile_enable(0) switches it off and clears the table. */
int m0_profile_enable(int enable);
int m0_profile_get(const char* name, double* total_ms, long long* launches);
/* forward(x, return_ssl=True) (resnet.py:736-745): d_ssl_out[h] float32[B][k_h][8][8] for each SSL head (fp32 path) */
int m0_net_forward_ssl(m0_net* net, const float* d_planes, int B, float* d_logits, float* d_values, float* const* d_ssl_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* MATRIX0_B200_H */
