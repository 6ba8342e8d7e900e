// C-ABI of the device-resident self-play game loop (selfplay_kernels.cu).
#include "engine_host.cuh"
#include <string.h>

namespace m0 {
__global__ void selfplay_start_kernel(EngineView E, SelfPlayState S, int all, unsigned long long step);
template <bool GUMBEL>
__global__ void selfplay_advance_kernel(EngineView E, SelfPlayState S, unsigned long long step, u16* out_move, GumbelView GB);
__global__ void clear_trees_kernel(EngineView E);
}  // namespace m0

// selfplay: section of the reference config (internal.py:347-381), host mirror
struct m0_selfplay_config {
  double temperature_start, temperature_end, resign_threshold, resign_min_entropy, resign_value_margin;
  int temperature_moves, max_game_len, min_resign_plies, resign_window, resign_consecutive_bad, opening_random_plies;
  unsigned long long seed;
  int argmax_after_plies, low_visit_threshold;
  int draw_enabled, draw_min_plies, draw_window, draw_min_unique, draw_halfmove_cap, draw_material_threshold;
};

struct m0_finished_game {
  int game, plies;
  float z;
  int reason;
  float avg_entropy;
};

#define TRY(x)            \
  do {                    \
    int _r = (x);         \
    if (_r != M0_OK) return _r; \
  } while (0)

static int sp_ensure(m0_engine* e) {
  if (e->sp.ply) return M0_OK;
  const size_t G = e->v.G;
  SelfPlayState& s = e->sp;
  TRY(dev_alloc(e, &s.ply, G));
  TRY(dev_alloc(e, &s.consec_bad, G));
  TRY(dev_alloc(e, &s.recent_n, G));
  TRY(dev_alloc(e, &s.ent_n, G));
  TRY(dev_alloc(e, &s.ent_total, G));
  TRY(dev_alloc(e, &s.recent_val, G * SP_WINDOW));
  TRY(dev_alloc(e, &s.recent_ent, G * SP_WINDOW));
  TRY(dev_alloc(e, &s.ent_sum, G));
  TRY(dev_alloc(e, &s.last_value, G));
  TRY(dev_alloc(e, &s.games_started, G));
  TRY(dev_alloc(e, &s.need_start, G));
  TRY(dev_alloc(e, &s.hist_move, G * (size_t)e->v.hist_cap));
  TRY(dev_alloc(e, &s.start_budget, 1));
  {
    const int unlimited = 1 << 30;
    M0_CUDA_TRY(cudaMemcpy(s.start_budget, &unlimited, sizeof(int), cudaMemcpyHostToDevice));
  }
  s.uniforms = nullptr;
  s.finished_cap = (int)(G * 4 > 65536 ? G * 4 : 65536);
  TRY(dev_alloc(e, &s.finished, (size_t)s.finished_cap));
  TRY(dev_alloc(e, &s.finished_count, 1));
  TRY(dev_alloc(e, &e->d_sp_params, 1));
  s.params = e->d_sp_params;
  e->sp_step = 0;
  e->finished_read = 0;
  return M0_OK;
}

extern "C" {

// selfplay_worker configuration (internal.py:269-381): temperatures, resign rule, game length, opening plies
int m0_selfplay_configure(m0_engine* e, const m0_selfplay_config* c, void* stream) {
  if (!e || !c) { m0_set_error("m0_selfplay_configure: invalid argument"); return M0_ERR_ARG; }
  m0::DeviceGuard device_guard(e->device);
  M0_CUDA_TRY(device_guard.err);
  TRY(sp_ensure(e));
  SelfPlayParams p;
  memset(&p, 0, sizeof(p));
  p.temperature_start = c->temperature_start;
  p.temperature_end = c->temperature_end;
  p.resign_threshold = c->resign_threshold;
  p.resign_min_entropy = c->resign_min_entropy;
  p.resign_value_margin = c->resign_value_margin;
  p.temperature_moves = c->temperature_moves;
  p.max_game_len = c->max_game_len;
  p.min_resign_plies = c->min_resign_plies;
  p.resign_window = c->resign_window;
  p.resign_consecutive_bad = c->resign_consecutive_bad;
  p.opening_random_plies = c->opening_random_plies;
  p.seed = c->seed;
  p.argmax_after_plies = c->argmax_after_plies;
  p.low_visit_threshold = c->low_visit_threshold;
  p.draw_enabled = c->draw_enabled;
  p.draw_min_plies = c->draw_min_plies;
  p.draw_window = c->draw_window;
  p.draw_min_unique = c->draw_min_unique;
  p.draw_halfmove_cap = c->draw_halfmove_cap;
  p.draw_material_threshold = c->draw_material_threshold;
  M0_CUDA_TRY(cudaMemcpyAsync(e->d_sp_params, &p, sizeof(p), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  M0_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return M0_OK;
}

// start a new game in every slot (start position + opening_random_plies random legal moves, internal.py:326-379)
int m0_selfplay_start(m0_engine* e, void* stream) {
  if (!e) { m0_set_error("m0_selfplay_start: invalid argument"); return M0_ERR_ARG; }
  TRY(sp_ensure(e));
  e->sp_step += 1;
  selfplay_start_kernel<<<(e->v.G + 3) / 4, 128, 0, (cudaStream_t)stream>>>(e->v, e->sp, 1, e->sp_step);
  return m0_check_launch("m0_selfplay_start");
}

// selfplay_worker plays exactly `games` games (internal.py:326): at most `games` more games are STARTED from now on (by
// m0_selfplay_start and by the restarts of finished slots); slots that find the budget empty go idle, so every started game is played
// to its end and none is discarded.  games < 0: unlimited (the default).
int m0_selfplay_set_start_budget(m0_engine* e, long long games, void* stream) {
  if (!e) { m0_set_error("m0_selfplay_set_start_budget: invalid argument"); return M0_ERR_ARG; }
  TRY(sp_ensure(e));
  const int v = (games < 0 || games >= (1 << 30)) ? (1 << 30) : (int)games;
  M0_CUDA_TRY(cudaMemcpyAsync(e->sp.start_budget, &v, sizeof(int), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  M0_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  return M0_OK;
}

// d_uniforms float64[G]: the np.random draw sample_move_from_counts makes for each game in the NEXT m0_selfplay_advance calls
// (internal.py:734 np.random.choice -> one uniform in [0, 1)); NULL returns to the device generator.  The buffer must stay alive.
int m0_selfplay_set_uniforms(m0_engine* e, const double* d_uniforms) {
  if (!e) { m0_set_error("m0_selfplay_set_uniforms: invalid argument"); return M0_ERR_ARG; }
  TRY(sp_ensure(e));
  e->sp.uniforms = d_uniforms;
  return M0_OK;
}

// number of slots that currently hold a game (int, host): 0 once the start budget is spent and every started game has ended
int m0_selfplay_active_games(m0_engine* e, int* h_out, void* stream) {
  if (!e || !h_out) { m0_set_error("m0_selfplay_active_games: invalid argument"); return M0_ERR_ARG; }
  std::vector<unsigned char> act((size_t)e->v.G);
  M0_CUDA_TRY(cudaMemcpyAsync(act.data(), e->v.active, (size_t)e->v.G, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  M0_CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
  int n = 0;
  for (unsigned char a : act) n += a ? 1 : 0;
  *h_out = n;
  return M0_OK;
}

// One ply of the game loop for every slot whose search has finished (internal.py:408-539 + loop condition :382-384):
// sample the move, resign rule, push, finish / restart games.  d_out_move uint16[G] (optional) receives the moves played.
int m0_selfplay_advance(m0_engine* e, uint16_t* d_out_move, void* stream) {
  if (!e || !e->sp.ply) { m0_set_error("m0_selfplay_advance: self-play not configured"); return M0_ERR_STATE; }
  e->sp_step += 1;
  selfplay_advance_kernel<false><<<(e->v.G + 3) / 4, 128, 0, (cudaStream_t)stream>>>(e->v, e->sp, e->sp_step, d_out_move, GumbelView{});
  return m0_check_launch("m0_selfplay_advance");
}

// The same ply after a Gumbel search (m0_gumbel_result): the move is the search's choice, the search value and the entropy of the
// policy target feed the resign rule and avg_policy_entropy; temperature and visit sampling do not apply.
int m0_selfplay_advance_gumbel(m0_engine* e, uint16_t* d_out_move, void* stream) {
  if (!e || !e->sp.ply || !e->gb.logit) { m0_set_error("m0_selfplay_advance_gumbel: self-play or the Gumbel search not configured"); return M0_ERR_STATE; }
  e->sp_step += 1;
  selfplay_advance_kernel<true><<<(e->v.G + 3) / 4, 128, 0, (cudaStream_t)stream>>>(e->v, e->sp, e->sp_step, d_out_move, e->gb);
  return m0_check_launch("m0_selfplay_advance_gumbel");
}

// Drop all trees (nodes + transposition tables), keep positions and histories: what constructing a fresh
// MCTS per move does in the reference.
int m0_trees_clear(m0_engine* e, void* stream) {
  if (!e) { m0_set_error("m0_trees_clear: invalid argument"); return M0_ERR_ARG; }
  int bx = (e->v.tt_cap / 2 + 255) / 256;
  if (bx > 16) bx = 16;
  if (bx < 1) bx = 1;
  clear_trees_kernel<<<dim3(bx, e->v.G), 256, 0, (cudaStream_t)stream>>>(e->v);
  return m0_check_launch("m0_trees_clear");
}

// Fetch finished-game records produced since the last call into a HOST buffer (synchronises the stream).
int m0_selfplay_finished(m0_engine* e, m0_finished_game* h_out, int max_records, int* n_out, void* stream) {
  if (!e || !h_out || !n_out || !e->sp.ply) { m0_set_error("m0_selfplay_finished: invalid argument"); return M0_ERR_ARG; }
  cudaStream_t s = (cudaStream_t)stream;
  unsigned total = 0;
  M0_CUDA_TRY(cudaMemcpyAsync(&total, e->sp.finished_count, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
  M0_CUDA_TRY(cudaStreamSynchronize(s));
  unsigned avail = total - e->finished_read;
  if (avail > (unsigned)e->sp.finished_cap) {  // ring overran: skip to the oldest record still present
    e->finished_read = total - (unsigned)e->sp.finished_cap;
    avail = (unsigned)e->sp.finished_cap;
  }
  int n = (int)(avail < (unsigned)max_records ? avail : (unsigned)max_records);
  for (int i = 0; i < n;) {
    unsigned pos = (e->finished_read + (unsigned)i) % (unsigned)e->sp.finished_cap;
    int run = n - i;
    if (pos + (unsigned)run > (unsigned)e->sp.finished_cap) run = (int)((unsigned)e->sp.finished_cap - pos);
    M0_CUDA_TRY(cudaMemcpyAsync(h_out + i, e->sp.finished + pos, sizeof(m0_finished_game) * run, cudaMemcpyDeviceToHost, s));
    i += run;
  }
  M0_CUDA_TRY(cudaStreamSynchronize(s));
  e->finished_read += (unsigned)n;
  *n_out = n;
  return M0_OK;
}

}  // extern "C"

extern "C" {
// len(states) of every game slot (int32[G], device) -- gates ply-dependent options such as dirichlet_plies
int m0_selfplay_plies(m0_engine* e, int32_t* d_out, void* stream) {
  if (!e || !d_out || !e->sp.ply) { m0_set_error("m0_selfplay_plies: invalid argument"); return M0_ERR_ARG; }
  M0_CUDA_TRY(cudaMemcpyAsync(d_out, e->sp.ply, sizeof(int) * e->v.G, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return M0_OK;
}
}
