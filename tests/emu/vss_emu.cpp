// vss_emu.cpp — TEST HARNESS: runs the product's per-lane step code (csrc/vss_lane.cuh,
// the exact source the CUDA kernel compiles) on the host, one tile at a time, so the
// step logic can be checked against the oracle in the GPU-less build container. The
// orchestration below mirrors k_step, k_step_cta and k_reset_dones in csrc/vss_step.cu for every
// variant: the full contract, the views, the match step and the opponent views.
// Not part of the product: libvss_b200.so has no host execution path.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../rsoccer_isaac_cleanrl_b200/csrc/vss_lane.cuh"

using namespace vss;

static const ObsTable g_tab = make_obs_table();

// Mirror of k_step (one warp per 32-field tile), phases 1-5.
template <int VIEW, bool INJECT>
static void emu_step_warp(const StepArgs& a, const DevParams& P) {
  constexpr int PER_FIELD = ViewShape<VIEW>::F4_PER;
  const long long tiles = (a.n + 31) / 32;
#pragma omp parallel for schedule(static)
  for (long long tile = 0; tile < tiles; ++tile) {
    std::vector<float> Tbuf(TILE_WORDS, 0.0f);
    float* T = Tbuf.data();
    const long long env0 = tile * 32;
    const int valid = (int)std::min(32LL, a.n - env0);
    bool done[32] = {false}, ended[32] = {false};
    uint32_t done_mask = 0;
    for (int lane = 0; lane < valid; ++lane) lane_phase1a<VIEW>(T + lane, env0 + lane, a, P, make_key(a, env0 + lane));
    if (INJECT) {
      for (int lane = 0; lane < valid; ++lane) lane_inject(T + lane, env0 + lane, a);
    } else {  // physics_tile of vss_step.cu: wall tasks compacted over the warp
      for (int it = 0; it < P.substeps; ++it) {
        std::vector<int> queue;
        for (int lane = 0; lane < valid; ++lane) {
          uint32_t m = substep_pre_lane(T + lane, P);
          for (int r = 0; r < 6; ++r) if (m & (1u << r)) queue.push_back((lane << 3) | r);
        }
        for (int q : queue) robot_walls_task(T + (q >> 3), q & 7, P);
        for (int lane = 0; lane < valid; ++lane) substep_ball_walls_lane(T + lane, P);
      }
    }
    for (int lane = 0; lane < valid; ++lane) {
      const int code = lane_phase1d<VIEW>(T + lane, env0 + lane, a, P, make_key(a, env0 + lane));
      done[lane] = code == LANE_DONE;
      ended[lane] = code != LANE_RUNNING;
      if (done[lane]) done_mask |= 1u << lane;
    }
    const auto [ob, tob, obh, pk] = tile_out<VIEW>(a, env0);
    if (VIEW != VIEW_MATCH)  // (a match writes no terminal observation: every row is written once, after the reset)
      for (int lane = 0; lane < 32; ++lane) {
        if (PER_FIELD >= 32) write_obs_tile_rows<PER_FIELD>(T, g_tab.v, lane, valid, tob, ob, done_mask, obh, pk);
        else write_obs_tile(T, g_tab.v, lane, valid, PER_FIELD, tob, ob, done_mask, obh, pk);
      }
    for (int lane = 0; lane < valid; ++lane)
      if (done[lane]) reset_lane(T + lane, P, make_key(a, env0 + lane));
    for (int lane = 0; lane < 32; ++lane) {
      if (VIEW == VIEW_MATCH) write_match_tile(T, g_tab.v, lane, valid, env0, a);
      else write_obs_fields(T, g_tab.v, lane, PER_FIELD, ob, done_mask, obh, pk);
      if (VIEW >= VIEW_OPP) write_opp_tile(T, g_tab.v, lane, valid, env0, a);
    }
    for (int lane = 0; lane < valid; ++lane) lane_phase5<VIEW>(T + lane, env0 + lane, a, ended[lane]);
  }
}

// Mirror of k_step_cta (one tile shared by NW warps: W = NW - 1 body warps with the bodies dealt to them,
// and a helper warp that computes the resets speculatively into shadow columns): the phases below are the
// kernel's, each CTA barrier becomes the end of a loop over (warp, lane).
template <int VIEW, bool INJECT>
static void emu_step_cta(const StepArgs& a, const DevParams& P, int NW, int F) {
  constexpr int PER_FIELD = ViewShape<VIEW>::F4_PER;
  const int W = NW - 1;
  const long long tiles = (a.n + F - 1) / F;  // F = 32, 16 or 8 fields per tile (vss_set_step_fields_per_tile)
#pragma omp parallel for schedule(static)
  for (long long tile = 0; tile < tiles; ++tile) {
    std::vector<float> Tbuf(TILE_CTA_WORDS, 0.0f);
    float* T = Tbuf.data();
    const long long env0 = tile * F;
    const int valid = (int)std::min((long long)F, a.n - env0);
#define EACH_THREAD for (int warp = 0; warp < NW; ++warp) for (int lane = 0; lane < valid; ++lane)
#define EACH_BODY_THREAD for (int warp = 0; warp < W; ++warp) for (int lane = 0; lane < valid; ++lane)
    EACH_THREAD load_state_words(T + lane, a.state, a.ld, env0 + lane, warp, NW);
    EACH_BODY_THREAD {
      float* S = T + lane;
      const long long env = env0 + lane;
      const RngKey key = make_key(a, env);
      for (int b = warp; b < 3; b += W) actions_block<VIEW>(S, env, a, P, key, b);
      if (warp == 3 % W && a.reset_buf[env] != 0) S[VSS_W_PROGRESS * LDS] = bitsf(0u);
      for (int b = warp; b < 7; b += W) prev_term_body(S, b, P);
    }
    for (int lane = 0; lane < valid; ++lane) {  // the helper warp
      float* S = T + lane;
      float* Sh = S + W_SHADOW * LDS;
      Sh[VSS_W_EPISODE * LDS] = S[VSS_W_EPISODE * LDS];
      reset_lane(Sh, P, make_key(a, env0 + lane));
    }
    if (INJECT) {
      for (int lane = 0; lane < valid; ++lane) lane_inject(T + lane, env0 + lane, a);
    } else {
      for (int it = 0; it < P.substeps; ++it) {
        EACH_BODY_THREAD for (int b = warp; b < 7; b += W) { if (b < 6) integrate_robot(T + lane, b, P); else integrate_ball(T + lane, P); }
        EACH_BODY_THREAD {
          uint32_t m = 0u;
          for (int q = warp; q < 21; q += W) m |= broadphase_pair(T + lane, q, P);
          T[(W_SCR + warp) * LDS + lane] = bitsf(m);
        }
        EACH_BODY_THREAD if (lane % W == warp) {
          uint32_t m = 0u;
          for (int j = 0; j < W; ++j) m |= fbits(T[(W_SCR + j) * LDS + lane]);
          if (m) contacts_task(T + lane, m, P);
        }
        EACH_BODY_THREAD for (int b = warp; b < 7; b += W) walls_body(T + lane, b, P);
      }
    }
    bool finite[32];
    for (int lane = 0; lane < valid; ++lane) {
      finite[lane] = state_finite(T + lane);
      if (!finite[lane]) lane_sanitise(T + lane, a, P, make_key(a, env0 + lane));
    }
    const auto [ob, tob, obh, pk] = tile_out<VIEW>(a, env0);
    // warps 1 .. NW-1 write the rows of ALL fields (before warp 0's outputs are known; a match writes none) ...
    if (VIEW != VIEW_MATCH)
      for (int warp = 1; warp < NW; ++warp)
        for (int lane = 0; lane < 32; ++lane) {
          if (PER_FIELD >= 32) write_obs_tile_rows<PER_FIELD, true>(T, g_tab.v, lane, valid, tob, ob, 0u, obh, pk, warp - 1, NW - 1);
          else write_obs_tile(T, g_tab.v, lane, valid, PER_FIELD, tob, ob, 0u, obh, pk, warp - 1, NW - 1);
        }
    // ... while warp 0 computes them
    uint32_t done_mask = 0, ended_mask = 0;
    for (int lane = 0; lane < valid; ++lane) {
      const int code = lane_outputs<VIEW>(T + lane, env0 + lane, a, P, finite[lane]);
      if (code == LANE_DONE) done_mask |= 1u << lane;
      if (code != LANE_RUNNING) ended_mask |= 1u << lane;
    }
    EACH_THREAD if ((done_mask >> lane) & 1u)
      for (int w = warp; w < VSS_STATE_WORDS; w += NW)
        if (w != VSS_W_PROGRESS) T[w * LDS + lane] = T[(W_SHADOW + w) * LDS + lane];
    for (int warp = 0; warp < NW; ++warp)
      for (int lane = 0; lane < 32; ++lane) {
        if (VIEW == VIEW_MATCH) write_match_tile(T, g_tab.v, lane, valid, env0, a, warp, NW);
        else write_obs_fields(T, g_tab.v, lane, PER_FIELD, ob, done_mask, obh, pk, warp, NW);
        if (VIEW >= VIEW_OPP) write_opp_tile(T, g_tab.v, lane, valid, env0, a, warp, NW);
      }
    EACH_THREAD store_state_words(T + lane, a.state, a.ld, env0 + lane, warp, NW);
    if (VIEW != VIEW_FULL && VIEW != VIEW_MATCH)
      for (int lane = 0; lane < valid; ++lane)
        if ((ended_mask >> lane) & 1u) zero_action_row(env0 + lane, a);
#undef EACH_THREAD
#undef EACH_BODY_THREAD
  }
}

// One step in the launch shape wpt (1: k_step; 2 .. MAX_WPT: k_step_cta with fpt fields per tile). A match closes
// the step on its scoreboard after all tiles, as the kernels' last CTA does (step_done).
template <int VIEW, bool INJECT = false>
static int emu_shape(const StepArgs& a, const DevParams& P, int wpt, int fpt) {
  if (wpt > 1) emu_step_cta<VIEW, INJECT>(a, P, wpt, fpt);
  else emu_step_warp<VIEW, INJECT>(a, P);
  if (VIEW == VIEW_MATCH) board_close_step(a.board, a.n_matches);
  return 0;
}

// The step of variant `view` (VIEW_FULL, VSS_VIEW_*, VIEW_MATCH or VIEW_OPP + VSS_VIEW_*) with the step index `step`.
static int emu_run(const vss_params* p, int view, StepArgs& a, unsigned int step, int wpt, int fpt) {
  if (wpt > 1 && (wpt > MAX_WPT || (fpt != 8 && fpt != 16 && fpt != 32))) return -1;
  unsigned long long step_ctr[3] = {step, 0, 0};  // index, CTA count, sanitised fields
  a.step_ctr = step_ctr; a.grid = 1;
  const DevParams P = derive_params(*p);
  switch (view) {
    case VIEW_FULL: return a.inject ? emu_shape<VIEW_FULL, true>(a, P, wpt, fpt) : emu_shape<VIEW_FULL>(a, P, wpt, fpt);
    case VSS_VIEW_SA: return emu_shape<VSS_VIEW_SA>(a, P, wpt, fpt);
    case VSS_VIEW_CMA: return emu_shape<VSS_VIEW_CMA>(a, P, wpt, fpt);
    case VSS_VIEW_DMA: return emu_shape<VSS_VIEW_DMA>(a, P, wpt, fpt);
    case VIEW_MATCH: return emu_shape<VIEW_MATCH>(a, P, wpt, fpt);
    case VIEW_OPP + VSS_VIEW_SA: return emu_shape<VIEW_OPP + VSS_VIEW_SA>(a, P, wpt, fpt);
    case VIEW_OPP + VSS_VIEW_CMA: return emu_shape<VIEW_OPP + VSS_VIEW_CMA>(a, P, wpt, fpt);
    case VIEW_OPP + VSS_VIEW_DMA: return emu_shape<VIEW_OPP + VSS_VIEW_DMA>(a, P, wpt, fpt);
    default: return -1;
  }
}

static StepArgs base_args(float* state, long long n, long long ld, unsigned long long goff, unsigned long long seed) {
  StepArgs a;
  memset(&a, 0, sizeof(a));
  a.state = state; a.n = n; a.ld = ld; a.goff = goff;
  a.seed_lo = (uint32_t)seed; a.seed_hi = (uint32_t)(seed >> 32);
  return a;
}

extern "C" {

// The full contract (view = VIEW_FULL) and the views (VSS_VIEW_*).
__attribute__((visibility("default"))) int emu_step(
    const vss_params* p, int view, float* state, long long n, long long ld, unsigned long long goff,
    unsigned long long seed, unsigned int step, const float* actions, const float* inject, long long* reset_buf,
    float* obs, float* term_obs, float* rew, uint8_t* timeout, float* progress_f, const float* policy_action,
    float* action_buf, float* reward_v, long long* done_v, float* ep_ret, int* ep_len, float* ret_ret,
    int* ret_len, void* packed, int wpt, int fpt) {
  if (view < VIEW_FULL || view > VSS_VIEW_DMA) return -1;
  StepArgs a = base_args(state, n, ld, goff, seed);
  a.actions = actions; a.inject = inject; a.reset_buf = reset_buf; a.obs = obs; a.term_obs = term_obs;
  a.rew = rew; a.timeout = timeout; a.progress_f = progress_f; a.policy_action = policy_action;
  a.action_buf = action_buf; a.reward_v = reward_v; a.done_v = done_v; a.ep_ret = ep_ret; a.ep_len = ep_len;
  a.ret_ret = ret_ret; a.ret_len = ret_len; a.packed = packed;
  return emu_run(p, view, a, step, wpt, fpt);
}

// The match step (vss_step_match). teams: modes[2], policy actions[2] (f32), bf16 rows[2] (uint16); board =
// vss_match_board.
__attribute__((visibility("default"))) int emu_step_match(
    const vss_params* p, float* state, long long n, long long ld, unsigned long long goff, unsigned long long seed,
    unsigned int step, const int* modes, const float* act0, const float* act1, void* rows0, void* rows1,
    float* action_buf, long long* reset_buf, float* obs, long long count_envs, long long n_matches,
    vss_match_board* board, int wpt, int fpt) {
  StepArgs a = base_args(state, n, ld, goff, seed);
  a.action_buf = action_buf; a.reset_buf = reset_buf; a.obs = obs;
  a.team_mode[0] = modes[0]; a.team_mode[1] = modes[1];
  a.team_action[0] = act0; a.team_action[1] = act1; a.team_rows[0] = rows0; a.team_rows[1] = rows1;
  a.count_envs = count_envs; a.n_matches = n_matches; a.board = board;
  return emu_run(p, VIEW_MATCH, a, step, wpt, fpt);
}

// One opponent view step: the arguments of vss_step_view (no aux / packed outputs) + the vss_view_opponent fields.
// (Mode OU runs the opponent variant with the draw kept: the tests check that it equals the plain view.)
__attribute__((visibility("default"))) int emu_step_view_opp(
    const vss_params* p, int view, float* state, long long n, long long ld, unsigned long long goff,
    unsigned long long seed, unsigned int step, long long* reset_buf, float* obs, float* term_obs, float* rew,
    uint8_t* timeout, float* progress_f, const float* policy_action, float* action_buf, float* reward_v,
    long long* done_v, float* ep_ret, int* ep_len, float* ret_ret, int* ret_len, int opp_mode,
    const float* opp_action, void* opp_rows, float* opp_obs, int wpt, int fpt) {
  if (view < VSS_VIEW_SA || view > VSS_VIEW_DMA || opp_mode < VSS_TEAM_ZERO || opp_mode > VSS_TEAM_EXTERNAL) return -1;
  StepArgs a = base_args(state, n, ld, goff, seed);
  a.reset_buf = reset_buf; a.obs = obs; a.term_obs = term_obs; a.rew = rew; a.timeout = timeout;
  a.progress_f = progress_f; a.policy_action = policy_action; a.action_buf = action_buf; a.reward_v = reward_v;
  a.done_v = done_v; a.ep_ret = ep_ret; a.ep_len = ep_len; a.ret_ret = ret_ret; a.ret_len = ret_len;
  a.team_mode[1] = opp_mode; a.team_action[1] = opp_action; a.team_rows[1] = opp_rows; a.opp_obs = opp_obs;
  return emu_run(p, VIEW_OPP + view, a, step, wpt, fpt);
}

__attribute__((visibility("default"))) int emu_reset_dones(const vss_params* p, float* state, long long n,
                                                           long long ld, unsigned long long goff,
                                                           unsigned long long seed, const long long* reset_buf,
                                                           float* obs) {
  const DevParams P = derive_params(*p);
  const StepArgs a = base_args(state, n, ld, goff, seed);
  const long long tiles = (n + 31) / 32;
  for (long long tile = 0; tile < tiles; ++tile) {
    std::vector<float> Tbuf(TILE_WORDS, 0.0f);
    float* T = Tbuf.data();
    const long long env0 = tile * 32;
    const int valid = (int)std::min(32LL, n - env0);
    for (int lane = 0; lane < valid; ++lane) {
      load_state(T + lane, state, ld, env0 + lane);
      if (reset_buf[env0 + lane] != 0) {
        reset_lane(T + lane, P, make_key(a, env0 + lane));
        store_state(T + lane, state, ld, env0 + lane);
      }
    }
    if (obs)
      for (int lane = 0; lane < 32; ++lane)
        write_obs_tile(T, g_tab.v, lane, valid, F4_PER_FIELD, nullptr, obs + env0 * VSS_OBS_PER_FIELD, 0u);
  }
  return 0;
}

}  // extern "C"
