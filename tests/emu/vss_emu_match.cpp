// vss_emu_match.cpp — TEST HARNESS: the match mode of the step kernels (vss_step_match, VIEW_MATCH of
// csrc/vss_lane.cuh) run on the host, one tile at a time, like vss_emu.cpp does for the other modes. The
// orchestration mirrors the VIEW_MATCH paths of k_step (wpt = 1) and k_step_cta (wpt > 1) in csrc/vss_step.cu; the
// end of the step (step_done) becomes one board_close_step after all tiles. Not part of the product.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../rsoccer_isaac_cleanrl_b200/csrc/vss_lane.cuh"

using namespace vss;

static const ObsTable g_tab = make_obs_table();

static void emu_match_warp(const StepArgs& a, const DevParams& P) {
  const long long tiles = (a.n + 31) / 32;
#pragma omp parallel for schedule(static)
  for (long long tile = 0; tile < tiles; ++tile) {
    std::vector<float> Tbuf(TILE_WORDS, 0.0f);
    float* T = Tbuf.data();
    const long long env0 = tile * 32;
    const int valid = (int)std::min(32LL, a.n - env0);
    bool done[32] = {false};
    for (int lane = 0; lane < valid; ++lane)
      lane_phase1a<VIEW_MATCH>(T + lane, env0 + lane, a, P, make_key(a, env0 + lane));
    for (int it = 0; it < P.substeps; ++it) {
      std::vector<int> queue;
      for (int lane = 0; lane < valid; ++lane) {
        uint32_t m = substep_pre_lane(T + lane, P);
        for (int r = 0; r < 6; ++r) if (m & (1u << r)) queue.push_back((lane << 3) | r);
      }
      for (int q : queue) robot_walls_task(T + (q >> 3), q & 7, P);
      for (int lane = 0; lane < valid; ++lane) substep_ball_walls_lane(T + lane, P);
    }
    for (int lane = 0; lane < valid; ++lane)
      done[lane] = lane_phase1d<VIEW_MATCH>(T + lane, env0 + lane, a, P, make_key(a, env0 + lane)) == LANE_DONE;
    for (int lane = 0; lane < valid; ++lane)
      if (done[lane]) reset_lane(T + lane, P, make_key(a, env0 + lane));
    for (int lane = 0; lane < 32; ++lane) write_match_tile(T, g_tab.v, lane, valid, env0, a);
    for (int lane = 0; lane < valid; ++lane) lane_phase5<VIEW_MATCH>(T + lane, env0 + lane, a, done[lane]);
  }
}

static void emu_match_cta(const StepArgs& a, const DevParams& P, int NW, int F) {
  const int W = NW - 1;
  const long long tiles = (a.n + F - 1) / F;
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
      for (int b = warp; b < 3; b += W) actions_block<VIEW_MATCH>(S, env, a, P, key, b);
      if (warp == 3 % W && a.reset_buf[env] != 0) S[VSS_W_PROGRESS * LDS] = bitsf(0u);
      for (int b = warp; b < 7; b += W) prev_term_body(S, b, P);
    }
    for (int lane = 0; lane < valid; ++lane) {  // the helper warp
      float* Sh = T + lane + W_SHADOW * LDS;
      Sh[VSS_W_EPISODE * LDS] = T[VSS_W_EPISODE * LDS + lane];
      reset_lane(Sh, P, make_key(a, env0 + lane));
    }
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
    bool finite[32];
    for (int lane = 0; lane < valid; ++lane) {
      finite[lane] = state_finite(T + lane);
      if (!finite[lane]) lane_sanitise(T + lane, a, P, make_key(a, env0 + lane));
    }
    uint32_t done_mask = 0;
    for (int lane = 0; lane < valid; ++lane)
      if (lane_outputs<VIEW_MATCH>(T + lane, env0 + lane, a, P, finite[lane]) == LANE_DONE) done_mask |= 1u << lane;
    EACH_THREAD if ((done_mask >> lane) & 1u)
      for (int w = warp; w < VSS_STATE_WORDS; w += NW)
        if (w != VSS_W_PROGRESS) T[w * LDS + lane] = T[(W_SHADOW + w) * LDS + lane];
    for (int warp = 0; warp < NW; ++warp)
      for (int lane = 0; lane < 32; ++lane) write_match_tile(T, g_tab.v, lane, valid, env0, a, warp, NW);
    EACH_THREAD store_state_words(T + lane, a.state, a.ld, env0 + lane, warp, NW);
#undef EACH_THREAD
#undef EACH_BODY_THREAD
  }
}

extern "C" {

// teams: modes[2], policy actions[2] (f32), bf16 rows[2] (uint16); board = vss_match_board.
__attribute__((visibility("default"))) int emu_step_match(
    const vss_params* p, float* state, long long n, long long ld, unsigned long long goff, unsigned long long seed,
    unsigned int step, const int* modes, const float* act0, const float* act1, void* rows0, void* rows1,
    float* action_buf, long long* reset_buf, float* obs, long long count_envs, long long n_matches,
    vss_match_board* board, int wpt, int fpt) {
  const DevParams P = derive_params(*p);
  StepArgs a;
  memset(&a, 0, sizeof(a));
  unsigned long long step_ctr[3] = {step, 0, 0};
  a.state = state; a.n = n; a.ld = ld; a.goff = goff;
  a.seed_lo = (uint32_t)seed; a.seed_hi = (uint32_t)(seed >> 32); a.step_ctr = step_ctr; a.grid = 1;
  a.action_buf = action_buf; a.reset_buf = reset_buf; a.obs = obs;
  a.team_mode[0] = modes[0]; a.team_mode[1] = modes[1];
  a.team_action[0] = act0; a.team_action[1] = act1; a.team_rows[0] = rows0; a.team_rows[1] = rows1;
  a.count_envs = count_envs; a.n_matches = n_matches; a.board = board;
  if (wpt > 1) {
    if (wpt > MAX_WPT || (fpt != 8 && fpt != 16 && fpt != 32)) return -1;
    emu_match_cta(a, P, wpt, fpt);
  } else {
    emu_match_warp(a, P);
  }
  board_close_step(board, n_matches);
  return 0;
}

}  // extern "C"
