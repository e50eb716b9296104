// vss_emu_opp.cpp — TEST HARNESS: the opponent views of the step kernels (vss_step_view with vss_set_view_opponent,
// VIEW_OPP + VSS_VIEW_* of csrc/vss_lane.cuh) run on the host, one tile at a time, like vss_emu.cpp does for the
// other views. The orchestration mirrors the view paths of k_step (wpt = 1) and k_step_cta (wpt > 1) in
// csrc/vss_step.cu, with the opponent's post-reset rows written after the reset. Not part of the product.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <vector>

#include "../../rsoccer_isaac_cleanrl_b200/csrc/vss_lane.cuh"

using namespace vss;

static const ObsTable g_tab = make_obs_table();

template <int VIEW>
static void emu_opp_warp(const StepArgs& a, const DevParams& P) {
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
    for (int it = 0; it < P.substeps; ++it) {
      std::vector<int> queue;
      for (int lane = 0; lane < valid; ++lane) {
        uint32_t m = substep_pre_lane(T + lane, P);
        for (int r = 0; r < 6; ++r) if (m & (1u << r)) queue.push_back((lane << 3) | r);
      }
      for (int q : queue) robot_walls_task(T + (q >> 3), q & 7, P);
      for (int lane = 0; lane < valid; ++lane) substep_ball_walls_lane(T + lane, P);
    }
    for (int lane = 0; lane < valid; ++lane) {
      const int code = lane_phase1d<VIEW>(T + lane, env0 + lane, a, P, make_key(a, env0 + lane));
      done[lane] = code == LANE_DONE;
      ended[lane] = code != LANE_RUNNING;
      if (done[lane]) done_mask |= 1u << lane;
    }
    float* ob = a.obs + env0 * (PER_FIELD * 4);
    float* tob = a.term_obs ? a.term_obs + env0 * (PER_FIELD * 4) : nullptr;
    for (int lane = 0; lane < 32; ++lane) {
      if (PER_FIELD >= 32) write_obs_tile_rows<PER_FIELD>(T, g_tab.v, lane, valid, tob, ob, done_mask);
      else write_obs_tile(T, g_tab.v, lane, valid, PER_FIELD, tob, ob, done_mask);
    }
    for (int lane = 0; lane < valid; ++lane)
      if (done[lane]) reset_lane(T + lane, P, make_key(a, env0 + lane));
    for (int lane = 0; lane < 32; ++lane) write_obs_fields(T, g_tab.v, lane, PER_FIELD, ob, done_mask);
    for (int lane = 0; lane < 32; ++lane) write_opp_tile(T, g_tab.v, lane, valid, env0, a);
    for (int lane = 0; lane < valid; ++lane) lane_phase5<VIEW>(T + lane, env0 + lane, a, ended[lane]);
  }
}

template <int VIEW>
static void emu_opp_cta(const StepArgs& a, const DevParams& P, int NW, int F) {
  constexpr int PER_FIELD = ViewShape<VIEW>::F4_PER;
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
      for (int b = warp; b < 3; b += W) actions_block<VIEW>(S, env, a, P, key, b);
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
    float* ob = a.obs + env0 * (PER_FIELD * 4);
    float* tob = a.term_obs ? a.term_obs + env0 * (PER_FIELD * 4) : nullptr;
    for (int warp = 1; warp < NW; ++warp)
      for (int lane = 0; lane < 32; ++lane) {
        if (PER_FIELD >= 32) write_obs_tile_rows<PER_FIELD, true>(T, g_tab.v, lane, valid, tob, ob, 0u, nullptr, nullptr, warp - 1, NW - 1);
        else write_obs_tile(T, g_tab.v, lane, valid, PER_FIELD, tob, ob, 0u, nullptr, nullptr, warp - 1, NW - 1);
      }
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
        write_obs_fields(T, g_tab.v, lane, PER_FIELD, ob, done_mask, nullptr, nullptr, warp, NW);
        write_opp_tile(T, g_tab.v, lane, valid, env0, a, warp, NW);
      }
    EACH_THREAD store_state_words(T + lane, a.state, a.ld, env0 + lane, warp, NW);
    for (int lane = 0; lane < valid; ++lane)
      if ((ended_mask >> lane) & 1u) zero_action_row(env0 + lane, a);
#undef EACH_THREAD
#undef EACH_BODY_THREAD
  }
}

template <int VIEW>
static int emu_opp(const StepArgs& a, const DevParams& P, int wpt, int fpt) {
  if (wpt > 1) {
    if (wpt > MAX_WPT || (fpt != 8 && fpt != 16 && fpt != 32)) return -1;
    emu_opp_cta<VIEW>(a, P, wpt, fpt);
  } else {
    emu_opp_warp<VIEW>(a, P);
  }
  return 0;
}

extern "C" {

// One opponent view step: the arguments of vss_step_view (no aux / packed outputs) + the vss_view_opponent fields.
__attribute__((visibility("default"))) int emu_step_view_opp(
    const vss_params* p, int view, float* state, long long n, long long ld, unsigned long long goff,
    unsigned long long seed, unsigned int step, long long* reset_buf, float* obs, float* term_obs, float* rew,
    uint8_t* timeout, float* progress_f, const float* policy_action, float* action_buf, float* reward_v,
    long long* done_v, float* ep_ret, int* ep_len, float* ret_ret, int* ret_len, int opp_mode,
    const float* opp_action, void* opp_rows, float* opp_obs, int wpt, int fpt) {
  // (mode OU runs the opponent variant with the draw kept: the tests check that it equals the plain view)
  if (opp_mode < VSS_TEAM_ZERO || opp_mode > VSS_TEAM_EXTERNAL) return -1;
  const DevParams P = derive_params(*p);
  StepArgs a;
  memset(&a, 0, sizeof(a));
  unsigned long long step_ctr[3] = {step, 0, 0};
  a.state = state; a.n = n; a.ld = ld; a.goff = goff;
  a.seed_lo = (uint32_t)seed; a.seed_hi = (uint32_t)(seed >> 32); a.step_ctr = step_ctr; a.grid = 1;
  a.reset_buf = reset_buf; a.obs = obs; a.term_obs = term_obs; a.rew = rew; a.timeout = timeout;
  a.progress_f = progress_f; a.policy_action = policy_action; a.action_buf = action_buf; a.reward_v = reward_v;
  a.done_v = done_v; a.ep_ret = ep_ret; a.ep_len = ep_len; a.ret_ret = ret_ret; a.ret_len = ret_len;
  a.team_mode[1] = opp_mode; a.team_action[1] = opp_action; a.team_rows[1] = opp_rows; a.opp_obs = opp_obs;
  switch (view) {
    case VSS_VIEW_SA: return emu_opp<VIEW_OPP + VSS_VIEW_SA>(a, P, wpt, fpt);
    case VSS_VIEW_CMA: return emu_opp<VIEW_OPP + VSS_VIEW_CMA>(a, P, wpt, fpt);
    case VSS_VIEW_DMA: return emu_opp<VIEW_OPP + VSS_VIEW_DMA>(a, P, wpt, fpt);
    default: return -1;
  }
}

}  // extern "C"
