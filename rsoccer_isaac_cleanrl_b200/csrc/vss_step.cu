// vss_step.cu — the fused VSS env-step kernels for sm_100a and their C-ABI.
//
// One warp = one tile of 32 consecutive fields. Phase structure of a step:
//   1. per lane : coalesced SoA load of the 60 state words into a shared-memory column,
//                 actions / OU noise, physics substeps, rewards, dones, per-field outputs
//   2. warp     : terminal observation (and the final observation of fields that are not
//                 reset) written row-major with 128-bit fully coalesced stores, gathered
//                 from the staged columns through a 78-entry permutation/sign table
//   3. per lane : masked reset (Philox rejection sampling) of done fields
//   4. warp     : observation rows of the fields that were reset
//   5. per lane : coalesced SoA store of the state
// HBM traffic per field-step (full VSS.step contract): 240 B state in + 240 B out, 48 B
// actions, 8+8 B reset flags, 1248 B obs, 1248 B terminal obs, 96 B rewards, 5 B flags.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>

#include "vss_lane.cuh"
#include "vss_render.cuh"

namespace vss {

__constant__ ObsTable c_obs_table = make_obs_table();

constexpr int TAB_WORDS = 80;  // 78 table entries, padded
constexpr int CTR_WORDS = 4;   // task counters of the CTA-wide queues

// Shared-memory layout of a CTA of W warps (words):
//   [0, TAB_WORDS)                     observation permutation/sign table
//   + W * TILE_STATE_WORDS             the staged state columns, one 32-field tile per warp
//   + W * QUEUE_WORDS                  task queues
//   + CTR_WORDS                        task counters
__host__ __device__ constexpr size_t smem_words(int wpb) {
  return TAB_WORDS + (size_t)wpb * TILE_WORDS + CTR_WORDS;
}


// Physics of one tile (replaces gym.simulate), warp-local version: per substep, phases A-C per lane,
// then the robot-wall contacts as (field, robot) tasks compacted over the warp — any lane can work
// on any field of the tile because the state columns live in shared memory — then the ball-wall
// phase per lane.
template <bool SYNC>
__device__ __forceinline__ void physics_tile(float* T, uint8_t* queue, int lane, bool active, const DevParams& P) {
  float* S = T + lane;
#pragma unroll 1
  for (int it = 0; it < P.substeps; ++it) {
    // keep the warps of a CTA in the same code region: the kernel is instruction-fetch bound
    // (85 KB of SASS, "no instruction" stalls), and warps that run the same 128-byte lines at the
    // same time share them in the instruction caches
    if (SYNC) __syncthreads();
    uint32_t m = active ? substep_pre_lane(S, P) : 0u;
    const int cnt = __popc(m);
    int incl = cnt;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int v = __shfl_up_sync(0xffffffffu, incl, d);
      if (lane >= d) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    int pos = incl - cnt;
    while (m) {
      const int r = __ffs((int)m) - 1;
      m &= m - 1;
      queue[pos++] = (uint8_t)((lane << 3) | r);
    }
    __syncwarp();
#pragma unroll 1
    for (int t0 = 0; t0 < total; t0 += 32) {  // warp-uniform trip count: usually one pass, rarely more
      if (t0 + lane < total) {
        const int q = queue[t0 + lane];
        robot_walls_task(T + (q >> 3), q & 7, P);
      }
    }
    __syncwarp();
    if (active) substep_ball_walls_lane(S, P);
  }
}

__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// The last warp of a CTA to finish counts the CTA as done (StepArgs::step_ctr[1]): every warp of the CTA
// has read the step index (phase 1a) by then. The CTA that completes the step — `a.grid` CTAs, over all
// the range launches of one step — clears the count and advances the step index (step_ctr[0]); launches
// of the next step are ordered after every launch of this one, so they read the new index.
// Match mode: every thread fences its scoreboard adds before its warp is counted, and the completing CTA fences
// again before it reads the count and closes the step (the last-block pattern of a threadfence reduction).
template <int VIEW>
__device__ __forceinline__ void step_done(const StepArgs& a, uint32_t* ctr) {
  if (VIEW == VIEW_MATCH) __threadfence();
  __syncwarp();
  if ((threadIdx.x & 31) == 0 && atomicAdd(&ctr[3], 1u) == (blockDim.x >> 5) - 1u) {
    if (VIEW == VIEW_MATCH) __threadfence();
    unsigned long long* done_ctas = a.step_ctr + 1;
    if (atomicAdd(done_ctas, 1ull) == (unsigned long long)a.grid - 1ull) {
      if (VIEW == VIEW_MATCH) {
        __threadfence();
        board_close_step(a.board, a.n_matches);
      }
      atomicExch(done_ctas, 0ull);
      atomicAdd(a.step_ctr, 1ull);
    }
  }
}

// SYNC: false = warps run free (small batches: 1-2 warps per CTA); true = CTA-wide barriers at substep
// and phase boundaries (large batches: 4 warps per CTA kept in the same code region).
template <int VIEW, bool INJECT, bool SYNC>
__global__ void __launch_bounds__(384)
k_step(const __grid_constant__ StepArgs a, const __grid_constant__ DevParams P) {
  extern __shared__ __align__(16) float smem[];
  uint32_t* tab = reinterpret_cast<uint32_t*>(smem);
  for (int i = threadIdx.x; i < F4_PER_FIELD; i += blockDim.x) tab[i] = c_obs_table.v[i];
  float* tiles = smem + TAB_WORDS;
  uint32_t* queue = reinterpret_cast<uint32_t*>(tiles + (blockDim.x >> 5) * TILE_STATE_WORDS);
  uint32_t* ctr = queue + (blockDim.x >> 5) * QUEUE_WORDS;
  if (threadIdx.x == 0) ctr[3] = 0u;  // warps of this CTA that have finished
  // The CTAs of the first wave all start at once and would run their load / compute / store phases in
  // lock-step (memory idle while they all compute, then all storing); the CTAs that take their slots
  // later inherit the rhythm. Start the co-resident CTAs of an SM a little apart.
  if (a.stagger_ns > 0 && blockIdx.x < 148u * 6u) {
    // CTAs are handed out round-robin over the 148 SMs: the k-th CTA of an SM is blockIdx / 148
    const unsigned wait_ns = ((blockIdx.x / 148u) % 6u) * (unsigned)a.stagger_ns;
    const unsigned long long t0 = globaltimer_ns();
    while (globaltimer_ns() - t0 < wait_ns) __nanosleep(1000);
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long tile = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  const long long env0 = a.env_begin + tile * a.fpw;
  if (!SYNC && env0 >= a.n) { if (VIEW != VIEW_FULL) step_done<VIEW>(a, ctr); return; }  // (with block-level syncs every warp stays until the end)
  float* T = tiles + warp * TILE_STATE_WORDS;
  float* S = T + lane;
  const long long env = env0 + lane;
  const bool active = lane < a.fpw && env < a.n;
  const int valid = (int)max(0LL, min((long long)a.fpw, a.n - env0));
  constexpr int PER_FIELD = ViewShape<VIEW>::F4_PER;
  const RngKey key = make_key(a, env);
  // 1. per lane: load, actions, physics, rewards, dones
  if (active) lane_phase1a<VIEW>(S, env, a, P, key);
  if (INJECT) { if (active) lane_inject(S, env, a); }
  else physics_tile<SYNC>(T, reinterpret_cast<uint8_t*>(queue + warp * QUEUE_WORDS), lane, active, P);
  if (SYNC) __syncthreads();
  int code = LANE_RUNNING;
  if (active) code = lane_phase1d<VIEW>(S, env, a, P, key);
  const bool done = code == LANE_DONE;   // needs the masked reset of phase 3
  __syncwarp();
  if (SYNC) __syncthreads();
  // 2. terminal observation + observation of the fields that keep their state (vss.py:195-196)
  const uint32_t done_mask = __ballot_sync(0xffffffffu, done);
  const auto [ob, tob, obh, pk] = tile_out<VIEW>(a, env0);
  if (VIEW == VIEW_MATCH) {}  // (no terminal observation: every row is written once, after the reset)
  else if (PER_FIELD >= 32) write_obs_tile_rows<PER_FIELD>(T, tab, lane, valid, tob, ob, done_mask, obh, pk);
  else write_obs_tile(T, tab, lane, valid, PER_FIELD, tob, ob, done_mask, obh, pk);
  __syncwarp();
  // 3. masked reset (vss.py:202, 267-333)
  if (done) reset_lane(S, P, key);
  __syncwarp();
  // 4. observation of the fields that were reset (vss.py:203)
  if (VIEW == VIEW_MATCH) write_match_tile(T, tab, lane, valid, env0, a);
  else write_obs_fields(T, tab, lane, PER_FIELD, ob, done_mask, obh, pk);
  if (VIEW >= VIEW_OPP) write_opp_tile(T, tab, lane, valid, env0, a);  // the opponent's next input
  // 5. state out
  if (SYNC) __syncthreads();
  if (active) lane_phase5<VIEW>(S, env, a, code != LANE_RUNNING);
  // only the views draw OU noise: the full-contract step neither reads nor advances the index (the
  // extra memory operation at the end of every CTA costs 1 % of the launch at 2^20 fields)
  if (VIEW != VIEW_FULL) step_done<VIEW>(a, ctr);
}

// ----------------------------------------------------------------------------------------
// k_step_cta — the same step with ONE 32-field tile per CTA, shared by NW = blockDim / 32 warps:
// W = NW - 1 "body" warps and one helper warp.
// Small and medium batches leave SMs idle and are bound by the critical path of a tile (one warp
// = one field per lane walks 6 robots + the ball one after the other: ~12 000 dependent instructions,
// 31-37 us). Here body warp j owns the bodies j, j + W, ... (0-5 = robots, 6 = ball) of all 32 fields:
// every dense phase still runs with 32 active lanes, lane = field, conflict-free on the same staged
// columns, but up to 7 bodies advance side by side. Phases that couple bodies are separated by CTA
// barriers: integrate | broadphase (pairs dealt round-robin to the warps, partial masks in the
// scratch words) | pair contacts (field l by warp l mod W: the sequential impulse order inside a
// field is unchanged) | walls (per body, in place).
// The helper warp spends the physics phase computing the masked reset of EVERY field of the tile
// into a shadow set of columns (the reset depends only on (seed, field id, episode counter), all
// known at the start): 32 dense lanes, off the critical path; phase 3 copies the shadow columns of
// the fields that did end. Without it the ~1 100 dependent instructions of a reset (4-5 Philox
// blocks, 21 distance tests, 6 sincos) sit at the end of whichever tile has a done field — and with
// >= 100 tiles per launch some tile always has one.
// After the physics, warp 0 computes rewards / dones / per-field outputs while the other warps
// already write the observation rows (for all fields: the rows of fields that turn out to be done
// are written again after the reset, phase 4). The cooperative parts — state load / store by words,
// observation rows by field groups — are dealt to all NW warps.
// Results are bit-identical to k_step: the same per-body code in the same order per field.
// ----------------------------------------------------------------------------------------
// Barrier over the W body warps of a k_step_cta CTA only (named barrier 1): the helper warp runs its
// speculative resets meanwhile and joins the others at the next __syncthreads().
__device__ __forceinline__ void body_barrier(int W) {
  asm volatile("bar.sync 1, %0;" ::"r"(W * 32) : "memory");
}

// Profiling build only (-DVSS_PHASE_PROFILE, profiles/step_phase_profile.py): per-CTA clock totals of the phases of
// k_step_cta as seen by warp 0 after the barrier that ends each phase (= the slowest warp of the phase), plus one
// extra barrier after the wall phase so that its imbalance is not booked on the next integrate. Not in the product.
#ifdef VSS_PHASE_PROFILE
__device__ unsigned long long g_phase_prof[65536 * 8];
__device__ unsigned long long g_integ_prof[4096 * 16];  // per CTA: [warp] integrate compute, [8 + warp] wait at its barrier
#define PROF_DECL unsigned long long pf_t = clock64(), pf_acc[7] = {0, 0, 0, 0, 0, 0, 0}; const unsigned long long pf_t0 = pf_t;
#define PROF_MARK(i) do { const unsigned long long pf_n = clock64(); pf_acc[i] += pf_n - pf_t; pf_t = pf_n; } while (0)
#define PROF_STORE do { if (threadIdx.x == 0 && blockIdx.x < 65536) { pf_acc[6] = clock64() - pf_t0; \
    for (int i = 0; i < 7; ++i) g_phase_prof[blockIdx.x * 8 + i] = pf_acc[i]; } } while (0)
#else
#define PROF_DECL
#define PROF_MARK(i)
#define PROF_STORE
#endif

template <int VIEW, bool INJECT>
__global__ void __launch_bounds__(32 * MAX_WPT)
k_step_cta(const __grid_constant__ StepArgs a, const __grid_constant__ DevParams P) {
  extern __shared__ __align__(16) float smem[];
  uint32_t* tab = reinterpret_cast<uint32_t*>(smem);
  for (int i = threadIdx.x; i < F4_PER_FIELD; i += blockDim.x) tab[i] = c_obs_table.v[i];
  float* T = smem + TAB_WORDS;
  uint32_t* ctr = reinterpret_cast<uint32_t*>(T + TILE_CTA_WORDS);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, NW = blockDim.x >> 5, W = NW - 1;
  const bool helper = warp == W;
  if (threadIdx.x == 0) ctr[3] = 0u;  // warps of this CTA that have finished
  // a.fpw fields per tile (32, 16 or 8): lanes >= fpw idle in the per-field phases and help in the cooperative ones
  const long long env0 = a.env_begin + (long long)blockIdx.x * a.fpw;
  float* S = T + lane;
  float* Sh = S + W_SHADOW * LDS;  // the field's shadow column
  const long long env = env0 + lane;
  const bool active = lane < a.fpw && env < a.n;
  const int valid = (int)max(0LL, min((long long)a.fpw, a.n - env0));
  constexpr int PER_FIELD = ViewShape<VIEW>::F4_PER;
  const RngKey key = make_key(a, env);
  PROF_DECL
  // 1a. state in (words dealt to the warps), then actions / OU noise per Philox block, progress restart,
  //     prev_* clones per body
  if (active) load_state_words(S, a.state, a.ld, env, warp, NW);
  __syncthreads();
  if (active && !helper) {
    for (int b = warp; b < 3; b += W) actions_block<VIEW>(S, env, a, P, key, b);
    if (warp == 3 % W && a.reset_buf[env] != 0) S[VSS_W_PROGRESS * LDS] = bitsf(0u);  // vss.py:182-183
    for (int b = warp; b < 7; b += W) prev_term_body(S, b, P);
  }
  __syncthreads();
  PROF_MARK(0);
  // physics (replaces gym.simulate) on the body warps, which synchronise among themselves (body_barrier);
  // speculative resets on the helper warp meanwhile.
  if (helper && active) {
    Sh[VSS_W_EPISODE * LDS] = S[VSS_W_EPISODE * LDS];
    reset_lane(Sh, P, key);
  }
  if (INJECT) {
    if (warp == 0 && active) lane_inject(S, env, a);
  } else {
    if (!helper) {
#pragma unroll 1
      for (int it = 0; it < P.substeps; ++it) {
#ifdef VSS_PHASE_PROFILE
        const unsigned long long ig0 = clock64();
#endif
        if (active)
          for (int b = warp; b < 7; b += W) { if (b < 6) integrate_robot(S, b, P); else integrate_ball(S, P); }
#ifdef VSS_PHASE_PROFILE
        const unsigned long long ig1 = clock64();
#endif
        body_barrier(W);
#ifdef VSS_PHASE_PROFILE
        if (lane == 0 && blockIdx.x < 4096) {
          const unsigned long long ig2 = clock64();
          if (it == 0) { g_integ_prof[blockIdx.x * 16 + warp] = 0; g_integ_prof[blockIdx.x * 16 + 8 + warp] = 0; }
          g_integ_prof[blockIdx.x * 16 + warp] += ig1 - ig0;
          g_integ_prof[blockIdx.x * 16 + 8 + warp] += ig2 - ig1;
        }
#endif
        PROF_MARK(1);
        {
          uint32_t m = 0u;
          if (active)
            for (int q = warp; q < 21; q += W) m |= broadphase_pair(S, q, P);
          S[(W_SCR + warp) * LDS] = bitsf(m);
        }
        body_barrier(W);
        PROF_MARK(2);
        if (active && lane % W == warp) {
          uint32_t m = 0u;
          for (int j = 0; j < W; ++j) m |= fbits(S[(W_SCR + j) * LDS]);
          if (m) contacts_task(S, m, P);
        }
        body_barrier(W);
        PROF_MARK(3);
        if (active)
          for (int b = warp; b < 7; b += W) walls_body(S, b, P);  // (the next integrate of a body is by the same thread)
#ifdef VSS_PHASE_PROFILE
        body_barrier(W);
        PROF_MARK(4);
#endif
      }
    }
  }
  __syncthreads();
  // non-finite guard: every warp looks at the same 32 fields, so the branch is uniform over the CTA
  const bool finite = !active || state_finite(S);
  if (__ballot_sync(0xffffffffu, !finite)) {
    __syncthreads();
    if (warp == 0 && !finite) lane_sanitise(S, a, P, key);
    __syncthreads();
  }
  // 1d. post_physics_step per field (warp 0): progress, rewards, dones, per-field outputs — while the other
  // warps write 2. terminal observation + observation (vss.py:195-196) of all fields
  const auto [ob, tob, obh, pk] = tile_out<VIEW>(a, env0);
  if (warp == 0) {
    int code = LANE_RUNNING;
    if (active) code = lane_outputs<VIEW>(S, env, a, P, finite);
    const uint32_t dm = __ballot_sync(0xffffffffu, code == LANE_DONE);      // needs the masked reset of phase 3
    const uint32_t em = __ballot_sync(0xffffffffu, code != LANE_RUNNING);  // episode ended (done or sanitised)
    if (lane == 0) { ctr[0] = dm; ctr[1] = em; }
  } else if (VIEW == VIEW_MATCH) {
    // (no terminal observation: every row is written once, after the reset)
  } else if (PER_FIELD >= 32) {
    write_obs_tile_rows<PER_FIELD, true>(T, tab, lane, valid, tob, ob, 0u, obh, pk, warp - 1, NW - 1);
  } else {
    write_obs_tile(T, tab, lane, valid, PER_FIELD, tob, ob, 0u, obh, pk, warp - 1, NW - 1);
  }
  __syncthreads();
  const uint32_t done_mask = ctr[0], ended_mask = ctr[1];
  // 3. masked reset (vss.py:202, 267-333): the shadow column replaces the state (not the progress counter,
  //    which restarts at the next step's pre_physics_step)
  if ((done_mask >> lane) & 1u)
    for (int w = warp; w < VSS_STATE_WORDS; w += NW)
      if (w != VSS_W_PROGRESS) S[w * LDS] = Sh[w * LDS];
  __syncthreads();
  // 4. observation of the fields that were reset (vss.py:203); 5. state out
  if (VIEW == VIEW_MATCH) write_match_tile(T, tab, lane, valid, env0, a, warp, NW);
  else write_obs_fields(T, tab, lane, PER_FIELD, ob, done_mask, obh, pk, warp, NW);
  if (VIEW >= VIEW_OPP) write_opp_tile(T, tab, lane, valid, env0, a, warp, NW);  // the opponent's next input
  if (active) store_state_words(S, a.state, a.ld, env, warp, NW);
  if (VIEW == VIEW_MATCH) {
    step_done<VIEW>(a, ctr);  // (done rows keep their actions: play_matches carries the OU state over)
  } else if (VIEW != VIEW_FULL) {
    if (warp == 0 && ((ended_mask >> lane) & 1u)) zero_action_row(env, a);  // wrappers.py:105-107
    step_done<VIEW>(a, ctr);
  }
  PROF_MARK(5);
  PROF_STORE;
}

// reset_dones() + compute_observations(): vss.py:72-73, 267-333, 205-216
__global__ void __launch_bounds__(384)
k_reset_dones(float* state, long long n, long long ld, unsigned long long goff, uint32_t seed_lo,
              uint32_t seed_hi, const long long* reset_buf, float* obs, const __grid_constant__ DevParams P) {
  extern __shared__ __align__(16) float smem[];
  uint32_t* tab = reinterpret_cast<uint32_t*>(smem);
  for (int i = threadIdx.x; i < F4_PER_FIELD; i += blockDim.x) tab[i] = c_obs_table.v[i];
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long tile = (long long)blockIdx.x * (blockDim.x >> 5) + warp;
  const long long env0 = tile * 32;
  if (env0 >= n) return;
  float* T = smem + TAB_WORDS + warp * TILE_STATE_WORDS;
  float* S = T + lane;
  const long long env = env0 + lane;
  const bool active = env < n;
  const int valid = (int)min(32LL, n - env0);
  bool flagged = false;
  if (active) {
    load_state(S, state, ld, env);
    flagged = reset_buf[env] != 0;
    if (flagged) {
      const unsigned long long gid = goff + (unsigned long long)env;
      reset_lane(S, P, RngKey{seed_lo, seed_hi, (uint32_t)gid, (uint32_t)(gid >> 32)});
      store_state(S, state, ld, env);
    }
  }
  __syncwarp();
  if (obs) write_obs_tile(T, tab, lane, valid, F4_PER_FIELD, nullptr, obs + env0 * VSS_OBS_PER_FIELD, 0u);
}

// ----------------------------------------------------------------------------------------
// GAE reverse scan: ppo_continuous_action_isaacgym.py:282-296. One thread per env column,
// coalesced across envs, the T loop in registers, loads unrolled 8 deep ahead of the
// (serial) recurrence. 28 B of HBM traffic per (t, env).
// ----------------------------------------------------------------------------------------
struct GaeRows { float r, v, nv, d, to; };

__device__ __forceinline__ GaeRows gae_load(const float* __restrict__ rewards, const float* __restrict__ values,
                                            const float* __restrict__ next_values, const float* __restrict__ next_dones,
                                            const float* __restrict__ next_timeouts, long long i) {
  return GaeRows{__ldg(rewards + i), __ldg(values + i), __ldg(next_values + i), __ldg(next_dones + i),
                 __ldg(next_timeouts + i)};
}

// One step of the recurrence (ppo…:284-296), in the oracle's operation order.
__device__ __forceinline__ float gae_step(const GaeRows& x, float last, float gamma, float gamma_lambda,
                                          float* __restrict__ advantages, float* __restrict__ returns, long long i) {
  const float nnt = (x.d != 0.0f && !(x.to != 0.0f)) ? 0.0f : 1.0f;
  const float delta = fsub(fadd(x.r, fmul(fmul(gamma, x.nv), nnt)), x.v);
  last = fadd(delta, fmul(fmul(gamma_lambda, fsub(1.0f, x.d)), last));
  advantages[i] = last;
  returns[i] = fadd(last, x.v);
  return last;
}

// The recurrence is serial in t, the loads are not: the rows of the NEXT group of U time steps are
// requested before the current group is consumed (two register buffers), so a thread always has
// 5 U loads in flight. Without this the kernel is bound by T / U DRAM round trips (52 us at
// T = 128, N = 65536, whatever the CTA size).
// PREFETCH = false (many columns: enough warps per SM to cover the round trips, and 80 loads in
// flight per thread then only thrash DRAM pages): the next group is requested after the current one.
template <bool PREFETCH>
__global__ void __launch_bounds__(128)
k_gae(const float* __restrict__ rewards, const float* __restrict__ values, const float* __restrict__ next_values,
      const float* __restrict__ next_dones, const float* __restrict__ next_timeouts,
      float* __restrict__ advantages, float* __restrict__ returns, int T, long long N, float gamma,
      float gamma_lambda) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float last = 0.0f;
  constexpr int U = 8;
  int t = T - 1;
  if (t >= U - 1) {
    GaeRows cur[U], nxt[U];
#pragma unroll
    for (int k = 0; k < U; ++k)
      cur[k] = gae_load(rewards, values, next_values, next_dones, next_timeouts, (long long)(t - k) * N + n);
    for (; t >= U - 1; t -= U) {
      const bool more = t - U >= U - 1;  // another full group follows: request it now (or after this one)
      if (PREFETCH && more) {
#pragma unroll
        for (int k = 0; k < U; ++k)
          nxt[k] = gae_load(rewards, values, next_values, next_dones, next_timeouts, (long long)(t - U - k) * N + n);
      }
#pragma unroll
      for (int k = 0; k < U; ++k)
        last = gae_step(cur[k], last, gamma, gamma_lambda, advantages, returns, (long long)(t - k) * N + n);
      if (more) {
#pragma unroll
        for (int k = 0; k < U; ++k)
          cur[k] = PREFETCH ? nxt[k]
                            : gae_load(rewards, values, next_values, next_dones, next_timeouts,
                                       (long long)(t - U - k) * N + n);
      }
    }
  }
  for (; t >= 0; --t) {
    const long long i = (long long)t * N + n;
    last = gae_step(gae_load(rewards, values, next_values, next_dones, next_timeouts, i), last, gamma, gamma_lambda,
                    advantages, returns, i);
  }
}

// ---------------------------------------------------------------------------------------- frames (vss_render)
// One CTA per (frame, band of RENDER_THREADS 16-pixel segments = a band of rows); the field's RENDER_WORDS state
// words are read once into shared memory. Each thread draws 16 consecutive pixels of a row (csrc/vss_render.cuh)
// and stores their 48 bytes with three 16-byte stores: a warp writes 1 536 contiguous bytes of a row.
constexpr int RENDER_THREADS = 128;

__global__ void __launch_bounds__(RENDER_THREADS)
k_render(const float* __restrict__ state, long long ld, long long first, int height, int width,
         long long ctas_per_frame, RenderFrame g, uint8_t* __restrict__ rgb) {
  __shared__ float f[RENDER_WORDS];
  const long long frame = blockIdx.x / ctas_per_frame;
  const int band = (int)(blockIdx.x - frame * ctas_per_frame);
  if (threadIdx.x < RENDER_WORDS) f[threadIdx.x] = state[(long long)render_word(threadIdx.x) * ld + first + frame];
  __syncthreads();
  const int segs_per_row = width >> 4;
  const int seg = band * RENDER_THREADS + (int)threadIdx.x;
  if (seg >= height * segs_per_row) return;
  const int i = seg / segs_per_row, j0 = (seg - i * segs_per_row) << 4;
  uint32_t w[12];
  render_segment(g, f, i, j0, w);
  uint4* out = reinterpret_cast<uint4*>(rgb + ((frame * height + i) * (long long)width + j0) * 3);
  out[0] = make_uint4(w[0], w[1], w[2], w[3]);
  out[1] = make_uint4(w[4], w[5], w[6], w[7]);
  out[2] = make_uint4(w[8], w[9], w[10], w[11]);
}

}  // namespace vss

// ========================================================================================
// C-ABI
// ========================================================================================
using namespace vss;

struct vss_engine {
  int device;
  int64_t n, ld, goff;
  uint64_t seed;
  unsigned long long* d_step;  // device words: [0] step index (keys the OU stream), [1] CTAs of the current step that
                               // finished, [2] fields re-randomised by the non-finite guard
  vss_params params;
  DevParams dp;
  float* state;
  void* aux_obs_bf16; float* aux_done_f; float* aux_timeout_f;  // vss_set_step_aux
  void* packed_rows;                                            // vss_set_step_packed
  int wpt_override;                                             // vss_set_step_warps_per_tile (0 = automatic)
  int fpt_override;                                             // vss_set_step_fields_per_tile (0 = automatic)
  int64_t range_first, range_count;                             // vss_set_step_range (count 0 = all fields)
  vss_view_opponent opp;                                        // vss_set_view_opponent (mode OU = none)
  cudaStream_t host_stream[2];                                  // vss_step_view_host: the two pipeline streams ...
  cudaEvent_t host_start, host_done[2];                         // ... and their fork / join events (created on first use)
  bool host_ready;
};

static thread_local std::string g_last_error;

static int fail(int code, const char* what, cudaError_t e = cudaSuccess) {
  g_last_error = what;
  if (e != cudaSuccess) { g_last_error += ": "; g_last_error += cudaGetErrorString(e); }
  return code;
}
#define VSS_CUDA(call)                                        \
  do {                                                        \
    cudaError_t e_ = (call);                                  \
    if (e_ != cudaSuccess) return fail(VSS_E_CUDA, #call, e_); \
  } while (0)

// Launch shape of the step kernels (a function of the engine's field count only, so that every
// launch of an engine — whole or one range of vss_set_step_range — uses the same CTA shape).
// Large batches: 4 warps per CTA with CTA-wide barriers at phase boundaries — the step kernel is
// instruction-fetch bound (profiles/r01_b_*.md), and warps that execute the same code region at the
// same time share its lines in the instruction caches (+25 % measured); 6 CTAs of 4 warps per SM
// (measured at 2^20 fields: 4 / 6 / 8 / 12 warps per CTA -> 0.672 / 0.671 / 0.652 / 0.592 of the HBM
// roofline). Small batches: 1-2 warps per CTA so that at least 148 CTAs exist; no barriers (up to ~3
// resident warps per scheduler the barriers only add latency: 2^16 fields 61.5 us vs 68.0 us with 4
// warps + barriers; 2^17 fields 117 vs 109 us, so the switch sits between them).
// `fpw` (fields per warp): small batches leave most SMs empty and are bound by one warp's critical
// path, which grows with the number of fields it owns (every contact of any of its fields is
// serialised): 16 or 8 fields per warp (the other lanes idle in the per-field phases and help in the
// cooperative observation writes). Measured (k_step<sa>, us per step at 32 / 16 / 8 fields per warp):
// 1024 fields 43.7 / 35.7 / 33.8; 4096: 46.4 / 40.0 / 36.2; 8192: 47.7 / 40.2 / 40.3; 16384: 48.7 /
// 44.4 / 47.5; 21845: 51.2 / 47.4 / 53.7; 32768: 53.9 / 53.8 / 84.2.
// First-wave stagger (profiles/r01_g_*.md): 5 us per resident CTA of an SM, measured best of 0-12 us
// at 2^20 fields (675 -> 652 us per step); only for the barrier-synchronised shape and only when the
// launch is longer than one wave of 148 x 6 CTAs.
// `wpt` (warps per tile) > 1 selects k_step_cta: one 32-field tile per CTA shared by wpt - 1 body warps (bodies
// dealt to the warps) and a helper warp. It shortens a tile's critical path and is used while the batch cannot
// fill the SMs with one warp per tile.
struct LaunchShape {
  int wpb, fpw, stagger_ns, wpt;
  bool sync;
  unsigned grid;  // CTAs of a whole-engine launch
  size_t smem;
};

static int auto_wpt(int64_t n) {
  const int64_t tiles = (n + 31) / 32;
  // measured (profiles/r02_g_step_shapes.txt, us per launch, sa view, 1 / 8 warps per tile): 1 024 fields 31.0 / 29.0;
  // 4 096: 32.5 / 30.3; 8 192: 36.2 / 33.2; 16 384: 39.5 / 45+: from ~3 CTAs per SM on, the idle lanes of the
  // one-warp shape (8 or 16 fields per warp) are the cheaper way to shorten the critical path
  return tiles <= 256 ? 8 : 1;
}

// Fields per tile of the k_step_cta shape: the smallest tile that still gives at most one CTA per SM. Measured
// (profiles/r02_ae_step_shapes_fpt.txt, us per launch, full contract, 8 warps per tile, 32 / 16 / 8 fields per tile):
// 1 024 fields 28.2 / 26.9 / 25.8; 4 096: 32.9 / 34.1 / 35.3; 8 192: 35.1 / 37.0 / 51.7 — smaller tiles only pay
// while every tile still has an SM to itself (the launch is bound by ONE field's contact chain, not by the number
// of fields that share a warp).
static int auto_cta_fields(int64_t n) { return n <= 148 * 8 ? 8 : (n <= 148 * 16 ? 16 : 32); }

static LaunchShape launch_shape(int64_t n, bool step_kernel = true, int wpt_override = 0, int fpt_override = 0) {
  LaunchShape s;
  s.wpt = !step_kernel ? 1 : (wpt_override > 0 ? wpt_override : auto_wpt(n));
  if (s.wpt > 1) {
    s.wpb = s.wpt; s.sync = true; s.stagger_ns = 0;
    s.fpw = fpt_override > 0 ? fpt_override : auto_cta_fields(n);
    s.grid = (unsigned)((n + s.fpw - 1) / s.fpw);
    s.smem = sizeof(float) * (TAB_WORDS + TILE_CTA_WORDS + CTR_WORDS);
    return s;
  }
  s.fpw = !step_kernel ? 32 : (fpt_override > 0 ? fpt_override : (n < 148 * 40 ? 8 : (n < 148 * 192 ? 16 : 32)));
  const int64_t tiles = (n + s.fpw - 1) / s.fpw;
  s.wpb = tiles < 148 * 2 ? 1 : (tiles < 148 * 20 ? 2 : 4);
  s.sync = s.wpb == 4;
  s.grid = (unsigned)((tiles + s.wpb - 1) / s.wpb);
  s.smem = sizeof(float) * smem_words(s.wpb);
  s.stagger_ns = (s.sync && s.grid > 148u * 6u) ? 5000 : 0;
  return s;
}

static int use_device(vss_handle h) {
  int cur = -1;
  VSS_CUDA(cudaGetDevice(&cur));
  if (cur != h->device) VSS_CUDA(cudaSetDevice(h->device));
  return VSS_OK;
}

static StepArgs base_args(vss_handle h) {
  StepArgs a;
  memset(&a, 0, sizeof(a));
  a.state = h->state; a.n = h->n; a.ld = h->ld; a.goff = (unsigned long long)h->goff;
  a.seed_lo = (uint32_t)h->seed; a.seed_hi = (uint32_t)(h->seed >> 32); a.step_ctr = h->d_step;
  return a;
}

template <int VIEW, bool INJECT>
static int launch_step(vss_handle h, StepArgs a, void* stream) {
  const LaunchShape ls = launch_shape(h->n, true, h->wpt_override, h->fpt_override);
  a.fpw = ls.fpw; a.stagger_ns = ls.stagger_ns;
  a.grid = ls.grid;  // a step is complete when this many CTAs have finished, over all its range launches
  unsigned grid = ls.grid;
  if (h->range_count > 0) {  // vss_set_step_range: this launch covers [first, first + count) — same CTA shape, fewer CTAs
    const int64_t per_cta = ls.wpt > 1 ? ls.fpw : (int64_t)ls.wpb * ls.fpw;
    if (h->range_first % per_cta != 0 || (h->range_count % per_cta != 0 && h->range_first + h->range_count != h->n))
      return fail(VSS_E_INVALID, "step range: first / count must be multiples of vss_step_granularity()");
    a.env_begin = h->range_first;
    a.n = h->range_first + h->range_count;
    grid = (unsigned)((h->range_count + per_cta - 1) / per_cta);
  }
  if (ls.wpt > 1) k_step_cta<VIEW, INJECT><<<grid, ls.wpt * 32, ls.smem, (cudaStream_t)stream>>>(a, h->dp);
  else if (ls.sync) k_step<VIEW, INJECT, true><<<grid, ls.wpb * 32, ls.smem, (cudaStream_t)stream>>>(a, h->dp);
  else k_step<VIEW, INJECT, false><<<grid, ls.wpb * 32, ls.smem, (cudaStream_t)stream>>>(a, h->dp);
  VSS_CUDA(cudaGetLastError());
  return VSS_OK;
}

extern "C" {

VSS_API const char* vss_last_error(void) { return g_last_error.c_str(); }
VSS_API const char* vss_version(void) { return "vss_b200 0.1 (sm_100a)"; }

VSS_API int vss_default_params(vss_params* p) {
  if (!p) return fail(VSS_E_INVALID, "vss_default_params: null");
  const double PI = 3.14159265358979323846;
  p->dt = 0.05f; p->substeps = 4; p->max_episode_length = 400;
  p->field_half_length = 0.75f; p->field_half_width = 0.65f; p->goal_half_width = 0.2f; p->goal_depth = 0.1f;
  p->ball_radius = 0.02134f;
  p->ball_mass = (float)(1130.0 * 4.0 / 3.0 * PI * 0.02134 * 0.02134 * 0.02134);
  p->ball_drag = (float)(0.5 * 2.0 / 7.0);
  p->robot_half_size = 0.035f; p->robot_mass = 0.44f;
  p->robot_inertia = (float)(0.4 * (0.07 * 0.07 + 0.07 * 0.07) / 12.0 + 2.0 * 0.02 * 0.03375 * 0.03375);
  p->wheel_radius = 0.024f; p->wheel_half_track = 0.03375f; p->wheel_coll_radius = 0.024f;
  p->max_wheel_rad_s = 42.0f; p->drive_damping = 0.01f; p->drive_max_torque = 0.1f;
  p->wheel_inertia = (float)(0.0002 + 0.4 * 0.02 * 0.024 * 0.024);
  p->mu_traction = 0.7f; p->mu_lateral = 0.55f; p->gravity = 9.81f;
  p->restitution = 0.0f; p->mu_ball_robot = 0.5f; p->mu_ball_wall = 1.0f; p->mu_robot_wall = 0.5f;
  p->reset_scale_x = (float)(1.5 - 0.14); p->reset_scale_y = (float)(1.3 - 0.14);
  p->min_placement_dist = 0.07f; p->ball_reset_speed = 1.0f;
  p->w_goal = 10.0f; p->w_grad = 2.0f; p->w_move = 3.0f; p->w_energy = 0.0f;
  p->ou_theta = 0.1f; p->ou_sigma = 0.15f;
  return VSS_OK;
}

VSS_API int vss_create(vss_handle* out, const vss_params* p, int64_t num_envs, int64_t global_env_offset,
                       int device, uint64_t seed) {
  if (!out || !p) return fail(VSS_E_INVALID, "vss_create: null argument");
  if (num_envs <= 0) return fail(VSS_E_INVALID, "vss_create: num_envs must be > 0");
  if (p->substeps < 0 || p->substeps > 64) return fail(VSS_E_INVALID, "vss_create: substeps out of range");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(VSS_E_NODEVICE, "vss_create: no CUDA device (this library has no CPU fallback)", e);
  if (device < 0 || device >= count) return fail(VSS_E_INVALID, "vss_create: bad device index");
  cudaDeviceProp prop;
  VSS_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10)
    return fail(VSS_E_NODEVICE, "vss_create: kernels are built for sm_100a only (Blackwell B200)");
  VSS_CUDA(cudaSetDevice(device));
  vss_engine* h = new (std::nothrow) vss_engine();
  if (!h) return fail(VSS_E_NOMEM, "vss_create: host allocation failed");
  h->device = device; h->n = num_envs; h->ld = (num_envs + 31) / 32 * 32; h->goff = global_env_offset;
  h->aux_obs_bf16 = nullptr; h->aux_done_f = nullptr; h->aux_timeout_f = nullptr; h->packed_rows = nullptr;
  h->range_first = 0; h->range_count = 0; h->wpt_override = 0; h->fpt_override = 0; h->host_ready = false;
  h->opp = vss_view_opponent{VSS_TEAM_OU, 0, nullptr, nullptr, nullptr};
  h->seed = seed; h->d_step = nullptr; h->params = *p; h->dp = derive_params(*p); h->state = nullptr;
  const size_t bytes = sizeof(float) * VSS_STATE_WORDS * (size_t)h->ld;
  e = cudaMalloc(&h->state, bytes);
  if (e != cudaSuccess) { delete h; return fail(VSS_E_NOMEM, "vss_create: cudaMalloc(state)", e); }
  e = cudaMemset(h->state, 0, bytes);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_step, 3 * sizeof(unsigned long long));
  if (e == cudaSuccess) e = cudaMemset(h->d_step, 0, 3 * sizeof(unsigned long long));
  if (e != cudaSuccess) { cudaFree(h->state); cudaFree(h->d_step); delete h; return fail(VSS_E_CUDA, "vss_create: cudaMemset", e); }
  *out = h;
  return VSS_OK;
}

VSS_API int vss_destroy(vss_handle h) {
  if (!h) return VSS_OK;
  if (h->host_ready) {
    for (int i = 0; i < 2; ++i) { cudaStreamDestroy(h->host_stream[i]); cudaEventDestroy(h->host_done[i]); }
    cudaEventDestroy(h->host_start);
  }
  cudaFree(h->state);
  cudaFree(h->d_step);
  delete h;
  return VSS_OK;
}

VSS_API int64_t vss_num_envs(vss_handle h) { return h ? h->n : 0; }
VSS_API int64_t vss_state_ld(vss_handle h) { return h ? h->ld : 0; }
// The counter lives on the device; these two synchronise (tests / checkpointing only).
VSS_API uint64_t vss_step_count(vss_handle h) {
  if (!h) return 0;
  unsigned long long v = 0;
  if (use_device(h) != VSS_OK) return 0;
  if (cudaMemcpy(&v, h->d_step, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
  return v;
}
VSS_API uint64_t vss_sanitised_count(vss_handle h) {
  if (!h) return 0;
  unsigned long long v = 0;
  if (use_device(h) != VSS_OK) return 0;
  if (cudaMemcpy(&v, h->d_step + 2, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return 0;
  return v;
}
VSS_API int vss_set_step_count(vss_handle h, uint64_t n) {
  if (!h) return fail(VSS_E_INVALID, "null handle");
  if (int rc = use_device(h)) return rc;
  // the index is one 32-bit word of the Philox counter of the OU stream
  if (n > 0xFFFFFFFFull) return fail(VSS_E_INVALID, "vss_set_step_count: the step index is a 32-bit counter");
  const unsigned long long v[2] = {(unsigned long long)n, 0ull};  // also forgets a partially issued step
  VSS_CUDA(cudaMemcpy(h->d_step, v, sizeof(v), cudaMemcpyHostToDevice));
  return VSS_OK;
}

VSS_API int vss_set_reward_weights(vss_handle h, const float w[4]) {
  if (!h || !w) return fail(VSS_E_INVALID, "vss_set_reward_weights: null");
  h->params.w_goal = w[0]; h->params.w_grad = w[1]; h->params.w_move = w[2]; h->params.w_energy = w[3];
  h->dp.w_goal = w[0]; h->dp.w_grad = w[1]; h->dp.w_move = w[2]; h->dp.w_energy = w[3];
  return VSS_OK;
}

VSS_API int vss_reset_dones(vss_handle h, const int64_t* reset_buf, float* obs, void* stream) {
  if (!h || !reset_buf) return fail(VSS_E_INVALID, "vss_reset_dones: null argument");
  if (int rc = use_device(h)) return rc;
  const LaunchShape ls = launch_shape(h->n, false);
  k_reset_dones<<<ls.grid, ls.wpb * 32, ls.smem, (cudaStream_t)stream>>>(
      h->state, h->n, h->ld, (unsigned long long)h->goff, (uint32_t)h->seed, (uint32_t)(h->seed >> 32),
      reinterpret_cast<const long long*>(reset_buf), obs, h->dp);
  VSS_CUDA(cudaGetLastError());
  return VSS_OK;
}

VSS_API int vss_step(vss_handle h, const float* actions, int64_t* reset_buf, float* obs, float* term_obs,
                     float* rew, uint8_t* timeout, float* progress_f, void* stream) {
  if (!h || !actions || !reset_buf || !obs || !rew || !timeout)
    return fail(VSS_E_INVALID, "vss_step: null argument");
  if (int rc = use_device(h)) return rc;
  StepArgs a = base_args(h);
  a.actions = actions; a.reset_buf = reinterpret_cast<long long*>(reset_buf); a.obs = obs; a.term_obs = term_obs;
  a.rew = rew; a.timeout = timeout; a.progress_f = progress_f;
  return launch_step<VIEW_FULL, false>(h, a, stream);
}

VSS_API int vss_step_injected(vss_handle h, const float* actions, const float* post_state, int64_t* reset_buf,
                              float* obs, float* term_obs, float* rew, uint8_t* timeout, float* progress_f,
                              void* stream) {
  if (!h || !actions || !post_state || !reset_buf || !obs || !rew || !timeout)
    return fail(VSS_E_INVALID, "vss_step_injected: null argument");
  if (int rc = use_device(h)) return rc;
  StepArgs a = base_args(h);
  a.actions = actions; a.inject = post_state; a.reset_buf = reinterpret_cast<long long*>(reset_buf); a.obs = obs;
  a.term_obs = term_obs; a.rew = rew; a.timeout = timeout; a.progress_f = progress_f;
  return launch_step<VIEW_FULL, true>(h, a, stream);
}

VSS_API int vss_step_view(vss_handle h, int view, const float* policy_action, float* action_buf,
                          int64_t* reset_buf, float* obs_v, float* term_obs_v, float* rews_v, float* reward_v,
                          int64_t* done_v, uint8_t* timeout_v, float* progress_v, float* ep_ret, int32_t* ep_len,
                          float* ret_ret, int32_t* ret_len, void* stream) {
  if (!h || !policy_action || !action_buf || !reset_buf || !obs_v || !rews_v || !reward_v || !done_v || !timeout_v)
    return fail(VSS_E_INVALID, "vss_step_view: null argument");
  if (ep_ret && (!ep_len || !ret_ret || !ret_len))
    return fail(VSS_E_INVALID, "vss_step_view: episode statistics need all four buffers");
  if (int rc = use_device(h)) return rc;
  StepArgs a = base_args(h);
  a.policy_action = policy_action; a.action_buf = action_buf; a.reset_buf = reinterpret_cast<long long*>(reset_buf);
  a.obs = obs_v; a.term_obs = term_obs_v; a.rew = rews_v; a.reward_v = reward_v;
  a.done_v = reinterpret_cast<long long*>(done_v); a.timeout = timeout_v; a.progress_f = progress_v;
  a.ep_ret = ep_ret; a.ep_len = ep_len; a.ret_ret = ret_ret; a.ret_len = ret_len;
  a.obs_bf16 = h->aux_obs_bf16; a.done_f = h->aux_done_f; a.timeout_f = h->aux_timeout_f;
  a.packed = h->packed_rows;
  if (h->opp.mode != VSS_TEAM_OU) {  // the opponent variant of the view (today's kernel without one)
    a.team_mode[1] = h->opp.mode; a.team_action[1] = h->opp.policy_action; a.team_rows[1] = h->opp.rows_bf16;
    a.opp_obs = h->opp.obs_f32;
    switch (view) {
      case VSS_VIEW_SA: return launch_step<VIEW_OPP + VSS_VIEW_SA, false>(h, a, stream);
      case VSS_VIEW_CMA: return launch_step<VIEW_OPP + VSS_VIEW_CMA, false>(h, a, stream);
      case VSS_VIEW_DMA: return launch_step<VIEW_OPP + VSS_VIEW_DMA, false>(h, a, stream);
      default: return fail(VSS_E_INVALID, "vss_step_view: unknown view");
    }
  }
  switch (view) {
    case VSS_VIEW_SA: return launch_step<VSS_VIEW_SA, false>(h, a, stream);
    case VSS_VIEW_CMA: return launch_step<VSS_VIEW_CMA, false>(h, a, stream);
    case VSS_VIEW_DMA: return launch_step<VSS_VIEW_DMA, false>(h, a, stream);
    default: return fail(VSS_E_INVALID, "vss_step_view: unknown view");
  }
}

VSS_API int vss_step_match(vss_handle h, const vss_match_team teams[2], float* action_buf, int64_t* reset_buf,
                           float* obs, int64_t count_envs, int64_t n_matches, vss_match_board* board, void* stream) {
  // everything that needs no handle first
  if (!teams) return fail(VSS_E_INVALID, "vss_step_match: null argument");
  for (int t = 0; t < 2; ++t) {
    const int m = teams[t].mode;
    if (m < VSS_TEAM_ZERO || m > VSS_TEAM_EXTERNAL) return fail(VSS_E_INVALID, "vss_step_match: unknown team mode");
    if ((m == VSS_TEAM_SA || m == VSS_TEAM_CMA || m == VSS_TEAM_DMA) && !teams[t].policy_action)
      return fail(VSS_E_INVALID, "vss_step_match: a policy team needs its policy action");
  }
  if (n_matches < 1) return fail(VSS_E_INVALID, "vss_step_match: n_matches must be >= 1");
  if (!h || !action_buf || !reset_buf || !board) return fail(VSS_E_INVALID, "vss_step_match: null argument");
  if (count_envs < 1 || count_envs > h->n) return fail(VSS_E_INVALID, "vss_step_match: count_envs outside [1, num_envs]");
  if (h->range_count > 0) return fail(VSS_E_INVALID, "vss_step_match: whole-engine launches only (a step range is set)");
  if (int rc = use_device(h)) return rc;
  StepArgs a = base_args(h);
  a.action_buf = action_buf; a.reset_buf = reinterpret_cast<long long*>(reset_buf); a.obs = obs;
  for (int t = 0; t < 2; ++t) {
    a.team_mode[t] = teams[t].mode; a.team_action[t] = teams[t].policy_action; a.team_rows[t] = teams[t].rows_bf16;
  }
  a.count_envs = count_envs; a.n_matches = n_matches; a.board = board;
  return launch_step<VIEW_MATCH, false>(h, a, stream);
}

VSS_API int vss_step_view_host(vss_handle h, int view, const vss_view_buffers* dev, const float* policy_action_host,
                               void* rows_host, int num_ranges, void* stream) {
  if (!h || !dev || !policy_action_host || !rows_host || !dev->packed_rows || !dev->policy_action)
    return fail(VSS_E_INVALID, "vss_step_view_host: null argument");
  if (view != VSS_VIEW_SA && view != VSS_VIEW_CMA && view != VSS_VIEW_DMA) return fail(VSS_E_INVALID, "vss_step_view_host: unknown view");
  if (h->opp.mode != VSS_TEAM_OU) return fail(VSS_E_INVALID, "vss_step_view_host: no opponents on the host-buffer path");
  if (int rc = use_device(h)) return rc;
  if (!h->host_ready) {
    for (int i = 0; i < 2; ++i) {
      VSS_CUDA(cudaStreamCreateWithFlags(&h->host_stream[i], cudaStreamNonBlocking));
      VSS_CUDA(cudaEventCreateWithFlags(&h->host_done[i], cudaEventDisableTiming));
    }
    VSS_CUDA(cudaEventCreateWithFlags(&h->host_start, cudaEventDisableTiming));
    h->host_ready = true;
  }
  cudaStream_t st = (cudaStream_t)stream;
  const int agents = view == VSS_VIEW_DMA ? 3 : 1, adim = view == VSS_VIEW_CMA ? 6 : 2;
  const int64_t gran = vss_step_granularity(h);
  if (num_ranges < 1) num_ranges = 1;
  int64_t per = (h->n + num_ranges - 1) / num_ranges;
  per = (per + gran - 1) / gran * gran;
  void* const saved_packed = h->packed_rows;
  const int64_t saved_first = h->range_first, saved_count = h->range_count;
  h->packed_rows = dev->packed_rows;
  VSS_CUDA(cudaEventRecord(h->host_start, st));
  int rc = VSS_OK, used = 0;
  for (int64_t f0 = 0; f0 < h->n && rc == VSS_OK; f0 += per, ++used) {
    const int64_t cnt = f0 + per <= h->n ? per : h->n - f0;
    const int64_t v0 = f0 * agents, nv = cnt * agents;
    cudaStream_t s = h->host_stream[used & 1];
    cudaError_t e = cudaStreamWaitEvent(s, h->host_start, 0);
    if (e == cudaSuccess)
      e = cudaMemcpyAsync(dev->policy_action + v0 * adim, policy_action_host + v0 * adim, sizeof(float) * nv * adim,
                          cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) { rc = fail(VSS_E_CUDA, "vss_step_view_host: H2D copy", e); break; }
    h->range_first = f0; h->range_count = (f0 == 0 && cnt == h->n) ? 0 : cnt;
    rc = vss_step_view(h, view, dev->policy_action, dev->action_buf, dev->reset_buf, dev->obs_v, dev->term_obs_v, dev->rews_v,
                       dev->reward_v, dev->done_v, dev->timeout_v, dev->progress_v, dev->ep_ret, dev->ep_len, dev->ret_ret,
                       dev->ret_len, s);
    if (rc != VSS_OK) break;
    e = cudaMemcpyAsync(static_cast<char*>(rows_host) + v0 * VSS_PACKED_ROW_BYTES,
                        static_cast<const char*>(dev->packed_rows) + v0 * VSS_PACKED_ROW_BYTES,
                        (size_t)nv * VSS_PACKED_ROW_BYTES, cudaMemcpyDeviceToHost, s);
    if (e != cudaSuccess) { rc = fail(VSS_E_CUDA, "vss_step_view_host: D2H copy", e); break; }
  }
  h->packed_rows = saved_packed; h->range_first = saved_first; h->range_count = saved_count;
  for (int i = 0; i < 2 && i < used; ++i) {  // join (also after an error: nothing of this call stays in flight)
    cudaEventRecord(h->host_done[i], h->host_stream[i]);
    cudaStreamWaitEvent(st, h->host_done[i], 0);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (rc != VSS_OK) {  // a step abandoned after some of its range launches: forget the partial CTA count
    unsigned long long zero = 0;
    cudaMemcpy(h->d_step + 1, &zero, sizeof(zero), cudaMemcpyHostToDevice);
    return rc;
  }
  if (e != cudaSuccess) return fail(VSS_E_CUDA, "vss_step_view_host: synchronize", e);
  return VSS_OK;
}

VSS_API int vss_set_step_aux(vss_handle h, void* obs_bf16, float* done_f32, float* timeout_f32) {
  if (!h) return fail(VSS_E_INVALID, "vss_set_step_aux: null handle");
  h->aux_obs_bf16 = obs_bf16; h->aux_done_f = done_f32; h->aux_timeout_f = timeout_f32;
  return VSS_OK;
}

VSS_API int vss_set_view_opponent(vss_handle h, const vss_view_opponent* opp) {
  if (opp) {  // everything that needs no handle first
    const int m = opp->mode;
    if (m < VSS_TEAM_ZERO || m > VSS_TEAM_EXTERNAL) return fail(VSS_E_INVALID, "vss_set_view_opponent: unknown team mode");
    if ((m == VSS_TEAM_SA || m == VSS_TEAM_CMA || m == VSS_TEAM_DMA) && !opp->policy_action)
      return fail(VSS_E_INVALID, "vss_set_view_opponent: a policy opponent needs its policy action");
  }
  if (!h) return fail(VSS_E_INVALID, "vss_set_view_opponent: null handle");
  h->opp = opp ? *opp : vss_view_opponent{VSS_TEAM_OU, 0, nullptr, nullptr, nullptr};
  return VSS_OK;
}

VSS_API int vss_set_step_packed(vss_handle h, void* rows) {
  if (!h) return fail(VSS_E_INVALID, "vss_set_step_packed: null handle");
  if (reinterpret_cast<uintptr_t>(rows) & 15u) return fail(VSS_E_INVALID, "vss_set_step_packed: rows must be 16-byte aligned");
  h->packed_rows = rows;
  return VSS_OK;
}

VSS_API int vss_set_step_warps_per_tile(vss_handle h, int warps) {
  if (!h) return fail(VSS_E_INVALID, "vss_set_step_warps_per_tile: null handle");
  if (warps < 0 || warps > MAX_WPT) return fail(VSS_E_INVALID, "vss_set_step_warps_per_tile: 0 (automatic) .. 8");
  h->wpt_override = warps;
  return VSS_OK;
}
VSS_API int vss_step_warps_per_tile(vss_handle h) {
  return h ? launch_shape(h->n, true, h->wpt_override, h->fpt_override).wpt : 0;
}

VSS_API int vss_set_step_fields_per_tile(vss_handle h, int fields) {
  if (!h) return fail(VSS_E_INVALID, "vss_set_step_fields_per_tile: null handle");
  if (fields != 0 && fields != 8 && fields != 16 && fields != 32)
    return fail(VSS_E_INVALID, "vss_set_step_fields_per_tile: 0 (automatic), 8, 16 or 32");
  h->fpt_override = fields;
  return VSS_OK;
}
VSS_API int vss_step_fields_per_tile(vss_handle h) {
  return h ? launch_shape(h->n, true, h->wpt_override, h->fpt_override).fpw : 0;
}

#ifdef VSS_PHASE_PROFILE
VSS_API int vss_prof_read_integrate(unsigned long long* out, int ctas) {  // out[ctas][16]
  return cudaMemcpyFromSymbol(out, vss::g_integ_prof, sizeof(unsigned long long) * 16 * (size_t)ctas) == cudaSuccess ? 0 : -1;
}
VSS_API int vss_prof_read(unsigned long long* out, int ctas) {  // profiling build only: out[ctas][8] clock totals
  return cudaMemcpyFromSymbol(out, vss::g_phase_prof, sizeof(unsigned long long) * 8 * (size_t)ctas) == cudaSuccess ? 0 : -1;
}
#endif

VSS_API int64_t vss_step_granularity(vss_handle h) {
  if (!h) return 0;
  const LaunchShape ls = launch_shape(h->n, true, h->wpt_override, h->fpt_override);
  return ls.wpt > 1 ? ls.fpw : (int64_t)ls.wpb * ls.fpw;
}

VSS_API int vss_set_step_range(vss_handle h, int64_t first_field, int64_t num_fields) {
  if (!h) return fail(VSS_E_INVALID, "vss_set_step_range: null handle");
  if (first_field < 0 || num_fields < 0 || first_field + num_fields > h->n)
    return fail(VSS_E_INVALID, "vss_set_step_range: range outside [0, num_envs)");
  h->range_first = num_fields ? first_field : 0; h->range_count = num_fields;
  return VSS_OK;
}

VSS_API int vss_get_state(vss_handle h, float* state_out, void* stream) {
  if (!h || !state_out) return fail(VSS_E_INVALID, "vss_get_state: null argument");
  if (int rc = use_device(h)) return rc;
  VSS_CUDA(cudaMemcpyAsync(state_out, h->state, sizeof(float) * VSS_STATE_WORDS * (size_t)h->ld,
                           cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return VSS_OK;
}

VSS_API int vss_render(vss_handle h, int64_t first_field, int32_t num_fields, int32_t height, int32_t width,
                       uint8_t* rgb, void* stream) {
  if (!rgb) return fail(VSS_E_INVALID, "vss_render: null rgb");
  if (reinterpret_cast<uintptr_t>(rgb) & 15u) return fail(VSS_E_INVALID, "vss_render: rgb must be 16-byte aligned");
  if (height % 16 != 0 || height < 64 || height > 4096)
    return fail(VSS_E_INVALID, "vss_render: height must be a multiple of 16 in [64, 4096]");
  if (width % 16 != 0 || width < 64 || width > 4096)
    return fail(VSS_E_INVALID, "vss_render: width must be a multiple of 16 in [64, 4096]");
  if (!h) return fail(VSS_E_INVALID, "vss_render: null handle");
  if (num_fields < 1) return fail(VSS_E_INVALID, "vss_render: num_fields must be >= 1");
  if (first_field < 0 || first_field > h->n - num_fields)
    return fail(VSS_E_INVALID, "vss_render: fields outside [0, num_envs)");
  const long long ctas_per_frame = ((long long)height * (width / 16) + RENDER_THREADS - 1) / RENDER_THREADS;
  if (ctas_per_frame * num_fields > 0x7FFFFFFFLL)
    return fail(VSS_E_INVALID, "vss_render: too many pixels for one launch (split the fields)");
  if (int rc = use_device(h)) return rc;
  const RenderFrame g = render_frame(h->params, height, width);
  k_render<<<(unsigned)(ctas_per_frame * num_fields), RENDER_THREADS, 0, (cudaStream_t)stream>>>(
      h->state, h->ld, first_field, height, width, ctas_per_frame, g, rgb);
  VSS_CUDA(cudaGetLastError());
  return VSS_OK;
}

VSS_API int vss_set_state(vss_handle h, const float* state_in, void* stream) {
  if (!h || !state_in) return fail(VSS_E_INVALID, "vss_set_state: null argument");
  if (int rc = use_device(h)) return rc;
  VSS_CUDA(cudaMemcpyAsync(h->state, state_in, sizeof(float) * VSS_STATE_WORDS * (size_t)h->ld,
                           cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return VSS_OK;
}

VSS_API int vss_gae(const float* rewards, const float* values, const float* next_values, const float* next_dones,
                    const float* next_timeouts, float* advantages, float* returns, int32_t T, int64_t N,
                    double gamma, double gae_lambda, void* stream) {
  if (!rewards || !values || !next_values || !next_dones || !next_timeouts || !advantages || !returns)
    return fail(VSS_E_INVALID, "vss_gae: null argument");
  if (T <= 0 || N <= 0) return fail(VSS_E_INVALID, "vss_gae: T and N must be > 0");
  // 64 columns per CTA: at N = 65536 that is 1024 CTAs = 6.9 per SM (128 per CTA: 3.46 per SM, i.e. a
  // quarter of the SMs carry a third more columns than the rest)
  const int gae_block = 64;
  const unsigned grid = (unsigned)((N + gae_block - 1) / gae_block);
  // prefetch while the batch has fewer than ~28 warps per SM (measured: N = 65536 51.7 -> 39.8 us with it,
  // N = 196608 112.8 -> 122.9 us)
  const bool prefetch = N <= 131072;
  if (prefetch)
    k_gae<true><<<grid, gae_block, 0, (cudaStream_t)stream>>>(rewards, values, next_values, next_dones, next_timeouts,
                                                            advantages, returns, T, N, (float)gamma,
                                                            (float)(gamma * gae_lambda));
  else
    k_gae<false><<<grid, gae_block, 0, (cudaStream_t)stream>>>(rewards, values, next_values, next_dones, next_timeouts,
                                                             advantages, returns, T, N, (float)gamma,
                                                             (float)(gamma * gae_lambda));
  VSS_CUDA(cudaGetLastError());
  return VSS_OK;
}

VSS_API void vss_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
  const U4 r = philox4x32_10(U4{ctr[0], ctr[1], ctr[2], ctr[3]}, key[0], key[1]);
  out[0] = r.x; out[1] = r.y; out[2] = r.z; out[3] = r.w;
}

}  // extern "C"
