/*
 * vss_b200.h — C-ABI of libvss_b200.so, the B200-native VSS (3v3 robot soccer)
 * hot path: fused env step, masked reset, agent views, GAE, PPO MLP.
 *
 * This is the drop-in boundary UNDER the reference's Python seam (envs/vss.py
 * class VSS, envs/wrappers.py views, ppo_continuous_action_isaacgym.py loop).
 * The reference has no FFI of its own: every entry point below replaces a run of
 * IsaacGym `gymapi`/`gymtorch` calls plus torch-jit code, cited per function as
 * `file:line` into the reference tree.
 *
 * Conventions
 *   - plain C: pointers + sizes, no torch types. All `float*`/`int64_t*`/`uint8_t*`
 *     data pointers are DEVICE pointers owned by the caller (torch); the engine
 *     borrows them for the duration of the call. Layouts are the reference's
 *     row-major tensor layouts, stated per argument.
 *   - `stream` is a `cudaStream_t` passed as `void*` (0 = legacy default stream).
 *     Every call only enqueues work; there is NO host synchronisation inside.
 *   - return 0 on success, negative `VSS_E_*` on failure; `vss_last_error()` gives
 *     the message (thread-local).
 *   - one handle per device; a handle is not thread-safe.
 *   - there is no CPU fallback: `vss_create` fails if the device is not sm_100.
 */
#ifndef VSS_B200_H
#define VSS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VSS_API __attribute__((visibility("default")))

/* ---- fixed problem shape (envs/vss.py:24-25,80-92; vss.yaml:4-5) ---- */
#define VSS_NUM_TEAMS 2
#define VSS_NUM_ROBOTS 3
#define VSS_NUM_OBS 52
#define VSS_NUM_ACTIONS 2
#define VSS_NUM_REW 4
#define VSS_OBS_PER_FIELD (VSS_NUM_TEAMS * VSS_NUM_ROBOTS * VSS_NUM_OBS) /* 312 */
#define VSS_ACT_PER_FIELD (VSS_NUM_TEAMS * VSS_NUM_ROBOTS * VSS_NUM_ACTIONS) /* 12 */
#define VSS_REW_PER_FIELD (VSS_NUM_TEAMS * VSS_NUM_ROBOTS * VSS_NUM_REW) /* 24 */

/* Engine state, SoA in HBM: word w of field e lives at state[w * ld + e].
 * Words 0..3   ball x, y, vx, vy
 * Words 4+9r+k robot r = team*3 + idx; k: x, y, vx, vy, cos(yaw), sin(yaw), yaw-rate,
 *              last action left, last action right      (= vss.py:541-551 feature order)
 * Word 58      progress counter (int32 bit pattern)     (vss.py:95 progress_buf)
 * Word 59      episode counter  (uint32 bit pattern; keys the reset RNG)            */
#define VSS_STATE_FLOATS 58
#define VSS_STATE_WORDS 60
#define VSS_W_PROGRESS 58
#define VSS_W_EPISODE 59

/* error codes */
#define VSS_OK 0
#define VSS_E_INVALID (-1)   /* bad argument */
#define VSS_E_CUDA (-2)      /* CUDA runtime error */
#define VSS_E_NODEVICE (-3)  /* no sm_100 device / no CPU fallback */
#define VSS_E_NOMEM (-4)

/* agent views, envs/wrappers.py:89-180 */
#define VSS_VIEW_SA 0  /* SingleAgent: controls blue robot 0          */
#define VSS_VIEW_CMA 1 /* CMA: one 6-dim action for blue robots 0-2   */
#define VSS_VIEW_DMA 2 /* DMA: blue robots 0-2 as 3 separate agents   */

typedef struct vss_engine* vss_handle;

/* Physical + task constants. Defaults (vss_default_params) are extracted from the
 * reference scene code: envs/vss.py:48-49,342-345,368-434,436-522, vss_robot.urdf,
 * vss.yaml. The physics model itself is new (PhysX is closed); see DESIGN.md §3. */
typedef struct vss_params {
  /* simulation, vss.yaml:16, vss.yaml:6 */
  float dt;                   /* 0.05 s control step */
  int32_t substeps;           /* physics substeps per control step (4) */
  int32_t max_episode_length; /* 400 */
  /* field, vss.py:342-345 */
  float field_half_length;    /* 0.75  (field_width / 2) */
  float field_half_width;     /* 0.65  (field_height / 2) */
  float goal_half_width;      /* 0.2   (goal_height / 2) */
  float goal_depth;           /* 0.1   (goal_width) */
  /* ball, vss.py:380-389 */
  float ball_radius;          /* 0.02134 */
  float ball_mass;            /* 0.046 kg (density 1130) */
  float ball_drag;            /* 1/s: rolling sphere under PhysX angular damping 0.5 -> 2/7*0.5 */
  /* robot, vss_robot.urdf:3-68 */
  float robot_half_size;      /* 0.035 (0.07 collision box) */
  float robot_mass;           /* 0.44 kg = body 0.4 + 2 wheels 0.02 */
  float robot_inertia;        /* yaw inertia, kg m^2 */
  float wheel_radius;         /* 0.024 */
  float wheel_half_track;     /* 0.03375 */
  float wheel_coll_radius;    /* 0.024 wheel collision sphere (robot-robot only) */
  /* wheel drive, vss.py:47,427-434, urdf:59,67 */
  float max_wheel_rad_s;      /* 42.0 */
  float drive_damping;        /* 0.01 N m s/rad velocity-drive gain */
  float drive_max_torque;     /* 0.1 N m effort limit */
  float wheel_inertia;        /* armature 2e-4 + sphere 0.4 m r^2 */
  float mu_traction;          /* 0.7 longitudinal traction limit */
  float mu_lateral;           /* 0.55 lateral sliding friction */
  float gravity;              /* 9.81 */
  /* contacts */
  float restitution;          /* 0 (PhysX default materials) */
  float mu_ball_robot;        /* 0.5 */
  float mu_ball_wall;         /* 1.0 */
  float mu_robot_wall;        /* 0.5 */
  /* reset distribution, vss.py:49,142-147,267-327 */
  float reset_scale_x;        /* 1.5 - 0.14 */
  float reset_scale_y;        /* 1.3 - 0.14 */
  float min_placement_dist;   /* 0.07 */
  float ball_reset_speed;     /* 1.0: ball velocity ~ (U-0.5)*this */
  /* reward weights, vss.yaml:8-12 (mutable at run time, ppo...:389-392) */
  float w_goal, w_grad, w_move, w_energy;
  /* OU noise of uncontrolled robots, wrappers.py:5-19 */
  float ou_theta;             /* 0.1 */
  float ou_sigma;             /* 0.15 */
} vss_params;

/* Fill `p` with the reference's constants. */
VSS_API int vss_default_params(vss_params* p);

/* Replaces VSS.__init__ -> create_sim / allocate_buffers / _acquire_tensors
 * (envs/vss.py:32-175, 341-522): allocates the SoA state for `num_envs` fields on
 * CUDA device `device`. `global_env_offset` is the global id of local field 0 (keys
 * the counter-based RNG so results do not depend on how fields are sharded). All
 * fields start flagged for reset, like reset_buf = ones (vss.py:93). */
VSS_API int vss_create(vss_handle* out, const vss_params* p, int64_t num_envs,
                       int64_t global_env_offset, int device, uint64_t seed);
VSS_API int vss_destroy(vss_handle h);

VSS_API int64_t vss_num_envs(vss_handle h);
/* leading dimension (in fields) of the SoA state: num_envs rounded up to 32 */
VSS_API int64_t vss_state_ld(vss_handle h);

/* w = {goal, grad, move, energy}; replaces attribute writes at ppo...:389-392. */
VSS_API int vss_set_reward_weights(vss_handle h, const float w[4]);

/* Replaces reset_dones() + compute_observations() (envs/vss.py:72-73, 267-333,
 * 205-216): re-randomise every field whose reset_buf entry is != 0 (reset_buf is
 * NOT cleared, as in the reference), then write obs (N,2,3,52) for all fields.
 * reset_buf: (N) int64, device. */
VSS_API int vss_reset_dones(vss_handle h, const int64_t* reset_buf, float* obs, void* stream);

/* Replaces VecTask.step -> pre_physics_step / gym.simulate / post_physics_step
 * (envs/vss.py:180-203, 218-333 and the six jit functions :530-655).
 *   actions   in  (N,2,3,2) f32, clamped to [-1,1] inside (vss.yaml:7)
 *   reset_buf io  (N) int64: flags from the previous step in, this step's dones out
 *   obs       out (N,2,3,52) post-reset observation          (vss.py:203)
 *   term_obs  out (N,2,3,52) pre-reset "terminal_observation" (vss.py:195-196); may be NULL
 *   rew       out (N,2,3,4)  {goal,grad,move,energy} * weights (vss.py:223-255)
 *   timeout   out (N) uint8  (progress >= max_len-1) & reset  (VecTask.step)
 *   progress_f out (N) f32   un-reset progress counter         (vss.py:198-200); may be NULL */
VSS_API int vss_step(vss_handle h, const float* actions, int64_t* reset_buf, float* obs,
                     float* term_obs, float* rew, uint8_t* timeout, float* progress_f,
                     void* stream);

/* Parity hook ("identical input states"): same as vss_step, but the physics phase
 * is replaced by loading the post-physics state from `post_state` (58 x ld floats,
 * SoA as above; the two last-action words are ignored and taken from `actions`).
 * Everything else (progress, rewards, dones, obs, masked reset, timeouts) runs
 * through the same code as vss_step. */
VSS_API int vss_step_injected(vss_handle h, const float* actions, const float* post_state,
                              int64_t* reset_buf, float* obs, float* term_obs, float* rew,
                              uint8_t* timeout, float* progress_f, void* stream);

/* Fused agent-view step: replaces SingleAgent/CMA/DMA.step (envs/wrappers.py:101-115,
 * 133-148, 163-180) + random_ou (:5-19) + VSS.step + RecordEpisodeStatisticsTorch.step
 * (:66-87) in ONE launch. N' = N (sa, cma) or 3N (dma); A = 2 (sa, dma) or 6 (cma).
 *   policy_action in  (N',A) f32
 *   action_buf    io  (N,2,3,2) f32 persistent OU state of the view (wrappers.py:94)
 *   reset_buf     io  (N) int64 (the VSS reset_buf)
 *   obs_v         out (N',52)  view observation after reset
 *   term_obs_v    out (N',52)  view terminal observation
 *   rews_v        out (N',4)   infos['rews']
 *   reward_v      out (N')     rews.sum(-1)
 *   done_v        out (N') int64
 *   timeout_v     out (N') uint8
 *   progress_v    out (N') f32
 *   ep_ret/ep_len io  (N',4) f32 / (N') int32 running episode statistics, or NULL
 *   ret_ret/ret_len out (N',4) f32 / (N') int32 statistics snapshot before masking, or NULL */
VSS_API int vss_step_view(vss_handle h, int view, const float* policy_action, float* action_buf,
                          int64_t* reset_buf, float* obs_v, float* term_obs_v, float* rews_v,
                          float* reward_v, int64_t* done_v, uint8_t* timeout_v, float* progress_v,
                          float* ep_ret, int32_t* ep_len, float* ret_ret, int32_t* ret_len,
                          void* stream);

#define VSS_PACKED_ROW_BYTES 112
/* The same step for a caller on the HOST side of the PCIe link: one call takes the policy action from pinned
 * host memory and returns one packed VSS_PACKED_ROW_BYTES-byte row per view env (see vss_set_step_packed) in
 * pinned host memory — what `SingleAgent/CMA/DMA.step` hands the policy (envs/wrappers.py:108-115). Internally the
 * fields are cut into `num_ranges` ranges, each with its own H2D copy of its actions, kernel launch and ONE D2H
 * copy of its rows, alternating over two streams owned by the engine, so that the copies of one range overlap the
 * kernel of the next; the call orders itself after the work already queued on `stream` and returns when the rows
 * are in host memory. `dev` holds the view's device buffers exactly as vss_step_view takes them (+ the device
 * staging for the rows); they keep the ordinary outputs of the step. Results are bit-identical to one vss_step_view
 * launch over all fields. */
typedef struct vss_view_buffers {
  float* policy_action;   /* device copy of the action, (N', act dim) */
  float* action_buf;
  int64_t* reset_buf;
  float* obs_v;
  float* term_obs_v;
  float* rews_v;
  float* reward_v;
  int64_t* done_v;
  uint8_t* timeout_v;
  float* progress_v;
  float* ep_ret;          /* the four statistics buffers may be NULL together */
  int32_t* ep_len;
  float* ret_ret;
  int32_t* ret_len;
  void* packed_rows;      /* device staging, N' x VSS_PACKED_ROW_BYTES */
} vss_view_buffers;
VSS_API int vss_step_view_host(vss_handle h, int view, const vss_view_buffers* dev, const float* policy_action_host,
                               void* rows_host, int num_ranges, void* stream);

/* Optional side outputs of the following vss_step_view launches (each may be NULL = off), for a
 * caller that feeds the observation straight into a bf16 tensor-core MLP and the flags into a float
 * GAE (the PPO loop, ppo_continuous_action_isaacgym.py:258-272, 282-296):
 *   obs_bf16     (N',64) bf16: the view observation rounded to nearest even; columns 52..63 are
 *                never written (zero the buffer once);
 *   done_f32     (N') f32: done_v as 0.0f / 1.0f;   timeout_f32 (N') f32: timeout_v as 0.0f / 1.0f.
 * Host-side state of the handle (no device work, no synchronisation); the pointers are read when
 * vss_step_view is called, so they may change from step to step. */
VSS_API int vss_set_step_aux(vss_handle h, void* obs_bf16, float* done_f32, float* timeout_f32);

/* Optional packed per-agent output of the following vss_step_view launches (NULL = off), for a caller
 * on the HOST side of the PCIe link (what SingleAgent/CMA/DMA.step returns to the policy,
 * envs/wrappers.py:108-115, in as few bytes as carry it): one row of VSS_PACKED_ROW_BYTES = 112 bytes
 * per view env,
 *   bytes   0..103  the 52 observation values as bf16 (round to nearest even)
 *   bytes 104..107  the scalar reward, f32
 *   byte  108       done (0 / 1)          byte 109  time-out (0 / 1)          bytes 110..111  zero
 * `rows` is any pointer the device can write: device memory (staging for one cudaMemcpyAsync per field
 * range) or pinned host memory (cudaHostAlloc is device-mapped under unified addressing: the kernel then
 * stores straight across PCIe and no copy is issued at all). Host-side state of the handle, like
 * vss_set_step_aux. */
VSS_API int vss_set_step_packed(vss_handle h, void* rows);

/* Restricts the following vss_step / vss_step_view launches to the fields [first_field, first_field +
 * num_fields) (num_fields = 0: the whole engine again). Buffers keep their whole-engine shapes and base
 * pointers; only the rows of the range are read and written. For a caller that pipelines one step over
 * several streams (host copies of chunk c overlapping the kernel of chunk c+1): the chunks of ONE step
 * may run concurrently, every field must be covered exactly once per step, and the next step's launches
 * must be ordered after all of them (the OU-noise step index is counted over the whole engine).
 * first_field and num_fields must be multiples of vss_step_granularity(h), except that the last range
 * may end at num_envs. Host-side state of the handle, like vss_set_step_aux. */
VSS_API int64_t vss_step_granularity(vss_handle h);

/* Launch shape of the step kernels: how many warps share one 32-field tile. 1 = one warp per tile (one
 * lane per field walks the 6 robots and the ball in turn: the shape of large batches, HBM-bound);
 * 2..8 = the bodies of a tile are dealt to that many warps, which shortens the critical path of a tile
 * (small and medium batches, latency-bound). 0 (default) = chosen from num_envs. Every shape computes
 * bit-identical results; the setter exists for tuning runs and for the parity tests that cover all of
 * them. Changes vss_step_granularity(). Host-side state of the handle. */
VSS_API int vss_set_step_warps_per_tile(vss_handle h, int warps);
VSS_API int vss_step_warps_per_tile(vss_handle h);

/* Launch shape of the step kernels, second knob: how many fields form a tile (32, 16 or 8; 0 = chosen from
 * num_envs). With fewer fields per tile the lanes beyond the tile idle in the per-field phases (and help in
 * the cooperative observation writes), there are more tiles to spread over the SMs, and the divergent
 * contact code of a tile - which runs field after field - forms a shorter chain. Bit-identical results for
 * every value; covered by the same parity tests as vss_set_step_warps_per_tile. Changes
 * vss_step_granularity(). Host-side state of the handle. */
VSS_API int vss_set_step_fields_per_tile(vss_handle h, int fields);
VSS_API int vss_step_fields_per_tile(vss_handle h);
VSS_API int vss_set_step_range(vss_handle h, int64_t first_field, int64_t num_fields);

/* ---- match evaluation: play.py::play_matches (reference play.py:131-164) on the device ----
 * One team per side, each driving its 6 action slots of the (N,2,3,2) buffer in one of these modes
 * (reference play.py:26-64):
 *   ZERO      TeamZero: act[:] *= 0 (the previous values times 0: the sign of zero is kept)
 *   OU        TeamOU: the OU draw (wrappers.py:5-19)
 *   SA        TeamSA: the OU draw, then robot 0 = policy_action (N,2)
 *   CMA       TeamCMA: the 6 slots = policy_action (N,6)
 *   DMA       TeamDMA / ppo-sa-x3: the 6 slots = policy_action (3N,2) (= (N,6))
 *   EXTERNAL  any other team: the slots are left as the caller wrote them into the buffer */
#define VSS_TEAM_ZERO 0
#define VSS_TEAM_OU 1
#define VSS_TEAM_SA 2
#define VSS_TEAM_CMA 3
#define VSS_TEAM_DMA 4
#define VSS_TEAM_EXTERNAL 5
typedef struct vss_match_team {
  int32_t mode;                /* VSS_TEAM_* */
  int32_t reserved;
  const float* policy_action;  /* SA (N,2), CMA (N,6), DMA (3N,2) f32; required by those modes, ignored otherwise */
  void* rows_bf16;             /* SA / CMA (N,64), DMA (3N,64) bf16, or NULL: the team's rows of the post-reset
                                  observation (robot 0, or robots 0-2; yellow = the mirrored obs[:,1] rows) rounded
                                  to nearest even, columns 52..63 never written - the input of the team's next
                                  policy call. Ignored by the other modes. */
} vss_match_team;
/* Scoreboard of a match evaluation (device memory, 40 bytes, zeroed by the caller before the first step):
 * the statistics the reference's loop accumulates (play.py:152-164). */
typedef struct vss_match_board {
  int64_t matches;     /* episodes that ended among the fields < count_envs, counted while not frozen */
  int64_t length_sum;  /* sum of their un-reset progress counters (info["progress_buffer"]) */
  double score_sum;    /* sum of their rew[env,0,0,0]: the goal term of blue robot 0 with the weights as set */
  int64_t steps;       /* steps counted, the one that froze the board included */
  uint32_t frozen;     /* set at the end of the step in which `matches` reached n_matches; later steps count
                          nothing, so a caller may run steps past it (a captured chunk) without changing the
                          result: score = score_sum / matches, length = length_sum / matches */
  uint32_t reserved;
} vss_match_board;
/* One step of a two-team match: what play_matches does per iteration (both team calls + VSS.step +
 * the statistics), in one launch. The action prologue reads action_buf, draws the views' OU noise
 * (Philox stream 2 keyed by the device step index) on all 12 slots, applies each team's mode, stores
 * the buffer back un-clamped and clamps it into the state; a done field's row is NOT zeroed (play_matches
 * carries the OU state across resets). Outputs: reset_buf (io, as vss_step), the teams' bf16 rows, obs
 * (N,2,3,52) f32 post-reset (may be NULL: only EXTERNAL teams need it) and the scoreboard. No terminal
 * observation, no f32 rewards. Advances the step index like vss_step_view. Whole-engine launches only:
 * rejected while vss_set_step_range is active. */
VSS_API int vss_step_match(vss_handle h, const vss_match_team teams[2], float* action_buf, int64_t* reset_buf,
                           float* obs, int64_t count_envs, int64_t n_matches, vss_match_board* board, void* stream);

/* ---- training against an opponent: a team in the yellow slots of the view step ----
 * With an opponent set, every vss_step_view launch (whole-engine or a vss_set_step_range range) is one opponent view
 * step. Restatement (what the tests check the kernels against):
 *   1. action_buf = random_ou(action_buf) on all 12 slots (Philox stream 2 keyed by the device step index, as today);
 *   2. the learner's slots = policy_action, exactly as the view does without an opponent;
 *   3. the 6 yellow slots follow the opponent's mode (VSS_TEAM_*):
 *        OU        keep the draw: no opponent; vss_step_view runs today's kernel
 *        ZERO      draw x 0 (act[:] *= 0 on the drawn buffer: the sign of zero is kept)
 *        SA        robot 0 = policy_action (N,2); robots 1-2 keep the draw
 *        CMA / DMA the 6 slots = policy_action (N,6) / (3N,2)
 *        EXTERNAL  the slots as the caller wrote them before the step (the noise is drawn, not stored there);
 *   4. everything else is the view step: the buffer is stored un-clamped and clamped into the state; physics,
 *      rewards, dones, the learner's outputs, episode statistics and aux outputs are unchanged; done rows of
 *      action_buf are zeroed (all 12 slots);
 *   5. after the masked reset, for every field: rows_bf16 = the opponent's policy input, the yellow rows (the
 *      mirrored obs[:,1]) rounded to nearest even and padded to 64 columns, columns 52..63 never written: robot 0
 *      -> row env (SA / CMA), robot i -> row 3 env + i (DMA); obs_f32 = the yellow team's (N,3,52) observation.
 * Extra HBM bytes per field-step: policy action in 8 (SA) / 24 (CMA, DMA); bf16 rows out 104 (SA, CMA) / 312 (DMA);
 * obs_f32 624 when requested. */
typedef struct vss_view_opponent {
  int32_t mode;               /* VSS_TEAM_*; OU = no opponent (today's kernel) */
  int32_t reserved;
  const float* policy_action; /* SA (N,2), CMA (N,6), DMA (3N,2); required by those modes */
  void* rows_bf16;            /* SA/CMA (N,64), DMA (3N,64) bf16, or NULL */
  float* obs_f32;             /* (N,3,52) yellow post-reset obs, or NULL */
} vss_view_opponent;
/* Sets (opp) or clears (NULL) the opponent of the following vss_step_view launches. Host-side state of the handle,
 * like vss_set_step_aux: the struct is copied, its pointers are read when vss_step_view is called, so a captured
 * graph records them. Arguments are checked before anything else (unknown mode, a policy mode without
 * policy_action, then the handle). vss_step_view_host returns VSS_E_INVALID while an opponent is set; vss_step and
 * vss_step_match ignore it. */
VSS_API int vss_set_view_opponent(vss_handle h, const vss_view_opponent* opp);

/* State access for parity tests and checkpointing: copies the SoA state
 * (VSS_STATE_WORDS x ld 32-bit words) device->device. */
VSS_API int vss_get_state(vss_handle h, float* state_out, void* stream);
VSS_API int vss_set_state(vss_handle h, const float* state_in, void* stream);
/* The reference's viewer / RecordVideo frames (ppo…:213-221, play.py:134-142, vss.py:16-23,389,412-417), drawn
 * from the state on the device: renders fields [first_field, first_field + num_fields) of the current state into
 * `rgb`, (num_fields, height, width, 3) uint8 RGB, row-major. The picture is exact and defined per pixel in
 * csrc/vss_render.cuh (DESIGN.md §4.7): field, goals, lines, ball, and the six robots with their team colour
 * behind and their ID colour in front of the centre; 560 x 720 is 400 px/m. A frame shows the state as it is
 * (after a step, a field that ended an episode is shown already reset). Reads the state only: no counter or handle
 * state changes; no synchronisation and no allocation, so a CUDA graph can capture it. Arguments are checked
 * before anything else (rgb null or not 16-byte aligned; height / width not a multiple of 16 in [64, 4096]; then
 * the handle; then num_fields >= 1 and the range inside [0, num_envs)). */
VSS_API int vss_render(vss_handle h, int64_t first_field, int32_t num_fields, int32_t height, int32_t width,
                       uint8_t* rgb, void* stream);
/* number of view steps executed so far (keys the OU-noise RNG of the views; vss_step draws no noise
 * and does not advance it). The counter is device-resident and advanced by the step kernel itself — by
 * the CTA that completes the step, counted over all the range launches of that step — so CUDA-graph
 * replays of a captured vss_step_view launch advance it too; these two calls synchronise with the
 * device. vss_set_step_count also forgets a partially issued step (a caller that abandons a step after
 * some of its range launches must call it before the next step); values above UINT32_MAX are rejected
 * (the index is one 32-bit word of the Philox counter). */
VSS_API uint64_t vss_step_count(vss_handle h);
/* Safety net that the reference does not have: a field whose state is not finite at the end of the
 * physics (a blow-up of the 2-D model; never observed in the stress tests) is re-randomised on the spot
 * and reported with done = 1, time-out = 0 and zero reward, so that one bad field cannot poison a
 * training run. This returns how many fields that has happened to over the engine's life (device
 * counter; the call synchronises). A non-zero value is worth a look. */
VSS_API uint64_t vss_sanitised_count(vss_handle h);
VSS_API int vss_set_step_count(vss_handle h, uint64_t n);

/* Replaces the GAE loop, ppo_continuous_action_isaacgym.py:282-296. All arrays (T,N) f32
 * row-major, device. adv and ret are outputs. gamma/lambda are the python doubles; they are
 * rounded to f32 exactly where torch rounds them (gamma, gamma*lambda). */
VSS_API int vss_gae(const float* rewards, const float* values, const float* next_values,
                    const float* next_dones, const float* next_timeouts, float* advantages,
                    float* returns, int32_t T, int64_t N, double gamma, double gae_lambda,
                    void* stream);

/* Tensor-core GEMM of the PPO MLPs (tcgen05 / TMEM / TMA, csrc/tc_gemm.cu): replaces the cuBLAS
 * GEMM + bias + tanh launches behind nn.Linear/nn.Tanh of the reference's Agent
 * (ppo_continuous_action_isaacgym.py:127-164) and their autograd backward (:352).
 *   C[M,N] = epilogue(op(A) * op(B)^T), bf16 operands, fp32 accumulation.
 *   mn_major = 0: A [M,K], B [N,K] row-major (forward: A = activations, B = nn.Linear weight;
 *                 dgrad: A = dZ, B = weight^T). mn_major = 1: A [K,M], B [K,N] row-major (wgrad:
 *                 dW = dZ^T X with the batch as K; no transposed copies needed).
 *   epilogue: 0 out_bf16 = tanh(acc + bias[n]); 1 out_bf16 = acc * (1 - aux[m,n]^2) (aux bf16);
 *             2 out_f32 += acc (atomic, split-K; caller zeroes out); 3 out_f32 = acc + bias[n].
 *   lda/ldb/ldo/ld_aux in elements; K multiple of 64 (K-major), N multiple of 64. lda/ldb: multiples of 8, at least
 *   the row they hold (K; M/N with mn_major). ldo >= N, a multiple of 8 for bf16 outputs and of 4 for epilogue 3;
 *   out (epilogues 0, 1, 3) and bias 16-byte aligned; epilogue 1: ld_aux >= N, a multiple of 8, aux 16-byte
 *   aligned. Other layouts return VSS_E_INVALID before any CUDA call. */
VSS_API int vss_gemm_bf16_tn(const void* A, int lda, const void* B, int ldb, void* out, int ldo, int M,
                             int N, int K, int epilogue, const float* bias, const void* aux, int ld_aux,
                             int splits, int mn_major, void* stream);
/* The same with one more output (dgrad epilogue 1 only, mn_major = 0, N <= 512): colsum[N] (f32) +=
 * column sums of the bf16 output, i.e. the bias gradient of the layer below; NULL = plain GEMM. */
VSS_API int vss_gemm_bf16_tn_colsum(const void* A, int lda, const void* B, int ldb, void* out, int ldo, int M,
                                    int N, int K, int epilogue, const float* bias, const void* aux, int ld_aux,
                                    int splits, int mn_major, float* colsum, void* stream);
VSS_API const char* vss_gemm_last_error(void);
/* out[N] (f32) += column sums of the bf16 matrix x [M,N] (row stride ld): bias gradients. N and ld even, ld >= N,
 * x 4-byte aligned. */
VSS_API int vss_colsum_bf16(const void* x, int ld, int M, int N, float* out, void* stream);
/* dst [M,ncol_pad] bf16 = zero-padded src[idx[m] (or m if idx is NULL), :ncol] f32: the minibatch
 * gather b_obs[mb_inds] (ppo...:314) fused with the bf16 conversion and K padding. ncol_pad even, dst 4-byte
 * aligned. */
VSS_API int vss_gather_pad_bf16(const float* src, const int64_t* idx, int M, int ncol, int ncol_pad, void* dst,
                                void* stream);

/* Output head of the Agent MLPs (Linear 256 -> n_out in {1,2,6}, ppo...:138,151) and its backward
 * fused with tanh' of the last hidden layer: dz = (dout W) * (1 - h^2) (bf16), dW += dout^T h,
 * db += sum dout; dz_colsum [256] += column sums of dz (bias gradient of the last hidden layer) when
 * not NULL. h [M,256] bf16, W [n_out,256] f32, out/dout [M,n_out] f32. ldh/ldz >= 256 and multiples of 8, h and dz
 * 16-byte aligned. */
VSS_API int vss_head_forward(const void* h, int ldh, const float* W, const float* b, float* out, int M, int n_out,
                             void* stream);
VSS_API int vss_head_backward(const float* dout, const void* h, int ldh, const float* W, void* dz, int ldz,
                              float* dW, float* db, float* dz_colsum, int M, int n_out, void* stream);

/* The whole Agent MLP forward in ONE launch (csrc/mlp_fused.cu): for each of n_nets (1 or 2) networks that share the
 * input rows - the actor mean and the critic value of the same observations, Agent.get_action_and_value,
 * ppo...:155-164 called once per rollout step at ppo...:259-261 -
 *   out [M, n_out] f32 = Linear(256, n_out)(tanh-MLP(x)),  MLP = obs -> 256 -> 512 -> 512 -> 256 (ppo...:130-152).
 * x16 [M, 64] bf16: the observations zero-padded to 64 columns (what vss_set_step_aux's obs_bf16 output and
 * vss_gather_pad_bf16 produce), row stride ldx elements. w[l] bf16 row-major [256,64], [512,256], [512,512], [256,512]
 * (nn.Linear layout, the first K-padded to 64), b[l] f32; head_w f32 [n_out, 256], head_b f32 [n_out]; n_out in
 * {1, 2, 6}. The hidden activations never leave the SM (shared memory / TMEM); same per-element arithmetic as four
 * vss_gemm_bf16_tn(EPI_BIAS_TANH_BF16) + vss_head_forward. epilogue_warps: 0 (default), 4 or 8 - a tuning knob with
 * identical results. All pointers 16-byte aligned. */
typedef struct vss_mlp_net {
  const void* w[4];
  const float* b[4];
  const float* head_w;
  const float* head_b;
  float* out;
  int32_t n_out;
  int32_t reserved;
} vss_mlp_net;
/* Optional: draw the action in the same launch (network 0 = the actor mean, n_out = action width 2 or 6):
 * action = Normal(out_0, exp(logstd)).sample(), logprob = log_prob(action).sum(1) - the arithmetic and the Philox stream
 * of vss_policy_sample, with call index *counter + call_offset. The launch does NOT advance *counter: a caller that
 * captures T steps in a CUDA graph passes call_offset = 0..T-1 and adds T to the counter once per rollout.
 * nets[0].out may then be NULL (the mean is not stored). */
typedef struct vss_mlp_sampling {
  const float* logstd;      /* f32 [n_out] */
  const uint32_t* counter;  /* device word */
  uint64_t seed;
  uint32_t call_offset;
  uint32_t reserved;
  float* action;            /* f32 [M, n_out] */
  float* logprob;           /* f32 [M] */
} vss_mlp_sampling;
VSS_API int vss_mlp_forward_fused(const void* x16, int ldx, int M, const vss_mlp_net* nets, int n_nets,
                                  const vss_mlp_sampling* sampling, int epilogue_warps, void* stream);
/* The same launch with a profiling hook: the first CTA records 11 %globaltimer stamps (ns) at its phase boundaries
 * into stamps (device memory, NULL = none): [0] entry, [1] barriers + TMEM ready, [2 + 2l] first accumulator chunk of
 * hidden layer l complete, [3 + 2l] epilogue of layer l done (one epilogue warp's view), [10] exit. */
VSS_API int vss_mlp_forward_fused_timed(const void* x16, int ldx, int M, const vss_mlp_net* nets, int n_nets,
                                        const vss_mlp_sampling* sampling, int epilogue_warps,
                                        unsigned long long* stamps, void* stream);

/* ---- the small pieces of the PPO loop, one launch each (ppo_continuous_action_isaacgym.py) ------
 * Normal(mean, exp(logstd)).sample() and .log_prob(action).sum(1) of Agent.get_action_and_value
 * (ppo...:155-164). mean/action (M,A) f32, logstd (A), logprob (M); A in {2,6}. Normals come from
 * Philox4x32-10 keyed by (seed, *counter, row); `counter` is a device word that the call advances
 * (stream-ordered, so CUDA-graph replays draw fresh noise). */
VSS_API int vss_policy_sample(const float* mean, const float* logstd, int64_t M, int A, uint64_t seed,
                              uint32_t* counter, float* action, float* logprob, void* stream);
/* The rows of a rollout whose step ended an episode, as a compact list (any order): list[k] = index of the k-th
 * non-zero entry of flags[0..n), *count = their number (device words; *count may exceed cap - entries beyond cap are
 * dropped and the caller must check). And its inverse for per-row results: dst[list[k]] = src[k], k < min(*count, cap).
 * Used for V(terminal_observation) (ppo...:272): for a row that did NOT end an episode the terminal observation IS the
 * next observation, whose value the per-step critic pass has already produced, so only the listed rows need the critic. */
VSS_API int vss_compact_nonzero(const float* flags, int64_t n, int64_t* list, int cap, int* count, void* stream);
VSS_API int vss_scatter_rows_f32(float* dst, const int64_t* list, const float* src, const int* count, int cap,
                                 void* stream);
/* One PPO minibatch loss and its gradient w.r.t. the network outputs (ppo...:314-352):
 *   j = inds[i] (or i when inds is NULL) gathers the rollout arrays b_* (flattened (T*N,...) f32);
 *   mean (B,A) / value (B) are the fresh network outputs for those rows; logstd (A).
 *   ratio, approx-KL, clip fraction, advantage normalisation (mean / unbiased std + 1e-8) when
 *   norm_adv, clipped surrogate, value loss (clipped when clip_vloss; b_val may be NULL otherwise),
 *   entropy bonus; loss = pg - ent_coef * entropy + vf_coef * v_loss.
 * Outputs: d_mean (B,A), d_value (B) = d loss / d output; d_logstd (A) is ACCUMULATED (caller
 * zeroes); stats[8] = {pg_loss, v_loss, entropy, old_approx_kl, approx_kl, clipfrac, loss, 0};
 * scratch = 2 doubles of device workspace. */
VSS_API int vss_ppo_loss(const float* mean, const float* value, const float* logstd, const float* b_action,
                         const float* b_logprob, const float* b_adv, const float* b_ret, const float* b_val,
                         const int64_t* inds, int64_t B, int A, float clip_coef, float ent_coef, float vf_coef,
                         int norm_adv, int clip_vloss, float* d_mean, float* d_value, float* d_logstd, float* stats,
                         double* scratch, void* stream);
/* bf16 copies of fp32 matrices in one launch: dst[r, c] = src[r, c], or dst[c, r] = src[r, c] when
 * transpose; src (rows, cols) contiguous, dst row stride ld_dst elements (K padding of the first
 * layer: the caller zeroes the pad columns once). Up to VSS_MAX_CONVERT_JOBS matrices per call. */
#define VSS_MAX_CONVERT_JOBS 8
typedef struct vss_convert_job {
  const float* src;
  void* dst;
  int32_t rows, cols, ld_dst, transpose;
} vss_convert_job;
VSS_API int vss_convert_bf16_batch(const vss_convert_job* jobs, int njobs, void* stream);
/* nn.utils.clip_grad_norm_(max_grad_norm) + Adam.step() (torch semantics, no weight decay) on flat
 * buffers of n f32 (ppo...:353-354). The gradient is first scaled by grad_scale (1 / world size after
 * a sum all-reduce). state (device, 3 f32) = {step count, learning rate, 0}; the call increments the
 * step count on the device, so it can be replayed from a CUDA graph. grads holds the clipped
 * gradient afterwards. */
VSS_API int vss_clip_adam(float* params, float* grads, float* exp_avg, float* exp_avg_sq, int64_t n, float* state,
                          float grad_scale, float max_grad_norm, float beta1, float beta2, float eps, void* stream);
VSS_API const char* vss_ppo_last_error(void);

/* ---- the PPO gradient all-reduce over NVLink peer memory (csrc/peer_reduce.cu) -----------------------
 * Replaces `torch.distributed.all_reduce(flat_grad)` — the data-parallel form of the reference's
 * single-GPU `loss.backward(); clip_grad_norm_; optimizer.step()` (ppo…:352-354) — for the ranks of ONE
 * node: one process per GPU, every rank keeps its flat gradient in a buffer of its vss_peer group that
 * the other ranks map through CUDA IPC, and vss_peer_allreduce is ONE kernel per rank that synchronises
 * with the peers through flag words in those buffers and sums all P gradients in rank order (bit-
 * identical results on all ranks), with no host involvement; graph-capturable.
 *   vss_peer_create      allocates the group's buffer on `device` (num_floats floats, rounded up to 4)
 *   vss_peer_ipc_handle  64 opaque bytes to hand to the other ranks (any host-side exchange, e.g.
 *                        torch.distributed.all_gather)
 *   vss_peer_connect     all_handles = world x 64 bytes in rank order (own entry ignored)
 *   vss_peer_buffer      the rank's gradient buffer (device pointer): the backward pass accumulates here
 *   vss_peer_allreduce   out_sum[i] = sum over ranks of buffer_rank[i]; when it has completed on the
 *                        stream the rank's buffer may be overwritten. Collective: every rank must
 *                        call it the same number of times. */
typedef struct vss_peer_group* vss_peer;
#define VSS_PEER_HANDLE_BYTES 64
VSS_API int vss_peer_create(vss_peer* out, int device, int rank, int world, int64_t num_floats);
VSS_API int vss_peer_ipc_handle(vss_peer h, void* handle64);
VSS_API int vss_peer_connect(vss_peer h, const void* all_handles);
VSS_API float* vss_peer_buffer(vss_peer h);
VSS_API int64_t vss_peer_num_floats(vss_peer h);
VSS_API int vss_peer_allreduce(vss_peer h, float* out_sum, void* stream);
VSS_API int vss_peer_destroy(vss_peer h);
VSS_API const char* vss_peer_last_error(void);

/* Philox4x32-10 known-answer hook (host side; same code as the device generator). */
VSS_API void vss_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);

VSS_API const char* vss_last_error(void);
VSS_API const char* vss_version(void);

#ifdef __cplusplus
}
#endif
#endif /* VSS_B200_H */
