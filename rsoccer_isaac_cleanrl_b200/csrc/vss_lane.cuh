// vss_lane.cuh — per-field ("lane") logic of the fused VSS step.
//
// One thread owns one field. Its 60 state words live in a shared-memory column
// S[w * LDS] (LDS = 33: conflict-free both for "every lane reads its own column"
// and for the cooperative row-major observation write). Everything here is plain
// per-lane code with no warp collectives, so the same source also compiles for the
// host (tests/emu) to check the logic without a GPU. The warp-cooperative parts
// (coalesced obs writes, ballots) live in vss_step.cu.
//
// Reference behaviour replaced (file:line in the reference tree):
//   pre_physics_step            envs/vss.py:180-187
//   gym.simulate (PhysX)        new 2-D model, DESIGN.md §3 (scene spec vss.py:341-522)
//   compute_rewards_and_dones   envs/vss.py:218-265, jit :578-655
//   compute_obs                 envs/vss.py:530-575 (obs_entry table below)
//   reset_dones                 envs/vss.py:267-333
//   random_ou                   envs/wrappers.py:5-19
#pragma once
#include <stdint.h>
#include <math.h>
#include <string.h>
#if defined(__CUDACC__)
#include <cuda_bf16.h>
#endif

#include "../../include/vss_b200.h"

#if defined(__CUDACC__)
#define VSS_HD __host__ __device__ __forceinline__
#define VSS_HD_COLD inline __host__ __device__ __noinline__  // rare paths kept out of the hot instruction stream
#else
#define VSS_HD inline
#define VSS_HD_COLD inline
#endif

#ifndef VSS_INTEG_UNROLL
// Robots integrated side by side per lane: instruction-level parallelism vs code size. Since the CTAs of an SM
// no longer run in lock-step (first-wave stagger) the instruction caches are the scarcer resource: same box,
// 2^20 fields, 656.9 us per step at 2, 644.9 us at 1 (before the stagger: 681.8 vs 684.5).
#define VSS_INTEG_UNROLL 1
#endif

namespace vss {

constexpr int INTEG_UNROLL = VSS_INTEG_UNROLL;
#ifndef VSS_OBS_UNROLL
#define VSS_OBS_UNROLL 1  // fields per iteration of the row-owner observation writer: 8 / 4 / 2 / 1 -> 657.3 / 644.5 / 640.2 /
                          // 636.5 us per step at 2^20 fields (code size beats loop overhead: the kernel is fetch-bound)
#endif
constexpr int OBS_UNROLL = VSS_OBS_UNROLL;
constexpr int LDS = 33;       // shared-memory column stride in words
constexpr int W_PREV = 60;    // 7 words of pre-physics reward terms: ball potential, 6 robot-ball distances
constexpr int SM_WORDS = 67;  // words per field staged in shared memory
constexpr int TILE_STATE_WORDS = SM_WORDS * LDS;  // the staged columns of one 32-field tile
// Task queues, per warp of the CTA: 32 x 6 (field, robot) wall tasks of 2 bytes + 32 ball-wall tasks
// of 1 byte (the per-field contact tasks, 32 x 4 bytes, reuse the same space in an earlier phase)
constexpr int QUEUE_WORDS = 104;
constexpr int TILE_WORDS = TILE_STATE_WORDS + QUEUE_WORDS;  // shared-memory words per warp
// k_step_cta (one tile shared by up to MAX_WPT warps): the staged columns + one scratch word per warp
// and field (the warp's share of the broadphase candidate mask)
constexpr int MAX_WPT = 8;
constexpr int W_SCR = SM_WORDS;
constexpr int W_SHADOW = SM_WORDS + MAX_WPT;  // a second set of state columns: the helper warp's speculative resets
constexpr int TILE_CTA_WORDS = (W_SHADOW + VSS_STATE_WORDS) * LDS;
constexpr int F4_PER_FIELD = VSS_OBS_PER_FIELD / 4;  // 78 float4 per (2,3,52) observation
constexpr int F4_PER_ROW = VSS_NUM_OBS / 4;          // 13
constexpr int RESET_MAX_ATTEMPTS = 64;

// Constants derived once on the host (double precision) from vss_params.
struct DevParams {
  float h, H, rb, b, rw, rwc, inv_rw;
  float kd_imp, tmax, wmax, fv, fw, dv_max, du_max, ball_decay;
  float k_act, k_v, k_w;  // wheel torque before the clamp = k_act a - k_v v -+ k_w w (kd_imp folded in)
  float inv_mr, inv_ir, inv_mb, e1, mu_br, mu_bw, mu_rw;
  float HL, HW, GH, GD, br_reach2, rr_reach2, wall_rej_x, wall_rej_y;
  float reset_sx, reset_sy, min_d2, ball_speed;
  float w_goal, w_grad, w_move, w_energy;
  float ou_theta, ou_sigma;
  int substeps, max_len;
};

inline DevParams derive_params(const vss_params& p) {
  DevParams q;
  const double h = (double)p.dt / (double)p.substeps, rw = p.wheel_radius, b = p.wheel_half_track;
  const double jw_lin = (double)p.wheel_inertia / (rw * rw);
  const double m_eff = p.robot_mass + 2.0 * jw_lin, i_eff = p.robot_inertia + 2.0 * jw_lin * b * b;
  const double j_wheel_eq = 0.5 * m_eff * rw * rw;
  const double sq2 = 1.4142135623730951, H = p.robot_half_size;
  q.h = (float)h; q.H = (float)H; q.rb = p.ball_radius; q.b = (float)b; q.rw = (float)rw;
  q.rwc = p.wheel_coll_radius; q.inv_rw = (float)(1.0 / rw);
  q.kd_imp = (float)(p.drive_damping / (1.0 + h * p.drive_damping / j_wheel_eq));
  q.tmax = p.drive_max_torque; q.wmax = p.max_wheel_rad_s;
  {
    const double kd = p.drive_damping / (1.0 + h * p.drive_damping / j_wheel_eq);
    q.k_act = (float)(kd * p.max_wheel_rad_s); q.k_v = (float)(kd / rw); q.k_w = (float)(kd * b / rw);
  }
  q.fv = (float)(h / (rw * m_eff)); q.fw = (float)(b * h / (rw * i_eff));
  q.dv_max = (float)((double)p.mu_traction * p.gravity * h);
  q.du_max = (float)((double)p.mu_lateral * p.gravity * h);
  q.ball_decay = (float)exp(-(double)p.ball_drag * h);
  q.inv_mr = (float)(1.0 / p.robot_mass); q.inv_ir = (float)(1.0 / p.robot_inertia);
  q.inv_mb = (float)(1.0 / p.ball_mass); q.e1 = 1.0f + p.restitution;
  q.mu_br = p.mu_ball_robot; q.mu_bw = p.mu_ball_wall; q.mu_rw = p.mu_robot_wall;
  q.HL = p.field_half_length; q.HW = p.field_half_width; q.GH = p.goal_half_width; q.GD = p.goal_depth;
  const double br = p.ball_radius + H * sq2 + 0.005;
  const double rr0 = H * sq2, wr0 = b + p.wheel_coll_radius;
  const double rr = 2.0 * (rr0 > wr0 ? rr0 : wr0) + 0.01;
  q.br_reach2 = (float)(br * br); q.rr_reach2 = (float)(rr * rr);
  q.wall_rej_x = (float)(p.field_half_length - H * sq2); q.wall_rej_y = (float)(p.field_half_width - H * sq2);
  q.reset_sx = p.reset_scale_x; q.reset_sy = p.reset_scale_y;
  q.min_d2 = p.min_placement_dist * p.min_placement_dist; q.ball_speed = p.ball_reset_speed;
  q.w_goal = p.w_goal; q.w_grad = p.w_grad; q.w_move = p.w_move; q.w_energy = p.w_energy;
  q.ou_theta = p.ou_theta; q.ou_sigma = p.ou_sigma;
  q.substeps = p.substeps; q.max_len = p.max_episode_length;
  return q;
}

// ---- IEEE single ops that must not be contracted into FMAs (bit parity with the oracle) ----
#if defined(__CUDA_ARCH__)
VSS_HD float fadd(float a, float b) { return __fadd_rn(a, b); }
VSS_HD float fsub(float a, float b) { return __fsub_rn(a, b); }
VSS_HD float fmul(float a, float b) { return __fmul_rn(a, b); }
VSS_HD float ffma(float a, float b, float c) { return __fmaf_rn(a, b, c); }
VSS_HD float fsqrt(float a) { return __fsqrt_rn(a); }
VSS_HD float fdiv(float a, float b) { return __fdiv_rn(a, b); }
VSS_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return __umulhi(a, b); }
VSS_HD int ffs32(uint32_t m) { return __ffs((int)m); }
VSS_HD uint32_t fbits(float f) { return __float_as_uint(f); }
VSS_HD float bitsf(uint32_t u) { return __uint_as_float(u); }
#else
VSS_HD float fadd(float a, float b) { return a + b; }  // host build uses -ffp-contract=off
VSS_HD float fsub(float a, float b) { return a - b; }
VSS_HD float fmul(float a, float b) { return a * b; }
VSS_HD float ffma(float a, float b, float c) { return fmaf(a, b, c); }
VSS_HD float fsqrt(float a) { return sqrtf(a); }
VSS_HD float fdiv(float a, float b) { return a / b; }
VSS_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }
VSS_HD int ffs32(uint32_t m) { return __builtin_ffs((int)m); }
VSS_HD uint32_t fbits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
VSS_HD float bitsf(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
#endif

// Quick division / reciprocal square root for the contact code (2 ulp on the device; the physics is
// compared with the fp64 oracle under a tolerance, unlike the rewards, which use the _rn forms above).
// Without -ftz the CUDA intrinsics wrap every MUFU in denormal scaling (9 instructions per
// division); the flush-to-zero forms are one MUFU (+ one FMUL), and no contact quantity is denormal.
#if defined(__CUDA_ARCH__)
VSS_HD float qrcp(float b) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(b)); return r; }
VSS_HD float qdiv(float a, float b) { return a * qrcp(b); }
VSS_HD float qrsqrt(float a) { float r; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(a)); return r; }
#else
VSS_HD float qrcp(float b) { return 1.0f / b; }
VSS_HD float qdiv(float a, float b) { return a / b; }
VSS_HD float qrsqrt(float a) { return 1.0f / sqrtf(a); }
#endif
VSS_HD float clampf(float v, float lo, float hi) { return fminf(fmaxf(v, lo), hi); }
VSS_HD float sgnf(float v) { return v < 0.0f ? -1.0f : 1.0f; }

// ---- Philox4x32-10 (Salmon et al. 2011) ----
struct U4 { uint32_t x, y, z, w; };

VSS_HD U4 philox4x32_10(U4 c, uint32_t k0, uint32_t k1) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    const uint32_t hi0 = mulhi32(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
    const uint32_t hi1 = mulhi32(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
    c = U4{hi1 ^ c.y ^ k0, lo1, hi0 ^ c.w ^ k1, lo0};
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return c;
}

constexpr uint32_t STREAM_RESET_POS = 0, STREAM_RESET_MISC = 1, STREAM_OU = 2;

struct RngKey { uint32_t seed_lo, seed_hi, gid_lo, gid_hi; };

VSS_HD U4 rng_block(const RngKey& k, uint32_t a, uint32_t stream, uint32_t b) {
  return philox4x32_10(U4{k.gid_lo, k.gid_hi, a, (stream << 28) | b}, k.seed_lo, k.seed_hi);
}
VSS_HD float u01(uint32_t x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
VSS_HD float u01_open(uint32_t x) { return (float)((x >> 8) + 1u) * (1.0f / 16777216.0f); }

// ---- observation table: output element (team t, robot i, slot k) -> state word, sign ----
// Layout restated from envs/vss.py:539-574 (SURVEY App. A.1). bit 7 = negate.
constexpr uint32_t obs_entry(int t, int i, int k) {
  int team = 0, robot = 0, f = 0, word = 0;
  bool ball = false;
  if (k < 4) { ball = true; word = k; f = 0; }
  else if (k < 31) { const int m = (k - 4) / 9; f = (k - 4) % 9; team = t; robot = (i + m) % 3; }
  else { const int m = (k - 31) / 7; f = (k - 31) % 7; team = 1 - t; robot = m; }
  if (!ball) word = 4 + 9 * (team * 3 + robot) + f;
  const bool neg = (t == 1) && (ball || f < 6);
  return (uint32_t)word | (neg ? 0x80u : 0u);
}
struct ObsTable { uint32_t v[F4_PER_FIELD]; };
constexpr ObsTable make_obs_table() {
  ObsTable tab{};
  for (int j = 0; j < F4_PER_FIELD; ++j) {
    const int row = j / F4_PER_ROW, q = j % F4_PER_ROW, t = row / 3, i = row % 3;
    uint32_t e = 0;
    for (int c = 0; c < 4; ++c) e |= obs_entry(t, i, 4 * q + c) << (8 * c);
    tab.v[j] = e;
  }
  return tab;
}

struct F4 { float x, y, z, w; };

// One float4 of the observation of field column `e` of the tile whose staging area starts
// at T (T = warp base, NOT lane-offset).
VSS_HD F4 obs_gather(const float* T, uint32_t entry, int e) {
  float v[4];
#pragma unroll
  for (int c = 0; c < 4; ++c) {
    const uint32_t by = (entry >> (8 * c)) & 0xFFu;
    v[c] = bitsf(fbits(T[(by & 0x7Fu) * LDS + e]) ^ ((by >> 7) << 31));
  }
  return F4{v[0], v[1], v[2], v[3]};
}

// ---- rigid bodies -------------------------------------------------------------------
struct Body { float x, y, vx, vy, c, s, w, invm, invi; };

VSS_HD Body load_robot(const float* S, int r, const DevParams& P) {
  const float* b = S + (4 + 9 * r) * LDS;
  return Body{b[0], b[LDS], b[2 * LDS], b[3 * LDS], b[4 * LDS], b[5 * LDS], b[6 * LDS], P.inv_mr, P.inv_ir};
}
VSS_HD void store_robot(float* S, int r, const Body& B) {
  float* b = S + (4 + 9 * r) * LDS;
  b[0] = B.x; b[LDS] = B.y; b[2 * LDS] = B.vx; b[3 * LDS] = B.vy; b[4 * LDS] = B.c; b[5 * LDS] = B.s;
  b[6 * LDS] = B.w;
}
VSS_HD Body load_ball(const float* S, const DevParams& P) {
  return Body{S[0], S[LDS], S[2 * LDS], S[3 * LDS], 1.0f, 0.0f, 0.0f, P.inv_mb, 0.0f};
}
VSS_HD void store_ball(float* S, const Body& B) {
  S[0] = B.x; S[LDS] = B.y; S[2 * LDS] = B.vx; S[3 * LDS] = B.vy;
}
VSS_HD Body static_body() { return Body{0.f, 0.f, 0.f, 0.f, 1.f, 0.f, 0.f, 0.f, 0.f}; }

// Inelastic contact; unit normal n points from P to Q; cp = contact point (world).
VSS_HD void resolve(Body& P, Body& Q, float nx, float ny, float depth, float cpx, float cpy, float e1,
                    float mu, float kt_extra) {
  const float rpx = cpx - P.x, rpy = cpy - P.y, rqx = cpx - Q.x, rqy = cpy - Q.y;
  const float wsum = P.invm + Q.invm;
  if (!(wsum > 0.0f)) return;
  const float iw = qdiv(1.0f, wsum), wp = P.invm * iw, wq = Q.invm * iw;
  P.x -= nx * depth * wp; P.y -= ny * depth * wp;
  Q.x += nx * depth * wq; Q.y += ny * depth * wq;
  float vrx = (Q.vx - Q.w * rqy) - (P.vx - P.w * rpy);
  float vry = (Q.vy + Q.w * rqx) - (P.vy + P.w * rpx);
  const float vn = vrx * nx + vry * ny;
  if (vn >= 0.0f) return;
  const float rnp = rpx * ny - rpy * nx, rnq = rqx * ny - rqy * nx;
  const float kn = wsum + rnp * rnp * P.invi + rnq * rnq * Q.invi;
  const float jn = qdiv(-e1 * vn, kn);
  P.vx -= jn * nx * P.invm; P.vy -= jn * ny * P.invm; P.w -= jn * rnp * P.invi;
  Q.vx += jn * nx * Q.invm; Q.vy += jn * ny * Q.invm; Q.w += jn * rnq * Q.invi;
  if (mu > 0.0f) {
    const float tx = -ny, ty = nx;
    vrx = (Q.vx - Q.w * rqy) - (P.vx - P.w * rpy);
    vry = (Q.vy + Q.w * rqx) - (P.vy + P.w * rpx);
    const float vt = vrx * tx + vry * ty;
    const float rtp = rpx * ty - rpy * tx, rtq = rqx * ty - rqy * tx;
    const float kt = wsum + rtp * rtp * P.invi + rtq * rtq * Q.invi + kt_extra;
    const float jt = clampf(qdiv(-vt, kt), -mu * jn, mu * jn);
    P.vx -= jt * tx * P.invm; P.vy -= jt * ty * P.invm; P.w -= jt * rtp * P.invi;
    Q.vx += jt * tx * Q.invm; Q.vy += jt * ty * Q.invm; Q.w += jt * rtq * Q.invi;
  }
}

// resolve() against a static body (walls, goal posts): Q is the dynamic body and the unit normal n
// points from the wall into Q. Same impulse model with the wall's inverse mass and inertia taken
// as the zeros they are (one division less and none of the dead arithmetic on the wall side; a
// contact `resolve(R, wall, n)` with the robot on the P side is `resolve_static(R, -n)`).
VSS_HD void resolve_static(Body& Q, float nx, float ny, float depth, float cpx, float cpy, float e1, float mu,
                           float kt_extra) {
  const float rqx = cpx - Q.x, rqy = cpy - Q.y;
  Q.x += nx * depth; Q.y += ny * depth;
  float vrx = Q.vx - Q.w * rqy, vry = Q.vy + Q.w * rqx;
  const float vn = vrx * nx + vry * ny;
  if (vn >= 0.0f) return;
  const float rnq = rqx * ny - rqy * nx;
  const float jn = qdiv(-e1 * vn, Q.invm + rnq * rnq * Q.invi);
  Q.vx += jn * nx * Q.invm; Q.vy += jn * ny * Q.invm; Q.w += jn * rnq * Q.invi;
  if (mu > 0.0f) {
    const float tx = -ny, ty = nx;
    vrx = Q.vx - Q.w * rqy; vry = Q.vy + Q.w * rqx;
    const float vt = vrx * tx + vry * ty;
    const float rtq = rqx * ty - rqy * tx;
    const float jt = clampf(qdiv(-vt, Q.invm + rtq * rtq * Q.invi + kt_extra), -mu * jn, mu * jn);
    Q.vx += jt * tx * Q.invm; Q.vy += jt * ty * Q.invm; Q.w += jt * rtq * Q.invi;
  }
}

struct Hit { bool hit; float nx, ny, depth, cpx, cpy; };

// Circle (centre (lx,ly) in the frame of box B, radius rho; rho = 0 -> point) against the oriented
// box of B. Normal (world frame) points out of B towards the circle.
struct Pose { float x, y, c, s; };
VSS_HD Hit circle_vs_box_local(const Pose& B, float H, float lx, float ly, float rho) {
  Hit r;
  r.hit = false; r.nx = r.ny = r.depth = r.cpx = r.cpy = 0.0f;
  float nlx, nly, clx, cly;
  bool face = fabsf(lx) <= H && fabsf(ly) <= H;  // centre inside (or exactly on) the box
  if (!face) {
    const float qx = clampf(lx, -H, H), qy = clampf(ly, -H, H);
    const float ex = lx - qx, ey = ly - qy;
    const float d2 = ex * ex + ey * ey;
    if (d2 >= rho * rho) return r;
    if (d2 > 1e-20f) {
      const float id = qrsqrt(d2);
      nlx = ex * id; nly = ey * id; r.depth = rho - d2 * id; clx = qx; cly = qy;
    } else {
      face = true;  // centre within rounding of the surface: no direction to normalise, use the face rule
    }
  }
  if (face) {  // face of least penetration
    const float pxd = H - fabsf(lx), pyd = H - fabsf(ly);
    if (pxd < pyd) { nlx = sgnf(lx); nly = 0.0f; r.depth = pxd + rho; clx = sgnf(lx) * H; cly = ly; }
    else { nlx = 0.0f; nly = sgnf(ly); r.depth = pyd + rho; clx = lx; cly = sgnf(ly) * H; }
  }
  r.hit = true;
  r.nx = nlx * B.c - nly * B.s; r.ny = nlx * B.s + nly * B.c;
  r.cpx = B.x + clx * B.c - cly * B.s; r.cpy = B.y + clx * B.s + cly * B.c;
  return r;
}
// The same with the circle's centre (px,py) given in the world frame.
VSS_HD Hit circle_vs_box(const Body& B, float H, float px, float py, float rho) {
  const float dx = px - B.x, dy = py - B.y;
  return circle_vs_box_local(Pose{B.x, B.y, B.c, B.s}, H, dx * B.c + dy * B.s, -dx * B.s + dy * B.c, rho);
}

VSS_HD void corner_xy(int k, float H, float& lx, float& ly) {
  lx = (k == 0 || k == 3) ? H : -H;  // (+,+) (-,+) (-,-) (+,-)
  ly = (k < 2) ? H : -H;
}

VSS_HD void ball_robot(float* S, int r, const DevParams& P) {
  Body ball = load_ball(S, P), R = load_robot(S, r, P);
  const Hit h = circle_vs_box(R, P.H, ball.x, ball.y, P.rb);
  if (h.hit) {
    resolve(R, ball, h.nx, h.ny, h.depth, h.cpx, h.cpy, P.e1, P.mu_br, 2.5f * P.inv_mb);
    store_ball(S, ball);
    store_robot(S, r, R);
  }
}

// Detection of the 6 features of one robot (4 box corners, 2 wheel circles) against the box of
// the other, done in the box's frame: (lx, ly) = owner centre, (cr, sr) = rotation of the owner
// relative to the box. Returns bits 0-3 for corners, 4-5 for wheels.
VSS_HD uint32_t features_in_box(float lx, float ly, float cr, float sr, const DevParams& P) {
  const float H = P.H;
  uint32_t hits = 0;
  const float ch = cr * H, sh = sr * H;
  // corner (cx, cy) in (+,+) (-,+) (-,-) (+,-): offset = R_rel * (cx H, cy H)
  const float ox[4] = {ch - sh, -ch - sh, -ch + sh, ch + sh};
  const float oy[4] = {sh + ch, -sh + ch, -sh - ch, sh - ch};
#pragma unroll
  for (int q = 0; q < 4; ++q)
    if (fabsf(lx + ox[q]) < H && fabsf(ly + oy[q]) < H) hits |= 1u << q;
#pragma unroll
  for (int w = 0; w < 2; ++w) {  // wheel centres at local (0, +-b)
    const float wy = w ? -P.b : P.b;
    const float px = lx - sr * wy, py = ly + cr * wy;
    const float ex = px - clampf(px, -H, H), ey = py - clampf(py, -H, H);
    if (ex * ex + ey * ey < P.rwc * P.rwc) hits |= 16u << w;  // (inside the box: ex = ey = 0)
  }
  return hits;
}

// Hits of the features of F flagged in `mask` (4 corners, or 2 wheel circles if `wheels`) against
// the box of G. (lx,ly) = F's centre and (cr,sr) = F's rotation in G's frame at entry, (f0x,f0y) and
// (g0x,g0y) the entry positions; the penetration of each hit is reduced by the separation already
// gained along its normal.
VSS_HD void rr_hits(Body& F, Body& G, float f0x, float f0y, float g0x, float g0y, float lx, float ly, float cr,
                    float sr, uint32_t mask, bool wheels, const DevParams& P) {
  const Pose G0{g0x, g0y, G.c, G.s};  // (contacts move a body but do not turn it)
  while (mask) {
    const int q = ffs32(mask) - 1;
    mask &= mask - 1;
    float fx, fy, rho;  // the feature in F's own frame
    if (wheels) { fx = 0.0f; fy = q ? -P.b : P.b; rho = P.rwc; }
    else { corner_xy(q, P.H, fx, fy); rho = 0.0f; }
    const Hit h = circle_vs_box_local(G0, P.H, lx + (fx * cr - fy * sr), ly + (fx * sr + fy * cr), rho);
    if (h.hit) {
      const float gained = ((F.x - f0x) - (G.x - g0x)) * h.nx + ((F.y - f0y) - (G.y - g0y)) * h.ny;
      resolve(G, F, h.nx, h.ny, fmaxf(h.depth - gained, 0.0f), h.cpx, h.cpy, P.e1, 0.0f, 0.0f);
    }
  }
}

// Robot-robot contact (DESIGN.md §3 C). The 12 features — corners of A in B, corners of B in A,
// wheels of A, wheels of B — are all tested against the poses at entry (one snapshot); the hits
// are then resolved in that order, each penetration reduced by the separation already gained
// along its normal.
VSS_HD void robot_robot(float* S, int i, int j, const DevParams& P) {
  Body A = load_robot(S, i, P), B = load_robot(S, j, P);
  const float dx = A.x - B.x, dy = A.y - B.y;
  const float cd = A.c * B.c + A.s * B.s, sd = A.s * B.c - A.c * B.s;  // rotation of A relative to B
  const float lxb = dx * B.c + dy * B.s, lyb = dy * B.c - dx * B.s;    // A's centre in B's frame
  const float lxa = -(dx * A.c + dy * A.s), lya = -(dy * A.c - dx * A.s);  // B's centre in A's frame
  {  // exact reject (separating-axis bound on the four box axes): nothing can touch
    const float acd = fabsf(cd), asd = fabsf(sd), hc = P.H * (acd + asd);
    const float ex = fmaxf(hc, P.b * asd + P.rwc) + P.H + 1e-5f, ey = fmaxf(hc, P.b * acd + P.rwc) + P.H + 1e-5f;
    const bool a_in_b = fabsf(lxb) < ex && fabsf(lyb) < ey;
    const bool b_in_a = fabsf(lxa) < ex && fabsf(lya) < ey;
    if (!(a_in_b || b_in_a)) return;
  }
  const uint32_t ha = features_in_box(lxb, lyb, cd, sd, P);   // features of A against box B
  const uint32_t hb = features_in_box(lxa, lya, cd, -sd, P);  // features of B against box A
  if (!(ha | hb)) return;
  // resolution order: A corners, B corners, A wheels, B wheels. Feature positions are taken in the
  // box's frame straight from the relative pose of the entry snapshot (as features_in_box did).
  const float a0x = A.x, a0y = A.y, b0x = B.x, b0y = B.y;
#pragma unroll 1
  for (int w = 0; w < 2; ++w) {
    rr_hits(A, B, a0x, a0y, b0x, b0y, lxb, lyb, cd, sd, w ? ha >> 4 : ha & 15u, w != 0, P);
    rr_hits(B, A, b0x, b0y, a0x, a0y, lxa, lya, cd, -sd, w ? hb >> 4 : hb & 15u, w != 0, P);
  }
  store_robot(S, i, A);
  store_robot(S, j, B);
}

// Circle of radius rho at the centre of body Q (the ball) against the static walls.
// Three wall families, each resolved at once with the position re-evaluated.
VSS_HD bool circle_vs_walls(Body& Q, float rho, float mu, float kt_extra, const DevParams& P) {
  bool any = false;
#pragma unroll 1
  for (int pass = 0; pass < 3; ++pass) {
    const float px = Q.x, py = Q.y;
    const float ax = fabsf(px), ay = fabsf(py), sx = sgnf(px), sy = sgnf(py);
    float nx = 0.0f, ny = 0.0f, depth = 0.0f;
    bool hit = false;
    if (pass == 0) {  // side walls y = +-HW
      if (ay > P.HW - rho) { nx = 0.0f; ny = -sy; depth = ay - (P.HW - rho); hit = true; }
    } else if (pass == 1) {  // end-wall blocks [HL,inf) x [GH,inf) in each quadrant
      if (ax >= P.HL && ay >= P.GH) {
        const float dx = ax - P.HL, dy = ay - P.GH;
        if (dx < dy) { nx = -sx; ny = 0.0f; depth = dx + rho; }
        else { nx = 0.0f; ny = -sy; depth = dy + rho; }
        hit = true;
      } else {
        const float qx = fmaxf(ax, P.HL), qy = fmaxf(ay, P.GH);
        const float ex = ax - qx, ey = ay - qy;
        const float d2 = ex * ex + ey * ey;
        if (d2 < rho * rho && d2 > 1e-20f) {
          const float id = qrsqrt(d2);
          nx = sx * ex * id; ny = sy * ey * id; depth = rho - d2 * id; hit = true;
        } else if (d2 < rho * rho) {  // on the block's surface within rounding: push out along x
          nx = -sx; ny = 0.0f; depth = rho; hit = true;
        }
      }
    } else {  // goal back wall x = +-(HL+GD)
      if (ax > P.HL + P.GD - rho) { nx = -sx; ny = 0.0f; depth = ax - (P.HL + P.GD - rho); hit = true; }
    }
    if (hit) {
      resolve_static(Q, nx, ny, depth, px - nx * rho, py - ny * rho, P.e1, mu, kt_extra);
      any = true;
    }
  }
  return any;
}

// The box can reach a wall or a goal post: conservative test with the circumradius H sqrt(2) instead
// of the exact axis-aligned extent H(|c|+|s|) (no heading loads; a robot queued in vain finds no
// corner outside the field and is left untouched, so the result is the same).
VSS_HD bool robot_near_walls(const float* S, int r, const DevParams& P) {
  const float* b = S + (4 + 9 * r) * LDS;
  return !(fabsf(b[0]) < P.wall_rej_x && fabsf(b[LDS]) < P.wall_rej_y);
}

// Wall contacts of robot r of the field whose column starts at S. Touches only that robot, so
// tasks of different (field, robot) pairs are independent and can run on any lane.
// The four box corners are points (radius 0) tested against the same three wall families as the
// ball, in the same order, each hit resolved at once and the corner re-evaluated: a point can only
// touch the end-wall blocks or the goal back wall from |x| >= HL, so those two passes are skipped
// for corners that are not there. Then the goal posts (+-HL, +-GH) against the box faces: a post
// can only be inside the box if it is the one in the robot's own quadrant (the others are at
// least 2 GH = 0.4 m away, the box's circumradius is 0.05 m).
VSS_HD void robot_walls_task(float* S, int r, const DevParams& P) {
  Body R = load_robot(S, r, P);
  bool dirty = false;
  // corner offsets in the world frame; contacts do not change the heading. Corners in the order
  // (+,+) (-,+) (-,-) (+,-): each is the previous one rotated by 90 degrees.
  float ox = P.H * R.c - P.H * R.s, oy = P.H * R.s + P.H * R.c;
#pragma unroll 1
  for (int k = 0; k < 4; ++k) {
    // a corner inside |x| < HL, |y| <= HW touches nothing (most corners of most tasks); hits only push
    // it further inside, so the test need not be repeated between the passes
    if (fabsf(R.y + oy) > P.HW || fabsf(R.x + ox) >= P.HL) {
#pragma unroll 1
      for (int pass = 0; pass < 3; ++pass) {  // uniform trip count: the lanes of a warp stay together
        const float px = R.x + ox, py = R.y + oy;
        const float ax = fabsf(px), ay = fabsf(py);
        float nx = 0.0f, ny = 0.0f, depth = 0.0f;
        bool hit = false;
        if (pass == 0) {  // side walls y = +-HW
          if (ay > P.HW) { ny = -sgnf(py); depth = ay - P.HW; hit = true; }
        } else if (pass == 1) {  // end-wall blocks [HL,inf) x [GH,inf) per quadrant
          if (ax >= P.HL && ay >= P.GH) {
            const float dx = ax - P.HL, dy = ay - P.GH;
            if (dx < dy) { nx = -sgnf(px); depth = dx; }
            else { ny = -sgnf(py); depth = dy; }
            hit = true;
          }
        } else {  // goal back wall x = +-(HL+GD)
          if (ax > P.HL + P.GD) { nx = -sgnf(px); depth = ax - (P.HL + P.GD); hit = true; }
        }
        if (hit) {
          resolve_static(R, nx, ny, depth, px, py, P.e1, P.mu_rw, 0.0f);
          dirty = true;
        }
      }
    }
    const float t = ox; ox = -oy; oy = t;
  }
  {  // the goal post of the robot's quadrant against the box faces
    const float gx = R.x < 0.0f ? -P.HL : P.HL, gy = R.y < 0.0f ? -P.GH : P.GH;
    const float dx = gx - R.x, dy = gy - R.y;
    const float lx = dx * R.c + dy * R.s, ly = -dx * R.s + dy * R.c;
    if (fabsf(lx) <= P.H && fabsf(ly) <= P.H) {  // face of least penetration
      const float pxd = P.H - fabsf(lx), pyd = P.H - fabsf(ly);
      float nlx, nly, depth;
      if (pxd < pyd) { nlx = sgnf(lx); nly = 0.0f; depth = pxd; }
      else { nlx = 0.0f; nly = sgnf(ly); depth = pyd; }
      // the normal points out of the box towards the post: the robot is pushed the other way
      const float nx = nlx * R.c - nly * R.s, ny = nlx * R.s + nly * R.c;
      // contact point on the box face, as circle_vs_box reports it
      const float clx = pxd < pyd ? sgnf(lx) * P.H : lx, cly = pxd < pyd ? ly : sgnf(ly) * P.H;
      resolve_static(R, -nx, -ny, depth, R.x + clx * R.c - cly * R.s, R.y + clx * R.s + cly * R.c, P.e1, P.mu_rw,
                     0.0f);
      dirty = true;
    }
  }
  if (dirty) store_robot(S, r, R);
}

// sin/cos of the small per-substep yaw increment
VSS_HD void sincos_small(float a, float& sa, float& ca) {
  if (fabsf(a) < 0.5f) {  // |w| < 40 rad/s at h = 12.5 ms: Taylor to a^7 / a^8, error < 6e-9
    const float a2 = a * a;
    sa = a * (1.0f + a2 * (-1.0f / 6 + a2 * (1.0f / 120 + a2 * (-1.0f / 5040))));
    ca = 1.0f + a2 * (-0.5f + a2 * (1.0f / 24 + a2 * (-1.0f / 720 + a2 * (1.0f / 40320))));
    return;
  }
#if defined(__CUDA_ARCH__)
  __sincosf(a, &sa, &ca);  // |a| = |w| h stays below a few radians: the fast intrinsic is accurate to ~1e-6 there
#else
  sa = sinf(a); ca = cosf(a);
#endif
}
// A. wheel drive + integration of robot r (DESIGN.md §3)
VSS_HD void integrate_robot(float* S, int r, const DevParams& P) {
  float* b = S + (4 + 9 * r) * LDS;
  float x = b[0], y = b[LDS], vx = b[2 * LDS], vy = b[3 * LDS], c = b[4 * LDS], s = b[5 * LDS];
  float w = b[6 * LDS];
  const float al = b[7 * LDS], ar = b[8 * LDS];
  float v = vx * c + vy * s, u = -vx * s + vy * c;
  // torque = k_imp (42 a - wheel speed), wheel speeds (v -+ w b) / r_w: the constants are folded
  const float tv = P.k_v * v, tw = P.k_w * w;
  const float tl = clampf(P.k_act * al - tv + tw, -P.tmax, P.tmax);
  const float tr = clampf(P.k_act * ar - tv - tw, -P.tmax, P.tmax);
  v += clampf((tl + tr) * P.fv, -P.dv_max, P.dv_max);
  w += (tr - tl) * P.fw;
  u -= clampf(u, -P.du_max, P.du_max);
  vx = v * c - u * s; vy = v * s + u * c;
  x += vx * P.h; y += vy * P.h;
  float sa, ca;
  sincos_small(w * P.h, sa, ca);
  const float c2 = c * ca - s * sa, s2 = s * ca + c * sa;
  // |(c2,s2)|^2 = 1 + O(1e-7): one Newton step of 1/sqrt around 1 renormalises to below 1e-13
  const float inv = 1.5f - 0.5f * (c2 * c2 + s2 * s2);
  b[0] = x; b[LDS] = y; b[2 * LDS] = vx; b[3 * LDS] = vy; b[4 * LDS] = c2 * inv; b[5 * LDS] = s2 * inv;
  b[6 * LDS] = w;
}
// B. ball: exponential rolling drag
VSS_HD void integrate_ball(float* S, const DevParams& P) {
  const float vx = S[2 * LDS] * P.ball_decay, vy = S[3 * LDS] * P.ball_decay;
  S[2 * LDS] = vx; S[3 * LDS] = vy;
  S[0] += vx * P.h; S[LDS] += vy * P.h;
}
// C. broadphase of pair q (0-5: ball-robot q; 6-20: robot pairs in lexicographic order): the bit of the
// candidate mask, from the post-integration positions. PAIR_A / PAIR_B: x word of the two bodies of pair
// q (the y word is the next one): ball = word 0, robot r = word 4 + 9 r. (Constant memory on the device: a
// local constexpr array indexed at run time is rebuilt on the stack at every call.)
#if defined(__CUDACC__)
#define VSS_D __device__ __forceinline__
#define VSS_TABLE __constant__ const
#else
#define VSS_D inline
#define VSS_TABLE static const
#endif
VSS_TABLE unsigned char PAIR_A[21] = {0, 0, 0, 0, 0, 0, 4, 4, 4, 4, 4, 13, 13, 13, 13, 22, 22, 22, 31, 31, 40};
VSS_TABLE unsigned char PAIR_B[21] = {4, 13, 22, 31, 40, 49, 13, 22, 31, 40, 49, 22, 31, 40, 49, 31, 40, 49, 40, 49, 49};
VSS_D uint32_t broadphase_pair(const float* S, int q, const DevParams& P) {
  const float* pa = S + PAIR_A[q] * LDS;
  const float* pb = S + PAIR_B[q] * LDS;
  const float dx = pa[0] - pb[0], dy = pa[LDS] - pb[LDS];
  return dx * dx + dy * dy < (q < 6 ? P.br_reach2 : P.rr_reach2) ? 1u << q : 0u;
}
// The whole candidate mask of one field: bits 0-5 ball-robot r, bits 6-20 robot pairs.
VSS_HD uint32_t broadphase_lane(const float* S, const DevParams& P) {
  uint32_t mask = 0;
  const float bx = S[0], by = S[LDS];
  float rx[6], ry[6];
#pragma unroll
  for (int r = 0; r < 6; ++r) { rx[r] = S[(4 + 9 * r) * LDS]; ry[r] = S[(5 + 9 * r) * LDS]; }
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    const float dx = bx - rx[r], dy = by - ry[r];
    if (dx * dx + dy * dy < P.br_reach2) mask |= 1u << r;
  }
  int bit = 6;
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = i + 1; j < 6; ++j) {
      const float dx = rx[i] - rx[j], dy = ry[i] - ry[j];
      if (dx * dx + dy * dy < P.rr_reach2) mask |= 1u << bit;
      ++bit;
    }
  return mask;
}
// Phases A-B of a substep for one field plus the broadphase of phase C. Returns the 21-bit
// candidate mask: bits 0-5 ball-robot r, bits 6-20 robot pairs in lexicographic order.
VSS_HD uint32_t substep_integrate_lane(float* S, const DevParams& P) {
#pragma unroll(INTEG_UNROLL)
  for (int r = 0; r < 6; ++r) integrate_robot(S, r, P);
  integrate_ball(S, P);
  return broadphase_lane(S, P);  // C. broadphase once, then flagged pairs in fixed order
}

// Narrow phase + impulses of the flagged pairs of one field, in fixed order. Touches only that
// field's column, so any thread of the CTA can run it.
VSS_HD void contacts_task(float* S, uint32_t mask, const DevParams& P) {
  uint32_t mb = mask & 63u;
  while (mb) {
    const int r = ffs32(mb) - 1;
    mb &= mb - 1;
    ball_robot(S, r, P);
  }
  uint32_t mr = mask >> 6;
  while (mr) {
    const int p = ffs32(mr) - 1;
    mr &= mr - 1;
    // lexicographic pair index -> (i, j), 3 bits each
    const uint64_t PI = 0x0 | (0ull << 0) | (0ull << 3) | (0ull << 6) | (0ull << 9) | (0ull << 12) | (1ull << 15) |
                        (1ull << 18) | (1ull << 21) | (1ull << 24) | (2ull << 27) | (2ull << 30) | (2ull << 33) |
                        (3ull << 36) | (3ull << 39) | (4ull << 42);
    const uint64_t PJ = (1ull << 0) | (2ull << 3) | (3ull << 6) | (4ull << 9) | (5ull << 12) | (2ull << 15) |
                        (3ull << 18) | (4ull << 21) | (5ull << 24) | (3ull << 27) | (4ull << 30) | (5ull << 33) |
                        (4ull << 36) | (5ull << 39) | (5ull << 42);
    robot_robot(S, (int)((PI >> (3 * p)) & 7), (int)((PJ >> (3 * p)) & 7), P);
  }
}

// D. which robots can touch a wall (bits 0-5)
VSS_HD uint32_t robots_near_walls_lane(const float* S, const DevParams& P) {
  uint32_t walls = 0;
#pragma unroll
  for (int r = 0; r < 6; ++r) walls |= robot_near_walls(S, r, P) ? (1u << r) : 0u;
  return walls;
}
VSS_HD bool ball_near_walls(const float* S, const DevParams& P) {
  return !(fabsf(S[0]) + P.rb <= P.HL && fabsf(S[LDS]) + P.rb <= P.HW);  // else: cannot touch any wall family
}
VSS_HD void ball_walls_task(float* S, const DevParams& P) {
  Body ball = load_ball(S, P);
  if (circle_vs_walls(ball, P.rb, P.mu_bw, 2.5f * P.inv_mb, P)) store_ball(S, ball);
}

// Phases A-C of a substep for one field. Returns the 6-bit mask of robots that need the wall
// phase D, which the caller runs as (field, robot) tasks spread over the lanes of the warp.
VSS_HD uint32_t substep_pre_lane(float* S, const DevParams& P) {
  const uint32_t mask = substep_integrate_lane(S, P);
  contacts_task(S, mask, P);
  return robots_near_walls_lane(S, P);
}

// Phase E of a substep: ball vs walls.
VSS_HD void substep_ball_walls_lane(float* S, const DevParams& P) {
  if (ball_near_walls(S, P)) ball_walls_task(S, P);
}

// ---- rewards and dones: envs/vss.py:218-265, 578-655 -----------------------------------
VSS_HD float norm2(float x, float y) { return fsqrt(fadd(fmul(x, x), fmul(y, y))); }
VSS_HD float ball_potential(float bx, float by, float gx) {
  return fsub(norm2(fadd(bx, gx), by), norm2(fsub(bx, gx), by));
}
VSS_HD bool is_goal(float bx, float by, const DevParams& P) { return fabsf(bx) > P.HL && fabsf(by) < P.GH; }

// rew[r*4 + c] for r = team*3 + idx. The "prev" halves of the grad and move terms (functions
// of the pre-physics positions only, vss.py:219-220) were staged at W_PREV before the physics.
VSS_HD void rewards_lane(const float* S, const DevParams& P, float rew[VSS_REW_PER_FIELD]) {
  const float bx = S[0], by = S[LDS];
#pragma unroll
  for (int k = 0; k < VSS_REW_PER_FIELD; ++k) rew[k] = 0.0f;
  if (P.w_goal > 0.0f) {
    const bool g = is_goal(bx, by, P);
    // the reference's goal term is an int64 in {-1,0,1} (vss.py:589-594): no negative zero
    float gv = 0.0f, gy = 0.0f;
    if (g && bx > 0.0f) { gv = 1.0f; gy = -1.0f; }
    if (g && bx < 0.0f) { gv = -1.0f; gy = 1.0f; }
#pragma unroll
    for (int r = 0; r < 6; ++r) rew[4 * r + 0] = fmul(r < 3 ? gv : gy, P.w_goal);
  }
  if (P.w_grad > 0.0f) {
    const float grad = fsub(ball_potential(bx, by, P.HL), S[W_PREV * LDS]);
#pragma unroll
    for (int r = 0; r < 6; ++r) rew[4 * r + 1] = fmul(r < 3 ? grad : -grad, P.w_grad);
  }
  if (P.w_move > 0.0f) {
#pragma unroll
    for (int r = 0; r < 6; ++r) {
      const float x = S[(4 + 9 * r) * LDS], y = S[(5 + 9 * r) * LDS];
      const float p_dist = S[(W_PREV + 1 + r) * LDS];
      const float dist = norm2(fsub(x, bx), fsub(y, by));
      rew[4 * r + 2] = fmul(fsub(p_dist, dist), P.w_move);
    }
  }
  if (P.w_energy > 0.0f) {
#pragma unroll
    for (int r = 0; r < 6; ++r) {
      const float al = S[(11 + 9 * r) * LDS], ar = S[(12 + 9 * r) * LDS];
      rew[4 * r + 3] = fmul(-fmul(fadd(fabsf(al), fabsf(ar)), 0.5f), P.w_energy);
    }
  }
}

// ---- masked reset of one field: envs/vss.py:267-333 ---------------------------------------
VSS_HD_COLD void reset_lane(float* S, const DevParams& P, const RngKey& key) {
  const uint32_t ep = fbits(S[VSS_W_EPISODE * LDS]);
  float px[7], py[7];
#pragma unroll 1
  for (uint32_t attempt = 0; attempt < (uint32_t)RESET_MAX_ATTEMPTS; ++attempt) {
    uint32_t u[16];
#pragma unroll
    for (uint32_t b = 0; b < 4; ++b) {
      const U4 g = rng_block(key, ep, STREAM_RESET_POS, (attempt << 2) | b);
      u[4 * b] = g.x; u[4 * b + 1] = g.y; u[4 * b + 2] = g.z; u[4 * b + 3] = g.w;
    }
#pragma unroll
    for (int e = 0; e < 7; ++e) {
      px[e] = fmul(fsub(u01(u[2 * e]), 0.5f), P.reset_sx);
      py[e] = fmul(fsub(u01(u[2 * e + 1]), 0.5f), P.reset_sy);
    }
    bool too_close = false;
#pragma unroll
    for (int a = 0; a < 7; ++a)
#pragma unroll
      for (int b = a + 1; b < 7; ++b) {
        const float dx = fsub(px[a], px[b]), dy = fsub(py[a], py[b]);
        too_close |= ffma(dy, dy, fmul(dx, dx)) < P.min_d2;
      }
    if (!too_close) break;
  }
  const U4 m0 = rng_block(key, ep, STREAM_RESET_MISC, 0), m1 = rng_block(key, ep, STREAM_RESET_MISC, 1);
  const uint32_t m[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
  S[0] = px[0]; S[LDS] = py[0];
  S[2 * LDS] = fmul(fsub(u01(m[6]), 0.5f), P.ball_speed);
  S[3 * LDS] = fmul(fsub(u01(m[7]), 0.5f), P.ball_speed);
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    float* b = S + (4 + 9 * r) * LDS;
    const float yaw = fsub(fmul(u01(m[r]), 6.283185307179586f), 3.141592653589793f);
    b[0] = px[1 + r]; b[LDS] = py[1 + r];
    b[2 * LDS] = 0.0f; b[3 * LDS] = 0.0f;
    b[4 * LDS] = cosf(yaw); b[5 * LDS] = sinf(yaw);
    b[6 * LDS] = 0.0f; b[7 * LDS] = 0.0f; b[8 * LDS] = 0.0f;
  }
  S[VSS_W_EPISODE * LDS] = bitsf(ep + 1u);
}

// ---- OU noise on the 12 action slots of one field: envs/wrappers.py:5-19 -------------------
// Philox block b of the step's OU stream drives slots 4b .. 4b+3 (robots 2b and 2b+1).
VSS_HD void ou_block(float a4[4], const DevParams& P, const RngKey& key, uint32_t step, uint32_t b) {
  const U4 g = rng_block(key, step, STREAM_OU, b);
  const uint32_t u[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const float rad = fsqrt(fmul(-2.0f, logf(u01_open(u[2 * h]))));
    const float ang = fmul(6.283185307179586f, u01(u[2 * h + 1]));
    const float z[2] = {fmul(rad, cosf(ang)), fmul(rad, sinf(ang))};
#pragma unroll
    for (int c = 0; c < 2; ++c) {
      float& v = a4[2 * h + c];
      v = clampf(fadd(fsub(v, fmul(P.ou_theta, v)), fmul(P.ou_sigma, z[c])), -1.0f, 1.0f);
    }
  }
}
VSS_HD void ou_lane(float a[VSS_ACT_PER_FIELD], const DevParams& P, const RngKey& key, uint32_t step) {
#pragma unroll
  for (uint32_t b = 0; b < 3; ++b) ou_block(a + 4 * b, P, key, step, b);
}


// ---- 128-bit / 64-bit global accesses -------------------------------------------------------
#if defined(__CUDA_ARCH__)
VSS_HD F4 ld4(const float* p) { const float4 v = *reinterpret_cast<const float4*>(p); return F4{v.x, v.y, v.z, v.w}; }
VSS_HD void st4(float* p, const F4& v) { *reinterpret_cast<float4*>(p) = make_float4(v.x, v.y, v.z, v.w); }
// streaming store (evict-first): observations are written once and never re-read by this kernel
VSS_HD void st4_stream(float* p, const F4& v) { __stcs(reinterpret_cast<float4*>(p), make_float4(v.x, v.y, v.z, v.w)); }
VSS_HD float ldg(const float* p) { return __ldg(p); }
// four floats -> four bf16 (round to nearest even), one 8-byte store at element offset `off` of `base`
VSS_HD void st_bf16x4(void* base, long long off, const F4& v) {
  const uint32_t lo = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v.x)) |
                      ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v.y)) << 16);
  const uint32_t hi = (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v.z)) |
                      ((uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(v.w)) << 16);
  *reinterpret_cast<uint2*>(reinterpret_cast<unsigned short*>(base) + off) = make_uint2(lo, hi);
}
#else
VSS_HD F4 ld4(const float* p) { return F4{p[0], p[1], p[2], p[3]}; }
VSS_HD void st4(float* p, const F4& v) { p[0] = v.x; p[1] = v.y; p[2] = v.z; p[3] = v.w; }
VSS_HD void st4_stream(float* p, const F4& v) { st4(p, v); }
VSS_HD float ldg(const float* p) { return *p; }
VSS_HD uint32_t bf16_rne(float f) {  // round to nearest even, as __float2bfloat16_rn (NaN stays NaN)
  const uint32_t u = fbits(f);
  if ((u & 0x7FFFFFFFu) > 0x7F800000u) return 0x7FFFu;
  return (u + 0x7FFFu + ((u >> 16) & 1u)) >> 16;
}
VSS_HD void st_bf16x4(void* base, long long off, const F4& v) {
  unsigned short* p = reinterpret_cast<unsigned short*>(base) + off;
  p[0] = (unsigned short)bf16_rne(v.x); p[1] = (unsigned short)bf16_rne(v.y);
  p[2] = (unsigned short)bf16_rne(v.z); p[3] = (unsigned short)bf16_rne(v.w);
}
#endif

constexpr int VIEW_FULL = -1;
constexpr int VIEW_MATCH = 3;  // vss_step_match: two teams, the scoreboard, no terminal observation / f32 rewards
// VIEW_OPP + VSS_VIEW_*: the view step with an opponent in the yellow slots (vss_set_view_opponent). Everything the
// view does is unchanged; the yellow slots follow the opponent's mode instead of the OU draw, and the yellow team's
// post-reset observation is written for the opponent's next call.
constexpr int VIEW_OPP = 8;
VSS_HD constexpr int view_base(int view) { return view >= VIEW_OPP ? view - VIEW_OPP : view; }

struct StepArgs {
  float* state; long long n, ld; unsigned long long goff;  // n = end of the field range of this launch
  long long env_begin;         // first field of this launch (0 unless vss_set_step_range restricts it)
  uint32_t seed_lo, seed_hi;
  // Device words: step_ctr[2] = fields the non-finite guard has re-randomised so far; step_ctr[0] =
  // device-resident step index (keys the OU stream), step_ctr[1] = CTAs of the current step that have finished. The CTA that brings the count to `grid` (the CTAs of a whole-engine
  // launch; a step issued as several range launches adds up to the same number) clears it and advances
  // the index, so a CUDA graph that replays the launch advances the index without a second kernel.
  unsigned long long* step_ctr;
  uint32_t grid;
  const float* actions;        // full: (N,2,3,2)
  const float* inject;         // injected post-physics state (58 x ld) or null
  long long* reset_buf;        // (N) io
  float* obs;                  // full: (N,2,3,52); view: (N',52)
  float* term_obs;             // may be null
  float* rew;                  // full: (N,2,3,4); view: rews_v (N',4)
  uint8_t* timeout;            // (N) or (N')
  float* progress_f;           // (N) or (N'), may be null
  // view mode only
  const float* policy_action; float* action_buf; float* reward_v; long long* done_v;
  float* ep_ret; int* ep_len; float* ret_ret; int* ret_len;
  // optional side outputs of the views (vss_set_step_aux): the observation as bf16 rows padded to 64
  // columns (what the tensor-core MLP reads), done / timeout as floats (what the GAE kernel reads)
  void* obs_bf16; float* done_f; float* timeout_f;
  // optional packed per-agent rows (vss_set_step_packed): 52 bf16 obs | f32 reward | u8 done | u8 timeout | 0
  void* packed;
  int fpw;                     // fields per warp: 32, or 16 / 8 for small batches (idle lanes, shorter critical path)
  int stagger_ns;              // first-wave CTAs start (blockIdx / 148 % 6) * stagger_ns late (0 = off)
  // match mode only (vss_step_match): per team (blue, yellow) its VSS_TEAM_* mode, policy action and bf16 rows; the
  // scoreboard counts the episodes of the fields < count_envs until n_matches
  int team_mode[2];
  const float* team_action[2];
  void* team_rows[2];
  long long count_envs, n_matches;
  // opponent views (VIEW_OPP + v) use team_mode / team_action / team_rows [1] for the yellow team and opp_obs for its
  // (N,3,52) f32 post-reset observation (or null); sharing the board's word keeps the kernel parameters' layout
  union {
    vss_match_board* board;
    float* opp_obs;
  };
};

template <int VIEW>
struct ViewShape {
  static constexpr int F4_PER = (VIEW == VIEW_FULL || VIEW == VIEW_MATCH)
                                    ? F4_PER_FIELD
                                    : (view_base(VIEW) == VSS_VIEW_DMA ? 3 * F4_PER_ROW : F4_PER_ROW);
  static constexpr int AGENTS = view_base(VIEW) == VSS_VIEW_DMA ? 3 : 1;  // view "envs" per field
};

// The output rows of the tile whose first field is env0: observation, terminal observation (or null) and, for the
// views only, the same rows as bf16 padded to 64 columns and the packed rows (each or null).
struct TileOut { float* ob; float* tob; void* obh; void* pk; };
template <int VIEW>
VSS_HD TileOut tile_out(const StepArgs& a, long long env0) {
  constexpr int PER_FIELD = ViewShape<VIEW>::F4_PER, AGENTS = ViewShape<VIEW>::AGENTS;
  TileOut o;
  o.ob = a.obs + env0 * (PER_FIELD * 4);
  o.tob = a.term_obs ? a.term_obs + env0 * (PER_FIELD * 4) : nullptr;
  o.obh = (VIEW != VIEW_FULL && a.obs_bf16)
              ? static_cast<void*>(static_cast<unsigned short*>(a.obs_bf16) + env0 * (AGENTS * 64))
              : nullptr;
  o.pk = (VIEW != VIEW_FULL && a.packed)
             ? static_cast<void*>(static_cast<char*>(a.packed) + env0 * (AGENTS * VSS_PACKED_ROW_BYTES))
             : nullptr;
  return o;
}

VSS_HD uint32_t step_index(const StepArgs& a) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__ldcg(a.step_ctr);  // read at L2, where the advancing CTA's add lands
#else
  return (uint32_t)*a.step_ctr;
#endif
}

VSS_HD RngKey make_key(const StepArgs& a, long long env) {
  const unsigned long long gid = a.goff + (unsigned long long)env;
  return RngKey{a.seed_lo, a.seed_hi, (uint32_t)gid, (uint32_t)(gid >> 32)};
}

VSS_HD void load_state(float* S, const float* state, long long ld, long long env) {
  const float* src = state + env;
#pragma unroll
  for (int w = 0; w < VSS_STATE_WORDS; ++w) S[w * LDS] = ldg(src + (long long)w * ld);
}
VSS_HD void store_state(const float* S, float* state, long long ld, long long env) {
  float* dst = state + env;
#pragma unroll
  for (int w = 0; w < VSS_STATE_WORDS; ++w) dst[(long long)w * ld] = S[w * LDS];
}

// Does the step draw OU noise? The views do; a match does if a team needs it (TeamOU, and robots 1-2 of TeamSA).
template <int VIEW>
VSS_HD bool draws_ou(const StepArgs& a) {
  if (VIEW != VIEW_MATCH) return VIEW != VIEW_FULL;
  return a.team_mode[0] == VSS_TEAM_OU || a.team_mode[0] == VSS_TEAM_SA || a.team_mode[1] == VSS_TEAM_OU ||
         a.team_mode[1] == VSS_TEAM_SA;
}
// Action slot k (0..5) of a team after its call (play.py:34-64), from the team's mode and policy action (SA (N,2),
// CMA (N,6), DMA (3N,2): the same 6 floats per field). `found` is the buffer as the team finds it (the previous value
// in a match, the OU draw in a view), `prev` the value the caller wrote, `ou` the slot's OU draw. The C-ABI entries
// accept only the VSS_TEAM_* modes.
VSS_HD float team_slot(int mode, const float* action, long long env, int k, float found, float prev, float ou) {
  switch (mode) {
    case VSS_TEAM_ZERO: return fmul(found, 0.0f);  // act[:] *= 0 keeps the sign of zero
    case VSS_TEAM_SA: return k < 2 ? action[2 * env + k] : ou;
    case VSS_TEAM_CMA:
    case VSS_TEAM_DMA: return action[6 * env + k];
    case VSS_TEAM_EXTERNAL: return prev;
    default: return ou;  // OU
  }
}

// The slots 4b .. 4b+3 (robots 2b, 2b+1) that drive the step, un-clamped (vss.py:180-187; wrappers.py:102-103), in
// place: `act` holds the block's OU draw where draws_ou (else the loaded values), `prev` the values loaded from the
// buffer. Full contract: the caller's actions. Views: the OU draw with the learner's policy action in its slots and,
// with an opponent, the opponent's yellow slots. Match: each team's slots.
template <int VIEW>
VSS_HD void action_slots(float act[4], const float prev[4], long long env, const StepArgs& a, int b) {
  if (VIEW == VIEW_MATCH) {
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int s = 4 * b + q, t = s >= 6 ? 1 : 0;
      act[q] = team_slot(a.team_mode[t], a.team_action[t], env, s - 6 * t, prev[q], prev[q], act[q]);
    }
  } else if (VIEW != VIEW_FULL) {
    if (view_base(VIEW) == VSS_VIEW_SA) {  // act_view[:] = action
      if (b == 0) { act[0] = a.policy_action[2 * env]; act[1] = a.policy_action[2 * env + 1]; }
    } else {  // cma (N,6) and dma (3N,2): the same 6 contiguous floats per field
      for (int q = 4 * b; q < 6 && q < 4 * b + 4; ++q) act[q - 4 * b] = a.policy_action[6 * env + q];
    }
    if (VIEW >= VIEW_OPP) {  // the opponent's call on act[:, 1] (slots 6..11)
#pragma unroll
      for (int q = 0; q < 4; ++q)
        if (4 * b + q >= 6)
          act[q] = team_slot(a.team_mode[1], a.team_action[1], env, 4 * b + q - 6, act[q], prev[q], act[q]);
    }
  }
}

// Phase 1a of a step for one field: state in, actions (+OU noise), progress restart, prev clones.
template <int VIEW>
VSS_HD void lane_phase1a(float* S, long long env, const StepArgs& a, const DevParams& P, const RngKey& key) {
  // state in: 60 coalesced loads in flight per lane
  load_state(S, a.state, a.ld, env);
  // actions: the whole row is loaded before any OU work
  float act[VSS_ACT_PER_FIELD];
  {
    const float* ap = (VIEW == VIEW_FULL ? a.actions : a.action_buf) + env * VSS_ACT_PER_FIELD;
#pragma unroll
    for (int q = 0; q < 3; ++q) {
      const F4 v = ld4(ap + 4 * q);
      act[4 * q] = v.x; act[4 * q + 1] = v.y; act[4 * q + 2] = v.z; act[4 * q + 3] = v.w;
    }
  }
  float prev[VSS_ACT_PER_FIELD];
#pragma unroll
  for (int q = 0; q < VSS_ACT_PER_FIELD; ++q) prev[q] = act[q];
  if (draws_ou<VIEW>(a)) ou_lane(act, P, key, step_index(a));
#pragma unroll
  for (int b = 0; b < 3; ++b) action_slots<VIEW>(act + 4 * b, prev + 4 * b, env, a, b);
  if (VIEW != VIEW_FULL) {  // the buffer keeps the un-clamped values (views zero done rows in phase 5, a match does not)
    float* ap = a.action_buf + env * VSS_ACT_PER_FIELD;
#pragma unroll
    for (int q = 0; q < 3; ++q) st4(ap + 4 * q, F4{act[4 * q], act[4 * q + 1], act[4 * q + 2], act[4 * q + 3]});
  }
  if (a.reset_buf[env] != 0) S[VSS_W_PROGRESS * LDS] = bitsf(0u);  // flags of the previous step, vss.py:182-183
#pragma unroll
  for (int r = 0; r < 6; ++r) {  // dof_velocity_buf[:] = clamp(actions), vss.py:184 + VecTask clip
    S[(11 + 9 * r) * LDS] = clampf(act[2 * r], -1.0f, 1.0f);
    S[(12 + 9 * r) * LDS] = clampf(act[2 * r + 1], -1.0f, 1.0f);
  }
  // prev_* clones, vss.py:219-220
  {
    const float pbx = S[0], pby = S[LDS];
    S[W_PREV * LDS] = ball_potential(pbx, pby, P.HL);
#pragma unroll
    for (int r = 0; r < 6; ++r)
      S[(W_PREV + 1 + r) * LDS] = norm2(fsub(S[(4 + 9 * r) * LDS], pbx), fsub(S[(5 + 9 * r) * LDS], pby));
  }
}

// ---- the same phase 1a in pieces, for the kernel that spreads one tile over several warps -------
// (k_step_cta: warp j owns bodies j, j+W, ...; body 0-5 = robot, 6 = ball).
VSS_HD void load_state_words(float* S, const float* state, long long ld, long long env, int w0, int wstep) {
  const float* src = state + env;
  for (int w = w0; w < VSS_STATE_WORDS; w += wstep) S[w * LDS] = ldg(src + (long long)w * ld);
}
VSS_HD void store_state_words(const float* S, float* state, long long ld, long long env, int w0, int wstep) {
  float* dst = state + env;
  for (int w = w0; w < VSS_STATE_WORDS; w += wstep) dst[(long long)w * ld] = S[w * LDS];
}
// Action slots 4b .. 4b+3 of the field (robots 2b, 2b+1): load, action_slots, write-back of the buffer, clamp into
// the state.
template <int VIEW>
VSS_HD void actions_block(float* S, long long env, const StepArgs& a, const DevParams& P, const RngKey& key, int b) {
  float* ab = const_cast<float*>(VIEW == VIEW_FULL ? a.actions : a.action_buf) + env * VSS_ACT_PER_FIELD + 4 * b;
  const F4 v = ld4(ab);
  float act[4] = {v.x, v.y, v.z, v.w};
  const float prev[4] = {v.x, v.y, v.z, v.w};
  if (draws_ou<VIEW>(a)) ou_block(act, P, key, step_index(a), (uint32_t)b);
  action_slots<VIEW>(act, prev, env, a, b);
  if (VIEW != VIEW_FULL) st4(ab, F4{act[0], act[1], act[2], act[3]});
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int r = 2 * b + k;
    S[(11 + 9 * r) * LDS] = clampf(act[2 * k], -1.0f, 1.0f);
    S[(12 + 9 * r) * LDS] = clampf(act[2 * k + 1], -1.0f, 1.0f);
  }
}
// prev_* clone of one body (vss.py:219-220): ball potential (body 6) or robot-ball distance
VSS_HD void prev_term_body(float* S, int body, const DevParams& P) {
  const float pbx = S[0], pby = S[LDS];
  if (body == 6) S[W_PREV * LDS] = ball_potential(pbx, pby, P.HL);
  else S[(W_PREV + 1 + body) * LDS] = norm2(fsub(S[(4 + 9 * body) * LDS], pbx), fsub(S[(5 + 9 * body) * LDS], pby));
}
// Walls of one body after the pair contacts (phases D / E), in place
VSS_HD void walls_body(float* S, int body, const DevParams& P) {
  if (body == 6) { if (ball_near_walls(S, P)) ball_walls_task(S, P); }
  else if (robot_near_walls(S, body, P)) robot_walls_task(S, body, P);
}

// Parity hook: take the post-physics state from `inject` instead of simulating.
VSS_HD void lane_inject(float* S, long long env, const StepArgs& a) {
  const float* inj = a.inject + env;
#pragma unroll
  for (int w = 0; w < VSS_STATE_FLOATS; ++w) {
    const bool is_act = w >= 4 && ((w - 4) % 9) >= 7;
    if (!is_act) S[w * LDS] = ldg(inj + (long long)w * a.ld);
  }
}

// All dynamic state words of the field are finite.
VSS_HD bool state_finite(const float* S) {
  float acc = 0.0f;
#pragma unroll
  for (int w = 0; w < VSS_STATE_FLOATS; ++w) {
    const bool is_act = w >= 4 && ((w - 4) % 9) >= 7;
    if (!is_act) acc = fmaf(S[w * LDS], 0.0f, acc);  // 0 * finite = 0; 0 * inf = NaN; NaN stays NaN
  }
  return acc == 0.0f;
}

enum : int { LANE_RUNNING = 0, LANE_DONE = 1, LANE_SANITISED = 2 };

// step_ctr[2]: fields re-randomised by the non-finite guard over the engine's life (vss_sanitised_count)
VSS_HD_COLD void count_sanitised(const StepArgs& a) {
#if defined(__CUDA_ARCH__)
  atomicAdd(a.step_ctr + 2, 1ull);
#else
#pragma omp atomic
  a.step_ctr[2] += 1ull;
#endif
}

// Phase 1d: post_physics_step — progress, rewards, dones, per-field outputs (vss.py:189-193,
// 218-265). Returns LANE_DONE if the episode ended this step (masked reset follows in phase 3).
// Safety net (not in the reference): a field whose state is not finite is re-randomised on the
// spot and reported as done with zero reward (LANE_SANITISED), so that one bad field cannot
// poison a training run.
// `finite` = state_finite(S) at the end of the physics; a field that was not finite has already been
// re-randomised by the caller (lane_sanitise).
VSS_HD_COLD void lane_sanitise(float* S, const StepArgs& a, const DevParams& P, const RngKey& key) {
  reset_lane(S, P, key);
  count_sanitised(a);
}
// ---- match scoreboard (vss_match_board): adds of the fields during a step, frozen by the end of the step ----
VSS_HD bool board_frozen(const StepArgs& a) {
#if defined(__CUDA_ARCH__)
  return __ldcg(&a.board->frozen) != 0u;  // set by the last CTA of an earlier launch: read at L2
#else
  return a.board->frozen != 0u;
#endif
}
VSS_HD void board_add(const StepArgs& a, float score, int progress) {
#if defined(__CUDA_ARCH__)
  atomicAdd(reinterpret_cast<unsigned long long*>(&a.board->matches), 1ull);
  atomicAdd(reinterpret_cast<unsigned long long*>(&a.board->length_sum), (unsigned long long)progress);
  atomicAdd(&a.board->score_sum, (double)score);
#else
#pragma omp atomic
  a.board->matches += 1;
#pragma omp atomic
  a.board->length_sum += progress;
#pragma omp atomic
  a.board->score_sum += (double)score;
#endif
}
// Called once per step after every field's adds: the step counts, and the board freezes once the count is reached
// (play.py:152: the loop stops after the step in which ep_count reaches n_matches, with all of that step's dones).
VSS_HD void board_close_step(volatile vss_match_board* b, long long n_matches) {
  if (b->frozen) return;
  b->steps = b->steps + 1;
  if (b->matches >= n_matches) b->frozen = 1u;
}

// Match mode: dones and the scoreboard (play.py:152-160). A field < count_envs whose episode ended adds its
// rew[env,0,0,0] (the goal term of blue robot 0, as rewards_lane computes it) and its un-reset progress.
VSS_HD int match_outputs(const float* S, long long env, const StepArgs& a, const DevParams& P, bool finite,
                         int progress) {
  const bool goal = is_goal(S[0], S[LDS], P);
  const bool done = !finite || goal || progress >= P.max_len;
  a.reset_buf[env] = done ? 1 : 0;
  if (done && env < a.count_envs && !board_frozen(a)) {
    float score = 0.0f;
    if (finite && P.w_goal > 0.0f) {
      float gv = 0.0f;
      if (goal && S[0] > 0.0f) gv = 1.0f;
      if (goal && S[0] < 0.0f) gv = -1.0f;
      score = fmul(gv, P.w_goal);
    }
    board_add(a, score, progress);
  }
  return !done ? LANE_RUNNING : (finite ? LANE_DONE : LANE_SANITISED);
}

template <int VIEW>
VSS_HD int lane_outputs(float* S, long long env, const StepArgs& a, const DevParams& P, bool finite) {
  constexpr int AGENTS = ViewShape<VIEW>::AGENTS;
  const int progress = (int)fbits(S[VSS_W_PROGRESS * LDS]) + 1;
  S[VSS_W_PROGRESS * LDS] = bitsf((uint32_t)progress);
  if (VIEW == VIEW_MATCH) return match_outputs(S, env, a, P, finite, progress);
  float rew[VSS_REW_PER_FIELD];
  if (finite) {
    rewards_lane(S, P, rew);
  } else {
#pragma unroll
    for (int k = 0; k < VSS_REW_PER_FIELD; ++k) rew[k] = 0.0f;
  }
  const bool done = !finite || is_goal(S[0], S[LDS], P) || progress >= P.max_len;
  const bool tmo = done && finite && progress >= P.max_len - 1;  // VecTask.step timeout_buf
  a.reset_buf[env] = done ? 1 : 0;
  if (VIEW == VIEW_FULL) {
    float* rp = a.rew + env * VSS_REW_PER_FIELD;
#pragma unroll
    for (int q = 0; q < 6; ++q) st4(rp + 4 * q, F4{rew[4 * q], rew[4 * q + 1], rew[4 * q + 2], rew[4 * q + 3]});
    a.timeout[env] = tmo ? 1 : 0;
    if (a.progress_f) a.progress_f[env] = (float)progress;
  } else {
#pragma unroll
    for (int j = 0; j < AGENTS; ++j) {
      const long long v = env * AGENTS + j;
      float r4[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) {
        if (view_base(VIEW) == VSS_VIEW_CMA) r4[c] = fdiv(fadd(fadd(rew[c], rew[4 + c]), rew[8 + c]), 3.0f);  // .mean(1)
        else r4[c] = rew[4 * j + c];
      }
      st4(a.rew + 4 * v, F4{r4[0], r4[1], r4[2], r4[3]});
      a.reward_v[v] = fadd(fadd(fadd(r4[0], r4[1]), r4[2]), r4[3]);
      a.done_v[v] = done ? 1 : 0;
      a.timeout[v] = tmo ? 1 : 0;
      if (a.done_f) a.done_f[v] = done ? 1.0f : 0.0f;
      if (a.timeout_f) a.timeout_f[v] = tmo ? 1.0f : 0.0f;
      if (a.progress_f) a.progress_f[v] = (float)progress;
      if (a.packed) {  // bytes 104..111 of the agent's packed row
        uint32_t* tail = reinterpret_cast<uint32_t*>(static_cast<char*>(a.packed) + v * VSS_PACKED_ROW_BYTES + 104);
        tail[0] = fbits(fadd(fadd(fadd(r4[0], r4[1]), r4[2]), r4[3]));
        tail[1] = (done ? 1u : 0u) | (tmo ? 0x100u : 0u);
      }
      if (a.ep_ret) {  // RecordEpisodeStatisticsTorch.step, wrappers.py:68-75
        const float keep = done ? 0.0f : 1.0f;
        F4 er = ld4(a.ep_ret + 4 * v);
        er = F4{fadd(er.x, r4[0]), fadd(er.y, r4[1]), fadd(er.z, r4[2]), fadd(er.w, r4[3])};
        st4(a.ret_ret + 4 * v, er);
        st4(a.ep_ret + 4 * v, F4{fmul(er.x, keep), fmul(er.y, keep), fmul(er.z, keep), fmul(er.w, keep)});
        const int el = a.ep_len[v] + 1;
        a.ret_len[v] = el;
        a.ep_len[v] = done ? 0 : el;
      }
    }
  }
  return !done ? LANE_RUNNING : (finite ? LANE_DONE : LANE_SANITISED);
}
template <int VIEW>
VSS_HD int lane_phase1d(float* S, long long env, const StepArgs& a, const DevParams& P, const RngKey& key) {
  const bool finite = state_finite(S);
  if (!finite) lane_sanitise(S, a, P, key);
  return lane_outputs<VIEW>(S, env, a, P, finite);
}

// Phase 5: state out (+ zero the view's action buffer row of a done field, wrappers.py:105-107)
VSS_HD void zero_action_row(long long env, const StepArgs& a) {
  float* ap = a.action_buf + env * VSS_ACT_PER_FIELD;
#pragma unroll
  for (int q = 0; q < 3; ++q) {
    const F4 v = ld4(ap + 4 * q);  // `*= 0` keeps the sign of zero
    st4(ap + 4 * q, F4{fmul(v.x, 0.0f), fmul(v.y, 0.0f), fmul(v.z, 0.0f), fmul(v.w, 0.0f)});
  }
}
template <int VIEW>
VSS_HD void lane_phase5(const float* S, long long env, const StepArgs& a, bool done) {
  store_state(S, a.state, a.ld, env);
  if (VIEW != VIEW_FULL && VIEW != VIEW_MATCH && done) zero_action_row(env, a);
}

// Cooperative, coalesced observation write of one tile (all 32 lanes call it).
//   per_field = float4 per field in this layout (78 full, 13 sa/cma, 39 dma)
//   skip_mask = fields whose `ob` row is NOT written now (they are reset first)
// Element offset, in a (rows, 64) bf16 matrix, of float4 slot f of a (rows, 52) f32 matrix.
VSS_HD int bf16_pad_offset(int f) { const int row = f / F4_PER_ROW; return row * 64 + (f - row * F4_PER_ROW) * 4; }
// The same for the packed rows of vss_set_step_packed (112 bytes = 56 bf16 elements per row).
constexpr int PACKED_ROW_ELEMS = VSS_PACKED_ROW_BYTES / 2;
VSS_HD int packed_offset(int f) { const int row = f / F4_PER_ROW; return row * PACKED_ROW_ELEMS + (f - row * F4_PER_ROW) * 4; }

// (part, parts): this caller is warp `part` of `parts` warps that share the tile (k_step_cta); 0, 1 = alone.
VSS_HD void write_obs_tile(const float* T, const uint32_t* tab, int lane, int valid, int per_field, float* tob,
                           float* ob, uint32_t skip_mask, void* obh = nullptr, void* pk = nullptr, int part = 0,
                           int parts = 1) {
  const int total = valid * per_field;
#pragma unroll 4
  for (int f = lane + 32 * part; f < total; f += 32 * parts) {
    const int e = f / per_field, j = f - e * per_field;
    const F4 v = obs_gather(T, tab[j], e);
    if (tob) st4(tob + 4 * f, v);
    if (!((skip_mask >> e) & 1u)) {
      st4(ob + 4 * f, v);
      if (obh) st_bf16x4(obh, bf16_pad_offset(f), v);
      if (pk) st_bf16x4(pk, packed_offset(f), v);
    }
  }
}

// Same result as write_obs_tile for layouts with at least 32 float4 per field (full contract: 78,
// dma: 39), organised the other way round: lane l owns the float4 slots j = l, l+32 of EVERY
// field, so its gather offsets and sign masks are loop-invariant registers and the loop over the
// fields of the tile needs no index arithmetic or table look-ups (3x fewer instructions; the
// observation write is the largest single consumer of issue slots in the step kernel). Each
// warp-wide store of a full slot covers 512 contiguous bytes. The slots left over after the full
// ones (78 = 2 x 32 + 14, 39 = 32 + 7) are packed G fields to a store instruction: lane group g
// (16 or 8 lanes wide) writes the tail of field e + g.
template <int PER_FIELD, bool MULTI = false>
VSS_HD void write_obs_tile_rows(const float* T, const uint32_t* tab, int lane, int valid, float* tob, float* ob,
                                uint32_t skip_mask, void* obh = nullptr, void* pk = nullptr, int part = 0,
                                int parts = 1) {
  constexpr int FULL = PER_FIELD / 32, TAIL = PER_FIELD - 32 * FULL;
  constexpr int TW = TAIL <= 1 ? 1 : TAIL <= 2 ? 2 : TAIL <= 4 ? 4 : TAIL <= 8 ? 8 : TAIL <= 16 ? 16 : 32;
  constexpr int G = 32 / TW, SLOTS = FULL + (TAIL ? 1 : 0);
  int off[SLOTS][4];
  uint32_t sgn[SLOTS][4];
  const int sub = lane / TW, jt = 32 * FULL + (lane % TW);
  const bool tail_lane = TAIL && (lane % TW) < TAIL;
#pragma unroll
  for (int sl = 0; sl < SLOTS; ++sl) {
    const int j = sl < FULL ? lane + 32 * sl : jt;
    const uint32_t entry = j < PER_FIELD ? tab[j] : 0u;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const uint32_t by = (entry >> (8 * c)) & 0xFFu;
      off[sl][c] = (int)(by & 0x7Fu) * LDS + (sl < FULL ? 0 : sub);
      sgn[sl][c] = (by >> 7) << 31;
    }
  }
  // MULTI (k_step_cta: `parts` warps share the tile): warp `part` takes the field groups part, part + parts,
  // ... of GRP consecutive fields, so that the packed tail slots of a group stay with one warp.
  constexpr int GRP = MULTI ? (TAIL ? G : 1) : 32;
  const int e_first = MULTI ? part * GRP : 0, e_jump = MULTI ? parts * GRP : 32;
#pragma unroll 1
  for (int e0 = e_first; e0 < valid; e0 += e_jump) {
    const int e1 = e0 + GRP < valid ? e0 + GRP : valid;
#pragma unroll(OBS_UNROLL)
    for (int e = e0; e < e1; ++e) {
      const bool keep = !((skip_mask >> e) & 1u);
#pragma unroll
      for (int sl = 0; sl < FULL; ++sl) {
        const F4 v{bitsf(fbits(T[off[sl][0] + e]) ^ sgn[sl][0]), bitsf(fbits(T[off[sl][1] + e]) ^ sgn[sl][1]),
                   bitsf(fbits(T[off[sl][2] + e]) ^ sgn[sl][2]), bitsf(fbits(T[off[sl][3] + e]) ^ sgn[sl][3])};
        const int idx = 4 * (e * PER_FIELD + lane + 32 * sl);
        if (tob) st4_stream(tob + idx, v);
        if (keep) {
          st4_stream(ob + idx, v);
          if (obh) st_bf16x4(obh, bf16_pad_offset(idx >> 2), v);
          if (pk) st_bf16x4(pk, packed_offset(idx >> 2), v);
        }
      }
      if (TAIL && (e % G) == 0 && tail_lane && e + sub < valid) {  // fields e .. e+G-1, one lane group each
        constexpr int sl = SLOTS - 1;
        const F4 v{bitsf(fbits(T[off[sl][0] + e]) ^ sgn[sl][0]), bitsf(fbits(T[off[sl][1] + e]) ^ sgn[sl][1]),
                   bitsf(fbits(T[off[sl][2] + e]) ^ sgn[sl][2]), bitsf(fbits(T[off[sl][3] + e]) ^ sgn[sl][3])};
        const int idx = 4 * ((e + sub) * PER_FIELD + jt);
        if (tob) st4_stream(tob + idx, v);
        if (!((skip_mask >> (e + sub)) & 1u)) {
          st4_stream(ob + idx, v);
          if (obh) st_bf16x4(obh, bf16_pad_offset(idx >> 2), v);
          if (pk) st_bf16x4(pk, packed_offset(idx >> 2), v);
        }
      }
    }
  }
}

VSS_HD void write_obs_fields(const float* T, const uint32_t* tab, int lane, int per_field, float* ob,
                             uint32_t field_mask, void* obh = nullptr, void* pk = nullptr, int part = 0, int parts = 1) {
  int k = 0;
  while (field_mask) {
    const int e = ffs32(field_mask) - 1;
    field_mask &= field_mask - 1;
    if ((k++) % parts != part) continue;  // the k-th flagged field goes to warp k mod parts
    for (int j = lane; j < per_field; j += 32) {
      const F4 v = obs_gather(T, tab[j], e);
      st4(ob + 4 * (e * per_field + j), v);
      if (obh) st_bf16x4(obh, bf16_pad_offset(e * per_field + j), v);
      if (pk) st_bf16x4(pk, packed_offset(e * per_field + j), v);
    }
  }
}

// A policy team's bf16 row of the observation of its robot i in field env (SA / CMA: robot 0 -> row env; DMA: robot
// i -> row 3 env + i), or -1 for none.
VSS_HD long long team_row(int mode, long long env, int i) {
  if (mode == VSS_TEAM_DMA) return 3 * env + i;
  return i == 0 && (mode == VSS_TEAM_SA || mode == VSS_TEAM_CMA) ? env : -1;
}

// Match mode: the post-reset observation of the tile's fields (cooperative, all 32 lanes of `parts` warps): the f32
// (N,2,3,52) obs when a.obs is set, and each policy team's bf16 rows (the yellow rows are the mirrored obs[:,1]
// rows). Slots that go nowhere are not gathered.
VSS_HD void write_match_tile(const float* T, const uint32_t* tab, int lane, int valid, long long env0, const StepArgs& a,
                             int part = 0, int parts = 1) {
  const int total = valid * F4_PER_FIELD;
  for (int f = lane + 32 * part; f < total; f += 32 * parts) {
    const int e = f / F4_PER_FIELD, j = f - e * F4_PER_FIELD;
    const int row = j / F4_PER_ROW, t = row / 3, i = row - 3 * t;
    void* rows = a.team_rows[t];
    const long long r = rows ? team_row(a.team_mode[t], env0 + e, i) : -1;  // the team's bf16 row of this slot
    if (!a.obs && r < 0) continue;
    const F4 v = obs_gather(T, tab[j], e);
    if (a.obs) st4(a.obs + 4 * (env0 * F4_PER_FIELD + f), v);
    if (r >= 0) st_bf16x4(rows, r * 64 + (j - row * F4_PER_ROW) * 4, v);
  }
}

// Opponent view: the yellow team's post-reset observation of the tile's fields (cooperative, all 32 lanes of `parts`
// warps), gathered through obs-table entries 39..77 (the mirrored obs[:,1] rows): the f32 (N,3,52) rows when
// a.opp_obs is set, and the policy opponent's bf16 rows. Only robot 0 is gathered when nothing else goes anywhere.
VSS_HD void write_opp_tile(const float* T, const uint32_t* tab, int lane, int valid, long long env0, const StepArgs& a,
                           int part = 0, int parts = 1) {
  const int m = a.team_mode[1];
  void* rows = (m == VSS_TEAM_SA || m == VSS_TEAM_CMA || m == VSS_TEAM_DMA) ? a.team_rows[1] : nullptr;
  if (!rows && !a.opp_obs) return;
  constexpr int TEAM = 3 * F4_PER_ROW;
  const int per = (a.opp_obs || m == VSS_TEAM_DMA) ? TEAM : F4_PER_ROW;
  const int total = valid * per;
  for (int f = lane + 32 * part; f < total; f += 32 * parts) {
    const int e = f / per, j = f - e * per, i = j / F4_PER_ROW;
    const F4 v = obs_gather(T, tab[TEAM + j], e);
    if (a.opp_obs) st4(a.opp_obs + 4 * ((env0 + e) * TEAM + j), v);
    const long long r = team_row(m, env0 + e, i);
    if (rows && r >= 0) st_bf16x4(rows, r * 64 + (j - i * F4_PER_ROW) * 4, v);
  }
}

}  // namespace vss
