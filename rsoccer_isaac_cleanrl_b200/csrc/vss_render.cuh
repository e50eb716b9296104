// vss_render.cuh — the picture of one field: an exact, per-pixel definition of the RGB frame that
// vss_render (csrc/vss_step.cu) writes, compiled by the kernel and by the host emulator of the tests
// (tests/emu/vss_render_emu.cpp), like vss_lane.cuh.
//
// Every float operation is one f32 operation with one rounding (the non-contracting fadd / fsub / fmul /
// fdiv of vss_lane.cuh: no FMA, no fast-math), so a numpy float32 restatement that follows the same
// operation order (oracle/vss_render.py) agrees bit for bit. No anti-aliasing, no text: DESIGN.md §4.7.
//
// Window: X = (L + D) + 0.05, Y = Wf + 0.05; pixel (i, j) has its centre at x = (j + 0.5) px - X,
// y = Y - (i + 0.5) py with px = 2X / width, py = 2Y / height (row 0 at the top, +x right, +y up).
// Painter's order: margin, carpet, goal interiors, lines (carpet only), ball, robots 0..5 (body, then the
// 0.8-size patch: team colour behind the centre, ID colour in front of it, so the patch shows the heading).
#pragma once
#include "vss_lane.cuh"

namespace vss {

// state words a frame reads: ball x, y, then x, y, cos(yaw), sin(yaw) of robots 0..5 (4 + 9r + {0, 1, 4, 5})
constexpr int RENDER_WORDS = 2 + 4 * 6;
VSS_HD int render_word(int k) { return k < 2 ? k : 4 + 9 * ((k - 2) >> 2) + ((k - 2) & 3) + ((k - 2) & 2); }

// RGB colours, packed 0x00BBGGRR (byte 0 = red)
#define VSS_RGB(r, g, b) ((uint32_t)(r) | ((uint32_t)(g) << 8) | ((uint32_t)(b) << 16))
constexpr uint32_t RC_MARGIN = VSS_RGB(32, 32, 32);
constexpr uint32_t RC_CARPET = VSS_RGB(20, 90, 40);
constexpr uint32_t RC_GOAL_LEFT = VSS_RGB(60, 60, 140);    // x < 0: the goal blue defends
constexpr uint32_t RC_GOAL_RIGHT = VSS_RGB(140, 130, 40);  // x > 0: the goal yellow defends
constexpr uint32_t RC_LINE = VSS_RGB(230, 230, 230);
constexpr uint32_t RC_BALL = VSS_RGB(255, 140, 0);
constexpr uint32_t RC_BODY = VSS_RGB(16, 16, 16);
constexpr uint32_t RC_BLUE = VSS_RGB(30, 90, 255);
constexpr uint32_t RC_YELLOW = VSS_RGB(255, 220, 0);
VSS_HD uint32_t render_id_colour(int idx) {
  return idx == 0 ? VSS_RGB(230, 40, 40) : (idx == 1 ? VSS_RGB(40, 200, 60) : VSS_RGB(200, 60, 220));
}
#undef VSS_RGB

// Per-frame constants, derived from vss_params and the frame size in a fixed operation order.
struct RenderFrame {
  float X, Y, px, py;  // window half-extents, metres per pixel
  float L, Wf, G, LD;  // field half-length / half-width, goal half-width, L + goal depth
  float line_x, line_y, t, ring_lo2, ring_hi2;  // lines: L - 2t, Wf - 2t, t, (0.2 - t)^2, (0.2 + t)^2
  float rb2, h, p;  // ball radius^2, robot half-size, patch half-size 0.8 h
  float reach;      // 2.01 h: no pixel farther than this (in x or in y) from a robot's centre is drawn by it
};

VSS_HD RenderFrame render_frame(const vss_params& prm, int height, int width) {
  RenderFrame g;
  g.L = prm.field_half_length; g.Wf = prm.field_half_width; g.G = prm.goal_half_width;
  g.LD = fadd(g.L, prm.goal_depth);
  g.X = fadd(g.LD, 0.05f);
  g.Y = fadd(g.Wf, 0.05f);
  g.px = fdiv(fmul(2.0f, g.X), (float)width);
  g.py = fdiv(fmul(2.0f, g.Y), (float)height);
  g.t = 0.005f;
  const float t2 = fmul(2.0f, g.t);
  g.line_x = fsub(g.L, t2);
  g.line_y = fsub(g.Wf, t2);
  const float lo = fsub(0.2f, g.t), hi = fadd(0.2f, g.t);
  g.ring_lo2 = fmul(lo, lo);
  g.ring_hi2 = fmul(hi, hi);
  g.rb2 = fmul(prm.ball_radius, prm.ball_radius);
  g.h = prm.robot_half_size;
  g.p = fmul(0.8f, g.h);
  g.reach = fmul(2.01f, g.h);
  return g;
}

VSS_HD float render_x(const RenderFrame& g, int j) { return fsub(fmul(fadd((float)j, 0.5f), g.px), g.X); }
VSS_HD float render_y(const RenderFrame& g, int i) { return fsub(g.Y, fmul(fadd((float)i, 0.5f), g.py)); }

// The colour of pixel (i, j); f = the RENDER_WORDS state words of the field (render_word order). A non-finite
// coordinate fails every comparison and draws nothing. Robots whose bit in `live` is clear are skipped: the caller
// clears it only for a robot that cannot draw this pixel (render_segment), so the colour does not depend on it.
VSS_HD uint32_t render_pixel(const RenderFrame& g, const float* f, int i, int j, uint32_t live = 0x3Fu) {
  const float x = render_x(g, j);
  const float y = render_y(g, i);
  const float ax = fabsf(x), ay = fabsf(y);
  uint32_t c = RC_MARGIN;
  if (ax <= g.L && ay <= g.Wf) {
    c = RC_CARPET;
    const float r2 = fadd(fmul(x, x), fmul(y, y));
    if (ax > g.line_x || ay > g.line_y || ax <= g.t || (r2 >= g.ring_lo2 && r2 <= g.ring_hi2)) c = RC_LINE;
  } else if (ax > g.L && ax <= g.LD && ay < g.G) {
    c = x < 0.0f ? RC_GOAL_LEFT : RC_GOAL_RIGHT;
  }
  {
    const float dx = fsub(x, f[0]), dy = fsub(y, f[1]);
    if (fadd(fmul(dx, dx), fmul(dy, dy)) <= g.rb2) c = RC_BALL;
  }
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    if (!((live >> r) & 1u)) continue;
    const float* q = f + 2 + 4 * r;  // x, y, cos, sin
    const float dx = fsub(x, q[0]), dy = fsub(y, q[1]);
    const float u = fadd(fmul(dx, q[2]), fmul(dy, q[3]));
    const float v = fsub(fmul(dy, q[2]), fmul(dx, q[3]));
    const float au = fabsf(u), av = fabsf(v);
    if (au <= g.h && av <= g.h) c = RC_BODY;
    if (au <= g.p && av <= g.p) c = u < 0.0f ? (r < 3 ? RC_BLUE : RC_YELLOW) : render_id_colour(r % 3);
  }
  return c;
}

// Robots that may draw a pixel of the segment (i, j0 .. j0 + 15): a culling test that never changes a colour.
// With q = c^2 + s^2, u^2 + v^2 = q (dx^2 + dy^2), so a drawn pixel (|u|, |v| <= h) has dx^2 + dy^2 <= 2 h^2 / q; for
// 0.5 <= q <= 2 (any unit (cos, sin) pair; otherwise nothing is culled) and the f32 rounding of u and v that bounds
// |dx| and |dy| by 2.0001 h < reach. dx = x - rx is non-decreasing in j (every operation of render_x and the
// subtraction are monotone), so its values at the segment's two ends bound it for all 16 pixels; dy is the row's.
VSS_HD uint32_t render_live_robots(const RenderFrame& g, const float* f, int i, int j0) {
  const float y = render_y(g, i), xa = render_x(g, j0), xb = render_x(g, j0 + 15);
  uint32_t live = 0u;
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    const float* q = f + 2 + 4 * r;
    const float qq = fadd(fmul(q[2], q[2]), fmul(q[3], q[3]));
    const float dy = fsub(y, q[1]), dxa = fsub(xa, q[0]), dxb = fsub(xb, q[0]);
    const bool far = qq >= 0.5f && qq <= 2.0f && (fabsf(dy) > g.reach || dxa > g.reach || dxb < -g.reach);
    live |= (far ? 0u : 1u) << r;
  }
  return live;
}

// 16 consecutive pixels (i, j0 .. j0 + 15) as 48 RGB bytes in 12 little-endian words (what one thread of
// the kernel stores with three 16-byte stores).
VSS_HD void render_segment(const RenderFrame& g, const float* f, int i, int j0, uint32_t w[12]) {
  const uint32_t live = render_live_robots(g, f, i, j0);
#pragma unroll
  for (int k = 0; k < 12; ++k) w[k] = 0u;
#pragma unroll
  for (int q = 0; q < 16; ++q) {
    const uint32_t c = render_pixel(g, f, i, j0 + q, live);
#pragma unroll
    for (int ch = 0; ch < 3; ++ch) {
      const int b = 3 * q + ch;
      w[b >> 2] |= ((c >> (8 * ch)) & 255u) << (8 * (b & 3));
    }
  }
}

}  // namespace vss
