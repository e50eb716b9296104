"""numpy float32 restatement of the field picture — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The definition is DESIGN.md §4.7 (csrc/vss_render.cuh is the product's source). Every array operation
below is one float32 operation with one rounding, in the order vss_render.cuh performs it, so the
restatement, the host emulator and the kernel agree byte for byte.
"""
import numpy as np

F32 = np.float32
MARGIN, CARPET = (32, 32, 32), (20, 90, 40)
GOAL_LEFT, GOAL_RIGHT = (60, 60, 140), (140, 130, 40)
LINE, BALL, BODY = (230, 230, 230), (255, 140, 0), (16, 16, 16)
BLUE, YELLOW = (30, 90, 255), (255, 220, 0)
ID_COLOURS = ((230, 40, 40), (40, 200, 60), (200, 60, 220))


def _get(params, k):
    return F32(params[k] if isinstance(params, dict) else getattr(params, k))


def frame_constants(params, height, width):
    """The per-frame constants of render_frame(), in its operation order."""
    g = {}
    g["L"], g["Wf"], g["G"] = _get(params, "field_half_length"), _get(params, "field_half_width"), _get(params, "goal_half_width")
    g["LD"] = F32(g["L"] + _get(params, "goal_depth"))
    g["X"] = F32(g["LD"] + F32(0.05))
    g["Y"] = F32(g["Wf"] + F32(0.05))
    g["px"] = F32(F32(F32(2.0) * g["X"]) / F32(width))
    g["py"] = F32(F32(F32(2.0) * g["Y"]) / F32(height))
    g["t"] = F32(0.005)
    t2 = F32(F32(2.0) * g["t"])
    g["line_x"], g["line_y"] = F32(g["L"] - t2), F32(g["Wf"] - t2)
    lo, hi = F32(F32(0.2) - g["t"]), F32(F32(0.2) + g["t"])
    g["ring_lo2"], g["ring_hi2"] = F32(lo * lo), F32(hi * hi)
    rb = _get(params, "ball_radius")
    g["rb2"] = F32(rb * rb)
    g["h"] = _get(params, "robot_half_size")
    g["p"] = F32(F32(0.8) * g["h"])
    return g


def pixel_centres(g, height, width):
    """(x, y) of every pixel centre: float32 arrays of shape (H, W)."""
    j = np.arange(width, dtype=F32)
    i = np.arange(height, dtype=F32)
    x = ((j + F32(0.5)) * g["px"]) - g["X"]
    y = g["Y"] - ((i + F32(0.5)) * g["py"])
    return np.broadcast_to(x[None, :], (height, width)), np.broadcast_to(y[:, None], (height, width))


def render_field(g, words, x, y):
    """One frame (H, W, 3) uint8. words: the field's 58 state words (include/vss_b200.h layout)."""
    w = np.asarray(words, F32)
    out = np.empty(x.shape + (3,), np.uint8)
    out[...] = MARGIN
    with np.errstate(invalid="ignore", over="ignore"):
        ax, ay = np.abs(x), np.abs(y)
        carpet = (ax <= g["L"]) & (ay <= g["Wf"])
        out[carpet] = CARPET
        goal = ~carpet & (ax > g["L"]) & (ax <= g["LD"]) & (ay < g["G"])
        out[goal & (x < 0)] = GOAL_LEFT
        out[goal & ~(x < 0)] = GOAL_RIGHT
        r2 = (x * x) + (y * y)
        line = carpet & ((ax > g["line_x"]) | (ay > g["line_y"]) | (ax <= g["t"]) |
                         ((r2 >= g["ring_lo2"]) & (r2 <= g["ring_hi2"])))
        out[line] = LINE
        dx, dy = x - w[0], y - w[1]
        out[((dx * dx) + (dy * dy)) <= g["rb2"]] = BALL
        for r in range(6):
            b = 4 + 9 * r
            rx, ry, c, s = w[b], w[b + 1], w[b + 4], w[b + 5]
            dx, dy = x - rx, y - ry
            u = (dx * c) + (dy * s)
            v = (dy * c) - (dx * s)
            au, av = np.abs(u), np.abs(v)
            out[(au <= g["h"]) & (av <= g["h"])] = BODY
            patch = (au <= g["p"]) & (av <= g["p"])
            out[patch & (u < 0)] = BLUE if r < 3 else YELLOW
            out[patch & ~(u < 0)] = ID_COLOURS[r % 3]
    return out


def render(params, soa, first_field, num_fields, height=560, width=720):
    """Frames (num_fields, H, W, 3) uint8 of fields [first_field, first_field + num_fields) of a SoA state
    (STATE_WORDS x ld float32, word w of field e at soa[w, e])."""
    soa = np.asarray(soa, F32)
    g = frame_constants(params, height, width)
    x, y = pixel_centres(g, height, width)
    return np.stack([render_field(g, soa[:58, e], x, y) for e in range(first_field, first_field + num_fields)])


def pixel_of(params, height, width, px_x, px_y):
    """The (row, column) whose pixel contains the point (px_x, px_y) in metres (for hand-checked tests)."""
    g = frame_constants(params, height, width)
    return int((g["Y"] - px_y) / g["py"]), int((px_x + g["X"]) / g["px"])
