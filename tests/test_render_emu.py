"""CPU: the field picture (DESIGN.md §4.7). The numpy restatement is pinned by hand-checkable facts, the host
build of the product's per-pixel code (csrc/vss_render.cuh) equals it byte for byte, vss_render rejects bad
arguments without a device, and the video helpers lay out and write frames."""
import ctypes as C
import math

import numpy as np
import pytest

import render_checks as rc
from oracle import vss_oracle as orc
from oracle import vss_render as vr

H, W = 560, 720


def _empty(ld=32):
    """A field with the ball and every robot far outside the window: nothing but the field is drawn."""
    s = np.zeros((60, ld), np.float32)
    s[0:2] = 10.0
    for r in range(6):
        b = 4 + 9 * r
        s[b], s[b + 1], s[b + 4] = 10.0 + r, 10.0, 1.0
    return s


def _at(img, x, y, p=None):
    i, j = vr.pixel_of(p or orc.default_params(), img.shape[0], img.shape[1], x, y)
    return tuple(int(c) for c in img[i, j])


def _one(s, p=None, h=H, w=W):
    return vr.render(p or orc.default_params(), s, 0, 1, h, w)[0]


def test_window_is_400_px_per_metre():
    g = vr.frame_constants(orc.default_params(), H, W)
    assert g["px"] == pytest.approx(1 / 400, rel=1e-6) and g["py"] == pytest.approx(1 / 400, rel=1e-6)
    assert g["X"] == pytest.approx(0.9, rel=1e-6) and g["Y"] == pytest.approx(0.7, rel=1e-6)


def test_empty_field_margin_carpet_goals_lines():
    img = _one(_empty())
    assert tuple(img[0, 0]) == vr.MARGIN and tuple(img[-1, -1]) == vr.MARGIN
    assert _at(img, 0.4, 0.3) == vr.CARPET and _at(img, -0.5, -0.45) == vr.CARPET
    assert _at(img, -0.8, 0.05) == vr.GOAL_LEFT    # blue defends the left goal (blue attacks +x)
    assert _at(img, 0.8, -0.05) == vr.GOAL_RIGHT
    assert _at(img, -0.8, 0.3) == vr.MARGIN        # beside the goal, behind the end line
    assert _at(img, 0.001, 0.4) == vr.LINE         # half-way line
    assert _at(img, 0.745, 0.3) == vr.LINE and _at(img, -0.3, -0.646) == vr.LINE  # border lines
    assert _at(img, 0.2, 0.0) == vr.LINE and _at(img, 0.0, -0.2) == vr.LINE      # centre circle
    assert _at(img, 0.1, 0.05) == vr.CARPET and _at(img, 0.25, 0.1) == vr.CARPET  # inside / outside the circle
    # the picture is symmetric in y (x is not: the goal tints differ)
    assert np.array_equal(img, img[::-1])


def test_ball_centre_pixel_is_orange_and_one_and_a_half_radii_away_is_not():
    p = orc.default_params()
    s = _empty()
    s[0, 0], s[1, 0] = 0.3, 0.2
    img = _one(s)
    assert _at(img, 0.3, 0.2) == vr.BALL
    assert _at(img, 0.3 + 1.5 * p.ball_radius, 0.2) == vr.CARPET
    assert _at(img, 0.3, 0.2 - 1.5 * p.ball_radius) == vr.CARPET


@pytest.mark.parametrize("yaw, front", [(0.0, (1, 0)), (math.pi / 2, (0, 1)), (math.pi, (-1, 0))])
def test_robot_patch_shows_the_heading(yaw, front):
    p = orc.default_params()
    h = p.robot_half_size
    for r in (0, 4):  # a blue robot (ID 0) and a yellow one (ID 1)
        s = _empty()
        rx, ry = -0.3, -0.2
        b = 4 + 9 * r
        s[b, 0], s[b + 1, 0], s[b + 4, 0], s[b + 5, 0] = rx, ry, np.cos(yaw), np.sin(yaw)
        img = _one(s)
        d = 0.5 * 0.8 * h
        assert _at(img, rx + d * front[0], ry + d * front[1]) == vr.ID_COLOURS[r % 3]
        assert _at(img, rx - d * front[0], ry - d * front[1]) == (vr.BLUE if r < 3 else vr.YELLOW)
        assert _at(img, rx + 0.9 * h * front[0], ry + 0.9 * h * front[1]) == vr.BODY
        assert _at(img, rx + 1.2 * h * front[0], ry + 1.2 * h * front[1]) == vr.CARPET


def test_robot_drawn_over_the_ball_covers_it():
    s = _empty()
    s[0, 0], s[1, 0] = 0.3, 0.2
    s[4, 0], s[5, 0], s[8, 0], s[9, 0] = 0.3, 0.2, 1.0, 0.0
    img = _one(s)
    assert _at(img, 0.3, 0.2) != vr.BALL
    assert not (img == np.array(vr.BALL, np.uint8)).all(-1).any()


def test_non_finite_coordinates_draw_nothing():
    s = _empty()
    s[0, 0] = np.nan
    s[4, 0], s[5, 0] = np.inf, 0.0
    s[13, 0], s[14, 0], s[17, 0] = 0.1, 0.1, np.nan
    assert np.array_equal(_one(s), _one(_empty()))


@pytest.mark.parametrize("h, w", rc.SIZES)
def test_emulator_equals_restatement_on_random_states(h, w):
    p = orc.default_params()
    n = 80 if (h, w) == (560, 720) else 120
    s = rc.random_states(n, seed=h * 7 + w)
    assert np.array_equal(rc.emu_render(p, s, 0, n, h, w), vr.render(p, s, 0, n, h, w))


def test_emulator_equals_restatement_on_oracle_rollouts():
    p = orc.default_params()
    for k, s in enumerate(rc.oracle_rollout_states(16, 30, seed=5)[::6]):
        h, w = rc.SIZES[k % 3]
        assert np.array_equal(rc.emu_render(p, s, 3, 13, h, w), vr.render(p, s, 3, 13, h, w)), k


def test_emulator_equals_restatement_with_other_geometry():
    p = orc.default_params()
    p.field_half_length, p.field_half_width, p.goal_half_width, p.goal_depth = 1.1, 0.9, 0.35, 0.18
    p.ball_radius, p.robot_half_size = 0.03, 0.05
    s = rc.random_states(24, seed=3, spread=1.4)
    assert np.array_equal(rc.emu_render(p, s, 0, 24, 128, 64), vr.render(p, s, 0, 24, 128, 64))


def test_vss_render_validates_without_a_device():
    from rsoccer_isaac_cleanrl_b200 import _lib
    lib = _lib.load_library()
    buf = (C.c_uint8 * 64)()
    p = C.addressof(buf) + (-C.addressof(buf)) % 16
    assert lib.vss_render(None, 0, 1, 100, 720, p, None) == -1
    assert "height" in lib.vss_last_error().decode()
    assert lib.vss_render(None, 0, 1, 560, 100, p, None) == -1
    assert "width" in lib.vss_last_error().decode()
    assert lib.vss_render(None, 0, 1, 560, 4112, p, None) == -1
    assert lib.vss_render(None, 0, 1, 48, 720, p, None) == -1
    assert lib.vss_render(None, 0, 1, 560, 720, None, None) == -1
    assert "rgb" in lib.vss_last_error().decode()
    assert lib.vss_render(None, 0, 1, 560, 720, p + 8, None) == -1
    assert "aligned" in lib.vss_last_error().decode()
    assert lib.vss_render(None, 0, 1, 560, 720, p, None) == -1
    assert "handle" in lib.vss_last_error().decode()


def test_mosaic_layout():
    torch = pytest.importorskip("torch")
    from rsoccer_isaac_cleanrl_b200.video import mosaic
    for f in (1, 2, 4, 5, 7, 9, 10):
        fr = torch.randint(1, 256, (f, 16, 24, 3), dtype=torch.uint8)
        m = mosaic(fr)
        cols = math.ceil(math.sqrt(f))
        rows = math.ceil(f / cols)
        assert m.shape == (rows * 16, cols * 24, 3)
        for k in range(rows * cols):
            tile = m[(k // cols) * 16:(k // cols + 1) * 16, (k % cols) * 24:(k % cols + 1) * 24]
            assert torch.equal(tile, fr[k]) if k < f else not tile.any()


def test_video_writer_round_trip(tmp_path):
    cv2 = pytest.importorskip("cv2")
    from rsoccer_isaac_cleanrl_b200.video import FPS, VideoWriter
    p = orc.default_params()
    frames = vr.render(p, rc.random_states(3, seed=1), 0, 3, 64, 80)
    path = str(tmp_path / "sub" / "v.mp4")
    with VideoWriter(path) as w:
        w.write_frames(frames[:, None])   # (K, 1, H, W, 3): one field per frame
        w.write_frames(frames)            # (K, H, W, 3)
    assert w.frames == 6
    path4 = str(tmp_path / "four.mp4")
    with VideoWriter(path4) as w4:
        w4.write_frames(np.repeat(frames[:, None], 4, axis=1))  # four fields per frame: a 2 x 2 mosaic
    for pth, n_want, shape in ((path, 6, (64, 80, 3)), (path4, 3, (128, 160, 3))):
        cap = cv2.VideoCapture(pth)
        assert cap.get(cv2.CAP_PROP_FPS) == pytest.approx(FPS)
        n = 0
        while True:
            ok, img = cap.read()
            if not ok:
                break
            assert img.shape == shape
            n += 1
        cap.release()
        assert n == n_want


def test_video_writer_rejects_a_size_change(tmp_path):
    pytest.importorskip("cv2")
    from rsoccer_isaac_cleanrl_b200.video import VideoWriter
    with VideoWriter(str(tmp_path / "v.mp4")) as w:
        w.write(np.zeros((64, 80, 3), np.uint8))
        with pytest.raises(ValueError):
            w.write(np.zeros((64, 96, 3), np.uint8))


def test_safe_name():
    from rsoccer_isaac_cleanrl_b200.video import safe_name
    assert safe_name("ppo-sa:runs/x y/agent.pt") == "ppo-sa_runs_x_y_agent.pt"
    assert safe_name("ou") == "ou"


def test_robot_culling_never_changes_a_pixel():
    """Robots placed where the per-segment culling of vss_render.cuh decides: centres around the edges of 16-pixel
    segments at the largest extent (yaw 45 degrees), and (cos, sin) pairs that are not unit vectors (culled only
    for 0.5 <= c^2 + s^2 <= 2). The host build of the product equals the restatement, which does not cull."""
    p = orc.default_params()
    rng = np.random.default_rng(11)
    n = 96
    s = _empty(ld=n)
    for h, w in ((560, 720), (128, 64)):
        g = vr.frame_constants(p, h, w)
        for r in range(6):
            b = 4 + 9 * r
            j0 = 16 * rng.integers(1, w // 16 - 1, n)
            edge = (j0 - 0.5 * (1 + np.sign(rng.uniform(-1, 1, n))) * 1.0) * g["px"] - g["X"]
            s[b] = edge + rng.choice([-1, 1], n) * p.robot_half_size * rng.uniform(1.38, 2.05, n)
            s[b + 1] = rng.uniform(-0.6, 0.6, n)
            a = np.where(rng.uniform(size=n) < 0.5, np.pi / 4, rng.uniform(-np.pi, np.pi, n))
            scale = rng.choice([1.0, 1.0, 0.0, 0.3, 0.69, 0.72, 1.4, 1.43, 3.0], n)
            s[b + 4], s[b + 5] = scale * np.cos(a), scale * np.sin(a)
        assert np.array_equal(rc.emu_render(p, s, 0, n, h, w), vr.render(p, s, 0, n, h, w)), (h, w)
