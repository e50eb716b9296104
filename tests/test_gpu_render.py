"""B200: vss_render (the field picture, DESIGN.md §4.7) byte for byte against the numpy restatement, its
argument checks on a live handle, graph capture, and the videos of VSS.render, play_matches(_fused) and
ppo.train(--capture-video)."""
import os

import numpy as np
import pytest

import render_checks as rc
from backends import GpuBackend
from oracle import vss_render as vr

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _restated(eng, first, num, h, w):
    return vr.render(eng.params, eng.get_state().cpu().numpy(), first, num, h, w)


def _assert_frames(eng, first, num, h, w):
    got = eng.render(first, num, h, w)
    torch.cuda.synchronize()
    want = _restated(eng, first, num, h, w)
    diff = got.cpu().numpy() != want
    assert not diff.any(), (first, num, h, w, int(diff.any(-1).sum()), np.argwhere(diff.any(-1))[:5])


def _vss(n, seed):
    from rsoccer_isaac_cleanrl_b200.envs import VSS, load_cfg
    cfg = load_cfg()
    cfg["env"]["numEnvs"] = n
    envs = VSS(cfg, "cuda:0", "cuda:0", 0, True, seed=seed)
    envs.w_goal, envs.w_grad, envs.w_move, envs.w_energy = 1.0, 0.0, 0.0, 0.0
    return envs


# ------------------------------------------------------------------ the kernel against the restatement
@pytest.mark.parametrize("h, w", rc.SIZES + ((1024, 1280),))
def test_render_set_states(h, w):
    n = 200
    be = GpuBackend(n, seed=3)
    be.set_state(rc.random_states(n, seed=h + w, ld=be.ld))
    big = h * w > 1e6
    for first, num in (((0, 1), (5, 7), (n - 2, 2)) if big else ((0, 1), (3, 7), (0, 64), (n - 64, 64), (n - 7, 7))):
        _assert_frames(be.eng, first, num, h, w)
    be.eng.close()


@pytest.mark.parametrize("view", [-1, 0, 1, 2], ids=["full", "sa", "cma", "dma"])
def test_render_after_steps(view):
    """States after 50 steps of the full contract and of each view (goals, resets, collisions)."""
    n = 300
    be = GpuBackend(n, seed=11 + view)
    rng = np.random.default_rng(4)
    rb = np.ones(n, np.int64)
    be.reset_dones(rb)
    rb[:] = 0
    nv = 3 * n if view == 2 else n
    abuf = np.zeros((n, 2, 3, 2), np.float32)
    for _ in range(50):
        if view < 0:
            be.step(rng.uniform(-1, 1, (n, 2, 3, 2)).astype(np.float32), rb)
        else:
            be.step_view(view, rng.uniform(-1, 1, (nv, 6 if view == 1 else 2)).astype(np.float32), abuf, rb)
    for k, (first, num) in enumerate(((0, 1), (17, 7), (n - 64, 64))):
        _assert_frames(be.eng, first, num, *rc.SIZES[k])
    be.eng.close()


def test_render_changes_nothing():
    """The state words are bit-identical before and after a render, and a step after renders equals the same step of
    a twin engine that did not render (outputs and state)."""
    import rsoccer_isaac_cleanrl_b200 as R
    n = 1065
    outs = []
    for renders in (True, False):
        eng = R.Engine(n, "cuda:0", seed=8)
        z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device="cuda")
        rb = torch.ones(n, dtype=torch.int64, device="cuda")
        eng.reset_dones(rb, z(n, 2, 3, 52))
        gen = torch.Generator(device="cuda").manual_seed(2)
        bufs = [z(n, 2, 3, 52), z(n, 2, 3, 52), z(n, 2, 3, 4), z(n, dt=torch.uint8), z(n)]
        for t in range(6):
            if renders:
                before = eng.get_state().clone()
                eng.render(0, 64)
                eng.render(n - 100, 100, 64, 80)
                torch.cuda.synchronize()
                assert torch.equal(before.view(torch.int32), eng.get_state().view(torch.int32))
            eng.step(torch.rand((n, 2, 3, 2), device="cuda", generator=gen) * 2 - 1, rb, *bufs)
        torch.cuda.synchronize()
        outs.append([eng.get_state().view(torch.int32), rb.clone()] + [b.clone() for b in bufs] + [eng.step_count])
        eng.close()
    for a, b in zip(*outs):
        assert torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b


def test_render_validation_with_a_live_handle():
    import rsoccer_isaac_cleanrl_b200 as R
    from rsoccer_isaac_cleanrl_b200 import _lib
    lib = _lib.load_library()
    n = 100
    eng = R.Engine(n, "cuda:0", seed=1)
    buf = torch.zeros(4 * 560 * 720 * 3 + 16, dtype=torch.uint8, device="cuda")
    p = buf.data_ptr()
    s = torch.cuda.current_stream().cuda_stream
    cases = [((n - 3, 4, 560, 720, p), "outside"), ((0, 0, 560, 720, p), "num_fields"), ((-1, 1, 560, 720, p), "outside"),
             ((0, n + 1, 560, 720, p), "outside"), ((0, 1, 560, 720, None), "rgb"), ((0, 1, 560, 720, p + 4), "aligned"),
             ((0, 1, 568, 720, p), "height"), ((0, 1, 560, 4608, p), "width")]
    for args, word in cases:
        assert lib.vss_render(eng._h, *args, s) == -1, args
        assert word in lib.vss_last_error().decode(), (args, lib.vss_last_error())
    torch.cuda.synchronize()   # nothing was launched: no error is pending
    assert not buf.any()
    assert lib.vss_render(eng._h, n - 4, 4, 560, 720, p, s) == 0
    torch.cuda.synchronize()
    eng.close()


def test_render_in_a_cuda_graph():
    """Renders captured in a CUDA graph and replayed give the frames of eager renders of the same state."""
    be = GpuBackend(500, seed=2)
    be.set_state(rc.random_states(500, seed=9, ld=be.ld))
    eng = be.eng
    out = torch.zeros((3, 16, 560, 720, 3), dtype=torch.uint8, device="cuda")
    small = torch.zeros((5, 128, 64, 3), dtype=torch.uint8, device="cuda")

    def renders():
        eng.render(0, 16, out=out[0])
        eng.render(100, 16, out=out[1])
        eng.render(484, 16, out=out[2])
        eng.render(7, 5, 128, 64, out=small)
    renders()
    torch.cuda.synchronize()
    eager = out.clone(), small.clone()
    out.zero_(); small.zero_()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        renders()
    torch.cuda.synchronize()
    assert not out.any()
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(out, eager[0]) and torch.equal(small, eager[1])
    assert np.array_equal(eager[1].cpu().numpy(), _restated(eng, 7, 5, 128, 64))
    eng.close()


def test_vss_render_method():
    from rsoccer_isaac_cleanrl_b200.video import mosaic
    envs = _vss(64, seed=4)
    envs.step(torch.rand((64, 2, 3, 2), device="cuda") * 2 - 1)
    img = envs.render()
    assert img.dtype == np.uint8 and img.shape == (560, 720, 3)
    assert np.array_equal(img, _restated(envs.engine, 0, 1, 560, 720)[0])
    img5 = envs.render(fields=5, height=128, width=160)
    want = mosaic(torch.from_numpy(_restated(envs.engine, 0, 5, 128, 160))).numpy()
    assert img5.shape == (2 * 128, 3 * 160, 3) and np.array_equal(img5, want)
    with pytest.raises(NotImplementedError):
        envs.render(mode="human")
    envs.close()


# ------------------------------------------------------------------ match videos
@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory):
    """A (barely trained) ppo-sa checkpoint in the reference's state_dict format."""
    from rsoccer_isaac_cleanrl_b200 import ppo
    args = ppo.parse_args(["--env-id", "sa", "--num-envs", "128", "--num-steps", "8", "--total-timesteps",
                           str(128 * 8), "--quiet"])
    st = ppo.train(args)
    path = str(tmp_path_factory.mktemp("render") / "agent.pt")
    torch.save(st["agent"].state_dict(), path)
    return path


def _mp4_frames(path):
    import cv2
    cap = cv2.VideoCapture(path)
    n, shape = 0, None
    while True:
        ok, img = cap.read()
        if not ok:
            break
        shape = img.shape
        n += 1
    cap.release()
    return n, shape


def _external_ou():
    from rsoccer_isaac_cleanrl_b200 import play
    ou = play.TeamOU()
    return lambda act, obs: ou(act, obs)


@pytest.mark.parametrize("blue,yellow", [("zero", "ou"), ("ppo-sa", "ou"), ("external", "ou")])
def test_play_matches_fused_video(blue, yellow, checkpoint, tmp_path):
    from rsoccer_isaac_cleanrl_b200 import play
    fields = 1 if blue == "zero" else 4
    n_matches = 150 if blue == "external" else 400
    runs = []
    for video, graphs in ((False, True), (True, True), (True, False)):
        envs = _vss(1065, seed=17)
        team = _external_ou() if blue == "external" else play.get_team(blue, checkpoint if blue != "zero" else None)
        path = str(tmp_path / f"{blue}_{graphs}.mp4") if video else None
        torch.manual_seed(3)
        r = play._run_matches_fused(envs, team, play.get_team(yellow), n_matches, seed=6, graphs=graphs,
                                    video_path=path, video_fields=fields)
        torch.cuda.synchronize()
        r["state"] = envs.engine.get_state()
        if video:
            fr = r["buffers"]["frames"]
            assert fr is not None and fr.shape[1:] == (fields, 560, 720, 3)
            n, shape = _mp4_frames(path)
            assert n == r["video_frames"] >= r["steps"] > 0
            assert n - r["steps"] < play._CHUNK
            assert shape == ((560, 720, 3) if fields == 1 else (1120, 1440, 3))
            assert np.array_equal(fr[-1].cpu().numpy(), _restated(envs.engine, 0, fields, 560, 720))
        else:
            assert r["buffers"]["frames"] is None and r["video_frames"] == 0
        runs.append(r)
        envs.close()
    for r in runs[1:]:
        assert (r["score"], r["length"], r["matches"], r["steps"]) == \
            (runs[0]["score"], runs[0]["length"], runs[0]["matches"], runs[0]["steps"])
        assert torch.equal(r["state"].view(torch.int32), runs[0]["state"].view(torch.int32))
    assert runs[1]["video_frames"] == runs[2]["video_frames"]
    assert torch.equal(runs[1]["buffers"]["frames"], runs[2]["buffers"]["frames"])


def test_play_matches_eager_video(tmp_path):
    from rsoccer_isaac_cleanrl_b200 import play
    out = []
    for video in (False, True):
        envs = _vss(1065, seed=23)
        steps = [0]
        zero = play.TeamZero()

        def counted(act, obs):
            steps[0] += 1
            zero(act, obs)
        torch.manual_seed(5)
        path = str(tmp_path / "eager.mp4") if video else None
        out.append(play.play_matches(envs, counted, play.get_team("ou"), 200, video_path=path) + (steps[0],))
        envs.close()
    assert out[0] == out[1]
    assert _mp4_frames(str(tmp_path / "eager.mp4")) == (out[1][2], (560, 720, 3))


def test_play_cli_writes_one_video_per_opponent(tmp_path):
    from rsoccer_isaac_cleanrl_b200 import play
    d = str(tmp_path / "out")
    play.main(["--blue", "zero", "--yellow", "ou", "--num-envs", "256", "--matches", "20", "--video", d])
    n, shape = _mp4_frames(os.path.join(d, "zero_vs_ou.mp4"))
    assert n > 0 and n % play._CHUNK == 0 and shape == (560, 720, 3)


# ------------------------------------------------------------------ ppo --capture-video
def _train(tmp_path, backend, capture):
    from rsoccer_isaac_cleanrl_b200 import ppo
    T, N = 16, 256
    argv = ["--env-id", "sa", "--num-envs", str(N), "--num-steps", str(T), "--total-timesteps", str(N * T * 5),
            "--quiet", "--tensorboard", "false", "--mlp-backend", backend, "--save-path", str(tmp_path),
            "--record-video-step-frequency", str(2 * T), "--seed", "3"]
    args = ppo.parse_args(argv + (["--capture-video"] if capture else []))
    seen = []

    def hook(update, d):
        rec = dict(update=update, stats={k: v.detach().clone() for k, v in d["stats"].items()},
                   flat=d["flat"].detach().clone(), rewards=d["rewards"].clone(), actions=d["actions"].clone())
        fr = d["frames"]
        rec["frames"] = None if fr is None else fr.clone()
        if fr is not None:
            rec["restated"] = _restated(d["env"].engine, 0, 1, 560, 720)
        seen.append(rec)
    st = ppo.train(args, hook=hook)
    return st, seen


def test_capture_video_torch_backend_is_bit_identical(tmp_path):
    """--mlp-backend torch is reproducible run to run: with and without the flag, every per-update statistic and the
    final parameters are bit-identical (updates 1, 3 and 5 record: eager, capturing and replaying)."""
    st0, seen0 = _train(tmp_path / "a", "torch", False)
    st1, seen1 = _train(tmp_path / "b", "torch", True)
    assert st0["videos"] == [] and len(st1["videos"]) == 3
    assert [r["frames"] is not None for r in seen1] == [True, False, True, False, True]
    for a, b in zip(seen0, seen1):
        for k in a["stats"]:
            assert torch.equal(a["stats"][k], b["stats"][k]), (a["update"], k)
        for k in ("flat", "rewards", "actions"):
            assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), (a["update"], k)
    for k in ("lr", "minibatches", "epochs"):
        assert st0[k] == st1[k]
    p0 = torch.cat([p.detach().reshape(-1) for p in st0["agent"].parameters()])
    p1 = torch.cat([p.detach().reshape(-1) for p in st1["agent"].parameters()])
    assert torch.equal(p0.view(torch.int32), p1.view(torch.int32))
    assert not os.path.exists(os.path.join(str(tmp_path / "a"), "None_ppo-sa_3", "videos"))


def test_capture_video_tc_backend(tmp_path):
    st, seen = _train(tmp_path, "tc", True)
    want = [os.path.join(str(tmp_path), "None_ppo-sa_3", "videos", f"update-{u:06d}.mp4") for u in (1, 3, 5)]
    assert st["videos"] == want
    for p in want:
        assert _mp4_frames(p) == (16, (560, 720, 3))
    rec = [r for r in seen if r["frames"] is not None]
    assert [r["update"] for r in rec] == [1, 3, 5]
    for r in rec:
        assert r["frames"].shape == (16, 1, 560, 720, 3)
        assert np.array_equal(r["frames"][-1, 0].cpu().numpy(), r["restated"][0]), r["update"]
        assert not torch.equal(r["frames"][0], r["frames"][-1])
