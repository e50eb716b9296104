"""B200: the match step (vss_step_match) and play.play_matches_fused against the oracle, the full-contract step,
the views' OU stream, the fused actor launch and the eager play_matches loop."""
import numpy as np
import pytest

import match_checks as mc
from backends import GpuBackend, with_wpt

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _cfg(n):
    from rsoccer_isaac_cleanrl_b200.envs import load_cfg
    cfg = load_cfg()
    cfg["env"]["numEnvs"] = n
    return cfg


def _vss(n, seed):
    from rsoccer_isaac_cleanrl_b200.envs import VSS
    envs = VSS(_cfg(n), "cuda:0", "cuda:0", 0, True, seed=seed)
    envs.w_goal, envs.w_grad, envs.w_move, envs.w_energy = 1.0, 0.0, 0.0, 0.0   # ppo…:389-392
    return envs


@pytest.fixture(scope="module")
def checkpoint(tmp_path_factory):
    """A (barely trained) ppo-sa checkpoint in the reference's state_dict format, as test_gpu_api uses."""
    from rsoccer_isaac_cleanrl_b200 import ppo
    args = ppo.parse_args(["--env-id", "sa", "--num-envs", "128", "--num-steps", "8", "--total-timesteps",
                           str(128 * 8), "--quiet"])
    st = ppo.train(args)
    path = str(tmp_path_factory.mktemp("match") / "agent.pt")
    torch.save(st["agent"].state_dict(), path)
    return path


# ------------------------------------------------------------------ the step against the oracle and its twins
@pytest.mark.parametrize("modes", [(mc.SA, mc.OU), (mc.ZERO, mc.OU), (mc.CMA, mc.DMA), (mc.DMA, mc.ZERO),
                                   (mc.EXTERNAL, mc.SA)], ids=lambda m: f"{m[0]}v{m[1]}")
def test_match_step_parity(modes):
    """Team slots, OU within 2e-6 of the restated draw, bit-exact against the full step from the same state (state,
    reset flags, obs, bf16 rows), oracle physics within tolerance, scoreboard = the loop's statistics."""
    mc.check_match(GpuBackend, modes=modes)


@pytest.mark.parametrize("wpt,fpt", [(1, 32), (1, 16), (1, 8), (2, 32), (4, 16), (7, 8), (8, 32), (8, 16), (8, 8)])
def test_match_step_every_launch_shape(wpt, fpt):
    """Every launch shape computes the same match step (checked bit-exact against the full step of that shape,
    whose shapes are pinned bit-identical by the parity suite)."""
    mc.check_match(with_wpt(GpuBackend, wpt, fpt), modes=(mc.SA, mc.DMA), n=1065, steps=6)


def test_match_shapes_bit_identical():
    """The same match run under every launch shape: identical state, actions, rows and scoreboard."""
    import rsoccer_isaac_cleanrl_b200 as R
    n, results = 1065, []
    for wpt, fpt in [(0, 0), (1, 32), (1, 16), (1, 8), (2, 32), (4, 16), (7, 8), (8, 32), (8, 16), (8, 8)]:
        eng = R.Engine(n, "cuda:0", seed=3)
        eng.warps_per_tile, eng.fields_per_tile = wpt, fpt
        rb = torch.ones(n, dtype=torch.int64, device="cuda")
        obs = torch.zeros((n, 2, 3, 52), device="cuda")
        eng.reset_dones(rb, obs)
        g = torch.Generator(device="cuda").manual_seed(5)
        ab = torch.zeros((n, 2, 3, 2), device="cuda")
        board = torch.zeros(5, dtype=torch.int64, device="cuda")
        rows = torch.zeros((n, 64), dtype=torch.bfloat16, device="cuda")
        for _ in range(30):
            act = torch.rand((n, 2), device="cuda", generator=g) * 2 - 1
            eng.step_match([(mc.SA, act, rows), (mc.OU, None, None)], ab, rb, board, 1000, 50, obs=obs)
        results.append([eng.get_state().view(torch.int32), ab.view(torch.int32), rows.view(torch.int16), board,
                        obs.view(torch.int32)])
        eng.close()
    for r in results[1:]:
        for a, b in zip(results[0], r):
            assert torch.equal(a, b)


def test_rows_equal_gather_pad_of_the_full_step_obs():
    """Blue rows = gather_pad_bf16(obs[:,0] rows), yellow rows = gather_pad_bf16 of the mirrored obs[:,1] rows."""
    import rsoccer_isaac_cleanrl_b200 as R
    from rsoccer_isaac_cleanrl_b200.engine import gather_pad_bf16
    n = 777
    e1, e2 = R.Engine(n, "cuda:0", seed=8), R.Engine(n, "cuda:0", seed=8)
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device="cuda")
    rb1, rb2 = torch.ones(n, dtype=torch.int64, device="cuda"), torch.ones(n, dtype=torch.int64, device="cuda")
    o1, o2 = z(n, 2, 3, 52), z(n, 2, 3, 52)
    e1.reset_dones(rb1, o1); e2.reset_dones(rb2, o2)
    ab = torch.rand((n, 2, 3, 2), device="cuda") * 2 - 1
    act_b, act_y = torch.rand((n, 6), device="cuda"), torch.rand((3 * n, 2), device="cuda")
    rows_b, rows_y = z(n, 64, dt=torch.bfloat16), z(3 * n, 64, dt=torch.bfloat16)
    board = z(5, dt=torch.int64)
    for _ in range(12):
        e1.step_match([(mc.CMA, act_b, rows_b), (mc.DMA, act_y, rows_y)], ab, rb1, board, n, 10 ** 6)
        e2.step(ab.clone(), rb2, o2, z(n, 2, 3, 52), z(n, 2, 3, 4), z(n, dt=torch.uint8), z(n))
        flat = o2.view(n * 6, 52)
        ar = torch.arange(n, device="cuda")
        assert torch.equal(rows_b.view(torch.int16), gather_pad_bf16(flat, 6 * ar, 64).view(torch.int16))
        idx_y = (6 * ar[:, None] + 3 + torch.arange(3, device="cuda")).reshape(-1)
        assert torch.equal(rows_y.view(torch.int16), gather_pad_bf16(flat, idx_y, 64).view(torch.int16))
        assert torch.equal(rb1, rb2)


def test_ou_slots_equal_the_views_draw():
    """The OU slots are the SingleAgent view's OU draw at the same step index, bit for bit."""
    import rsoccer_isaac_cleanrl_b200 as R
    n = 512
    e1, e2 = R.Engine(n, "cuda:0", seed=2), R.Engine(n, "cuda:0", seed=2)
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device="cuda")
    rb = torch.ones(n, dtype=torch.int64, device="cuda")
    e1.reset_dones(rb, z(n, 2, 3, 52)); e2.reset_dones(rb, z(n, 2, 3, 52))
    rb.zero_()
    e1.step_count = e2.step_count = 17
    prev = torch.rand((n, 2, 3, 2), device="cuda") * 2 - 1
    ab1, ab2 = prev.clone(), prev.clone()
    act = torch.rand((n, 2), device="cuda")
    e1.step_match([(mc.SA, act, z(n, 64, dt=torch.bfloat16)), (mc.OU, None, None)], ab1, rb.clone(),
                  z(5, dt=torch.int64), n, 1)
    e2.step_view(R._lib.VIEW_SA, act, ab2, rb.clone(), z(n, 52), z(n, 52), z(n, 4), z(n), z(n, dt=torch.int64),
                 z(n, dt=torch.uint8), z(n))
    torch.cuda.synchronize()
    assert e1.step_count == e2.step_count == 18
    # (the view zeroes done rows afterwards; the match keeps them)
    keep = ab2.view(n, 12).abs().sum(1) != 0
    assert torch.equal(ab1.view(n, 12)[keep].view(torch.int32), ab2.view(n, 12)[keep].view(torch.int32))


def test_policy_slots_equal_policy_sample_of_the_layer_by_layer_mean(checkpoint):
    from rsoccer_isaac_cleanrl_b200 import play
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused, policy_sample
    from rsoccer_isaac_cleanrl_b200.tc_mlp import forward_explicit
    n = 1065
    for algo in ("ppo-sa", "ppo-dma"):
        team = play.get_team(algo, checkpoint)
        mode = play._team_mode(team)
        obs = torch.randn((n * 6, 52), device="cuda")
        pol = play._DevicePolicy(team, mode, 1, obs, n, play._team_seed(3, 1))
        pol.launch(0)
        mean_layers, _ = forward_explicit(pol.mw, pol.rows)
        # the fused launch's own mean (same arithmetic as the layer-by-layer path up to the stated tolerance)
        mean_fused = mlp_forward_fused(pol.rows, [(pol.mw.w16, pol.mw.bs, pol.mw.head_w, pol.mw.head_b, None)])[0]
        sw = sum(float(w.detach().abs().sum()) for w in pol.mw.ws + [pol.mw.head_w])
        assert float((mean_fused - mean_layers).abs().max()) <= 2e-5 * (sw + float(mean_layers.abs().max()))
        ref, _ = policy_sample(mean_fused, pol.logstd, pol.seed, torch.zeros(1, dtype=torch.int32, device="cuda"))
        assert torch.equal(pol.action.view(torch.int32), ref.view(torch.int32))   # bit-equal noise
        assert pol.rows.shape[0] == (3 * n if algo == "ppo-dma" else n)


def test_noise_of_the_two_teams_is_uncorrelated(checkpoint):
    """Self-play with one checkpoint: the same rows through both teams' samplers, |corr(noise)| < 0.01."""
    from rsoccer_isaac_cleanrl_b200 import play
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused
    team = play.get_team("ppo-sa", checkpoint)
    n = 131072
    obs = torch.randn((n * 6, 52), device="cuda")
    pols = [play._DevicePolicy(team, play._lib.TEAM_SA, 0, obs, n, play._team_seed(0, side)) for side in (0, 1)]
    pols[1].rows.copy_(pols[0].rows)
    for p in pols:
        p.launch(0)
    mean = mlp_forward_fused(pols[0].rows, [(pols[0].mw.w16, pols[0].mw.bs, pols[0].mw.head_w, pols[0].mw.head_b, None)])[0]
    a, b = (pols[0].action - mean).flatten().double(), (pols[1].action - mean).flatten().double()
    corr = float(((a - a.mean()) * (b - b.mean())).mean() / (a.std() * b.std()))
    assert abs(corr) < 0.01, corr
    assert float(a.std()) > 0.1 and float(b.std()) > 0.1


# ------------------------------------------------------------------ play_matches_fused
def test_external_teams_bit_parity_with_play_matches(checkpoint):
    """zero / ou / ppo-sa / ppo-dma team objects wrapped as EXTERNAL: identical score, length, steps, action buffers
    and final state as play_matches on a twin VSS (same torch seed, same engine seed)."""
    from rsoccer_isaac_cleanrl_b200 import play
    teams = {k: play.get_team(k, None if k in ("zero", "ou") else checkpoint) for k in ("zero", "ou", "ppo-sa", "ppo-dma")}
    for blue_k, yellow_k in (("ou", "zero"), ("ppo-sa", "ppo-dma"), ("ppo-dma", "ou")):
        runs = []
        for fused in (False, True):
            envs = _vss(1065, seed=21)
            seen = {"steps": 0}

            def wrap(team, side):
                def ext(act, obs):
                    if side == 0:
                        seen["steps"] += 1
                    seen[side] = act
                    team(act, obs)
                return ext
            torch.manual_seed(1234)
            run = play.play_matches_fused if fused else play.play_matches
            score, length = run(envs, wrap(teams[blue_k], 0), wrap(teams[yellow_k], 1), 300)
            torch.cuda.synchronize()
            runs.append((score, length, seen["steps"], seen[0].clone(), seen[1].clone(),
                         envs.engine.get_state().view(torch.int32)))
            envs.close()
        (s0, l0, n0, b0, y0, st0), (s1, l1, n1, b1, y1, st1) = runs
        assert (s0, l0, n0) == (s1, l1, n1), (blue_k, yellow_k, runs[0][:3], runs[1][:3])
        assert torch.equal(b0.view(torch.int32), b1.view(torch.int32)) and torch.equal(y0.view(torch.int32), y1.view(torch.int32))
        assert torch.equal(st0, st1)


def test_graph_replay_equals_eager_steps():
    """A captured chunk of match steps replayed equals the same steps run eagerly: state, scoreboard, actions;
    the step index advances with every replayed step."""
    import rsoccer_isaac_cleanrl_b200 as R
    n, K = 1065, 8
    out = []
    for graph in (False, True):
        eng = R.Engine(n, "cuda:0", seed=6)
        z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device="cuda")
        rb = torch.ones(n, dtype=torch.int64, device="cuda")
        eng.reset_dones(rb, z(n, 2, 3, 52))
        ab, board = z(n, 2, 3, 2), z(5, dt=torch.int64)
        act = torch.rand((n, 6), device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)) * 2 - 1
        rows = z(n, 64, dt=torch.bfloat16)

        def chunk():
            for _ in range(K):
                eng.step_match([(mc.OU, None, None), (mc.CMA, act, rows)], ab, rb, board, 1000, 10 ** 6)
        if graph:
            chunk()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                chunk()
            for _ in range(3):
                g.replay()
        else:
            for _ in range(4):
                chunk()
        torch.cuda.synchronize()
        assert eng.step_count == 4 * K
        out.append([eng.get_state().view(torch.int32), ab.view(torch.int32), board, rows.view(torch.int16)])
        eng.close()
    for a, b in zip(*out):
        assert torch.equal(a, b)
    assert mc.board_dict(out[0][2].cpu().numpy())["steps"] == 4 * K


def _play_matches_recorded(envs, blue_team, yellow_team, n_matches, count_envs=1065):
    """play_matches (play.py) with the per-match values kept: (scores, lengths) of every counted episode."""
    envs.reset_buf[:] = 1
    envs.reset_dones()
    n = envs.cfg["env"]["numEnvs"]
    action_buf = torch.zeros((n,) + envs.action_space.shape, device=envs.device)
    obs = envs.reset()["obs"]
    count_envs = min(count_envs, n)
    scores, lengths = [], []
    while sum(len(x) for x in scores) < n_matches:
        blue_team(action_buf[:, 0], obs[:, 0])
        yellow_team(action_buf[:, 1], obs[:, 1])
        obs, rew, dones, info = envs.step(action_buf)
        obs = obs["obs"]
        env_ids = dones[:count_envs].nonzero(as_tuple=False).squeeze(-1)
        if len(env_ids):
            scores.append(rew[env_ids, 0, 0, 0].double().cpu())
            lengths.append(info["progress_buffer"][env_ids].double().cpu())
    return torch.cat(scores).numpy(), torch.cat(lengths).numpy()


@pytest.mark.parametrize("blue,yellow", [("ou", "zero"), ("ppo-sa", "ou")])
def test_fused_statistics_agree_with_play_matches(blue, yellow, checkpoint):
    """10 000 matches each way: fused and eager mean score and length within 4 standard errors of their
    difference, the standard errors from the per-match spread of the eager run."""
    from rsoccer_isaac_cleanrl_b200 import play
    n_matches = 10000
    path = checkpoint if blue.startswith("ppo") else None
    runs = []
    for recorded in (False, True):  # play_matches, then its restatement that keeps the per-match values
        torch.manual_seed(7)
        envs = _vss(1065, seed=31)
        run = _play_matches_recorded if recorded else play.play_matches
        runs.append(run(envs, play.get_team(blue, path), play.get_team(yellow), n_matches))
        if not recorded:
            envs.close()
    (s_e, l_e), (scores, lengths) = runs
    # the restatement reproduces play_matches exactly (same engine seed, same torch seed)
    assert (float(scores.sum()) / len(scores), float(lengths.sum()) / len(lengths)) == (s_e, l_e)
    r = play._run_matches_fused(envs, play.get_team(blue, path), play.get_team(yellow), n_matches, seed=5)
    assert r["matches"] >= n_matches and r["steps"] > 0
    k = np.sqrt(1.0 / len(scores) + 1.0 / r["matches"])
    se_score, se_length = scores.std(ddof=1) * k, lengths.std(ddof=1) * k
    assert se_score > 0 and se_length > 0
    assert abs(r["score"] - s_e) <= 4 * se_score, (r["score"], s_e, se_score)
    assert abs(r["length"] - l_e) <= 4 * se_length, (r["length"], l_e, se_length)


@pytest.mark.parametrize("blue,yellow", [("ppo-sa", "ppo-dma"), ("ppo-sa", "ppo-sa"), ("ppo-cma", "ppo-dma")])
def test_two_policy_graph_replays_equal_eager_chunks(blue, yellow, checkpoint, tmp_path):
    """Two policy teams, well past the first (eager) chunk: the graph replays record both actors (the second on a
    side stream) and equal the same chunks run eagerly, bit for bit: state, scoreboard, action buffer, both teams'
    last sampled actions."""
    from rsoccer_isaac_cleanrl_b200 import play
    out = []
    for graphs in (False, True):
        envs = _vss(1065, seed=13)
        teams = [play.get_team(k, _ckpt(k, checkpoint, tmp_path)) for k in (blue, yellow)]
        r = play._run_matches_fused(envs, teams[0], teams[1], 600, seed=2, graphs=graphs)
        torch.cuda.synchronize()
        assert r["steps"] > 4 * play._CHUNK
        b = r["buffers"]
        out.append([r["score"], r["length"], r["matches"], r["steps"], envs.engine.get_state().view(torch.int32),
                    b["action_buf"].view(torch.int32), b["policy_action"][0].view(torch.int32),
                    b["policy_action"][1].view(torch.int32)])
        envs.close()
    for a, b in zip(*out):
        assert (torch.equal(a, b) if isinstance(a, torch.Tensor) else a == b)


def _ckpt(algo, checkpoint, tmp_path):
    """The ppo-sa checkpoint serves sa / sa-x3 / dma teams; a cma team gets a freshly initialised 6-action Agent."""
    if algo != "ppo-cma":
        return checkpoint
    from collections import namedtuple
    from rsoccer_isaac_cleanrl_b200.envs.spaces import Box
    from rsoccer_isaac_cleanrl_b200.ppo import Agent
    path = tmp_path / "cma.pt"
    if not path.exists():
        d = namedtuple("d", ["single_observation_space", "single_action_space"])
        torch.manual_seed(0)
        agent = Agent(d(Box(-np.inf, np.inf, (52,)), Box(-1.0, 1.0, (6,))), mlp_backend="tc")
        torch.save(agent.state_dict(), str(path))
    return str(path)


def test_fused_match_runner_stops_on_the_scoreboard(checkpoint):
    from rsoccer_isaac_cleanrl_b200 import play
    envs = _vss(1065, seed=4)
    for yellow in ("zero", "ou"):
        r = play._run_matches_fused(envs, play.get_team("ppo-sa", checkpoint), play.get_team(yellow), 500)
        assert 500 <= r["matches"] < 500 + 1065 and -1.0 <= r["score"] <= 1.0 and 1.0 <= r["length"] <= 400.0
    # obs_buf is rebuilt from the state on the next read
    assert envs._obs_stale
    envs.reset()
    assert not envs._obs_stale


def test_step_match_rejects_ranges_and_count_envs():
    import rsoccer_isaac_cleanrl_b200 as R
    n = 256
    eng = R.Engine(n, "cuda:0", seed=1)
    z = lambda *s, dt=torch.float32: torch.zeros(s, dtype=dt, device="cuda")
    ab, rb, board = z(n, 2, 3, 2), z(n, dt=torch.int64), z(5, dt=torch.int64)
    teams = [(mc.OU, None, None), (mc.ZERO, None, None)]
    for bad in (0, n + 1):
        with pytest.raises(RuntimeError, match="count_envs"):
            eng.step_match(teams, ab, rb, board, bad, 10)
    eng.set_step_range(0, eng.step_granularity)
    with pytest.raises(RuntimeError, match="whole-engine"):
        eng.step_match(teams, ab, rb, board, n, 10)
    eng.set_step_range(0, 0)
    eng.step_match(teams, ab, rb, board, n, 10)
    torch.cuda.synchronize()
    assert eng.step_count == 1
