"""B200: the opponent view step (vss_set_view_opponent + vss_step_view), the views' set_opponent and PPO's --opponent,
against the restatement through the full-contract step, an EXTERNAL twin, the eager rollout and the field's symmetry."""
import numpy as np
import pytest

import opponent_checks as oc
from backends import VIEW_CMA, VIEW_DMA, VIEW_SA, GpuBackend, with_wpt

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

VIEWS = (VIEW_SA, VIEW_CMA, VIEW_DMA)


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _train(argv, hook=None):
    from rsoccer_isaac_cleanrl_b200 import ppo
    return ppo.train(ppo.parse_args(argv + ["--quiet", "--tensorboard", "false"]), hook=hook)


@pytest.fixture(scope="module")
def checkpoints(tmp_path_factory):
    """Barely trained sa and cma checkpoints in the reference's state_dict format (as test_gpu_match builds one)."""
    out = {}
    for env_id in ("sa", "cma"):
        st = _train(["--env-id", env_id, "--num-envs", "128", "--num-steps", "8", "--total-timesteps", str(128 * 8)])
        path = str(tmp_path_factory.mktemp("opp") / f"{env_id}.pt")
        torch.save(st["agent"].state_dict(), path)
        out[env_id] = path
    return out


# ------------------------------------------------------------------ the step against the restatement
@pytest.mark.parametrize("mode", oc.OPP_MODES)
@pytest.mark.parametrize("view", VIEWS)
def test_opponent_view_parity(view, mode):
    oc.check_opponent(GpuBackend, view, mode)


@pytest.mark.parametrize("n", [1000, 2300, 6000, 20000, 140000])
def test_opponent_view_every_automatic_shape(n):
    """Sizes that select each automatic launch shape (k_step_cta with 8 / 16 / 32 fields per tile, k_step with 1, 2
    and 4 warps per CTA)."""
    view, mode = VIEWS[n % 3], oc.OPP_MODES[n % 5]
    oc.check_opponent(GpuBackend, view, mode, n=n, steps=4)


@pytest.mark.parametrize("fpt", [32, 16, 8])
@pytest.mark.parametrize("wpt", [1, 2, 4, 7, 8])
def test_opponent_view_explicit_shapes(wpt, fpt):
    view, mode = VIEWS[(wpt + fpt) % 3], oc.OPP_MODES[(wpt * 3 + fpt) % 5]
    oc.check_opponent(with_wpt(GpuBackend, wpt, fpt), view, mode, n=1065, steps=5)


@pytest.mark.parametrize("view,mode", [(VIEW_SA, oc.SA), (VIEW_DMA, oc.CMA), (VIEW_CMA, oc.EXTERNAL)])
def test_opponent_view_split_into_ranges(view, mode):
    """The step issued as three vss_set_step_range launches equals the restatement (so the whole-engine launch)."""
    oc.check_opponent(GpuBackend, view, mode, n=5000, steps=5, step_range=3)


@pytest.mark.parametrize("view", VIEWS)
def test_mode_ou_equals_no_opponent(view):
    oc.check_ou_mode_is_no_opponent(GpuBackend, view)


def test_host_buffer_path_rejects_an_opponent():
    from rsoccer_isaac_cleanrl_b200 import _lib
    from rsoccer_isaac_cleanrl_b200.envs import VSS, SingleAgent, load_cfg
    cfg = load_cfg()
    cfg["env"]["numEnvs"] = 256
    view = SingleAgent(VSS(cfg, "cuda:0", "cuda:0", 0, True, seed=1))
    view.reset()
    eng = view.task.engine
    eng.set_view_opponent((_lib.TEAM_ZERO, None, None, None))
    buf = _lib.ViewBuffers()
    dev_act, dev_rows = torch.zeros((256, 2), device="cuda"), torch.zeros((256, _lib.PACKED_ROW_BYTES), device="cuda",
                                                                         dtype=torch.uint8)
    buf.policy_action, buf.packed_rows = dev_act.data_ptr(), dev_rows.data_ptr()
    act = torch.zeros((256, 2)).pin_memory()
    rows = torch.zeros((256, _lib.PACKED_ROW_BYTES), dtype=torch.uint8).pin_memory()
    rc = eng.lib.vss_step_view_host(eng._h, _lib.VIEW_SA, buf, act.data_ptr(), rows.data_ptr(), 1, None)
    assert rc == -1 and b"host-buffer path" in eng.lib.vss_last_error()
    eng.set_view_opponent(None)


# ------------------------------------------------------------------ views with a device policy opponent
def _view(env_id, n, seed):
    from rsoccer_isaac_cleanrl_b200.envs import CMA, DMA, VSS, SingleAgent, load_cfg
    cfg = load_cfg()
    cfg["env"]["numEnvs"] = n
    return {"sa": SingleAgent, "cma": CMA, "dma": DMA}[env_id](VSS(cfg, "cuda:0", "cuda:0", 0, True, seed=seed))


@pytest.mark.parametrize("algo", ["ppo-sa-x3", "ppo-cma"])
def test_device_policy_opponent_equals_an_external_twin(algo, checkpoints):
    """A view with a device policy opponent against a twin whose EXTERNAL opponent writes the first run's sampled
    opponent actions into the yellow slots: bit-identical over 50 steps. The sampled actions are vss_policy_sample
    of the fused actor's mean on the rows the kernel wrote. (DMA and CMA modes drive all six yellow slots; an SA
    opponent's robots 1-2 keep the kernel's OU draw, which no caller can write for the fields that end in the step;
    its slots are covered by the restatement parity above.)"""
    from rsoccer_isaac_cleanrl_b200 import play
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused, policy_sample
    team = play.get_team(algo, checkpoints["cma" if algo == "ppo-cma" else "sa"])
    n, steps = 1065, 50
    dev_view, twin = _view("sa", n, 5), _view("sa", n, 5)
    dev_view.set_opponent(team, seed=11)
    sampled = []

    def external(act, obs):
        act[:] = sampled[-1].view(-1, 3, 2)
    twin.set_opponent(external)
    dev_view.reset()
    twin.reset()
    pol = dev_view.opponent.device
    g = torch.Generator(device="cuda").manual_seed(3)
    dones = 0
    for step in range(steps):
        rows, counter = pol.rows.clone(), pol.counter.clone()
        action = torch.rand((n, 2), device="cuda", generator=g) * 2 - 1
        o1, r1, d1, _ = dev_view.step(action)
        o1, r1, d1 = o1["obs"].clone(), r1.clone(), d1.clone()
        sampled.append(pol.action.clone())
        mean = mlp_forward_fused(rows, [(pol.mw.w16, pol.mw.bs, pol.mw.head_w, pol.mw.head_b, None)])[0]
        ref, _ = policy_sample(mean, pol.logstd, pol.seed, counter)
        assert torch.equal(sampled[-1].view(torch.int32), ref.view(torch.int32)), step
        o2, r2, d2, _ = twin.step(action)
        assert torch.equal(o1.view(torch.int32), o2["obs"].view(torch.int32)), step
        assert torch.equal(r1.view(torch.int32), r2.view(torch.int32)) and torch.equal(d1, d2), step
        assert torch.equal(dev_view.action_buf.view(torch.int32), twin.action_buf.view(torch.int32)), step
        assert torch.equal(dev_view.task.engine.get_state().view(torch.int32), twin.task.engine.get_state().view(torch.int32))
        # the rows the kernel wrote for the next call are the yellow rows of the twin's f32 observation
        want = twin.opponent.obs_f32
        want = want.reshape(-1, 52) if algo == "ppo-sa-x3" else want[:, 0]
        assert torch.equal(pol.rows[:, :52].view(torch.int16), want.to(torch.bfloat16).view(torch.int16)), step
        dones += int(d1.sum())
    assert dones > 0


def test_symmetric_self_play_has_no_goal_bias(checkpoints):
    """Learner and opponent are the same sa checkpoint (the learner's action sampled from it on its own stream): by the
    mirror symmetry of the field, the observation and the reset distribution, the mean blue goal term over >= 5000
    ended episodes is within 4 standard errors of 0."""
    from rsoccer_isaac_cleanrl_b200 import _lib, play
    from rsoccer_isaac_cleanrl_b200.engine import gather_pad_bf16
    team = play.get_team("ppo-sa", checkpoints["sa"])
    n = 8192
    view = _view("sa", n, 77)
    view.set_opponent(team, seed=101)
    view.reset()
    blue = play._DevicePolicy(team, _lib.TEAM_SA, 0, view.task.obs_buf.view(n * 6, -1), n, play._team_seed(202, 0))
    goals, count = [], 0
    with torch.no_grad():
        for _ in range(1200):
            blue.launch(0)
            o, r, d, info = view.step(blue.action)
            blue.counter.add_(1)
            blue.rows.copy_(gather_pad_bf16(o["obs"], None, 64))
            ended = d.nonzero().flatten()
            if ended.numel():
                goals.append(info["rews"][ended, 0].double())
                count += ended.numel()
            if count >= 6000:
                break
    g = torch.cat(goals)
    mean, se = float(g.mean()), float(g.std() / g.numel() ** 0.5)
    assert g.numel() >= 5000
    assert int((g != 0).sum()) >= 20, "too few goals for the statistic to say anything"
    assert abs(mean) <= 4 * se, (mean, se, int((g > 0).sum()), int((g < 0).sum()))


# ------------------------------------------------------------------ PPO
def _collect(store):
    def hook(update, t):
        opp = t["opponent"]
        store.append(dict(obs=t["obs"].clone(), actions=t["actions"].clone(), rewards=t["rewards"].clone(),
                          dones=t["next_dones"].clone(), opp_action=opp.device.action.clone(),
                          state=t["env"].engine.get_state().clone()))
    return hook


@pytest.mark.parametrize("opponent", ["checkpoint", "self"])
def test_rollout_graph_replay_equals_eager_rollout(opponent, checkpoints):
    """With the weights held fixed (--update-epochs 0), rollouts replayed from the captured graph equal the same
    rollouts issued eagerly, bit for bit: obs, actions, rewards, dones, the opponent's actions and the state."""
    spec = f"ppo-cma:{checkpoints['cma']}" if opponent == "checkpoint" else "self"
    runs = []
    for graph in ("true", "false"):
        store = []
        _train(["--env-id", "dma", "--num-envs", "1536", "--num-steps", "16", "--total-timesteps", str(1536 * 16 * 3),
                "--update-epochs", "0", "--opponent", spec, "--cuda-graph", graph], hook=_collect(store))
        runs.append(store)
    for u, (a, b) in enumerate(zip(*runs)):
        for k in a:
            assert torch.equal(a[k].view(torch.int32), b[k].view(torch.int32)), (u + 1, k)
    assert len(runs[0]) == 3


def test_self_play_snapshots_follow_the_refresh_period():
    """--opponent self --opponent-refresh 2: the opponent's weights (fp32 and bf16) equal the learner's conversion at
    the refresh updates (1, 3, 5) and do not change in between, while the learner's do."""
    from rsoccer_isaac_cleanrl_b200.tc_mlp import MlpWeights
    seen = []

    def hook(update, t):
        opp = t["opponent"].device
        learner = MlpWeights(t["agent"].actor_mean)
        seen.append(dict(opp16=[w.clone() for w in opp.mw.w16], opp32=[w.detach().clone() for w in opp.mw.ws],
                         logstd=opp.logstd.clone(), learner16=[w.clone() for w in learner.w16],
                         learner_logstd=t["agent"].actor_logstd.detach().reshape(-1).clone()))
    _train(["--env-id", "sa", "--num-envs", "512", "--num-steps", "8", "--total-timesteps", str(512 * 8 * 5),
            "--opponent", "self", "--opponent-refresh", "2"], hook=hook)
    same = lambda xs, ys: all(torch.equal(x.view(torch.int16 if x.dtype == torch.bfloat16 else torch.int32),
                                          y.view(torch.int16 if y.dtype == torch.bfloat16 else torch.int32))
                              for x, y in zip(xs, ys))
    assert len(seen) == 5
    for u in (1, 3):  # (seen[u] = after update u + 1)
        assert same(seen[u]["opp16"], seen[u - 1]["opp16"]) and same(seen[u]["opp32"], seen[u - 1]["opp32"])
        assert not same(seen[u]["learner16"], seen[u - 1]["learner16"])
    for u in (2, 4):  # snapshots before updates 3 and 5: the learner as it left updates 2 and 4
        assert same(seen[u]["opp16"], seen[u - 1]["learner16"]), u
        assert same([seen[u]["logstd"]], [seen[u - 1]["learner_logstd"]]), u
        assert not same(seen[u]["opp16"], seen[u - 2]["opp16"])


@pytest.mark.parametrize("env_id,opponent,backend", [("sa", "zero", "auto"), ("cma", "self", "auto"),
                                                     ("dma", "ppo-cma", "auto"), ("sa", "self", "torch"),
                                                     ("cma", "ppo-sa", "torch")])
def test_ppo_with_opponents_trains_and_saves(env_id, opponent, backend, checkpoints, tmp_path):
    """Small runs finish with finite losses; the saved checkpoint loads as a play.py team."""
    from rsoccer_isaac_cleanrl_b200 import play
    spec = f"{opponent}:{checkpoints[opponent[4:]]}" if opponent.startswith("ppo-") else opponent
    losses = []
    num = 768 if env_id == "dma" else 256
    st = _train(["--env-id", env_id, "--num-envs", str(num), "--num-steps", "8", "--total-timesteps", str(num * 8 * 3),
                 "--opponent", spec, "--opponent-refresh", "2", "--mlp-backend", backend],
                hook=lambda u, t: losses.append([float(t["stats"][k]) for k in ("pg_loss", "v_loss", "entropy")]))
    assert len(losses) == 3 and np.isfinite(np.array(losses)).all(), losses
    path = str(tmp_path / "agent.pt")
    torch.save(st["agent"].state_dict(), path)
    algo = {"sa": "ppo-sa", "cma": "ppo-cma", "dma": "ppo-dma"}[env_id]
    team = play.get_team(algo, path)
    assert play._team_mode(team) in (play._lib.TEAM_SA, play._lib.TEAM_CMA, play._lib.TEAM_DMA)
