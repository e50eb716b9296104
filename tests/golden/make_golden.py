"""Generate golden vectors by EXECUTING THE REFERENCE'S OWN CODE.

Run in the build container only (needs /root/reference, which does not exist on the GPU
box):   python tests/golden/make_golden.py
Outputs (committed): tests/golden/jit_functions.npz, gae.npz, wrappers.npz, agent.npz, ppo_update.npz,
play.npz, ppo_schedule.npz, ppo_defaults.json

Nothing from the reference is copied into the repo: the source ranges below are read from
/root/reference at generation time and exec'd in a scratch namespace.
  - envs/vss.py:530-655       the six @torch.jit.script functions (obs, 4 rewards, dones);
                              `device="cuda:0"` at :536 is rewritten to "cpu" (no GPU here), and
                              isaacgym.torch_utils.get_euler_xyz (un-vendored) is supplied by a
                              stand-in restating its published formula (SURVEY App. C).
  - ppo_continuous_action_isaacgym.py:282-296   the GAE loop, verbatim.
  - ppo_continuous_action_isaacgym.py:121-164   layer_init + Agent, verbatim.
  - ppo_continuous_action_isaacgym.py:48-118    parse_args, verbatim (flag names and defaults).
  - envs/wrappers.py (whole file)  executed against a 20-line `gym` shim (gym 0.23.1 is
                              un-vendored) and a fake task that replays fixed VSS.step outputs.
"""
import os
import sys
import textwrap
import types

import numpy as np
import torch

REF = os.environ.get("VSS_REFERENCE", "/root/reference")
OUT = os.path.dirname(os.path.abspath(__file__))


def _lines(path, lo, hi):
    with open(os.path.join(REF, path)) as f:
        src = f.readlines()
    return "".join(src[lo - 1:hi])


# ------------------------------------------------------------------ reference jit functions
def load_ref_jit():
    src = _lines("envs/vss.py", 526, 655).replace('device="cuda:0"', 'device="cpu"')
    prelude = textwrap.dedent('''
        import numpy as np
        import torch
        from torch import Tensor
        from typing import Tuple

        @torch.jit.script
        def get_euler_xyz(q):
            # type: (Tensor) -> Tuple[Tensor, Tensor, Tensor]
            qx, qy, qz, qw = 0, 1, 2, 3
            sinr_cosp = 2.0 * (q[:, qw] * q[:, qx] + q[:, qy] * q[:, qz])
            cosr_cosp = q[:, qw] * q[:, qw] - q[:, qx] * q[:, qx] - q[:, qy] * q[:, qy] + q[:, qz] * q[:, qz]
            roll = torch.atan2(sinr_cosp, cosr_cosp)
            sinp = 2.0 * (q[:, qw] * q[:, qy] - q[:, qz] * q[:, qx])
            pitch = torch.where(torch.abs(sinp) >= 1, torch.sign(sinp) * (3.141592653589793 / 2.0), torch.asin(sinp))
            siny_cosp = 2.0 * (q[:, qw] * q[:, qz] + q[:, qx] * q[:, qy])
            cosy_cosp = q[:, qw] * q[:, qw] + q[:, qx] * q[:, qx] - q[:, qy] * q[:, qy] - q[:, qz] * q[:, qz]
            yaw = torch.atan2(siny_cosp, cosy_cosp)
            return roll % (2 * 3.141592653589793), pitch % (2 * 3.141592653589793), yaw % (2 * 3.141592653589793)
    ''')
    # torch.jit.script needs real source files -> write a scratch module outside the repo
    import importlib.util
    import tempfile
    d = tempfile.mkdtemp(prefix="vss_ref_jit_")
    path = os.path.join(d, "ref_jit_scratch.py")
    with open(path, "w") as f:
        f.write(prelude + "\n" + src)
    spec = importlib.util.spec_from_file_location("ref_jit_scratch", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def make_states(rng, n):
    """Random field states in the reference's tensor layouts, with edge cases."""
    ball_pos = rng.uniform(-1, 1, (n, 2)).astype(np.float32) * np.float32([0.85, 0.65])
    prev_ball_pos = (ball_pos + rng.normal(0, 0.03, (n, 2))).astype(np.float32)
    # edge cases: balls inside both goals, on the goal line, just outside the mouth, at the origin
    ball_pos[0] = [0.80, 0.05]
    ball_pos[1] = [-0.78, -0.19]
    ball_pos[2] = [0.75, 0.0]       # on the line: not > 0.75 -> no goal
    ball_pos[3] = [0.76, 0.2]       # |y| == 0.2 -> no goal
    ball_pos[4] = [-0.7500001, 0.1]
    ball_pos[5] = [0.0, 0.0]
    ball_pos[6] = [0.8, 0.3]        # behind the end wall, outside the mouth
    ball_vel = rng.uniform(-1.5, 1.5, (n, 2)).astype(np.float32)
    ball_vel[5] = 0.0               # exercises the -0.0 of the mirrored view
    r_pos = (rng.uniform(-1, 1, (n, 2, 3, 2)) * [0.85, 0.65]).astype(np.float32)
    prev_r_pos = (r_pos + rng.normal(0, 0.03, (n, 2, 3, 2))).astype(np.float32)
    r_vel = rng.uniform(-1.2, 1.2, (n, 2, 3, 2)).astype(np.float32)
    yaw = rng.uniform(-np.pi, np.pi, (n, 2, 3))
    yaw[5] = 0.0
    yaw[6, 0, 0] = np.pi / 2
    yaw[6, 0, 1] = -np.pi
    quats = np.zeros((n, 2, 3, 4), np.float32)  # xyzw, rotation about z (vss.py:313-315)
    quats[..., 2] = np.sin(yaw / 2)
    quats[..., 3] = np.cos(yaw / 2)
    r_w = rng.uniform(-30, 30, (n, 2, 3, 1)).astype(np.float32)
    r_w[5] = 0.0
    acts = rng.uniform(-1, 1, (n, 2, 3, 2)).astype(np.float32)
    acts[5] = 0.0
    progress = rng.integers(0, 405, (n,)).astype(np.int64)
    progress[7], progress[8], progress[9] = 399, 400, 401
    reset_buf = rng.integers(0, 2, (n,)).astype(np.int64)
    return dict(ball_pos=ball_pos, prev_ball_pos=prev_ball_pos, ball_vel=ball_vel, r_pos=r_pos,
                prev_r_pos=prev_r_pos, r_vel=r_vel, quats=quats, r_w=r_w, acts=acts, progress=progress,
                reset_buf=reset_buf)


def gen_jit(mod):
    rng = np.random.default_rng(20261018)
    s = make_states(rng, 96)
    t = {k: torch.from_numpy(v) for k, v in s.items()}
    perms = torch.tensor([[0, 1, 2], [1, 2, 0], [2, 0, 1]])      # vss.py:173-175
    mirror = torch.tensor([-1.0] * 6 + [1.0] * 3)                # vss.py:166-171
    yellow_goal = torch.tensor([1.5 / 2, 0.0])                   # vss.py:154-159
    out = dict(s)
    out["obs"] = mod.compute_obs(t["ball_pos"], t["ball_vel"], t["r_pos"], t["r_vel"], t["quats"], t["r_w"],
                                 t["acts"], perms, mirror).numpy()
    out["goal_rew"] = mod.compute_goal_rew(t["reset_buf"], t["ball_pos"], 1.5, 0.4).numpy()
    out["grad_rew"] = mod.compute_grad_rew(t["prev_ball_pos"], t["ball_pos"], yellow_goal).numpy()
    out["move_rew"] = mod.compute_move_rew(t["prev_r_pos"], t["r_pos"], t["prev_ball_pos"], t["ball_pos"]).numpy()
    out["energy_rew"] = mod.compute_energy_rew(t["acts"]).numpy()
    out["dones"] = mod.compute_vss_dones(t["ball_pos"], t["reset_buf"], t["progress"], 400.0, 1.5, 0.4).numpy()
    # (cos, sin) of the yaw the engine stores instead of quaternions, from the same quats in f64
    q = s["quats"].astype(np.float64)
    c = q[..., 3] ** 2 + q[..., 0] ** 2 - q[..., 1] ** 2 - q[..., 2] ** 2
    sn = 2.0 * (q[..., 3] * q[..., 2] + q[..., 0] * q[..., 1])
    nrm = np.sqrt(c * c + sn * sn)
    out["r_rot"] = np.stack([c / nrm, sn / nrm], -1).astype(np.float32)
    assert out["obs"].shape == (96, 2, 3, 52) and out["goal_rew"].dtype == np.int64
    np.savez_compressed(os.path.join(OUT, "jit_functions.npz"), **out)
    print("jit_functions.npz", {k: v.shape for k, v in out.items() if k in ("obs", "goal_rew", "dones")})


# ------------------------------------------------------------------ GAE loop
def gen_gae():
    src = textwrap.dedent(_lines("ppo_continuous_action_isaacgym.py", 282, 296))
    assert src.startswith("with torch.no_grad():") and "returns = advantages + values" in src
    rng = np.random.default_rng(7)
    cases = {}
    for name, (T, N) in {"a": (16, 8), "b": (128, 33), "c": (1, 5)}.items():
        rewards = rng.normal(0, 1, (T, N)).astype(np.float32)
        values = rng.normal(0, 2, (T, N)).astype(np.float32)
        next_values = rng.normal(0, 2, (T, N)).astype(np.float32)
        next_dones = (rng.uniform(size=(T, N)) < 0.15).astype(np.float32)
        next_timeouts = ((rng.uniform(size=(T, N)) < 0.5) * next_dones).astype(np.float32)
        next_timeouts[0, 0] = 1.0  # timeout flag without done (cannot happen, but defined)
        ns = dict(torch=torch, device="cpu", args=types.SimpleNamespace(num_steps=T, gamma=0.99, gae_lambda=0.95),
                  rewards=torch.from_numpy(rewards), values=torch.from_numpy(values),
                  next_values=torch.from_numpy(next_values), next_dones=torch.from_numpy(next_dones),
                  next_timeouts=torch.from_numpy(next_timeouts))
        exec(src, ns)
        for k, v in dict(rewards=rewards, values=values, next_values=next_values, next_dones=next_dones,
                         next_timeouts=next_timeouts, advantages=ns["advantages"].numpy(),
                         returns=ns["returns"].numpy()).items():
            cases[f"{name}_{k}"] = v
    np.savez_compressed(os.path.join(OUT, "gae.npz"), **cases)
    print("gae.npz", sorted(cases)[:3], "...")


# ------------------------------------------------------------------ wrappers against a fake task
def _gym_shim():
    gym = types.ModuleType("gym")

    class Box:
        def __init__(self, low, high, shape):
            self.low, self.high, self.shape = low, high, tuple(shape)

    class Wrapper:
        def __init__(self, env):
            self.env = env

        def __getattr__(self, name):
            if name.startswith("_"):
                raise AttributeError(name)
            return getattr(self.env, name)

        def reset(self, **kw):
            return self.env.reset(**kw)

        def step(self, action):
            return self.env.step(action)

    gym.Wrapper = Wrapper
    gym.spaces = types.SimpleNamespace(Box=Box)
    return gym


class FakeTask:
    """Replays fixed VSS.step outputs; records the action buffer it is stepped with."""

    def __init__(self, steps):
        self.steps = steps
        self.num_envs = steps[0]["obs"].shape[0]
        self.num_obs, self.num_actions = 52, 2
        self.device = "cpu"
        self.dof_velocity_buf = torch.zeros((self.num_envs, 2, 3, 2))
        self.t = 0
        self.seen_actions = []

    def reset(self):
        return {"obs": torch.from_numpy(self.steps[0]["obs0"]).clone()}

    def step(self, actions):
        self.seen_actions.append(actions.clone().numpy())
        s = self.steps[self.t]
        self.t += 1
        infos = {"time_outs": torch.from_numpy(s["timeout"]).clone(),
                 "terminal_observation": torch.from_numpy(s["term_obs"]).clone(),
                 "progress_buffer": torch.from_numpy(s["progress_f"]).clone()}
        return ({"obs": torch.from_numpy(s["obs"]).clone()}, torch.from_numpy(s["rew"]).clone(),
                torch.from_numpy(s["reset"]).clone(), infos)


def gen_wrappers():
    sys.modules["gym"] = _gym_shim()
    import importlib.util
    spec = importlib.util.spec_from_file_location("ref_wrappers", os.path.join(REF, "envs/wrappers.py"))
    W = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(W)
    rng = np.random.default_rng(11)
    n, T = 7, 4
    steps = []
    for t in range(T):
        reset = (rng.uniform(size=n) < 0.4).astype(np.int64)
        steps.append(dict(
            obs0=rng.normal(size=(n, 2, 3, 52)).astype(np.float32),
            obs=rng.normal(size=(n, 2, 3, 52)).astype(np.float32),
            term_obs=rng.normal(size=(n, 2, 3, 52)).astype(np.float32),
            rew=rng.normal(size=(n, 2, 3, 4)).astype(np.float32),
            reset=reset, timeout=((rng.uniform(size=n) < 0.5) & (reset != 0)),
            progress_f=rng.integers(1, 400, n).astype(np.float32)))
    out = {"n": np.int64(n), "T": np.int64(T)}
    for t, s in enumerate(steps):
        for k, v in s.items():
            out[f"in{t}_{k}"] = v
    for name, cls, adim in (("sa", W.SingleAgent, 2), ("cma", W.CMA, 6), ("dma", W.DMA, 2)):
        torch.manual_seed(5)
        task = FakeTask(steps)
        env = W.RecordEpisodeStatisticsTorch(_ExtractObs(cls(task)), "cpu")
        nv = n * 3 if name == "dma" else n
        env.num_envs = nv  # the PPO script sizes the statistics by args.num_envs (= 3*fields for dma)
        o0 = env.reset()
        out[f"{name}_obs0"] = o0.numpy()
        for t in range(T):
            act = torch.from_numpy(rng.uniform(-1, 1, (nv, adim)).astype(np.float32))
            obs, reward, dones, infos = env.step(act)
            out[f"{name}{t}_policy_action"] = act.numpy()
            out[f"{name}{t}_stepped_actions"] = task.seen_actions[t]
            out[f"{name}{t}_action_buf_after"] = _view_action_buf(env).clone().numpy()
            out[f"{name}{t}_obs"] = obs.numpy().copy()
            out[f"{name}{t}_reward"] = reward.numpy().copy()
            out[f"{name}{t}_done"] = dones.numpy().copy()
            out[f"{name}{t}_term_obs"] = infos["terminal_observation"].numpy().copy()
            out[f"{name}{t}_rews"] = infos["rews"].numpy().copy()
            out[f"{name}{t}_timeout"] = infos["time_outs"].numpy().copy()
            out[f"{name}{t}_progress"] = infos["progress_buffer"].numpy().copy()
            out[f"{name}{t}_ret_ret"] = env.returned_episode_returns.numpy().copy()
            out[f"{name}{t}_ret_len"] = env.returned_episode_lengths.numpy().copy()
            out[f"{name}{t}_ep_ret"] = env.episode_returns.numpy().copy()
            out[f"{name}{t}_ep_len"] = env.episode_lengths.numpy().copy()
    np.savez_compressed(os.path.join(OUT, "wrappers.npz"), **out)
    print("wrappers.npz", len(out), "arrays")


class _ExtractObs:
    """ExtractObsWrapper (ppo...:167-169) over the gym shim."""

    def __init__(self, env):
        self.env = env

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.env, name)

    def reset(self, **kw):
        return self.env.reset(**kw)["obs"]

    def step(self, a):
        o, r, d, i = self.env.step(a)
        return o["obs"], r, d, i


def _view_action_buf(env):
    e = env
    while not hasattr(e, "action_buf") or "action_buf" not in vars(e):
        e = e.env
    return e.action_buf


# ------------------------------------------------------------------ Agent (MLPs)
def gen_agent():
    sys.modules.setdefault("gym", _gym_shim())
    src = _lines("ppo_continuous_action_isaacgym.py", 121, 164)
    ns = dict(torch=torch, nn=torch.nn, np=np)
    exec("from torch.distributions.normal import Normal\n" + src, ns)
    out = {}
    for name, adim in (("a2", 2),):
        torch.manual_seed(3)
        envs = types.SimpleNamespace(single_observation_space=types.SimpleNamespace(shape=(52,)),
                                     single_action_space=types.SimpleNamespace(shape=(adim,)))
        agent = ns["Agent"](envs)
        with torch.no_grad():
            agent.actor_logstd.copy_(torch.linspace(-0.5, 0.3, adim).view(1, adim))
        x = torch.randn(40, 52)
        action = torch.randn(40, adim)
        _, logp, ent, value = agent.get_action_and_value(x, action)
        mean = agent.actor_mean(x)
        # one PPO-style scalar loss to pin the backward pass
        adv = torch.randn(40)
        ret = torch.randn(40)
        loss = (-(adv * logp.exp())).mean() - 0.005 * ent.mean() + 4 * 0.5 * ((value.view(-1) - ret) ** 2).mean()
        agent.zero_grad()
        loss.backward()
        for k, v in agent.state_dict().items():
            if v.numel() <= 52 * 256:
                out[f"{name}_sd_{k}"] = v.detach().numpy().copy()
            else:  # the hidden 256/512-wide weights: the test rebuilds them from the seed and checks these
                out[f"{name}_sum_{k}"] = weight_checksum(v)
                out[f"{name}_sample_{k}"] = weight_sample(v)
        for k, p in agent.named_parameters():
            g = p.grad.detach().numpy()
            out[f"{name}_gradnorm_{k}"] = np.float64(np.sqrt((g.astype(np.float64) ** 2).sum()))
            if g.size <= 52 * 256:  # full gradients only for the small layers (keeps the fixture small)
                out[f"{name}_grad_{k}"] = g.copy()
        for k, v in dict(x=x, action=action, logp=logp, ent=ent, value=value, mean=mean, adv=adv, ret=ret,
                         loss=loss).items():
            out[f"{name}_{k}"] = v.detach().numpy().copy()
    np.savez_compressed(os.path.join(OUT, "agent.npz"), **out)
    print("agent.npz", len(out), "arrays")


# ------------------------------------------------------------------ one PPO minibatch update
def gen_ppo_update():
    """Executes the reference's own minibatch code (ppo…:314-354: loss, backward, clip_grad_norm_,
    Adam step) on its own Agent (ppo…:121-164) and records the statistics, the gradient w.r.t. the
    network outputs (captured with forward hooks) and a sample of the updated parameters."""
    sys.modules.setdefault("gym", _gym_shim())
    ns = dict(torch=torch, nn=torch.nn, np=np)
    exec("from torch.distributions.normal import Normal\n" + _lines("ppo_continuous_action_isaacgym.py", 121, 164), ns)
    body = textwrap.dedent(_lines("ppo_continuous_action_isaacgym.py", 314, 352))        # ... loss.backward()
    body_step = textwrap.dedent(_lines("ppo_continuous_action_isaacgym.py", 353, 354))   # clip_grad_norm_, optimizer.step()
    out = {}
    for name, adim, clip_vloss in (("a2", 2, False), ("a6v", 6, True)):
        torch.manual_seed(11)
        envs = types.SimpleNamespace(single_observation_space=types.SimpleNamespace(shape=(52,)),
                                     single_action_space=types.SimpleNamespace(shape=(adim,)))
        agent = ns["Agent"](envs)
        with torch.no_grad():
            agent.actor_logstd.copy_(torch.linspace(-0.4, 0.1, adim).view(1, adim))
            agent.actor_mean[8].weight.mul_(20.0)   # (initialised with std 0.01: make the mean matter)
        R, B = 160, 64
        b_obs, b_actions = torch.randn(R, 52), torch.randn(R, adim) * 0.7
        with torch.no_grad():
            _, lp, _, val = agent.get_action_and_value(b_obs, b_actions)
        b_logprobs = lp + 0.3 * torch.randn(R)        # ratios on both sides of the clip range
        b_values = val.view(-1) + 0.3 * torch.randn(R)
        b_advantages, b_returns = torch.randn(R) * 1.5 + 0.2, torch.randn(R)
        mb_inds = torch.randperm(R)[:B]
        args = types.SimpleNamespace(clip_coef=0.2, norm_adv=True, clip_vloss=clip_vloss, ent_coef=0.005, vf_coef=4.0,
                                     max_grad_norm=1.5)
        optimizer = torch.optim.Adam(agent.parameters(), lr=1e-3, eps=1e-5)
        captured = {}

        def keep(key):
            def hook(module, inputs, output):   # (returns None: the output is not replaced)
                output.retain_grad()
                captured[key] = output
            return hook

        hooks = [agent.actor_mean.register_forward_hook(keep("mean")), agent.critic.register_forward_hook(keep("value"))]
        for k, v in dict(b_obs=b_obs, b_actions=b_actions, b_logprobs=b_logprobs, b_values=b_values,
                         b_advantages=b_advantages, b_returns=b_returns, mb_inds=mb_inds,
                         logstd=agent.actor_logstd.detach().clone().view(-1)).items():
            out[f"{name}_{k}"] = v.numpy().copy()
        env = dict(ns, agent=agent, b_obs=b_obs, b_actions=b_actions, b_logprobs=b_logprobs, b_values=b_values,
                   b_advantages=b_advantages, b_returns=b_returns, mb_inds=mb_inds, args=args, optimizer=optimizer,
                   clipfracs=[])
        exec(body, env)
        for h in hooks:
            h.remove()
        out[f"{name}_d_logstd"] = agent.actor_logstd.grad.view(-1).numpy().copy()
        gn0 = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in agent.parameters()))
        out[f"{name}_grad_norm"] = np.float64(gn0.item())
        exec(body_step, env)
        for k in ("pg_loss", "v_loss", "entropy_loss", "old_approx_kl", "approx_kl", "loss"):
            out[f"{name}_{k}"] = np.float32(env[k].item())
        out[f"{name}_clipfrac"] = np.float32(env["clipfracs"][0])
        out[f"{name}_mean"] = captured["mean"].detach().numpy().copy()
        out[f"{name}_value"] = captured["value"].detach().numpy().copy()
        out[f"{name}_d_mean"] = captured["mean"].grad.numpy().copy()
        out[f"{name}_d_value"] = captured["value"].grad.numpy().copy()
        # after clip_grad_norm_: .grad holds the clipped gradient; logstd's is d_logstd * clip coefficient
        gn = torch.sqrt(sum((p.grad.double() ** 2).sum() for p in agent.parameters()))
        out[f"{name}_clipped_grad_norm"] = np.float64(gn.item())
        out[f"{name}_clipped_d_logstd"] = agent.actor_logstd.grad.view(-1).numpy().copy()
        out[f"{name}_logstd_after"] = agent.actor_logstd.detach().view(-1).numpy().copy()
    np.savez_compressed(os.path.join(OUT, "ppo_update.npz"), **out)
    print("ppo_update.npz", len(out), "arrays")



# ------------------------------------------------------------------ play.py: teams + match runner
class FakeMatchTask:
    """Raw-task stand-in for play_matches (play.py:131-164): replays fixed VSS.step outputs, records
    every action buffer it is stepped with."""

    def __init__(self, steps, obs0):
        self.steps, self.obs0 = steps, obs0
        n = obs0.shape[0]
        self.cfg = {"env": {"numEnvs": n}}
        self.device = "cpu"
        self.action_space = types.SimpleNamespace(shape=(2, 3, 2))
        self.observation_space = types.SimpleNamespace(shape=(2, 3, 52))
        self.reset_buf = torch.zeros(n, dtype=torch.long)
        self.reset_dones_calls, self.t, self.seen_actions = 0, 0, []

    def reset_dones(self):
        assert bool((self.reset_buf == 1).all())  # play.py:132-133 forces a full reset first
        self.reset_dones_calls += 1

    def reset(self):
        return {"obs": torch.from_numpy(self.obs0).clone()}

    def step(self, actions):
        self.seen_actions.append(actions.clone().numpy())
        s = self.steps[self.t]
        self.t += 1
        infos = {"progress_buffer": torch.from_numpy(s["progress_f"]).clone()}
        return ({"obs": torch.from_numpy(s["obs"]).clone()}, torch.from_numpy(s["rew"]).clone(),
                torch.from_numpy(s["reset"]).clone(), infos)


def play_fixture(rng, n=1100, T=6):
    obs0 = rng.normal(size=(n, 2, 3, 52)).astype(np.float32)
    steps = []
    for t in range(T):
        reset = (rng.uniform(size=n) < 0.02).astype(np.int64)
        reset[1065:] = 1  # fields beyond the first 1065 are never counted (play.py:158)
        rew = np.zeros((n, 2, 3, 4), np.float32)
        rew[..., 0] = rng.choice([-1.0, 0.0, 1.0], size=(n, 1, 1)).astype(np.float32) * np.float32([[1], [-1]])
        steps.append(dict(obs=rng.normal(size=(n, 2, 3, 52)).astype(np.float32), rew=rew, reset=reset,
                          progress_f=rng.integers(1, 401, n).astype(np.float32)))
    return obs0, steps


def weight_checksum(t):
    """(sum, sum of |x|) in float64: identifies a weight tensor without storing it."""
    a = t.detach().double()
    return np.float64([a.sum().item(), a.abs().sum().item()])


def weight_sample(t, stride=97, count=256):
    """A strided sample of a tensor's elements (keeps the fixtures small)."""
    return t.detach().reshape(-1)[::stride][:count].numpy().copy()


def gen_play():
    """Executes the reference's play.py:1-102 (teams, get_team) and :131-164 (play_matches) — 'cuda:0'
    rewritten to 'cpu', BASELINE_TEAMS (:105-128, loads the missing base_nets at import) left out — over
    the gym shim, the reference's own Agent (ppo…:121-164) and a fake task that replays fixed outputs."""
    import tempfile
    gym = _gym_shim()

    class ObservationWrapper(gym.Wrapper):
        def reset(self, **kw):
            return self.observation(self.env.reset(**kw))

        def step(self, action):
            o, r, d, i = self.env.step(action)
            return self.observation(o), r, d, i

    gym.ObservationWrapper = ObservationWrapper
    sys.modules["gym"] = gym
    ppo_ns = dict(torch=torch, nn=torch.nn, np=np, gym=gym)
    exec("from torch.distributions.normal import Normal\n" + _lines("ppo_continuous_action_isaacgym.py", 121, 169), ppo_ns)
    fake_ppo = types.ModuleType("ppo_continuous_action_isaacgym")
    fake_ppo.Agent, fake_ppo.ExtractObsWrapper = ppo_ns["Agent"], ppo_ns["ExtractObsWrapper"]
    sys.modules["ppo_continuous_action_isaacgym"] = fake_ppo
    src = (_lines("play.py", 1, 102) + "\n" + _lines("play.py", 131, 164)).replace("'cuda:0'", "'cpu'")
    P = {}
    exec(src, P)
    rng = np.random.default_rng(21)
    obs0, steps = play_fixture(rng)
    # (the inputs are not stored: the test regenerates them with play_fixture(default_rng(21)); a checksum
    # guards against a numpy whose generator streams differ)
    out = {"T": np.int64(len(steps)), "obs0_sum": np.float64(obs0.astype(np.float64).sum()),
           "last_obs_sum": np.float64(steps[-1]["obs"].astype(np.float64).sum())}
    # checkpoints in the reference's own format: torch.save(agent.state_dict()) (ppo…:379)
    tmp = tempfile.mkdtemp(prefix="vss_play_")
    dummy = lambda adim: types.SimpleNamespace(single_observation_space=types.SimpleNamespace(shape=(52,)),
                                               single_action_space=types.SimpleNamespace(shape=(adim,)))
    ckpt = {}
    for adim in (2, 6):
        torch.manual_seed(40 + adim)
        agent = ppo_ns["Agent"](dummy(adim))
        with torch.no_grad():
            agent.actor_mean[8].weight.mul_(30.0)
            agent.actor_logstd.fill_(-1.0)
        ckpt[adim] = os.path.join(tmp, f"agent{adim}.pt")
        torch.save(agent.state_dict(), ckpt[adim])
        # (weights are not stored: the test rebuilds them from the same seed with the product's Agent — same
        # layer order and initialisers — and checks these per-tensor checksums)
        for k, v in agent.state_dict().items():
            out[f"ckpt{adim}_sum_{k}"] = weight_checksum(v)
    cases = {"zero_vs_ou": ("zero", None, "ou", None), "sa_vs_zero": ("ppo-sa", 2, "zero", None),
             "cma_vs_dma": ("ppo-cma", 6, "ppo-dma", 2), "sax3_vs_sa": ("ppo-sa-x3", 2, "ppo-sa", 2)}
    for name, (ba, bd, ya, yd) in cases.items():
        torch.manual_seed(77)
        blue = P["get_team"](ba, ckpt.get(bd))
        yellow = P["get_team"](ya, ckpt.get(yd))
        task = FakeMatchTask(steps, obs0)
        n_matches = 60
        score, length = P["play_matches"](task, blue, yellow, n_matches)
        assert task.reset_dones_calls == 1
        out[f"{name}_score"], out[f"{name}_length"] = np.float64(score), np.float64(length)
        out[f"{name}_steps"] = np.int64(task.t)
        for t, a in enumerate(task.seen_actions):
            out[f"{name}_act{t}"] = a
    np.savez_compressed(os.path.join(OUT, "play.npz"), **out)
    print("play.npz", len(out), "arrays")


# ------------------------------------------------------------------ PPO update schedule
def schedule_fixture(adim=2, R=14):
    g = torch.Generator().manual_seed(123)
    r = lambda *s: torch.randn(*s, generator=g)
    return dict(obs=r(R, 52), actions=r(R, adim) * 0.7, dlogp=0.3 * r(R), dval=0.3 * r(R), adv=r(R) * 1.5 + 0.2, ret=r(R))


def gen_ppo_schedule():
    """Executes the reference's whole optimisation phase (ppo…:298-365: flatten, epochs, randperm,
    minibatches incl. the shorter remainder, adaptive LR, target-KL stop) and its LR annealing lines
    (:250-254) on its own Agent, batch 14 = 7 envs x 2 steps, minibatch 14 // 4 = 3 (-> 3,3,3,3,2)."""
    sys.modules.setdefault("gym", _gym_shim())
    ns0 = dict(torch=torch, nn=torch.nn, np=np)
    exec("from torch.distributions.normal import Normal\n" + _lines("ppo_continuous_action_isaacgym.py", 121, 164), ns0)
    body = textwrap.dedent(_lines("ppo_continuous_action_isaacgym.py", 298, 365))
    anneal = textwrap.dedent(_lines("ppo_continuous_action_isaacgym.py", 250, 254))
    out = {}
    fx = schedule_fixture()
    for k, v in fx.items():
        out[f"fx_{k}"] = v.numpy().copy()
    cases = {"plain": {}, "adaptive": dict(adaptative_lr=True, threshold_kl=0.008),
             "adaptive_up": dict(adaptative_lr=True, threshold_kl=50.0),
             "target_kl": dict(target_kl=0.002), "clipv_nonorm": dict(clip_vloss=True, norm_adv=False)}
    for name, over in cases.items():
        torch.manual_seed(9)
        envs = types.SimpleNamespace(single_observation_space=types.SimpleNamespace(shape=(52,)),
                                     single_action_space=types.SimpleNamespace(shape=(2,)))
        agent = ns0["Agent"](envs)
        with torch.no_grad():
            agent.actor_mean[8].weight.mul_(20.0)
            agent.actor_logstd.fill_(-0.3)
        if name == "plain":
            for k, v in agent.state_dict().items():
                out[f"init_sum_{k}"] = weight_checksum(v)
        with torch.no_grad():
            _, lp, _, val = agent.get_action_and_value(fx["obs"], fx["actions"])
        T, N = 2, 7
        args = types.SimpleNamespace(num_envs=N, num_steps=T, batch_size=T * N, minibatch_size=(T * N) // 4,
                                     update_epochs=3, clip_coef=0.2, norm_adv=True, clip_vloss=False, ent_coef=0.005,
                                     vf_coef=4.0, max_grad_norm=1.5, adaptative_lr=False, threshold_kl=0.008,
                                     target_kl=None, learning_rate=3e-3)
        for k, v in over.items():
            setattr(args, k, v)
        optimizer = torch.optim.Adam(agent.parameters(), lr=args.learning_rate, eps=1e-5)
        lr_trace, kl_trace = [], []

        class Spy(torch.optim.Adam):
            pass

        orig_step = optimizer.step

        def step_spy(*a, **k):
            lr_trace.append(optimizer.param_groups[0]["lr"])
            return orig_step(*a, **k)

        optimizer.step = step_spy
        env = dict(ns0, agent=agent, args=args, optimizer=optimizer, device="cpu", envs=envs,
                   obs=fx["obs"].view(T, N, 52), logprobs=(lp + fx["dlogp"]).view(T, N),
                   actions=fx["actions"].view(T, N, 2), advantages=fx["adv"].view(T, N), returns=fx["ret"].view(T, N),
                   values=(val.view(-1) + fx["dval"]).view(T, N))
        torch.manual_seed(31)  # the randperm stream of the update phase
        exec(body, env)
        out[f"{name}_lr_at_step"] = np.float64(lr_trace)
        out[f"{name}_lr_final"] = np.float64(optimizer.param_groups[0]["lr"])
        out[f"{name}_minibatches"] = np.int64(len(lr_trace))
        out[f"{name}_last_kl"] = np.float32(env["approx_kl"].item())
        out[f"{name}_clipfracs"] = np.float32(env["clipfracs"])
        for k, v in agent.state_dict().items():
            out[f"{name}_final_{k}"] = weight_sample(v)
    # annealing: lr at update u of num_updates
    lrs = []
    for u in (1, 2, 7, 48):
        opt = types.SimpleNamespace(param_groups=[{"lr": None}])
        env = dict(args=types.SimpleNamespace(anneal_lr=True, learning_rate=1e-3), update=u, num_updates=48, optimizer=opt)
        exec(anneal, env)
        lrs.append(opt.param_groups[0]["lr"])
    out["anneal_updates"], out["anneal_lr"] = np.int64([1, 2, 7, 48]), np.float64(lrs)
    np.savez_compressed(os.path.join(OUT, "ppo_schedule.npz"), **out)
    print("ppo_schedule.npz", len(out), "arrays", {k: int(out[f"{k}_minibatches"]) for k in cases})



def gen_ppo_defaults():
    """Defaults of every CLI flag: the reference's parse_args (ppo…:48-118) executed with no argv."""
    import argparse
    import json

    def strtobool(x):  # distutils.util.strtobool (removed from python 3.12)
        x = x.lower()
        if x in ("y", "yes", "t", "true", "on", "1"):
            return 1
        if x in ("n", "no", "f", "false", "off", "0"):
            return 0
        raise ValueError(x)

    ns = dict(argparse=argparse, strtobool=strtobool)
    exec(_lines("ppo_continuous_action_isaacgym.py", 48, 118), ns)
    old = sys.argv
    sys.argv = ["ppo"]
    try:
        d = vars(ns["parse_args"]())
        sys.argv = ["ppo", "--env-id", "dma", "--num-envs", "65535", "--num-steps", "64", "--anneal-lr", "--norm-adv", "false"]
        d2 = vars(ns["parse_args"]())
    finally:
        sys.argv = old
    with open(os.path.join(OUT, "ppo_defaults.json"), "w") as f:
        json.dump({"defaults": d, "dma_case": d2}, f, indent=1, sort_keys=True)
    print("ppo_defaults.json", len(d), "flags")


if __name__ == "__main__":
    torch.set_num_threads(1)
    gen_ppo_defaults()
    gen_jit(load_ref_jit())
    gen_gae()
    gen_wrappers()
    gen_agent()
    gen_ppo_update()
    gen_play()
    gen_ppo_schedule()
