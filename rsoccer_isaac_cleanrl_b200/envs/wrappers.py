"""Agent views — drop-ins for the reference's `envs/wrappers.py`.

`SingleAgent`, `CMA`, `DMA`, `RecordEpisodeStatisticsTorch` and `make_env` keep the reference's
names, constructor arguments and return conventions (envs/wrappers.py:21-180). Each view's
`step()` is ONE kernel launch (`vss_step_view`): OU noise for the uncontrolled robots
(wrappers.py:5-19), the policy-action overwrite, the env step, the view slicing / reward
aggregation and the running episode statistics are fused; only the policy-visible 52-float rows
are written to HBM (208 B per agent instead of 1248 B per field).
"""
import os

import numpy as np
import torch

from .._lib import VIEW_CMA, VIEW_DMA, VIEW_SA
from .spaces import Box, Wrapper


def random_ou(prev):
    """Ornstein-Uhlenbeck update of an action buffer (torch version, for callers such as team
    policies that own their buffer; the views do this inside the step kernel)."""
    ou_theta, ou_sigma = 0.1, 0.15
    return torch.clamp(prev * (1.0 - ou_theta) + ou_sigma * torch.randn_like(prev), -1.0, 1.0)


def make_env(args):
    """(raw VSS task, agent view) for args.env_id in {'sa','cma','dma'} (wrappers.py:21-48).
    `args.num_envs` counts AGENTS: for 'dma' it must be divisible by 3 and the task gets a third
    as many fields. Under torchrun each rank builds its own shard of fields (global ids offset by
    rank) on its own GPU."""
    from .vss import VSS, load_cfg
    cfg = load_cfg(getattr(args, "cfg_path", None))
    assert args.cuda, "the VSS engine is CUDA-only"
    cfg["env"]["numEnvs"] = args.num_envs
    if args.env_id == "dma":
        assert args.num_envs % 3 == 0
        cfg["env"]["numEnvs"] = int(args.num_envs / 3)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    device = f"cuda:{local_rank}"
    envs = VSS(cfg=cfg, rl_device=device, sim_device=device, graphics_device_id=0,
               headless=not getattr(args, "capture_video", False),
               virtual_screen_capture=getattr(args, "capture_video", False), force_render=False,
               seed=getattr(args, "seed", 0), global_env_offset=rank * cfg["env"]["numEnvs"])
    wrappers = {"sa": SingleAgent, "cma": CMA, "dma": DMA}
    return envs, wrappers[args.env_id](envs)


class _FusedView(Wrapper):
    VIEW = None
    AGENTS = 1   # view "envs" per field
    ACT_DIM = 2

    def __init__(self, env):
        super().__init__(env)
        task = env.unwrapped
        self.task = task
        n, dev = task.num_fields, task.device
        nv = n * self.AGENTS
        self.num_view_envs = nv
        f32 = torch.float32
        self._action_space = Box(-1.0, 1.0, (self.ACT_DIM,))
        self._observation_space = Box(-np.inf, np.inf, (task.num_obs,))
        self.action_buf = torch.zeros((n, 2, 3, 2), device=dev, dtype=f32)  # env.dof_velocity_buf.clone()
        self._obs = torch.zeros((nv, task.num_obs), device=dev, dtype=f32)
        self._term_obs = torch.zeros_like(self._obs)
        self._rews = torch.zeros((nv, 4), device=dev, dtype=f32)
        self._reward = torch.zeros(nv, device=dev, dtype=f32)
        self._done = torch.zeros(nv, device=dev, dtype=torch.long)
        self._timeout_u8 = torch.zeros(nv, device=dev, dtype=torch.uint8)
        self._progress = torch.zeros(nv, device=dev, dtype=f32)
        self.episode_returns = self.episode_lengths = None
        self.returned_episode_returns = self.returned_episode_lengths = None
        self._host = None
        self._packed_out = None  # optional: where a step()'s packed rows go (vss_set_step_packed)
        self.opponent = None     # set_opponent: the team in the yellow slots (None = OU noise, the reference's view)

    # ---- running episode statistics fused into the step epilogue (wrappers.py:50-87)
    def enable_episode_stats(self):
        nv, dev = self.num_view_envs, self.task.device
        self.episode_returns = torch.zeros((nv, 4), dtype=torch.float32, device=dev)
        self.episode_lengths = torch.zeros(nv, dtype=torch.int32, device=dev)
        self.returned_episode_returns = torch.zeros((nv, 4), dtype=torch.float32, device=dev)
        self.returned_episode_lengths = torch.zeros(nv, dtype=torch.int32, device=dev)

    def _slice_obs(self, full):
        raise NotImplementedError

    def reset(self, **kwargs):
        observations = self.env.reset(**kwargs)
        if self.opponent is not None:
            self.opponent.load(observations["obs"])
        return {"obs": self._slice_obs(observations["obs"])}

    def set_opponent(self, team, seed=0):
        """Puts a team in the yellow slots of every following step: None (OU noise, the reference's view), a play.py
        team object (TeamZero, TeamOU, TeamSA, TeamCMA, TeamDMA) or any `team(act, obs)` callable, which fills
        act (N,3,2) in place from the yellow team's mirrored observation obs (N,3,52). Policy teams run on the
        device (their actor, sampled with their own Philox stream from `seed`); see include/vss_b200.h,
        vss_set_view_opponent, for what one step then computes. Call reset() afterwards: the opponent's first
        input is the post-reset observation."""
        from .. import _lib
        from ..play import _team_mode
        mode = _team_mode(team) if team is not None else _lib.TEAM_OU
        self.opponent = None if mode == _lib.TEAM_OU else _Opponent(self, team, mode, seed)
        if self.opponent is None:
            self.task.engine.set_view_opponent(None)

    def step(self, action, obs_out=None, term_obs_out=None, reward_out=None, obs_bf16_out=None, done_f_out=None,
             timeout_f_out=None, opponent_issued=False):
        """One fused step. The optional `*_out` tensors (contiguous, right shape) make the kernel write
        the observation / terminal observation / scalar reward straight into caller storage — e.g. the
        `(T, N, …)` rollout slabs of the PPO loop (ppo…:258-272) — instead of the view's own buffers.
        `obs_bf16_out (N',64) bf16`, `done_f_out`, `timeout_f_out (N') f32` are extra copies in the form the
        tensor-core MLP and the GAE kernel read (no conversion launches between the steps).
        With an opponent (set_opponent) the step first runs the opponent's call (its actor launch, or the team
        callable on its observation), then the kernel. `opponent_issued=True`: the caller has already issued the
        device opponent's actor (`opponent.launch`) and advances its counter itself (the PPO rollout)."""
        task = self.task
        if action.device != task.device or action.dtype != torch.float32 or not action.is_contiguous():
            action = action.to(task.device, torch.float32).contiguous()
        obs = self._obs if obs_out is None else obs_out
        term_obs = self._term_obs if term_obs_out is None else term_obs_out
        reward = self._reward if reward_out is None else reward_out
        opp = self.opponent
        if opp is not None and not opponent_issued:
            opp.act(self.action_buf)
        task.engine.step_view(self.VIEW, action, self.action_buf, task.reset_buf, obs, term_obs,
                              self._rews, reward, self._done, self._timeout_u8, self._progress,
                              self.episode_returns, self.episode_lengths, self.returned_episode_returns,
                              self.returned_episode_lengths, obs_bf16=obs_bf16_out, done_f=done_f_out,
                              timeout_f=timeout_f_out, packed=self._packed_out,
                              opponent=None if opp is None else opp.spec)
        if opp is not None and not opponent_issued and opp.device is not None:
            opp.device.counter.add_(1)
        task._obs_stale = True
        infos = task.extras
        infos["rews"] = self._rews
        infos["terminal_observation"] = term_obs
        infos["time_outs"] = self._timeout_u8.view(torch.bool)
        infos["progress_buffer"] = self._progress
        return {"obs": obs}, reward, self._done, infos

    # ---- the same call with HOST buffers (pinned): action in, (obs, reward, done) out
    HOST_CHUNKS = 8            # large batches are stepped in this many field ranges ...
    HOST_CHUNK_MIN_FIELDS = 1 << 17   # ... when there are at least this many fields
    # Packed rows go to a device staging buffer and cross PCIe as ONE cudaMemcpyAsync per field range.
    # (The kernel can also store straight into the mapped pinned buffer — `vss_set_step_packed` takes any
    # device-accessible pointer — but 8-byte stores across PCIe reach 21 GB/s where the copy engine reaches
    # 55 GB/s: 5.51 vs 2.37 ms per 2^20-field step, profiles/r02_a_e2e_host_rows.md.)

    def _host_buffers(self, packed):
        from .. import _lib
        from ..hostmem import pinned_empty
        task, nv = self.task, self.num_view_envs
        if self._host is None:
            self._host = dict(
                act=torch.empty((nv, self.ACT_DIM), device=task.device, dtype=torch.float32),
                streams=[torch.cuda.Stream(device=task.device) for _ in range(2)])
        h = self._host
        if packed and "rows" not in h:
            rows = pinned_empty((nv, _lib.PACKED_ROW_BYTES), torch.uint8, task.device)
            h["rows"] = rows
            h["rows_dev"] = torch.zeros((nv, _lib.PACKED_ROW_BYTES), device=task.device, dtype=torch.uint8)
            # zero-copy views of the 112-byte rows (include/vss_b200.h: vss_set_step_packed)
            h["obs16"] = rows.view(torch.bfloat16)[:, :task.num_obs]
            h["reward_p"] = rows.view(torch.float32)[:, 26]
            h["done_p"], h["timeout_p"] = rows[:, 108], rows[:, 109]
        if not packed and "obs" not in h:
            h["obs"] = pinned_empty((nv, task.num_obs), torch.float32, task.device)
            h["reward"] = pinned_empty((nv,), torch.float32, task.device)
            h["done"] = pinned_empty((nv,), torch.long, task.device)
        return h

    def step_host(self, action_host, obs_dtype=torch.bfloat16):
        """One step with HOST buffers: pinned policy action in, what `step()` returns to the policy out
        (envs/wrappers.py:108-115: observation, scalar reward, done) in pinned host memory.

        `obs_dtype=torch.bfloat16` (default): one packed 112-byte row per view env (52 bf16 observation
        values, f32 reward, u8 done, u8 time-out), written by the step kernel itself; returns zero-copy
        views `(obs (N',52) bf16, reward (N') f32, done (N') uint8)` of that buffer (`host_timeouts` is the
        fourth column). `obs_dtype=torch.float32`: the reference's own types (f32 observation, int64 done),
        220 bytes per view env, copied from the view's device buffers.

        Large batches are pipelined: the fields are split into ranges (`vss_set_step_range`), each with its
        own H2D copy -> kernel (-> D2H copy) on one of two side streams. Same kernels, same RNG keys: the
        device-side results are bit-identical to `step()`."""
        task, nv = self.task, self.num_view_envs
        if self.opponent is not None:
            raise NotImplementedError("step_host: opponents run on the device path only (step())")
        packed = obs_dtype == torch.bfloat16
        if not packed and obs_dtype != torch.float32:
            raise ValueError("step_host: obs_dtype must be torch.bfloat16 or torch.float32")
        h = self._host_buffers(packed)
        n, agents = task.num_fields, nv // task.num_fields
        chunks = self.HOST_CHUNKS if n >= self.HOST_CHUNK_MIN_FIELDS else 1
        if packed:
            # one C call: the range pipeline (H2D of the range's actions, kernel, ONE D2H of its rows, two streams)
            # runs inside the library — a Python loop over the ranges cannot keep a 2 ms step fed on a busy host
            if "bufs" not in h:
                from .. import _lib
                p = lambda t: None if t is None else t.data_ptr()
                h["bufs"] = _lib.ViewBuffers(
                    p(h["act"]), p(self.action_buf), p(task.reset_buf), p(self._obs), p(self._term_obs), p(self._rews),
                    p(self._reward), p(self._done), p(self._timeout_u8), p(self._progress), p(self.episode_returns),
                    p(self.episode_lengths), p(self.returned_episode_returns), p(self.returned_episode_lengths),
                    p(h["rows_dev"]))
                h["bufs_stats"] = self.episode_returns is not None
            assert h["bufs_stats"] == (self.episode_returns is not None), "enable_episode_stats() after the first step_host"
            act_host = action_host.view(h["act"].shape)
            if not act_host.is_pinned():
                h.setdefault("act_pinned", torch.empty(tuple(h["act"].shape), dtype=torch.float32).pin_memory()).copy_(act_host)
                act_host = h["act_pinned"]
            task.engine.step_view_host(self.VIEW, h["bufs"], act_host, h["rows"], chunks)
            task._obs_stale = True
            return h["obs16"], h["reward_p"], h["done_p"]
        act_host = action_host.view(h["act"].shape)
        cur = torch.cuda.current_stream(task.device)
        g = task.engine.step_granularity
        per = -(-n // (chunks * g)) * g
        start = torch.cuda.Event()
        start.record(cur)
        ok = False
        try:
            for c in range(chunks):
                f0 = c * per
                cnt = min(per, n - f0)
                if cnt <= 0:
                    break
                v0, v1 = f0 * agents, (f0 + cnt) * agents
                s = h["streams"][c & 1] if chunks > 1 else cur
                with torch.cuda.stream(s):
                    s.wait_event(start)
                    h["act"][v0:v1].copy_(act_host[v0:v1], non_blocking=True)
                    if chunks > 1:
                        task.engine.set_step_range(f0, cnt)
                    obs, reward, done, _ = self.step(h["act"])
                    h["obs"][v0:v1].copy_(obs["obs"][v0:v1], non_blocking=True)
                    h["reward"][v0:v1].copy_(reward[v0:v1], non_blocking=True)
                    h["done"][v0:v1].copy_(done[v0:v1], non_blocking=True)
            ok = True
        finally:
            if chunks > 1:
                task.engine.set_step_range(0, 0)
            if not ok:  # a step abandoned after some of its range launches: forget the partial CTA count
                torch.cuda.synchronize(task.device)
                task.engine.step_count = task.engine.step_count
        if chunks > 1:
            for s in h["streams"]:
                cur.wait_stream(s)
        cur.synchronize()
        return h["obs"], h["reward"], h["done"]

    @property
    def host_timeouts(self):
        """(N') uint8 view of the time-out column of the packed rows of the last `step_host`."""
        return self._host["timeout_p"]

    @staticmethod
    def host_outputs_as_f32(obs, reward, done):
        """The reference's own types (f32 observation, f32 reward, int64 done) from either host format."""
        return obs.float(), reward.float().contiguous(), done.long()

    def d2h_bytes(self, obs_dtype=torch.bfloat16):
        from .. import _lib
        per = _lib.PACKED_ROW_BYTES if obs_dtype == torch.bfloat16 else self.task.num_obs * 4 + 4 + 8
        return self.num_view_envs * per

    @property
    def h2d_bytes_per_step(self):
        return self.num_view_envs * self.ACT_DIM * 4

    @property
    def d2h_bytes_per_step(self):
        return self.d2h_bytes(torch.bfloat16)


class _Opponent:
    """The yellow team of a fused view (set_opponent): its device mode and the buffers the step kernel reads and
    writes for it. `spec` is the `opponent` argument of Engine.step_view.
      policy teams, tc backend  play._DevicePolicy: bf16 actor weights, its own Philox seed / counter, its bf16 rows
                                (written by the step kernel) and the action of one fused actor launch (`launch`);
      policy teams, fp32 Agent  (mlp_backend "torch") the Agent's sampled action on the f32 observation, passed in
                                the same SA / CMA / DMA mode (the OU slots still come from the kernel);
      EXTERNAL                  the callable, run on the f32 observation before the step;
      ZERO                      nothing."""

    def __init__(self, view, team, mode, seed):
        from .. import _lib
        from ..play import _DevicePolicy, _team_seed
        task = view.task
        n, dev = task.num_fields, task.device
        self.team, self.mode = team, mode
        self.device = None
        self.obs_f32 = None
        policy = mode in (_lib.TEAM_SA, _lib.TEAM_CMA, _lib.TEAM_DMA)
        if policy and getattr(team.agent, "mlp_backend", "tc") == "tc":
            self.device = _DevicePolicy(team, mode, 1, task.obs_buf.view(n * 6, -1), n, _team_seed(seed, 1))
            self.spec = (mode, self.device.action, self.device.rows, None)
            return
        self.obs_f32 = torch.zeros((n, 3, task.num_obs), device=dev, dtype=torch.float32)
        self.obs_f32.copy_(task.obs_buf[:, 1])
        if policy:
            self.action = torch.zeros((3 * n, 2) if mode == _lib.TEAM_DMA else (n, 6 if mode == _lib.TEAM_CMA else 2),
                                      device=dev, dtype=torch.float32)
            self.spec = (mode, self.action, None, self.obs_f32)
        else:
            self.spec = (mode, None, None, self.obs_f32 if mode == _lib.TEAM_EXTERNAL else None)

    def load(self, full_obs):
        """The opponent's input from a full (N,2,3,52) post-reset observation: obs[:, 1]."""
        if self.device is not None:
            self.device.load_rows(full_obs.reshape(-1, full_obs.shape[-1]))
        if self.obs_f32 is not None:
            self.obs_f32.copy_(full_obs[:, 1])

    def launch(self, call_offset=0):
        """The device opponent's fused actor launch (sampling call index = counter + call_offset)."""
        self.device.launch(call_offset)

    def act(self, action_buf):
        """The opponent's call before a step."""
        from .. import _lib
        if self.device is not None:
            self.launch(0)
        elif self.mode == _lib.TEAM_EXTERNAL:
            self.team(action_buf[:, 1], self.obs_f32)
        elif self.mode in (_lib.TEAM_SA, _lib.TEAM_CMA, _lib.TEAM_DMA):
            x = self.obs_f32.view(-1, self.obs_f32.shape[-1]) if self.mode == _lib.TEAM_DMA else self.obs_f32[:, 0]
            with torch.no_grad():
                self.action.copy_(self.team.agent.get_action_and_value(x.contiguous())[0].view(self.action.shape))


class SingleAgent(_FusedView):
    """Controls blue robot 0; the other five follow OU noise (wrappers.py:89-115)."""
    VIEW, AGENTS, ACT_DIM = VIEW_SA, 1, 2

    @property
    def act_view(self):
        return self.action_buf[:, 0, 0, :]

    def _slice_obs(self, full):
        return full[:, 0, 0, :]


class CMA(_FusedView):
    """Centralised multi-agent: one 6-dim action drives blue robots 0-2, observing robot 0's view;
    reward = mean over the three blue robots (wrappers.py:118-148)."""
    VIEW, AGENTS, ACT_DIM = VIEW_CMA, 1, 6

    def __init__(self, env):
        super().__init__(env)
        self.num_envs = getattr(env, "num_envs", 1)
        self.device = env.device

    @property
    def act_view(self):
        return self.action_buf[:, 0, :, :].view(-1, 6)

    def _slice_obs(self, full):
        return full[:, 0, 0, :]


class DMA(_FusedView):
    """Decentralised multi-agent: blue robots 0-2 are three agents, field-major (wrappers.py:151-180)."""
    VIEW, AGENTS, ACT_DIM = VIEW_DMA, 3, 2

    def __init__(self, env):
        super().__init__(env)
        setattr(env.unwrapped, "num_environments", getattr(env, "num_envs", 1) * 3)

    def _slice_obs(self, full):
        return full[:, 0, :, :].reshape(-1, self.task.num_obs)


def _find_fused(env):
    e = env
    while e is not None:
        if isinstance(e, _FusedView):
            return e
        e = getattr(e, "env", None) if isinstance(e, Wrapper) else None
    return None


class _EpisodeReturns(dict):
    """`infos["r"]` of RecordEpisodeStatisticsTorch.step (envs/wrappers.py:76-83): the four reward components of the
    last finished episode are views of the statistics buffer; their sum ("return") is computed when it is read, not
    once per step (one launch less inside the captured rollout)."""

    def __init__(self, r):
        super().__init__(goal=r[:, 0], grad=r[:, 1], move=r[:, 2], energy=r[:, 3])
        self._r = r

    def __missing__(self, key):
        if key == "return":
            return self._r.sum(1)
        raise KeyError(key)

    def __contains__(self, key):
        return key == "return" or super().__contains__(key)

    def get(self, key, default=None):
        return self[key] if key in self else default

    def keys(self):
        return list(super().keys()) + ["return"]


class RecordEpisodeStatisticsTorch(Wrapper):
    """Per-env running sums of the 4 reward components and the episode length
    (wrappers.py:50-87). Over a fused view the sums are maintained by the step kernel;
    over any other env they are computed with torch ops."""

    def __init__(self, env, device):
        super().__init__(env)
        self.num_envs = getattr(env, "num_envs", 1)
        self.device = device
        self._fused = _find_fused(env)
        self.episode_returns = None
        self.episode_lengths = None

    def reset(self, **kwargs):
        observations = super().reset(**kwargs)
        if self._fused is not None:
            v = self._fused
            v.enable_episode_stats()
            self.episode_returns, self.episode_lengths = v.episode_returns, v.episode_lengths
            self.returned_episode_returns = v.returned_episode_returns
            self.returned_episode_lengths = v.returned_episode_lengths
            return observations
        z = lambda shape, dt: torch.zeros(shape, dtype=dt, device=self.device)
        self.episode_returns, self.episode_lengths = z((self.num_envs, 4), torch.float32), z(self.num_envs, torch.int32)
        self.returned_episode_returns = z((self.num_envs, 4), torch.float32)
        self.returned_episode_lengths = z(self.num_envs, torch.int32)
        return observations

    def step(self, action, **out):
        observations, rewards, dones, infos = self.env.step(action, **out) if out else super().step(action)
        if self._fused is None:
            self.episode_returns += infos["rews"]
            self.episode_lengths += 1
            self.returned_episode_returns[:] = self.episode_returns
            self.returned_episode_lengths[:] = self.episode_lengths
            self.episode_returns *= 1 - dones.unsqueeze(1)
            self.episode_lengths *= 1 - dones
        infos["r"] = _EpisodeReturns(self.returned_episode_returns)
        infos["l"] = self.returned_episode_lengths
        return observations, rewards, dones, infos
