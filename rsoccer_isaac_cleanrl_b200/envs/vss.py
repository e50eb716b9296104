"""VSS task — drop-in for the reference's `envs/vss.py::VSS(VecTask)`.

Same constructor signature, attributes and `reset()/step()/reset_dones()` contract
(reference envs/vss.py:32-73,180-203,267-333 and IsaacGymEnvs `VecTask.step/reset`), but
everything below the Python seam is one fused sm_100a kernel launch per step
(`vss_step` in libvss_b200.so) instead of IsaacGym/PhysX plus ~150 torch launches.

Differences a caller can observe (all documented in DESIGN.md):
  * physics is the engine's own 2-D model (PhysX is closed source);
  * reset RNG is counter-based Philox keyed by (seed, global field id, episode), not the
    torch global generator — same distribution, different stream;
  * `root_state`-derived views (`ball_pos`, `robots_pos`, …) are read-only snapshots.
"""
import math
import os

import numpy as np
import torch

from .. import _lib
from ..engine import Engine
from .spaces import Box

NUM_TEAMS = 2
NUM_ROBOTS = 3
BLUE_TEAM, YELLOW_TEAM = 0, 1

_HERE = os.path.dirname(os.path.abspath(__file__))


def load_cfg(path=None):
    """Plain-YAML replacement of the reference's hydra compose (envs/wrappers.py:22-26)."""
    import yaml
    with open(path or os.path.join(_HERE, "vss.yaml")) as f:
        return yaml.safe_load(f)


class VSS:
    def __init__(self, cfg, rl_device="cuda:0", sim_device="cuda:0", graphics_device_id=0, headless=True,
                 virtual_screen_capture=False, force_render=False, seed=0, global_env_offset=0):
        env = cfg["env"]
        self.cfg = cfg
        self.num_fields = int(env["numEnvs"])
        self.num_environments = self.num_fields  # DMA overwrites this with 3N (wrappers.py:154)
        self.num_agents = 1
        self.num_obs = int(env.get("numObservations", 52))
        self.num_states = int(env.get("numStates", 0))
        self.num_actions = int(env.get("numActions", 2))
        self.max_episode_length = int(env["maxEpisodeLength"])
        self.control_freq_inv = int(env.get("controlFrequencyInv", 1))
        self.clip_obs = float(env.get("clipObservations", math.inf))
        self.clip_actions = float(env.get("clipActions", math.inf))
        if self.num_obs != 52 or self.num_actions != 2:
            raise ValueError("the VSS kernels are built for numObservations=52, numActions=2")
        if self.clip_actions != 1.0 or self.control_freq_inv != 1:
            raise ValueError("the VSS kernels implement clipActions=1, controlFrequencyInv=1 (vss.yaml)")
        if not str(sim_device).startswith("cuda"):
            raise RuntimeError("VSS runs on a CUDA device only: there is no CPU pipeline in this engine")
        self.device = torch.device(sim_device)
        self.rl_device = torch.device(rl_device)
        self.graphics_device_id = graphics_device_id
        self.headless = headless
        self.virtual_screen_capture = virtual_screen_capture
        self.force_render = force_render
        self.viewer = None
        self.robot_max_wheel_rad_s = 42.0
        self.min_robot_placement_dist = 0.07
        self.field_width, self.field_height = 1.5, 1.3
        self.goal_width, self.goal_height = 0.1, 0.4

        p = _lib.default_params()
        sim = cfg.get("sim", {})
        p.dt = float(sim.get("dt", p.dt))
        p.substeps = int(sim.get("substeps", p.substeps))
        p.max_episode_length = self.max_episode_length
        w = env["rew_weights"]
        p.w_goal, p.w_grad, p.w_move, p.w_energy = float(w["goal"]), float(w["grad"]), float(w["move"]), float(w["energy"])
        self._w = [p.w_goal, p.w_grad, p.w_move, p.w_energy]
        self.seed = int(seed)
        self.global_env_offset = int(global_env_offset)
        self.engine = Engine(self.num_fields, self.device, seed=self.seed, global_env_offset=self.global_env_offset,
                             params=p)

        self.obs_space = Box(-np.inf, np.inf, (NUM_TEAMS, NUM_ROBOTS, self.num_obs))
        self.state_space = Box(-np.inf, np.inf, (NUM_TEAMS, NUM_ROBOTS, self.num_states))
        self.act_space = Box(-1.0, 1.0, (NUM_TEAMS, NUM_ROBOTS, self.num_actions))
        self.allocate_buffers()
        self.reset_dones()  # reset_buf starts as ones: every field is randomised (vss.py:72,93)

    # ------------------------------------------------------------------ VecTask surface
    @property
    def num_envs(self):
        return self.num_environments

    @property
    def observation_space(self):
        return self.obs_space

    @property
    def action_space(self):
        return self.act_space

    @property
    def unwrapped(self):
        return self

    def allocate_buffers(self):
        n, dev = self.num_fields, self.device
        f32 = torch.float32
        self.obs_buf = torch.zeros((n, NUM_TEAMS, NUM_ROBOTS, self.num_obs), device=dev, dtype=f32)
        self.terminal_obs_buf = torch.zeros_like(self.obs_buf)
        self.rew_buf = torch.zeros((n, NUM_TEAMS, NUM_ROBOTS, 4), device=dev, dtype=f32)
        self.reset_buf = torch.ones(n, device=dev, dtype=torch.long)
        self._timeout_u8 = torch.zeros(n, device=dev, dtype=torch.uint8)
        self.timeout_buf = self._timeout_u8.view(torch.bool)
        self._progress_f = torch.zeros(n, device=dev, dtype=f32)
        self.extras = {}
        self.obs_dict = {}
        self._obs_stale = False

    # reward weights are plain attributes in the reference, re-read every step (vss.py:225-253)
    def _set_w(self, i, v):
        self._w[i] = float(v)
        self.engine.set_reward_weights(*self._w)

    w_goal = property(lambda s: s._w[0], lambda s, v: s._set_w(0, v))
    w_grad = property(lambda s: s._w[1], lambda s, v: s._set_w(1, v))
    w_move = property(lambda s: s._w[2], lambda s, v: s._set_w(2, v))
    w_energy = property(lambda s: s._w[3], lambda s, v: s._set_w(3, v))

    def _obs_out(self):
        if self._obs_stale:  # a fused view stepped the engine: rebuild obs_buf from the state (no re-randomising)
            self.engine.reset_dones(torch.zeros_like(self.reset_buf), self.obs_buf)
            self._obs_stale = False
        obs = self.obs_buf if math.isinf(self.clip_obs) else torch.clamp(self.obs_buf, -self.clip_obs, self.clip_obs)
        self.obs_dict["obs"] = obs.to(self.rl_device)
        return self.obs_dict

    def reset(self):
        """VecTask.reset: returns the current observation buffer; does not re-randomise."""
        return self._obs_out()

    def reset_dones(self):
        """Re-randomise the fields flagged in `reset_buf` (which callers may write, play.py:132-133)
        and refresh `obs_buf` (vss.py:267-333 + compute_observations)."""
        self.engine.reset_dones(self.reset_buf, self.obs_buf)

    def compute_observations(self):
        """obs_buf is always current after reset_dones()/step(); kept for API compatibility."""
        return self.obs_buf

    def step(self, actions):
        """One control step: (obs_dict, rew_buf (N,2,3,4), reset_buf (N) int64, extras)."""
        if actions.device != self.device:
            actions = actions.to(self.device, non_blocking=True)
        if actions.dtype != torch.float32 or not actions.is_contiguous():
            actions = actions.contiguous().float()
        self.engine.step(actions, self.reset_buf, self.obs_buf, self.terminal_obs_buf, self.rew_buf,
                         self._timeout_u8, self._progress_f)
        self._obs_stale = False
        self.extras["terminal_observation"] = self.terminal_obs_buf.to(self.rl_device)
        self.extras["progress_buffer"] = self._progress_f.to(self.rl_device)
        self.extras["time_outs"] = self.timeout_buf.to(self.rl_device)
        return self._obs_out(), self.rew_buf.to(self.rl_device), self.reset_buf.to(self.rl_device), self.extras

    def render(self, mode="rgb_array", fields=1, height=560, width=720):
        """Fields [0, fields) as one (H', W', 3) uint8 numpy picture: each field rendered on the device
        (Engine.render, DESIGN.md §4.7), laid out by video.mosaic. The picture is the current state: after a
        step, a field that ended an episode is shown already reset. mode="human" needs a display, which this
        engine does not have."""
        if mode != "rgb_array":
            raise NotImplementedError(f"render mode {mode!r}: only 'rgb_array' is supported (there is no display)")
        from ..video import mosaic
        with torch.cuda.device(self.device):
            frames = self.engine.render(0, fields, height, width)
            return mosaic(frames).cpu().numpy()

    def close(self):
        self.engine.close()

    # ------------------------------------------------------------------ state snapshots
    def _state(self):
        return self.engine.get_state()[:, :self.num_fields]

    def _robot_words(self, k0, k1):
        s = self._state()
        idx = [4 + 9 * r + k for r in range(6) for k in range(k0, k1)]
        return s[idx].t().reshape(self.num_fields, NUM_TEAMS, NUM_ROBOTS, k1 - k0).contiguous()

    @property
    def progress_buf(self):
        return self._state()[_lib.W_PROGRESS].view(torch.int32).long()

    @property
    def ball_pos(self):
        return self._state()[0:2].t().contiguous()

    @property
    def ball_vel(self):
        return self._state()[2:4].t().contiguous()

    @property
    def robots_pos(self):
        return self._robot_words(0, 2)

    @property
    def robots_vel(self):
        return self._robot_words(2, 4)

    @property
    def robots_rot(self):
        """(N,2,3,2) cos/sin of the yaw (the reference stores quaternions, vss.py:118-121)."""
        return self._robot_words(4, 6)

    @property
    def robots_quats(self):
        cs = self.robots_rot
        yaw = torch.atan2(cs[..., 1], cs[..., 0])
        z = torch.zeros_like(yaw)
        return torch.stack([z, z, torch.sin(yaw / 2), torch.cos(yaw / 2)], -1)

    @property
    def robots_ang_vel(self):
        return self._robot_words(6, 7)

    @property
    def dof_velocity_buf(self):
        """(N,2,3,2) last commanded (clamped) wheel actions, zero after a reset (vss.py:137-141,184,333)."""
        return self._robot_words(7, 9)
