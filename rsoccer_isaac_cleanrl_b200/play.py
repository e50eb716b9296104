"""Team policies and the match runner — drop-in for the reference's `play.py`.

Same names and call conventions (reference play.py:26-164): a team is a callable
`team(act, obs)` that fills its slice `act (N,3,2)` of the `(N,2,3,2)` action buffer in place
from its own observations `obs (N,3,52)`; the yellow team receives the 180-degree mirrored
observations, so one policy plays either side. `play_matches` steps the raw `VSS` task (one fused
kernel launch per step).

Difference: the reference builds `BASELINE_TEAMS` from `base_nets/*/agent.pt` at import time;
those checkpoints are missing from the reference tree (`.MISSING_LARGE_BLOBS`), so here the table
is built lazily by `baseline_teams(base_dir)` and only lists the checkpoints that exist (plus
the parameter-free `zero` and `ou` teams).
"""
import argparse
import json
import os
import time
from abc import ABC, abstractmethod
from collections import namedtuple

import numpy as np
import torch

from . import _lib
from .envs.spaces import Box
from .envs.wrappers import random_ou
from .ppo import Agent


class Team(ABC):
    def __init__(self, path=None, env_d=None):
        pass

    @abstractmethod
    def __call__(self, act, obs):
        pass


class TeamZero(Team):
    def __call__(self, act, obs):
        act[:] *= 0


class TeamOU(Team):
    def __call__(self, act, obs):
        act[:] = random_ou(act)


class TeamAgent(Team):
    def __init__(self, path, env_d, device="cuda:0", mlp_backend="tc"):
        self.agent = Agent(env_d, mlp_backend=mlp_backend).to(device)
        self.agent.load_state_dict(torch.load(path, map_location=device))  # reference state_dict keys
        self.agent.eval()

    @classmethod
    def from_agent(cls, agent):
        """The team of an Agent already in memory (a self-play snapshot, for instance): no checkpoint is read."""
        team = cls.__new__(cls)
        team.agent = agent
        return team


class TeamSA(TeamAgent):
    """A single-agent policy drives robot 0; robots 1-2 follow OU noise (play.py:51-54)."""

    @torch.no_grad()
    def __call__(self, act, obs):
        act[:] = random_ou(act)
        act[:, 0, :] = self.agent.get_action_and_value(obs[:, 0, :].contiguous())[0]


class TeamCMA(TeamAgent):
    """One centralised 6-dim action for the three robots, from robot 0's view (play.py:57-59)."""

    @torch.no_grad()
    def __call__(self, act, obs):
        act[:] = self.agent.get_action_and_value(obs[:, 0, :].contiguous())[0].view(-1, 3, 2)


class TeamDMA(TeamAgent):
    """The same policy applied to each robot's own view (play.py:62-64)."""

    @torch.no_grad()
    def __call__(self, act, obs):
        n = obs.shape[0]
        act[:] = self.agent.get_action_and_value(obs.reshape(n * 3, -1))[0].view(n, 3, 2)


def get_team(algo, path=None, device="cuda:0", mlp_backend="tc"):
    dummy_env = namedtuple("dummy_env", ["single_observation_space", "single_action_space"])
    obs_space = Box(-np.inf, np.inf, (52,))
    if algo == "ppo-sa":
        return TeamSA(path, dummy_env(obs_space, Box(-1.0, 1.0, (2,))), device, mlp_backend)
    if algo in ("ppo-sa-x3", "ppo-dma"):
        return TeamDMA(path, dummy_env(obs_space, Box(-1.0, 1.0, (2,))), device, mlp_backend)
    if algo == "ppo-cma":
        return TeamCMA(path, dummy_env(obs_space, Box(-1.0, 1.0, (6,))), device, mlp_backend)
    if algo == "zero":
        return TeamZero()
    if algo == "ou":
        return TeamOU()
    raise ValueError(f"Unknown algo: {algo}")


def baseline_teams(base_dir="base_nets", device="cuda:0"):
    """The reference's BASELINE_TEAMS table (play.py:105-128), restricted to checkpoints that exist."""
    teams = {"zero": {"00": get_team("zero")}, "ou": {"00": get_team("ou")}}
    for algo, sub in (("ppo-sa", "ppo-sa"), ("ppo-sa-x3", "ppo-sa"), ("ppo-cma", "ppo-cma"), ("ppo-dma", "ppo-dma")):
        for seed in ("10", "20", "30"):
            path = os.path.join(base_dir, f"exp000_{sub}_{seed}", "agent.pt")
            if os.path.exists(path):
                teams.setdefault(algo, {})[seed] = get_team(algo, path, device)
    return teams


def play_matches(envs, blue_team, yellow_team, n_matches, video_path=None, count_envs=1065, video_fields=1):
    """Mean blue goal score and mean episode length over `n_matches` finished episodes
    (reference play.py:131-164). Only the first `count_envs` fields are counted, as the
    reference does (hard-coded 1065 there). With `video_path`, fields [0, video_fields) are rendered after every
    step (one mp4 frame per loop iteration, several fields as a mosaic; the state after the step: a field that
    ended an episode is shown already reset)."""
    writer = None
    if video_path:
        from .video import HEIGHT, WIDTH, VideoWriter
        writer = VideoWriter(video_path)
        frame = torch.empty((int(video_fields), HEIGHT, WIDTH, 3), dtype=torch.uint8, device=envs.device)
    envs.reset_buf[:] = 1
    envs.reset_dones()
    ep_count = 0
    rew_sum = 0.0
    len_sum = 0.0
    n = envs.cfg["env"]["numEnvs"]
    action_buf = torch.zeros((n,) + envs.action_space.shape, device=envs.device)
    obs = envs.reset()["obs"]
    count_envs = min(count_envs, n)
    while ep_count < n_matches:
        blue_team(action_buf[:, 0], obs[:, 0])
        yellow_team(action_buf[:, 1], obs[:, 1])
        obs, rew, dones, info = envs.step(action_buf)
        obs = obs["obs"]
        if writer is not None:
            writer.write_frames(envs.engine.render(0, video_fields, HEIGHT, WIDTH, out=frame)[None])
        env_ids = dones[:count_envs].nonzero(as_tuple=False).squeeze(-1)
        if len(env_ids):
            ep_count += len(env_ids)
            rew_sum += rew[env_ids, 0, 0, 0].sum().item()
            len_sum += info["progress_buffer"][env_ids].sum().item()
    if writer is not None:
        writer.close()
    return rew_sum / ep_count, len_sum / ep_count


# ---------------------------------------------------------------------------------------------------------------
# play_matches on the device: one vss_step_match launch per step (both teams' action prologue, the env step, the
# scoreboard) and one fused actor launch per policy team, captured in CUDA graphs of _CHUNK steps.
_CHUNK = 16  # steps per graph replay; the host reads the scoreboard once per replay
_POLICY_MODES = (_lib.TEAM_SA, _lib.TEAM_CMA, _lib.TEAM_DMA)


def _team_mode(team):
    """The device mode of a team object; any other callable (or a subclass with its own __call__) is EXTERNAL."""
    return {TeamZero: _lib.TEAM_ZERO, TeamOU: _lib.TEAM_OU, TeamSA: _lib.TEAM_SA, TeamCMA: _lib.TEAM_CMA,
            TeamDMA: _lib.TEAM_DMA}.get(type(team), _lib.TEAM_EXTERNAL)


def _team_seed(seed, side):
    """The Philox seed of a team's action sampling: distinct for the two sides of one match."""
    return ((int(seed) * 2 + side) * 0x9E3779B97F4A7C15 + 0x5EED) & (2 ** 64 - 1)


class _DevicePolicy:
    """One policy team on the device: bf16 actor weights (converted once), its sampling stream and its buffers."""

    def __init__(self, team, mode, side, obs_flat, n, seed):
        from .engine import gather_pad_bf16
        from .tc_mlp import MlpWeights
        agent = team.agent
        self.mw = MlpWeights(agent.actor_mean)
        assert self.mw.k0 == 64, self.mw.k0
        self.logstd = agent.actor_logstd.detach().reshape(-1).contiguous()
        dev = self.logstd.device
        robots = 3 if mode == _lib.TEAM_DMA else 1
        nv = n * robots
        # the team's rows of the observation: (field, team, robot) -> row 6 field + 3 team + robot of obs (N*6, 52)
        self._idx = (6 * torch.arange(n, device=dev)[:, None] + 3 * side + torch.arange(robots, device=dev)[None]).reshape(-1)
        self.rows = gather_pad_bf16(obs_flat, self._idx, 64)
        self.action = torch.zeros((nv, 6 if mode == _lib.TEAM_CMA else 2), device=dev, dtype=torch.float32)
        self.logprob = torch.empty(nv, device=dev, dtype=torch.float32)
        self.counter = torch.zeros(1, device=dev, dtype=torch.int32)
        self.seed = seed

    def load_rows(self, obs_flat):
        """Re-gathers the team's rows from a full (N*6, 52) observation (after a reset), into the same buffer."""
        from .engine import gather_pad_bf16
        self.rows.copy_(gather_pad_bf16(obs_flat, self._idx, 64))

    def launch(self, call_offset):
        from .engine import mlp_forward_fused
        mw = self.mw
        mlp_forward_fused(self.rows, [(mw.w16, mw.bs, mw.head_w, mw.head_b, False)],
                          sampling=dict(logstd=self.logstd, counter=self.counter, seed=self.seed,
                                        call_offset=call_offset, action=self.action, logprob=self.logprob))


def _run_matches_fused(envs, blue_team, yellow_team, n_matches, count_envs=1065, seed=0, graphs=True, video_path=None,
                       video_fields=1):
    """play_matches_fused with its scoreboard: dict(score, length, matches, steps, video_frames, buffers). `buffers`
    holds the final action buffer, the policy teams' last sampled actions and, with a video, the last chunk's device
    frames (K, F, H, W, 3). graphs=False runs every chunk eagerly: the same launches in the same order, which the
    tests compare the graph replays against. With `video_path` every chunk also renders fields [0, video_fields)
    after each step (inside the captured graph) and the host writes the chunk's frames after it: the video holds
    every executed step, the steps a chunk runs past the end of the evaluation included; video_frames counts them.
    Without a video the launches are exactly those of a run without the feature."""
    n = envs.num_fields
    dev = envs.device
    count_envs = min(int(count_envs), n)
    if n_matches < 1:
        raise ValueError("n_matches must be >= 1")
    teams = (blue_team, yellow_team)
    modes = [_team_mode(t) for t in teams]
    with torch.no_grad():
        envs.reset_buf[:] = 1  # as play_matches: re-randomise every field, then play
        envs.reset_dones()
        action_buf = torch.zeros((n,) + envs.action_space.shape, device=dev)
        board = torch.zeros(_lib.BOARD_WORDS, device=dev, dtype=torch.int64)
        obs_flat = envs.obs_buf.view(n * 6, -1)
        # distinct Philox seeds and counters per team: the two teams' noise is independent, also in self-play
        pol = [_DevicePolicy(t, m, side, obs_flat, n, _team_seed(seed, side))
               if m in _POLICY_MODES else None for side, (t, m) in enumerate(zip(teams, modes))]
        external = _lib.TEAM_EXTERNAL in modes
        obs = envs.obs_buf if external else None
        specs = [(m, None if p is None else p.action, None if p is None else p.rows) for m, p in zip(modes, pol)]
        side_stream = torch.cuda.Stream(device=dev)
        writer = frames = None
        if video_path:
            from .video import HEIGHT, WIDTH, VideoWriter
            writer = VideoWriter(video_path)
            frames = torch.zeros((_CHUNK, int(video_fields), HEIGHT, WIDTH, 3), dtype=torch.uint8, device=dev)
        shown = [0]  # frames of the last chunk (all _CHUNK except, on the EXTERNAL path, possibly the last)

        def render(k):
            if frames is not None:
                envs.engine.render(0, frames.shape[1], frames.shape[2], frames.shape[3], out=frames[k])

        def flush(k):
            if writer is not None and k:
                writer.write_frames(frames[:k])
                shown[0] = k

        def policies(call_offset):
            active = [p for p in pol if p is not None]
            if len(active) == 2:  # the two actors side by side (each fills a fraction of the SMs at 1 065 fields)
                # the stream current at call time: under graph capture that is the capture stream, and the fork /
                # join below records the side stream's launch into the graph
                main = torch.cuda.current_stream(dev)
                side_stream.wait_stream(main)
                with torch.cuda.stream(side_stream):
                    active[1].launch(call_offset)
                active[0].launch(call_offset)
                main.wait_stream(side_stream)
            elif active:
                active[0].launch(call_offset)

        def step(call_offset):
            policies(call_offset)
            envs.engine.step_match(specs, action_buf, envs.reset_buf, board, count_envs, n_matches, obs=obs)

        def frozen():
            return (int(board[4].item()) & 0xFFFFFFFF) != 0

        if external:  # EXTERNAL teams run eagerly on the step's f32 observation: no graph, one check per step
            k = 0
            while not frozen():
                for side, (t, m) in enumerate(zip(teams, modes)):
                    if m == _lib.TEAM_EXTERNAL:
                        t(action_buf[:, side], obs[:, side])
                step(0)
                for p in pol:
                    if p is not None:
                        p.counter.add_(1)
                render(k)
                k += 1
                if k == _CHUNK:
                    flush(k)
                    k = 0
            flush(k)
        else:
            def chunk():
                for k in range(_CHUNK):
                    step(k)
                    render(k)
                for p in pol:
                    if p is not None:
                        p.counter.add_(_CHUNK)

            chunk()  # eager first chunk (also the warm-up of everything the graph records)
            flush(_CHUNK)
            if not graphs:
                while not frozen():
                    chunk()
                    flush(_CHUNK)
            elif not frozen():
                torch.cuda.synchronize(dev)
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph):
                    chunk()
                while True:
                    graph.replay()
                    flush(_CHUNK)
                    if frozen():
                        break
        b = board.cpu()
        if writer is not None:
            writer.close()
    envs._obs_stale = True  # the step wrote neither obs_buf (unless EXTERNAL) nor the reward / terminal buffers
    matches = int(b[0])
    return dict(score=float(b[2:3].view(torch.float64)[0]) / matches, length=int(b[1]) / matches, matches=matches,
                steps=int(b[3]), video_frames=writer.frames if writer is not None else 0,
                buffers=dict(action_buf=action_buf, policy_action=[p and p.action for p in pol],
                             frames=None if frames is None else frames[:shown[0]]))


def play_matches_fused(envs, blue_team, yellow_team, n_matches, count_envs=1065, seed=0, video_path=None,
                       video_fields=1):
    """play_matches on the device: (mean blue goal score, mean episode length) over the first `n_matches`
    episodes that end among the first `count_envs` fields, exactly as play_matches defines them. TeamZero /
    TeamOU / TeamSA / TeamCMA / TeamDMA run inside the step (policy teams: the actor only, from bf16 copies of
    team.agent's weights, sampled in the same launch); any other team callable runs eagerly on the step's f32
    observation. The teams' OU noise comes from the engine's counter-based stream and the policy noise from a
    per-team Philox stream derived from `seed`, so results match play_matches in distribution, not draw for draw.
    With `video_path`, fields [0, video_fields) are rendered on the device after every executed step (inside the
    captured chunks; a frame is the state after its step) and written as an mp4 (see _run_matches_fused)."""
    r = _run_matches_fused(envs, blue_team, yellow_team, n_matches, count_envs, seed, video_path=video_path,
                           video_fields=video_fields)
    return r["score"], r["length"]


def parse_team(spec, device="cuda:0"):
    """'zero', 'ou' or 'ALGO:PATH' (ALGO = ppo-sa, ppo-sa-x3, ppo-cma, ppo-dma)."""
    algo, _, path = spec.partition(":")
    return get_team(algo, path or None, device)


def main(argv=None):
    """test.py without W&B: one checkpoint against a team or against every baseline team, one JSON line each."""
    ap = argparse.ArgumentParser(prog="python -m rsoccer_isaac_cleanrl_b200.play")
    ap.add_argument("--blue", required=True, help="ALGO:PATH of the evaluated team (or zero / ou)")
    ap.add_argument("--yellow", default=None, help="the opponent's team spec; default: every baseline team")
    ap.add_argument("--base-dir", default="base_nets", help="baseline checkpoints (play.baseline_teams)")
    ap.add_argument("--num-envs", type=int, default=1065)
    ap.add_argument("--matches", type=int, default=10000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--eager", action="store_true", help="run play_matches (the reference loop) instead")
    ap.add_argument("--video", default=None, metavar="DIR",
                    help="write one mp4 per opponent, DIR/<blue>_vs_<yellow>.mp4, of every step of fields [0, F)")
    ap.add_argument("--video-fields", type=int, default=1, metavar="F", help="fields per video frame (a mosaic)")
    args = ap.parse_args(argv)
    from .envs import VSS, load_cfg
    cfg = load_cfg()
    cfg["env"]["numEnvs"] = args.num_envs
    torch.manual_seed(args.seed)
    envs = VSS(cfg, "cuda:0", "cuda:0", 0, True, seed=args.seed)
    envs.w_goal, envs.w_grad, envs.w_move, envs.w_energy = 1.0, 0.0, 0.0, 0.0  # ppo…:389-392, test.py:45-48
    blue = parse_team(args.blue)
    if args.yellow:
        opponents = {args.yellow: parse_team(args.yellow)}
    else:
        opponents = {f"{algo}/{s}": t for algo, by_seed in baseline_teams(args.base_dir).items()
                     for s, t in by_seed.items()}
    for name, yellow in opponents.items():
        video = None
        if args.video:
            from .video import safe_name
            video = os.path.join(args.video, f"{safe_name(args.blue)}_vs_{safe_name(name)}.mp4")
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if args.eager:
            steps = [0]

            def counted(act, obs, team=blue):
                steps[0] += 1
                team(act, obs)
            score, length = play_matches(envs, counted, yellow, args.matches, count_envs=args.num_envs,
                                         video_path=video, video_fields=args.video_fields)
            r = dict(score=score, length=length, matches=args.matches, steps=steps[0])
        else:
            f = _run_matches_fused(envs, blue, yellow, args.matches, count_envs=args.num_envs, seed=args.seed,
                                   video_path=video, video_fields=args.video_fields)
            r = dict(score=f["score"], length=f["length"], matches=args.matches, steps=f["steps"],
                     counted_matches=f["matches"])  # (the step that reaches the count adds all its episodes)
        torch.cuda.synchronize()
        r["seconds"] = time.perf_counter() - t0
        if video:
            r["video"] = video
        print(json.dumps(dict(blue=args.blue, yellow=name, path="eager" if args.eager else "fused", **r)), flush=True)


if __name__ == "__main__":
    main()
