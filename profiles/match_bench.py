"""Match evaluation on the B200: the eager play_matches loop against play_matches_fused (one vss_step_match launch
plus one fused actor launch per policy team per step, CUDA graphs of play._CHUNK steps).

Workloads: zero-vs-ou, sa-vs-ou and cma-vs-dma at 1 065 fields (the reference's evaluation size, count_envs 1065),
and the fused path at 16 384 fields with count_envs = N. The policies are freshly initialised Agents (the timing does
not depend on the weights). Each workload runs warm-up matches first, then old and new alternate `--reps` times in
the same process; a time is the host clock around a run that ends in a device synchronise. Reported per run: µs per
env step and matches per second. The GPU name and power limit are read in the same call and written beside them.

    python profiles/match_bench.py [--matches 10000] [--reps 3] [--out profiles/match_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import namedtuple

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--matches", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "match_bench needs the GPU"
    from rsoccer_isaac_cleanrl_b200 import play
    from rsoccer_isaac_cleanrl_b200.envs import VSS, load_cfg
    from rsoccer_isaac_cleanrl_b200.envs.spaces import Box
    from rsoccer_isaac_cleanrl_b200.ppo import Agent

    def envs_of(n):
        cfg = load_cfg()
        cfg["env"]["numEnvs"] = n
        e = VSS(cfg, "cuda:0", "cuda:0", 0, True, seed=0)
        e.w_goal, e.w_grad, e.w_move, e.w_energy = 1.0, 0.0, 0.0, 0.0
        return e

    def agent_team(cls, adim):
        d = namedtuple("d", ["single_observation_space", "single_action_space"])
        t = cls.__new__(cls)
        torch.manual_seed(0)
        t.agent = Agent(d(Box(-np.inf, np.inf, (52,)), Box(-1.0, 1.0, (adim,))), mlp_backend="tc").cuda().eval()
        return t

    teams = {"zero": play.TeamZero(), "ou": play.TeamOU(), "sa": agent_team(play.TeamSA, 2),
             "cma": agent_team(play.TeamCMA, 6), "dma": agent_team(play.TeamDMA, 2)}

    def run(path, envs, blue, yellow, matches, count_envs):
        steps = [0]

        def counted(act, obs):
            steps[0] += 1
            blue(act, obs)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        if path == "eager":
            score, length = play.play_matches(envs, counted, yellow, matches, count_envs=count_envs)
            n_steps, counted_matches = steps[0], None
        else:
            r = play._run_matches_fused(envs, blue, yellow, matches, count_envs=count_envs)
            score, length, n_steps, counted_matches = r["score"], r["length"], r["steps"], r["matches"]
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        return dict(path=path, seconds=dt, steps=n_steps, us_per_step=1e6 * dt / n_steps, matches_per_s=matches / dt,
                    score=score, length=length, counted_matches=counted_matches)

    results = dict(gpu=gpu_info(), matches=args.matches, reps=args.reps, runs=[])
    work = [("zero", "ou", 1065, ("eager", "fused")), ("sa", "ou", 1065, ("eager", "fused")),
            ("cma", "dma", 1065, ("eager", "fused")), ("sa", "ou", 16384, ("fused",))]
    for blue, yellow, n, paths in work:
        envs = envs_of(n)
        for path in paths:  # warm-up: module loads, graph capture, allocator
            run(path, envs, teams[blue], teams[yellow], 500, n)
        for rep in range(args.reps):
            for path in paths:  # old and new alternate
                r = run(path, envs, teams[blue], teams[yellow], args.matches, n)
                r.update(blue=blue, yellow=yellow, num_envs=n, rep=rep)
                results["runs"].append(r)
                print(json.dumps(r), flush=True)
        envs.close()
    summary = {}
    for r in results["runs"]:
        k = f"{r['blue']}-vs-{r['yellow']}@{r['num_envs']}/{r['path']}"
        summary.setdefault(k, []).append(r["us_per_step"])
    results["median_us_per_step"] = {k: float(np.median(v)) for k, v in summary.items()}
    print(json.dumps(results["median_us_per_step"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
