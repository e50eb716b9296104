"""PPO against opponents on the B200: rollout time and steady PPO SPS per opponent.

Workloads: sa at 4 096 agents, cma at 16 384 and dma at 65 535 (bench.py's PPO legs), each with the opponents
  ou          OU noise in the yellow slots (the reference's view, today's kernel)
  zero        TeamZero (the opponent variant of the view kernel, no actor)
  checkpoint  a same-algorithm checkpoint (ppo-sa / ppo-cma / ppo-dma): one fused actor launch per step on its own
              stream beside the learner's forward
  self        a frozen snapshot of the learner (the same launches; the snapshot is refreshed every 10 updates)
The checkpoints are freshly initialised Agents (the timing does not depend on the weights). Each run is ppo.train
with the default hyperparameters for --updates updates; the first two (eager, then graph capture) are warm-up.
Reported per run: the median rollout time of the remaining updates (128 steps, the host clock around a replay that
ends in a device synchronise) and steady SPS = agents x steps / (rollout + update) of those updates. The
configurations alternate in one process, --reps times; the summary is the median over the reps. The GPU name and
power limit are read in the same call and written beside the numbers.

    python profiles/opponent_bench.py [--reps 5] [--updates 5] [--out profiles/opponent_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
from collections import namedtuple

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

LEGS = (("sa", 4096), ("cma", 16384), ("dma", 65535))
OPPONENTS = ("ou", "zero", "checkpoint", "self")


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--updates", type=int, default=5)
    ap.add_argument("--steps", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "opponent_bench needs the GPU"
    from rsoccer_isaac_cleanrl_b200 import ppo
    from rsoccer_isaac_cleanrl_b200.envs.spaces import Box

    tmp = tempfile.mkdtemp(prefix="opponent_bench_")
    ckpt = {}
    for env_id, adim in (("sa", 2), ("cma", 6), ("dma", 2)):
        d = namedtuple("d", ["single_observation_space", "single_action_space"])
        torch.manual_seed(0)
        agent = ppo.Agent(d(Box(-np.inf, np.inf, (52,)), Box(-1.0, 1.0, (adim,))))
        ckpt[env_id] = os.path.join(tmp, f"{env_id}.pt")
        torch.save(agent.state_dict(), ckpt[env_id])

    def run(env_id, n, opponent):
        spec = f"ppo-{env_id}:{ckpt[env_id]}" if opponent == "checkpoint" else opponent
        a = ppo.parse_args(["--env-id", env_id, "--num-envs", str(n), "--num-steps", str(args.steps),
                            "--total-timesteps", str(n * args.steps * args.updates), "--opponent", spec,
                            "--quiet", "--tensorboard", "false"])
        st = ppo.train(a)
        roll, upd = np.array(st["rollout_wall"][2:]), np.array(st["update_wall"][2:])
        r = dict(env_id=env_id, num_envs=n, opponent=opponent, rollout_ms=1e3 * float(np.median(roll)),
                 steady_sps=float(np.median(n * args.steps / (roll + upd))), rollout_ms_all=(1e3 * roll).tolist())
        del st
        torch.cuda.empty_cache()
        return r

    results = dict(gpu=gpu_info(), steps=args.steps, updates=args.updates, reps=args.reps, runs=[])
    for rep in range(args.reps):
        for env_id, n in LEGS:
            for opponent in OPPONENTS:  # the opponents alternate
                r = run(env_id, n, opponent)
                r["rep"] = rep
                results["runs"].append(r)
                print(json.dumps(r), flush=True)
    summary = {}
    for r in results["runs"]:
        k = f"{r['env_id']}@{r['num_envs']}/{r['opponent']}"
        summary.setdefault(k, {"rollout_ms": [], "steady_sps": []})
        summary[k]["rollout_ms"].append(r["rollout_ms"])
        summary[k]["steady_sps"].append(r["steady_sps"])
    results["median"] = {k: {m: float(np.median(v)) for m, v in d.items()} for k, d in summary.items()}
    print(json.dumps(results["median"]), flush=True)
    if args.out:
        with open(args.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
