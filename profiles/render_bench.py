"""Field rendering on the B200: vss_render per launch, match videos and recording PPO updates.

1. `vss_render` at 560 x 720 and F = 1 / 16 / 64 / 256 fields per launch: device events around `--launches`
   back-to-back launches after a warm-up, µs per launch; bytes written F * H * W * 3 over that time as GB/s, and as
   a share of the project's HBM roofline (`hbm_gbs` of MEASURED_PEAKS.json when the box has one, else the 6 650 GB/s
   fallback bench.py uses; the kernel reads 104 B of state per frame, which is left out). At F = 1 and 16 the
   output (1.2 / 19 MB) stays in the 126 MB L2 from launch to launch; at 64 and 256 (77 / 310 MB) it does not.
2. `play_matches_fused` at 1 065 fields, sa-vs-ou (a freshly initialised actor: the timing does not depend on the
   weights), without a video, with F = 1 and with F = 4 fields per frame: the three alternate `--reps` times in one
   process after a warm-up run each; host clock around each run (ends in a synchronise), µs per executed step,
   median over the reps. The host time inside the video writer (device-to-host copy, mosaic, RGB->BGR, mp4v
   encode) is reported separately.
3. ppo-sa, 4 096 agents, T = 128: the rollout time (host clock around the rollout + synchronise) of recording and of
   plain updates, `--record-video-step-frequency 2T` so updates alternate; updates 1-3 (eager, the two captures)
   are left out, median of the rest of each kind.

The GPU name and power limit are read in the same run and written beside the numbers.

    python profiles/render_bench.py [--launches 200] [--reps 5] [--matches 2000] [--out profiles/render_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from collections import namedtuple

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

H, W = 560, 720


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(0), nvidia_smi=q.stdout.strip())


def hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback 6650 GB/s (bench.py)"


def bench_kernel(launches):
    import rsoccer_isaac_cleanrl_b200 as R
    n = 4096
    eng = R.Engine(n, "cuda:0", seed=0)
    eng.reset_dones(torch.ones(n, dtype=torch.int64, device="cuda"), torch.zeros((n, 2, 3, 52), device="cuda"))
    peak, src = hbm_peak()
    rows = []
    for f in (1, 16, 64, 256):
        out = torch.empty((f, H, W, 3), dtype=torch.uint8, device="cuda")
        for _ in range(20):
            eng.render(0, f, out=out)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(launches):
            eng.render(0, f, out=out)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / launches
        nbytes = f * H * W * 3
        gbs = nbytes / (us * 1e-6) / 1e9
        rows.append(dict(fields=f, height=H, width=W, launches=launches, us_per_launch=us, bytes_written=nbytes,
                         gb_per_s=gbs, hbm_roofline_gbs=peak, roofline_source=src, frac_of_roofline=gbs / peak,
                         output_fits_l2=nbytes < 126e6))
        print(json.dumps(rows[-1]), flush=True)
    eng.close()
    return rows


def bench_matches(reps, matches, tmp):
    from rsoccer_isaac_cleanrl_b200 import play, video
    from rsoccer_isaac_cleanrl_b200.envs import VSS, load_cfg
    from rsoccer_isaac_cleanrl_b200.envs.spaces import Box
    from rsoccer_isaac_cleanrl_b200.ppo import Agent
    cfg = load_cfg()
    cfg["env"]["numEnvs"] = 1065
    envs = VSS(cfg, "cuda:0", "cuda:0", 0, True, seed=0)
    envs.w_goal, envs.w_grad, envs.w_move, envs.w_energy = 1.0, 0.0, 0.0, 0.0
    d = namedtuple("d", ["single_observation_space", "single_action_space"])
    sa = play.TeamSA.__new__(play.TeamSA)
    torch.manual_seed(0)
    sa.agent = Agent(d(Box(-np.inf, np.inf, (52,)), Box(-1.0, 1.0, (2,))), mlp_backend="tc").cuda().eval()
    ou = play.TeamOU()

    encode = [0.0]
    write_frames = video.VideoWriter.write_frames

    def timed_write(self, frames):
        t0 = time.perf_counter()
        write_frames(self, frames)
        encode[0] += time.perf_counter() - t0
    video.VideoWriter.write_frames = timed_write

    def run(fields):
        encode[0] = 0.0
        path = os.path.join(tmp, f"m{fields}.mp4") if fields else None
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = play._run_matches_fused(envs, sa, ou, matches, seed=1, video_path=path, video_fields=max(fields, 1))
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        executed = r["video_frames"] if fields else -(-r["steps"] // play._CHUNK) * play._CHUNK
        return dict(video_fields=fields, seconds=dt, board_steps=r["steps"], executed_steps=executed,
                    us_per_step=1e6 * dt / executed, writer_host_s=encode[0],
                    writer_host_us_per_frame=1e6 * encode[0] / executed if fields else 0.0)

    for f in (0, 1, 4):
        run(f)  # warm-up (graph capture, cv2 import, codec start-up)
    runs = []
    for rep in range(reps):
        for f in (0, 1, 4):
            runs.append(dict(rep=rep, **run(f)))
            print(json.dumps(runs[-1]), flush=True)
    video.VideoWriter.write_frames = write_frames
    envs.close()
    summary = {}
    for f in (0, 1, 4):
        rs = [r for r in runs if r["video_fields"] == f]
        summary[f"fields_{f}" if f else "no_video"] = dict(
            median_us_per_step=statistics.median(r["us_per_step"] for r in rs),
            median_writer_host_us_per_frame=statistics.median(r["writer_host_us_per_frame"] for r in rs))
    return dict(workload=f"sa-vs-ou, 1065 fields, {matches} matches, fresh tc actor", runs=runs, summary=summary)


def bench_ppo(tmp):
    from rsoccer_isaac_cleanrl_b200 import ppo
    T, N, updates = 128, 4096, 9
    args = ppo.parse_args(["--env-id", "sa", "--num-envs", str(N), "--num-steps", str(T), "--total-timesteps",
                           str(N * T * updates), "--quiet", "--tensorboard", "false", "--capture-video",
                           "--record-video-step-frequency", str(2 * T), "--save-path", tmp])
    recorded = {}
    st = ppo.train(args, hook=lambda u, d: recorded.__setitem__(u, d["frames"] is not None))
    rows = [dict(update=u, recording=recorded[u], rollout_ms=1e3 * st["rollout_wall"][u - 1]) for u in range(1, updates + 1)]
    later = [r for r in rows if r["update"] >= 4]
    return dict(workload=f"ppo-sa, {N} agents, T={T}, tc backend, 1 field per frame", updates=rows,
                median_rollout_ms_recording=statistics.median(r["rollout_ms"] for r in later if r["recording"]),
                median_rollout_ms_plain=statistics.median(r["rollout_ms"] for r in later if not r["recording"]),
                videos=len(st["videos"]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--matches", type=int, default=2000)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "render_bench needs the GPU"
    res = dict(gpu=gpu_info())
    with tempfile.TemporaryDirectory() as tmp:  # the videos are written and thrown away
        res["vss_render"] = bench_kernel(args.launches)
        res["play_matches_fused"] = bench_matches(args.reps, args.matches, tmp)
        res["ppo_rollout"] = bench_ppo(tmp)
    res["gpu_after"] = gpu_info()
    s = json.dumps(res, indent=1)
    print(s)
    if args.out:
        with open(args.out, "w") as f:
            f.write(s + "\n")


if __name__ == "__main__":
    main()
