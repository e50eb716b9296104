#!/usr/bin/env python
"""bench.py — VSS env-steps/s (and PPO SPS) on N B200s, with roofline, CPU baseline and e2e.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--envs E_PER_GPU] [--impl native|reference] [--dump-outputs DIR]
  torchrun --nproc-per-node N bench.py --gpus N ...        (one rank per GPU, NCCL only for timing / PPO grads)

A "step" is one pass of the hot path over one batch: one fused `vss_step` launch advancing E
fields per GPU by one control step (full VSS.step contract: obs + terminal obs + rewards + dones
+ masked reset). Fields shard across GPUs with no data-path collective (weak scaling).
Prints ONE JSON line on rank 0.

Legs of the native arm (all in the one line):
  value / roofline   K timed `VSS.step` launches at E fields per GPU, inputs resident in HBM (+ a 400-step
                     "sustained" region when K < 200)
  e2e                `SingleAgent.step_host`: pinned host action in, packed host rows out, every step
                     (+ the f32 variant, + the full VSS.step contract with host buffers)
  cpu_baseline       the oracle's view step on the host cores, same view and field count as e2e (N = 1 only)
  sweep              1K … 1M fields per GPU (BASELINE configs[4])
  gae                the reverse-scan kernel at T = 128
  ppo                ppo-sa 4096 / ppo-cma 16384 / ppo-dma 65535 agents per GPU (BASELINE configs[1-3])
  reference_torch    what the reference itself runs on the GPU, restated in torch (oracle/torch_ref.py):
                     obs/rewards/dones op sequence, the python GAE loop, the fp32 autograd minibatch (N = 1 only)
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic HBM bytes of one field-step of the full VSS.step contract (DESIGN.md §4.1):
# state 240 in + 240 out, actions 48, reset flags 8 in + 8 out, obs 1248, terminal obs 1248,
# rewards 96, timeout 1, progress 4
BYTES_PER_FIELD_STEP = 240 + 240 + 48 + 8 + 8 + 1248 + 1248 + 96 + 1 + 4
# host bytes of the full contract per field-step: actions in; obs, terminal obs, rewards, reset, timeout, progress out
FULL_H2D, FULL_D2H = 48, 1248 + 1248 + 96 + 8 + 1 + 4
# fields sampled by --dump-outputs: 2.6 KB of outputs per field keeps a dump near 43 MB
DUMP_FIELDS = 16384


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=400)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--envs", type=int, default=1 << 20, help="fields per GPU")
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-ppo", action="store_true")
    ap.add_argument("--skip-reference-torch", action="store_true")
    ap.add_argument("--no-sweep", action="store_true", help="skip the N in {1K..1M} sweep (BASELINE configs[4])")
    ap.add_argument("--ppo-legs", default="sa:4096,cma:16384,dma:65535",
                    help="env-id:agents-per-GPU of the PPO legs (BASELINE configs[1-3])")
    ap.add_argument("--ppo-updates", type=int, default=0,
                    help="updates per PPO leg (1 eager + 1 capturing + steady); 0 = about 2e7 samples per GPU and leg, "
                         "at least 8 and at most 40 updates, so that the reference's own SPS metric (global_step / wall, "
                         "start-up included) is not dominated by the two start-up updates")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed VSS.step returned as DIR/<name>.npy "
                         f"(float32 / float64; the same {DUMP_FIELDS} sampled fields in every run, all fields when "
                         "there are fewer; rank 0's fields)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "native":
        ap.error("--dump-outputs dumps the native arm's outputs: use it with --impl native")
    return args


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock and throttle reasons sampled through NVML every 5 ms from a thread of this process (the
    `nvidia-smi -lms` poller cannot go below ~50 ms and missed short timed regions altogether)."""

    def __init__(self, index, period=0.005):
        self.index, self.period = index, period
        self.samples, self.reasons, self.mx = [], set(), None
        self._stop = threading.Event()
        self.thread = None
        self.error = None

    def start(self):
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            p = torch.cuda.get_device_properties(self.index)
            bus = f"{p.pci_domain_id:08x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
            self.h = pynvml.nvmlDeviceGetHandleByPciBusId(bus.encode())
            self.nv = pynvml
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()
        except Exception as e:
            self.error = f"{type(e).__name__}: {e}"

    def _run(self):
        nv = self.nv
        bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception as e:
                self.error = f"{type(e).__name__}: {e}"
                return
            self._stop.wait(self.period)

    def mark(self):
        """Forget what was sampled so far (called right before the timed region starts)."""
        self.samples, self.reasons = [], set()

    def stop(self):
        self._stop.set()
        if self.thread is not None:
            self.thread.join(timeout=1)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.mx, "samples": 0, "reasons": [self.error or "no samples"]}
        sm = sorted(self.samples)
        return {"sm_mhz": sm[len(sm) // 2], "sm_min_mhz": sm[0], "sm_max_mhz": self.mx, "samples": len(sm),
                "reasons": sorted(self.reasons), "how": "NVML, 5 ms period, timed region only"}


# ----------------------------------------------------------------------------- CPU arm (oracle)
def cpu_oracle_run(n_envs, seconds=None, steps=None, warmup=1, contract="sa_view"):
    """Times the oracle (CPU restatement, all host threads that help) on a bounded sample.
    contract "sa_view": SingleAgent.step — OU opponents, env step, view slicing (what the native e2e arm
    delivers); "full": the raw VSS.step contract (what the native device-timed `value` runs)."""
    import numpy as np
    from oracle import vss_oracle as orc
    p = orc.default_params()
    st = orc.State(n_envs)
    rb = np.ones(n_envs, np.int64)
    orc.reset_dones(p, 0, 0, st, rb)
    rb[:] = 0
    rng = np.random.default_rng(0)
    st.progress[:] = rng.integers(0, 400, n_envs)
    if contract == "full":
        acts = [rng.uniform(-1, 1, (n_envs, 2, 3, 2)).astype(np.float32) for _ in range(2)]
        bufs = orc.step(p, 0, 0, st, acts[0], rb)   # persistent output buffers, as the reference's obs_buf / rew_buf
        fn = lambda i: orc.step(p, 0, 0, st, acts[i & 1], rb, out=bufs)
    else:
        acts = [rng.uniform(-1, 1, (n_envs, 2)).astype(np.float32) for _ in range(2)]
        abuf = np.zeros((n_envs, 2, 3, 2), np.float32)
        bufs = orc.step_view(p, 0, 0, 0, st, orc.VIEW_SA, acts[0], abuf, rb)
        fn = lambda i: orc.step_view(p, 0, 0, i, st, orc.VIEW_SA, acts[i & 1], abuf, rb, out=bufs)
    # use as many host threads as actually help (containers often expose more cpus than their quota)
    best = (None, 1)
    for nt in sorted({1, max(1, (os.cpu_count() or 1) // 2), os.cpu_count() or 1}):
        orc.set_num_threads(nt)
        fn(0)
        t0 = time.perf_counter()
        fn(1)
        dt = time.perf_counter() - t0
        if best[0] is None or dt < best[0]:
            best = (dt, nt)
    orc.set_num_threads(best[1])
    for i in range(warmup):
        fn(i)
    t0 = time.perf_counter()
    k = 0
    while True:
        fn(k)
        k += 1
        el = time.perf_counter() - t0
        if (steps is not None and k >= steps) or (steps is None and el >= seconds and k >= 3):
            break
    what = "SingleAgent.step (OU opponents + env step + view slicing)" if contract != "full" else "VSS.step (full contract)"
    return {"value": n_envs * k / el, "unit": "env-steps/s", "cores": orc.num_threads(), "kind": "port",
            "sample": f"{k} oracle {what} calls over {n_envs} fields ({el:.1f} s, OpenMP over fields, "
                      f"{os.cpu_count()} host cpus); CPU restatement incl. the new 2-D physics, NOT PhysX"}, el / k


def run_reference(args):
    """The reference arm: the reference's CPU PhysX pipeline cannot run (IsaacGym is absent), so this times
    the oracle port on the host cores — the SAME workload as the native arm's e2e (SingleAgent view, the same
    field count), every step a full pass over all the fields."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.envs
    # a CPU step over 2^20 fields takes ~0.15 s: bound the run to a few minutes whatever K the driver asks for
    k = max(1, min(args.steps, 200))
    w = max(1, min(args.warmup, 10))
    cb, sec_per_step = cpu_oracle_run(n, steps=k, warmup=w, contract="sa_view")
    full, sec_full = cpu_oracle_run(n, steps=max(3, k // 4), warmup=1, contract="full")
    line = {
        "impl": "reference", "metric": "vss_env_steps_per_s", "value": cb["value"], "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": k, "warmup": w, "ms_per_step": sec_per_step * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"random-action VSS 3v3 env step through the SingleAgent view, {n} fields per step on "
                               "the host cores (the native arm's e2e workload: same view, same field count)",
                   "envs_per_gpu": n,
                   "note": "the reference's own CPU PhysX pipeline cannot run (IsaacGym absent); this is the "
                           "oracle port: reference obs/reward/reset/view semantics + the new 2-D physics"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "full_contract": {"value": full["value"], "unit": "env-steps/s", "ms_per_step": sec_full * 1e3,
                          "sample": full["sample"]},
        "gpu_launches": 0,
    }
    emit(line)


# ----------------------------------------------------------------------------- native arm
def time_steps(torch, dist, world, fn, steps, warmup, on_start=None):
    for i in range(warmup):
        fn(i)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if on_start is not None:
        on_start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = float(t.item())
    return ms


def make_task(torch, n, rank, local, seed=0):
    """The public task object (drop-in VSS) with progress counters staggered to steady state."""
    from rsoccer_isaac_cleanrl_b200.envs import VSS, load_cfg
    cfg = load_cfg()
    cfg["env"]["numEnvs"] = n
    dev = f"cuda:{local}"
    envs = VSS(cfg, dev, dev, 0, True, seed=seed, global_env_offset=rank * n)
    envs.reset_buf.zero_()
    st = envs.engine.get_state()
    g = torch.Generator(device=dev); g.manual_seed(1234 + rank)
    st[58, :n] = torch.randint(0, 400, (n,), device=dev, generator=g, dtype=torch.int32).view(torch.float32)
    envs.engine.set_state(st)
    del st
    acts = [torch.rand((n, 2, 3, 2), device=dev, generator=g) * 2 - 1 for _ in range(4)]
    return envs, acts


def full_contract_host_step(torch, envs, local):
    """`VSS.step` with HOST buffers: pinned (N,2,3,2) actions in; obs, terminal obs, rewards, reset, time-outs
    and progress out to pinned host memory, every step."""
    from rsoccer_isaac_cleanrl_b200.hostmem import pinned_empty
    n, dev = envs.num_fields, f"cuda:{local}"
    act_h = torch.rand((n, 2, 3, 2)).mul_(2).sub_(1).pin_memory()
    act_d = torch.empty((n, 2, 3, 2), device=dev)
    outs = []

    def step(i):
        act_d.copy_(act_h, non_blocking=True)
        obs, rew, reset, extras = envs.step(act_d)
        src = (obs["obs"], extras["terminal_observation"], rew, reset, extras["time_outs"], extras["progress_buffer"])
        if not outs:
            outs.extend(pinned_empty(tuple(t.shape), t.dtype, dev) for t in src)
        for h, d in zip(outs, src):
            h.copy_(d, non_blocking=True)
        torch.cuda.current_stream().synchronize()
    return step


def dump_outputs(torch, out_dir, step_out):
    """Writes what one `VSS.step` returned, `(obs_dict, rew, reset, extras)`, as out_dir/<name>.npy: floats as
    float32, the int64 reset flags as float64 (exact), the bool time-outs as float32 0 / 1. Fields beyond
    DUMP_FIELDS are sampled with a fixed seed, so two runs with the same arguments dump the same fields."""
    import numpy as np
    obs, rew, reset, extras = step_out
    arrays = {"obs": obs["obs"], "rew": rew, "reset": reset, "terminal_observation": extras["terminal_observation"],
              "time_outs": extras["time_outs"], "progress_buffer": extras["progress_buffer"]}
    n = reset.shape[0]
    rows = None
    if n > DUMP_FIELDS:
        rows = np.sort(np.random.default_rng(0).choice(n, DUMP_FIELDS, replace=False))
        rows = torch.from_numpy(rows).to(reset.device)
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        a = (t if rows is None else t.index_select(0, rows)).cpu().numpy()
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64 if a.dtype == np.int64 else np.float32))


def reference_torch_legs(torch, peak):
    """BASELINE.md B2-B4: the reference's own torch code paths (restated, oracle/torch_ref.py) on this GPU."""
    import types

    import numpy as np

    from oracle import torch_ref as tr
    from rsoccer_isaac_cleanrl_b200 import ppo as ppo_mod
    from rsoccer_isaac_cleanrl_b200.engine import gae as gae_kernel
    from rsoccer_isaac_cleanrl_b200.envs.spaces import Box
    dev = "cuda"
    out = {"note": "torch restatements of the reference's GPU code, pinned to the golden vectors in "
                   "tests/test_torch_ref_golden.py; eager torch on the same B200, CUDA-event timed"}

    def timeit(fn, reps, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / reps   # us

    # B2: obs x2 + rewards + dones (vss.py:189-265, :530-655) — excludes PhysX, the masked reset and the wrappers
    b2 = []
    for n in (4096, 65536):
        g = torch.Generator(device=dev); g.manual_seed(n)
        r = lambda *s: torch.rand(s, device=dev, generator=g) * 2 - 1
        yaw = r(n, 2, 3) * 3.14159
        quats = torch.stack([torch.zeros_like(yaw), torch.zeros_like(yaw), torch.sin(yaw / 2), torch.cos(yaw / 2)], -1)
        s = dict(ball_pos=r(n, 2) * 0.7, ball_vel=r(n, 2), prev_ball_pos=r(n, 2) * 0.7, r_pos=r(n, 2, 3, 2) * 0.6,
                 prev_r_pos=r(n, 2, 3, 2) * 0.6, r_vel=r(n, 2, 3, 2), quats=quats, r_w=r(n, 2, 3, 1), acts=r(n, 2, 3, 2),
                 reset_buf=torch.zeros(n, dtype=torch.long, device=dev),
                 progress=torch.randint(0, 400, (n,), device=dev, generator=g))
        us = timeit(lambda: tr.obs_rewards_dones(s), 30)
        b2.append({"fields": n, "us_per_step": us, "field_steps_per_s": n / (us * 1e-6)})
    out["obs_rewards_dones_torch"] = b2
    # B3: the python GAE loop vs vss_gae on the same tensors
    b3 = []
    for T, N in ((128, 4096), (128, 65536)):
        a = [torch.randn((T, N), device=dev) for _ in range(3)]
        d = (torch.rand((T, N), device=dev) < 0.01).float()
        to = d * (torch.rand((T, N), device=dev) < 0.5).float()
        us_ref = timeit(lambda: tr.gae_loop(*a, d, to), 5, 2)
        adv, ret = torch.empty_like(d), torch.empty_like(d)
        us_k = timeit(lambda: gae_kernel(*a, d, to, 0.99, 0.95, adv, ret), 50, 5)
        ra, _ = tr.gae_loop(*a, d, to)
        b3.append({"T": T, "N": N, "torch_loop_us": us_ref, "vss_gae_us": us_k, "speedup": us_ref / us_k,
                   "max_abs_diff": float((ra - adv).abs().max())})
    out["gae_loop_torch"] = b3
    # B4: one fp32 autograd minibatch (ppo…:314-354) at the default minibatch of 4096 x 128 / 4 rows
    B, R = 131072, 524288
    envs_d = types.SimpleNamespace(single_observation_space=Box(-np.inf, np.inf, (52,)),
                                   single_action_space=Box(-1.0, 1.0, (2,)))
    args = ppo_mod.parse_args(["--num-envs", "4096", "--quiet"])
    b4 = {}
    for name, tf32 in (("fp32", False), ("tf32", True)):
        torch.backends.cuda.matmul.allow_tf32 = tf32
        torch.manual_seed(0)
        agent = ppo_mod.Agent(envs_d, mlp_backend="torch").to(dev)
        opt = torch.optim.Adam(agent.parameters(), lr=1e-3, eps=1e-5)
        batch = dict(b_obs=torch.randn(R, 52, device=dev), b_actions=torch.randn(R, 2, device=dev),
                     b_logprobs=torch.randn(R, device=dev) * 0.1 - 2.0, b_advantages=torch.randn(R, device=dev),
                     b_returns=torch.randn(R, device=dev), b_values=torch.randn(R, device=dev))
        inds = torch.randperm(R, device=dev)[:B]
        us = timeit(lambda: tr.agent_update(agent, opt, args, batch, inds), 10, 3)
        b4[name] = {"us_per_minibatch": us, "samples_per_s_update_phase": B / (us * 1e-6) / 8,
                    "tflops": 3 * 2 * 1.076e6 * B / (us * 1e-6) / 1e12}
        del agent, opt, batch
    torch.backends.cuda.matmul.allow_tf32 = False
    b4["note"] = ("minibatch of 131072 rows, torch autograd + clip_grad_norm_ + torch.optim.Adam; tflops = 3 x forward "
                  "FLOPs of both MLPs; samples_per_s_update_phase divides by the 8 epochs every sample is visited")
    out["agent_update_torch"] = b4
    torch.cuda.empty_cache()
    return out


def run_ppo_leg(torch, world, env_id, agents, updates):
    from rsoccer_isaac_cleanrl_b200 import ppo as ppo_mod
    torch.cuda.empty_cache()
    pa_ = ppo_mod.parse_args(["--env-id", env_id, "--num-envs", str(agents), "--quiet",
                              "--total-timesteps", str(agents * 128 * world * updates)])
    st = ppo_mod.train(pa_)
    # steady state: updates after the eager first one and the graph-capturing second one
    tail_r, tail_u = st["rollout_wall"][2:] or st["rollout_wall"], st["update_wall"][2:] or st["update_wall"]
    per_update = sorted(a + b for a, b in zip(tail_r, tail_u))[len(tail_r) // 2]
    res = {"env_id": env_id, "agents_per_gpu": agents,
           "sps": st["final_sps"], "unit": "samples/s (global_step / wall, ppo…:257,376), all GPUs",
           "sps_steady": agents * 128 * world / per_update,
           "steady_note": "median over updates >= 3 (update 1 runs eagerly, update 2 records the CUDA graphs)",
           "rollout_s_steady": sorted(tail_r)[len(tail_r) // 2], "update_s_steady": sorted(tail_u)[len(tail_u) // 2],
           "workload": f"ppo-{env_id}, {agents} agents per GPU x 128 steps, 4 minibatches x 8 epochs, "
                       f"{st['updates']} updates, defaults of ppo…:71-108",
           "rollout_s": st["rollout_s"], "update_s": st["update_s"], "wall_s": st["wall"],
           "mlp_backend": st.get("mlp_backend", "torch-fp32"), "nccl_in_graph": st.get("nccl_in_graph"),
           "grad_allreduce": st.get("grad_allreduce"),
           "sanitised_fields": st.get("sanitised_fields"), "n_gpus": world}
    del st
    torch.cuda.empty_cache()
    return res


def run_native(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl native needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n = args.envs
    envs, acts = make_task(torch, n, rank, local)

    def step_full(i):
        return envs.step(acts[i & 3])  # the drop-in VSS.step: one fused vss_step launch

    last = {}

    def timed_step(i):
        last["out"] = step_full(i)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()   # before the warm-up; `mark` drops the warm-up samples when the timed region starts
    ms = time_steps(torch, dist, world, timed_step, args.steps, args.warmup, on_start=sampler.mark)
    clocks = sampler.stop() if rank == 0 else None
    value = world * n * args.steps / (ms * 1e-3)
    if args.dump_outputs and rank == 0:   # before the legs below step the same fields again
        dump_outputs(torch, args.dump_outputs, last["out"])
    last.clear()

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = BYTES_PER_FIELD_STEP * n / (ms * 1e-3 / args.steps) / 1e9
    traffic = None
    try:  # dram__bytes_read.sum + dram__bytes_write.sum of one `ncu --set full` capture, scaled per field
        tr = json.load(open(os.path.join(ROOT, "profiles", "r02_step_traffic.json")))
        traffic = tr["dram_bytes_per_field_step"] * n
    except Exception:
        pass
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic,
                "traffic_source": "ncu capture profiles/r02_step_traffic.json (per field-step x fields), not re-measured in this run",
                "kernel": "k_step<full>", "algorithmic_bytes_per_launch": BYTES_PER_FIELD_STEP * n,
                "region": f"{args.steps} back-to-back launches" + (" (burst: shorter than the power-cap time constant)"
                                                                   if args.steps < 200 else " (sustained)"),
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s"}
    launches = args.steps  # timed region: K x k_step
    if args.steps < 200:   # the same kernel over a region long enough for the power cap to set in
        ms_s = time_steps(torch, dist, world, step_full, 400, 20)
        ach_s = BYTES_PER_FIELD_STEP * n / (ms_s * 1e-3 / 400) / 1e9
        roofline["sustained"] = {"steps": 400, "ms_per_step": ms_s / 400, "achieved": ach_s, "frac": ach_s / peak,
                                 "value": world * n * 400 / (ms_s * 1e-3)}
        launches += 420

    # ---- GAE reverse scan (BASELINE roofline row: 28 B per (t, env)), T = 128
    gae_res = None
    if world == 1:
        from rsoccer_isaac_cleanrl_b200.engine import gae as gae_kernel
        # T=128 x 65536 columns (configs[3] read as 65 536 agents: 235 MB per call, latency and launch ramp
        # still visible) and T=128 x 196608 (65 536 dma fields = 196 608 agents: 705 MB per call)
        gae_res = []
        for Tn, Nn in ((128, 65536), (128, 196608)):
            gin = [torch.randn((Tn, Nn), device="cuda") for _ in range(3)]
            gd = (torch.rand((Tn, Nn), device="cuda") < 0.01).float()
            gto = gd * (torch.rand((Tn, Nn), device="cuda") < 0.5).float()
            adv, ret = torch.empty_like(gd), torch.empty_like(gd)
            # >= 235 MB per call: larger than L2, so consecutive calls do not hit in cache
            ms_g = time_steps(torch, dist, 1, lambda i: gae_kernel(*gin, gd, gto, 0.99, 0.95, adv, ret), 50, 5)
            gbs = 28.0 * Tn * Nn / (ms_g * 1e-3 / 50) / 1e9
            gae_res.append({"elements_per_s": Tn * Nn * 50 / (ms_g * 1e-3), "us_per_call": ms_g * 1e3 / 50,
                            "achieved_gbs": gbs, "frac": gbs / peak,
                            "workload": f"vss_gae T={Tn} N={Nn}, 28 B per (t, env)"})
        del gin, gd, gto, adv, ret

    # ---- e2e: the user-facing call with HOST buffers (SingleAgent view): pinned policy action ->
    #      device, fused view step, packed view rows -> pinned host, every step.
    e2e = None
    if not args.skip_e2e:
        from rsoccer_isaac_cleanrl_b200.envs import SingleAgent
        from rsoccer_isaac_cleanrl_b200.hostmem import pinned_empty
        view = SingleAgent(envs)
        pa = [torch.rand((n, 2)).mul_(2).sub_(1).pin_memory() for _ in range(2)]
        k_e2e = max(10, min(args.steps, 100))
        chunks = view.HOST_CHUNKS if n >= view.HOST_CHUNK_MIN_FIELDS else 1
        variants = {}
        for name, dt in (("bf16_packed_rows", torch.bfloat16), ("f32_reference_types", torch.float32)):
            ms_v = time_steps(torch, dist, world, lambda i: view.step_host(pa[i & 1], obs_dtype=dt), k_e2e, 3)
            variants[name] = {"value": world * n * k_e2e / (ms_v * 1e-3), "ms_per_step": ms_v / k_e2e,
                              "d2h_bytes_per_step": view.d2h_bytes(dt)}
            launches += (k_e2e + 3) * chunks
        # the ceiling: a plain cudaMemcpyAsync of the same bytes, device -> pinned host, all ranks at once
        nbytes = view.d2h_bytes(torch.bfloat16)
        src = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
        dst = pinned_empty((nbytes,), torch.uint8, f"cuda:{local}")
        ms_c = time_steps(torch, dist, world, lambda i: dst.copy_(src, non_blocking=True), 20, 3)
        d2h_gbs = nbytes * 20 / (ms_c * 1e-3) / 1e9
        del src, dst
        # the full VSS.step contract with host buffers (2.6 KB per field-step across PCIe)
        k_full = 5
        ms_f = time_steps(torch, dist, world, full_contract_host_step(torch, envs, local), k_full, 2)
        launches += k_full + 2
        best = variants["bf16_packed_rows"]
        e2e = {"value": best["value"], "unit": "env-steps/s",
               "h2d_bytes_per_step": view.h2d_bytes_per_step, "d2h_bytes_per_step": best["d2h_bytes_per_step"],
               "steps": k_e2e, "ms_per_step": best["ms_per_step"],
               "api": "SingleAgent.step_host(pinned policy action (N,2)) -> pinned packed rows (N,112 B): obs (N,52) "
                      "bf16, reward (N) f32, done (N) u8, time-out (N) u8 (what envs/wrappers.py:108-115 returns to "
                      f"the policy); the step runs as {chunks} field ranges (vss_set_step_range) on two streams, one "
                      "cudaMemcpyAsync per range; host sync every step",
               "variants": variants,
               "d2h_memcpy_gbs_per_gpu": d2h_gbs,
               "d2h_memcpy_note": f"plain device->pinned copies of the same bytes, {world} rank(s) at once: the "
                                  "ceiling of this box's PCIe / host memory path",
               "d2h_frac_of_memcpy": best["d2h_bytes_per_step"] / (best["ms_per_step"] * 1e-3) / 1e9 / d2h_gbs,
               "full_contract": {"value": world * n * k_full / (ms_f * 1e-3), "ms_per_step": ms_f / k_full,
                                 "h2d_bytes_per_step": FULL_H2D * n, "d2h_bytes_per_step": FULL_D2H * n,
                                 "api": "VSS.step with pinned host buffers: (N,2,3,2) actions in; obs, terminal obs, "
                                        "rewards, reset, time-outs, progress out"}}
        del view, pa

    sweep = None
    if not args.no_sweep:
        # BASELINE configs[4]: random-action step throughput from 1K to 1M fields per GPU (same full
        # VSS.step contract; sizes below ~64K fields fit in L2 and are launch/latency bound)
        sweep = []
        del envs, acts
        for ne in (1024, 4096, 16384, 65536, 262144, 1048576):
            e2, a2 = make_task(torch, ne, rank, local)
            f = lambda i: e2.step(a2[i & 3])
            m = time_steps(torch, dist, world, f, 200, 20)
            sweep.append({"envs_per_gpu": ne, "env_steps_per_s": world * ne * 200 / (m * 1e-3),
                          "us_per_step": m * 1e3 / 200,
                          "hbm_frac": BYTES_PER_FIELD_STEP * ne / (m * 1e-3 / 200) / 1e9 / peak})
            del e2, a2

    # ---- PPO SPS (BASELINE configs[1-3]; OU-noise opponents as in training)
    ppo_res = None
    if not args.skip_ppo:
        try:
            del envs, acts
        except NameError:
            pass
        ppo_res = []
        for leg in args.ppo_legs.split(","):
            env_id, agents = leg.split(":")
            updates = args.ppo_updates or max(8, min(40, int(2.1e7 // (int(agents) * 128))))
            ppo_res.append(run_ppo_leg(torch, world, env_id, int(agents), updates))

    ref_torch = None
    if world == 1 and not args.skip_reference_torch:
        try:
            del envs, acts
        except NameError:
            pass
        torch.cuda.empty_cache()
        ref_torch = reference_torch_legs(torch, peak)

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.skip_cpu_baseline:
        cpu_baseline, _ = cpu_oracle_run(n, seconds=args.cpu_seconds, contract="sa_view")

    if rank == 0:
        line = {
            "metric": "vss_env_steps_per_s", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"random-action VSS 3v3 env step (BASELINE configs[4] sweep top), full VSS.step "
                                   f"contract, {n} fields per GPU, U(-1,1) actions resident in HBM, progress "
                                   "counters staggered to the steady-state reset rate; e2e and cpu_baseline: the "
                                   "same fields stepped through the SingleAgent view",
                       "envs_per_gpu": n, "l2": f"per-step working set {BYTES_PER_FIELD_STEP * n / 1e6:.0f} MB "
                                               "(> 126 MB L2 when envs_per_gpu >= 65536)",
                       "parallelism": f"fields sharded over {world} GPU(s), no data-path collective"},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": launches,
            "clocks": clocks, "ppo": ppo_res[0] if ppo_res else None, "ppo_legs": ppo_res, "gae": gae_res,
            "reference_torch": ref_torch,
        }
        if sweep:
            line["sweep"] = sweep
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def emit(line):
    """The ONE JSON line goes to the real stdout; everything libraries print (e.g. NCCL's version
    banner) was diverted to stderr at start-up."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


if __name__ == "__main__":
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
