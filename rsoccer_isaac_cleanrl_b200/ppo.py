"""PPO training loop — drop-in for the reference's `ppo_continuous_action_isaacgym.py`.

Same CLI flags and defaults (reference ppo…:48-118), same `Agent` (attribute names and
state_dict keys `critic.{0,2,4,6,8}.*`, `actor_mean.{0,2,4,6,8}.*`, `actor_logstd`, :121-164),
same rollout / GAE / clipped-surrogate update (:231-365), with
  * the env step, OU opponents, view slicing and episode statistics in ONE kernel per step
    (`vss_step_view`),
  * GAE as one reverse-scan kernel (`vss_gae`) instead of a 128-iteration python loop,
  * no per-minibatch `.item()` host syncs (the reference syncs at :322; statistics are
    accumulated on the device and read once per update),
  * data-parallel over GPUs: each rank owns `--num-envs` agents on its own fields; the only
    collective is one all-reduce of the flat gradient per minibatch (NCCL over NVLink).

Run:  python -m rsoccer_isaac_cleanrl_b200.ppo --env-id sa --num-envs 4096 --total-timesteps 2000000
      torchrun --nproc-per-node 8 -m rsoccer_isaac_cleanrl_b200.ppo --env-id dma --num-envs 196608
"""
import argparse
import os
import random
import time

import numpy as np
import torch
import torch.nn as nn

from .engine import gae as gae_kernel
from .envs.spaces import ObservationWrapper


def _strtobool(x):
    x = str(x).lower()
    if x in ("y", "yes", "t", "true", "on", "1"):
        return True
    if x in ("n", "no", "f", "false", "off", "0"):
        return False
    raise ValueError(f"invalid truth value {x!r}")


def parse_args(argv=None):
    b = lambda x: bool(_strtobool(x))
    p = argparse.ArgumentParser()
    p.add_argument("--exp-name", type=str, help="the name of this experiment")
    p.add_argument("--seed", type=int, default=1)
    p.add_argument("--torch-deterministic", type=b, default=True, nargs="?", const=True,
                   help="sets torch.backends.cudnn.deterministic as the reference does; run-to-run bit "
                        "reproducibility additionally needs --mlp-backend torch (the tcgen05 path reduces "
                        "split-K partial sums and statistics with floating-point atomics in arbitrary order)")
    p.add_argument("--cuda", type=b, default=True, nargs="?", const=True)
    p.add_argument("--track", type=b, default=False, nargs="?", const=True)
    p.add_argument("--wandb-project-name", type=str, default="ppo-isaac-cleanrl")
    p.add_argument("--wandb-entity", type=str, default=None)
    p.add_argument("--capture-video", type=b, default=False, nargs="?", const=True)
    # algorithm
    p.add_argument("--env-id", type=str, default="sa")
    p.add_argument("--total-timesteps", type=int, default=1000000000)
    p.add_argument("--learning-rate", type=float, default=0.001)
    p.add_argument("--num-envs", type=int, default=4095, help="parallel agents PER GPU")
    p.add_argument("--num-steps", type=int, default=128)
    p.add_argument("--anneal-lr", type=b, default=False, nargs="?", const=True)
    p.add_argument("--adaptative-lr", type=b, default=False, nargs="?", const=True)
    p.add_argument("--gamma", type=float, default=0.99)
    p.add_argument("--gae-lambda", type=float, default=0.95)
    p.add_argument("--num-minibatches", type=int, default=4)
    p.add_argument("--update-epochs", type=int, default=8)
    p.add_argument("--norm-adv", type=b, default=True, nargs="?", const=True)
    p.add_argument("--clip-coef", type=float, default=0.2)
    p.add_argument("--clip-vloss", type=b, default=False, nargs="?", const=True)
    p.add_argument("--ent-coef", type=float, default=0.005)
    p.add_argument("--vf-coef", type=float, default=4)
    p.add_argument("--max-grad-norm", type=float, default=1.5)
    p.add_argument("--target-kl", type=float, default=None)
    p.add_argument("--threshold-kl", type=float, default=0.008)
    p.add_argument("--reward-scaler", type=float, default=1000)  # parsed and unused, as in the reference
    p.add_argument("--record-video-step-frequency", type=int, default=20000)
    p.add_argument("--test", type=b, default=False, nargs="?", const=True)
    # engine-specific additions
    p.add_argument("--save-path", type=str, default="runs")
    p.add_argument("--mlp-backend", type=str, default="auto", choices=["auto", "tc", "torch"],
                   help="tc: hand-written tcgen05 GEMMs (bf16 in, fp32 accumulate); torch: fp32 library GEMMs")
    p.add_argument("--cuda-graph", type=b, default=True, nargs="?", const=True,
                   help="capture the whole T-step rollout (+ critic on terminal obs + GAE) in one CUDA graph")
    p.add_argument("--grad-allreduce", type=str, default="auto", choices=["auto", "peer", "nccl"],
                   help="multi-GPU gradient sum: peer = one hand-written kernel per rank over NVLink peer memory "
                        "(CUDA IPC, one node); nccl = torch.distributed.all_reduce; auto = peer when it can be set up")
    p.add_argument("--opponent", type=str, default="ou",
                   help="the yellow team during training: ou (OU noise, the reference), zero, self (a frozen snapshot "
                        "of the learner) or ppo-sa|ppo-sa-x3|ppo-cma|ppo-dma:PATH (a checkpoint)")
    p.add_argument("--opponent-refresh", type=int, default=10,
                   help="--opponent self: the snapshot is taken before update 1 and then every K updates")
    p.add_argument("--quiet", type=b, default=False, nargs="?", const=True)
    p.add_argument("--tensorboard", type=b, default=True, nargs="?", const=True,
                   help="write the reference's scalar tags (losses/*, Charts/SPS, rws/episodic_*) with SummaryWriter")
    args = p.parse_args(argv)
    args.batch_size = int(args.num_envs * args.num_steps)
    args.minibatch_size = int(args.batch_size // args.num_minibatches)
    return args


def layer_init(layer, std=np.sqrt(2), bias_const=0.0):
    torch.nn.init.orthogonal_(layer.weight, std)
    torch.nn.init.constant_(layer.bias, bias_const)
    return layer


def _mlp(n_in, n_out, out_std):
    return nn.Sequential(
        layer_init(nn.Linear(n_in, 256)), nn.Tanh(),
        layer_init(nn.Linear(256, 512)), nn.Tanh(),
        layer_init(nn.Linear(512, 512)), nn.Tanh(),
        layer_init(nn.Linear(512, 256)), nn.Tanh(),
        layer_init(nn.Linear(256, n_out), std=out_std))


class Agent(nn.Module):
    """Two independent 52-256-512-512-256-{A,1} tanh MLPs + state-independent log-std."""

    def __init__(self, envs, mlp_backend="torch"):
        super().__init__()
        self.mlp_backend = mlp_backend  # "tc": tcgen05 GEMMs (bf16 in, fp32 accumulate); "torch": fp32 library
        n_obs = int(np.array(envs.single_observation_space.shape).prod())
        n_act = int(np.prod(envs.single_action_space.shape))
        self.critic = _mlp(n_obs, 1, 1.0)
        self.actor_mean = _mlp(n_obs, n_act, 0.01)
        self.actor_logstd = nn.Parameter(torch.zeros(1, n_act))

    def _mlp(self, seq, x):
        if self.mlp_backend == "tc" and x.is_cuda:
            from .tc_mlp import mlp_forward
            return mlp_forward(seq, x.contiguous())
        return seq(x)

    def get_value(self, x):
        return self._mlp(self.critic, x)

    def get_action_and_value(self, x, action=None):
        action_mean = self._mlp(self.actor_mean, x)
        action_logstd = self.actor_logstd.expand_as(action_mean)
        action_std = torch.exp(action_logstd)
        if action is None:
            action = action_mean + action_std * torch.randn_like(action_mean)  # Normal.sample()
        # Normal(mean, std).log_prob(action).sum(1) and .entropy().sum(1)
        var = action_std * action_std
        logp = (-((action - action_mean) ** 2) / (2 * var) - action_logstd - 0.5 * np.log(2 * np.pi)).sum(1)
        entropy = (0.5 + 0.5 * np.log(2 * np.pi) + action_logstd).sum(1)
        return action, logp, entropy, self._mlp(self.critic, x)


class ExtractObsWrapper(ObservationWrapper):
    def observation(self, obs):
        return obs["obs"]


def flat_size(module):
    """Floats of the flat parameter buffer of `flatten_parameters` (every tensor padded to a multiple of 4)."""
    return sum((p.numel() + 3) // 4 * 4 for p in module.parameters())


def flatten_parameters(module, grad_buffer=None):
    """Re-home every parameter (and its .grad) as a view of one flat buffer, so the gradient
    all-reduce, the norm clip and Adam each touch ONE tensor. `grad_buffer`: an existing zeroed f32 tensor to
    hold the flat gradient (e.g. the peer-mapped buffer of `PeerGradients`)."""
    params = list(module.parameters())
    # every tensor starts on a 16-byte boundary (the 1-element biases of the value head would otherwise leave all
    # later tensors at odd offsets: the split-K wgrad reduces with 16-byte vector atomics); the padding words stay
    # zero in the parameters, the gradient and the Adam moments
    starts, off = [], 0
    for p in params:
        starts.append(off)
        off += (p.numel() + 3) // 4 * 4
    flat = torch.zeros(off, device=params[0].device, dtype=params[0].dtype)
    flat_grad = torch.zeros_like(flat) if grad_buffer is None else grad_buffer[:off]
    for p, o in zip(params, starts):
        n = p.numel()
        flat[o:o + n].copy_(p.data.view(-1))
        p.data = flat[o:o + n].view_as(p.data)
        p.grad = flat_grad[o:o + n].view_as(p.data)
    return flat, flat_grad


class FlatAdam:
    """Adam (eps 1e-5, no weight decay; torch.optim.Adam semantics) over the flat buffer. The step
    count and the learning rate live in device tensors so that step() can sit inside a CUDA graph."""

    def __init__(self, flat, flat_grad, lr, eps=1e-5, betas=(0.9, 0.999)):
        self.flat, self.grad, self.eps, self.b1, self.b2 = flat, flat_grad, eps, betas[0], betas[1]
        self.m, self.v = torch.zeros_like(flat), torch.zeros_like(flat)
        self.state = torch.zeros(3, device=flat.device, dtype=torch.float32)  # [step count, lr, scratch]
        self.t, self.lr_t = self.state[0], self.state[1]
        self.lr_t.fill_(lr)
        self.param_groups = [{"lr": lr}]
        self._lr_host = lr

    def sync_lr(self):
        """Push param_groups[0]['lr'] (annealing / adaptive schedule) to the device scalar."""
        lr = self.param_groups[0]["lr"]
        if lr != self._lr_host:
            self.lr_t.fill_(lr)
            self._lr_host = lr

    def step(self):
        g = self.grad
        self.t += 1
        self.m.mul_(self.b1).add_(g, alpha=1 - self.b1)
        self.v.mul_(self.b2).addcmul_(g, g, value=1 - self.b2)
        bc1 = 1 - torch.pow(self.b1, self.t)
        bc2 = 1 - torch.pow(self.b2, self.t)
        denom = (self.v.sqrt() / bc2.sqrt()).add_(self.eps)
        self.flat.sub_((self.m / denom) * (self.lr_t / bc1))

    def clip_and_step_fused(self, max_grad_norm, grad_scale=1.0):
        """clip_grad_norm_(max_grad_norm) on grad * grad_scale, then step(): three launches
        (`vss_clip_adam`) instead of ~25."""
        from .engine import clip_adam
        clip_adam(self.flat, self.grad, self.m, self.v, self.state, grad_scale, max_grad_norm, self.b1, self.b2,
                  self.eps)


def anneal_lr(update, num_updates, learning_rate):
    """ppo…:250-254: linear decay, `update` counts from 1."""
    return (1.0 - (update - 1.0) / num_updates) * learning_rate


def torch_minibatch_grad(agent, args, batch, inds, stats=None, clipfrac_sum=None):
    """One minibatch of ppo…:314-352 with torch autograd (fp32): the clipped-surrogate / value / entropy
    loss of the rows `inds` of `batch` (dict of b_obs, b_actions, b_logprobs, b_advantages, b_returns,
    b_values) and its gradient into the parameters' .grad buffers (zeroed first). No host sync: the
    statistics go to the device scalars in `stats`."""
    _, newlogprob, entropy, newvalue = agent.get_action_and_value(batch["b_obs"][inds], batch["b_actions"][inds])
    logratio = newlogprob - batch["b_logprobs"][inds]
    ratio = logratio.exp()
    with torch.no_grad():
        if stats is not None:
            stats["old_approx_kl"].copy_((-logratio).mean())
            stats["approx_kl"].copy_(((ratio - 1) - logratio).mean())
        if clipfrac_sum is not None:
            clipfrac_sum.add_(((ratio - 1.0).abs() > args.clip_coef).float().mean())
    mb_advantages = batch["b_advantages"][inds]
    if args.norm_adv:
        mb_advantages = (mb_advantages - mb_advantages.mean()) / (mb_advantages.std() + 1e-8)
    pg_loss = torch.max(-mb_advantages * ratio,
                        -mb_advantages * torch.clamp(ratio, 1 - args.clip_coef, 1 + args.clip_coef)).mean()
    newvalue = newvalue.view(-1)
    mb_returns = batch["b_returns"][inds]
    if args.clip_vloss:
        mb_values = batch["b_values"][inds]
        v_clipped = mb_values + torch.clamp(newvalue - mb_values, -args.clip_coef, args.clip_coef)
        v_loss = 0.5 * torch.max((newvalue - mb_returns) ** 2, (v_clipped - mb_returns) ** 2).mean()
    else:
        v_loss = 0.5 * ((newvalue - mb_returns) ** 2).mean()
    entropy_loss = entropy.mean()
    loss = pg_loss - args.ent_coef * entropy_loss + v_loss * args.vf_coef
    if stats is not None:
        with torch.no_grad():
            stats["v_loss"].copy_(v_loss); stats["pg_loss"].copy_(pg_loss); stats["entropy"].copy_(entropy_loss)
    for p in agent.parameters():
        if p.grad is not None:
            p.grad.zero_()
    loss.backward()
    return loss


def update_policy(args, batch_size, randperm, run_minibatch, optimizer, read_kl):
    """The epoch / minibatch schedule of ppo…:308-365 around a caller-supplied minibatch step.

    `run_minibatch(mb_inds)` does forward, loss, backward, gradient clip and the optimiser step for the
    given rows (including the shorter remainder minibatch that `range(0, batch_size, minibatch_size)`
    visits when batch_size is not a multiple of it, ppo…:310-312). `read_kl()` returns the approx-KL of the
    LAST minibatch as a float (mean over ranks); it is only called when a flag needs it, because it
    synchronises. Adaptive LR (ppo…:356-361) looks at every minibatch; the target-KL stop (ppo…:363-365)
    looks at the last minibatch of an epoch, after the inner loop. Returns (minibatches run, epochs run)."""
    n_mb = 0
    epochs = 0
    for epoch in range(args.update_epochs):
        epochs += 1
        b_inds = randperm(batch_size)
        for start in range(0, batch_size, args.minibatch_size):
            run_minibatch(b_inds[start:start + args.minibatch_size])
            n_mb += 1
            if args.adaptative_lr:
                kl = read_kl()
                current_lr = optimizer.param_groups[0]["lr"]
                if kl > 2.0 * args.threshold_kl:
                    optimizer.param_groups[0]["lr"] = max(current_lr / 1.5, 1e-6)
                elif kl < 0.5 * args.threshold_kl:
                    optimizer.param_groups[0]["lr"] = min(current_lr * 1.5, 1e-2)
        if args.target_kl is not None and read_kl() > args.target_kl:
            break
    return n_mb, epochs



def _make_writer(args, rank, log):
    """SummaryWriter of ppo…:195-199 (rank 0; None when --quiet, --tensorboard false or tensorboard is not
    installed). W&B (--track) and video capture are out of scope (SURVEY §2 #18, #22): say so instead of
    silently ignoring the flags."""
    if rank != 0:
        return None
    if args.track:
        log("warning: --track (Weights & Biases) is not implemented by this engine; the TensorBoard event file "
            "carries the same scalars")
    if args.capture_video:
        log("warning: --capture-video is not implemented by this engine (no renderer); flag ignored")
    if args.quiet or not getattr(args, "tensorboard", True):
        return None
    try:
        from torch.utils.tensorboard import SummaryWriter
    except Exception as e:
        log(f"warning: tensorboard is not available ({e}); no event file is written")
        return None
    run_name = f"{args.exp_name}_ppo-{args.env_id}_{args.seed}"
    writer = SummaryWriter(os.path.join(getattr(args, "save_path", "runs"), run_name))
    writer.add_text("hyperparameters", "|param|value|\n|-|-|\n%s" % (
        "\n".join([f"|{key}|{value}|" for key, value in vars(args).items()])))
    return writer


_SELF_TEAM = {"sa": "TeamSA", "cma": "TeamCMA", "dma": "TeamDMA"}


def make_opponent(args, agent, envs, device, backend):
    """(team, frozen Agent or None) for --opponent; team None = OU noise (the reference's view, today's kernel)."""
    from . import play
    spec = getattr(args, "opponent", "ou")
    if spec == "ou":
        return None, None
    if spec == "self":  # a frozen copy of the learner's actor, in the learner's own mode
        frozen = Agent(envs, mlp_backend=backend).to(device)
        frozen.load_state_dict(agent.state_dict())
        frozen.requires_grad_(False)
        frozen.eval()
        return getattr(play, _SELF_TEAM[args.env_id]).from_agent(frozen), frozen
    algo, _, path = spec.partition(":")
    if algo not in ("zero", "ppo-sa", "ppo-sa-x3", "ppo-cma", "ppo-dma") or (algo != "zero" and not path):
        raise ValueError(f"--opponent: expected ou, zero, self or ALGO:PATH, got {spec!r}")
    return play.get_team(algo, path or None, str(device), backend), None


def train(args, log=print, hook=None):
    import torch.distributed as dist
    from .envs import RecordEpisodeStatisticsTorch, make_env
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    random.seed(args.seed); np.random.seed(args.seed); torch.manual_seed(args.seed + rank)
    torch.backends.cudnn.deterministic = args.torch_deterministic
    device = torch.device("cuda", local)

    writer = _make_writer(args, rank, log)
    unwrapped_env, envs = make_env(args)
    view = envs
    envs = ExtractObsWrapper(envs)
    envs = RecordEpisodeStatisticsTorch(envs, device)
    envs.single_action_space = envs.action_space
    envs.single_observation_space = envs.observation_space

    torch.manual_seed(args.seed)  # identical initial weights on every rank
    backend = "tc" if args.mlp_backend in ("auto", "tc") else "torch"
    agent = Agent(envs, mlp_backend=backend).to(device)
    torch.manual_seed(args.seed + 1000 * (rank + 1))
    # the flat gradient lives in a buffer the other ranks of the node can read (peer.py) when that can be set up
    peer_grads = None
    mode = getattr(args, "grad_allreduce", "auto")
    if world > 1 and mode != "nccl":
        one_node = int(os.environ.get("LOCAL_WORLD_SIZE", str(world))) == world
        try:
            if not one_node:   # (the same on every rank)
                raise RuntimeError("the ranks span several nodes (CUDA IPC reaches one node)")
            from .peer import PeerGradients
            peer_grads = PeerGradients(flat_size(agent), device, rank, world)
        except Exception as e:
            if mode == "peer":
                raise
            log(f"[rank {rank}] peer-memory gradient all-reduce unavailable ({type(e).__name__}: {e}); using NCCL")
            peer_grads = None   # (PeerGradients raises on every rank or on none)
    flat, flat_grad = flatten_parameters(agent, None if peer_grads is None else peer_grads.buffer)
    if world > 1:
        dist.broadcast(flat, 0)
    # what clip + Adam read: the summed gradient (a local buffer with the peer kernel, flat_grad itself with NCCL)
    grad_sum = flat_grad if peer_grads is None else torch.zeros_like(flat)
    optimizer = FlatAdam(flat, grad_sum, lr=args.learning_rate, eps=1e-5)

    # the yellow team (--opponent): its own Philox stream per rank, like the learner's sampling stream
    opp_team, opp_frozen = make_opponent(args, agent, envs, device, backend)
    opp = opp_dev = None
    if opp_team is not None:
        from .play import _team_seed
        view.set_opponent(opp_team, seed=_team_seed(args.seed + 7919 * (rank + 1), 1))
        opp = view.opponent
        opp_dev = opp.device if opp is not None else None   # a policy opponent whose actor runs on the device

    def opponent_snapshot(update):
        """--opponent self: copy the learner's weights into the frozen Agent's static fp32 buffers and their bf16
        copies, outside any graph: later rollout replays read the new snapshot."""
        with torch.no_grad():
            for p_o, p_l in zip(opp_frozen.parameters(), agent.parameters()):
                p_o.copy_(p_l)
            if opp_dev is not None:
                opp_dev.mw.refresh()

    T, N = args.num_steps, args.num_envs
    oshape, ashape = envs.single_observation_space.shape, envs.single_action_space.shape
    z = lambda *s: torch.zeros(s, dtype=torch.float32, device=device)
    obs_all, actions = z(T + 1, N, *oshape), z(T, N, *ashape)   # obs_all[t + 1] is written by env step t
    obs = obs_all[:T]
    logprobs, rewards, next_dones, next_timeouts, values, next_values = (z(T, N) for _ in range(6))
    advantages, returns = z(T, N), z(T, N)
    term_obs_all = z(T, N, *oshape)

    fused = backend == "tc"
    if fused:
        from .engine import compact_nonzero, gather_pad_bf16, mlp_forward_fused, ppo_loss, scatter_rows
        from .tc_mlp import MlpWeights, backward_explicit, forward_explicit
        mw_actor, mw_critic = MlpWeights(agent.actor_mean), MlpWeights(agent.critic)
        sample_ctr = torch.zeros(1, device=device, dtype=torch.int32)
        sample_seed = args.seed + 7919 * (rank + 1)
        logstd_flat = agent.actor_logstd.detach().view(-1)
        k0 = mw_actor.k0
        # the critic runs beside the actor on a second stream (fork/join inside the captured graphs): at
        # 4096 rows one network's GEMMs fill less than half of the SMs
        side = torch.cuda.Stream(device=device)
        # the opponent's actor runs beside the learner's forward on a stream of its own
        opp_stream = torch.cuda.Stream(device=device) if opp_dev is not None else None

    def on_side(fn):
        """Run fn() on the side stream, ordered after everything queued so far on the current one.
        The caller joins with `join_side()` before the tensors fn touched are released or read."""
        if side is None:
            return fn()
        side.wait_stream(torch.cuda.current_stream(device))
        with torch.cuda.stream(side):
            return fn()

    def join_side():
        if side is not None:
            torch.cuda.current_stream(device).wait_stream(side)

    if fused:
        # the env step writes the next observation a second time as bf16 rows padded to k0 = 64 columns
        # (what the first tcgen05 GEMM reads) and done / timeout as floats (what the GAE kernel reads):
        # no conversion launches between the steps. Two buffers: step t reads one, writes the other.
        assert k0 == 64, k0
        x16_buf = [torch.zeros((N, k0), device=device, dtype=torch.bfloat16) for _ in range(2)]
        # V(terminal observation) (ppo…:272) is only computed where it differs from the next step's value: the rows
        # whose step ended an episode, compacted into a list of fixed capacity (1/8 of the rollout; checked per update)
        term_cap = max(128, (T * N // 8 + 127) // 128 * 128)
        term_list = torch.zeros(term_cap, device=device, dtype=torch.int64)
        term_count = torch.zeros(1, device=device, dtype=torch.int32)
        term_values = torch.zeros(term_cap, device=device, dtype=torch.float32)

    def rollout_fused(first_obs):
        """rollout() as two launches per step: the fused MLP forward (both networks' four tcgen05 layers + heads,
        action sample and log-prob written into the rollout slabs, the critic's value into values[step]) and the env
        step (obs / reward / done / timeout slabs and the next bf16 MLP input)."""
        with torch.no_grad():
            obs_all[0] = first_obs
            x16_buf[0].copy_(gather_pad_bf16(obs_all[0], None, k0))
            mw_actor.refresh(); mw_critic.refresh()
            nets = [(mw.w16, mw.bs, mw.head_w, mw.head_b) for mw in (mw_actor, mw_critic)]
            # One launch covers both networks while its CTAs (one per 128 rows and network) fit the SMs at once; with
            # more rows the critic gets its own launch on the side stream and runs beside the env step.
            one_launch = 2 * ((N + 127) // 128) <= torch.cuda.get_device_properties(device).multi_processor_count
            for step in range(T):
                # actor mean + action sample + log-prob (and the critic's value) in ONE launch (csrc/mlp_fused.cu); the
                # sampling stream's call index is counter + step, the counter advances by T once per rollout
                x16 = x16_buf[step & 1]
                if opp_dev is not None:  # its rows were written by the previous env step; its action is read by this one
                    opp_stream.wait_stream(torch.cuda.current_stream(device))
                    with torch.cuda.stream(opp_stream):
                        opp_dev.launch(step)
                samp = dict(logstd=logstd_flat, counter=sample_ctr, seed=sample_seed, call_offset=step,
                            action=actions[step], logprob=logprobs[step])
                if one_launch:
                    mlp_forward_fused(x16, [nets[0] + (False,), nets[1] + (values[step],)], sampling=samp)
                else:
                    on_side(lambda: mlp_forward_fused(x16, [nets[1] + (values[step],)]))
                    mlp_forward_fused(x16, [nets[0] + (False,)], sampling=samp)
                if opp_dev is not None:
                    torch.cuda.current_stream(device).wait_stream(opp_stream)
                envs.step(actions[step], obs_out=obs_all[step + 1], term_obs_out=term_obs_all[step],
                          reward_out=rewards[step], obs_bf16_out=x16_buf[(step + 1) & 1],
                          done_f_out=next_dones[step], timeout_f_out=next_timeouts[step],
                          opponent_issued=opp_dev is not None)
                if not one_launch:
                    join_side()
            sample_ctr.add_(T)
            if opp_dev is not None:
                opp_dev.counter.add_(T)
            # V(terminal observation) (ppo…:272). Where the step did not end an episode the terminal observation IS the
            # next observation (the step kernel writes both from the same registers), so its value is the next step's
            # critic output, bit for bit (every row of the fused forward is computed independently of its neighbours):
            # a shifted copy. Left to the critic: the observation after the last step and the rows that ended an
            # episode — one launch on a compacted list of fixed capacity instead of one over all T x N rows.
            if T > 1:
                next_values[:T - 1].copy_(values[1:])
            mlp_forward_fused(x16_buf[T & 1], [nets[1] + (next_values[T - 1],)])
            compact_nonzero(next_dones, term_list, term_count)
            mlp_forward_fused(gather_pad_bf16(term_obs_all.view(T * N, -1), term_list, k0), [nets[1] + (term_values,)])
            scatter_rows(next_values, term_list, term_values, term_count)
            gae_kernel(rewards, values, next_values, next_dones, next_timeouts, args.gamma, args.gae_lambda,
                       advantages, returns)
        return obs_all[T]

    def rollout(first_obs):
        """T env steps + V(terminal obs) + GAE (ppo…:256-296). No host sync anywhere, so the whole
        thing can be captured in a CUDA graph."""
        if fused:
            return rollout_fused(first_obs)
        with torch.no_grad():
            obs_all[0] = first_obs
            for step in range(T):
                cur = obs_all[step]
                action, logprob, _, value = agent.get_action_and_value(cur)
                values[step] = value.flatten()
                actions[step] = action
                logprobs[step] = logprob
                # the step kernel writes next obs / terminal obs / reward straight into the rollout slabs
                _, _, next_done, info = envs.step(action, obs_out=obs_all[step + 1],
                                                  term_obs_out=term_obs_all[step], reward_out=rewards[step])
                next_dones[step] = next_done
                next_timeouts[step] = info["time_outs"]
            cur = obs_all[T]
            # V(terminal_observation) for the whole rollout in one batched pass (ppo…:272 does it per step)
            next_values.copy_(agent.get_value(term_obs_all.view(T * N, *oshape)).view(T, N))
            gae_kernel(rewards, values, next_values, next_dones, next_timeouts, args.gamma, args.gae_lambda,
                       advantages, returns)
        return cur

    b_obs = obs.reshape((-1,) + oshape)
    b_logprobs, b_actions = logprobs.reshape(-1), actions.reshape((-1,) + ashape)
    b_advantages, b_returns, b_values = advantages.reshape(-1), returns.reshape(-1), values.reshape(-1)
    mb_inds = torch.zeros(args.minibatch_size, dtype=torch.long, device=device)
    clipfrac_sum = torch.zeros((), device=device)
    stats_buf = torch.zeros(8, device=device)  # vss_ppo_loss: pg_loss v_loss entropy old_kl kl clipfrac loss
    loss_scratch = torch.zeros(2, device=device, dtype=torch.float64)
    mb_stats = {"pg_loss": stats_buf[0], "v_loss": stats_buf[1], "entropy": stats_buf[2],
                "old_approx_kl": stats_buf[3], "approx_kl": stats_buf[4]}

    def forward_backward_fused():
        """forward_backward() without autograd: gather+pad once, both MLPs forward, ONE loss kernel
        that also produces d loss / d (mean, value, logstd), explicit backward into flat_grad."""
        x16 = gather_pad_bf16(b_obs, mb_inds, k0)
        mw_actor.refresh(); mw_critic.refresh()
        flat_grad.zero_()
        value, hs_c = on_side(lambda: forward_explicit(mw_critic, x16))
        mean, hs_a = forward_explicit(mw_actor, x16)
        join_side()
        d_mean, d_value, _ = ppo_loss(mean, value, logstd_flat, b_actions, b_logprobs, b_advantages, b_returns,
                                      b_values, mb_inds, args.clip_coef, args.ent_coef, args.vf_coef, args.norm_adv,
                                      args.clip_vloss, agent.actor_logstd.grad.view(-1), stats=stats_buf,
                                      scratch=loss_scratch)
        clipfrac_sum.add_(stats_buf[5])
        on_side(lambda: backward_explicit(mw_critic, hs_c, d_value))
        backward_explicit(mw_actor, hs_a, d_mean)
        join_side()

    batch = dict(b_obs=b_obs, b_actions=b_actions, b_logprobs=b_logprobs, b_advantages=b_advantages,
                 b_returns=b_returns, b_values=b_values)

    def forward_backward(inds=None):
        """One minibatch: clipped-surrogate loss and its gradient into flat_grad (ppo…:314-352).
        Reads the static index buffer mb_inds (or `inds`: the eager path of a remainder minibatch); no
        host sync (the reference's `.item()` at :322 is replaced by device-side accumulation), so it can
        be replayed as a CUDA graph."""
        if fused and inds is None:
            return forward_backward_fused()
        torch_minibatch_grad(agent, args, batch, mb_inds if inds is None else inds, mb_stats, clipfrac_sum)

    def clip_and_step():
        """nn.utils.clip_grad_norm_ + Adam on the flat buffer (ppo…:353-354); flat_grad holds the SUM
        over ranks at this point."""
        if fused:
            return optimizer.clip_and_step_fused(args.max_grad_norm, 1.0 / world)
        if world > 1:
            grad_sum.div_(world)
        gnorm = torch.linalg.vector_norm(grad_sum)
        grad_sum.mul_(torch.clamp(args.max_grad_norm / (gnorm + 1e-6), max=1.0))
        optimizer.step()

    def reduce_gradient():
        """The one collective of the path: sum of the flat gradient over ranks (clip_and_step divides)."""
        if peer_grads is not None:
            peer_grads.allreduce(grad_sum)   # one kernel over NVLink peer memory (csrc/peer_reduce.cu)
        elif world > 1:
            dist.all_reduce(flat_grad)

    # Can this process group's all-reduce be recorded into a CUDA graph? (Then the whole minibatch —
    # forward, backward, all-reduce, clip, Adam — is ONE graph replay and the collective no longer sits
    # between two replays with Python in between.) Probed once on a scratch tensor.
    nccl_in_graph = False
    if world > 1 and args.cuda_graph and peer_grads is None:
        try:
            probe = torch.zeros(1024, device=device)
            dist.all_reduce(probe)            # (communicator set-up happens outside capture)
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                dist.all_reduce(probe)
            g.replay()
            torch.cuda.synchronize()
            nccl_in_graph = True
            del g, probe
        except Exception as e:  # keep the collective between the graphs, as before
            log(f"[rank {rank}] NCCL all-reduce is not graph-capturable here ({type(e).__name__}: {e}); using the eager collective")
            torch.cuda.synchronize()

    def minibatch_step():
        """forward + backward + all-reduce + clip + Adam of the rows in mb_inds (graph-capturable)."""
        forward_backward()
        reduce_gradient()
        clip_and_step()

    rollout_graph = None
    mb_graph = fb_graph = opt_graph = None
    state = {"update": 0}

    def run_minibatch(inds):
        optimizer.sync_lr()
        if inds.numel() != args.minibatch_size:
            # the shorter remainder minibatch of ppo…:310-312 (only when batch_size is not a multiple of
            # num_minibatches): eager, torch autograd, its own index tensor
            forward_backward(inds)
            reduce_gradient()
            clip_and_step()
            return
        nonlocal mb_graph, fb_graph, opt_graph
        mb_inds.copy_(inds)
        capture = args.cuda_graph and state["update"] >= 2
        if world == 1 or nccl_in_graph or peer_grads is not None:
            if mb_graph is not None:
                mb_graph.replay()
            elif capture:
                torch.cuda.synchronize()
                mb_graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(mb_graph):
                    minibatch_step()
                mb_graph.replay()
            else:
                minibatch_step()
            return
        if fb_graph is not None:
            fb_graph.replay()
        elif capture:
            torch.cuda.synchronize()
            fb_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(fb_graph):
                forward_backward()
            fb_graph.replay()
        else:
            forward_backward()
        reduce_gradient()
        if opt_graph is not None:
            opt_graph.replay()
        elif capture:
            torch.cuda.synchronize()
            opt_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(opt_graph):
                clip_and_step()
            opt_graph.replay()
        else:
            clip_and_step()

    def read_kl():
        kl = mb_stats["approx_kl"].detach().clone()
        if world > 1:
            dist.all_reduce(kl); kl /= world
        return float(kl)

    global_step = 0
    start_time = time.time()
    next_obs = envs.reset()
    num_updates = args.total_timesteps // (args.batch_size * world)
    stats = {"sps": [], "updates": 0, "update_wall": [], "rollout_wall": [], "lr": [], "minibatches": [], "epochs": []}
    t_roll = t_upd = 0.0
    for update in range(1, num_updates + 1):
        state["update"] = update
        if opp_frozen is not None and (update - 1) % max(1, args.opponent_refresh) == 0:
            opponent_snapshot(update)
            if writer is not None:
                writer.add_scalar("opponent/snapshot_update", update, global_step)
        if args.anneal_lr:
            optimizer.param_groups[0]["lr"] = anneal_lr(update, num_updates, args.learning_rate)
        tr0 = time.time()
        global_step += T * N * world
        if rollout_graph is not None:
            rollout_graph.replay()
        elif args.cuda_graph and update >= 2:
            # every buffer the rollout touches is static by now (next_obs is the view's own output
            # buffer): record the T steps once, replay them for all later updates
            torch.cuda.synchronize()
            rollout_graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(rollout_graph):
                rollout(next_obs)
            rollout_graph.replay()
        else:
            next_obs = rollout(next_obs)
        torch.cuda.synchronize()
        tu0 = time.time()
        t_roll += tu0 - tr0
        if fused and int(term_count.item()) > term_cap:
            raise RuntimeError(f"{int(term_count.item())} of {T * N} rollout rows ended an episode: more than the "
                               f"{term_cap} rows the terminal-value list holds")

        clipfrac_sum.zero_()
        n_mb, n_ep = update_policy(args, args.batch_size, lambda n_: torch.randperm(n_, device=device), run_minibatch,
                                   optimizer, read_kl)
        stats["lr"].append(optimizer.param_groups[0]["lr"]); stats["minibatches"].append(n_mb); stats["epochs"].append(n_ep)
        torch.cuda.synchronize()
        t_upd += time.time() - tu0
        if hook is not None:  # diagnostics: called once per update with the live tensors
            hook(update, dict(obs=obs_all, actions=actions, logprobs=logprobs, rewards=rewards, values=values,
                              next_values=next_values, advantages=advantages, returns=returns, flat=flat,
                              flat_grad=flat_grad, term_obs=term_obs_all, next_dones=next_dones,
                              agent=agent, env=unwrapped_env, stats=mb_stats, opponent=opp))
        stats["rollout_wall"].append(tu0 - tr0)
        stats["update_wall"].append(time.time() - tu0)
        sps = int(global_step / (time.time() - start_time))
        stats["sps"].append(sps)
        stats["updates"] = update
        if writer is not None:  # the reference's tags (ppo…:273-279, 367-376); one host read per update
            writer.add_scalar("losses/learning_rate", optimizer.param_groups[0]["lr"], global_step)
            writer.add_scalar("losses/value_loss", mb_stats["v_loss"].item(), global_step)
            writer.add_scalar("losses/policy_loss", mb_stats["pg_loss"].item(), global_step)
            writer.add_scalar("losses/entropy", mb_stats["entropy"].item(), global_step)
            writer.add_scalar("losses/old_approx_kl", mb_stats["old_approx_kl"].item(), global_step)
            writer.add_scalar("losses/approx_kl", mb_stats["approx_kl"].item(), global_step)
            writer.add_scalar("losses/clipfrac", (clipfrac_sum / max(n_mb, 1)).item(), global_step)
            writer.add_scalar("Charts/SPS", sps, global_step)
            writer.add_scalar("engine/sanitised_fields", unwrapped_env.engine.sanitised_count, global_step)
            # an episode that ended on the rollout's last step (the reference samples steps 0-2 of the rollout
            # on the host; here the rollout is one CUDA graph, so the sample is taken after it)
            ended = next_dones[T - 1].nonzero()
            if ended.numel():
                idx = int(ended[0])
                r4 = envs.returned_episode_returns[idx]
                for j, key in enumerate(("goal", "grad", "move", "energy")):
                    writer.add_scalar(f"rws/episodic_{key}", r4[j].item(), global_step)
                writer.add_scalar("rws/episodic_return", r4.sum().item(), global_step)
                writer.add_scalar("rws/episodic_length", envs.returned_episode_lengths[idx].item(), global_step)
        if rank == 0 and not args.quiet:
            r = envs.returned_episode_returns.sum(1)
            log(f"update {update}/{num_updates} step {global_step} SPS {sps} lr {optimizer.param_groups[0]['lr']:.2e} "
                f"v_loss {mb_stats['v_loss'].item():.4f} pg_loss {mb_stats['pg_loss'].item():.4f} "
                f"ent {mb_stats['entropy'].item():.3f} kl {mb_stats['approx_kl'].item():.5f} "
                f"clipfrac {(clipfrac_sum / max(n_mb, 1)).item():.3f} ep_ret(last) {r.mean().item():.3f}")
    stats.update(global_step=global_step, wall=time.time() - start_time, rollout_s=t_roll, update_s=t_upd,
                 final_sps=(global_step / max(time.time() - start_time, 1e-9)))
    stats["mlp_backend"] = "tcgen05-bf16" if backend == "tc" else "torch-fp32"
    stats["nccl_in_graph"] = nccl_in_graph
    stats["grad_allreduce"] = "none" if world == 1 else ("peer-memory kernel" if peer_grads is not None else "nccl")
    stats["sanitised_fields"] = unwrapped_env.engine.sanitised_count
    if writer is not None:
        writer.close()
    if peer_grads is not None:   # the gradient views point into the peer buffer: drop them before it is freed
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()       # no rank unmaps while another may still be reading
        for p_ in agent.parameters():
            p_.grad = None
        del flat_grad
        peer_grads.close()
    stats["agent"] = agent
    stats["env"] = unwrapped_env
    stats["opponent"] = opp
    return stats


def main(argv=None):
    args = parse_args(argv)
    if args.test:
        args.total_timesteps = 1000000
    run_name = f"{args.exp_name}_ppo-{args.env_id}_{args.seed}"
    stats = train(args)
    if int(os.environ.get("RANK", "0")) == 0:
        os.makedirs(os.path.join(args.save_path, run_name), exist_ok=True)
        path = os.path.join(args.save_path, run_name, f"{run_name}-agent.pt")
        torch.save(stats["agent"].state_dict(), path)  # ppo…:379, same state_dict keys
        print(f"saved {path}; SPS {stats['final_sps']:.0f} (rollout {stats['rollout_s']:.1f}s, "
              f"update {stats['update_s']:.1f}s)")


if __name__ == "__main__":
    main()
