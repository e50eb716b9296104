"""GPU: the fused MLP forward (csrc/mlp_fused.cu: k_mlp_fwd<4>, k_mlp_fwd<8>) and the policy's action sampling
(csrc/ppo_sample.cuh sample_row, through k_policy_sample<2/6> and the fused launch) against exact and fp64
references, element by element.

(A) Hidden activations, bit for bit: a one-hot head (w[a, c] = 1, b = 0) makes out[:, a] the fused kernel's last
    hidden activation h4[:, c] exactly (one exact product, every other product a zero), compared with the layer-by-
    layer path (forward_explicit, exact-checked in test_gpu_tc_reference.py). The head with Gaussian weights against
    fp64 within 256 * 2^-24 * (|h4| |W|^T) + one rounding, with the bound shown tight. Outputs inside NaN guard
    buffers; an input with a padded row stride.
(B) Sampling against a numpy restatement of sample_row: Philox4x32-10 counter (row_lo, row_hi, call, 0x50504f00 + b),
    key (seed_lo, seed_hi), the uniforms and the angle in fp32 (exact), log / sqrt / cos / sin in fp64, within
    bounds from CUDA's documented maximum errors. The bounds reject a reference with the wrong call index, row,
    cos / sin order or block order at more than 99 % of the elements.
(C) The rollout's sampling stream end to end: actions, log-probs and values of three PPO updates (eager, captured,
    replayed) against (B) on the fused actor mean of the recorded observations.
(E) A profiler run checks that the cases reach every kernel instantiation."""
import re

import numpy as np
import pytest

from parity_checks import philox4x32_10_np
from test_gpu_tc_reference import (TINY, U32, _assert_bits, _assert_guard, _assert_within, _bits, _mlp, _out_buf,
                                   _strided)

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

F32 = torch.float32
PAIR_MIN_M = 256 * 74            # rows from which the layer-by-layer GEMMs take the CTA-pair kernel
STREAM_TAG = 0x50504F00          # 4th Philox counter word of the sampling stream (+ block index)
TWO_PI_F32 = np.float32(6.283185307179586)
ULP_REL = 2.0 ** -23             # one ulp of a normal fp32 x is at most 2^-23 |x|
LOGF_ULP, SINCOSF_ULP, EXPF_ULP = 1, 2, 2   # CUDA C Programming Guide, maximum ulp errors (no --use_fast_math)
HALF_LOG_2PI = 0.5 * np.log(2.0 * np.pi)
SEED = 0x9E3779B97F4A7C15 ^ 12345          # both key words non-zero


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _x16(M, seed):
    from rsoccer_isaac_cleanrl_b200.engine import gather_pad_bf16
    return gather_pad_bf16(torch.randn(M, 52, device="cuda", generator=_gen(seed)), None, 64)


def _net(mw, head_w=None, head_b=None, out=None):
    hw = mw.head_w.detach() if head_w is None else head_w
    hb = mw.head_b.detach() if head_b is None else head_b
    return (mw.w16, [b.detach() for b in mw.bs], hw.contiguous(), hb.contiguous(), out)


# ---------------------------------------------------------------------------------------------------------------
# (A) the fused forward
# ---------------------------------------------------------------------------------------------------------------
def _one_hot(cols):
    w = torch.zeros((len(cols), 256), device="cuda")
    w[torch.arange(len(cols)), torch.tensor(cols)] = 1.0
    return w, torch.zeros(len(cols), device="cuda")


def _report_rows(out, ref, what):
    ne = (_bits(out) != _bits(ref)).any(1)
    if ne.any():
        rows = ne.nonzero().view(-1)
        tiles = sorted(set((rows // 128).tolist()))
        raise AssertionError(f"{what}: {int(ne.sum())} of {ne.numel()} rows differ, first rows "
                             f"{rows[:8].tolist()}, in {len(tiles)} row tiles (first {tiles[:8]})")


@pytest.mark.parametrize("M", [1, 77, 128, 129, 4096, 16384 + 77, 65535, 1 << 20])
def test_hidden_activations_are_the_bits_of_the_layer_by_layer_path(M):
    """All 256 columns of h4 read out through one-hot heads: 22 launches of two 6-output networks (the same hidden
    weights in both slots, different columns), then (1, 6), (2, 1) and (6, 2) outputs in slots (0, 1), so that the
    second network slot runs every head width. Both epilogue shapes. Below 18 944 rows the layer-by-layer GEMMs run
    on one CTA per tile, from there on CTA pairs."""
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused
    from rsoccer_isaac_cleanrl_b200.tc_mlp import forward_explicit
    mw = _mlp(6, 100 + M % 97)
    x16 = _x16(M, M)
    h4 = forward_explicit(mw, x16)[1][4].float()
    for ew in (4, 8):
        rec = torch.full((M, 256), float("nan"), device="cuda")
        for k in range(22):
            c0 = [(12 * k + j) % 256 for j in range(6)]
            c1 = [(12 * k + 6 + j) % 256 for j in range(6)]
            o0, o1 = mlp_forward_fused(x16, [_net(mw, *_one_hot(c0)), _net(mw, *_one_hot(c1))], epilogue_warps=ew)
            rec[:, c0], rec[:, c1] = o0, o1
        _report_rows(rec, h4, f"h4 of the fused forward (EW={ew}, M={M}) vs forward_explicit")
        for n0, n1, off in ((1, 6, 3), (2, 1, 101), (6, 2, 250)):
            c0 = [(off + 7 * j) % 256 for j in range(n0)]
            c1 = [(off + 11 * j + 1) % 256 for j in range(n1)]
            o0, o1 = mlp_forward_fused(x16, [_net(mw, *_one_hot(c0)), _net(mw, *_one_hot(c1))], epilogue_warps=ew)
            _assert_bits(o0, h4[:, c0], f"slot 0 n_out={n0} EW={ew} M={M}")
            _assert_bits(o1, h4[:, c1], f"slot 1 n_out={n1} EW={ew} M={M}")
    print(f"[bits] h4 M={M}: all 256 columns equal for EW 4 and 8")


@pytest.mark.parametrize("M", [77, 4096, 16384 + 77, 65535])
def test_head_within_per_element_fp64_bound(M):
    """out = h4 W^T + b summed by the kernel in fp32 in its own order (head_chunk's fmaf chains, the EW = 8 halves
    combined) within 256 * 2^-24 * (|h4| |W|^T) + 2^-24 |ref| + TINY, against fp64 of the layer-by-layer h4 (the
    same bits, checked above). The bound rejects the reference with one 32-column chunk dropped and with one row
    tile shifted by one row."""
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused
    from rsoccer_isaac_cleanrl_b200.tc_mlp import forward_explicit
    x16 = _x16(M, M + 1)
    worst = 0.0
    for n0, n1 in ((2, 1), (6, 1), (1, 2)):
        nets = [_mlp(n0, 7 * n0 + M % 31), _mlp(n1, 7 * n1 + 3 + M % 31)]
        for mw in nets:   # Gaussian head weights of unit scale
            with torch.no_grad():
                mw.head_w.copy_(torch.randn(mw.head_w.shape, device="cuda", generator=_gen(mw.head_w.shape[0] + M)) / 16)
                mw.head_b.normal_(0, 0.5)
        hs = [forward_explicit(mw, x16)[1][4].double() for mw in nets]
        for ew in (4, 8):
            outs = mlp_forward_fused(x16, [_net(mw) for mw in nets], epilogue_warps=ew)
            for slot, (mw, h4, out) in enumerate(zip(nets, hs, outs)):
                W, b = mw.head_w.detach().double(), mw.head_b.detach().double()
                acc = h4 @ W.t()
                ref = acc + b
                bound = 256 * U32 * (h4.abs() @ W.abs().t()) + U32 * ref.abs() + TINY
                chunk = slice(96, 128)
                drop = h4[:, chunk] @ W[:, chunk].t()
                worst = max(worst, _assert_within(f"head n_out={mw.head_w.shape[0]} slot {slot} EW={ew} M={M}", out,
                                                  lambda a: a + b, acc, bound, drop, M))   # noqa: B023
    print(f"[err/bound] head M={M}: largest {worst:.4g}")


@pytest.mark.parametrize("M", [77, 16384 + 77])
def test_outputs_stay_inside_their_buffers_and_a_strided_input_reads_64_columns(M):
    """out, action and logprob are views inside NaN-filled buffers with 128 extra rows: nothing outside [M, n_out]
    is written. x16 with row stride 72 whose columns 64..71 hold NaN gives the bits of the contiguous input."""
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused
    actor, critic = _mlp(6, 41), _mlp(1, 42)
    x16 = _x16(M, M + 2)
    xs = _strided(x16, 72)
    assert xs.stride(0) == 72 and torch.isnan(xs.as_strided((M, 8), (72, 1), 64).float()).all()
    logstd = torch.linspace(-0.7, 0.2, 6, device="cuda")
    for ew in (4, 8):
        ref = mlp_forward_fused(x16, [_net(actor), _net(critic)], epilogue_warps=ew)
        bases, views = zip(_out_buf(M, 6, 6, F32), _out_buf(M, 1, 1, F32), _out_buf(M, 6, 6, F32), _out_buf(M, 1, 1, F32))
        out_a, out_c, act, lp = views
        ctr = torch.full((1,), 5, device="cuda", dtype=torch.int32)
        samp = dict(logstd=logstd, counter=ctr, seed=SEED, call_offset=5, action=act, logprob=lp.view(-1))
        mlp_forward_fused(xs, [_net(actor, out=out_a), _net(critic, out=out_c)], epilogue_warps=ew, sampling=samp)
        torch.cuda.synchronize()
        for base, n, what in zip(bases, (6, 1, 6, 1), ("actor out", "critic out", "action", "logprob")):
            _assert_guard(base, M, n, f"{what} EW={ew} M={M}")
        _assert_bits(out_a, ref[0], f"actor, strided input, EW={ew}")
        _assert_bits(out_c, ref[1], f"critic, strided input, EW={ew}")
        z_ref = _sample_reference(ref[0].cpu().numpy(), logstd.cpu().numpy(), np.arange(M), 10, SEED)
        _check_sample(act, lp.view(-1), ref[0], logstd, z_ref, f"strided EW={ew} M={M}")


# ---------------------------------------------------------------------------------------------------------------
# (B) sampling
# ---------------------------------------------------------------------------------------------------------------
def _normals(rows, call, seed, A, swap_cs=False, swap_blocks=False):
    """fp64 z [n, A] of sample_row for the given rows and call index, and the bound on |z_fp32 - z|."""
    rows = np.asarray(rows, np.int64)
    n, nb = rows.size, (A + 3) // 4
    lo, hi = (rows & 0xFFFFFFFF).astype(np.uint32), (rows >> 32).astype(np.uint32)
    key = (seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
    u = np.concatenate([philox4x32_10_np(np.stack([lo, hi, np.full(n, call % 2 ** 32, np.uint32),
                                                   np.full(n, STREAM_TAG + b, np.uint32)], 1), key)
                        for b in range(nb)], 1)
    if swap_blocks:
        u = np.concatenate([u[:, 4:8], u[:, 0:4]], 1)
    # vss::u01_open and vss::u01 (24-bit integers times 2^-24: exact), and the angle as the device rounds it
    u_open = ((u[:, 0::2] >> np.uint32(8)) + np.uint32(1)).astype(np.float32) * np.float32(2.0 ** -24)
    theta = TWO_PI_F32 * ((u[:, 1::2] >> np.uint32(8)).astype(np.float32) * np.float32(2.0 ** -24))
    L = np.log(u_open.astype(np.float64))
    rad = np.sqrt(-2.0 * L)
    cs, sn = np.cos(theta.astype(np.float64)), np.sin(theta.astype(np.float64))
    if swap_cs:
        cs, sn = sn, cs
    # logf: 1 ulp relative to |log u|; -2 * is exact; sqrtf is correctly rounded and halves the relative error
    e_rad = rad * (0.5 * LOGF_ULP * ULP_REL + U32) * (1 + 2.0 ** -20)
    z = np.empty((n, 4 * nb))
    e_z = np.empty((n, 4 * nb))
    for k, trig in ((0, cs), (1, sn)):
        e_trig = SINCOSF_ULP * ULP_REL * np.abs(trig) + TINY          # sincosf: 2 ulp each
        prod = rad * trig
        e_prod = e_rad * np.abs(trig) + (rad + e_rad) * e_trig
        z[:, k::2] = prod
        e_z[:, k::2] = e_prod + U32 * (np.abs(prod) + e_prod)          # rad * cs: one rounding
    return z[:, :A], e_z[:, :A]


def _sample_reference(mean, logstd, rows, call, seed, **wrong):
    """fp64 action = mean + exp(logstd) z and its bound: expf 2 ulp, and one rounding for mean + sd * z (nvcc
    contracts it into an fma)."""
    A = mean.shape[1]
    z, e_z = _normals(rows, call, seed, A, **wrong)
    mu, ls = mean.astype(np.float64), logstd.astype(np.float64)
    sd = np.exp(ls)
    e_sd = EXPF_ULP * ULP_REL * sd
    act = mu + sd * z
    e_pre = sd * e_z + e_sd * (np.abs(z) + e_z)
    return act, e_pre + U32 * (np.abs(act) + e_pre) + TINY


def _logprob_reference(act, mean, logstd):
    """fp64 log-density of Normal(mean, exp(logstd)) at the kernel's action, and the bound on the fp32 sum:
    q = (d*d) / (2*sd*sd) with d = act - mean (one rounding), sd = expf (2 ulp), three products and a division
    carries 15 roundings; each of the A terms - q - logstd - 0.5 log 2 pi, and the running sum, one per addition
    (the fp32 constant 0.5 log 2 pi is within one rounding of its value)."""
    d = act.astype(np.float64) - mean.astype(np.float64)
    ls = logstd.astype(np.float64)
    q = d * d / (2.0 * np.exp(2.0 * ls))
    A = act.shape[1]
    lp = (-q - ls - HALF_LOG_2PI).sum(1)
    terms = (q + np.abs(ls) + HALF_LOG_2PI).sum(1)
    return lp, 15 * U32 * q.sum(1) + (A + 3) * U32 * terms + TINY


def _check_sample(act, lp, mean, logstd, ref, what):
    act, lp, mean, logstd = (t.detach().cpu().numpy() for t in (act, lp, mean, logstd))
    a_ref, a_bound = ref
    ra = (np.abs(act.astype(np.float64) - a_ref) / a_bound).max()
    assert ra <= 1.0, f"{what}: action max err/bound = {ra:.4g}"
    l_ref, l_bound = _logprob_reference(act, mean, logstd)
    rl = (np.abs(lp.astype(np.float64) - l_ref) / l_bound).max()
    assert rl <= 1.0, f"{what}: log-prob max err/bound = {rl:.4g}"
    return max(ra, rl), ra, rl


def _assert_teeth(act, mean, logstd, rows, call, seed, what):
    """The bound rejects the references of the wrong call index, row, cos / sin order and block order."""
    act = act.detach().cpu().numpy().astype(np.float64)
    mean, logstd = mean.detach().cpu().numpy(), logstd.detach().cpu().numpy()
    wrongs = {"call - 1": dict(call=call - 1), "call + 1": dict(call=call + 1), "row + 1": dict(rows=rows + 1),
              "cos / sin swapped": dict(swap_cs=True)}
    if mean.shape[1] == 6:
        wrongs["blocks 0 and 1 exchanged"] = dict(swap_blocks=True)
    for name, w in wrongs.items():
        kw = dict(rows=rows, call=call)
        kw.update({k: v for k, v in w.items() if k in kw})
        ref, bound = _sample_reference(mean, logstd, kw["rows"], kw["call"], seed,
                                       **{k: v for k, v in w.items() if k not in kw})
        frac = (np.abs(act - ref) > bound).mean()
        assert frac > 0.99, f"{what}: the bound rejects the {name} reference at only {100 * frac:.2f} % of the elements"


SAMPLE_MS = (1, 255, 257, 65535, 131040)
COUNTERS = (0, 5, -3)   # -3 = 0xFFFFFFFD: with call_offset 5 the fused call index wraps to 2


@pytest.mark.parametrize("A", [2, 6])
def test_policy_sample_against_the_philox_reference(A):
    """vss_policy_sample (k_policy_sample<A>): call index = the counter word, advanced by one per call (mod 2^32)."""
    from rsoccer_isaac_cleanrl_b200.engine import policy_sample
    logstd = torch.linspace(-0.7, 0.2, A, device="cuda")
    worst = (0.0, 0.0)
    for M in SAMPLE_MS:
        mean = torch.randn(M, A, device="cuda", generator=_gen(M + A)) * 2
        for c in COUNTERS:
            ctr = torch.full((1,), c, device="cuda", dtype=torch.int32)
            act, lp = policy_sample(mean, logstd, SEED, ctr)
            assert int(ctr.item()) == c + 1
            rows = np.arange(M)
            ref = _sample_reference(mean.cpu().numpy(), logstd.cpu().numpy(), rows, c % 2 ** 32, SEED)
            _, ra, rl = _check_sample(act, lp, mean, logstd, ref, f"policy_sample A={A} M={M} counter={c}")
            worst = (max(worst[0], ra), max(worst[1], rl))
            if M == 65535 and c != 5:
                _assert_teeth(act, mean, logstd, rows, c % 2 ** 32, SEED, f"policy_sample A={A} counter={c}")
    print(f"[err/bound] policy_sample A={A}: action {worst[0]:.4g}, log-prob {worst[1]:.4g}")


FUSED_MODES = [(ew, critic, store) for ew in (4, 8) for critic in (False, True) for store in (True, False)]


@pytest.mark.parametrize("A", [2, 6])
def test_fused_sampling_against_the_philox_reference(A):
    """The fused forward's sampling (network 0 = the actor): call index = counter + call_offset (mod 2^32), the
    counter is not advanced; every (epilogue warps, with / without the critic, mean stored or not) mode at several
    sizes, each mode at least twice. The mean is the fused kernel's own output (checked in (A))."""
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused
    actor, critic = _mlp(A, 60 + A), _mlp(1, 61)
    logstd = torch.linspace(-0.7, 0.2, A, device="cuda")
    worst, k = (0.0, 0.0), 0
    seen = set()
    for M in SAMPLE_MS:
        x16 = _x16(M, M + 3)
        means = {ew: mlp_forward_fused(x16, [_net(actor)], epilogue_warps=ew)[0] for ew in (4, 8)}
        for c in COUNTERS:
            ew, with_critic, store = FUSED_MODES[k % len(FUSED_MODES)]
            k += 1
            seen.add((ew, with_critic, store))
            ctr = torch.full((1,), c, device="cuda", dtype=torch.int32)
            act, lp = torch.empty((M, A), device="cuda"), torch.empty(M, device="cuda")
            samp = dict(logstd=logstd, counter=ctr, seed=SEED, call_offset=5, action=act, logprob=lp)
            nets = [_net(actor, out=None if store else False)] + ([_net(critic)] if with_critic else [])
            outs = mlp_forward_fused(x16, nets, epilogue_warps=ew, sampling=samp)
            assert int(ctr.item()) == c
            if store:
                _assert_bits(outs[0], means[ew], f"stored mean EW={ew} M={M}")
            else:
                assert outs[0] is None
            what = f"fused A={A} M={M} counter={c} EW={ew} critic={with_critic} store={store}"
            call = (c + 5) % 2 ** 32
            ref = _sample_reference(means[ew].cpu().numpy(), logstd.cpu().numpy(), np.arange(M), call, SEED)
            _, ra, rl = _check_sample(act, lp, means[ew], logstd, ref, what)
            worst = (max(worst[0], ra), max(worst[1], rl))
            if M == 65535:
                _assert_teeth(act, means[ew], logstd, np.arange(M), call, SEED, what)
    assert seen == set(FUSED_MODES), sorted(set(FUSED_MODES) - seen)
    print(f"[err/bound] fused sampling A={A}: action {worst[0]:.4g}, log-prob {worst[1]:.4g}")


# ---------------------------------------------------------------------------------------------------------------
# (C) the rollout's stream
# ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("env_id,N", [("sa", 700), ("cma", 16384)])
def test_rollout_actions_logprobs_and_values_follow_the_sampling_stream(env_id, N):
    """ppo.train with a zero learning rate (the hook sees the weights the rollout used): for every step t of update u,
    the actions and log-probs are the reference draws on the fused actor mean of the recorded observation, seed
    args.seed + 7919, call index T (u - 1) + t; the values are the fused critic's bits. Update 1 runs eagerly,
    update 2 is captured and replayed, update 3 replayed. sa with 700 envs: one launch for both networks; cma with
    16 384 envs (A = 6): 256 CTAs, more than the SMs, so the critic runs in its own launch on the side stream."""
    from rsoccer_isaac_cleanrl_b200 import ppo
    from rsoccer_isaac_cleanrl_b200.engine import gather_pad_bf16, mlp_forward_fused
    from rsoccer_isaac_cleanrl_b200.tc_mlp import MlpWeights
    T = 4
    args = ppo.parse_args(["--env-id", env_id, "--num-envs", str(N), "--num-steps", str(T), "--total-timesteps",
                           str(T * N * 3), "--update-epochs", "1", "--quiet", "--seed", "11", "--learning-rate", "0"])
    one_launch = 2 * ((N + 127) // 128) <= torch.cuda.get_device_properties(0).multi_processor_count
    assert one_launch == (env_id == "sa")
    seen = []

    def hook(update, t):
        ag = t["agent"]
        mw_a, mw_c = MlpWeights(ag.actor_mean), MlpWeights(ag.critic)
        logstd = ag.actor_logstd.detach().reshape(-1).contiguous()
        worst = 0.0
        for s in range(T):
            x16 = gather_pad_bf16(t["obs"][s].contiguous(), None, 64)
            mean, value = mlp_forward_fused(x16, [_net(mw_a), _net(mw_c)])
            _assert_bits(t["values"][s], value.view(-1), f"{env_id} update {update} step {s}: values")
            call = T * (update - 1) + s
            ref = _sample_reference(mean.cpu().numpy(), logstd.cpu().numpy(), np.arange(N), call, args.seed + 7919)
            worst = max(worst, _check_sample(t["actions"][s], t["logprobs"][s], mean, logstd, ref,
                                             f"{env_id} update {update} step {s}")[0])
        seen.append((update, worst))

    stats = ppo.train(args, hook=hook)
    assert stats["updates"] == 3 and [u for u, _ in seen] == [1, 2, 3]
    print(f"[err/bound] rollout {env_id} N={N}: " + ", ".join(f"update {u} {w:.4g}" for u, w in seen))


# ---------------------------------------------------------------------------------------------------------------
# (E) coverage
# ---------------------------------------------------------------------------------------------------------------
def test_the_cases_reach_every_kernel_instantiation():
    """The calls of the cases above launch k_mlp_fwd<4>, k_mlp_fwd<8>, k_policy_sample<2>, k_policy_sample<6>,
    k_ppo_loss<2>, k_ppo_loss<6> and k_adv_stats."""
    from torch.profiler import ProfilerActivity, profile
    from rsoccer_isaac_cleanrl_b200.engine import mlp_forward_fused, policy_sample, ppo_loss
    actor = _mlp(6, 5)
    x16 = _x16(300, 1)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for ew in (4, 8):
            mlp_forward_fused(x16, [_net(actor)], epilogue_warps=ew)
        for A in (2, 6):
            mean = torch.randn(300, A, device="cuda")
            logstd = torch.zeros(A, device="cuda")
            policy_sample(mean, logstd, 1, torch.zeros(1, device="cuda", dtype=torch.int32))
            v = torch.randn(300, 1, device="cuda")
            ppo_loss(mean, v, logstd, mean.clone(), torch.randn(300, device="cuda"), torch.randn(300, device="cuda"),
                     torch.randn(300, device="cuda"), None, None, 0.2, 0.0, 0.5, True, False,
                     torch.zeros(A, device="cuda"))
        torch.cuda.synchronize()
    names = {re.sub(r"\s+", "", e.name) for e in prof.events()}
    found = set()
    for nm in names:
        for pat in (r"k_mlp_fwd<\d+>", r"k_policy_sample<\d+>", r"k_ppo_loss<\d+>", r"k_adv_stats"):
            found.update(re.findall(pat, nm))
    want = {"k_mlp_fwd<4>", "k_mlp_fwd<8>", "k_policy_sample<2>", "k_policy_sample<6>", "k_ppo_loss<2>",
            "k_ppo_loss<6>", "k_adv_stats"}
    assert want <= found, ("not launched:", sorted(want - found), "launched:", sorted(found))
    print("[coverage] launched:", ", ".join(sorted(found & want)))
