"""GPU: the fused PPO pieces (csrc/ppo_ops.cu) against plain PyTorch fp32 references of the same
expressions — the reference's own formulas (ppo_continuous_action_isaacgym.py:155-164, 314-354)
evaluated with torch autograd / torch.optim.Adam. Tolerances are fp32 rounding (1e-5 relative)."""
import math
import os
import types

import numpy as np
import pytest

from oracle import ppo_oracle as po

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _close(a, b, rtol=2e-5, atol=1e-6):
    err = (a - b).abs().max().item()
    lim = atol + rtol * b.abs().max().item()
    assert err <= lim, (err, lim)


@pytest.mark.parametrize("A", [2, 6])
def test_policy_sample_matches_normal_log_prob_and_is_standard_normal(A):
    from rsoccer_isaac_cleanrl_b200.engine import policy_sample
    M = 200_003
    g = torch.Generator(device="cuda").manual_seed(1)
    mean = torch.randn(M, A, device="cuda", generator=g)
    logstd = torch.linspace(-1.0, 0.5, A, device="cuda")
    ctr = torch.zeros(1, device="cuda", dtype=torch.int32)
    act, lp = policy_sample(mean, logstd, 1234, ctr)
    assert ctr.item() == 1
    dist = torch.distributions.Normal(mean, logstd.exp().expand_as(mean))
    _close(lp, dist.log_prob(act).sum(1), rtol=1e-5, atol=2e-5)
    z = (act - mean) / logstd.exp()
    assert abs(z.mean().item()) < 5e-3 and abs(z.std().item() - 1.0) < 5e-3
    assert abs((z ** 3).mean().item()) < 2e-2 and abs((z ** 4).mean().item() - 3.0) < 5e-2
    # columns are independent draws; a second call draws fresh noise; same counter -> same noise
    assert abs((z[:, 0] * z[:, 1]).mean().item()) < 1e-2  # 4.5 sigma at this M
    act2, _ = policy_sample(mean, logstd, 1234, ctr)
    assert ctr.item() == 2 and (act2 != act).float().mean().item() > 0.99
    ctr.fill_(0)
    act3, lp3 = policy_sample(mean, logstd, 1234, ctr)
    assert torch.equal(act3, act) and torch.equal(lp3, lp)


def _torch_loss(mean, value, logstd, act, old_lp, adv, ret, old_v, clip, ent_coef, vf_coef, norm_adv, clip_vloss):
    """ppo…:314-352 verbatim in torch."""
    std = logstd.exp().expand_as(mean)
    dist = torch.distributions.Normal(mean, std)
    newlogprob, entropy = dist.log_prob(act).sum(1), dist.entropy().sum(1)
    logratio = newlogprob - old_lp
    ratio = logratio.exp()
    old_kl, kl = (-logratio).mean(), ((ratio - 1) - logratio).mean()
    clipfrac = ((ratio - 1.0).abs() > clip).float().mean()
    if norm_adv:
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    pg_loss = torch.max(-adv * ratio, -adv * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    newvalue = value.view(-1)
    if clip_vloss:
        v_un = (newvalue - ret) ** 2
        v_cl = old_v + torch.clamp(newvalue - old_v, -clip, clip)
        v_loss = 0.5 * torch.max(v_un, (v_cl - ret) ** 2).mean()
    else:
        v_loss = 0.5 * ((newvalue - ret) ** 2).mean()
    ent = entropy.mean()
    loss = pg_loss - ent_coef * ent + v_loss * vf_coef
    return loss, dict(pg_loss=pg_loss, v_loss=v_loss, entropy=ent, old_approx_kl=old_kl, approx_kl=kl,
                      clipfrac=clipfrac, loss=loss)


@pytest.mark.parametrize("A,norm_adv,clip_vloss", [(2, True, False), (6, True, False), (2, False, True), (6, True, True)])
def test_ppo_loss_and_gradients_match_torch_autograd(A, norm_adv, clip_vloss):
    from rsoccer_isaac_cleanrl_b200.engine import PPO_STATS, ppo_loss
    R, B = 50_000, 16_411
    g = torch.Generator(device="cuda").manual_seed(3)
    rn = lambda *s: torch.randn(*s, device="cuda", generator=g)
    b_act, b_lp, b_adv, b_ret, b_val = rn(R, A), rn(R) * 0.3 - 2.0, rn(R) * 2 + 0.5, rn(R), rn(R)
    inds = torch.randperm(R, device="cuda", generator=g)[:B]
    mean = (b_act[inds] + 0.3 * rn(B, A)).requires_grad_()
    value = (b_val[inds] + 0.4 * rn(B)).view(B, 1).requires_grad_()
    logstd = torch.linspace(-0.3, 0.2, A, device="cuda").requires_grad_()
    # old log-probs near the new ones so that ratios straddle the clip range
    with torch.no_grad():
        d = torch.distributions.Normal(mean, logstd.exp().expand_as(mean))
        b_lp[inds] = d.log_prob(b_act[inds]).sum(1) + 0.25 * rn(B)
    loss, ref = _torch_loss(mean, value, logstd, b_act[inds], b_lp[inds], b_adv[inds], b_ret[inds], b_val[inds],
                            0.2, 0.005, 4.0, norm_adv, clip_vloss)
    loss.backward()
    d_logstd = torch.zeros(A, device="cuda")
    d_mean, d_value, stats = ppo_loss(mean.detach(), value.detach(), logstd.detach(), b_act, b_lp, b_adv, b_ret,
                                      b_val if clip_vloss else None, inds, 0.2, 0.005, 4.0, norm_adv, clip_vloss,
                                      d_logstd)
    for k, name in enumerate(PPO_STATS):
        if name == "clipfrac":  # a ratio within rounding of the clip boundary may fall on either side
            assert abs(stats[k].item() - ref[name].item()) <= 3.0 / B
        else:
            _close(stats[k], ref[name].detach(), rtol=3e-5, atol=2e-6)
    _close(d_mean, mean.grad, rtol=1e-4, atol=1e-9)
    _close(d_value, value.grad, rtol=1e-4, atol=1e-9)
    _close(d_logstd, logstd.grad, rtol=2e-4, atol=1e-6)
    # without an index array the rows are taken in order
    d_logstd2 = torch.zeros(A, device="cuda")
    d_mean2, _, stats2 = ppo_loss(mean.detach(), value.detach(), logstd.detach(), b_act[inds].contiguous(),
                                  b_lp[inds].contiguous(), b_adv[inds].contiguous(), b_ret[inds].contiguous(),
                                  b_val[inds].contiguous(), None, 0.2, 0.005, 4.0, norm_adv, clip_vloss, d_logstd2)
    _close(d_mean2, d_mean, rtol=1e-6)
    _close(stats2[:7], stats[:7], rtol=1e-5, atol=1e-6)  # (same kernel, same arithmetic per row)


def test_convert_bf16_batch_copies_pads_and_transposes():
    from rsoccer_isaac_cleanrl_b200.engine import convert_bf16_batch
    g = torch.Generator(device="cuda").manual_seed(5)
    shapes = [(256, 52), (512, 256), (512, 512), (256, 512), (33, 70)]
    srcs = [torch.randn(s, device="cuda", generator=g) for s in shapes]
    plain = [torch.full((s[0], (s[1] + 63) // 64 * 64), 7.0, device="cuda", dtype=torch.bfloat16) for s in shapes]
    trans = [torch.full((s[1], s[0] + 3), 7.0, device="cuda", dtype=torch.bfloat16) for s in shapes]
    convert_bf16_batch([(s, d, False) for s, d in zip(srcs, plain)] + [(s, d, True) for s, d in zip(srcs, trans)])
    for s, p, t in zip(srcs, plain, trans):
        R, C = s.shape
        assert torch.equal(p[:, :C], s.to(torch.bfloat16)) and (p[:, C:] == 7.0).all()
        assert torch.equal(t[:, :R], s.t().to(torch.bfloat16)) and (t[:, R:] == 7.0).all()


@pytest.mark.parametrize("scale,max_norm", [(1.0, 1.5), (0.5, 1e9)])
def test_clip_adam_matches_torch_clip_grad_norm_and_adam(scale, max_norm):
    from rsoccer_isaac_cleanrl_b200.ppo import FlatAdam
    n = 1_080_077
    g = torch.Generator(device="cuda").manual_seed(7)
    p0 = torch.randn(n, device="cuda", generator=g)
    ref_p = torch.nn.Parameter(p0.clone())
    ref_opt = torch.optim.Adam([ref_p], lr=1e-3, eps=1e-5)
    flat, grad = p0.clone(), torch.zeros(n, device="cuda")
    opt = FlatAdam(flat, grad, lr=1e-3, eps=1e-5)
    for it in range(5):
        gr = torch.randn(n, device="cuda", generator=g) * (10.0 if it % 2 == 0 else 1e-4)
        if it == 3:
            opt.param_groups[0]["lr"] = 5e-4
            ref_opt.param_groups[0]["lr"] = 5e-4
            opt.sync_lr()
        ref_p.grad = gr * scale
        torch.nn.utils.clip_grad_norm_([ref_p], max_norm)
        ref_opt.step()
        grad.copy_(gr)
        opt.clip_and_step_fused(max_norm, scale)
        _close(grad, ref_p.grad, rtol=1e-5, atol=1e-12)
        _close(flat, ref_p.detach(), rtol=0, atol=2e-6)
    assert opt.t.item() == 5.0


def test_explicit_mlp_training_path_matches_the_autograd_function():
    """forward_explicit / backward_explicit (no autograd, gradients accumulated straight into .grad)
    against TCMlp.apply + loss.backward() on the same weights and inputs."""
    from rsoccer_isaac_cleanrl_b200 import ppo, tc_mlp
    from rsoccer_isaac_cleanrl_b200.engine import gather_pad_bf16
    envs = types.SimpleNamespace(single_observation_space=types.SimpleNamespace(shape=(52,)),
                                 single_action_space=types.SimpleNamespace(shape=(6,)))
    torch.manual_seed(0)
    a = ppo.Agent(envs, "tc").cuda()
    b = ppo.Agent(envs, "tc").cuda()
    with torch.no_grad():
        a.actor_mean[8].weight.mul_(30.0)
    b.load_state_dict(a.state_dict())
    M = 8192 + 13
    pool = torch.randn(3 * M, 52, device="cuda")
    inds = torch.randperm(3 * M, device="cuda")[:M]
    dout = torch.randn(M, 6, device="cuda") / M
    out_a = tc_mlp.mlp_forward(a.actor_mean, pool[inds])
    out_a.backward(dout)
    flat, flat_grad = ppo.flatten_parameters(b)
    mw = tc_mlp.MlpWeights(b.actor_mean)
    out_b, hs = tc_mlp.forward_explicit(mw, gather_pad_bf16(pool, inds, mw.k0))
    tc_mlp.backward_explicit(mw, hs, dout)
    assert torch.equal(out_a.detach(), out_b)
    for (k, pa), (_, pb) in zip(a.actor_mean.named_parameters(), b.actor_mean.named_parameters()):
        num = (pa.grad - pb.grad).norm().item()
        assert num <= 1e-4 * pa.grad.norm().item() + 1e-12, (k, num)
    # a second backward accumulates
    tc_mlp.backward_explicit(mw, hs, dout)
    for (k, pa), (_, pb) in zip(a.actor_mean.named_parameters(), b.actor_mean.named_parameters()):
        assert (2 * pa.grad - pb.grad).norm().item() <= 2e-4 * pa.grad.norm().item() + 1e-12, k
    assert math.isfinite(flat_grad.norm().item())


GOLD = os.path.join(os.path.dirname(__file__), "golden", "ppo_update.npz")


@pytest.mark.parametrize("name,clip_vloss", [("a2", False), ("a6v", True)])
def test_ppo_loss_kernel_against_the_reference_update_golden(name, clip_vloss):
    """vss_ppo_loss on the inputs / fresh network outputs recorded while executing the reference's own
    minibatch code (ppo…:314-352): statistics and d loss / d (mean, value, logstd)."""
    from rsoccer_isaac_cleanrl_b200.engine import ppo_loss
    g = np.load(GOLD)
    k = lambda s_: torch.from_numpy(g[f"{name}_{s_}"]).cuda()
    A = k("logstd").numel()
    d_logstd = torch.zeros(A, device="cuda")
    d_mean, d_value, st = ppo_loss(k("mean").contiguous(), k("value").contiguous(), k("logstd"), k("b_actions"),
                                   k("b_logprobs"), k("b_advantages"), k("b_returns"), k("b_values"), k("mb_inds"),
                                   0.2, 0.005, 4.0, True, clip_vloss, d_logstd)
    ref = [g[f"{name}_{s_}"] for s_ in ("pg_loss", "v_loss", "entropy_loss", "old_approx_kl", "approx_kl", "clipfrac", "loss")]
    for i, r in enumerate(ref):
        assert abs(st[i].item() - float(r)) <= 3e-6 + 3e-5 * abs(float(r)), (i, st[i].item(), float(r))
    _close(d_mean, k("d_mean"), rtol=1e-4, atol=1e-9)
    _close(d_value, k("d_value"), rtol=1e-4, atol=1e-9)
    _close(d_logstd, k("d_logstd"), rtol=2e-4, atol=1e-7)


U32 = 2.0 ** -24   # unit roundoff of fp32
LOSS_GRID_ROWS = 148 * 4 * 256   # rows one pass of the vss_ppo_loss grid covers (592 blocks x 256 threads)


def _loss_sum_bounds(r, mean, value, logstd, b_act, b_lp, b_adv, b_ret, b_val, inds, clip, ent_coef, vf_coef,
                     norm_adv, clip_vloss):
    """Bounds on |kernel - oracle| of the statistics and d_logstd of vss_ppo_loss, from sums of |terms| in fp64.

    Each row's terms carry their own fp32 error (the log-probability, the ratio, the normalised advantage) and the
    sums add one rounding per addition on the longest chain: the rows of one thread in the grid-stride loop, the
    5-level warp tree, the 8 warps of a block, then one atomicAdd per block (and the scaling by 1/B)."""
    f = lambda t: t.detach().double().cpu().numpy()   # noqa: E731
    mean, value, logstd = f(mean), f(value).reshape(-1), f(logstd)
    j = f(inds).astype(np.int64)
    act, old_lp, adv_raw, ret, v0 = f(b_act)[j], f(b_lp)[j], f(b_adv)[j], f(b_ret)[j], f(b_val)[j]
    B, A = mean.shape
    grid = min((B + 255) // 256, 148 * 4)
    chain = -(-B // (grid * 256)) + 5 + 8 + grid + 2
    iv = np.exp(-2.0 * logstd)
    d = act - mean
    q = 0.5 * d * d * iv
    lr = (-q - logstd - po.HALF_LOG_2PI).sum(1) - old_lp
    ratio = np.exp(lr)
    # |fp32 log-ratio - lr|: q = d*d*(0.5/sd^2) with sd = expf (2 ulp) carries 15 roundings, the A + 3 additions of
    # each row's sum one each (the fp32 constant 0.5 log 2 pi is within one rounding of its value)
    e_lr = (A + 20) * U32 * ((q + np.abs(logstd) + po.HALF_LOG_2PI).sum(1) + np.abs(old_lp))
    if norm_adv:
        amean, ainv = adv_raw.mean(), 1.0 / (adv_raw.std(ddof=1) + 1e-8)
        adv = (adv_raw - amean) * ainv
        e_adv = 3 * U32 * (np.abs(adv_raw) + abs(amean)) * ainv + 4 * U32 * np.abs(adv)
    else:
        adv, e_adv = adv_raw, np.zeros(B)
    lo, hi = 1.0 - clip, 1.0 + clip
    t1, t2 = -adv * ratio, -adv * np.clip(ratio, lo, hi)
    e_ratio = ratio * (e_lr + 4 * U32)                       # expf: 2 ulp
    terms = {"pg_loss": np.maximum(t1, t2), "old_approx_kl": -lr, "approx_kl": (ratio - 1.0) - lr}
    errs = {"pg_loss": np.abs(adv) * e_ratio + ratio * e_adv + 4 * U32 * np.abs(terms["pg_loss"]),
            "old_approx_kl": e_lr, "approx_kl": np.abs(ratio - 1.0) * e_lr + 6 * U32 * (ratio + 1.0 + np.abs(lr))}
    if clip_vloss:
        vc = v0 + np.clip(value - v0, -clip, clip)
        terms["v_loss"] = 0.5 * np.maximum((value - ret) ** 2, (vc - ret) ** 2)
    else:
        terms["v_loss"] = 0.5 * (value - ret) ** 2
    errs["v_loss"] = 8 * U32 * (np.abs(value) + np.abs(ret) + np.abs(v0) + clip) ** 2
    bounds = {}
    for k in terms:
        bounds[k] = (errs[k].sum() + chain * U32 * np.abs(terms[k]).sum()) / B + 2 * U32 * abs(r[k])
    ent_terms = np.abs(0.5 + po.HALF_LOG_2PI + logstd).sum()
    bounds["entropy"] = (A + 2) * U32 * ent_terms
    bounds["loss"] = (bounds["pg_loss"] + vf_coef * bounds["v_loss"] + ent_coef * bounds["entropy"] +
                      (2 * grid + 2) * U32 * (np.abs(terms["pg_loss"]).sum() / B +
                                              vf_coef * np.abs(terms["v_loss"]).sum() / B + ent_coef * ent_terms))
    # clipfrac: a ratio within its error of the clip boundary may fall on either side; the counts are exact
    near = (np.abs(np.abs(ratio - 1.0) - clip) <= e_ratio + 4 * U32).sum()
    bounds["clipfrac"] = (near + 8) / B + chain * U32 * r["clipfrac"]
    # d_logstd[k] = sum_i g_lp_i (d^2 / sd^2 - 1) - ent_coef: the row terms cancel, so the bound is on their |sum|
    inside = (ratio >= lo) & (ratio <= hi)
    g_lp = np.where(inside | (t1 > t2), -adv, 0.0) * ratio / B
    w = d * d * iv
    dls = g_lp[:, None] * (w - 1.0)
    e_dls = (np.abs(g_lp)[:, None] * ((e_lr + 8 * U32)[:, None] * np.abs(w - 1.0) + 16 * U32 * w) +
             (ratio * e_adv / B)[:, None] * np.abs(w - 1.0))
    # a row whose ratio is within its error of lo or hi may take the other gradient branch: its whole term
    flip = (np.abs(ratio - lo) <= e_ratio + 4 * U32) | (np.abs(ratio - hi) <= e_ratio + 4 * U32)
    e_flip = (np.abs(adv) * ratio / B)[flip, None] * np.abs(w[flip] - 1.0)
    bounds["d_logstd"] = (e_dls.sum(0) + e_flip.sum(0) + chain * U32 * np.abs(dls).sum(0) +
                          2 * U32 * (np.abs(r["d_logstd"]) + ent_coef))
    return bounds


def _loss_case(B, R, A, norm_adv, clip_vloss, ident=None):
    return pytest.param(B, R, A, norm_adv, clip_vloss, id=ident or f"B{B}-R{R}-{A}-{norm_adv}-{clip_vloss}")


# B = 131 072 (one pass of the grid); 131 040 (the default sa minibatch); 524 288 (cma: 16 384 envs x 128 steps / 4);
# 1 048 560 and 2 097 120 (dma, the reference's and the benchmark's): every thread of the grid takes 1, 4, 7 and 14 rows
@pytest.mark.parametrize("B,R,A,norm_adv,clip_vloss", [
    _loss_case(131_072, 524_288, 2, True, False, "2-True-False"),
    _loss_case(131_072, 524_288, 6, False, True, "6-False-True"),
    _loss_case(131_040, 524_160, 6, True, True),
    _loss_case(524_288, 2_097_152, 6, True, False),
    _loss_case(524_288, 2_097_152, 2, False, True),
    _loss_case(1_048_560, 4_194_240, 2, False, False),
    _loss_case(2_097_120, 8_388_480, 2, True, False),
    _loss_case(2_097_120, 8_388_480, 2, False, False),
])
def test_ppo_loss_kernel_against_the_numpy_oracle_at_minibatch_size(B, R, A, norm_adv, clip_vloss):
    """Statistics and gradients against the fp64 oracle. Above 151 552 rows each thread of the loss and advantage
    kernels walks the grid-stride loop more than once; the minibatch indices reach the last row of the rollout.
    The statistics and d_logstd are also checked within bounds from sums of |terms| (_loss_sum_bounds): the
    d_logstd sum cancels, so a bound relative to the result does not hold at two million rows."""
    from rsoccer_isaac_cleanrl_b200.engine import PPO_STATS, ppo_loss
    gen = torch.Generator(device="cuda").manual_seed(21)
    rn = lambda *s_: torch.randn(*s_, device="cuda", generator=gen)
    b_act, b_adv, b_ret, b_val = rn(R, A), rn(R) * 3 - 1, rn(R), rn(R)
    perm = torch.randperm(R, device="cuda", generator=gen)
    inds = perm[:B].clone()
    if not bool((inds == R - 1).any()):
        inds[B // 2] = R - 1
    assert int(inds.max()) == R - 1
    mean, value = b_act[inds] + 0.4 * rn(B, A), (b_val[inds] + 0.5 * rn(B)).view(B, 1).contiguous()
    logstd = torch.linspace(-0.6, 0.3, A, device="cuda")
    b_lp = rn(R)
    lp, _ = po.log_prob_and_entropy(mean.cpu().numpy(), logstd.cpu().numpy(), b_act[inds].cpu().numpy())
    b_lp[inds] = torch.from_numpy(lp).float().cuda() + 0.2 * rn(B)
    d_logstd = torch.zeros(A, device="cuda")
    d_mean, d_value, st = ppo_loss(mean, value, logstd, b_act, b_lp, b_adv, b_ret, b_val, inds, 0.2, 0.005, 4.0,
                                   norm_adv, clip_vloss, d_logstd)
    c = lambda t: t.cpu().numpy()
    r = po.ppo_loss(c(mean), c(value), c(logstd), c(b_act), c(b_lp), c(b_adv), c(b_ret), c(b_val), c(inds), 0.2, 0.005,
                    4.0, norm_adv, clip_vloss)
    bounds = _loss_sum_bounds(r, mean, value, logstd, b_act, b_lp, b_adv, b_ret, b_val, inds, 0.2, 0.005, 4.0,
                              norm_adv, clip_vloss)
    ratios = []
    for i, nm in enumerate(PPO_STATS):
        if B <= LOSS_GRID_ROWS:
            tol = 8.0 / B if nm == "clipfrac" else 3e-6 + 5e-5 * abs(r[nm])
            assert abs(st[i].item() - r[nm]) <= tol, (nm, st[i].item(), r[nm])
        ratios.append(abs(st[i].item() - r[nm]) / bounds[nm])
        assert ratios[-1] <= 1.0, (nm, st[i].item(), r[nm], bounds[nm])
    # element-wise: a ratio within fp32 rounding of the clip boundary may take the other branch
    bad = (np.abs(c(d_mean) - r["d_mean"]) > 1e-9 + 2e-4 * np.abs(r["d_mean"])).any(1)
    assert bad.mean() < 2e-5, bad.sum()
    np.testing.assert_allclose(c(d_value).reshape(-1), r["d_value"], rtol=2e-4, atol=1e-10)
    if B <= LOSS_GRID_ROWS:
        np.testing.assert_allclose(c(d_logstd), r["d_logstd"], rtol=5e-4, atol=1e-6)
    e_ls = np.abs(c(d_logstd) - r["d_logstd"]) / bounds["d_logstd"]
    assert (e_ls <= 1.0).all(), (c(d_logstd), r["d_logstd"], bounds["d_logstd"])
    print(f"[err/bound] ppo loss B={B} A={A} norm_adv={norm_adv} clip_vloss={clip_vloss}: statistics "
          f"{max(ratios):.3g}, d_logstd {e_ls.max():.3g}")


def test_clip_adam_kernel_against_the_numpy_oracle():
    from rsoccer_isaac_cleanrl_b200.ppo import FlatAdam
    n = 200_003
    gen = torch.Generator(device="cuda").manual_seed(9)
    p = torch.randn(n, device="cuda", generator=gen)
    grad = torch.zeros(n, device="cuda")
    opt = FlatAdam(p.clone(), grad, lr=3e-4, eps=1e-5)
    P, M, V, t = p.cpu().numpy().astype(np.float64), np.zeros(n), np.zeros(n), 0
    for it in range(4):
        g = torch.randn(n, device="cuda", generator=gen) * (3.0 if it < 2 else 1e-3)
        grad.copy_(g)
        opt.clip_and_step_fused(1.5, 0.25)
        P, gc, M, V, t = po.clip_adam(P, g.cpu().numpy(), M, V, t, 3e-4, 1.5, grad_scale=0.25)
        np.testing.assert_allclose(grad.cpu().numpy(), gc, rtol=2e-5, atol=1e-12)
        np.testing.assert_allclose(opt.flat.cpu().numpy(), P, rtol=0, atol=3e-6)
