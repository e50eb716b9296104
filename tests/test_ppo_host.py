"""CPU: host-side PPO logic against golden vectors from the reference's own script."""
import json
import os
import sys
import types

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from rsoccer_isaac_cleanrl_b200 import ppo

sys.path.insert(0, GOLDEN)
import make_golden as mg  # noqa: E402  (checksum helpers only; the reference is not read here)


def test_cli_flags_and_defaults_match_reference():
    g = json.load(open(os.path.join(GOLDEN, "ppo_defaults.json")))
    mine = vars(ppo.parse_args([]))
    for k, v in g["defaults"].items():
        assert k in mine, k
        assert mine[k] == v, (k, mine[k], v)
    mine2 = vars(ppo.parse_args(["--env-id", "dma", "--num-envs", "65535", "--num-steps", "64", "--anneal-lr",
                                 "--norm-adv", "false"]))
    for k, v in g["dma_case"].items():
        assert mine2[k] == v, (k, mine2[k], v)


def _envs(adim):
    return types.SimpleNamespace(single_observation_space=types.SimpleNamespace(shape=(52,)),
                                 single_action_space=types.SimpleNamespace(shape=(adim,)))


def test_agent_state_dict_loads_reference_checkpoint_and_matches_outputs():
    z = np.load(os.path.join(GOLDEN, "agent.npz"))
    # the hidden 256/512-wide weights are not stored: rebuilt from the generator's seed with this Agent (same layer
    # order and initialisers), then pinned to the reference's by per-tensor checksum and a strided sample; one
    # thread, as the generator ran: orthogonal_'s QR rounds differently with more
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        torch.manual_seed(3)
        rebuilt = ppo.Agent(_envs(2)).state_dict()
    finally:
        torch.set_num_threads(threads)
    sd = {k[len("a2_sd_"):]: torch.from_numpy(z[k]) for k in z.files if k.startswith("a2_sd_")}
    for k in (k[len("a2_sum_"):] for k in z.files if k.startswith("a2_sum_")):
        np.testing.assert_allclose(mg.weight_checksum(rebuilt[k]), z[f"a2_sum_{k}"], rtol=1e-9, err_msg=k)
        np.testing.assert_array_equal(mg.weight_sample(rebuilt[k]), z[f"a2_sample_{k}"], err_msg=k)
        sd[k] = rebuilt[k]
    agent = ppo.Agent(_envs(2))
    assert set(sd) == set(agent.state_dict())           # same keys as the reference's Agent
    agent.load_state_dict(sd, strict=True)
    x, action = torch.from_numpy(z["a2_x"]), torch.from_numpy(z["a2_action"])
    _, logp, ent, value = agent.get_action_and_value(x, action)
    np.testing.assert_allclose(agent.actor_mean(x).detach().numpy(), z["a2_mean"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(logp.detach().numpy(), z["a2_logp"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(ent.detach().numpy(), z["a2_ent"], rtol=1e-6, atol=1e-6)
    np.testing.assert_allclose(value.detach().numpy(), z["a2_value"], rtol=1e-5, atol=1e-6)
    # the same scalar loss -> the same gradients
    adv, ret = torch.from_numpy(z["a2_adv"]), torch.from_numpy(z["a2_ret"])
    loss = (-(adv * logp.exp())).mean() - 0.005 * ent.mean() + 4 * 0.5 * ((value.view(-1) - ret) ** 2).mean()
    np.testing.assert_allclose(loss.item(), float(z["a2_loss"]), rtol=1e-5)
    agent.zero_grad()
    loss.backward()
    for k, p in agent.named_parameters():
        gn = float(np.sqrt((p.grad.numpy().astype(np.float64) ** 2).sum()))
        assert gn == pytest.approx(float(z[f"a2_gradnorm_{k}"]), rel=1e-4, abs=1e-7), k
        if f"a2_grad_{k}" in z.files:
            np.testing.assert_allclose(p.grad.numpy(), z[f"a2_grad_{k}"], rtol=1e-4, atol=1e-6)


def test_orthogonal_init_shapes_and_gains():
    torch.manual_seed(0)
    a = ppo.Agent(_envs(6))
    assert a.actor_mean[8].weight.shape == (6, 256) and a.critic[8].weight.shape == (1, 256)
    assert sum(p.numel() for p in a.parameters()) == 1080077  # SURVEY a17 (A=6)
    w = a.critic[2].weight.detach()                              # 512x256, orthogonal columns * sqrt(2)
    np.testing.assert_allclose((w.t() @ w).numpy(), 2 * np.eye(256), atol=1e-4)
    assert float(a.actor_mean[8].weight.abs().max()) < 0.01 and float(a.actor_logstd.abs().max()) == 0


def test_flat_parameters_and_adam_match_torch():
    torch.manual_seed(1)
    a, b = ppo.Agent(_envs(2)), ppo.Agent(_envs(2))
    b.load_state_dict(a.state_dict())
    flat, flat_grad = ppo.flatten_parameters(a)
    opt_a = ppo.FlatAdam(flat, flat_grad, lr=1e-3, eps=1e-5)
    opt_b = torch.optim.Adam(b.parameters(), lr=1e-3, eps=1e-5)
    x = torch.randn(64, 52)
    for it in range(3):
        for agent in (a, b):
            _, logp, ent, v = agent.get_action_and_value(x, torch.zeros(64, 2))
            loss = logp.mean() + v.pow(2).mean() - 0.01 * ent.mean()
            if agent is a:
                flat_grad.zero_()
            else:
                opt_b.zero_grad()
            loss.backward()
        gn = torch.linalg.vector_norm(flat_grad)
        flat_grad.mul_(torch.clamp(1.5 / (gn + 1e-6), max=1.0))
        torch.nn.utils.clip_grad_norm_(b.parameters(), 1.5)
        opt_a.step(); opt_b.step()
    for (k, pa), (_, pb) in zip(a.named_parameters(), b.named_parameters()):
        np.testing.assert_allclose(pa.detach().numpy(), pb.detach().numpy(), rtol=2e-5, atol=2e-6, err_msg=k)


def test_episode_returns_mapping_matches_the_reference_dict():
    """envs/wrappers.py:76-83 of the reference: infos["r"] = {goal, grad, move, energy, return = sum(1)}; here the four
    components are views and "return" is computed when read."""
    import torch
    from rsoccer_isaac_cleanrl_b200.envs.wrappers import _EpisodeReturns
    r = torch.arange(12, dtype=torch.float32).view(3, 4)
    m = _EpisodeReturns(r)
    assert set(m.keys()) == {"goal", "grad", "move", "energy", "return"} and "return" in m and "nope" not in m
    assert torch.equal(m["goal"], r[:, 0]) and torch.equal(m["energy"], r[:, 3])
    assert torch.equal(m["return"], r.sum(1)) and torch.equal(m.get("return"), r.sum(1)) and m.get("nope") is None
    r[0, 0] = 100.0   # views of the live statistics buffer, like the reference's slices
    assert float(m["goal"][0]) == 100.0 and float(m["return"][0]) == 100.0 + 1 + 2 + 3
    with __import__("pytest").raises(KeyError):
        m["nope"]
