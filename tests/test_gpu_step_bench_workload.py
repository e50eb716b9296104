"""B200: the full-contract step at the benchmark's own workload (bench.py's value leg).

bench.make_task builds 2^20 fields with the reset flags cleared and the progress counters staggered over [0, 400), then
bench.py issues 50 + 400 `VSS.step` launches back to back, cycling four action tensors, with nothing in the stream
between them. At that size the step runs as `k_step<…, sync=true>`: 32-field tiles, 4 warps per CTA, 8 192 CTAs (about
nine waves of 148 x 6) and the first-wave stagger. This file checks that workload as it is timed:

  * back to back == host-synchronised after every launch, bit for bit (state and outputs after step 450);
  * every other launch shape computes the same words at every one of the 450 steps;
  * chosen steps of the window against the oracle, all fields, in host chunks keyed by their global field id;
  * the injected-state step at 2^20 fields, bit-exact;
  * no output row is written outside its buffer slice, and none inside it is left unwritten.

Both sizes: 2^20, and 2^20 - 77 (a ragged last tile and a partly filled last CTA at the same shape).
"""
import numpy as np
import pytest

import parity_checks as pc
from oracle import vss_oracle as orc

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

WARMUP, TIMED = 50, 400            # bench.py's defaults: --warmup 50 --steps 400
STEPS = WARMUP + TIMED
SIZES = [1 << 20, (1 << 20) - 77]
SIZE_IDS = ["2^20", "2^20-77"]
# forced (warps per tile, fields per tile): one warp per 8- and 16-field tile (k_step, 4 warps per CTA), and k_step_cta
SHAPES = [(1, 8), (1, 16), (8, 32)]
# host chunks of the oracle comparison; a wave of the benchmark's shape is 148 x 6 CTAs of 128 fields
CHUNK = 131072
WAVE_FIELDS = 148 * 6 * 128
# what the per-step checksums cover: the state words, then VSS.step's outputs
SUM_NAMES = ("state", "obs", "term_obs", "rew", "reset", "time_outs", "progress")


_POS = {}


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    yield
    _POS.clear()   # the checksum weights: up to 2.6 GB of device memory
    torch.cuda.empty_cache()


def word_sum(t):
    """Position-weighted 64-bit sum of the int32 words of `t` (one-byte values widened to a word), on t's device:
    sum_i (i + 1) * w_i, wrapping modulo 2^64. Any changed word or any swap of two different words changes it."""
    w = t.reshape(-1)
    w = w.view(torch.int32) if w.element_size() >= 4 else w.to(torch.int32)
    k = w.numel()
    pos = _POS.get(w.device)
    if pos is None or pos.numel() < k:
        pos = _POS[w.device] = torch.arange(1, k + 1, dtype=torch.int64, device=w.device)
    return (w.to(torch.int64) * pos[:k]).sum()


def step_outputs(out):
    """(obs, terminal obs, rewards, reset flags, time-outs, progress) of one `VSS.step` return value."""
    obs, rew, reset, extras = out
    return (obs["obs"], extras["terminal_observation"], rew, reset, extras["time_outs"], extras["progress_buffer"])


def step_sums(envs, out):
    return torch.stack([word_sum(x) for x in (envs.engine.get_state(),) + step_outputs(out)])


def bits_equal(a, b):
    a, b = a.reshape(-1), b.reshape(-1)
    if a.element_size() >= 4:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return a.shape == b.shape and torch.equal(a, b)


def compare_with_oracle(p, seed, pre_state, pre_reset, actions, post, n, what, chunk=CHUNK):
    """One full-contract step against the oracle, from the state the step started from, in host chunks of `chunk`
    fields: the oracle is field-independent and keys its RNG by global field id, so chunk [c0, c1) is stepped with
    global offset c0. `post` = (obs, term_obs, rew, reset, time_outs, progress) as the step left them (tensors on any
    device). Returns the field count outside the physics tolerance and the chunks compared."""
    flips, chunks = 0, []
    for c0 in range(0, n, chunk):
        c1 = min(n, c0 + chunk)
        m = c1 - c0
        st = orc.State.from_soa(pre_state[:, c0:c1].cpu().numpy(), m)
        rb_ref = pre_reset[c0:c1].cpu().numpy().copy()   # the oracle updates the flags in place
        ref = orc.step(p, seed, c0, st, actions[c0:c1].cpu().numpy(), rb_ref)
        obs, tobs, rew, rb, tmo, prog = (x[c0:c1].cpu().numpy() for x in post)
        out = dict(obs=obs, term_obs=tobs, rew=rew, timeout=tmo.astype(np.uint8), progress_f=prog)
        flips += pc.compare_full_step(out, ref, np.ascontiguousarray(rb), rb_ref, m, f"{what} fields [{c0}, {c1})",
                                      exact_physics=False)
        chunks.append((c0, c1))
    return flips, chunks


def chosen_steps(progress0):
    """Steps of the window compared with the oracle: the first two, the last warm-up and first timed step, the step in
    which the most staggered counters reach 400 (a field with counter p times out at step 399 - p unless a goal ended
    its episode first), and the last step of each region."""
    counts = np.bincount(progress0, minlength=400)[:400]
    t_timeout = int(399 - np.argmax(counts))
    return sorted({0, 1, WARMUP - 1, WARMUP, t_timeout, 399, STEPS - 1}), t_timeout, int(counts.max())


def run_synchronised(n, shape=None, chosen=()):
    """The benchmark's task stepped STEPS times, synchronising with the host after every launch; per-step checksums
    (device) and, for the chosen steps, the pre-step state and flags and the step's outputs (device clones)."""
    import bench
    envs, acts = bench.make_task(torch, n, 0, 0)
    if shape is not None:
        envs.engine.warps_per_tile, envs.engine.fields_per_tile = shape
        assert (envs.engine.warps_per_tile, envs.engine.fields_per_tile) == shape
    start = envs.engine.get_state()
    sums = torch.zeros((STEPS, len(SUM_NAMES)), dtype=torch.int64, device=envs.device)
    events = torch.zeros((STEPS, 3), dtype=torch.int64, device=envs.device)   # resets, time-outs, goals
    kept = {}
    for i in range(STEPS):
        pre = (envs.engine.get_state(), envs.reset_buf.clone()) if i in chosen else None
        out = envs.step(acts[i & 3])
        sums[i] = step_sums(envs, out)
        obs, tobs, rew, reset, tmo, prog = step_outputs(out)
        events[i, 0], events[i, 1], events[i, 2] = reset.sum(), tmo.sum(), (rew[:, 0, 0, 0] != 0).sum()
        if pre is not None:
            kept[i] = pre + (acts[i & 3], tuple(x.clone() for x in step_outputs(out)))
        torch.cuda.synchronize()
    return dict(envs=envs, start=start, sums=sums, events=events.cpu().numpy(), kept=kept,
                final=envs.engine.get_state(), last=tuple(x.clone() for x in step_outputs(out)),
                step_count=envs.engine.step_count)


@pytest.fixture(scope="module", params=SIZES, ids=SIZE_IDS)
def window(request):
    """Run B (automatic shape, host-synchronised, with the oracle steps kept), run A (back to back), and the forced
    shapes, all built by bench.make_task with the same seeds."""
    import bench
    n = request.param
    res = {"n": n}
    probe, _ = bench.make_task(torch, n, 0, 0)
    progress0 = probe.engine.get_state()[58, :n].view(torch.int32).cpu().numpy()
    del probe
    res["chosen"], res["t_timeout"], res["timeouts_expected"] = chosen_steps(progress0)
    b = run_synchronised(n, chosen=set(res["chosen"]))
    res["b"] = b
    # run A: every launch right after the previous one, nothing else in the stream, no host synchronisation
    envs, acts = bench.make_task(torch, n, 0, 0)
    for i in range(STEPS):
        out = envs.step(acts[i & 3])
    torch.cuda.synchronize()
    res["a"] = dict(final=envs.engine.get_state(), last=step_outputs(out), step_count=envs.engine.step_count)
    del envs, acts
    res["shapes"] = {}
    for shape in SHAPES:
        r = run_synchronised(n, shape=shape)
        res["shapes"][shape] = dict(sums=r["sums"], final=r["final"], step_count=r["step_count"])
        del r
    torch.cuda.empty_cache()
    yield res
    res.clear()
    torch.cuda.empty_cache()


def test_back_to_back_equals_host_synchronised(window):
    """450 adjacent launches leave exactly the state and outputs of 450 host-synchronised ones: the whole SoA state
    (all 60 rows, incl. the progress and episode words) and every output of the last step."""
    a, b = window["a"], window["b"]
    assert bits_equal(a["final"], b["final"]), "state after the window"
    for name, x, y in zip(SUM_NAMES[1:], a["last"], b["last"]):
        assert bits_equal(x, y), f"{name} of step {STEPS - 1}"
    # vss_step draws no OU noise: it neither reads nor advances the views' step index (include/vss_b200.h)
    assert a["step_count"] == b["step_count"] == 0


def test_launch_shapes_agree_at_every_step(window):
    """1 warp x 8 fields, 1 warp x 16 fields and 8 warps x 32 fields per tile (k_step_cta) compute the automatic
    shape's words at every step of the window."""
    b = window["b"]
    for shape, r in window["shapes"].items():
        same = (r["sums"] == b["sums"]).all(1)
        if not bool(same.all()):
            t = int((~same).nonzero()[0, 0])
            bad = [SUM_NAMES[k] for k in range(len(SUM_NAMES)) if int(r["sums"][t, k]) != int(b["sums"][t, k])]
            pytest.fail(f"shape {shape}: step {t} differs from the automatic shape in {bad}")
        assert bits_equal(r["final"], b["final"]), f"shape {shape}: state after the window"
        assert r["step_count"] == 0


def test_chosen_steps_match_oracle(window):
    """Steps 0, 1, 49, 50, the step with the most time-outs of the staggered counters, 399 and 449 of run B against
    the oracle from the same pre-step state, every field (chunks of 131 072 fields with their global offsets)."""
    n, b = window["n"], window["b"]
    p = orc.default_params()
    seed = int(b["envs"].seed)
    for t in window["chosen"]:
        pre_state, pre_reset, actions, post = b["kept"][t]
        flips, chunks = compare_with_oracle(p, seed, pre_state, pre_reset, actions, post, n, f"step {t}")
        assert flips <= pc.FLIP_FRACTION * n, f"step {t}: {flips} fields outside the physics tolerance"
    # the chunks covered the first CTA, the CTAs on both sides of every wave boundary and the last, ragged CTA
    covered = lambda f: any(c0 <= f < c1 for c0, c1 in chunks)
    assert chunks[0][0] == 0 and chunks[-1][1] == n and all(x[1] == y[0] for x, y in zip(chunks, chunks[1:]))
    assert all(covered(k * WAVE_FIELDS - 1) and covered(k * WAVE_FIELDS) for k in range(1, n // WAVE_FIELDS + 1))
    ev = b["events"]
    assert ev[:, 0].sum() > 0 and ev[:, 1].sum() > 0 and ev[:, 2].sum() > 0, "resets, time-outs, goals in the window"
    assert ev[window["t_timeout"], 1] >= window["timeouts_expected"] // 2, (window["t_timeout"], ev[window["t_timeout"]])
    # fields reset twice inside the window (a counter at 399 - k times out at step k and again 400 steps later): the
    # episode word of the reset key has moved past its first value
    ep0 = b["start"][59, :n].view(torch.int32)
    ep1 = b["final"][59, :n].view(torch.int32)
    assert int((ep1 - ep0).max()) >= 2 and bool((ep1 >= ep0).all())


def test_injected_step_is_exact_at_benchmark_size():
    """Physics replaced by the same post-physics state on both sides: rewards, dones, time-outs, progress, obs and
    terminal obs bit-exact at 2^20 fields."""
    from backends import GpuBackend
    assert pc.check_injected(GpuBackend, n=1 << 20, steps=2, seed=20) > 0


@pytest.mark.parametrize("n", SIZES, ids=SIZE_IDS)
def test_full_contract_outputs_stay_inside_their_buffers(n):
    """Every output of `vss_step` is a slice of a larger buffer filled with a sentinel: the step writes every row of
    the slice and nothing outside it. The first launch runs with every reset flag set to a non-0/1 value (every field
    restarts its counter; the flags must all be overwritten), the second with the flags the first one returned."""
    import bench
    envs, acts = bench.make_task(torch, n, 0, 0)
    PAD, SENT = 300, -12345.0
    cols = {"obs": 312, "term_obs": 312, "rew": 24, "time_outs": 1, "progress": 1, "reset": 1}
    sent = {"time_outs": 0xA5, "reset": -7}
    dtype = {"time_outs": torch.uint8, "reset": torch.int64}
    big = {k: torch.full(((n + 2 * PAD) * c,), sent.get(k, SENT), device="cuda", dtype=dtype.get(k, torch.float32))
           for k, c in cols.items()}
    inner = {k: big[k][PAD * c:(PAD + n) * c] for k, c in cols.items()}
    for t in range(2):
        if t:
            for k in cols:
                if k != "reset":
                    inner[k].fill_(sent.get(k, SENT))
        envs.engine.step(acts[t], inner["reset"], inner["obs"], inner["term_obs"], inner["rew"], inner["time_outs"],
                         inner["progress"])
        torch.cuda.synchronize()
        for k, c in cols.items():
            s = sent.get(k, SENT)
            assert bool((big[k][:PAD * c] == s).all()) and bool((big[k][(PAD + n) * c:] == s).all()), (t, k, "outside")
            rows = inner[k].view(n, c) == s
            assert not bool(rows.any()), (t, k, "unwritten rows", rows.any(1).nonzero()[:5, 0].tolist())
        assert bool(((inner["reset"] == 0) | (inner["reset"] == 1)).all())
        assert bool(((inner["time_outs"] == 0) | (inner["time_outs"] == 1)).all())


def test_view_step_index_advances_once_per_back_to_back_launch():
    """The views key their OU noise by a device step index that the CTA completing a launch advances after clearing
    the CTA count; at the benchmark's size (8 192 CTAs) 64 adjacent SingleAgent launches advance it by exactly 64 and
    leave what 64 host-synchronised ones leave."""
    import bench
    from rsoccer_isaac_cleanrl_b200.envs import SingleAgent
    n, K = 1 << 20, 64
    runs = []
    for sync in (False, True):
        envs, _ = bench.make_task(torch, n, 0, 0)
        view = SingleAgent(envs)
        g = torch.Generator(device="cuda")
        g.manual_seed(7)
        pa = [torch.rand((n, 2), device="cuda", generator=g) * 2 - 1 for _ in range(4)]
        for i in range(K):
            out = view.step(pa[i & 3])
            if sync:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
        runs.append(dict(step_count=envs.engine.step_count, state=envs.engine.get_state(),
                         action_buf=view.action_buf.clone(), obs=out[0]["obs"].clone(), reward=out[1].clone()))
        del envs, view, pa, out
    a, b = runs
    assert a["step_count"] == b["step_count"] == K
    for k in ("state", "action_buf", "obs", "reward"):
        assert bits_equal(a[k], b[k]), k
