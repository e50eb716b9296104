"""Parity checks of the opponent view step (vss_step_view with vss_set_view_opponent), shared by the CPU (host
emulation) and GPU test files.

The restatement of one opponent view step (include/vss_b200.h):
  1. action_buf = random_ou(action_buf) on all 12 slots (the views' Philox stream 2 keyed by the step index);
  2. the learner's slots = the policy action, as the view does;
  3. the yellow slots follow the opponent's mode: ZERO draw x 0, SA robot 0 = its action, CMA / DMA all 6 = its
     action, EXTERNAL as the caller wrote them;
  4. the rest is the full-contract step driven with those 12 slots, sliced as the view slices it (oracle
     view_outputs), done rows of action_buf zeroed;
  5. the opponent's bf16 rows and f32 observation are the yellow rows of the full step's post-reset obs.

The 12 slots come from the restatement above, with the OU draw taken from the same backend's match step with two OU
teams (which stores the draw un-clamped and keeps done rows): it is the kernel's own draw, so the comparison can be
bit for bit. That draw is itself checked against match_checks.ou_draw (the numpy restatement) within 2e-6 (libm).
"""
import ctypes as C

import numpy as np

import match_checks as mc
import parity_checks as pc
from backends import VIEW_CMA, VIEW_DMA, VIEW_SA, EmuBackend, GpuBackend
from oracle import vss_oracle as orc

ZERO, OU, SA, CMA, DMA, EXTERNAL = mc.ZERO, mc.OU, mc.SA, mc.CMA, mc.DMA, mc.EXTERNAL
POLICY = mc.POLICY
OPP_MODES = (ZERO, SA, CMA, DMA, EXTERNAL)


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def nv_of_view(view, n):
    return 3 * n if view == VIEW_DMA else n


def adim_of_view(view):
    return 6 if view == VIEW_CMA else 2


def predicted_slots(view, mode, pa, opp_act, prev, ou):
    """The 12 slots of the restatement: (n,12) f32 from the caller's buffer `prev`, the OU draw and the two actions."""
    n = prev.shape[0]
    want = ou.reshape(n, 12).copy()
    if view == VIEW_SA:
        want[:, 0:2] = pa.reshape(n, 2)
    else:
        want[:, 0:6] = pa.reshape(n, 6)
    if mode == ZERO:
        want[:, 6:] = ou.reshape(n, 12)[:, 6:] * np.float32(0.0)
    elif mode == SA:
        want[:, 6:8] = opp_act.reshape(n, 2)
    elif mode in (CMA, DMA):
        want[:, 6:] = opp_act.reshape(n, 6)
    elif mode == EXTERNAL:
        want[:, 6:] = prev.reshape(n, 12)[:, 6:]
    return want


# ------------------------------------------------------------------ backends
class EmuOppBackend(mc.EmuMatchBackend):
    """EmuBackend + the opponent view step of the host emulation (emu_step_view_opp)."""

    def step_view_opp(self, view, policy_action, action_buf, reset_buf, ep_ret, ep_len, mode, opp_action,
                      want_obs=True):
        n, nv = self.n, nv_of_view(view, self.n)
        z = np.zeros
        out = dict(obs=z((nv, 52), np.float32), term_obs=z((nv, 52), np.float32), rews=z((nv, 4), np.float32),
                   reward=z((nv,), np.float32), done=z((nv,), np.int64), timeout=z((nv,), np.uint8),
                   progress=z((nv,), np.float32), ret_ret=z((nv, 4), np.float32), ret_len=z((nv,), np.int32))
        rows = z((mc.nv_of(mode, n), 64), np.uint16) if mode in POLICY else None
        opp_obs = z((n, 3, 52), np.float32) if want_obs else None
        oa = None if opp_action is None else np.ascontiguousarray(opp_action, np.float32)
        rc = self.lib().emu_step_view_opp(
            C.byref(self.params), C.c_int(view), _p(self.state), C.c_longlong(n), C.c_longlong(self.ld),
            C.c_ulonglong(self.goff), C.c_ulonglong(self.seed), C.c_uint(self.step_count & 0xFFFFFFFF), _p(reset_buf),
            _p(out["obs"]), _p(out["term_obs"]), _p(out["rews"]), _p(out["timeout"]), _p(out["progress"]),
            _p(np.ascontiguousarray(policy_action, np.float32)), _p(action_buf), _p(out["reward"]), _p(out["done"]),
            _p(ep_ret), _p(ep_len), _p(out["ret_ret"]), _p(out["ret_len"]), C.c_int(mode), _p(oa), _p(rows),
            _p(opp_obs), C.c_int(self.wpt), C.c_int(self.fpt))
        assert rc == 0
        self.step_count += 1
        out["rows"], out["opp_obs"] = rows, opp_obs
        return out


class GpuOppBackend(mc.GpuMatchBackend):
    """GpuBackend + Engine.step_view(..., opponent=...) (vss_set_view_opponent + vss_step_view)."""

    step_range = None  # a number of ranges: the step is issued as that many consecutive vss_set_step_range launches

    def step_view_opp(self, view, policy_action, action_buf, reset_buf, ep_ret, ep_len, mode, opp_action,
                      want_obs=True):
        t, n = self.torch, self.n
        nv = nv_of_view(view, n)
        z = lambda shape, dt: t.zeros(shape, dtype=dt, device=self.dev)
        rb, ab, er, el = self._t(reset_buf), self._t(action_buf), self._t(ep_ret), self._t(ep_len)
        obs, tobs, rews, reward = z((nv, 52), t.float32), z((nv, 52), t.float32), z((nv, 4), t.float32), z((nv,), t.float32)
        done, tout, prog = z((nv,), t.int64), z((nv,), t.uint8), z((nv,), t.float32)
        rr, rl = z((nv, 4), t.float32), z((nv,), t.int32)
        rows = z((mc.nv_of(mode, n), 64), t.bfloat16) if mode in POLICY else None
        opp_obs = z((n, 3, 52), t.float32) if want_obs else None
        opp = (mode, self._t(opp_action), rows, opp_obs)
        pa = self._t(np.ascontiguousarray(policy_action, np.float32))
        args = (view, pa, ab, rb, obs, tobs, rews, reward, done, tout, prog, er, el, rr, rl)
        if self.step_range is None:
            self.eng.step_view(*args, opponent=opp)
        else:
            g = self.eng.step_granularity
            per = -(-n // (self.step_range * g)) * g
            try:
                for f0 in range(0, n, per):
                    self.eng.set_step_range(f0, min(per, n - f0))
                    self.eng.step_view(*args, opponent=opp)
            finally:
                self.eng.set_step_range(0, 0)
        self.eng.set_view_opponent(None)
        t.cuda.synchronize()
        reset_buf[...] = rb.cpu().numpy()
        action_buf[...] = ab.cpu().numpy()
        ep_ret[...] = er.cpu().numpy()
        ep_len[...] = el.cpu().numpy()
        out = dict(obs=obs, term_obs=tobs, rews=rews, reward=reward, done=done, timeout=tout, progress=prog,
                   ret_ret=rr, ret_len=rl, opp_obs=opp_obs)
        out = {k: None if v is None else v.cpu().numpy() for k, v in out.items()}
        out["rows"] = None if rows is None else rows.view(t.int16).cpu().numpy().view(np.uint16)
        return out


def opp_backend(Backend):
    """The opponent-capable subclass of a parity_checks backend (keeps its launch-shape attributes)."""
    base = EmuOppBackend if issubclass(Backend, EmuBackend) else GpuOppBackend
    if issubclass(Backend, base):
        return Backend
    return type(f"Opp{Backend.__name__}", (base,), {k: getattr(Backend, k) for k in ("wpt", "fpt")})


def kernel_ou_draw(be_match, state, step_index, prev):
    """The backend's own OU draw of every slot: its match step with two OU teams from `state` (a scratch twin)."""
    n = be_match.n
    be_match.set_state(state)
    be_match.step_count = step_index
    abuf = np.ascontiguousarray(prev, np.float32).reshape(n, 2, 3, 2).copy()
    rb = np.zeros(n, np.int64)
    board = np.zeros(mc.BOARD_WORDS, np.int64)
    be_match.step_match((OU, OU), (None, None), abuf, rb, n, 1 << 40, board, want_obs=False)
    return abuf.reshape(n, 12)


# ------------------------------------------------------------------ the check
def check_opponent(Backend, view, mode, n=333, steps=12, seed=5, goff=777, want_obs=True, step_range=None):
    """An opponent view run on `Backend` against the restatement: bit for bit against the same backend's full-contract
    step driven with the predicted 12 slots and sliced as the view slices it (learner outputs, episode statistics,
    state, reset flags, action_buf with done rows zeroed, the opponent's bf16 rows and f32 observation)."""
    Opp = opp_backend(Backend)
    if step_range is not None:
        Opp = type(Opp.__name__ + "Ranges", (Opp,), {"step_range": step_range})
    be, p = pc.make_backend_pair(Opp, n, seed, goff)
    twin, _ = pc.make_backend_pair(Backend, n, seed, goff)
    draw, _ = pc.make_backend_pair(mc.match_backend(Backend), n, seed, goff)
    rng = np.random.default_rng(seed + 10 * view + mode)
    nv, adim = nv_of_view(view, n), adim_of_view(view)
    rb = np.ones(n, np.int64)
    be.reset_dones(rb)
    rb[:] = 0
    pc.stage_interesting_state(be, rng)
    abuf = rng.uniform(-1.2, 1.2, (n, 2, 3, 2)).astype(np.float32)
    abuf[:5] = -0.0
    ep_ret, ep_len = np.zeros((nv, 4), np.float32), np.zeros((nv,), np.int32)
    dones = 0
    for step in range(steps):
        st = be.get_state()
        step_index = be.step_count
        pa = rng.uniform(-1.2, 1.2, (nv, adim)).astype(np.float32)
        opp_act = (rng.uniform(-1.2, 1.2, (mc.nv_of(mode, n), mc.adim_of(mode))).astype(np.float32)
                   if mode in POLICY else None)
        if mode == EXTERNAL:  # what an EXTERNAL opponent writes into its slots before the step
            abuf[:, 1] = rng.uniform(-1.2, 1.2, (n, 3, 2)).astype(np.float32)
        rb_in, abuf_in, er_in, el_in = rb.copy(), abuf.copy(), ep_ret.copy(), ep_len.copy()
        out = be.step_view_opp(view, pa, abuf, rb, ep_ret, ep_len, mode, opp_act, want_obs=want_obs)
        # the restatement's 12 slots, with the kernel's own OU draw (itself within libm of the numpy restatement)
        ou = kernel_ou_draw(draw, st, step_index, abuf_in)
        np.testing.assert_allclose(ou, mc.ou_draw(p, seed, goff, step_index, abuf_in.reshape(n, 12)), rtol=0,
                                   atol=2e-6, err_msg=f"step {step}: OU draw")
        slots = predicted_slots(view, mode, pa, opp_act, abuf_in, ou).reshape(n, 2, 3, 2)
        # the full-contract step with those slots, sliced by the view
        twin.set_state(st)
        rb_twin = rb_in.copy()
        ref = twin.step(slots.copy(), rb_twin)
        abuf_ref = slots.copy()
        want = orc.view_outputs(view, ref["obs"], ref["term_obs"], ref["rew"], rb_twin, ref["timeout"],
                                ref["progress_f"], abuf_ref, er_in, el_in)
        what = f"view {view} opponent {mode} step {step}"
        assert np.array_equal(rb, rb_twin), what + ": reset_buf"
        pc.assert_bits_equal(be.get_state()[:, :n], twin.get_state()[:, :n], what + ": state")
        for k in ("obs", "term_obs", "rews", "reward", "progress", "ret_ret"):
            pc.assert_bits_equal(out[k], want[k], f"{what}: {k}")
        for k in ("done", "timeout", "ret_len"):
            assert np.array_equal(out[k], want[k]), f"{what}: {k}"
        pc.assert_bits_equal(ep_ret, er_in, what + ": ep_ret")
        assert np.array_equal(ep_len, el_in), what + ": ep_len"
        pc.assert_bits_equal(abuf, abuf_ref, what + ": action_buf")
        assert np.all(abuf[rb != 0] == 0)
        if mode in POLICY:
            assert np.array_equal(out["rows"], mc.expected_rows(mode, ref["obs"], 1)), what + ": rows_bf16"
        if want_obs:
            pc.assert_bits_equal(out["opp_obs"], ref["obs"][:, 1], what + ": obs_f32")
        dones += int(rb.sum())
    assert dones > 0
    return dict(dones=dones)


def check_ou_mode_is_no_opponent(Backend, view, n=200, steps=6, seed=3, goff=99):
    """Opponent mode OU computes exactly what the view computes without an opponent (on the device the setter clears
    the opponent; the host emulation runs the opponent variant with the draw kept)."""
    a, _ = pc.make_backend_pair(Backend, n, seed, goff)
    b, _ = pc.make_backend_pair(opp_backend(Backend), n, seed, goff)
    rng = np.random.default_rng(seed)
    nv, adim = nv_of_view(view, n), adim_of_view(view)
    rb = np.ones(n, np.int64)
    a.reset_dones(rb)
    b.reset_dones(rb)
    rb[:] = 0
    rb2 = rb.copy()
    abuf = rng.uniform(-1, 1, (n, 2, 3, 2)).astype(np.float32)
    abuf2 = abuf.copy()
    er, el = np.zeros((nv, 4), np.float32), np.zeros(nv, np.int32)
    er2, el2 = er.copy(), el.copy()
    for step in range(steps):
        pa = rng.uniform(-1.2, 1.2, (nv, adim)).astype(np.float32)
        x = a.step_view(view, pa, abuf, rb, er, el)
        y = b.step_view_opp(view, pa, abuf2, rb2, er2, el2, OU, None, want_obs=False)
        for k in x:
            pc.assert_bits_equal(x[k], y[k], f"step {step}: {k}")
        pc.assert_bits_equal(abuf, abuf2, f"step {step}: action_buf")
        assert np.array_equal(rb, rb2)
        pc.assert_bits_equal(a.get_state(), b.get_state(), f"step {step}: state")
