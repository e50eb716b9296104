"""Parity checks of the match step (vss_step_match), shared by the CPU (host emulation) and GPU test files.

The reference for one match step is restated here from the oracle's own pieces: the views' OU draw (Philox stream 2
keyed by the step index, restated in numpy from the Philox known answers the oracle pins), each team's mode applied
to the (N,2,3,2) buffer as play.py's teams do, then the oracle's VSS.step. Tolerances are parity_checks': OU slots
within 2e-6 (libm), physics within PHYS_ATOL / PHYS_RTOL with up to FLIP_FRACTION branch flips. Against the same
backend's full-contract step from the same state and with the same actions the match step is bit-exact.

Why a restatement here and not a match step in oracle/vss_oracle.c: the oracle is pinned to golden vectors produced
by executing the reference's own code (tests/golden), and the parity module and the oracle stay byte-for-byte as they
were pinned, so that a change to the engine cannot move its own yardstick. A match step adds nothing the oracle lacks:
it is the views' OU draw (the oracle's ou_one, which it does not export; the numpy restatement below is pinned to it
through orc.step_view by test_match_emu.py), a table of slot overwrites (play.py's teams) and orc.step, which is used
as is.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

import parity_checks as pc
from backends import ROOT, EmuBackend, GpuBackend
from oracle import vss_oracle as orc

ZERO, OU, SA, CMA, DMA, EXTERNAL = 0, 1, 2, 3, 4, 5
POLICY = (SA, CMA, DMA)
BOARD_WORDS = 5  # vss_match_board as int64 words: matches, length_sum, score_sum (f64 bits), steps, frozen


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def nv_of(mode, n):
    return 3 * n if mode == DMA else n


def adim_of(mode):
    return 6 if mode == CMA else 2


def board_dict(words):
    w = np.ascontiguousarray(words, np.int64)
    return dict(matches=int(w[0]), length_sum=int(w[1]), score_sum=float(w[2:3].view(np.float64)[0]),
                steps=int(w[3]), frozen=int(w[4]) & 0xFFFFFFFF)


# ------------------------------------------------------------------ numpy restatements
def _philox(c0, c1, c2, c3, k0, k1):
    m = np.uint64(0xFFFFFFFF)
    c = [np.asarray(x, np.uint64) for x in (c0, c1, c2, c3)]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c[0]
        p1 = np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & m, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & m]
        k0 = (k0 + np.uint64(0x9E3779B9)) & m
        k1 = (k1 + np.uint64(0xBB67AE85)) & m
    return [x.astype(np.uint32) for x in c]


def ou_draw(p, seed, goff, step, prev):
    """random_ou on all 12 slots of every field (wrappers.py:5-19, the views' Philox stream 2): (n,12) f32."""
    n = prev.shape[0]
    gid = np.arange(n, dtype=np.uint64) + np.uint64(goff)
    out = np.array(prev, np.float32).reshape(n, 12).copy()
    f = np.float32
    for b in range(3):
        u = _philox(gid & np.uint64(0xFFFFFFFF), gid >> np.uint64(32), np.full(n, step, np.uint64),
                    np.full(n, (2 << 28) | b, np.uint64), seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF)
        for h in range(2):
            uo = ((u[2 * h] >> 8) + np.uint32(1)).astype(np.float32) * f(1.0 / 16777216.0)
            uc = (u[2 * h + 1] >> 8).astype(np.float32) * f(1.0 / 16777216.0)
            rad = np.sqrt(f(-2.0) * np.log(uo))
            ang = f(6.283185307179586) * uc
            for c, z in enumerate((rad * np.cos(ang), rad * np.sin(ang))):
                v = out[:, 4 * b + 2 * h + c]
                out[:, 4 * b + 2 * h + c] = np.clip((v - f(p.ou_theta) * v) + f(p.ou_sigma) * z, -1.0, 1.0)
    return out


def team_actions(modes, acts, prev, ou):
    """play.py's team calls on the buffer: (n,12) f32 from the previous values and the OU draw of every slot."""
    n = prev.shape[0]
    new = prev.reshape(n, 12).copy()
    for t, m in enumerate(modes):
        s = slice(6 * t, 6 * t + 6)
        if m == ZERO:
            new[:, s] = prev.reshape(n, 12)[:, s] * np.float32(0.0)
        elif m == OU:
            new[:, s] = ou[:, s]
        elif m == SA:
            new[:, s] = ou[:, s]
            new[:, 6 * t:6 * t + 2] = acts[t].reshape(n, 2)
        elif m in (CMA, DMA):
            new[:, s] = acts[t].reshape(n, 6)
    return new


def bf16_bits(x):
    u = np.ascontiguousarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def expected_rows(mode, obs, t):
    """The team's bf16 rows (padded to 64 columns) of a post-reset (n,2,3,52) observation."""
    n = obs.shape[0]
    rows = obs[:, t] if mode == DMA else obs[:, t, :1]
    out = np.zeros((nv_of(mode, n), 64), np.uint16)
    out[:, :52] = bf16_bits(rows.reshape(-1, 52))
    return out


class LoopBoard:
    """The statistics of play_matches' loop (play.py:120-130), fed one step's dones, rewards and progress."""

    def __init__(self, count_envs, n_matches):
        self.count_envs, self.n_matches = count_envs, n_matches
        self.ep_count, self.rew_sum, self.len_sum, self.steps = 0, 0.0, 0.0, 0

    @property
    def finished(self):
        return self.ep_count >= self.n_matches

    def step(self, dones, rew, progress):
        if self.finished:
            return
        self.steps += 1
        ids = np.nonzero(dones[:self.count_envs])[0]
        if len(ids):
            self.ep_count += len(ids)
            self.rew_sum += float(rew[ids, 0, 0, 0].sum(dtype=np.float32))
            self.len_sum += float(progress[ids].sum(dtype=np.float32))


def assert_board_matches_loop(board, loop, what):
    b = board_dict(board)
    assert b["matches"] == loop.ep_count, (what, b, loop.ep_count)
    assert b["length_sum"] == loop.len_sum and b["score_sum"] == loop.rew_sum, (what, b, loop.len_sum, loop.rew_sum)
    assert b["steps"] == loop.steps and b["frozen"] == int(loop.finished), (what, b, loop.steps)


# ------------------------------------------------------------------ backends
class EmuMatchBackend(EmuBackend):
    """EmuBackend + the match step of tests/emu/vss_emu_match.cpp (compiled on first use into a temporary directory)."""

    _match_lib = None

    @classmethod
    def match_lib(cls):
        if cls._match_lib is None:
            d = tempfile.mkdtemp(prefix="vss_emu_match_")
            so = os.path.join(d, "libvss_emu_match.so")
            src = os.path.join(ROOT, "tests", "emu", "vss_emu_match.cpp")
            cxx = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"
            subprocess.run([cxx, "-O2", "-std=c++17", "-fPIC", "-ffp-contract=off", "-fopenmp", "-fvisibility=hidden",
                            "-shared", "-x", "c++", "-o", so, src, "-lm"], check=True, capture_output=True)
            cls._match_lib = C.CDLL(so)
        return cls._match_lib

    def step_match(self, modes, acts, action_buf, reset_buf, count_envs, n_matches, board, want_obs=True):
        n = self.n
        rows = [np.zeros((nv_of(m, n), 64), np.uint16) if m in POLICY else None for m in modes]
        acts = [None if a is None else np.ascontiguousarray(a, np.float32) for a in acts]
        obs = np.zeros((n, 2, 3, 52), np.float32) if want_obs else None
        mode_arr = np.array(modes, np.int32)
        rc = self.match_lib().emu_step_match(
            C.byref(self.params), _p(self.state), C.c_longlong(n), C.c_longlong(self.ld), C.c_ulonglong(self.goff),
            C.c_ulonglong(self.seed), C.c_uint(self.step_count & 0xFFFFFFFF), _p(mode_arr), _p(acts[0]), _p(acts[1]),
            _p(rows[0]), _p(rows[1]), _p(action_buf), _p(reset_buf), _p(obs), C.c_longlong(count_envs),
            C.c_longlong(n_matches), _p(board), C.c_int(self.wpt), C.c_int(self.fpt))
        assert rc == 0
        self.step_count += 1
        return dict(obs=obs, rows=rows)


class GpuMatchBackend(GpuBackend):
    """GpuBackend + Engine.step_match (vss_step_match through the C-ABI)."""

    def step_match(self, modes, acts, action_buf, reset_buf, count_envs, n_matches, board, want_obs=True):
        t, n = self.torch, self.n
        rows = [t.zeros((nv_of(m, n), 64), dtype=t.bfloat16, device=self.dev) if m in POLICY else None for m in modes]
        acts_t = [None if a is None else self._t(np.ascontiguousarray(a, np.float32)) for a in acts]
        ab, rb, bd = self._t(action_buf), self._t(reset_buf), self._t(board)
        obs = t.zeros((n, 2, 3, 52), dtype=t.float32, device=self.dev) if want_obs else None
        self.eng.step_match(list(zip(modes, acts_t, rows)), ab, rb, bd, count_envs, n_matches, obs=obs)
        t.cuda.synchronize()
        action_buf[...] = ab.cpu().numpy()
        reset_buf[...] = rb.cpu().numpy()
        board[...] = bd.cpu().numpy()
        return dict(obs=None if obs is None else obs.cpu().numpy(),
                    rows=[None if r is None else r.view(t.int16).cpu().numpy().view(np.uint16) for r in rows])


def match_backend(Backend):
    """The match-capable subclass of a parity_checks backend (keeps its launch-shape attributes)."""
    base = EmuMatchBackend if issubclass(Backend, EmuBackend) else GpuMatchBackend
    if issubclass(Backend, base):
        return Backend
    return type(f"Match{Backend.__name__}", (base,), {k: getattr(Backend, k) for k in ("wpt", "fpt")})


# ------------------------------------------------------------------ the check
def check_match(Backend, modes=(SA, OU), n=333, steps=14, seed=9, goff=4321, count_envs=None, n_matches=40):
    """A match run on `Backend` against (1) the same backend's full-contract step from the same state with the
    same actions: bit-exact state, reset flags, obs and bf16 rows; (2) the oracle restatement: every team's slots,
    OU within 2e-6, physics within the views' tolerances; (3) play_matches' loop statistics fed that step's
    dones, rewards and progress: the scoreboard, its freeze included."""
    Match = match_backend(Backend)
    count_envs = n - 17 if count_envs is None else count_envs
    be, p = pc.make_backend_pair(Match, n, seed, goff)
    twin, _ = pc.make_backend_pair(Backend, n, seed, goff)
    rng = np.random.default_rng(seed)
    rb = np.ones(n, np.int64)
    be.reset_dones(rb)
    rb[:] = 0
    pc.stage_interesting_state(be, rng)
    abuf = rng.uniform(-1.2, 1.2, (n, 2, 3, 2)).astype(np.float32)
    abuf[:5] = -0.0  # the sign of zero survives ZERO's `*= 0`
    board = np.zeros(BOARD_WORDS, np.int64)
    loop = LoopBoard(count_envs, n_matches)
    flips = dones_seen = 0
    for step in range(steps):
        st = be.get_state()
        rb_in, abuf_in, step_index = rb.copy(), abuf.copy(), be.step_count
        acts = [rng.uniform(-1.2, 1.2, (nv_of(m, n), adim_of(m))).astype(np.float32) if m in POLICY else None
                for m in modes]
        ext = rng.uniform(-1.2, 1.2, (n, 2, 3, 2)).astype(np.float32)   # what an EXTERNAL team writes
        for t, m in enumerate(modes):
            if m == EXTERNAL:
                abuf[:, t] = ext[:, t]
                abuf_in[:, t] = ext[:, t]
        out = be.step_match(modes, acts, abuf, rb, count_envs, n_matches, board)
        # (2a) the action prologue: every team writes exactly its slots; OU slots against the restated draw
        ou = ou_draw(p, seed, goff, step_index, abuf_in.reshape(n, 12))
        want = team_actions(modes, acts, abuf_in, ou)
        got = abuf.reshape(n, 12)
        is_ou = np.zeros((n, 12), bool)
        for t, m in enumerate(modes):
            if m == OU:
                is_ou[:, 6 * t:6 * t + 6] = True
            elif m == SA:
                is_ou[:, 6 * t + 2:6 * t + 6] = True
        pc.assert_bits_equal(got[~is_ou], want[~is_ou], f"step {step}: team slots")
        np.testing.assert_allclose(got[is_ou], want[is_ou], rtol=0, atol=2e-6, err_msg=f"step {step}: OU slots")
        # (1) the full-contract step of the same backend from the same state with the kernel's own actions
        twin.set_state(st)
        rb_twin = rb_in.copy()
        ref = twin.step(abuf.copy(), rb_twin)
        assert np.array_equal(rb, rb_twin), f"step {step}: reset_buf"
        pc.assert_bits_equal(be.get_state()[:, :n], twin.get_state()[:, :n], f"step {step}: state")
        pc.assert_bits_equal(out["obs"], ref["obs"], f"step {step}: obs")
        for t, m in enumerate(modes):
            if m in POLICY:
                assert np.array_equal(out["rows"][t], expected_rows(m, ref["obs"], t)), f"step {step}: team {t} rows"
        # (3) the scoreboard against the loop's statistics
        loop.step(rb_twin, ref["rew"], ref["progress_f"])
        assert_board_matches_loop(board, loop, f"step {step}")
        # (2b) the oracle's physics from the same state and actions
        ost = orc.State.from_soa(st, n)
        rb_ref = rb_in.copy()
        oref = orc.step(p, seed, goff, ost, abuf.copy(), rb_ref)
        flips += pc.compare_full_step(ref, oref, rb_twin, rb_ref, n, f"match step {step}", exact_physics=False)
        dones_seen += int(rb.sum())
    assert flips <= max(2, pc.FLIP_FRACTION * n * steps), f"{flips} field-steps outside the physics tolerance"
    assert dones_seen > 0
    return dict(board=board_dict(board), loop_steps=loop.steps, flips=flips)
