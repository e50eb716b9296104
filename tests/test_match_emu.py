"""CPU: the match step (vss_step_match) on the host emulation of the product's lane code, against the oracle and
play_matches' loop statistics; argument validation of the C-ABI entry without a device."""
import ctypes as C

import numpy as np
import pytest

import match_checks as mc
from backends import EmuBackend, with_wpt

MODE_PAIRS = [(mc.SA, mc.OU), (mc.ZERO, mc.OU), (mc.CMA, mc.DMA), (mc.DMA, mc.ZERO), (mc.EXTERNAL, mc.SA),
              (mc.OU, mc.EXTERNAL)]


@pytest.mark.parametrize("modes", MODE_PAIRS, ids=lambda m: f"{m[0]}v{m[1]}")
def test_match_step_one_warp_per_tile(modes):
    r = mc.check_match(EmuBackend, modes=modes)
    assert r["board"]["matches"] > 0


@pytest.mark.parametrize("wpt,fpt", [(8, 32), (7, 16), (2, 8)])
def test_match_step_shared_tile(wpt, fpt):
    mc.check_match(with_wpt(EmuBackend, wpt, fpt), modes=(mc.SA, mc.DMA))


def test_scoreboard_freezes_after_the_step_that_reaches_the_count():
    """n_matches reached after a few steps: later steps add nothing, the counting step adds all its dones."""
    r = mc.check_match(EmuBackend, modes=(mc.OU, mc.ZERO), n=256, steps=20, count_envs=100, n_matches=6)
    b = r["board"]
    assert b["frozen"] == 1 and b["matches"] >= 6 and b["steps"] == r["loop_steps"] < 20


def test_ou_restatement_matches_the_oracle_view():
    """The numpy OU draw used by the checks equals the oracle's own (SingleAgent view: slots 2..11 are OU)."""
    from oracle import vss_oracle as orc
    n, seed, goff, step = 64, 3, 99, 5
    p = orc.default_params()
    st = orc.State(n)
    rb = np.ones(n, np.int64)
    orc.reset_dones(p, seed, goff, st, rb)
    rb[:] = 0
    prev = np.random.default_rng(0).uniform(-1, 1, (n, 2, 3, 2)).astype(np.float32)
    abuf = prev.copy()
    orc.step_view(p, seed, goff, step, st, orc.VIEW_SA, np.zeros((n, 2), np.float32), abuf, rb)
    ou = mc.ou_draw(p, seed, goff, step, prev.reshape(n, 12))
    keep = rb == 0
    np.testing.assert_allclose(abuf.reshape(n, 12)[keep, 2:], ou[keep, 2:], rtol=0, atol=2e-6)


def test_step_match_argument_validation_without_a_device():
    """Bad arguments are rejected before any CUDA call."""
    from rsoccer_isaac_cleanrl_b200 import _lib
    lib = _lib.load_library()
    teams = (_lib.MatchTeam * 2)()
    buf = C.c_void_p(16)  # never dereferenced: every call below fails validation first

    def call(t, n_matches=10, h=None):
        return lib.vss_step_match(h, t, buf, buf, None, 1065, n_matches, buf, None)

    assert call(None) == -1 and b"null" in lib.vss_last_error()
    teams[0].mode, teams[1].mode = _lib.TEAM_OU, 17
    assert call(teams) == -1 and b"unknown team mode" in lib.vss_last_error()
    teams[1].mode = -1
    assert call(teams) == -1 and b"unknown team mode" in lib.vss_last_error()
    for mode in (_lib.TEAM_SA, _lib.TEAM_CMA, _lib.TEAM_DMA):
        teams[1].mode = mode
        assert call(teams) == -1 and b"policy action" in lib.vss_last_error()
    teams[1].mode = _lib.TEAM_ZERO
    assert call(teams, n_matches=0) == -1 and b"n_matches" in lib.vss_last_error()
    assert call(teams) == -1 and b"null" in lib.vss_last_error()   # null handle
