"""CPU: the opponent view step (vss_step_view with vss_set_view_opponent) on the host emulation of the product's lane
code, against the restatement driven through the emulated full-contract step; argument validation of the setter
without a device."""
import ctypes as C

import pytest

import opponent_checks as oc
from backends import VIEW_CMA, VIEW_DMA, VIEW_SA, EmuBackend, with_wpt

VIEWS = {"sa": VIEW_SA, "cma": VIEW_CMA, "dma": VIEW_DMA}
MODES = {"zero": oc.ZERO, "sa": oc.SA, "cma": oc.CMA, "dma": oc.DMA, "external": oc.EXTERNAL}


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("view", list(VIEWS))
def test_opponent_view_one_warp_per_tile(view, mode):
    oc.check_opponent(EmuBackend, VIEWS[view], MODES[mode])


@pytest.mark.parametrize("wpt,fpt", [(8, 32), (7, 16), (2, 8)])
@pytest.mark.parametrize("view,mode", [("sa", "sa"), ("cma", "dma"), ("dma", "external"), ("sa", "zero"),
                                       ("dma", "cma")])
def test_opponent_view_shared_tile(view, mode, wpt, fpt):
    oc.check_opponent(with_wpt(EmuBackend, wpt, fpt), VIEWS[view], MODES[mode], steps=10)


def test_opponent_rows_without_f32_observation():
    """obs_f32 is optional: the bf16 rows alone (the training path) are the same."""
    oc.check_opponent(EmuBackend, VIEW_SA, oc.SA, want_obs=False, steps=10)


@pytest.mark.parametrize("view", list(VIEWS))
def test_mode_ou_equals_no_opponent(view):
    oc.check_ou_mode_is_no_opponent(EmuBackend, VIEWS[view])


def test_set_view_opponent_argument_validation_without_a_device():
    """Bad arguments are rejected before anything else; NULL clears (a null handle is still an error)."""
    from rsoccer_isaac_cleanrl_b200 import _lib
    lib = _lib.load_library()
    opp = _lib.ViewOpponent()
    opp.mode = 17
    assert lib.vss_set_view_opponent(None, C.byref(opp)) == -1 and b"unknown team mode" in lib.vss_last_error()
    opp.mode = -1
    assert lib.vss_set_view_opponent(None, C.byref(opp)) == -1 and b"unknown team mode" in lib.vss_last_error()
    for mode in (_lib.TEAM_SA, _lib.TEAM_CMA, _lib.TEAM_DMA):
        opp.mode = mode
        assert lib.vss_set_view_opponent(None, C.byref(opp)) == -1 and b"policy action" in lib.vss_last_error()
    for mode in (_lib.TEAM_ZERO, _lib.TEAM_OU, _lib.TEAM_EXTERNAL):
        opp.mode = mode
        assert lib.vss_set_view_opponent(None, C.byref(opp)) == -1 and b"null handle" in lib.vss_last_error()
    opp.mode, opp.policy_action = _lib.TEAM_SA, 16
    assert lib.vss_set_view_opponent(None, C.byref(opp)) == -1 and b"null handle" in lib.vss_last_error()
    assert lib.vss_set_view_opponent(None, None) == -1 and b"null handle" in lib.vss_last_error()
