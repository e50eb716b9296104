"""Shared pieces of the picture tests: the host emulator of csrc/vss_render.cuh and random field states.

The emulator (tests/emu/vss_render_emu.cpp) compiles the product's per-pixel source on the host; the numpy
restatement (oracle/vss_render.py) is the independent statement of DESIGN.md §4.7 both are checked against.
"""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SIZES = ((560, 720), (64, 80), (128, 64))  # the default 400 px/m, a small one, and unequal x / y scales

_lib = None


def emu_lib():
    global _lib
    if _lib is None:
        d = os.path.join(ROOT, "tests", "emu")
        subprocess.run(["make", "-C", d, "-f", "render.mk"], check=True, capture_output=True)
        _lib = C.CDLL(os.path.join(d, "libvss_render_emu.so"))
    return _lib


def emu_render(params, soa, first, num, height, width):
    soa = np.ascontiguousarray(soa, np.float32)
    out = np.zeros((num, height, width, 3), np.uint8)
    rc = emu_lib().emu_render(C.byref(params), soa.ctypes.data_as(C.c_void_p), C.c_longlong(soa.shape[1]),
                              C.c_longlong(first), C.c_int(num), C.c_int(height), C.c_int(width),
                              out.ctypes.data_as(C.c_void_p))
    assert rc == 0
    return out


def _yaw(s, b, a):
    s[b + 4] = np.cos(a)
    s[b + 5] = np.sin(a)


def random_states(n, seed, ld=None, spread=1.2):
    """n SoA states (60 x ld): ball and robots uniform over [-spread, spread]^2 (the window is 0.9 x 0.7, so some
    lie beyond it), random yaws; every fourth field packs its robots and ball into a 0.1 m square (overlapping
    bodies)."""
    rng = np.random.default_rng(seed)
    ld = ld or (n + 31) // 32 * 32
    s = np.zeros((60, ld), np.float32)
    s[0:4, :n] = rng.uniform(-spread, spread, (4, n))
    for r in range(6):
        b = 4 + 9 * r
        s[b:b + 4, :n] = rng.uniform(-spread, spread, (4, n))
        _yaw(s[:, :n], b, rng.uniform(-np.pi, np.pi, n))
        s[b + 6:b + 9, :n] = rng.uniform(-1, 1, (3, n))
    packed = np.arange(n) % 4 == 3
    centre = rng.uniform(-0.7, 0.7, (2, n))
    for w in [0, 1] + [4 + 9 * r + k for r in range(6) for k in (0, 1)]:
        s[w, :n] = np.where(packed, centre[w % 2 if w < 2 else (w - 4) % 9] + rng.uniform(-0.05, 0.05, n), s[w, :n])
    return s


def oracle_rollout_states(n, steps, seed):
    """SoA states of an oracle rollout (reset, then `steps` steps of uniform random actions), one per step."""
    from oracle import vss_oracle as orc
    p = orc.default_params()
    st = orc.State(n)
    reset = np.ones(n, np.int64)
    orc.reset_dones(p, seed, 0, st, reset)
    reset[:] = 0
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(steps):
        orc.step(p, seed, 0, st, rng.uniform(-1, 1, (n, 2, 3, 2)).astype(np.float32), reset)
        out.append(st.to_soa())
    return out
