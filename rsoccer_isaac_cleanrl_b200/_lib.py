"""ctypes binding of libvss_b200.so (C-ABI declared in include/vss_b200.h).

The library is built in-tree by `csrc/Makefile` (nvcc, sm_100a) so that it travels with the
repo snapshot to the GPU box. Loading never falls back to anything else: a missing library
or a missing B200 raises.
"""
import ctypes as C
import os
import subprocess

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libvss_b200.so")
CSRC = os.path.join(_PKG, "csrc")

VIEW_SA, VIEW_CMA, VIEW_DMA = 0, 1, 2
STATE_FLOATS, STATE_WORDS = 58, 60
W_PROGRESS, W_EPISODE = 58, 59
PACKED_ROW_BYTES = 112  # VSS_PACKED_ROW_BYTES: 52 bf16 obs | f32 reward | u8 done | u8 timeout | 2 zero bytes


class VssParams(C.Structure):
    """`vss_params` of include/vss_b200.h."""

    _fields_ = [
        ("dt", C.c_float), ("substeps", C.c_int32), ("max_episode_length", C.c_int32),
        ("field_half_length", C.c_float), ("field_half_width", C.c_float),
        ("goal_half_width", C.c_float), ("goal_depth", C.c_float),
        ("ball_radius", C.c_float), ("ball_mass", C.c_float), ("ball_drag", C.c_float),
        ("robot_half_size", C.c_float), ("robot_mass", C.c_float), ("robot_inertia", C.c_float),
        ("wheel_radius", C.c_float), ("wheel_half_track", C.c_float), ("wheel_coll_radius", C.c_float),
        ("max_wheel_rad_s", C.c_float), ("drive_damping", C.c_float), ("drive_max_torque", C.c_float),
        ("wheel_inertia", C.c_float), ("mu_traction", C.c_float), ("mu_lateral", C.c_float),
        ("gravity", C.c_float),
        ("restitution", C.c_float), ("mu_ball_robot", C.c_float), ("mu_ball_wall", C.c_float),
        ("mu_robot_wall", C.c_float),
        ("reset_scale_x", C.c_float), ("reset_scale_y", C.c_float), ("min_placement_dist", C.c_float),
        ("ball_reset_speed", C.c_float),
        ("w_goal", C.c_float), ("w_grad", C.c_float), ("w_move", C.c_float), ("w_energy", C.c_float),
        ("ou_theta", C.c_float), ("ou_sigma", C.c_float),
    ]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ViewBuffers(C.Structure):
    """`vss_view_buffers` of include/vss_b200.h."""

    _fields_ = [(k, C.c_void_p) for k in (
        "policy_action", "action_buf", "reset_buf", "obs_v", "term_obs_v", "rews_v", "reward_v", "done_v", "timeout_v",
        "progress_v", "ep_ret", "ep_len", "ret_ret", "ret_len", "packed_rows")]


class ConvertJob(C.Structure):
    """`vss_convert_job` of include/vss_b200.h."""

    _fields_ = [("src", C.c_void_p), ("dst", C.c_void_p), ("rows", C.c_int32), ("cols", C.c_int32),
                ("ld_dst", C.c_int32), ("transpose", C.c_int32)]


MAX_CONVERT_JOBS = 8

TEAM_ZERO, TEAM_OU, TEAM_SA, TEAM_CMA, TEAM_DMA, TEAM_EXTERNAL = 0, 1, 2, 3, 4, 5


class MatchTeam(C.Structure):
    """`vss_match_team` of include/vss_b200.h."""

    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("policy_action", C.c_void_p), ("rows_bf16", C.c_void_p)]


class ViewOpponent(C.Structure):
    """`vss_view_opponent` of include/vss_b200.h."""

    _fields_ = [("mode", C.c_int32), ("reserved", C.c_int32), ("policy_action", C.c_void_p), ("rows_bf16", C.c_void_p),
                ("obs_f32", C.c_void_p)]


# `vss_match_board` of include/vss_b200.h as int64 words: matches, length_sum, score_sum (float64 bits), steps,
# frozen (low 32 bits)
BOARD_WORDS = 5


class MlpSampling(C.Structure):
    """`vss_mlp_sampling` of include/vss_b200.h."""

    _fields_ = [("logstd", C.c_void_p), ("counter", C.c_void_p), ("seed", C.c_uint64), ("call_offset", C.c_uint32),
                ("reserved", C.c_uint32), ("action", C.c_void_p), ("logprob", C.c_void_p)]


class MlpNet(C.Structure):
    """`vss_mlp_net` of include/vss_b200.h."""

    _fields_ = [("w", C.c_void_p * 4), ("b", C.c_void_p * 4), ("head_w", C.c_void_p), ("head_b", C.c_void_p),
                ("out", C.c_void_p), ("n_out", C.c_int32), ("reserved", C.c_int32)]


# every symbol include/vss_b200.h declares: name -> (restype, argtypes)
_VP = C.c_void_p
_SYMBOLS = {
    "vss_default_params": (C.c_int, [C.POINTER(VssParams)]),
    "vss_create": (C.c_int, [C.POINTER(_VP), C.POINTER(VssParams), C.c_int64, C.c_int64, C.c_int, C.c_uint64]),
    "vss_destroy": (C.c_int, [_VP]),
    "vss_num_envs": (C.c_int64, [_VP]),
    "vss_state_ld": (C.c_int64, [_VP]),
    "vss_set_reward_weights": (C.c_int, [_VP, C.POINTER(C.c_float)]),
    "vss_reset_dones": (C.c_int, [_VP, _VP, _VP, _VP]),
    "vss_step": (C.c_int, [_VP] * 9),
    "vss_step_injected": (C.c_int, [_VP] * 10),
    "vss_step_view": (C.c_int, [_VP, C.c_int] + [_VP] * 15),
    "vss_step_view_host": (C.c_int, [_VP, C.c_int, C.POINTER(ViewBuffers), _VP, _VP, C.c_int, _VP]),
    "vss_set_step_aux": (C.c_int, [_VP, _VP, _VP, _VP]),
    "vss_set_step_packed": (C.c_int, [_VP, _VP]),
    "vss_step_granularity": (C.c_int64, [_VP]),
    "vss_set_step_warps_per_tile": (C.c_int, [_VP, C.c_int]),
    "vss_step_warps_per_tile": (C.c_int, [_VP]),
    "vss_set_step_fields_per_tile": (C.c_int, [_VP, C.c_int]),
    "vss_step_fields_per_tile": (C.c_int, [_VP]),
    "vss_set_step_range": (C.c_int, [_VP, C.c_int64, C.c_int64]),
    "vss_step_match": (C.c_int, [_VP, C.POINTER(MatchTeam), _VP, _VP, _VP, C.c_int64, C.c_int64, _VP, _VP]),
    "vss_set_view_opponent": (C.c_int, [_VP, C.POINTER(ViewOpponent)]),
    "vss_get_state": (C.c_int, [_VP, _VP, _VP]),
    "vss_set_state": (C.c_int, [_VP, _VP, _VP]),
    "vss_step_count": (C.c_uint64, [_VP]),
    "vss_set_step_count": (C.c_int, [_VP, C.c_uint64]),
    "vss_sanitised_count": (C.c_uint64, [_VP]),
    "vss_gae": (C.c_int, [_VP] * 7 + [C.c_int32, C.c_int64, C.c_double, C.c_double, _VP]),
    "vss_gemm_bf16_tn": (C.c_int, [_VP, C.c_int, _VP, C.c_int, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _VP,
                                  _VP, C.c_int, C.c_int, C.c_int, _VP]),
    "vss_gemm_bf16_tn_colsum": (C.c_int, [_VP, C.c_int, _VP, C.c_int, _VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         _VP, _VP, C.c_int, C.c_int, C.c_int, _VP, _VP]),
    "vss_gemm_last_error": (C.c_char_p, []),
    "vss_head_forward": (C.c_int, [_VP, C.c_int, _VP, _VP, _VP, C.c_int, C.c_int, _VP]),
    "vss_mlp_forward_fused": (C.c_int, [_VP, C.c_int, C.c_int, C.POINTER(MlpNet), C.c_int, C.POINTER(MlpSampling),
                                        C.c_int, _VP]),
    "vss_mlp_forward_fused_timed": (C.c_int, [_VP, C.c_int, C.c_int, C.POINTER(MlpNet), C.c_int,
                                              C.POINTER(MlpSampling), C.c_int, _VP, _VP]),
    "vss_head_backward": (C.c_int, [_VP, _VP, C.c_int, _VP, _VP, C.c_int, _VP, _VP, _VP, C.c_int, C.c_int, _VP]),
    "vss_colsum_bf16": (C.c_int, [_VP, C.c_int, C.c_int, C.c_int, _VP, _VP]),
    "vss_gather_pad_bf16": (C.c_int, [_VP, _VP, C.c_int, C.c_int, C.c_int, _VP, _VP]),
    "vss_policy_sample": (C.c_int, [_VP, _VP, C.c_int64, C.c_int, C.c_uint64, _VP, _VP, _VP, _VP]),
    "vss_compact_nonzero": (C.c_int, [_VP, C.c_int64, _VP, C.c_int, _VP, _VP]),
    "vss_scatter_rows_f32": (C.c_int, [_VP, _VP, _VP, _VP, C.c_int, _VP]),
    "vss_ppo_loss": (C.c_int, [_VP] * 9 + [C.c_int64, C.c_int, C.c_float, C.c_float, C.c_float, C.c_int, C.c_int] +
                     [_VP] * 6),
    "vss_convert_bf16_batch": (C.c_int, [C.POINTER(ConvertJob), C.c_int, _VP]),
    "vss_clip_adam": (C.c_int, [_VP] * 4 + [C.c_int64, _VP, C.c_float, C.c_float, C.c_float, C.c_float, C.c_float,
                                            _VP]),
    "vss_ppo_last_error": (C.c_char_p, []),
    "vss_peer_create": (C.c_int, [C.POINTER(_VP), C.c_int, C.c_int, C.c_int, C.c_int64]),
    "vss_peer_ipc_handle": (C.c_int, [_VP, _VP]),
    "vss_peer_connect": (C.c_int, [_VP, _VP]),
    "vss_peer_buffer": (_VP, [_VP]),
    "vss_peer_num_floats": (C.c_int64, [_VP]),
    "vss_peer_allreduce": (C.c_int, [_VP, _VP, _VP]),
    "vss_peer_destroy": (C.c_int, [_VP]),
    "vss_peer_last_error": (C.c_char_p, []),
    "vss_philox4x32_10": (None, [_VP, _VP, _VP]),
    "vss_last_error": (C.c_char_p, []),
    "vss_version": (C.c_char_p, []),
}


def declared_symbols():
    return sorted(_SYMBOLS)


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into libvss_b200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC] + (["-B"] if force else [])
    r = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout, r.stderr)
    if r.returncode != 0:
        raise RuntimeError("building libvss_b200.so failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


_lib = None


def load_library():
    """Load libvss_b200.so; raises if it has not been built (there is no fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA extension is not built. Run "
                "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
                "This package has no CPU or PyTorch fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in _SYMBOLS.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int):
    if rc != 0:
        lib = load_library()
        msg = lib.vss_last_error().decode() or lib.vss_gemm_last_error().decode()
        raise RuntimeError(f"libvss_b200 error {rc}: {msg}")


def default_params() -> VssParams:
    p = VssParams()
    check(load_library().vss_default_params(C.byref(p)))
    return p
