"""Thin torch-facing wrapper of the C-ABI: borrows torch CUDA buffers by pointer, launches on
torch's current stream, owns nothing but the engine handle."""
import ctypes as C

import torch

from . import _lib
from ._lib import VIEW_CMA, VIEW_DMA, VIEW_SA, check


def _ptr(t, dtype, numel=None, name="tensor"):
    if t is None:
        return None
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f"{name}: expected a CUDA tensor")
    if t.dtype != dtype:
        raise TypeError(f"{name}: expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError(f"{name}: must be contiguous")
    if numel is not None and t.numel() != numel:
        raise ValueError(f"{name}: expected {numel} elements, got {t.numel()}")
    return t.data_ptr()


class Engine:
    """One engine per device: SoA field state in HBM + the fused step kernels."""

    def __init__(self, num_envs: int, device="cuda:0", seed: int = 0, global_env_offset: int = 0, params=None):
        self.lib = _lib.load_library()
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("rsoccer_isaac_cleanrl_b200 runs on a CUDA device only (no CPU fallback)")
        self.params = params if params is not None else _lib.default_params()
        self.num_envs = int(num_envs)
        self._h = C.c_void_p()
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        check(self.lib.vss_create(C.byref(self._h), C.byref(self.params), self.num_envs, int(global_env_offset),
                                  idx, int(seed) & 0xFFFFFFFFFFFFFFFF))
        self.ld = int(self.lib.vss_state_ld(self._h))
        self._aux_set = False
        self._packed_set = False
        self._opp_set = False

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.vss_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self):
        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- parameters
    def set_reward_weights(self, goal, grad, move, energy):
        w = (C.c_float * 4)(float(goal), float(grad), float(move), float(energy))
        check(self.lib.vss_set_reward_weights(self._h, w))

    # ---- state access
    def get_state(self):
        out = torch.empty((_lib.STATE_WORDS, self.ld), dtype=torch.float32, device=self.device)
        check(self.lib.vss_get_state(self._h, out.data_ptr(), self._stream()))
        return out

    def set_state(self, state):
        check(self.lib.vss_set_state(self._h, _ptr(state, torch.float32, _lib.STATE_WORDS * self.ld, "state"),
                                     self._stream()))

    @property
    def step_count(self):
        return int(self.lib.vss_step_count(self._h))

    @step_count.setter
    def step_count(self, n):
        check(self.lib.vss_set_step_count(self._h, int(n)))

    @property
    def sanitised_count(self):
        """Fields re-randomised by the non-finite guard so far (include/vss_b200.h); synchronises."""
        return int(self.lib.vss_sanitised_count(self._h))

    # ---- pipelining one step over several streams (include/vss_b200.h: vss_set_step_range)
    @property
    def step_granularity(self):
        return int(self.lib.vss_step_granularity(self._h))

    @property
    def warps_per_tile(self):
        """Launch shape of the step kernels (include/vss_b200.h: vss_set_step_warps_per_tile); 0 on write = automatic."""
        return int(self.lib.vss_step_warps_per_tile(self._h))

    @warps_per_tile.setter
    def warps_per_tile(self, w):
        check(self.lib.vss_set_step_warps_per_tile(self._h, int(w)))

    @property
    def fields_per_tile(self):
        """Fields per tile of the step kernels (include/vss_b200.h: vss_set_step_fields_per_tile); 0 on write = automatic."""
        return int(self.lib.vss_step_fields_per_tile(self._h))

    @fields_per_tile.setter
    def fields_per_tile(self, f):
        check(self.lib.vss_set_step_fields_per_tile(self._h, int(f)))

    def set_step_range(self, first_field=0, num_fields=0):
        check(self.lib.vss_set_step_range(self._h, int(first_field), int(num_fields)))

    # ---- hot path
    def reset_dones(self, reset_buf, obs):
        n = self.num_envs
        check(self.lib.vss_reset_dones(self._h, _ptr(reset_buf, torch.int64, n, "reset_buf"),
                                       _ptr(obs, torch.float32, n * 312, "obs"), self._stream()))

    def step(self, actions, reset_buf, obs, term_obs, rew, timeout, progress_f, post_state=None):
        n = self.num_envs
        args = [_ptr(actions, torch.float32, n * 12, "actions")]
        if post_state is not None:
            args.append(_ptr(post_state, torch.float32, None, "post_state"))
            if post_state.numel() < _lib.STATE_FLOATS * self.ld:
                raise ValueError("post_state: expected at least 58 x ld floats")
        args += [_ptr(reset_buf, torch.int64, n, "reset_buf"), _ptr(obs, torch.float32, n * 312, "obs"),
                 _ptr(term_obs, torch.float32, n * 312, "term_obs"), _ptr(rew, torch.float32, n * 24, "rew"),
                 _ptr(timeout, torch.uint8, n, "timeout"), _ptr(progress_f, torch.float32, n, "progress_f"),
                 self._stream()]
        fn = self.lib.vss_step if post_state is None else self.lib.vss_step_injected
        check(fn(self._h, *args))

    def step_view(self, view, policy_action, action_buf, reset_buf, obs_v, term_obs_v, rews_v, reward_v, done_v,
                  timeout_v, progress_v, ep_ret=None, ep_len=None, ret_ret=None, ret_len=None, obs_bf16=None,
                  done_f=None, timeout_f=None, packed=None, opponent=None):
        """`obs_bf16 (N',64) bf16`, `done_f (N') f32`, `timeout_f (N') f32`: optional side outputs
        (vss_set_step_aux) — the observation as the tensor-core MLP reads it, the flags as the GAE
        kernel reads them. `packed (N',112) uint8`: optional packed per-agent rows (vss_set_step_packed),
        a CUDA tensor or a pinned host tensor (the kernel then stores across PCIe).
        `opponent = (mode, policy_action or None, rows_bf16 or None, obs_f32 or None)`: the yellow team of this step
        (vss_set_view_opponent); None or mode TEAM_OU = no opponent, today's view step."""
        n = self.num_envs
        nv = n * 3 if view == VIEW_DMA else n
        adim = 6 if view == VIEW_CMA else 2
        if opponent is not None or self._opp_set:
            self.set_view_opponent(opponent)
        if obs_bf16 is not None or done_f is not None or timeout_f is not None or self._aux_set:
            check(self.lib.vss_set_step_aux(self._h, _ptr(obs_bf16, torch.bfloat16, nv * 64, "obs_bf16"),
                                            _ptr(done_f, torch.float32, nv, "done_f"),
                                            _ptr(timeout_f, torch.float32, nv, "timeout_f")))
            self._aux_set = obs_bf16 is not None or done_f is not None or timeout_f is not None
        if packed is not None or self._packed_set:
            ptr = None
            if packed is not None:
                if packed.dtype != torch.uint8 or not packed.is_contiguous() or packed.numel() != nv * _lib.PACKED_ROW_BYTES:
                    raise ValueError(f"packed: expected a contiguous uint8 tensor of {nv} x {_lib.PACKED_ROW_BYTES} bytes")
                if not (packed.is_cuda or packed.is_pinned()):
                    raise TypeError("packed: expected a CUDA tensor or a pinned host tensor")
                ptr = packed.data_ptr()
            check(self.lib.vss_set_step_packed(self._h, ptr))
            self._packed_set = packed is not None
        check(self.lib.vss_step_view(
            self._h, int(view), _ptr(policy_action, torch.float32, nv * adim, "policy_action"),
            _ptr(action_buf, torch.float32, n * 12, "action_buf"), _ptr(reset_buf, torch.int64, n, "reset_buf"),
            _ptr(obs_v, torch.float32, nv * 52, "obs_v"), _ptr(term_obs_v, torch.float32, nv * 52, "term_obs_v"),
            _ptr(rews_v, torch.float32, nv * 4, "rews_v"), _ptr(reward_v, torch.float32, nv, "reward_v"),
            _ptr(done_v, torch.int64, nv, "done_v"), _ptr(timeout_v, torch.uint8, nv, "timeout_v"),
            _ptr(progress_v, torch.float32, nv, "progress_v"), _ptr(ep_ret, torch.float32, nv * 4, "ep_ret"),
            _ptr(ep_len, torch.int32, nv, "ep_len"), _ptr(ret_ret, torch.float32, nv * 4, "ret_ret"),
            _ptr(ret_len, torch.int32, nv, "ret_len"), self._stream()))


    def set_view_opponent(self, opponent):
        """`vss_set_view_opponent`: opponent = (mode, policy_action, rows_bf16, obs_f32) as in step_view, or None."""
        n = self.num_envs
        if opponent is None or int(opponent[0]) == _lib.TEAM_OU:
            check(self.lib.vss_set_view_opponent(self._h, None))
            self._opp_set = False
            return
        mode, act, rows, obs = opponent
        mode = int(mode)
        ov = 3 * n if mode == _lib.TEAM_DMA else n
        policy = mode in (_lib.TEAM_SA, _lib.TEAM_CMA, _lib.TEAM_DMA)
        opp = _lib.ViewOpponent(
            mode, 0, _ptr(act, torch.float32, ov * (6 if mode == _lib.TEAM_CMA else 2), "policy_action") if policy else None,
            _ptr(rows, torch.bfloat16, ov * 64, "rows_bf16") if policy else None, _ptr(obs, torch.float32, n * 156, "obs_f32"))
        check(self.lib.vss_set_view_opponent(self._h, C.byref(opp)))
        self._opp_set = True

    def step_match(self, teams, action_buf, reset_buf, board, count_envs, n_matches, obs=None):
        """`vss_step_match`: one step of a two-team match (include/vss_b200.h). teams = [(mode, policy_action or
        None, rows_bf16 or None)] for blue and yellow; action_buf (N,2,3,2) f32 io; reset_buf (N) int64 io;
        board = int64 tensor of _lib.BOARD_WORDS words (the vss_match_board, zeroed before the first step);
        obs (N,2,3,52) f32 or None."""
        n = self.num_envs
        arr = (_lib.MatchTeam * 2)()
        for k, (mode, act, rows) in enumerate(teams):
            mode = int(mode)
            nv = 3 * n if mode == _lib.TEAM_DMA else n
            adim = 6 if mode == _lib.TEAM_CMA else 2
            policy = mode in (_lib.TEAM_SA, _lib.TEAM_CMA, _lib.TEAM_DMA)
            arr[k] = _lib.MatchTeam(mode, 0, _ptr(act, torch.float32, nv * adim, "policy_action") if policy else None,
                                    _ptr(rows, torch.bfloat16, nv * 64, "rows_bf16") if policy else None)
        check(self.lib.vss_step_match(
            self._h, arr, _ptr(action_buf, torch.float32, n * 12, "action_buf"),
            _ptr(reset_buf, torch.int64, n, "reset_buf"), _ptr(obs, torch.float32, n * 312, "obs"),
            int(count_envs), int(n_matches), _ptr(board, torch.int64, _lib.BOARD_WORDS, "board"), self._stream()))


def _engine_step_view_host(self, view, bufs, action_host, rows_host, num_ranges):
    """`vss_step_view_host`: pinned host action in, packed rows in pinned host memory out, pipelined over field
    ranges inside the library; returns when the rows are in host memory. `bufs`: _lib.ViewBuffers of device pointers."""
    if not (action_host.is_pinned() and rows_host.is_pinned()):
        raise TypeError("step_view_host: action_host and rows_host must be pinned host tensors")
    if action_host.dtype != torch.float32 or not action_host.is_contiguous():
        raise TypeError("step_view_host: action_host must be a contiguous float32 tensor")
    check(self.lib.vss_step_view_host(self._h, int(view), C.byref(bufs), action_host.data_ptr(), rows_host.data_ptr(),
                                      int(num_ranges), self._stream()))


Engine.step_view_host = _engine_step_view_host


def gae(rewards, values, next_values, next_dones, next_timeouts, gamma=0.99, gae_lambda=0.95, advantages=None,
        returns=None):
    """Reverse-scan GAE kernel (ppo_continuous_action_isaacgym.py:282-296). All (T,N) f32 CUDA."""
    lib = _lib.load_library()
    T, N = rewards.shape
    if advantages is None:
        advantages = torch.empty_like(rewards)
    if returns is None:
        returns = torch.empty_like(rewards)
    k = T * N
    check(lib.vss_gae(_ptr(rewards, torch.float32, k, "rewards"), _ptr(values, torch.float32, k, "values"),
                      _ptr(next_values, torch.float32, k, "next_values"),
                      _ptr(next_dones, torch.float32, k, "next_dones"),
                      _ptr(next_timeouts, torch.float32, k, "next_timeouts"),
                      _ptr(advantages, torch.float32, k, "advantages"), _ptr(returns, torch.float32, k, "returns"),
                      int(T), int(N), float(gamma), float(gae_lambda),
                      torch.cuda.current_stream(rewards.device).cuda_stream))
    return advantages, returns


EPI_BIAS_TANH_BF16, EPI_DTANH_BF16, EPI_ATOMIC_F32, EPI_BIAS_F32 = 0, 1, 2, 3


def gemm_bf16(a, b, out, epilogue, bias=None, aux=None, splits=1, mn_major=False, colsum=None):
    """tcgen05 GEMM (csrc/tc_gemm.cu). K-major: a [M,K], b [N,K]; MN-major: a [K,M], b [K,N]; bf16, last
    dimension contiguous. out [M,N] bf16 (epilogues 0,1) or f32 (2,3). colsum [N] f32 (dgrad epilogue
    only): += column sums of the output."""
    lib = _lib.load_library()
    if mn_major:
        K, M = a.shape
        N = b.shape[1]
        assert b.shape[0] == K
    else:
        M, K = a.shape
        N = b.shape[0]
        assert b.shape[1] == K
    assert a.dtype == torch.bfloat16 and b.dtype == torch.bfloat16 and a.stride(1) == 1 and b.stride(1) == 1
    assert out.shape == (M, N) and out.stride(1) == 1
    assert out.dtype == (torch.bfloat16 if epilogue in (EPI_BIAS_TANH_BF16, EPI_DTANH_BF16) else torch.float32)
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N and bias.is_contiguous()
    ld_aux = 0
    if aux is not None:
        assert aux.dtype == torch.bfloat16 and aux.shape == (M, N) and aux.stride(1) == 1
        ld_aux = aux.stride(0)
    if colsum is not None:
        assert colsum.dtype == torch.float32 and colsum.is_contiguous() and colsum.numel() == N
    rc = lib.vss_gemm_bf16_tn_colsum(a.data_ptr(), a.stride(0), b.data_ptr(), b.stride(0), out.data_ptr(),
                                     out.stride(0), M, N, K, int(epilogue), None if bias is None else bias.data_ptr(),
                                     None if aux is None else aux.data_ptr(), ld_aux, int(splits), int(bool(mn_major)),
                                     None if colsum is None else colsum.data_ptr(),
                                     torch.cuda.current_stream(a.device).cuda_stream)
    if rc != 0:
        raise RuntimeError(f"vss_gemm_bf16_tn failed ({rc}): {lib.vss_gemm_last_error().decode()}")
    return out


def colsum_bf16(x, out=None):
    """out[N] (f32) += column sums of x [M,N] bf16."""
    lib = _lib.load_library()
    M, N = x.shape
    assert x.dtype == torch.bfloat16 and x.stride(1) == 1
    if out is None:
        out = torch.zeros(N, device=x.device, dtype=torch.float32)
    rc = lib.vss_colsum_bf16(x.data_ptr(), x.stride(0), M, N, out.data_ptr(),
                             torch.cuda.current_stream(x.device).cuda_stream)
    if rc != 0:
        raise RuntimeError(lib.vss_gemm_last_error().decode())
    return out


def gather_pad_bf16(src, idx, ncol_pad):
    """[M, ncol_pad] bf16 = zero-padded src[idx] (src [R, ncol] f32 contiguous; idx int64 or None)."""
    lib = _lib.load_library()
    assert src.dtype == torch.float32 and src.is_contiguous() and src.dim() == 2
    M = src.shape[0] if idx is None else idx.numel()
    dst = torch.empty((M, ncol_pad), device=src.device, dtype=torch.bfloat16)
    rc = lib.vss_gather_pad_bf16(src.data_ptr(), None if idx is None else idx.data_ptr(), M, src.shape[1], ncol_pad,
                                 dst.data_ptr(), torch.cuda.current_stream(src.device).cuda_stream)
    if rc != 0:
        raise RuntimeError(lib.vss_gemm_last_error().decode())
    return dst


def head_forward(h, W, b, out=None):
    """out [M,n_out] f32 = h [M,256] bf16 @ W[n_out,256].T + b (CUDA-core kernel, one warp per row)."""
    lib = _lib.load_library()
    M, n_out = h.shape[0], W.shape[0]
    assert h.dtype == torch.bfloat16 and h.shape[1] == 256 and h.stride(1) == 1 and W.shape[1] == 256
    if out is None:
        out = torch.empty((M, n_out), device=h.device, dtype=torch.float32)
    assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == M * n_out
    rc = lib.vss_head_forward(h.data_ptr(), h.stride(0), W.contiguous().data_ptr(), b.contiguous().data_ptr(),
                              out.data_ptr(), M, n_out, torch.cuda.current_stream(h.device).cuda_stream)
    if rc != 0:
        raise RuntimeError(lib.vss_gemm_last_error().decode())
    return out


def mlp_forward_fused(x16, nets, epilogue_warps=0, stamps=None, sampling=None):
    """The whole MLP forward of 1 or 2 networks over the same rows in one launch (include/vss_b200.h:
    vss_mlp_forward_fused). x16 [M,64] bf16; nets = [(w16 list of 4 bf16 matrices, b list of 4 f32 vectors, head_w,
    head_b, out [M,n_out] f32 or None), ...]. sampling = dict(logstd, counter (uint32/int32 device word), seed,
    call_offset, action [M,A] f32, logprob [M] f32): also draws the action from network 0's output (then its `out`
    may be False = not stored). Returns the list of `out` tensors."""
    lib = _lib.load_library()
    M = x16.shape[0]
    assert x16.dtype == torch.bfloat16 and x16.shape[1] == 64 and x16.stride(1) == 1
    shapes = [(256, 64), (512, 256), (512, 512), (256, 512)]
    arr = (_lib.MlpNet * len(nets))()
    outs = []
    for k, (a, (w16, bs, head_w, head_b, out)) in enumerate(zip(arr, nets)):
        for l in range(4):
            assert w16[l].dtype == torch.bfloat16 and tuple(w16[l].shape) == shapes[l] and w16[l].is_contiguous()
            assert bs[l].dtype == torch.float32 and bs[l].is_contiguous() and bs[l].numel() == shapes[l][0]
            a.w[l], a.b[l] = w16[l].data_ptr(), bs[l].data_ptr()
        n_out = head_w.shape[0]
        assert head_w.dtype == torch.float32 and head_w.is_contiguous() and head_w.shape[1] == 256
        assert head_b.dtype == torch.float32 and head_b.is_contiguous()
        if out is False:
            assert k == 0 and sampling is not None
            out = None
        elif out is None:
            out = torch.empty((M, n_out), device=x16.device, dtype=torch.float32)
        if out is not None:
            assert out.dtype == torch.float32 and out.is_contiguous() and out.numel() == M * n_out
        a.head_w, a.head_b, a.n_out = head_w.data_ptr(), head_b.data_ptr(), n_out
        a.out = None if out is None else out.data_ptr()
        outs.append(out)
    samp = None
    if sampling is not None:
        A = nets[0][2].shape[0]
        act, lp, ls, ctr = sampling["action"], sampling["logprob"], sampling["logstd"], sampling["counter"]
        assert act.dtype == torch.float32 and act.is_contiguous() and act.numel() == M * A
        assert lp.dtype == torch.float32 and lp.is_contiguous() and lp.numel() == M
        assert ls.dtype == torch.float32 and ls.is_contiguous() and ls.numel() == A and ctr.element_size() == 4
        samp = _lib.MlpSampling(ls.data_ptr(), ctr.data_ptr(), int(sampling["seed"]) & (2 ** 64 - 1),
                                int(sampling.get("call_offset", 0)), 0, act.data_ptr(), lp.data_ptr())
    if stamps is not None:  # profiling hook: 11 int64 globaltimer stamps of the first CTA
        assert stamps.dtype == torch.int64 and stamps.is_cuda and stamps.numel() >= 11 and stamps.is_contiguous()
    rc = lib.vss_mlp_forward_fused_timed(x16.data_ptr(), x16.stride(0), M, arr, len(nets),
                                         None if samp is None else C.byref(samp), int(epilogue_warps),
                                         None if stamps is None else stamps.data_ptr(),
                                         torch.cuda.current_stream(x16.device).cuda_stream)
    if rc != 0:
        raise RuntimeError(lib.vss_gemm_last_error().decode())
    return outs


def head_backward(dout, h, W, dW=None, db=None, dz_colsum=None):
    """(dz [M,256] bf16, dW [n_out,256] f32, db [n_out] f32) of the head, tanh' of h fused into dz.
    dW / db, when given, are accumulated into (contiguous f32 buffers such as the .grad views)."""
    lib = _lib.load_library()
    M, n_out = dout.shape
    dout = dout.contiguous()
    dz = torch.empty((M, 256), device=h.device, dtype=torch.bfloat16)
    if dW is None:
        dW = torch.zeros((n_out, 256), device=h.device, dtype=torch.float32)
    if db is None:
        db = torch.zeros(n_out, device=h.device, dtype=torch.float32)
    assert dW.is_contiguous() and db.is_contiguous() and dW.numel() == n_out * 256 and db.numel() == n_out
    if dz_colsum is not None:  # += column sums of dz: the bias gradient of the last hidden layer
        assert dz_colsum.dtype == torch.float32 and dz_colsum.is_contiguous() and dz_colsum.numel() == 256
    rc = lib.vss_head_backward(dout.data_ptr(), h.data_ptr(), h.stride(0), W.contiguous().data_ptr(), dz.data_ptr(), 256,
                               dW.data_ptr(), db.data_ptr(), None if dz_colsum is None else dz_colsum.data_ptr(),
                               M, n_out, torch.cuda.current_stream(h.device).cuda_stream)
    if rc != 0:
        raise RuntimeError(lib.vss_gemm_last_error().decode())
    return dz, dW, db


def _ppo_check(lib, rc):
    if rc != 0:
        raise RuntimeError(lib.vss_ppo_last_error().decode())


def policy_sample(mean, logstd, seed, counter, action=None, logprob=None):
    """action = mean + exp(logstd) * N(0,1), logprob = Normal.log_prob(action).sum(1) in one launch
    (Agent.get_action_and_value without a given action, ppo…:155-164). `counter` is a device uint32
    word (int32 tensor of one element) advanced by the call."""
    lib = _lib.load_library()
    M, A = mean.shape
    assert mean.dtype == torch.float32 and mean.is_contiguous() and logstd.numel() == A and logstd.is_contiguous()
    assert counter.dtype == torch.int32 and counter.numel() == 1
    if action is None:
        action = torch.empty_like(mean)
    if logprob is None:
        logprob = torch.empty(M, device=mean.device, dtype=torch.float32)
    assert action.is_contiguous() and logprob.is_contiguous() and action.numel() == M * A and logprob.numel() == M
    _ppo_check(lib, lib.vss_policy_sample(mean.data_ptr(), logstd.data_ptr(), M, A, int(seed) & (2**64 - 1),
                                          counter.data_ptr(), action.data_ptr(), logprob.data_ptr(),
                                          torch.cuda.current_stream(mean.device).cuda_stream))
    return action, logprob


def compact_nonzero(flags, index_list, count):
    """index_list[k] = flat index of the k-th non-zero entry of `flags` (f32, any order), count[0] = how many there are
    (include/vss_b200.h: vss_compact_nonzero). Static shapes: index_list (int64, capacity rows) and count (int32, 1)
    are caller-owned; the caller checks count <= capacity."""
    lib = _lib.load_library()
    assert flags.dtype == torch.float32 and flags.is_contiguous() and index_list.dtype == torch.int64
    assert index_list.is_contiguous() and count.dtype == torch.int32 and count.numel() == 1
    _ppo_check(lib, lib.vss_compact_nonzero(flags.data_ptr(), flags.numel(), index_list.data_ptr(), index_list.numel(),
                                            count.data_ptr(), torch.cuda.current_stream(flags.device).cuda_stream))


def scatter_rows(dst, index_list, src, count):
    """dst.view(-1)[index_list[k]] = src[k] for k < min(count, capacity) (vss_scatter_rows_f32)."""
    lib = _lib.load_library()
    assert dst.dtype == torch.float32 and dst.is_contiguous() and src.dtype == torch.float32 and src.is_contiguous()
    assert src.numel() >= index_list.numel() and index_list.dtype == torch.int64 and count.dtype == torch.int32
    _ppo_check(lib, lib.vss_scatter_rows_f32(dst.data_ptr(), index_list.data_ptr(), src.data_ptr(), count.data_ptr(),
                                             index_list.numel(), torch.cuda.current_stream(dst.device).cuda_stream))


PPO_STATS = ("pg_loss", "v_loss", "entropy", "old_approx_kl", "approx_kl", "clipfrac", "loss")


def ppo_loss(mean, value, logstd, b_action, b_logprob, b_adv, b_ret, b_val, inds, clip_coef, ent_coef, vf_coef,
             norm_adv, clip_vloss, d_logstd, d_mean=None, d_value=None, stats=None, scratch=None):
    """One PPO minibatch loss and its gradients w.r.t. the network outputs (ppo…:314-352) in two
    launches. Returns (d_mean, d_value, stats[8]); d_logstd is accumulated in place."""
    lib = _lib.load_library()
    B, A = mean.shape
    dev = mean.device
    for t in (mean, value, logstd, b_action, b_logprob, b_adv, b_ret, d_logstd):
        assert t.dtype == torch.float32 and t.is_contiguous()
    assert value.numel() == B and d_logstd.numel() == A and (inds is None or (inds.dtype == torch.long and inds.numel() == B))
    d_mean = torch.empty_like(mean) if d_mean is None else d_mean
    d_value = torch.empty((B, 1), device=dev, dtype=torch.float32) if d_value is None else d_value
    stats = torch.empty(8, device=dev, dtype=torch.float32) if stats is None else stats
    scratch = torch.empty(2, device=dev, dtype=torch.float64) if scratch is None else scratch
    _ppo_check(lib, lib.vss_ppo_loss(
        mean.data_ptr(), value.data_ptr(), logstd.data_ptr(), b_action.data_ptr(), b_logprob.data_ptr(),
        b_adv.data_ptr(), b_ret.data_ptr(), None if b_val is None else b_val.data_ptr(),
        None if inds is None else inds.data_ptr(), B, A, float(clip_coef), float(ent_coef), float(vf_coef),
        int(bool(norm_adv)), int(bool(clip_vloss)), d_mean.data_ptr(), d_value.data_ptr(), d_logstd.data_ptr(),
        stats.data_ptr(), scratch.data_ptr(), torch.cuda.current_stream(dev).cuda_stream))
    return d_mean, d_value, stats


def convert_bf16_batch(jobs):
    """jobs: list of (src f32 [R,C] contiguous, dst bf16 2-D with unit column stride, transpose)."""
    lib = _lib.load_library()
    for start in range(0, len(jobs), _lib.MAX_CONVERT_JOBS):
        chunk = jobs[start:start + _lib.MAX_CONVERT_JOBS]
        arr = (_lib.ConvertJob * len(chunk))()
        for k, (src, dst, tr) in enumerate(chunk):
            assert src.dtype == torch.float32 and src.is_contiguous() and src.dim() == 2
            assert dst.dtype == torch.bfloat16 and dst.stride(1) == 1
            R, Cc = src.shape
            assert dst.shape[0] >= (Cc if tr else R) and dst.shape[1] >= (R if tr else Cc)
            arr[k] = _lib.ConvertJob(src.data_ptr(), dst.data_ptr(), R, Cc, dst.stride(0), int(bool(tr)))
        _ppo_check(lib, lib.vss_convert_bf16_batch(arr, len(chunk), torch.cuda.current_stream(chunk[0][0].device).cuda_stream))


def clip_adam(params, grads, exp_avg, exp_avg_sq, state, grad_scale, max_grad_norm, beta1, beta2, eps):
    """clip_grad_norm_ + Adam.step() on flat f32 buffers (ppo…:353-354); state = device [t, lr, 0]."""
    lib = _lib.load_library()
    for t in (params, grads, exp_avg, exp_avg_sq, state):
        assert t.dtype == torch.float32 and t.is_contiguous()
    _ppo_check(lib, lib.vss_clip_adam(params.data_ptr(), grads.data_ptr(), exp_avg.data_ptr(), exp_avg_sq.data_ptr(),
                                      params.numel(), state.data_ptr(), float(grad_scale), float(max_grad_norm),
                                      float(beta1), float(beta2), float(eps),
                                      torch.cuda.current_stream(params.device).cuda_stream))
