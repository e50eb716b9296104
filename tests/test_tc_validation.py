"""CPU: the C-ABI of the tensor-core GEMM, head, column-sum and gather kernels (csrc/tc_gemm.cu) rejects operand
layouts its kernels would fault on (short or unaligned row strides, unaligned pointers) before any CUDA call.

The calls use fake pointers that are never dereferenced, in a child process that sees no CUDA device: a layout that
passes validation ends in a CUDA error (VSS_E_CUDA), never in a launch, even on a machine with a GPU."""
import json
import os
import subprocess
import sys

from conftest import ROOT

# Runs in the child: loads libvss_b200.so through _lib (no torch import), makes every call of CASES and prints
# [name, return code, error message] per call as JSON.
_CHILD = r"""
import ctypes as C, importlib.util, json, sys
spec = importlib.util.spec_from_file_location("_lib", sys.argv[1])
_lib = importlib.util.module_from_spec(spec)
spec.loader.exec_module(_lib)
lib = _lib.load_library()
out = []
for name, fn, args in json.loads(sys.argv[2]):
    rc = getattr(lib, fn)(*args)
    out.append([name, rc, lib.vss_gemm_last_error().decode()])
print(json.dumps(out))
"""

P = 0x7f0000000000   # fake device address, 16-byte aligned; never dereferenced
INVALID, CUDA = -1, -2
EPI_BIAS_TANH_BF16, EPI_DTANH_BF16, EPI_ATOMIC_F32, EPI_BIAS_F32 = 0, 1, 2, 3


def _gemm(lda=64, ldb=64, out=P, ldo=256, M=256, N=256, K=64, epi=EPI_BIAS_TANH_BF16, bias=P, aux=None, ld_aux=0,
          splits=1, mn=0):
    return "vss_gemm_bf16_tn_colsum", [P, lda, P, ldb, out, ldo, M, N, K, epi, bias, aux, ld_aux, splits, mn, None, None]


def _head_fwd(h=P, ldh=256, n_out=2):
    return "vss_head_forward", [h, ldh, P, P, P, 100, n_out, None]


def _head_bwd(h=P, ldh=256, dz=P, ldz=256, n_out=2):
    return "vss_head_backward", [P, h, ldh, P, dz, ldz, P, P, None, 100, n_out, None]


def _colsum(x=P, ld=256, N=256):
    return "vss_colsum_bf16", [x, ld, 100, N, P, None]


def _gather(dst=P, ncol_pad=64):
    return "vss_gather_pad_bf16", [P, None, 100, 52, ncol_pad, dst, None]


# name -> (call, expected return code, substring of the message for VSS_E_INVALID)
CASES = {
    # layouts the kernels handle: validation passes and the first CUDA call fails (no device)
    "gemm forward ok": (_gemm(), CUDA, None),
    "gemm forward strided ok": (_gemm(lda=72, ldb=136, ldo=264), CUDA, None),
    "gemm forward pair ok": (_gemm(M=20000), CUDA, None),
    "gemm dgrad ok": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P, ld_aux=264), CUDA, None),
    "gemm dgrad pair ok": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P, ld_aux=256, M=20000), CUDA, None),
    "gemm bias f32 ok": (_gemm(epi=EPI_BIAS_F32, ldo=260), CUDA, None),
    "gemm bias f32 no bias ok": (_gemm(epi=EPI_BIAS_F32, bias=None), CUDA, None),
    "gemm atomic unaligned ok": (_gemm(epi=EPI_ATOMIC_F32, bias=None, out=P + 4, ldo=257, splits=3), CUDA, None),
    "gemm wgrad ok": (_gemm(lda=256, ldb=64, M=256, N=64, K=1000, epi=EPI_ATOMIC_F32, bias=None, ldo=64, mn=1,
                            splits=4), CUDA, None),
    "head fwd ok": (_head_fwd(ldh=264), CUDA, None),
    "head bwd ok": (_head_bwd(ldh=264, ldz=512, n_out=6), CUDA, None),
    "colsum ok": (_colsum(x=P + 4, ld=258, N=258), CUDA, None),
    "gather ok": (_gather(dst=P + 4, ncol_pad=54), CUDA, None),
    # gemm: row strides and alignment of every operand the epilogues touch with vector accesses
    "gemm ldo < N": (_gemm(ldo=192), INVALID, "ldo"),
    "gemm ldo % 8 (bf16)": (_gemm(ldo=260), INVALID, "ldo"),
    "gemm ldo % 8 (dgrad)": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P, ld_aux=256, ldo=257), INVALID, "ldo"),
    "gemm ldo % 4 (bias f32)": (_gemm(epi=EPI_BIAS_F32, ldo=258), INVALID, "ldo"),
    "gemm ldo < N (atomic)": (_gemm(epi=EPI_ATOMIC_F32, bias=None, ldo=255), INVALID, "ldo"),
    "gemm out unaligned (bf16)": (_gemm(out=P + 8), INVALID, "aligned"),
    "gemm out unaligned (dgrad)": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P, ld_aux=256, out=P + 2), INVALID, "aligned"),
    "gemm out unaligned (bias f32)": (_gemm(epi=EPI_BIAS_F32, out=P + 4), INVALID, "aligned"),
    "gemm bias unaligned": (_gemm(bias=P + 4), INVALID, "bias"),
    "gemm bias unaligned (bias f32)": (_gemm(epi=EPI_BIAS_F32, bias=P + 8), INVALID, "bias"),
    "gemm ld_aux odd": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P, ld_aux=257), INVALID, "ld_aux"),
    "gemm ld_aux odd (pair size)": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P, ld_aux=259, M=20000), INVALID, "ld_aux"),
    "gemm ld_aux < N": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P, ld_aux=248), INVALID, "ld_aux"),
    "gemm aux unaligned": (_gemm(epi=EPI_DTANH_BF16, bias=None, aux=P + 8, ld_aux=256), INVALID, "aux"),
    "gemm lda < K": (_gemm(lda=56), INVALID, "lda"),
    "gemm ldb < K": (_gemm(ldb=56), INVALID, "lda"),
    "gemm lda < M (MN-major)": (_gemm(lda=128, ldb=64, M=256, N=64, K=1000, epi=EPI_ATOMIC_F32, bias=None, ldo=64,
                                      mn=1), INVALID, "lda"),
    "gemm ldb < N (MN-major)": (_gemm(lda=256, ldb=56, M=256, N=64, K=1000, epi=EPI_ATOMIC_F32, bias=None, ldo=64,
                                      mn=1), INVALID, "lda"),
    "gemm MN-major forward": (_gemm(lda=256, ldb=256, mn=1), INVALID, "epilogue"),
    "gemm unknown epilogue": (_gemm(epi=4), INVALID, "epilogue"),
    # head kernels: h (and dz) rows are 16-byte vector accesses
    "head fwd ldh < 256": (_head_fwd(ldh=248), INVALID, "ldh"),
    "head fwd ldh % 8": (_head_fwd(ldh=260), INVALID, "ldh"),
    "head fwd h unaligned": (_head_fwd(h=P + 8), INVALID, "aligned"),
    "head bwd ldh % 8": (_head_bwd(ldh=257), INVALID, "ldh"),
    "head bwd ldh < 256": (_head_bwd(ldh=128), INVALID, "ldh"),
    "head bwd ldz < 256": (_head_bwd(ldz=248), INVALID, "ldz"),
    "head bwd ldz % 8": (_head_bwd(ldz=260), INVALID, "ldz"),
    "head bwd h unaligned": (_head_bwd(h=P + 2), INVALID, "aligned"),
    "head bwd dz unaligned": (_head_bwd(dz=P + 8), INVALID, "aligned"),
    # column sums read bf16 pairs; the gather writes them
    "colsum ld odd": (_colsum(ld=257), INVALID, "ld"),
    "colsum ld < N": (_colsum(ld=254), INVALID, "ld"),
    "colsum x unaligned": (_colsum(x=P + 2), INVALID, "aligned"),
    "gather dst unaligned": (_gather(dst=P + 2), INVALID, "aligned"),
}


def test_tc_c_abi_rejects_layouts_its_kernels_fault_on():
    from rsoccer_isaac_cleanrl_b200 import _lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    calls = [[name, fn, args] for name, ((fn, args), _, _) in CASES.items()]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    r = subprocess.run([sys.executable, "-c", _CHILD, os.path.join(ROOT, "rsoccer_isaac_cleanrl_b200", "_lib.py"),
                        json.dumps(calls)], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr
    got = {name: (rc, msg) for name, rc, msg in json.loads(r.stdout.strip().splitlines()[-1])}
    bad = []
    for name, (_, want_rc, want_msg) in CASES.items():
        rc, msg = got[name]
        if rc != want_rc or (want_msg is not None and want_msg not in msg):
            bad.append((name, rc, msg))
    assert not bad, bad
