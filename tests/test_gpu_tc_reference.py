"""GPU: every kernel path of the tensor-core GEMM family (csrc/tc_gemm.cu: k_gemm_tn, k_gemm_pair, k_head_fwd, k_head_bwd,
k_colsum_bf16, k_gather_pad_bf16) against exact or fp64 references, element by element.

(a) Exact-integer operands. Entries are small integer multiples of one power of two, so every product is exact in
    fp32 and every partial sum, in any order and with any internal rounding of the tensor core, is an integer multiple
    of the smallest product well below 2^24 of it (the bound is stated at each generator). The accumulator is then
    known exactly (fp64 on the GPU is exact for these values), and the epilogues, fixed IEEE fp32 operation sequences,
    are emulated in fp32 and compared bit for bit. Only tanh.approx.f32 cannot be emulated: it is compared with fp64
    tanh within its documented relative error plus one bf16 rounding.
(b) Gaussian operands at the MLP's layer shapes against fp64, within a per-element bound
    K * 2^-23 * (|A| |B|^T)_ij plus the epilogue's roundings.
(c) The production gradient path (forward_explicit / backward_explicit on two streams) against fp64 products of its
    own intermediates.
(d) A profiler run checks that the cases reach every kernel instantiation.

Every bound-based check also shows that its bound is tight: the same kernel output must fail the bound against the
fp64 reference with one 64-wide k-block dropped, and with one row tile shifted by one row."""
import re

import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

BF16, F32 = torch.bfloat16, torch.float32
EPI_BIAS_TANH_BF16, EPI_DTANH_BF16, EPI_ATOMIC_F32, EPI_BIAS_F32 = 0, 1, 2, 3
U32 = 2.0 ** -24            # unit roundoff of fp32
UBF = 2.0 ** -8             # unit roundoff of bf16 (8-bit significand)
TANH_REL = 2.0 ** -10.987   # PTX ISA: maximum relative error of tanh.approx.f32
TINY = 2.0 ** -126          # smallest normal fp32: absorbs underflow near zero
PAIR_MIN_M = 256 * 74       # the dispatch's CTA-pair threshold (rows)


@pytest.fixture(scope="module", autouse=True)
def _need_gpu():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _ints(shape, lo, hi, seed, scale=1.0, dtype=BF16):
    """Integers in [lo, hi] times `scale` (a power of two)."""
    return (torch.randint(lo, hi + 1, shape, device="cuda", generator=_gen(seed)).float() * scale).to(dtype)


def _sparse_rows(rows, cols, nnz, seed):
    """[rows, cols] bf16 with exactly nnz entries of +-1 per row, at random columns."""
    g = _gen(seed)
    pos = torch.rand(rows, cols, device="cuda", generator=g).argsort(1)[:, :nnz]
    val = torch.randint(0, 2, (rows, nnz), device="cuda", generator=g).float() * 2 - 1
    return torch.zeros(rows, cols, device="cuda").scatter_(1, pos, val).to(BF16)


def _strided(t, ld):
    """A copy of t [rows, cols] as a view with row stride ld; the padding columns hold NaN, so a kernel that reads
    them produces NaN."""
    base = torch.full((t.shape[0], ld), float("nan"), device="cuda", dtype=t.dtype)
    base[:, :t.shape[1]] = t
    return base[:, :t.shape[1]]


def _out_buf(M, N, ld, dtype, init=None, offset=0):
    """Output view [M, N] with row stride ld inside a NaN-filled buffer of M + 128 rows, starting `offset` elements
    into it: _assert_guard checks that nothing outside [M, N] was written."""
    flat = torch.full(((M + 128) * ld + offset,), float("nan"), device="cuda", dtype=dtype)
    base = flat[offset:].view(M + 128, ld)
    out = base[:M, :N]
    if init is not None:
        out.copy_(init)
    return base, out


def _assert_guard(base, M, N, what):
    assert torch.isnan(base[M:]).all() and torch.isnan(base[:M, N:]).all(), f"{what}: wrote outside the [M, N] output"


def _bits(t):
    return (t.float() + 0.0).view(torch.int32)   # (+0.0: the two zeros compare equal)


def _assert_bits(out, ref, what):
    ne = _bits(out) != _bits(ref)
    if ne.any():
        i = tuple(ne.nonzero()[0].tolist())
        raise AssertionError(f"{what}: {int(ne.sum())} of {ne.numel()} elements differ, first at {i}: "
                             f"{out[i].item()!r} vs {ref[i].item()!r}")


def _row_shifted(ref, M):
    """ref with one row tile (128 rows, fewer at the end) replaced by the rows one below it."""
    r0 = 128 * ((M // 128) // 2)
    n = min(128, M - r0 - 1)
    if n <= 0:
        return None
    s = ref.clone()
    s[r0:r0 + n] = ref[r0 + 1:r0 + 1 + n]
    return s


def _assert_within(what, out, ref_of, acc, bound, kblock_term, M):
    """|out - ref_of(acc)| <= bound element by element; and the bound is tight: it rejects ref_of(acc - one k-block)
    and the reference with one row tile shifted by one row. Returns the largest err / bound."""
    o = out.double()
    ratio = ((o - ref_of(acc)).abs() / bound).max().item()
    assert ratio <= 1.0, f"{what}: max err/bound = {ratio:.4g}"
    assert ((o - ref_of(acc - kblock_term)).abs() > bound).any(), \
        f"{what}: the bound does not reject a dropped k-block (max err/bound = {ratio:.4g})"
    shifted = _row_shifted(ref_of(acc), M)
    if shifted is not None:
        assert ((o - shifted).abs() > bound).any(), \
            f"{what}: the bound does not reject a row tile shifted by one row (max err/bound = {ratio:.4g})"
    print(f"[err/bound] {what}: {ratio:.4g}")
    return ratio


def _tanh_ref_and_bound(acc, bias, e_acc):
    """fp64 tanh(acc + bias) and the bound on bf16(tanh.approx(fl(acc_kernel + bias))), |acc_kernel - acc| <= e_acc:
    the fp32 add, the tanh (derivative <= 1), tanh.approx's relative error, one bf16 rounding."""
    z = acc + bias.double()
    t = torch.tanh(z)
    e_z = e_acc + U32 * (z.abs() + e_acc)
    e_t = e_z + TANH_REL * (t.abs() + e_z)
    return t, e_t + UBF * (t.abs() + e_t) + TINY


def _dtanh_ref(acc, y):
    return acc * (1.0 - y.double() ** 2)


def _dtanh_bound(acc, y, e_acc):
    """bf16(fl(acc_kernel * fl(1 - y*y))) against acc * (1 - y^2): y*y is exact for bf16 y, the subtraction and the
    product round once each, the bf16 conversion once."""
    t = 1.0 - y.double() ** 2
    pre = e_acc * (t + 2 * U32) + 2 * U32 * acc.abs()
    return pre + UBF * ((acc * t).abs() + pre) + TINY


# ---------------------------------------------------------------------------------------------------------------
# (a) exact-integer dispatch matrix
# ---------------------------------------------------------------------------------------------------------------
def _exact_gemm(M, N, K, epi, *, lda=None, ldb=None, ldo=None, ld_aux=None, splits=1, mn=False, bias=True,
                colsum=False, out_offset=0, seed=0, check=True, ops=None):
    """One vss_gemm_bf16_tn_colsum launch on exact-integer operands, checked against the exact reference.
    Returns (out, colsum, operands) so that callers can compare launches on the same operands."""
    from rsoccer_isaac_cleanrl_b200.engine import gemm_bf16
    what = f"epi {epi} {'MN' if mn else 'K'}-major M={M} N={N} K={K} lda={lda} ldb={ldb} ldo={ldo} " \
           f"ld_aux={ld_aux} splits={splits} bias={bias} colsum={colsum} offset={out_offset}"
    if ops is None:
        if mn:
            # wgrad: entries in {-1, 0, 1}; |any partial sum| <= K <= 2^17
            a, b = _ints((K, M), -1, 1, seed), _ints((K, N), -1, 1, seed + 1)
        elif epi == EPI_DTANH_BF16:
            # dgrad: A in {-1, 0, 1}, each row of B has 8 entries +-1: |acc| <= 8, an integer; times (1 - y^2) with
            # y in {0, +-0.5, +-1} a multiple of 0.25 of at most 8, exact in bf16; the column sums are multiples of
            # 0.25 of at most 8 M: at most 2^22 units of 0.25 for M <= 131 072
            a, b = _ints((M, K), -1, 1, seed), _sparse_rows(N, K, 8, seed + 1)
        else:
            # entries in {-2..2} * 2^-3: products are multiples of 2^-6 and |any partial sum| <= 4 K 2^-6 <= 2^5,
            # i.e. at most 2^11 units of 2^-6
            a, b = _ints((M, K), -2, 2, seed, 0.125), _ints((N, K), -2, 2, seed + 1, 0.125)
        y = _ints((M, N), -2, 2, seed + 2, 0.5) if epi == EPI_DTANH_BF16 else None
        bv = torch.randn(N, device="cuda", generator=_gen(seed + 3)) if bias and epi in (0, 3) else None
        ops = (a, b, y, bv)
    a, b, y, bv = ops
    A = _strided(a, lda) if lda else a
    B = _strided(b, ldb) if ldb else b
    Y = None if y is None else (_strided(y, ld_aux) if ld_aux else y)
    out_dtype = BF16 if epi in (EPI_BIAS_TANH_BF16, EPI_DTANH_BF16) else F32
    init = torch.zeros((M, N), device="cuda") if epi == EPI_ATOMIC_F32 else None
    base, out = _out_buf(M, N, ldo or N, out_dtype, init=init, offset=out_offset)
    cs0 = _ints((N,), -8, 8, seed + 4, dtype=F32) if colsum else None   # accumulated into
    cs = cs0.clone() if colsum else None
    gemm_bf16(A, B, out, epi, bias=bv, aux=Y, splits=splits, mn_major=mn, colsum=cs)
    torch.cuda.synchronize()
    _assert_guard(base, M, N, what)
    if not check:
        return out, cs, ops
    acc = a.double().t() @ b.double() if mn else a.double() @ b.double().t()
    if epi == EPI_DTANH_BF16:
        ref = (acc.float() * (1.0 - y.float() * y.float())).to(BF16)
        _assert_bits(out, ref, what)
        if colsum:
            _assert_bits(cs, (cs0.double() + ref.double().sum(0)).float(), what + " (column sums)")
    elif epi == EPI_ATOMIC_F32:
        _assert_bits(out, acc.float(), what)
    elif epi == EPI_BIAS_F32:
        _assert_bits(out, acc.float() + bv if bv is not None else acc.float(), what)
    else:
        kb = slice(64 * ((K // 64) // 2), 64 * ((K // 64) // 2) + 64)
        drop = a[:, kb].double() @ b[:, kb].double().t()
        t, bound = _tanh_ref_and_bound(acc, bv, 0.0)
        _assert_within(what, out, lambda x: torch.tanh(x + bv.double()), acc, bound, drop, M)
    return out, cs, ops


def _one_cta_cases():
    """(epi, bn, M, N, K, lda, ldb, ldo, ld_aux, splits, bias) for every K-major k_gemm_tn<BN, EPI, false>: one tile;
    ragged M (M % 128 = 1) with every stride padded; more tiles than resident CTAs (2 per SM) with M % 128 = 127;
    and again strided at M = 16 384. K-major split-K: 2 splits of 3 k-blocks, 3 of 8, and 20 of 4 (clamped to 4)."""
    cases = []
    for epi in (EPI_BIAS_TANH_BF16, EPI_DTANH_BF16, EPI_ATOMIC_F32, EPI_BIAS_F32):
        for bn in (64, 128):
            n_walk = 512 if bn == 128 else 320   # 129 x 4 / 129 x 5 tiles (BN = 128: the dgrad aux prefetch)
            sp = (lambda s: s if epi == EPI_ATOMIC_F32 else 1)
            cases += [
                (epi, bn, 128, bn, 64, None, None, None, None, 1, True),
                (epi, bn, 129, 3 * bn, 192, 200, 216, 3 * bn + 8, 3 * bn + 24, sp(2), epi != EPI_BIAS_F32),
                (epi, bn, 16384 + 127, n_walk, 512, None, None, None, None, sp(3), True),
                (epi, bn, 16384, n_walk, 256, 264, 320, n_walk + 8, n_walk + 64, sp(20), True),
            ]
    # N > 512: the bias is read from global memory instead of shared memory (one tile, and CTAs walking tiles)
    for epi in (EPI_BIAS_TANH_BF16, EPI_BIAS_F32):
        cases += [(epi, 128, 300, 640, 128, None, None, None, None, 1, True),
                  (epi, 128, 16384 + 1, 640, 64, None, None, 648, None, 1, True)]
    return cases


@pytest.mark.parametrize("epi,bn,M,N,K,lda,ldb,ldo,ld_aux,splits,bias", _one_cta_cases())
def test_one_cta_k_major_exact(epi, bn, M, N, K, lda, ldb, ldo, ld_aux, splits, bias):
    assert (N % 128 == 0) == (bn == 128)
    tiles = -(-M // 128) * (N // bn) * min(splits, K // 64)
    if M > 10000:
        assert tiles > 2 * _sms(), "the case must make CTAs walk more than one tile"
    _exact_gemm(M, N, K, epi, lda=lda, ldb=ldb, ldo=ldo, ld_aux=ld_aux if epi == EPI_DTANH_BF16 else None,
                splits=splits, bias=bias, colsum=(epi == EPI_DTANH_BF16 and M > 10000), seed=M + N + K + epi)


def test_one_cta_dgrad_column_sums_with_and_without():
    """The one-CTA dgrad column sums (shared-memory partial sums per CTA, then global atomics): exact, and the output
    is the same with and without them."""
    for M, N, K in ((128, 64, 64), (16384 + 1, 512, 256), (5000, 320, 512)):
        out, _, ops = _exact_gemm(M, N, K, EPI_DTANH_BF16, colsum=True, seed=M)
        out2, _, _ = _exact_gemm(M, N, K, EPI_DTANH_BF16, colsum=False, ops=ops, check=False)
        _assert_bits(out2, out, f"dgrad M={M} N={N} K={K} without column sums")


@pytest.mark.parametrize("M,N,batch,lda,ldb,ldo,splits,offset", [
    (128, 64, 64, None, None, None, 1, 0),            # BN = 64: one tile
    (256, 64, 19201, None, None, None, 301, 0),       # 2 x 301 tiles > resident; batch % 64 = 1
    (128, 64, 3903, 136, 72, 72, 7, 1),               # batch % 64 = 63, strided, out 4 bytes off 16-byte alignment
    (128, 128, 37, None, None, None, 1, 0),           # BN = 128: batch < 64
    (512, 384, 3969, None, None, None, 63, 0),        # 12 x 63 tiles; batch % 64 = 1
    (256, 128, 3903, 264, 136, 136, 5, 0),            # strided
    (128, 256, 64, None, None, None, 1, 0),           # BN = 256: one tile
    (512, 512, 131072, None, None, None, 37, 0),      # the minibatch reduction: 8 x 37 tiles > 148 resident
    (256, 256, 3969, 272, 264, 264, 9, 1),            # strided, unaligned out
    (256, 512, 1, None, None, None, 4, 0),            # batch 1: the split count clamps to 1
])
def test_one_cta_mn_major_wgrad_exact(M, N, batch, lda, ldb, ldo, splits, offset):
    _exact_gemm(M, N, batch, EPI_ATOMIC_F32, lda=lda, ldb=ldb, ldo=ldo, splits=splits, mn=True, out_offset=offset,
                seed=batch + N)


def test_k_major_atomic_accumulates_into_the_output():
    """EPI_ATOMIC_F32 adds to what the output holds."""
    from rsoccer_isaac_cleanrl_b200.engine import gemm_bf16
    a, b = _ints((300, 512), -2, 2, 1, 0.125), _ints((128, 512), -2, 2, 2, 0.125)
    start = _ints((300, 128), -64, 64, 3, 0.25, F32)
    out = start.clone()
    gemm_bf16(a, b, out, EPI_ATOMIC_F32, splits=3)
    _assert_bits(out, (start.double() + a.double() @ b.double().t()).float(), "atomic += ")


@pytest.mark.parametrize("epi,K,N", [(e, k, n) for e in (EPI_BIAS_TANH_BF16, EPI_DTANH_BF16) for k in (256, 512)
                                     for n in (256, 512)])
def test_cta_pair_exact(epi, K, N):
    """k_gemm_pair<EPI, EW>: EW = 8 for K <= 256, 4 for K = 512. At the threshold M = 18 944 and one row below it (the
    one-CTA kernel: the same bits); M % 256 in {1, 128, 129, 255} (1 and 128: the last tile's peer CTA holds only rows
    past M); the default minibatch of 131 040 rows. dgrad: with and without column sums, the same output."""
    Ms = [PAIR_MIN_M, PAIR_MIN_M - 1] + [20480 + r for r in (1, 128, 129, 255)] + [131040]
    ops_all = None
    for M in Ms:
        if M == PAIR_MIN_M - 1:   # the rows of the threshold case, one fewer
            a, b, y, bv = ops_all
            ops = (a[:M], b, None if y is None else y[:M], bv)
            out, cs, _ = _exact_gemm(M, N, K, epi, colsum=epi == EPI_DTANH_BF16, ops=ops)
            _assert_bits(out, out_thr[:M], f"epi {epi} K={K} N={N}: one-CTA M={M} vs pair M={PAIR_MIN_M}")
            continue
        out, cs, ops = _exact_gemm(M, N, K, epi, colsum=epi == EPI_DTANH_BF16, seed=M + K + N)
        if M == PAIR_MIN_M:
            ops_all, out_thr = ops, out
        if epi == EPI_DTANH_BF16:
            out2, _, _ = _exact_gemm(M, N, K, epi, colsum=False, ops=ops, check=False)
            _assert_bits(out2, out, f"dgrad pair M={M} K={K} N={N} without column sums")


def test_split_k_counts_that_do_not_divide_the_k_blocks():
    """K-major split-K: 8 k-blocks in 3 splits (3 + 3 + 2), 5 splits (clamped to 4 of 2), 9 and 64 splits (clamped to 8
    of 1); 7 k-blocks in 2 splits."""
    for K, splits in ((512, 3), (512, 5), (512, 9), (512, 64), (448, 2)):
        _exact_gemm(1000, 192, K, EPI_ATOMIC_F32, splits=splits, seed=K + splits)
        _exact_gemm(257, 256, K, EPI_ATOMIC_F32, splits=splits, seed=K + splits + 1)


# ---- head, column sums, gather ---------------------------------------------------------------------------------
HEAD_MS = (1, 7, 8, 33, 4173, 131072)


def _head_backward(dout, h, W, dz, dW, db, colsum):
    """vss_head_backward with the caller's dz (row stride dz.stride(0))."""
    from rsoccer_isaac_cleanrl_b200 import _lib
    lib = _lib.load_library()
    M, n_out = dout.shape
    rc = lib.vss_head_backward(dout.data_ptr(), h.data_ptr(), h.stride(0), W.data_ptr(), dz.data_ptr(), dz.stride(0),
                               dW.data_ptr(), db.data_ptr(), None if colsum is None else colsum.data_ptr(), M, n_out,
                               torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib.vss_gemm_last_error().decode()


@pytest.mark.parametrize("n_out", [1, 2, 6])
def test_head_forward_exact(n_out):
    """out = fl(sum_c h[m,c] W[j,c]) + b[j]: h in {-2..2} * 2^-3, W in {-2..2} * 2^-3, so the lane fmaf chains and the
    shuffle tree are exact (at most 256 * 4 units of 2^-6); the bias add is one fp32 rounding."""
    from rsoccer_isaac_cleanrl_b200.engine import head_forward
    for M in HEAD_MS:
        for ldh in (256, 264):
            h = _ints((M, 256), -2, 2, M + ldh, 0.125)
            W = _ints((n_out, 256), -2, 2, M + 1, 0.125, F32)
            b = torch.randn(n_out, device="cuda", generator=_gen(M))
            out = head_forward(_strided(h, ldh) if ldh != 256 else h, W, b)
            ref = (h.double() @ W.double().t()).float() + b
            _assert_bits(out, ref, f"head forward n_out={n_out} M={M} ldh={ldh}")


@pytest.mark.parametrize("n_out", [1, 2, 6])
def test_head_backward_exact(n_out):
    """dz = bf16(fl(sum_j dout W) * fl(1 - h^2)), dW += dout^T h, db += sum dout, dz_colsum += column sums of dz.
    dout in {-1, 0, 1}, W in {-1, 0, 1} * 2^-3, h in {0, +-0.5, +-1}: |sum_j dout W| <= 6 * 2^-3, dz a multiple of
    2^-5 of at most 0.75 (exact in bf16); dW a multiple of 0.5 of at most M; the column sums at most 24 M units of
    2^-5 <= 2^22. dW, db and the column sums start non-zero (the kernel accumulates)."""
    for M in HEAD_MS:
        for ldh, ldz in ((256, 256), (264, 512)):
            sd = M + n_out + ldz
            dout = _ints((M, n_out), -1, 1, sd, dtype=F32)
            h = _ints((M, 256), -2, 2, sd + 1, 0.5)
            W = _ints((n_out, 256), -1, 1, sd + 2, 0.125, F32)
            dW0, db0 = _ints((n_out, 256), -4, 4, sd + 3, 0.5, F32), _ints((n_out,), -4, 4, sd + 4, 1.0, F32)
            cs0 = _ints((256,), -8, 8, sd + 5, dtype=F32)
            g = dout.double() @ W.double()
            dz_ref = (g.float() * (1.0 - h.float() * h.float())).to(BF16)
            dW_ref = (dW0.double() + dout.double().t() @ h.double()).float()
            db_ref = (db0.double() + dout.double().sum(0)).float()
            what = f"head backward n_out={n_out} M={M} ldh={ldh} ldz={ldz}"
            H = _strided(h, ldh) if ldh != 256 else h
            for with_cs in (True, False):
                base, dz = _out_buf(M, 256, ldz, BF16)
                dW, db = dW0.clone(), db0.clone()
                cs = cs0.clone() if with_cs else None
                _head_backward(dout, H, W, dz, dW, db, cs)
                torch.cuda.synchronize()
                _assert_guard(base, M, 256, what)
                _assert_bits(dz, dz_ref, what + " dz")
                _assert_bits(dW, dW_ref, what + " dW")
                _assert_bits(db, db_ref, what + " db")
                if with_cs:
                    _assert_bits(cs, (cs0.double() + dz_ref.double().sum(0)).float(), what + " dz_colsum")


@pytest.mark.parametrize("N", [2, 62, 66, 258])
def test_colsum_bf16_exact(N):
    """x in {-3..3}: column sums of at most 3 M <= 2^19, exact; out starts non-zero and is accumulated into."""
    from rsoccer_isaac_cleanrl_b200.engine import colsum_bf16
    for M in (1, 7, 131077):
        for ld in (N, N + 6):
            x = _ints((M, N), -3, 3, M + N + ld)
            X = _strided(x, ld) if ld != N else x
            out0 = _ints((N,), -100, 100, M, dtype=F32)
            out = colsum_bf16(X, out0.clone())
            _assert_bits(out, (out0.double() + x.double().sum(0)).float(), f"colsum M={M} N={N} ld={ld}")


def test_gather_pad_bf16_exact():
    """dst = zero-padded src[idx].to(bfloat16): idx None, or int64 with repeats and out of order; odd ncol; ncol_pad =
    ncol + 1 and larger."""
    from rsoccer_isaac_cleanrl_b200.engine import gather_pad_bf16
    R = 5003
    for ncol, pads in ((51, (52, 64)), (53, (54, 128))):
        src = torch.randn(R, ncol, device="cuda", generator=_gen(ncol)) * 3
        idx_rep = torch.randint(0, R, (7001,), device="cuda", generator=_gen(ncol + 1))   # repeats, any order
        idx_rev = torch.arange(R - 1, -1, -2, device="cuda")
        for idx in (None, idx_rep, idx_rev):
            rows = src if idx is None else src[idx]
            for ncol_pad in pads:
                dst = gather_pad_bf16(src, idx, ncol_pad)
                ref = torch.zeros((rows.shape[0], ncol_pad), device="cuda", dtype=BF16)
                ref[:, :ncol] = rows.to(BF16)
                assert torch.equal(dst.view(torch.int16), ref.view(torch.int16)), (ncol, ncol_pad, idx is None)


# ---------------------------------------------------------------------------------------------------------------
# (b) Gaussian operands at the MLP's layer shapes against fp64, per element
# ---------------------------------------------------------------------------------------------------------------
FWD_LAYERS = [(64, 256), (256, 512), (512, 512), (512, 256)]   # (K, N); the first K is 52 observation columns + 12 zeros
DGRAD_LAYERS = [(256, 512), (512, 512), (512, 256)]            # (K = n_out of the layer, N = its k_in)


@pytest.mark.parametrize("M", [16384 + 77, 131040])
@pytest.mark.parametrize("epi", [EPI_BIAS_TANH_BF16, EPI_DTANH_BF16, EPI_BIAS_F32])
def test_gaussian_layers_within_per_element_fp64_bound(epi, M):
    """The accumulator error is bounded by K * 2^-23 * (|A| |B|^T)_ij (any summation order, fp32 partial sums with
    rounding or truncation); the epilogues add their fp32 roundings, tanh.approx's relative error and one bf16
    rounding. M = 16 461: the one-CTA kernel with CTAs walking several tiles; M = 131 040: the CTA-pair kernel
    (forward and dgrad; EPI_BIAS_F32 has only the one-CTA kernel)."""
    from rsoccer_isaac_cleanrl_b200.engine import gemm_bf16
    layers = DGRAD_LAYERS if epi == EPI_DTANH_BF16 else FWD_LAYERS
    worst = 0.0
    for li, (K, N) in enumerate(layers):
        g = _gen(1000 * li + M + epi)
        a = torch.randn(M, K, device="cuda", generator=g)
        if K == 64 and epi != EPI_DTANH_BF16:
            a[:, 52:] = 0
        a = a.to(BF16)
        b = (torch.randn(N, K, device="cuda", generator=g) * K ** -0.5).to(BF16)
        bias = torch.randn(N, device="cuda", generator=g) * 0.3
        y = torch.tanh(torch.randn(M, N, device="cuda", generator=g)).to(BF16) if epi == EPI_DTANH_BF16 else None
        out = torch.empty((M, N), device="cuda", dtype=F32 if epi == EPI_BIAS_F32 else BF16)
        gemm_bf16(a, b, out, epi, bias=None if epi == EPI_DTANH_BF16 else bias, aux=y)
        a64, b64 = a.double(), b.double()
        acc = a64 @ b64.t()
        e_acc = K * 2.0 ** -23 * (a64.abs() @ b64.abs().t())
        j = (K // 64) // 2
        drop = a64[:, 64 * j:64 * j + 64] @ b64[:, 64 * j:64 * j + 64].t()
        what = f"epi {epi} M={M} K={K} N={N}"
        if epi == EPI_BIAS_F32:
            ref_of = lambda x: x + bias.double()   # noqa: E731
            bound = e_acc * (1 + U32) + U32 * ref_of(acc).abs() + TINY
        elif epi == EPI_DTANH_BF16:
            ref_of = lambda x: _dtanh_ref(x, y)   # noqa: E731
            bound = _dtanh_bound(acc, y, e_acc)
        else:
            ref_of = lambda x: torch.tanh(x + bias.double())   # noqa: E731
            bound = _tanh_ref_and_bound(acc, bias, e_acc)[1]
        worst = max(worst, _assert_within(what, out, ref_of, acc, bound, drop, M))
        del acc, e_acc, drop, bound
    print(f"[err/bound] epi {epi} M={M}: largest over the layers {worst:.4g}")


# ---------------------------------------------------------------------------------------------------------------
# (c) the production gradient path
# ---------------------------------------------------------------------------------------------------------------
def _mlp(n_out, seed):
    from rsoccer_isaac_cleanrl_b200.tc_mlp import MlpWeights
    torch.manual_seed(seed)
    dims = [52, 256, 512, 512, 256]
    layers = []
    for i in range(4):
        layers += [torch.nn.Linear(dims[i], dims[i + 1]), torch.nn.Tanh()]
    layers.append(torch.nn.Linear(256, n_out))
    s = torch.nn.Sequential(*layers).cuda()
    with torch.no_grad():
        for m in s:
            if isinstance(m, torch.nn.Linear):
                m.weight.mul_(2.0)
                m.bias.normal_(0, 0.3)
    for p in s.parameters():   # the kernels accumulate: start from non-zero gradients
        p.grad = torch.randn(p.shape, device="cuda") * 1e-3
    return MlpWeights(s)


def _intermediates(mw, x16, dout):
    """hs (forward_explicit) and dz_l for l = 3..0 by the same kernels backward_explicit launches."""
    from rsoccer_isaac_cleanrl_b200.engine import EPI_DTANH_BF16 as DT, gemm_bf16, head_backward
    from rsoccer_isaac_cleanrl_b200.tc_mlp import forward_explicit
    out, hs = forward_explicit(mw, x16)
    dzs = [None] * 4
    dzs[3] = head_backward(dout, hs[4], mw.head_w.detach())[0]
    for l in (3, 2, 1):
        dzs[l - 1] = torch.empty((x16.shape[0], hs[l].shape[1]), device="cuda", dtype=BF16)
        gemm_bf16(dzs[l], mw.wt16[l], dzs[l - 1], DT, aux=hs[l])
    return out, hs, dzs


@pytest.mark.parametrize("M", [16384, 131040])
@pytest.mark.parametrize("n_act", [2, 6])
def test_production_gradient_path_against_fp64_of_its_intermediates(n_act, M):
    """forward_explicit + backward_explicit of an actor and a critic, the critic's backward on a side stream
    concurrently with the actor's (as ppo.forward_backward_fused runs them). Every .grad increment against fp64
    products of the kernels' own intermediates: dW_l = dz_l^T h_l, db_l = column sums of dz_l, dW0 sliced to the 52
    observation columns, the head from dout. M = 16 384: the one-CTA kernels, CTAs walking several tiles; 131 040:
    the CTA-pair kernels."""
    from rsoccer_isaac_cleanrl_b200.engine import gather_pad_bf16
    from rsoccer_isaac_cleanrl_b200.tc_mlp import backward_explicit, forward_explicit
    actor, critic = _mlp(n_act, 10 + n_act), _mlp(1, 20 + n_act)
    g = _gen(M + n_act)
    x16 = gather_pad_bf16(torch.randn(M, 52, device="cuda", generator=g), None, 64)
    douts = {"actor": torch.randn(M, n_act, device="cuda", generator=g) / M ** 0.5,
             "critic": torch.randn(M, 1, device="cuda", generator=g) / M ** 0.5}
    nets = {"actor": actor, "critic": critic}
    start = {k: [p.grad.clone() for p in mw.seq.parameters()] for k, mw in nets.items()}
    main, side = torch.cuda.current_stream(), torch.cuda.Stream()
    _, hs_a = forward_explicit(actor, x16)
    _, hs_c = forward_explicit(critic, x16)
    side.wait_stream(main)
    with torch.cuda.stream(side):
        backward_explicit(critic, hs_c, douts["critic"])
    backward_explicit(actor, hs_a, douts["actor"])
    main.wait_stream(side)
    torch.cuda.synchronize()
    for name, mw in nets.items():
        dout = douts[name]
        run1, run2 = _intermediates(mw, x16, dout), _intermediates(mw, x16, dout)
        for t1, t2 in zip([run1[0]] + run1[1] + run1[2], [run2[0]] + run2[1] + run2[2]):
            _assert_bits(t1, t2, f"{name}: intermediates of two runs")
        for t1, t2 in zip(run1[1], hs_a if name == "actor" else hs_c):
            _assert_bits(t1, t2, f"{name}: activations of the backward pass")
        _, hs, dzs = run1
        ref = []
        for l in range(4):
            dw = dzs[l].double().t() @ hs[l].double()
            ref += [dw[:, :52] if l == 0 else dw, dzs[l].double().sum(0)]
        ref += [dout.double().t() @ hs[4].double(), dout.double().sum(0)]
        errs = []
        for (pname, p), p0, r in zip(mw.seq.named_parameters(), start[name], ref):
            rel = ((p.grad.double() - p0.double() - r).norm() / r.norm()).item()
            errs.append((pname, rel))
            assert rel <= 1e-4, f"{name} M={M} {pname}: relative Frobenius error {rel:.3g}"
        print(f"[grad rel err] {name} n_act={n_act} M={M}: " + ", ".join(f"{k} {v:.2e}" for k, v in errs))


# ---------------------------------------------------------------------------------------------------------------
# (d) coverage
# ---------------------------------------------------------------------------------------------------------------
def test_the_cases_reach_every_kernel_instantiation():
    """Representative cases of every dispatch branch under the profiler: all 15 GEMM instantiations (11 one-CTA, 4
    CTA-pair) and the 6 head kernels are launched. A changed dispatch threshold fails here instead of silently
    testing another path."""
    from torch.profiler import ProfilerActivity, profile
    from rsoccer_isaac_cleanrl_b200.engine import head_forward
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for epi in range(4):
            for n in (64, 128):
                _exact_gemm(128, n, 64, epi, check=False, seed=epi + n)
        for n in (64, 128, 256):
            _exact_gemm(128, n, 64, EPI_ATOMIC_F32, mn=True, check=False, seed=n)
        for epi in (EPI_BIAS_TANH_BF16, EPI_DTANH_BF16):
            for k in (256, 512):
                _exact_gemm(PAIR_MIN_M, 256, k, epi, check=False, seed=k)
        for n_out in (1, 2, 6):
            h = _ints((33, 256), -2, 2, n_out, 0.125)
            W = _ints((n_out, 256), -2, 2, n_out, 0.125, F32)
            head_forward(h, W, torch.zeros(n_out, device="cuda"))
            _head_backward(torch.zeros(33, n_out, device="cuda"), h, W, torch.empty_like(h), torch.zeros_like(W),
                           torch.zeros(n_out, device="cuda"), None)
        torch.cuda.synchronize()
    names = {re.sub(r"\s+", "", e.name) for e in prof.events()}
    found = set()
    for nm in names:
        for pat in (r"k_gemm_tn<\d+,\d+,(?:true|false)>", r"k_gemm_pair<\d+,\d+>", r"k_head_(?:fwd|bwd)<\d+>"):
            found.update(re.findall(pat, nm))
    want = {f"k_gemm_tn<{bn},{e},false>" for bn in (64, 128) for e in range(4)}
    want |= {f"k_gemm_tn<{bn},2,true>" for bn in (64, 128, 256)}
    want |= {f"k_gemm_pair<{e},{ew}>" for e in (0, 1) for ew in (4, 8)}
    want |= {f"k_head_{d}<{n}>" for d in ("fwd", "bwd") for n in (1, 2, 6)}
    assert len(want) == 21 and want <= found, ("not launched:", sorted(want - found), "launched:", sorted(found))
    print("[coverage] launched:", ", ".join(sorted(found & want)))
