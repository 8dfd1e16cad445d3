"""Kernel-level tests of the dense FP64 building blocks of the C ABI (include/gpgp.h), one entry point at a time.

Where the arithmetic allows it, the inputs make the correct FP64 answer exact whatever the summation order, so that a
misplaced fragment, a dropped or duplicated k-slab, a wrong tile mask or a stale pipeline stage shows as a bit difference:
  - GEMMs, skinny products, dot products: integer operands in [-4, 4] (K <= 8192: every partial sum is an integer far
    below 2^53) and dyadic alpha / beta; float64 numpy in any order is the exact reference.
  - Cholesky and solves: a dyadic factor L (diagonal blocks 2 (I + N) with N^2 = 0, sparse small dyadic off-diagonal
    blocks, identity padding) for which every intermediate of a blocked Cholesky is representable: potrf(L L^T) must
    return L and potrs(L L^T y) must return y, bit for bit.
Regions a kernel promises not to read (skipped k ranges, skipped tiles, padding columns) hold NaN, and regions it
promises not to write hold a NaN sentinel that is compared bit for bit. Where no exact answer exists the bound is derived
from the operation and written next to the assert.

The tests marked gpu need a CUDA device; the unmarked ones check on the CPU that the exact references are exact."""

import ctypes
import math

import numpy
import pytest

gpu = pytest.mark.gpu

EPS = numpy.finfo(numpy.float64).eps
KR_FULL, KR_A_LOWER, KR_B_LOWER, KR_TN_LOWER = 0, 1, 2, 3      # csrc/gp_internal.h
TM_ALL, TM_LOWER = 0, 1
SENTINEL = numpy.array([0x7ff8dead0000beef], dtype=numpy.uint64).view(numpy.float64)[0]   # a NaN with a payload


# ------------------------------------------------------------------------------------------------ host-side references
def padded(n):
    return (n + 127) // 128 * 128


def int_matrix(rng, shape):
    return rng.integers(-4, 5, size=shape).astype(numpy.float64)


def dyadic_factor(n, rng):
    """Lower factor L (npad x npad) whose Cholesky intermediates are exact: diagonal 128-blocks 2 (I + N), N nonzero only
    in rows 64..127 x columns 0..63 of the block (N^2 = 0, inverse exactly (I - N) / 2), off-diagonal blocks in
    {-2..2} / 16 at density 1/8, identity padding."""
    npad = padded(n)
    L = numpy.tril(rng.integers(-2, 3, size=(npad, npad)) * (rng.random((npad, npad)) < 0.125) / 16.0, -1)
    for b in range(0, npad, 128):
        L[b:b + 128, b:b + 128] = 0.0
        N = rng.integers(-2, 3, size=(64, 64)) / 16.0
        L[b + 64:b + 128, b:b + 64] = 2.0 * N
        L[range(b, b + 128), range(b, b + 128)] = 2.0
    L[n:, :] = 0.0
    L[:, n:] = 0.0
    L[range(n, npad), range(n, npad)] = 1.0
    return L


def dyadic_rhs(rng, n, npad, p):
    y = numpy.zeros((npad, p))
    y[:n] = rng.integers(-8, 9, size=(n, p)) / 8.0
    return y


def nan_to_zero(a):
    return numpy.where(numpy.isnan(a), 0.0, a)


def bits(a):
    return numpy.ascontiguousarray(a).view(numpy.uint64)


def assert_equal(got, want, what):
    """exact equality (0.0 == -0.0); NaN anywhere in got fails"""
    bad = ~(got == want)
    assert not bad.any(), '%s: %d of %d entries differ, first at %s: %r vs %r' % (
        what, bad.sum(), bad.size, tuple(numpy.argwhere(bad)[0]), got[bad][0], want[bad][0])


def assert_untouched(got, want, what):
    bad = bits(got) != bits(want)
    assert not bad.any(), '%s: %d entries written that must stay untouched, first at %s' % (
        what, bad.sum(), tuple(numpy.argwhere(bad)[0]))


# ---------------------------------------------------------------------------------- CPU checks of the exact references
def test_integer_gemm_reference_is_exact():
    rng = numpy.random.default_rng(1)
    A, B = int_matrix(rng, (256, 8192)), int_matrix(rng, (8192, 128))
    exact = A.astype(numpy.int64) @ B.astype(numpy.int64)
    assert numpy.array_equal(A @ B, exact.astype(numpy.float64))
    assert numpy.array_equal(B.T @ A.T, exact.T.astype(numpy.float64))     # another summation order, same bits
    assert numpy.abs(exact).max() * 2 < 2 ** 53


@pytest.mark.parametrize('n', [129, 640])
def test_dyadic_factor_is_exact(n):
    rng = numpy.random.default_rng(n)
    L = dyadic_factor(n, rng)
    npad = L.shape[0]
    for b in range(0, npad, 128):                   # the diagonal blocks 2 (I + N) invert exactly to (I - N) / 2 = I - D / 4
        D = L[b:b + 128, b:b + 128]
        Dinv = numpy.eye(128) - D / 4.0
        v = max(0, min(128, n - b))                 # identity padding inverts to itself
        Dinv[v:, v:] = numpy.eye(128 - v)
        assert numpy.array_equal(D @ Dinv, numpy.eye(128))
    A = L @ L.T
    assert numpy.array_equal(numpy.linalg.cholesky(A), L)
    y = dyadic_rhs(rng, n, npad, 3)
    import scipy.linalg
    b = A @ y
    assert numpy.array_equal(scipy.linalg.cho_solve((L, True), b), y)


def test_numpy_ops_gemm_rejects_tables_off_the_k_slab():
    import torch
    from numpy_ops import NumpyOps
    C, A, B = torch.zeros(128, 128, dtype=torch.float64), torch.ones(128, 64, dtype=torch.float64), \
        torch.ones(128, 64, dtype=torch.float64)
    NumpyOps().gemm(C, A, B, 1.0, 0.0, kbeg=[16], kend=[48])
    assert (C.numpy() == 32.0).all()
    with pytest.raises(AssertionError):
        NumpyOps().gemm(C, A, B, 1.0, 0.0, kend=[40])


# ------------------------------------------------------------------------------------------------------- device plumbing
@pytest.fixture(scope='module')
def cu():
    from gaussian_proc import _device as dev
    dev.require_cuda()
    return dev


def _torch():
    import torch
    return torch


def dptr(t, offset=0):
    return ctypes.c_void_p(t.data_ptr() + 8 * offset)


def to_dev(a):
    torch = _torch()
    return torch.from_numpy(numpy.ascontiguousarray(a, dtype=numpy.float64)).cuda()


def to_host(t):
    torch = _torch()
    torch.cuda.synchronize()
    return t.cpu().numpy()


def run_gemm(dev, at, bt, M, N, K, alpha, beta, krange=KR_FULL, tmask=TM_ALL, pad=(0, 0, 0), offset=0, seed=0,
             kbeg=None, kend=None, c_nan=False, extra_k=0):
    """One gp_dgemm_f64 (tables None) or gp_dgemm_ktab_f64 call on integer operands; returns (got C, expected C, C0).
    pad: extra (NaN) columns of A, B, C storage; offset: every buffer starts 2 doubles (16 B) into its allocation.
    extra_k: the operands hold extra_k more k-columns / rows than K, all NaN."""
    torch = _torch()
    rng = numpy.random.default_rng(seed)
    Ka = K + extra_k
    A_log, B_log = int_matrix(rng, (M, Ka)), int_matrix(rng, (Ka, N))
    A_log[:, K:] = numpy.nan
    B_log[K:, :] = numpy.nan
    m, k, nn = numpy.arange(M)[:, None], numpy.arange(Ka)[None, :], numpy.arange(N)[None, :]
    kb = numpy.arange(Ka)[:, None]
    if krange == KR_A_LOWER:            # A(m, k) lower: zero right of the diagonal, NaN right of the diagonal block
        A_log[k > m] = 0.0
        A_log[k >= (m // 128 + 1) * 128] = numpy.nan
    if krange == KR_TN_LOWER:           # A(m, k) = W[k][m], W lower: zero for k < m, NaN left of the diagonal block
        A_log[k < m] = 0.0
        A_log[k < (m // 128) * 128] = numpy.nan
    if krange in (KR_B_LOWER, KR_TN_LOWER):   # B(k, n) lower: zero for k < n, NaN above the diagonal block
        B_log[kb < nn] = 0.0
        B_log[kb < (nn // 128) * 128] = numpy.nan
    if kbeg is not None or kend is not None:  # per-row-tile k ranges: every k outside the tile's range is NaN in A
        for t in range(M // 128):
            b0 = 0 if kbeg is None else min(kbeg[t], K)
            e0 = K if kend is None else min(kend[t], K)
            A_log[128 * t:128 * t + 128, :b0] = numpy.nan
            A_log[128 * t:128 * t + 128, max(e0, b0):] = numpy.nan
    ref = numpy.zeros((M, N))
    for t in range(M // 128):
        b0 = 0 if kbeg is None else min(kbeg[t], K)
        e0 = K if kend is None else min(kend[t], K)
        if e0 > b0:
            ref[128 * t:128 * t + 128] = nan_to_zero(A_log[128 * t:128 * t + 128, b0:e0]) @ nan_to_zero(B_log[b0:e0])
    C0 = numpy.full((M, N), numpy.nan) if c_nan else int_matrix(rng, (M, N))
    want = alpha * ref if beta == 0.0 else alpha * ref + beta * C0
    if tmask == TM_LOWER:
        C0[nn > m] = SENTINEL
        want[nn > m] = SENTINEL

    def store(log, transposed, padc):
        S = log.T if transposed else log
        rows, cols = S.shape
        flat = numpy.full(offset + rows * (cols + padc) + 2, numpy.nan)
        flat[offset:offset + rows * (cols + padc)].reshape(rows, cols + padc)[:, :cols] = S
        return to_dev(flat), cols + padc

    Ad, lda = store(A_log, at == 1, pad[0])            # at = 0: [m][k]; at = 1: [k][m]
    Bd, ldb = store(B_log, bt == 0, pad[1])            # bt = 0: [n][k]; bt = 1: [k][n]
    Cd, ldc = store(C0, False, pad[2])
    if kbeg is None and kend is None:
        rc = dev.lib.gp_dgemm_f64(at, bt, dptr(Cd, offset), ldc, dptr(Ad, offset), lda, dptr(Bd, offset), ldb, M, N, K,
                                  alpha, beta, krange, tmask, dev.stream_ptr())
    else:
        tabs = [None if t is None else torch.tensor(list(t), dtype=torch.int32, device='cuda') for t in (kbeg, kend)]
        rc = dev.lib.gp_dgemm_ktab_f64(at, bt, dptr(Cd, offset), ldc, dptr(Ad, offset), lda, dptr(Bd, offset), ldb, M, N,
                                       K, alpha, beta, None if tabs[0] is None else dptr(tabs[0]),
                                       None if tabs[1] is None else dptr(tabs[1]), dev.stream_ptr())
    assert rc == 0, 'gemm returned %d' % rc
    Cf = to_host(Cd)
    assert numpy.isnan(Cf[:offset]).all() and numpy.isnan(Cf[-2:]).all()
    Cs = Cf[offset:offset + M * ldc].reshape(M, ldc)
    assert numpy.isnan(Cs[:, N:]).all(), 'padding columns of C written'
    return Cs[:, :N], want, C0


def check_gemm(dev, *args, **kw):
    got, want, C0 = run_gemm(dev, *args, **kw)
    tmask = kw.get('tmask', TM_ALL)
    if tmask == TM_LOWER:
        up = numpy.triu(numpy.ones(got.shape, dtype=bool), 1)
        assert_untouched(got[up], want[up], 'TM_LOWER: C above the diagonal')
        assert_equal(got[~up], want[~up], 'gemm %r %r' % (args, kw))
    else:
        assert_equal(got, want, 'gemm %r %r' % (args, kw))


# (M, N, K, alpha, beta, krange, tmask, pad, offset): every k-range / tile-mask mode the library uses, K below the pipeline
# depth (32), K not a multiple of the 32-wide slab pairs (96, 160), K >= 2048 (many passes around the mbarrier ring), tile-row
# counts that are not multiples of RASTER_GROUP = 8 (9, 17), padded leading dimensions, 16-byte (not 128-byte) aligned views
GEMM_CASES = [
    (128, 128, 32, 1.0, 0.0, KR_FULL, TM_ALL, (0, 0, 0), 0),
    (1152, 2176, 96, -0.25, 0.5, KR_FULL, TM_ALL, (2, 6, 4), 2),
    (2176, 1152, 160, 3.0, -1.0, KR_FULL, TM_ALL, (6, 2, 2), 0),
    (1152, 1152, 2048, 0.5, 1.0, KR_FULL, TM_ALL, (0, 0, 0), 2),
    (2176, 2176, 128, -1.0, 1.0, KR_FULL, TM_LOWER, (2, 2, 2), 2),       # trailing update
    (1152, 640, 1152, -1.0, 0.0, KR_A_LOWER, TM_ALL, (0, 2, 0), 0),      # trtri: W21 = -W22 T
    (640, 1152, 1152, 1.0, 0.0, KR_B_LOWER, TM_ALL, (2, 0, 0), 2),       # trtri: T = L21 W11
    (1152, 1152, 1152, 1.0, 0.0, KR_TN_LOWER, TM_LOWER, (0, 0, 2), 0),   # lauum: W^T W
    (1152, 640, 1152, 0.5, -0.25, KR_TN_LOWER, TM_ALL, (2, 2, 2), 2),
]
LAYOUTS = [(0, 0), (0, 1), (1, 0), (1, 1)]


def gemm_suite(dev, cases=GEMM_CASES):
    """every case in every operand layout"""
    for i, case in enumerate(cases):
        M, N, K, alpha, beta, kr, tm, pad, off = case
        for at, bt in LAYOUTS:
            check_gemm(dev, at, bt, M, N, K, alpha, beta, krange=kr, tmask=tm, pad=pad, offset=off, seed=i)
    # beta = 0 must not read C (BLAS semantics): C full of NaN
    for at, bt in LAYOUTS:
        check_gemm(dev, at, bt, 1152, 1152, 96, -1.0, 0.0, c_nan=True, seed=7)
        check_gemm(dev, at, bt, 1152, 1152, 96, 1.0, 0.0, tmask=TM_LOWER, c_nan=True, seed=8)
    # K == 0: C = beta C (the operands hold 32 NaN k-columns that must not be read)
    for at, bt in LAYOUTS:
        check_gemm(dev, at, bt, 256, 256, 0, 1.0, 0.5, extra_k=32, seed=9)
        check_gemm(dev, at, bt, 256, 256, 0, 1.0, 0.0, c_nan=True, extra_k=32, seed=10)


@gpu
def test_gemm_tma_default(cu):
    gemm_suite(cu)


@gpu
@pytest.mark.parametrize('tiles', [9, 17])
@pytest.mark.parametrize('K', [32, 128, 512])
@pytest.mark.parametrize('alpha,beta', [(1.0, 0.0), (-0.5, 0.25)])
@pytest.mark.parametrize('pad', [0, 6])
def test_gemm_in_place_panel_solve(cu, tiles, K, alpha, beta, pad):
    """The one aliased form, C == A with a single 128-wide column tile (BN = 128: a CTA owns the row block it overwrites),
    as factor_panel's panel solve L21 = A21 inv(L_jj)^T uses it: C is the first 128 of A's K columns. tiles: tile rows,
    not a multiple of RASTER_GROUP; pad: extra columns of the leading dimension. Everything outside C (NaN around the
    block, A's columns past 128) must be left as it was; with beta = 0 the columns of C past K hold NaN, never read."""
    M, W = 128 * tiles, max(K, 128)
    r0, c0 = 3, 2                                       # the block starts inside the matrix, 16 bytes into a row
    ld = c0 + W + pad
    rng = numpy.random.default_rng(tiles + K)
    blk = int_matrix(rng, (M, W))
    if beta == 0.0:
        blk[:, K:] = numpy.nan
    full = numpy.full((r0 + M + 2, ld), numpy.nan)
    full[r0:r0 + M, c0:c0 + W] = blk
    B = numpy.full((128, K + 2), numpy.nan)             # inv(L_jj) stored [n][k], two NaN padding columns
    B[:, :K] = int_matrix(rng, (128, K))
    want = alpha * (blk[:, :K] @ B[:, :K].T)
    if beta != 0.0:
        want += beta * blk[:, :128]
    Ad = to_dev(full)
    C = dptr(Ad, r0 * ld + c0)
    assert cu.lib.gp_dgemm_f64(0, 0, C, ld, C, ld, dptr(to_dev(B)), K + 2, M, 128, K, alpha, beta, KR_FULL, TM_ALL,
                               cu.stream_ptr()) == 0
    got = to_host(Ad)
    assert_equal(got[r0:r0 + M, c0:c0 + 128], want, 'in-place panel solve')
    rest = numpy.ones(got.shape, dtype=bool)
    rest[r0:r0 + M, c0:c0 + 128] = False
    assert_untouched(got[rest], full[rest], 'in-place panel solve: outside C')


@gpu
def test_gemm_trailing_update_at_race_shape(cu):
    """The launch shape at which a stage released before its shared-memory loads had returned read a few entries from the
    wrong slab: trailing update, M = N = 7680, K = 512, two CTAs per SM (BN = 64), every entry compared; then the same
    product twice at once on two streams. Each launch runs once (a value check)."""
    torch = _torch()
    M, K = 7680, 512
    rng = numpy.random.default_rng(11)
    P = int_matrix(rng, (M, K))
    C0 = int_matrix(rng, (M, M))
    want = C0 - P @ P.T
    low = numpy.tril(numpy.ones((M, M), dtype=bool))
    Pd = to_dev(P)
    outs = []
    for streams in ([None], [torch.cuda.Stream(), torch.cuda.Stream()]):
        Cs = [to_dev(C0) for _ in streams]
        torch.cuda.synchronize()
        for s, Cd in zip(streams, Cs):
            with torch.cuda.stream(s if s is not None else torch.cuda.current_stream()):
                assert cu.lib.gp_dgemm_f64(0, 0, dptr(Cd), M, dptr(Pd), K, dptr(Pd), K, M, M, K, -1.0, 1.0, KR_FULL,
                                           TM_LOWER, cu.stream_ptr()) == 0
        outs += [to_host(Cd) for Cd in Cs]
    for got in outs:
        assert_equal(got[low], want[low], 'trailing update 7680 x 7680 x 512')
        assert_untouched(got[~low], C0[~low], 'trailing update: upper triangle')


@gpu
def test_gemm_ktab_tables(cu):
    M, N, K = 1152, 256, 512
    T = M // 128
    rng = numpy.random.default_rng(5)
    kb = [int(v) for v in rng.integers(0, K // 16 + 1, size=T) * 16]
    ke = [int(v) for v in rng.integers(0, K // 16 + 1, size=T) * 16]
    ke[0], kb[1], ke[2], kb[3], ke[4] = K + 96, K, 0, K + 64, -16     # kend > K; kbeg == K; empty; kbeg > K; negative
    for at, bt in LAYOUTS:
        for tabs in ((kb, None), (None, ke), (kb, ke)):
            check_gemm(cu, at, bt, M, N, K, -1.0, 0.5, kbeg=tabs[0], kend=tabs[1], seed=at + 2 * bt)
            check_gemm(cu, at, bt, M, N, K, 1.0, 0.0, kbeg=tabs[0], kend=tabs[1], c_nan=True, seed=at + 2 * bt)


def _ktab_through_entry(cu, at, bt, M, N, K, alpha, beta, kbeg, kend, extra_k=0, c_nan=False):
    """like check_gemm, but the call goes through gp_dgemm_ktab_f64 even when both tables are None"""
    torch = _torch()
    rng = numpy.random.default_rng(21)
    Ka = K + extra_k
    A = numpy.full((M, Ka) if at == 0 else (Ka, M), numpy.nan)
    B = numpy.full((N, Ka) if bt == 0 else (Ka, N), numpy.nan)
    C0 = numpy.full((M, N), numpy.nan) if c_nan else int_matrix(rng, (M, N))
    Ad, Bd, Cd = to_dev(A), to_dev(B), to_dev(C0)
    tabs = [None if t is None else torch.tensor(t, dtype=torch.int32, device='cuda') for t in (kbeg, kend)]
    rc = cu.lib.gp_dgemm_ktab_f64(at, bt, dptr(Cd), N, dptr(Ad), A.shape[1], dptr(Bd), B.shape[1], M, N, K, alpha, beta,
                                  None if tabs[0] is None else dptr(tabs[0]), None if tabs[1] is None else dptr(tabs[1]),
                                  cu.stream_ptr())
    assert rc == 0, rc
    return to_host(Cd), C0


@gpu
@pytest.mark.parametrize('at,bt', LAYOUTS)
def test_gemm_ktab_zero_depth_is_beta_c(cu, at, bt):
    """K == 0 with NULL tables: C = beta C. The operands hold 32 NaN k-columns past K, which must not be read."""
    got, C0 = _ktab_through_entry(cu, at, bt, 256, 256, 0, 1.0, 0.5, None, None, extra_k=32)
    assert_equal(got, 0.5 * C0, 'ktab, K = 0, beta = 0.5')
    got, C0 = _ktab_through_entry(cu, at, bt, 256, 256, 0, 1.0, 0.0, None, None, extra_k=32, c_nan=True)
    assert_equal(got, numpy.zeros_like(got), 'ktab, K = 0, beta = 0')
    # empty ranges from the tables at K > 0 (all NaN operands): C = beta C as well
    got, C0 = _ktab_through_entry(cu, at, bt, 256, 256, 64, 1.0, -1.0, [64, 32], [64, 16])
    assert_equal(got, -C0, 'ktab, empty ranges')
    # both tables NULL at K > 0: the plain product through the ktab entry point
    check_gemm(cu, at, bt, 1152, 256, 512, 1.0, 0.5, kbeg=[0] * 9, seed=at + 2 * bt)
    rng = numpy.random.default_rng(at + 2 * bt)
    A, B, C0 = int_matrix(rng, (256, 96)), int_matrix(rng, (96, 128)), int_matrix(rng, (256, 128))
    Ad = to_dev(A if at == 0 else A.T)
    Bd = to_dev(B.T if bt == 0 else B)
    Cd = to_dev(C0)
    assert cu.lib.gp_dgemm_ktab_f64(at, bt, dptr(Cd), 128, dptr(Ad), Ad.shape[1], dptr(Bd), Bd.shape[1], 256, 128, 96, -1.0,
                                    0.5, None, None, cu.stream_ptr()) == 0
    assert_equal(to_host(Cd), 0.5 * C0 - A @ B, 'ktab, NULL tables')


def blockcyclic_layout(P, nb, NB):
    from gaussian_proc._blockcyclic import snake_owner
    r = next(q for q in range(P - 1, 0, -1) if any(snake_owner(j, P) == q for j in range(NB)))
    return r, [j for j in range(NB) if snake_owner(j, P) == r]


def staircase_tables(I, nb, NB):
    """the kend tables of BlockCyclicCholesky.inverse_rows and the kbeg tables of inverse_traces for local block rows I"""
    tiles, nq = nb // 128, len(I)
    out = []
    for k in range(NB - 1, -1, -1):
        q0 = next((q for q, i in enumerate(I) if i > k), nq)
        if q0 < nq:
            out.append(('kend', k, q0, [(I[q] - k) * nb for q in range(q0, nq) for _ in range(tiles)]))
    for j in range(NB):
        q0 = next((q for q, i in enumerate(I) if i >= j), nq)
        if q0 < nq:
            out.append(('kbeg', j, q0, [(next((q for q in range(q0, nq) if I[q] >= jp), nq) - q0) * nb
                                        for jp in range(j, NB) for _ in range(tiles)]))
    return out


@gpu
@pytest.mark.parametrize('P,nb,NB', [(2, 256, 5), (3, 256, 5), (8, 128, 10)])
def test_gemm_ktab_blockcyclic_staircases(cu, P, nb, NB):
    """the staircase tables the distributed inverse builds on a rank != 0, with NaN right of the staircase"""
    _, I = blockcyclic_layout(P, nb, NB)
    for kind, k, q0, tab in staircase_tables(I, nb, NB):
        M = len(tab) * 128
        if kind == 'kend':       # T[rows] = X[rows, (k+1) nb:] panel^T   (at = 0, bt = 1)
            K = (NB - k - 1) * nb
            check_gemm(cu, 0, 1, M, nb, K, 1.0, 0.0, kend=tab, c_nan=True, seed=k)
        else:                    # C[:M] = X[rows, j nb:]^T X[rows, j nb:(j+1) nb]   (at = 1, bt = 1)
            K = (len(I) - q0) * nb
            check_gemm(cu, 1, 1, M, nb, K, 1.0, 0.0, kbeg=tab, c_nan=True, seed=k)


# --------------------------------------------------------------------------------------------- factorisation blocks
NS = [1, 127, 128, 129, 513, 640, 1152, 2177]


def potrf_dev(cu, A_host, n, info=None):
    torch = _torch()
    npad = A_host.shape[0]
    Ad = to_dev(A_host)
    ws = torch.empty(cu.lib.gp_potrf_workspace_bytes(npad) // 8, dtype=torch.float64, device='cuda')
    if info is None:
        info = torch.full((1,), 12345, dtype=torch.int32, device='cuda')
    assert cu.lib.gp_potrf_f64(dptr(Ad), n, npad, dptr(info), dptr(ws), cu.stream_ptr()) == 0
    return Ad, ws, info


def with_nan_upper(A):
    A = A.copy()
    A[numpy.triu_indices(A.shape[0], 1)] = numpy.nan
    return A


@gpu
@pytest.mark.parametrize('n', NS)
def test_potrf_potrs_dyadic_exact(cu, n):
    rng = numpy.random.default_rng(n)
    L = dyadic_factor(n, rng)
    npad = L.shape[0]
    A = with_nan_upper(L @ L.T)                          # the strict upper triangle is never referenced
    Ad, ws, info = potrf_dev(cu, A, n)
    got = to_host(Ad)
    low = numpy.tril(numpy.ones((npad, npad), dtype=bool))
    assert int(info.item()) == 0
    assert_equal(got[low], L[low], 'potrf n=%d' % n)
    assert_untouched(got[~low], A[~low], 'potrf: strict upper triangle')
    for nrhs in (1, 7, 8, 9, 16):
        ldb = nrhs + 3
        y = dyadic_rhs(rng, n, npad, nrhs)
        B = numpy.full((npad, ldb), numpy.nan)
        B[:, :nrhs] = (L @ L.T) @ y
        Bd = to_dev(B)
        assert cu.lib.gp_potrs_f64(dptr(Ad), npad, dptr(ws), dptr(Bd), nrhs, ldb, cu.stream_ptr()) == 0
        out = to_host(Bd)
        assert_equal(out[:, :nrhs], y, 'potrs n=%d nrhs=%d' % (n, nrhs))
        assert numpy.isnan(out[:, nrhs:]).all()


@gpu
@pytest.mark.parametrize('n,p', [(129, 1), (129, 32), (129, 33), (129, 128), (129, 129), (640, 129), (1152, 600),
                                 (1152, 1100), (2177, 700), (2177, 2177)])
def test_potrf_info_is_first_bad_pivot(cu, n, p):
    """A = L D L^T with D = I except D[p-1, p-1] = -1: the first non-positive pivot is exactly p. Pivot 600 of n = 1152 and
    700 of n = 2177 sit in the second outer panel, which is factored on the look-ahead stream; 1100 of n = 1152 in the
    last panel (the rest == 0 branch). A following call on a positive definite matrix reports 0 again."""
    rng = numpy.random.default_rng(p)
    L = dyadic_factor(n, rng)
    D = numpy.ones(L.shape[0])
    D[p - 1] = -1.0
    _, _, info = potrf_dev(cu, (L * D) @ L.T, n)
    assert int(info.item()) == p
    potrf_dev(cu, L @ L.T, n, info=info)
    assert int(info.item()) == 0


@gpu
@pytest.mark.parametrize('n', NS)
def test_trtri_lauum_potri(cu, n):
    import scipy.linalg
    torch = _torch()
    rng = numpy.random.default_rng(n + 1)
    L = dyadic_factor(n, rng)
    npad = L.shape[0]
    Ad, ws, _ = potrf_dev(cu, with_nan_upper(L @ L.T), n)
    tws = torch.empty(cu.lib.gp_potri_workspace_bytes(npad) // 8 + 1, dtype=torch.float64, device='cuda')
    Wd = to_dev(numpy.full((npad, npad), numpy.nan))
    assert cu.lib.gp_trtri_f64(dptr(Ad), dptr(Wd), npad, dptr(ws), dptr(tws), cu.stream_ptr()) == 0
    W = to_host(Wd)
    low = numpy.tril(numpy.ones((npad, npad), dtype=bool))
    blk = numpy.arange(npad) // 128
    diag_blk = blk[:, None] == blk[None, :]
    assert not numpy.isnan(W[low]).any()
    assert (W[diag_blk & ~low] == 0.0).all()                        # zero above the diagonal inside diagonal blocks
    assert numpy.isnan(W[~diag_blk & ~low]).all()                   # nothing written above the diagonal blocks
    assert (W[n:, :n] == 0.0).all()                                 # the padding inverts to the exact identity
    assert numpy.array_equal(numpy.tril(W[n:, n:]), numpy.eye(npad - n))
    Wl = numpy.where(low, W, 0.0)
    # triangular inverse (Higham, Accuracy and Stability, 14.2): |W L - I| <= c n u |W| |L|, c = 2 for the two products
    resid = numpy.abs(Wl @ L - numpy.eye(npad))
    assert (resid <= 2 * npad * EPS * (numpy.abs(Wl) @ numpy.abs(L)) + 1e-300).all()
    # against LAPACK dtrtri: each satisfies |W - X| <= n u |X| |L| |X|, so they differ by at most twice that
    X, info = scipy.linalg.lapack.dtrtri(L, lower=1)
    assert info == 0
    aX = numpy.abs(X)
    assert (numpy.abs(Wl - X) <= 2 * npad * EPS * (aX @ numpy.abs(L) @ aX) + 1e-300).all()
    # lauum: integer W with the same structure (lower, zero above the diagonal in the diagonal blocks, NaN above
    # them) -> W^T W exact; the strict upper triangle of the output stays untouched
    Wi = numpy.where(low, int_matrix(rng, (npad, npad)), numpy.where(diag_blk, 0.0, numpy.nan))
    Ci = numpy.full((npad, npad), SENTINEL)
    Cd = to_dev(Ci)
    assert cu.lib.gp_lauum_f64(dptr(to_dev(Wi)), dptr(Cd), npad, cu.stream_ptr()) == 0
    got = to_host(Cd)
    Wz = nan_to_zero(Wi)
    assert_equal(got[low], (Wz.T @ Wz)[low], 'lauum n=%d' % n)
    assert_untouched(got[~low], Ci[~low], 'lauum: strict upper triangle')
    # potri = trtri + lauum: lower triangle of inv(A) against numpy, error of W^T W with |dW| <= n u |W||L||W|:
    # |d(W^T W)| <= 2 |W|^T |dW| + n u |W|^T |W|, counted for both results
    Ad2, ws2, _ = potrf_dev(cu, with_nan_upper(L @ L.T), n)
    Wd2 = to_dev(numpy.full((npad, npad), numpy.nan))
    assert cu.lib.gp_potri_f64(dptr(Ad2), dptr(Wd2), npad, dptr(ws2), dptr(tws), cu.stream_ptr()) == 0
    Ainv = to_host(Ad2)
    ref = X.T @ X
    dW = npad * EPS * (aX @ numpy.abs(L) @ aX)
    bound = 2 * (2 * aX.T @ dW + npad * EPS * aX.T @ aX)
    assert (numpy.abs(Ainv[low] - ref[low]) <= bound[low] + 1e-300).all()
    assert numpy.array_equal(Ainv[n:, n:][numpy.tril_indices(npad - n)], numpy.eye(npad - n)[numpy.tril_indices(npad - n)])


@gpu
@pytest.mark.parametrize('n', [1, 129, 640, 2177])
def test_inverse_traces_exact_on_integers(cu, n):
    """kind 0: ||M||_F^2 over the lower triangle of the first n rows; kind 1: trace and ||M||_F^2 of the symmetric matrix
    whose lower triangle is stored. Integer entries make both sums exact."""
    torch = _torch()
    npad = padded(n)
    rng = numpy.random.default_rng(n)
    M = numpy.where(numpy.tril(numpy.ones((npad, npad), dtype=bool)), int_matrix(rng, (npad, npad)), numpy.nan)
    M[n:, :] = numpy.nan                                         # rows past n are not part of the n x n matrix
    Md = to_dev(M)
    ws = torch.empty(cu.lib.gp_traces_workspace_bytes(npad) // 8 + 1, dtype=torch.float64, device='cuda')
    Ml = nan_to_zero(M)[:n, :n]
    for kind in (0, 1):
        out = to_dev(numpy.full(8, numpy.nan))
        assert cu.lib.gp_inverse_traces(dptr(Md), n, npad, kind, dptr(out), dptr(ws), cu.stream_ptr()) == 0
        o = to_host(out)
        if kind == 0:
            assert o[1] == numpy.sum(Ml ** 2)
        else:
            assert o[1] == numpy.trace(Ml)
            assert o[2] == 2 * numpy.sum(Ml ** 2) - numpy.sum(numpy.diag(Ml) ** 2)


@gpu
@pytest.mark.parametrize('n', [1, 129, 2177])
def test_logdet_from_chol(cu, n):
    npad = padded(n)
    rng = numpy.random.default_rng(n)
    L = numpy.full((npad, npad), numpy.nan)
    d = numpy.exp(rng.uniform(-3.0, 3.0, size=npad))
    L[range(npad), range(npad)] = d
    out = to_dev(numpy.full(1, numpy.nan))
    assert cu.lib.gp_logdet_from_chol(dptr(to_dev(L)), n, npad, dptr(out), cu.stream_ptr()) == 0
    ref = 2.0 * math.fsum(numpy.log(d[:n]))
    # each device log within 1 ulp, a strided sum of <= n / 1024 + 1 terms and a 10-level tree: (n / 1024 + 12) u sum |log|
    bound = 2.0 * (n / 1024 + 12) * EPS * math.fsum(numpy.abs(numpy.log(d[:n])))
    assert abs(to_host(out)[0] - ref) <= bound


@gpu
@pytest.mark.parametrize('n', [1, 129, 1152])
def test_shift_copy_exact(cu, n):
    npad = padded(n)
    rng = numpy.random.default_rng(n)
    K = int_matrix(rng, (npad, npad)) / 8.0
    K[n:, :] = 0.0
    K[:, n:] = 0.0
    K[range(n, npad), range(n, npad)] = 1.0
    A0 = numpy.full((npad, npad), SENTINEL)
    Ad = to_dev(A0)
    eta = 0.375
    assert cu.lib.gp_shift_copy(dptr(to_dev(K)), n, npad, eta, dptr(Ad), cu.stream_ptr()) == 0
    A = to_host(Ad)
    blk = numpy.arange(npad) // 128
    lower_tiles = blk[:, None] >= blk[None, :]
    want = K.copy()
    want[range(n), range(n)] += eta
    assert_equal(A[lower_tiles], want[lower_tiles], 'shift_copy')
    assert (numpy.diag(A)[n:] == 1.0).all()
    assert_untouched(A[~lower_tiles], A0[~lower_tiles], 'shift_copy: upper tiles')


@gpu
@pytest.mark.parametrize('n', [1, 129, 1152])
@pytest.mark.parametrize('p', [1, 5, 16])
def test_symm_skinny_exact(cu, n, p):
    torch = _torch()
    npad = padded(n)
    rng = numpy.random.default_rng(n + p)
    K = int_matrix(rng, (npad, npad))
    K = numpy.tril(K) + numpy.tril(K, -1).T
    K[n:, :] = 0.0
    K[:, n:] = 0.0
    K[range(n, npad), range(n, npad)] = 1.0
    X = int_matrix(rng, (npad, p))
    X[n:] = numpy.nan                                        # rows >= n are ignored
    Yd = torch.full((npad, p), float('nan'), dtype=torch.float64, device='cuda')
    assert cu.lib.gp_symm_skinny(dptr(to_dev(K)), n, npad, dptr(to_dev(X)), p, dptr(Yd), cu.stream_ptr()) == 0
    want = numpy.zeros((npad, p))
    want[:n] = K[:n, :n] @ X[:n]
    assert_equal(to_host(Yd), want, 'symm_skinny n=%d p=%d' % (n, p))


def matern15(pts, rho):
    from numpy_ops import _matern
    x = numpy.sqrt((((pts[:, None, :] - pts[None, :, :]) / rho) ** 2).sum(-1))
    K, dK = _matern(x, 1.5, 1.0 / rho)
    numpy.fill_diagonal(dK, 0.0)
    return K, dK


@gpu
@pytest.mark.parametrize('flags', [0, 1, 2, 2 | 4, 1 | 8, 2 | 4 | 8])
@pytest.mark.parametrize('p', [1, 3, 16])
def test_loglik_dense_slots(cu, flags, p):
    torch = _torch()
    n, rho, eta = 300, 0.1, 0.1
    npad = padded(n)
    rng = numpy.random.default_rng(p)
    pts = rng.random((n, 2))
    Kh, dK = matern15(pts, rho)
    Kp = numpy.eye(npad)
    Kp[:n, :n] = Kh
    R = numpy.zeros((npad, p))
    R[:n] = rng.standard_normal((n, p))
    Kn = Kh + eta * numpy.eye(n)
    Ki = numpy.linalg.inv(Kn)
    lam = numpy.linalg.eigvalsh(Kn)
    kappa = lam[-1] / lam[0]
    Rn = R[:n]
    S = Ki @ Rn
    ref = {'G': Rn.T @ S, 'H': S.T @ S, 'Q': S.T @ dK @ S, 'T3': S.T @ Ki @ S}
    out_len = cu.lib.gp_loglik_out_len(p)
    out = to_dev(numpy.full(out_len, numpy.nan))
    A = to_dev(numpy.full((npad, npad), numpy.nan))                 # scratch: never read before it is written
    W = to_dev(numpy.full((npad, npad), numpy.nan))
    pws = torch.empty(cu.lib.gp_potrf_workspace_bytes(npad) // 8, dtype=torch.float64, device='cuda')
    ws = torch.empty(cu.lib.gp_loglik_workspace_bytes(npad) // 8 + 1, dtype=torch.float64, device='cuda')
    scale = numpy.array([rho, rho])
    ptsd = to_dev(pts)
    assert cu.lib.gp_loglik_dense(dptr(to_dev(Kp)), n, npad, dptr(to_dev(R)), p, eta, flags, dptr(ptsd), 2,
                                  cu.host_ptr(scale), 1.5, dptr(A), dptr(W), dptr(pws), dptr(ws), dptr(out),
                                  cu.stream_ptr()) == 0
    o = to_host(out)
    # a backward-stable factorisation gives relative errors of c n u kappa per solve with Kn; a quantity with k solves
    # (R^T Kn^-k R, tr Kn^-k) is within k n u kappa of its scale (normwise); c = 4
    tol = 4 * npad * EPS * kappa
    # log det: a backward error |dKn| <= c n u ||Kn|| moves it by tr(Kn^-1 dKn) <= n c n u kappa
    assert abs(o[0] - numpy.linalg.slogdet(Kn)[1]) <= n * tol
    assert o[4] == 0.0 and (o[5:8] == 0.0).all()
    if flags & 3:
        assert abs(o[1] - numpy.trace(Ki)) <= tol * numpy.trace(Ki)
    if flags & 2:
        assert abs(o[2] - numpy.sum(Ki * Ki)) <= 2 * tol * numpy.sum(Ki * Ki)
    if flags & 4:
        assert abs(o[3] - numpy.sum(Ki * dK)) <= tol * numpy.sum(numpy.abs(Ki) * numpy.abs(dK))
    nR2 = numpy.linalg.norm(Rn, 2) ** 2
    nKi = 1.0 / lam[0]
    blocks = {name: o[8 + i * p * p:8 + (i + 1) * p * p].reshape(p, p) for i, name in enumerate(('G', 'H', 'Q', 'T3'))}
    assert numpy.max(numpy.abs(blocks['G'] - ref['G'])) <= tol * nR2 * nKi
    assert numpy.max(numpy.abs(blocks['H'] - ref['H'])) <= 2 * tol * nR2 * nKi ** 2
    if flags & 4:
        assert numpy.max(numpy.abs(blocks['Q'] - ref['Q'])) <= 2 * tol * nR2 * nKi ** 2 * numpy.linalg.norm(dK, 2)
    else:
        assert (blocks['Q'] == 0.0).all()
    if flags & 8:
        assert numpy.max(numpy.abs(blocks['T3'] - ref['T3'])) <= 3 * tol * nR2 * nKi ** 3
    else:
        assert (blocks['T3'] == 0.0).all()


@gpu
@pytest.mark.parametrize('n,pivot', [(300, 1), (300, 129), (1152, 700)])
def test_loglik_dense_reports_pivot(cu, n, pivot):
    torch = _torch()
    rng = numpy.random.default_rng(pivot)
    L = dyadic_factor(n, rng)
    npad = L.shape[0]
    D = numpy.ones(npad)
    D[pivot - 1] = -1.0
    K = (L * D) @ L.T
    R = numpy.zeros((npad, 2))
    R[:n] = 1.0
    out = to_dev(numpy.full(cu.lib.gp_loglik_out_len(2), numpy.nan))
    A = torch.empty((npad, npad), dtype=torch.float64, device='cuda')
    pws = torch.empty(cu.lib.gp_potrf_workspace_bytes(npad) // 8, dtype=torch.float64, device='cuda')
    ws = torch.empty(cu.lib.gp_loglik_workspace_bytes(npad) // 8 + 1, dtype=torch.float64, device='cuda')
    assert cu.lib.gp_loglik_dense(dptr(to_dev(K)), n, npad, dptr(to_dev(R)), 2, 0.0, 0, None, 0, None, 0.5, dptr(A), None,
                                  dptr(pws), dptr(ws), dptr(out), cu.stream_ptr()) == 0
    assert to_host(out)[4] == float(pivot)


# ------------------------------------------------------------------------------ GpuOps == NumpyOps on other ranks' shapes
@gpu
@pytest.mark.parametrize('P,nb,NB', [(2, 256, 5), (3, 256, 5), (8, 128, 10)])
def test_gpu_ops_match_numpy_ops(cu, P, nb, NB):
    from gaussian_proc._blockcyclic import GpuOps
    from numpy_ops import NumpyOps, _matern
    g, h = GpuOps(), NumpyOps()
    npad = NB * nb
    n = npad - 77                                          # the last block has nvalid = nb - 77 < nb
    r, I = blockcyclic_layout(P, nb, NB)
    nq = len(I)
    rng = numpy.random.default_rng(P)

    def both(a):
        return g.from_host(a), h.from_host(a)

    def same(gd, hd, what):
        assert_equal(g.to_host(gd), h.to_host(hd), what)

    # staircase GEMMs of inverse_rows / inverse_traces on this rank's rows of W (NaN right of the staircase)
    X = int_matrix(rng, (nq * nb, npad))
    for q, i in enumerate(I):
        X[q * nb:(q + 1) * nb, (i + 1) * nb:] = numpy.nan
    Xg, Xh = both(X)
    panel = int_matrix(rng, (npad, nb))
    Pg, Ph = both(panel)
    for kind, k, q0, tab in staircase_tables(I, nb, NB):
        rows = slice(q0 * nb, nq * nb)
        if kind == 'kend':
            Tg, Th = g.zeros(((nq - q0) * nb, nb)), h.zeros(((nq - q0) * nb, nb))
            g.gemm(Tg, Xg[rows, (k + 1) * nb:], Pg[:(NB - k - 1) * nb], 1.0, 0.0, at=0, bt=1, kend=g.int_tensor(tab))
            h.gemm(Th, Xh[rows, (k + 1) * nb:], Ph[:(NB - k - 1) * nb], 1.0, 0.0, at=0, bt=1, kend=h.int_tensor(tab))
        else:
            M = npad - k * nb
            Tg, Th = g.zeros((M, nb)), h.zeros((M, nb))
            g.gemm(Tg, Xg[rows, k * nb:], Xg[rows, k * nb:(k + 1) * nb], 1.0, 0.0, at=1, bt=1, kbeg=g.int_tensor(tab))
            h.gemm(Th, Xh[rows, k * nb:], Xh[rows, k * nb:(k + 1) * nb], 1.0, 0.0, at=1, bt=1, kbeg=h.int_tensor(tab))
        same(Tg, Th, 'gemm %s k=%d' % (kind, k))
    # plain GEMM of a trailing block-column update (C -= panel rows x panel block^T)
    C0 = int_matrix(rng, (npad - nb, nb))
    Cg, Ch = both(C0)
    g.gemm(Cg, Pg[nb:], Pg[:nb], -1.0, 1.0)
    h.gemm(Ch, Ph[nb:], Ph[:nb], -1.0, 1.0)
    same(Cg, Ch, 'gemm')
    # skinny products: a slab of rows with a row stride wider than its width; rect_apply_t over M > 2048 rows
    p = 7
    slab = int_matrix(rng, (npad, npad))
    Sg, Sh = both(slab)
    Rm = int_matrix(rng, (npad - nb, p))
    Rg, Rh = both(Rm)
    Y0 = int_matrix(rng, (npad, p))
    Yg, Yh = both(Y0)
    g.rect_apply(Sg[:, nb:], Rg, Yg, alpha=-1.0, beta=1.0)
    h.rect_apply(Sh[:, nb:], Rh, Yh, alpha=-1.0, beta=1.0)
    same(Yg, Yh, 'rect_apply')
    Mt = max(npad, 2304)                                   # two 2048-row chunks of the two-stage reduction
    Xt = int_matrix(rng, (Mt, nb + 6))
    Xtg, Xth = both(Xt)
    Yt = int_matrix(rng, (Mt, p))
    Ytg, Yth = both(Yt)
    S0 = int_matrix(rng, (nb, p))
    S0g, S0h = both(S0)
    g.rect_apply_t(Xtg[:, 6:], Ytg, S0g, alpha=-1.0, beta=1.0)
    h.rect_apply_t(Xth[:, 6:], Yth, S0h, alpha=-1.0, beta=1.0)
    same(S0g, S0h, 'rect_apply_t')
    accg, acch = both(numpy.array([3.0, 0.0]))
    g.pair_dot(Sg[:nq * nb, nb:], Sg[:nq * nb, :npad - nb], nb // 2, 2.0, accg[0:1])
    h.pair_dot(Sh[:nq * nb, nb:], Sh[:nq * nb, :npad - nb], nb // 2, 2.0, acch[0:1])
    same(accg, acch, 'pair_dot')
    # generator blocks of this rank's columns (rows running into the padding) and of a lower block column
    d = 2
    pts = numpy.zeros((npad, d))
    pts[:n] = rng.random((n, d))
    scale = numpy.array([0.3, 0.3])
    cg = numpy.concatenate([numpy.arange(j * nb, (j + 1) * nb) for j in I]).astype(numpy.int32)
    for nu in (0.5, 1.5, 2.5):
        for j0 in (0, I[0]):
            rg = numpy.arange(j0 * nb, npad, dtype=numpy.int32)
            x = numpy.sqrt((((pts[rg][:, None, :] - pts[cg][None, :, :]) / scale) ** 2).sum(-1))
            outs = []
            for ops in (g, h):
                out = ops.zeros((len(rg), len(cg)))
                outd = ops.zeros((len(rg), len(cg)))
                ops.generate(ops.from_host(pts[rg]), ops.from_host(pts[cg]), ops.from_host(rg), ops.from_host(cg), n, scale,
                             nu, 0.25, out)
                ops.generate_dk(ops.from_host(pts[rg]), ops.from_host(pts[cg]), ops.from_host(rg), ops.from_host(cg), n,
                                scale, nu, outd)
                outs.append((ops.to_host(out), ops.to_host(outd)))
            # a few ulp of each value: distance, exp and polynomial each differ in the last bit, and a relative error d
            # of the distance moves the value by about sqrt(2 nu) x d (<= 2.3 x d): 16 (1 + x) ulp
            tolr = 16 * EPS * (1.0 + x)
            assert (numpy.abs(outs[0][0] - outs[1][0]) <= tolr * numpy.abs(outs[1][0]) + 1e-300).all(), nu
            assert (numpy.abs(outs[0][1] - outs[1][1]) <= tolr * numpy.abs(outs[1][1]) + 1e-300).all(), nu
        Sm = numpy.zeros((npad, p))
        Sm[:n] = rng.standard_normal((n, p))
        Vg, Vh = g.zeros((npad, p)), h.zeros((npad, p))
        g.dk_apply(g.from_host(pts[:n]), n, scale, nu, g.from_host(Sm), Vg)
        h.dk_apply(h.from_host(pts[:n]), n, scale, nu, h.from_host(Sm), Vh)
        xx = numpy.sqrt((((pts[:n][:, None, :] - pts[:n][None, :, :]) / scale) ** 2).sum(-1))
        absdk = numpy.abs(_matern(xx, nu, 1.0 / scale[0])[1])
        # n terms per entry, each value within 16 (1 + x) ulp (see above), then n - 1 additions: (n + 16 (1 + max x)) u |dK| |S|
        bound = (n + 16 * (1 + xx.max())) * EPS * (absdk @ numpy.abs(Sm[:n]))
        assert (numpy.abs(g.to_host(Vg)[:n] - h.to_host(Vh)[:n]) <= bound + 1e-300).all(), nu
        assert (g.to_host(Vg)[n:] == 0.0).all()
    # factor + inverse of the last diagonal block (nvalid < nb, identity padding) and its log-determinant
    nvalid = n - (NB - 1) * nb
    Dh = numpy.eye(nb)
    Kb, _ = matern15(rng.random((nvalid, 2)), 0.2)
    Dh[:nvalid, :nvalid] = Kb + 0.1 * numpy.eye(nvalid)
    Dg_, Dh_ = both(Dh)
    Lg_, Lh_ = g.zeros((nb, nb)), h.zeros((nb, nb))
    ig, ih = g.potrf_inv(Dg_, nvalid, Lg_), h.potrf_inv(Dh_, nvalid, Lh_)
    assert int(g.to_host(ig)[0]) == 0 and int(h.to_host(ih)[0]) == 0
    lam = numpy.linalg.eigvalsh(Dh)
    kappa = lam[-1] / lam[0]
    Lref = h.to_host(Dh_)
    Lgot = numpy.tril(g.to_host(Dg_))
    # Cholesky forward error (normwise): ||dL|| <= c n u kappa ||L||, c = 4; the same for inv(L)
    assert numpy.max(numpy.abs(Lgot - Lref)) <= 4 * nb * EPS * kappa * numpy.max(numpy.abs(Lref))
    Wref = h.to_host(Lh_)
    assert numpy.max(numpy.abs(g.to_host(Lg_) - Wref)) <= 4 * nb * EPS * kappa * numpy.max(numpy.abs(Wref))
    og, oh = g.zeros(1), h.zeros(1)
    g.logdet_chol(Dg_, nvalid, og)
    h.logdet_chol(Dh_, nvalid, oh)
    dg = numpy.diag(Lref)[:nvalid]
    # 2 sum |dL_ii| / L_ii with the bound on dL above, plus the summation of nvalid logs (see test_logdet_from_chol)
    bound = 2 * nvalid * 4 * nb * EPS * kappa * numpy.max(numpy.abs(Lref)) / dg.min() + \
        2 * (nvalid / 1024 + 12) * EPS * math.fsum(numpy.abs(numpy.log(dg)))
    assert abs(g.to_host(og)[0] - h.to_host(oh)[0]) <= bound
    assert r != 0
