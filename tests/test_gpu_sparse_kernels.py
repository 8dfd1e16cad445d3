"""Kernel-level tests of the sparse-operator entry points of the C ABI (include/gpgp.h), one entry point at a time,
on one GPU (peer = NULL).

The inputs make the correct FP64 answer exact whatever the summation order, so that a dropped or doubled entry, a
value in the wrong fragment row, a missing eta on a ragged block or a skipped Gram row shows as a bit difference:
  - matrices: nonzero integers in [-4, 4] (so the pattern is the set of nonzero values), blocks X, Y: integers in
    [-4, 4], eta, coefficients and the like: dyadic. Every partial sum is then an integer multiple of a power of two far
    below 2^53 (at most 16 x 3001 for the longest row used, 300 x 4 x 4 in sixteenths for the longest combine),
    so float64 NumPy in any order, the warp-shuffle sums and the DMMA path all give the same bits;
  - the row-blocked operator is decoded on the host with the fragment formula of gpgp.h (value (s, k) at
    64 (s/4) + 32 (k/8) + 4 (k%8) + s%4) and must equal P A P^T entry for entry, in the documented slot order.
Output buffers carry one extra row or block holding a NaN sentinel, compared bit for bit after the call. Lanczos and
CG have no exact answer: the bounds are derived from the recurrence and written next to each assert.

The tests marked gpu need a CUDA device; the unmarked ones check on the CPU that the exact references are exact."""

import ctypes

import numpy
import pytest
import scipy.sparse

gpu = pytest.mark.gpu

EPS = numpy.finfo(numpy.float64).eps
SENTINEL = numpy.array([0x7ff8dead0000beef], dtype=numpy.uint64).view(numpy.float64)[0]   # a NaN with a payload
ISENTINEL = -123456789
ROWS = 16                   # BCSR_ROWS, csrc/gp_internal.h
HMAX = 1536                 # distinct columns a row block may have on the hash path of bcsr_build_kernel
WIDTHS = [1, 2, 4, 8, 16, 32]
ETAS = [0.0, 0.75, -2.5]
NONZERO = numpy.array([-4, -3, -2, -1, 1, 2, 3, 4], dtype=numpy.float64)


# ------------------------------------------------------------------------------------------------ host-side references
def int_block(rng, shape):
    return rng.integers(-4, 5, size=shape).astype(numpy.float64)


def random_rows(rng, n, lengths):
    """a list of n column arrays (distinct columns per row, random order), lengths[i] entries in row i"""
    return [rng.choice(n, size=min(int(k), n), replace=False) for k in lengths]


def to_csr(rows, values, sort_rows):
    """(indptr int32, indices int32, data float64) with row i holding rows[i] and values[i]; sort_rows: by column"""
    ind, dat = [], []
    for c, v in zip(rows, values):
        p = numpy.argsort(c, kind='stable') if sort_rows else numpy.arange(len(c))
        ind.append(numpy.asarray(c, dtype=numpy.int32)[p])
        dat.append(numpy.asarray(v, dtype=numpy.float64)[p])
    indptr = numpy.zeros(len(rows) + 1, dtype=numpy.int32)
    indptr[1:] = numpy.cumsum([len(c) for c in rows])
    cat = lambda a, t: numpy.concatenate(a).astype(t) if a else numpy.zeros(0, t)   # noqa: E731
    return indptr, cat(ind, numpy.int32), cat(dat, numpy.float64)


def scipy_of(indptr, indices, data, n):
    return scipy.sparse.csr_matrix((data, indices, indptr), shape=(n, n))


def int_matrix(rng, n, max_len, empty=(), dense=(), sort_rows=True):
    """n x n CSR with nonzero integer values in [-4, 4]: row lengths uniform in [0, max_len], the rows in `empty` empty,
    the rows in `dense` full; rows in random column order unless sort_rows"""
    lengths = rng.integers(0, max_len + 1, size=n)
    lengths[list(empty)] = 0
    lengths[list(dense)] = n
    rows = random_rows(rng, n, lengths)
    values = [rng.choice(NONZERO, size=len(c)) for c in rows]
    return to_csr(rows, values, sort_rows)


def permuted_source(op_rows, op_values, order, sort_rows):
    """the source matrix A whose row-blocked form with this order is the operator M (rows op_rows / op_values in
    operator space): A[order[r], order[c]] = M[r, c]"""
    n = len(op_rows)
    rows, values = [None] * n, [None] * n
    for r in range(n):
        rows[order[r]] = order[op_rows[r]]
        values[order[r]] = op_values[r]
    return to_csr(rows, values, sort_rows)


def expected_blocks(indptr, indices, data, order, n):
    """The row-blocked form of P A P^T as gpgp.h describes it: per block of 16 rows, the distinct columns in order of
    first appearance (row 0's entries in the source row's order, then the new ones of row 1, ...), padded to a multiple of
    4 with zero slots. Returns nblk (per block), cols (per block, the real slots) and the (slot, row) values of the real
    slots, slots numbered from 0 in each block."""
    inv = numpy.argsort(order) if order is not None else None
    nrb = (n + ROWS - 1) // ROWS
    nblk, cols, vals = numpy.zeros(nrb, dtype=numpy.int64), [], []
    for rb in range(nrb):
        slot, lst, v = {}, [], {}
        for k in range(min(ROWS, n - rb * ROWS)):
            o = order[rb * ROWS + k] if order is not None else rb * ROWS + k
            for t in range(indptr[o], indptr[o + 1]):
                c = int(inv[indices[t]]) if inv is not None else int(indices[t])
                if c not in slot:
                    slot[c] = len(lst)
                    lst.append(c)
                v[(slot[c], k)] = data[t]
        nblk[rb] = (len(lst) + 3) // 4 * 4
        cols.append(lst)
        vals.append(v)
    return nblk, cols, vals


def fragment_positions(total):
    """index into bvals of value (slot s, row k): 64 (s/4) + 32 (k/8) + 4 (k%8) + s%4, as a (total, 16) array"""
    s = numpy.arange(total, dtype=numpy.int64)[:, None]
    k = numpy.arange(ROWS, dtype=numpy.int64)[None, :]
    return 64 * (s // 4) + 32 * (k // 8) + 4 * (k % 8) + s % 4


def decode_blocks(bptr, bidx, bvals, n):
    """the operator (n x n scipy CSR, duplicates summed) and the (total, 16) value table of a row-blocked operator"""
    total = int(bptr[-1])
    V = bvals[fragment_positions(total)]
    rb = numpy.repeat(numpy.arange(len(bptr) - 1), numpy.diff(bptr))
    rows = rb[:, None] * ROWS + numpy.arange(ROWS)[None, :]
    cols = numpy.broadcast_to(bidx[:total, None], V.shape)
    keep = V != 0.0
    assert (rows[keep] < n).all(), 'a value in a row past n'
    M = scipy.sparse.coo_matrix((V[keep], (rows[keep], cols[keep])), shape=(n, n)).tocsr()
    return M, V


def encode_blocks(nblk, cols, vals):
    """the inverse of decode_blocks for expected_blocks' description: (bptr, bidx with padding -1, bvals)"""
    bptr = numpy.concatenate([[0], numpy.cumsum(nblk)]).astype(numpy.int64)
    total = int(bptr[-1])
    bidx = numpy.full(total, -1, dtype=numpy.int64)
    table = numpy.zeros((total, ROWS))
    for rb in range(len(nblk)):
        bidx[bptr[rb]:bptr[rb] + len(cols[rb])] = cols[rb]
        for (s, k), v in vals[rb].items():
            table[bptr[rb] + s, k] = v
    bvals = numpy.zeros(total * ROWS)
    bvals[fragment_positions(total)] = table
    return bptr, bidx, bvals


def lanczos_ref(A, eta, V, m):
    """The recurrence of lanczos_run (csrc/gp_sparse_la.cu) in the same unnormalised form, column by column, in float64:
    u_0 = v, s_0 = 1 / ||v||; W = s_j (A + eta I) u_j, alpha_j = s_j u_j . W, u_{j+1} = W - alpha_j s_j u_j -
    beta_{j-1} s_{j-1} u_{j-1}, beta_j = ||u_{j+1}||, s_{j+1} = 1 / beta_j (0 after a breakdown)."""
    u = V.copy()
    up = numpy.zeros_like(u)
    s = 1.0 / numpy.sqrt((u * u).sum(axis=0))
    sp = numpy.zeros_like(s)
    bp = numpy.zeros_like(s)
    alpha, beta = numpy.zeros((m, V.shape[1])), numpy.zeros((m, V.shape[1]))
    for j in range(m):
        W = (A @ u + eta * u) * s
        al = s * (u * W).sum(axis=0)
        un = W - (al * s) * u - (bp * sp) * up
        bt = numpy.sqrt((un * un).sum(axis=0))
        alpha[j], beta[j] = al, bt
        up, u, sp, bp = u, un, s, bt
        with numpy.errstate(divide='ignore'):
            s = numpy.where(bt > 1e-300, 1.0 / bt, 0.0)
    return alpha, beta


def tridiag(alpha, beta, k):
    return numpy.diag(alpha[:k]) + numpy.diag(beta[:k - 1], 1) + numpy.diag(beta[:k - 1], -1)


def sym_int_matrix(rng, n, max_len):
    """symmetric integer matrix A + A^T without diagonal (|entries| <= 8) and its largest absolute row sum"""
    ip, ix, dt = int_matrix(rng, n, max_len)
    A = scipy_of(ip, ix, dt, n)
    S = (A + A.T).tocsr()
    S.setdiag(0.0)
    S.eliminate_zeros()
    S.sort_indices()
    return S, float(abs(S).sum(axis=1).max())


def bits(a):
    return numpy.ascontiguousarray(a).view(numpy.uint64)


def assert_equal(got, want, what):
    """exact equality (0.0 == -0.0); NaN anywhere in got fails"""
    bad = ~(got == want)
    assert not bad.any(), '%s: %d of %d entries differ, first at %s: %r vs %r' % (
        what, bad.sum(), bad.size, tuple(numpy.argwhere(bad)[0]), got[bad][0], want[bad][0])


def assert_untouched(got, want, what):
    bad = bits(got) != bits(want)
    assert not bad.any(), '%s: %d entries written that must stay untouched' % (what, bad.sum())


# ---------------------------------------------------------------------------------- CPU checks of the exact references
def test_integer_products_are_exact():
    """the longest row used (a dense row of 3001 entries) and the widest block: float64 in two summation orders equals
    int64 arithmetic, and every partial sum is far below 2^53"""
    rng = numpy.random.default_rng(1)
    n = 3001
    ip, ix, dt = int_matrix(rng, n, 40, empty=[5, 6], dense=[17])
    A = scipy_of(ip, ix, dt, n)
    X = int_block(rng, (n, 32))
    exact = A.astype(numpy.int64) @ X.astype(numpy.int64)
    assert numpy.array_equal(A @ X, exact.astype(numpy.float64))
    assert numpy.array_equal((X.T @ A.T.toarray()).T, exact.astype(numpy.float64))
    for eta in ETAS:          # dyadic eta: (A + eta I) X is a multiple of 1/4
        assert numpy.array_equal(A @ X + eta * X, (4 * exact + int(4 * eta) * X.astype(numpy.int64)) / 4.0)
    assert 16 * n * 4 < 2 ** 53


def test_block_combine_reference_is_exact():
    """the largest degree used (m = 300): coefficients k / 16 with |k| <= 64 and integer basis vectors in [-4, 4] give
    sums that are multiples of 1/16 below 300 * 64 * 4: the same bits in any order"""
    rng = numpy.random.default_rng(2)
    m, n, B = 300, 257, 32
    basis = int_block(rng, (m, n, B))
    coef = rng.integers(-64, 65, size=(m, B)) / 16.0
    exact = numpy.einsum('jc,jic->ic', (16 * coef).astype(numpy.int64), basis.astype(numpy.int64))
    want = exact / 16.0
    assert numpy.array_equal(numpy.einsum('jc,jic->ic', coef, basis), want)
    acc = numpy.zeros((n, B))
    for j in range(m):                                          # the kernel's order: j = 0 .. m - 1
        acc += coef[j] * basis[j]
    assert numpy.array_equal(acc, want)
    acc = numpy.zeros((n, B))
    for j in reversed(range(m)):
        acc += coef[j] * basis[j]
    assert numpy.array_equal(acc, want)
    assert 300 * 64 * 4 * 16 < 2 ** 53


@pytest.mark.parametrize('n,perm', [(1, False), (17, True), (300, True)])
def test_fragment_decoder_round_trips(n, perm):
    """encode_blocks (the slot / fragment layout gpgp.h documents) and decode_blocks are inverse: the decoded operator is
    P A P^T, every value lands on its own (row, column)"""
    rng = numpy.random.default_rng(n)
    ip, ix, dt = int_matrix(rng, n, min(n, 40), empty=[0], dense=[n // 2], sort_rows=False)
    order = rng.permutation(n).astype(numpy.int32) if perm else None
    nblk, cols, vals = expected_blocks(ip, ix, dt, order, n)
    bptr, bidx, bvals = encode_blocks(nblk, cols, vals)
    assert (nblk % 4 == 0).all()
    M, V = decode_blocks(bptr, numpy.where(bidx < 0, 0, bidx), bvals, n)
    A = scipy_of(ip, ix, dt, n)
    P = A if order is None else A[order][:, order]
    assert (M != P).nnz == 0 and M.nnz == A.nnz == int((bvals != 0).sum())
    # a swapped pair of 8-row fragments is visible: other values, or values in the rows past n of the last block
    if n > 8:
        swapped = bvals.reshape(-1, 2, 32)[:, ::-1].ravel()
        try:
            seen = (decode_blocks(bptr, numpy.where(bidx < 0, 0, bidx), swapped, n)[0] != P).nnz > 0
        except AssertionError:
            seen = True
        assert seen


def test_lanczos_reference_recurrence():
    """the NumPy recurrence run to m = n on a small matrix: the Ritz values of T are the eigenvalues of A + eta I; on a
    diagonal matrix with 5 distinct values it breaks down at step 5"""
    rng = numpy.random.default_rng(3)
    A, _ = tiny_dense_matrix(rng)
    V = int_block(rng, (A.shape[0], 4))
    alpha, beta = lanczos_ref(A, 0.5, V, A.shape[0])
    for c in range(4):
        ritz = numpy.linalg.eigvalsh(tridiag(alpha[:, c], beta[:, c], A.shape[0]))
        assert numpy.abs(ritz - numpy.linalg.eigvalsh(A + 0.5 * numpy.eye(A.shape[0]))).max() <= 1e-11
    D, vals = diagonal_matrix()
    alpha, beta = lanczos_ref(D.toarray(), 0.0, numpy.ones((D.shape[0], 1)), 10)
    k = len(vals)
    assert beta[k - 2, 0] > 0.1 and beta[k - 1, 0] <= 1e-12 and numpy.isfinite(alpha).all() and numpy.isfinite(beta).all()
    assert numpy.abs(numpy.linalg.eigvalsh(tridiag(alpha[:, 0], beta[:, 0], k)) - vals).max() <= 1e-12


def tiny_dense_matrix(rng, n=12):
    """symmetric n x n with every entry a nonzero integer in [-4, 4] (off-diagonal) and a diagonal 8 i that spreads the
    spectrum: eigenvalue gaps of a few units, so m = n Lanczos steps resolve every eigenvalue"""
    A = rng.choice(NONZERO, size=(n, n))
    A = numpy.triu(A, 1) + numpy.triu(A, 1).T
    A[range(n), range(n)] = 8.0 * numpy.arange(n)
    return A, n


def diagonal_matrix(n=40):
    """diag of 5 distinct values, each repeated: the Krylov space of any start vector with nonzero components has
    dimension 5"""
    vals = numpy.array([1.0, 2.0, 3.0, 5.0, 8.0])
    return scipy.sparse.diags(vals[numpy.arange(n) % 5]).tocsr(), vals


# ------------------------------------------------------------------------------------------------------- device plumbing
@pytest.fixture(scope='module')
def cu():
    from gaussian_proc import _device as dev
    dev.require_cuda()
    return dev


def _torch():
    import torch
    return torch


def dptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def to_dev(a, dtype=numpy.float64):
    torch = _torch()
    return torch.from_numpy(numpy.ascontiguousarray(a, dtype=dtype)).cuda()


def to_host(t):
    torch = _torch()
    torch.cuda.synchronize()
    return t.cpu().numpy()


def with_sentinel_rows(shape, extra=1, value=SENTINEL):
    """device buffer of shape[0] + extra rows, all `value` (the extra rows are the sentinel)"""
    return to_dev(numpy.full((shape[0] + extra,) + tuple(shape[1:]), value))


class DevCSR(object):
    def __init__(self, indptr, indices, data, ddata=None):
        self.n = len(indptr) - 1
        self.h = (indptr, indices, data, ddata)
        self.indptr, self.indices = to_dev(indptr, numpy.int32), to_dev(indices, numpy.int32)
        self.data = to_dev(data)
        self.ddata = to_dev(ddata) if ddata is not None else None


def build_blocks(cu, A, order, with_ddata):
    """gp_bcsr_count -> gp_scan_counts -> gp_bcsr_fill on a DevCSR; the outputs carry sentinels (one block of values,
    four indices) past the end. Returns dict of host arrays and device tensors."""
    torch = _torch()
    n, s = A.n, cu.stream_ptr()
    nrb = (n + ROWS - 1) // ROWS
    o = to_dev(order, numpy.int32) if order is not None else None
    inv = to_dev(numpy.argsort(order), numpy.int32) if order is not None else None
    nblk = to_dev(numpy.full(nrb + 1, ISENTINEL), numpy.int32)
    flag = to_dev(numpy.full(1, 7), numpy.int32)
    assert cu.lib.gp_bcsr_count(n, dptr(o), dptr(inv), dptr(A.indptr), dptr(A.indices), dptr(nblk), dptr(flag), s) == 0
    bptr = to_dev(numpy.full(nrb + 2, ISENTINEL), numpy.int64)
    assert cu.lib.gp_scan_counts(dptr(nblk), nrb, dptr(bptr), s) == 0
    bptr_h = to_host(bptr)
    total = int(bptr_h[nrb])
    bidx = to_dev(numpy.full(total + 4, ISENTINEL), numpy.int32)
    bvals = to_dev(numpy.full(16 * total + 64, SENTINEL))
    bdvals = to_dev(numpy.full(16 * total + 64, SENTINEL)) if with_ddata else None
    assert cu.lib.gp_bcsr_fill(n, dptr(o), dptr(inv), dptr(A.indptr), dptr(A.indices), dptr(A.data),
                               dptr(A.ddata) if with_ddata else None, dptr(bptr), total, dptr(bidx), dptr(bvals),
                               dptr(bdvals), s) == 0
    out = {'nblk': to_host(nblk), 'flag': int(to_host(flag)[0]), 'bptr': bptr_h, 'bidx': to_host(bidx),
           'bvals': to_host(bvals), 'bdvals': to_host(bdvals) if with_ddata else None, 'total': total}
    out['dev'] = (bptr, bidx, bvals, bdvals)
    return out


def csr_spmm(cu, A, eta, X, B):
    Y = with_sentinel_rows((A.n, B))
    rc = cu.lib.gp_csr_spmm(dptr(A.indptr), dptr(A.indices), dptr(A.data), A.n, eta, dptr(to_dev(X)), B, dptr(Y),
                            cu.stream_ptr())
    return rc, to_host(Y)


def bcsr_spmm(cu, blk, n, eta, X, B, values=None):
    bptr, bidx, bvals, _ = blk['dev']
    Y = with_sentinel_rows((n, B))
    rc = cu.lib.gp_bcsr_spmm(None, dptr(bptr), dptr(bidx), dptr(bvals if values is None else values), n, eta,
                             dptr(to_dev(X)), B, dptr(Y), cu.stream_ptr())
    return rc, to_host(Y)


def check_product(Y, want, n, B, what):
    assert_equal(Y[:n], want, what)
    assert_untouched(Y[n:], numpy.full((1, B), SENTINEL), what + ': row past n')


# ------------------------------------------------------------------------------------------------------------ SpMM
@gpu
@pytest.mark.parametrize('n', [1, 15, 16, 17, 3001])
def test_csr_spmm_exact(cu, n):
    """(A + eta I) X bit for bit, with empty rows and one dense row; widths outside {1, 2, 4, ..., 32} return -2"""
    rng = numpy.random.default_rng(n)
    empty = [i for i in (0, 3, n - 1) if i < n and i != n // 2]
    ip, ix, dt = int_matrix(rng, n, min(n, 40), empty=empty, dense=[n // 2], sort_rows=False)
    A = DevCSR(ip, ix, dt)
    As = scipy_of(ip, ix, dt, n)
    for B in WIDTHS:
        X = int_block(rng, (n, B))
        for eta in ETAS:
            rc, Y = csr_spmm(cu, A, eta, X, B)
            assert rc == 0
            check_product(Y, As @ X + eta * X, n, B, 'csr spmm n=%d B=%d eta=%g' % (n, B, eta))
    for B in (3, 64):
        assert csr_spmm(cu, A, 1.0, int_block(rng, (n, B)), B)[0] == -2


# (n, permuted, sorted source rows, with ddata, empty rows, dense rows): n < 16, n == 16, a ragged last block,
# unsorted rows on the hash path, a dense row (a block of n > HMAX distinct columns: the binary-search path)
BUILD_CASES = [
    (1, False, True, True, [], [0]),
    (15, True, False, False, [2], [7]),
    (16, False, False, True, [0, 15], [5]),
    (17, True, True, True, [16], [3]),
    (3001, True, False, True, [0, 1, 2, 1500, 3000], []),
    (3001, False, True, False, [4, 2999], [1000]),
    (3001, True, True, True, [], [2990]),
]


def check_blocks(blk, ip, ix, dt, ddt, order, n, with_ddata):
    """the device row blocks against expected_blocks: counts, prefix sums, slot order, values, zero padding, sentinels"""
    nrb = (n + ROWS - 1) // ROWS
    nblk, cols, vals = expected_blocks(ip, ix, dt, order, n)
    assert (blk['nblk'][:nrb] == nblk).all(), 'block-column counts'
    assert blk['nblk'][nrb] == ISENTINEL
    assert (blk['bptr'][:nrb + 1] == numpy.concatenate([[0], numpy.cumsum(nblk)])).all()
    assert blk['bptr'][nrb + 1] == ISENTINEL
    total = blk['total']
    bidx = blk['bidx']
    assert (bidx[total:] == ISENTINEL).all(), 'bidx past the end'
    assert_untouched(blk['bvals'][16 * total:], numpy.full(64, SENTINEL), 'bvals past the end')
    assert ((bidx[:total] >= 0) & (bidx[:total] < n)).all(), 'a block-column outside the matrix'
    _, want_bidx, want_vals = encode_blocks(nblk, cols, vals)
    real = want_bidx >= 0
    assert (bidx[:total][real] == want_bidx[real]).all(), 'slot order'
    assert_equal(blk['bvals'][:16 * total], want_vals, 'bvals')
    M, V = decode_blocks(blk['bptr'][:nrb + 1], bidx, blk['bvals'], n)
    A = scipy_of(ip, ix, dt, n)
    P = A if order is None else A[order][:, order]
    assert (M != P).nnz == 0 and int((blk['bvals'][:16 * total] != 0).sum()) == A.nnz
    assert (V[~real] == 0.0).all(), 'padding slots'
    if with_ddata:
        _, _, dvals = expected_blocks(ip, ix, ddt, order, n)
        assert_equal(blk['bdvals'][:16 * total], encode_blocks(nblk, cols, dvals)[2], 'bdvals')
        assert_untouched(blk['bdvals'][16 * total:], numpy.full(64, SENTINEL), 'bdvals past the end')
    return P


@gpu
@pytest.mark.parametrize('n,perm,sort_rows,with_ddata,empty,dense', BUILD_CASES)
def test_bcsr_build_and_spmm_exact(cu, n, perm, sort_rows, with_ddata, empty, dense):
    """gp_bcsr_count / gp_scan_counts / gp_bcsr_fill decode to P A P^T exactly, and gp_bcsr_spmm applies it bit for bit,
    including the ragged last block; B = 3 returns -2"""
    rng = numpy.random.default_rng(n + 10 * perm + 100 * sort_rows)
    ip, ix, dt = int_matrix(rng, n, min(n, 40), empty=empty, dense=dense, sort_rows=sort_rows)
    ddt = rng.choice(NONZERO, size=dt.size)
    order = rng.permutation(n).astype(numpy.int32) if perm else None
    blk = build_blocks(cu, DevCSR(ip, ix, dt, ddt), order, with_ddata)
    over = any(len(c) > HMAX for c in expected_blocks(ip, ix, dt, order, n)[1])
    assert blk['flag'] == int(over), 'needs_sorted flag'
    P = check_blocks(blk, ip, ix, dt, ddt, order, n, with_ddata)
    for B in WIDTHS:
        X = int_block(rng, (n, B))
        for eta in ETAS:
            rc, Y = bcsr_spmm(cu, blk, n, eta, X, B)
            assert rc == 0
            check_product(Y, P @ X + eta * X, n, B, 'bcsr spmm n=%d B=%d eta=%g' % (n, B, eta))
    if with_ddata:
        dP = scipy_of(ip, ix, ddt, n)
        dP = dP if order is None else dP[order][:, order]
        X = int_block(rng, (n, 16))
        rc, Y = bcsr_spmm(cu, blk, n, 0.75, X, 16, values=blk['dev'][3])
        assert rc == 0
        check_product(Y, dP @ X + 0.75 * X, n, 16, 'bcsr spmm on bdvals')
    assert bcsr_spmm(cu, blk, n, 1.0, int_block(rng, (n, 3)), 3)[0] == -2


def capacity_operator(rng, n, widths):
    """operator-space rows: block b of the first len(widths) blocks has exactly widths[b] distinct columns (disjoint
    rows, each column once), every other row a few random columns"""
    rows = random_rows(rng, n, rng.integers(0, 9, size=n))
    for b, w in enumerate(widths):
        cols = rng.permutation(n)[:w]
        for k, part in enumerate(numpy.array_split(cols, ROWS)):
            rows[b * ROWS + k] = part
    return rows, [rng.choice(NONZERO, size=len(c)) for c in rows]


@gpu
@pytest.mark.parametrize('widths,perm,sort_rows', [([HMAX], True, False), ([HMAX, HMAX + 1, 3000], True, True),
                                                   ([HMAX + 1], False, True)])
def test_bcsr_build_at_the_hash_capacity(cu, widths, perm, sort_rows):
    """a row block of exactly HMAX distinct columns stays on the hash path (unsorted source rows are fine there);
    HMAX + 1 and beyond go to the binary-search path and set needs_sorted_dev; both paths give the documented layout"""
    n = 3001
    rng = numpy.random.default_rng(len(widths) + 3 * perm)
    order = rng.permutation(n).astype(numpy.int32) if perm else numpy.arange(n, dtype=numpy.int32)
    op_rows, op_vals = capacity_operator(rng, n, widths)
    ip, ix, dt = permuted_source(op_rows, op_vals, order, sort_rows)
    ddt = rng.choice(NONZERO, size=dt.size)
    o = order if perm else None
    blk = build_blocks(cu, DevCSR(ip, ix, dt, ddt), o, True)
    assert blk['flag'] == int(max(widths) > HMAX)
    assert (blk['nblk'][:len(widths)] == (numpy.array(widths) + 3) // 4 * 4).all()
    P = check_blocks(blk, ip, ix, dt, ddt, o, n, True)
    for B in (1, 16):
        X = int_block(rng, (n, B))
        rc, Y = bcsr_spmm(cu, blk, n, -2.5, X, B)
        assert rc == 0
        check_product(Y, P @ X - 2.5 * X, n, B, 'bcsr spmm at the capacity B=%d' % B)


# ------------------------------------------------------------------------------------------------------ row sort
@gpu
@pytest.mark.parametrize('with_ddata', [False, True])
def test_csr_sort_rows_exact(cu, with_ddata):
    """every row sorted by column with data / ddata following, against numpy.lexsort: rows in reverse order, one-entry
    rows, empty rows, already sorted rows, rows of 512 / 513 / 2048 entries (the warp and CTA-wide sorts)"""
    rng = numpy.random.default_rng(5 + with_ddata)
    n = 4000
    lengths = rng.integers(0, 60, size=n)
    lengths[[0, 10, 11]] = 0
    lengths[[1, 12]] = 1
    lengths[[20, 21, 22]] = [512, 513, 2048]
    rows = random_rows(rng, n, lengths)
    rows[30] = numpy.arange(n)[::-1][:700]                       # reverse order, CTA-wide
    rows[31] = numpy.arange(50)[::-1]                            # reverse order, one warp
    rows[32] = numpy.arange(100, 180)                            # already sorted
    values = [rng.choice(NONZERO, size=len(c)) for c in rows]
    ip, ix, dt = to_csr(rows, values, False)
    ddt = numpy.arange(dt.size, dtype=numpy.float64) + 0.5          # distinct: each value is traceable
    nnz = dt.size
    ind_d = to_dev(numpy.concatenate([ix, [ISENTINEL]]), numpy.int32)
    dat_d = to_dev(numpy.concatenate([dt, [SENTINEL]]))
    ddat_d = to_dev(numpy.concatenate([ddt, [SENTINEL]])) if with_ddata else None
    flags = to_dev(numpy.zeros(2), numpy.int32)
    assert cu.lib.gp_csr_sort_rows(n, dptr(to_dev(ip, numpy.int32)), dptr(ind_d), dptr(dat_d), dptr(ddat_d), dptr(flags),
                                   cu.stream_ptr()) == 0
    rowid = numpy.repeat(numpy.arange(n), numpy.diff(ip))
    p = numpy.lexsort((ix, rowid))
    got_i, got_d = to_host(ind_d), to_host(dat_d)
    assert (got_i[:nnz] == ix[p]).all() and got_i[nnz] == ISENTINEL
    assert_equal(got_d[:nnz], dt[p], 'sorted data')
    assert_untouched(got_d[nnz:], numpy.array([SENTINEL]), 'data past the end')
    if with_ddata:
        got_dd = to_host(ddat_d)
        assert_equal(got_dd[:nnz], ddt[p], 'sorted ddata')
        assert_untouched(got_dd[nnz:], numpy.array([SENTINEL]), 'ddata past the end')


# ---------------------------------------------------------------------------------------------------- probes
@gpu
@pytest.mark.parametrize('n,B,seed,offset,mapped', [(1, 5, 0, 0, False), (1000, 1, 3, 0, False), (1000, 3, 11, 7, True),
                                                    (777, 16, 0xDEADBEEFCAFEF00D, 12345678901, True),
                                                    (64, 32, 1, 3, False)])
def test_rademacher_equals_the_oracle(cu, n, B, seed, offset, mapped):
    from oracle import slq
    rng = numpy.random.default_rng(n + B)
    N = 3 * n if mapped else n
    row_map = rng.choice(N, size=n, replace=False).astype(numpy.int32) if mapped else None
    V = with_sentinel_rows((n, B))
    assert cu.lib.gp_rademacher(dptr(V), n, B, seed, offset, dptr(to_dev(row_map, numpy.int32) if mapped else None),
                                cu.stream_ptr()) == 0
    ref = slq.rademacher(N, B, seed, offset)
    want = ref[row_map] if mapped else ref
    got = to_host(V)
    assert_equal(got[:n], want, 'rademacher')
    assert_untouched(got[n:], numpy.full((1, B), SENTINEL), 'rademacher: row past n')
    assert cu.lib.gp_rademacher(dptr(V), n, 0, seed, offset, None, cu.stream_ptr()) == -1


# ------------------------------------------------------------------------------------------------- reductions
@gpu
@pytest.mark.parametrize('B', WIDTHS)
def test_col_dot_exact(cu, B):
    """out[c] = sum_i X[i][c] Y[i][c] bit for bit, n from 1 to beyond one pass of the 592 x 256 threads of the
    first stage (each thread then sums several elements); B = 3 and 64 return -1"""
    torch = _torch()
    rng = numpy.random.default_rng(B)
    span = 592 * 256 // B
    for n in (1, 3, 600, span - 1, span, span + 1, 3 * span + 17):
        X, Y = int_block(rng, (n, B)), int_block(rng, (n, B))
        ws = torch.empty(cu.lib.gp_krylov_workspace_bytes(n, B) // 8 + 1, dtype=torch.float64, device='cuda')
        out = to_dev(numpy.full(B + 1, SENTINEL))
        assert cu.lib.gp_col_dot(None, dptr(to_dev(X)), dptr(to_dev(Y)), n, B, dptr(out), dptr(ws), cu.stream_ptr()) == 0
        got = to_host(out)
        assert_equal(got[:B], (X * Y).sum(axis=0), 'col_dot n=%d B=%d' % (n, B))
        assert_untouched(got[B:], numpy.array([SENTINEL]), 'col_dot past B')
    Xd = to_dev(numpy.zeros((4, 64)))
    for bad in (3, 64):
        assert cu.lib.gp_col_dot(None, dptr(Xd), dptr(Xd), 4, bad, dptr(Xd), dptr(Xd), cu.stream_ptr()) == -1


@gpu
def test_gram_skinny_exact(cu):
    """out[a B + b] = sum_i X[i][a] Y[i][b] for every B from 1 to 16, n around the 64-row tile and around 1184 CTAs x 64
    rows (one tile per CTA, then a second, partial one); B = 17 returns -1"""
    torch = _torch()
    rng = numpy.random.default_rng(6)
    sizes = [1, 63, 64, 65, 1184 * 64 - 1, 1184 * 64, 1184 * 64 + 1, 2 * 1184 * 64 + 3]
    Xa, Ya = int_block(rng, (max(sizes), 16)), int_block(rng, (max(sizes), 16))
    ws = torch.empty(cu.lib.gp_gram_workspace_bytes(16) // 8, dtype=torch.float64, device='cuda')
    for B in range(1, 17):
        for n in sizes:
            X, Y = numpy.ascontiguousarray(Xa[:n, :B]), numpy.ascontiguousarray(Ya[:n, :B])
            out = to_dev(numpy.full(B * B + 1, SENTINEL))
            assert cu.lib.gp_gram_skinny(dptr(to_dev(X)), dptr(to_dev(Y)), n, B, dptr(out), dptr(ws), cu.stream_ptr()) == 0
            got = to_host(out)
            assert_equal(got[:B * B], (X.T @ Y).ravel(), 'gram n=%d B=%d' % (n, B))
            assert_untouched(got[B * B:], numpy.array([SENTINEL]), 'gram past B^2')
    Xd = to_dev(numpy.zeros((4, 17)))
    assert cu.lib.gp_gram_skinny(dptr(Xd), dptr(Xd), 4, 17, dptr(Xd), dptr(ws), cu.stream_ptr()) == -1


# -------------------------------------------------------------------------------------------------- block combine
@gpu
@pytest.mark.parametrize('B', WIDTHS)
def test_block_combine_exact(cu, B):
    """X[i][c] = sum_j coef[j][c] basis[j][i][c] bit for bit for degrees 1, 7, 256 (one chunk of coefficients in shared
    memory), 257 and 300 (two chunks), odd n; nothing written past n B. B = 3 (and any width that is not a power of two
    up to 32) and m = 0 return -1 before any launch."""
    rng = numpy.random.default_rng(B)
    for n in (1, 1001):
        for m in (1, 7, 256, 257, 300):
            basis = int_block(rng, (m, n, B))
            coef = rng.integers(-64, 65, size=(m, B)) / 16.0
            X = with_sentinel_rows((n, B))
            assert cu.lib.gp_block_combine(dptr(to_dev(basis)), n, B, m, dptr(to_dev(coef)), dptr(X), cu.stream_ptr()) == 0
            got = to_host(X)
            assert_equal(got[:n], numpy.einsum('jc,jic->ic', coef, basis), 'block_combine n=%d B=%d m=%d' % (n, B, m))
            assert_untouched(got[n:], numpy.full((1, B), SENTINEL), 'block_combine past n B')
    Z = to_dev(numpy.zeros(64 * 8))
    for bad in (3, 5, 7, 12, 33, 64):
        assert cu.lib.gp_block_combine(dptr(Z), 4, bad, 2, dptr(Z), dptr(Z), cu.stream_ptr()) == -1
    assert cu.lib.gp_block_combine(dptr(Z), 4, B, 0, dptr(Z), dptr(Z), cu.stream_ptr()) == -1


# ------------------------------------------------------------------------------------------------------- Lanczos
def run_lanczos(cu, S, eta, V, m, blocked, keep_basis=True):
    """gp_lanczos (CSR) or gp_bcsr_lanczos (row blocks, identity order) on the symmetric scipy matrix S; alpha, beta and
    basis carry one sentinel row / vector past m. Returns alpha, beta (m x B), basis (m x n x B) or None."""
    torch = _torch()
    n, B = V.shape
    ip, ix, dt = S.indptr.astype(numpy.int32), S.indices.astype(numpy.int32), S.data.astype(numpy.float64)
    A = DevCSR(ip, ix, dt)
    alpha, beta = with_sentinel_rows((m, B)), with_sentinel_rows((m, B))
    basis = with_sentinel_rows((m, n, B)) if keep_basis else None
    ws = torch.empty(cu.lib.gp_krylov_workspace_bytes(n, B) // 8 + 1, dtype=torch.float64, device='cuda')
    Vd = to_dev(V)
    if blocked:
        bptr, bidx, bvals, _ = build_blocks(cu, A, None, False)['dev']
        rc = cu.lib.gp_bcsr_lanczos(None, dptr(bptr), dptr(bidx), dptr(bvals), n, eta, dptr(Vd), B, m, dptr(alpha),
                                    dptr(beta), dptr(basis), dptr(ws), cu.stream_ptr())
    else:
        rc = cu.lib.gp_lanczos(dptr(A.indptr), dptr(A.indices), dptr(A.data), n, eta, dptr(Vd), B, m, dptr(alpha),
                               dptr(beta), dptr(basis), dptr(ws), cu.stream_ptr())
    assert rc == 0
    a, b = to_host(alpha), to_host(beta)
    assert_untouched(a[m:], numpy.full((1, B), SENTINEL), 'alpha past m')
    assert_untouched(b[m:], numpy.full((1, B), SENTINEL), 'beta past m')
    U = None
    if keep_basis:
        U = to_host(basis)
        assert_untouched(U[m:], numpy.full((1, n, B), SENTINEL), 'basis past m')
        U = U[:m]
    return a[:m], b[:m], U


def check_lanczos_relations(S, eta, V, a, b, U, m):
    """Local checks of every step on the device's own numbers, each within the rounding of that step:
      u_0 = v; alpha_j = q_j^T (S + eta I) q_j and beta_j = ||u_{j+1}|| for the kept vectors u_j = beta_{j-1} q_j;
      the three-term relation s_j (S + eta I) u_j - alpha_j s_j u_j - beta_{j-1} s_{j-1} u_{j-1} - u_{j+1} = 0
    A sum of L products carries at most gamma_L = L u of the sum of their magnitudes. The device's and the host's
    evaluations each do that, plus 6 more roundings per element (eta term, scale, two axpys, subtraction): c = 2 (L + 8)
    with L the longest row (relation) or n (dot products, norms)."""
    n = V.shape[0]
    Aeta = S + eta * scipy.sparse.identity(n, format='csr')
    absA = abs(Aeta)
    L = int(numpy.diff(S.indptr).max()) + 1
    cr, cd = 2 * (L + 8) * EPS, 2 * (n + 8) * EPS
    assert_equal(U[0], V, 'u_0 = v')
    s = numpy.empty((m, V.shape[1]))
    s[0] = 1.0 / numpy.sqrt((V * V).sum(axis=0))
    s[1:] = 1.0 / b[:m - 1]
    for j in range(m):
        q = U[j] * s[j]
        Aq = Aeta @ q
        assert (numpy.abs(a[j] - (q * Aq).sum(axis=0)) <= cd * (numpy.abs(q) * (absA @ numpy.abs(q))).sum(axis=0)).all(), j
        if j + 1 < m:
            nrm = numpy.sqrt((U[j + 1] ** 2).sum(axis=0))
            assert (numpy.abs(b[j] - nrm) <= cd * nrm).all(), j
            prev = U[j - 1] * (b[j - 1] * s[j - 1]) if j > 0 else 0.0
            r = Aeta @ U[j] * s[j] - (a[j] * s[j]) * U[j] - prev - U[j + 1]
            mag = (absA @ numpy.abs(U[j])) * s[j] + numpy.abs(a[j] * s[j] * U[j]) + numpy.abs(prev) + numpy.abs(U[j + 1])
            assert (numpy.abs(r) <= cr * mag).all(), j


@gpu
@pytest.mark.parametrize('B', [1, 16, 32])
def test_lanczos_csr_and_row_blocked(cu, B):
    """m = 10 steps on a sparse symmetric integer matrix (n = 3001, a ragged last block): the local relations of every
    step, near-orthogonal kept vectors, and alpha / beta against the NumPy recurrence; the CSR and row-blocked runs agree"""
    rng = numpy.random.default_rng(B)
    n, m, eta = 3001, 10, 0.75
    S, _ = sym_int_matrix(rng, n, 6)
    V = int_block(rng, (n, B))
    V[0] = 1.0                                                  # no zero column
    ra, rb = lanczos_ref(S, eta, V, m)
    normA = float(abs(S).sum(axis=1).max()) + abs(eta)
    runs = [run_lanczos(cu, S, eta, V, m, blocked) for blocked in (False, True)]
    for a, b, U in runs:
        check_lanczos_relations(S, eta, V, a, b, U, m)
        # no Ritz value has converged in 10 steps (beta_j >= ||A|| / 16 below), so by Paige's theorem the kept vectors
        # stay orthogonal to the level of the local errors amplified by ||A|| / min beta: 16 x 2 (n + 8) u x m
        assert (b[:m - 1] >= normA / 16).all()
        for c in range(B):
            Q = U[:, :, c] / numpy.sqrt((U[:, :, c] ** 2).sum(axis=1))[:, None]
            assert numpy.abs(Q @ Q.T - numpy.eye(m)).max() <= 16 * 2 * (n + 8) * EPS * m
        # forward difference to the host recurrence: each step adds a local error of at most 2 (n + 8) u ||A|| and no
        # step amplifies an earlier one by more than ||A|| / min beta <= 16; over m steps: m 16 2 (n + 8) u ||A||
        tol = m * 16 * 2 * (n + 8) * EPS * normA
        assert numpy.abs(a - ra).max() <= tol and numpy.abs(b - rb).max() <= tol
    assert numpy.abs(runs[0][0] - runs[1][0]).max() <= 2 * tol and numpy.abs(runs[0][1] - runs[1][1]).max() <= 2 * tol


@gpu
@pytest.mark.parametrize('blocked', [False, True])
def test_lanczos_full_degree_and_breakdown(cu, blocked):
    """m = n on a dense 12 x 12 matrix: the Ritz values of T are the eigenvalues of A + eta I. A diagonal matrix with 5
    distinct values: beta breaks down at step 5, the later steps stay finite, T_5 has the 5 values as Ritz values."""
    rng = numpy.random.default_rng(4 + blocked)
    Ad, n = tiny_dense_matrix(rng)
    S = scipy.sparse.csr_matrix(Ad)
    for B in (1, 32):
        V = int_block(rng, (n, B))
        V[0] = 1.0
        a, b, U = run_lanczos(cu, S, 0.5, V, n, blocked)
        check_lanczos_relations(S, 0.5, V, a, b, U, n)
        lam = numpy.linalg.eigvalsh(Ad + 0.5 * numpy.eye(n))
        normA = numpy.abs(lam).max()
        assert numpy.diff(lam).min() >= 0.5
        for c in range(B):
            # eigenvalue gaps >= 1/2 (above): with local errors of 2 (n + 8) u ||A|| per step, every Ritz value is within
            # m times that, amplified by ||A|| / gap <= 2 ||A||, of its eigenvalue
            ritz = numpy.linalg.eigvalsh(tridiag(a[:, c], b[:, c], n))
            assert numpy.abs(ritz - lam).max() <= n * 2 * (n + 8) * EPS * normA * 2 * normA, c
    D, vals = diagonal_matrix()
    n, k, m = D.shape[0], len(vals), 10
    for B in (1, 32):
        V = numpy.where(int_block(rng, (n, B)) >= 0, 1.0, -1.0)
        a, b, _ = run_lanczos(cu, D, 0.0, V, m, blocked, keep_basis=False)
        assert numpy.isfinite(a).all() and numpy.isfinite(b).all()
        # beta_{k-1} = ||u_k|| is rounding noise: k steps of local errors 2 (n + 8) u ||D||, ||D|| = 8
        assert (b[k - 1] <= k * 2 * (n + 8) * EPS * 8).all() and (b[:k - 1] >= 0.1).all()
        ra, rb = lanczos_ref(D, 0.0, V, k)
        tol = k * 2 * (n + 8) * EPS * 8 * 8
        assert numpy.abs(a[:k] - ra).max() <= tol and numpy.abs(b[:k - 1] - rb[:k - 1]).max() <= tol
        for c in range(B):
            assert numpy.abs(numpy.linalg.eigvalsh(tridiag(a[:, c], b[:, c], k)) - vals).max() <= tol


@gpu
def test_lanczos_rejects_bad_widths(cu):
    Z = to_dev(numpy.zeros(64 * 64))
    Zi = to_dev(numpy.zeros(64), numpy.int32)
    for bad in (3, 64):
        assert cu.lib.gp_lanczos(dptr(Zi), dptr(Zi), dptr(Z), 4, 0.0, dptr(Z), bad, 2, dptr(Z), dptr(Z), None, dptr(Z),
                                 cu.stream_ptr()) == -2


# ------------------------------------------------------------------------------------------------------------- CG
def run_cg(cu, S, eta, R, tol, maxiter, blocked):
    """gp_cg_solve / gp_bcsr_cg_solve (identity order); X carries a sentinel row. Returns rc, iterations, X."""
    torch = _torch()
    n, B = R.shape
    A = DevCSR(S.indptr.astype(numpy.int32), S.indices.astype(numpy.int32), S.data.astype(numpy.float64))
    X = with_sentinel_rows((n, B))
    Rd = to_dev(R)
    it = ctypes.c_int64(-1)
    ws = torch.empty(cu.lib.gp_krylov_workspace_bytes(n, B) // 8 + 1, dtype=torch.float64, device='cuda')
    if blocked:
        bptr, bidx, bvals, _ = build_blocks(cu, A, None, False)['dev']
        rc = cu.lib.gp_bcsr_cg_solve(None, dptr(bptr), dptr(bidx), dptr(bvals), n, eta, dptr(Rd), dptr(X), B, tol, maxiter,
                                     ctypes.byref(it), dptr(ws), cu.stream_ptr())
    else:
        rc = cu.lib.gp_cg_solve(dptr(A.indptr), dptr(A.indices), dptr(A.data), n, eta, dptr(Rd), dptr(X), B, tol, maxiter,
                                ctypes.byref(it), dptr(ws), cu.stream_ptr())
    Xh = to_host(X)
    assert_untouched(Xh[n:], numpy.full((1, B), SENTINEL), 'cg: row past n')
    return rc, it.value, Xh[:n]


@gpu
@pytest.mark.parametrize('blocked', [False, True])
@pytest.mark.parametrize('B', [1, 16])
def test_cg_solve_residual_and_return_codes(cu, blocked, B):
    """0 with the true residual ||b - (S + eta I) x|| <= tol ||b|| per column (a zero column stays exactly 0 and does not
    hold the others back); 1 with iters == maxiter when maxiter is too small; 2 on an indefinite S + eta I"""
    rng = numpy.random.default_rng(B + 2 * blocked)
    n, tol = 3001, 1e-10
    S0, rmax = sym_int_matrix(rng, n, 4)
    S = (S0 + (rmax + 1.0) * scipy.sparse.identity(n, format='csr')).tocsr()     # spectrum in [1, 2 rmax + 1]
    S.sort_indices()
    eta = 0.5
    R = int_block(rng, (n, B))
    R[0] = 1.0
    if B > 1:
        R[:, 5] = 0.0
    rc, iters, X = run_cg(cu, S, eta, R, tol, 2000, blocked)
    assert rc == 0 and 0 < iters < 2000
    M = S + eta * scipy.sparse.identity(n, format='csr')
    # the recurrence stops at ||r_k|| <= tol ||b||; the true residual differs from the recursive one by the rounding of
    # the updates: at most c n u (|M| |x| + |b|) per element over the iterations, c = 2 (L + 8) iters
    L = int(numpy.diff(S.indptr).max()) + 1
    gap = 2 * (L + 8) * iters * EPS * numpy.linalg.norm(abs(M) @ numpy.abs(X) + numpy.abs(R), axis=0)
    res = numpy.linalg.norm(R - M @ X, axis=0)
    assert (res <= tol * numpy.linalg.norm(R, axis=0) + gap).all(), res
    if B > 1:
        assert (X[:, 5] == 0.0).all()
    rc, iters, _ = run_cg(cu, S, eta, R, tol, 3, blocked)
    assert rc == 1 and iters == 3
    # indefinite: eta = -(rmax + 1.5) puts every diagonal entry of S + eta I at -0.5 and the spectrum on both sides of 0;
    # b = e_i gives p^T A p = -0.5 in the first iteration
    E = numpy.zeros((n, B))
    E[rng.choice(n, size=B, replace=False), numpy.arange(B)] = 1.0
    rc, iters, _ = run_cg(cu, S, -0.5 - (rmax + 1.0), E, tol, 2000, blocked)
    assert rc == 2 and 0 < iters <= 8
    for bad in (3, 64):
        assert run_cg(cu, S, eta, int_block(rng, (n, bad)), tol, 10, blocked)[0] == -2


# ----------------------------------------------------------------------------------------- the engine at m > 256
@gpu
def test_engine_lanczos_degree_above_256(cu):
    """lanczos_degree = 300: tr(Kn^-1 dK/drho) takes the kept-Lanczos branch (gp_block_combine over two chunks of
    coefficients) and agrees with separate CG solves to the tolerance of test_hutchinson_dk_reuses_the_lanczos_basis"""
    from gaussian_proc._sparse import SparseEngine, generate_sparse_correlation
    rs = numpy.random.RandomState(1)
    pts = rs.rand(3000, 2)
    Kd = generate_sparse_correlation(pts, numpy.array([0.03, 0.03]), 0.5, 0.01, device=True, with_derivative=True)
    opts = {'seed': 2, 'lanczos_degree': 300, 'min_num_samples': 32, 'max_num_samples': 32, 'cg_tol': 1e-8}
    a = SparseEngine(Kd, 'slq', dict(opts, reuse_lanczos=True))
    b = SparseEngine(Kd, 'slq', dict(opts, reuse_lanczos=False))
    ta = a.traceinv_dK(2.0)
    assert a.last_dk_solver == 'lanczos'
    tb = b.traceinv_dK(2.0)
    assert a.last_info['num_samples'] == b.last_info['num_samples'] == 32
    assert abs(ta - tb) <= 1e-6 * abs(tb)
