"""
Sparse (kernel-threshold) path: device CSR generation and the stochastic estimators behind MixedCorrelation for a
sparse K (SpMM + batched Lanczos / CG in csrc/gp_sparse.cu, csrc/gp_sparse_la.cu).

Reference behaviour restated here:
  generate_sparse_correlation  gaussian_proc/generate_correlation/_generate_sparse_correlation.pyx:472-594
  logdet / traceinv (slq, hutchinson), solve (CG, tol 1e-6)
                               gaussian_proc/_mixed_correlation/mixed_correlation.py:193-209,263-268;
                               _linear_solver.py:49-68
imate (absent, unpinned dependency) is followed through its documented estimator: Rademacher probes, Lanczos
quadrature, min/max number of samples, relative error tolerance at a confidence level (SURVEY 8c). parity unpinned:
the reference's own 'slq' branches are dead code (mixed_correlation.py:141,207,266); the confidence band is checked
against exact values from the oracle in tests/test_gpu_sparse.py.
"""

import ctypes

import numpy
import scipy.linalg
import scipy.sparse
import scipy.special

from . import _device as dev
from ._device import lib, check

__all__ = ['DeviceCSR', 'DeviceRowBlocks', 'SparseEngine', 'generate_sparse_correlation', 'generate_sparse_operator',
           'estimate_kernel_threshold']

# imate's documented defaults for the stochastic estimators (SURVEY 8c)
DEFAULTS = dict(min_num_samples=10, max_num_samples=50, error_rtol=1e-2, error_atol=None, confidence_level=0.95,
                lanczos_degree=20, seed=0, batch=16, cg_tol=1e-6, cg_maxiter=2000, reuse_lanczos=True, overlap=True,
                shift_reuse=True, solve_degree=None, eager_rhs_basis=False)


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


_RHS_DEVICE_CACHE = []      # [(key, device block, X, z)]: see SparseEngine._rhs_block


def estimate_kernel_threshold(matrix_size, dimension, density, correlation_scale, nu):
    """tau for the requested density (_generate_sparse_correlation.pyx:294-413); ValueError when density*n < 1."""
    tau = ctypes.c_double()
    scale = dev.host_f64(correlation_scale)
    rc = lib.gp_kernel_threshold(int(matrix_size), int(dimension), float(density), dev.host_ptr(scale), float(nu),
                                 ctypes.byref(tau))
    if rc == -10:
        raise ValueError(
            'Adjacency: %0.2f. Correlation matrix will become identity since kernel radius is less than grid size. '
            'To increase adjacency, consider increasing density or correlation_scale.' % (density * matrix_size))
    check(rc, 'gp_kernel_threshold')
    return tau.value


class DeviceCSR(object):
    """CSR (int32 indptr / int32 indices, float64 data) resident on the GPU; `ddata` optionally holds d/d(rho) of every
    stored entry on the same pattern. The device generator leaves the rows in generation order (``sorted_rows`` False):
    the device operators do not need more; ``canonicalize()`` sorts every row by column - the reference's canonical CSR,
    bit-exact pattern - and is called by ``to_scipy()`` / whenever a consumer needs sorted rows."""

    def __init__(self, n, indptr, indices, data, ddata=None, kernel_threshold=None, order=None, sorted_rows=True):
        self.n = int(n)
        self.indptr, self.indices, self.data, self.ddata = indptr, indices, data, ddata
        self.kernel_threshold = kernel_threshold
        self.order = order      # optional spatially local ordering of the rows (device int32), see SparseEngine
        self.sorted_rows = bool(sorted_rows)
        self.dscale = None      # (device points, scale, nu): dK/d scale[k] per dimension, built with the row blocks

    def canonicalize(self):
        """sort every row by column index, in place (no-op when already sorted)"""
        if not self.sorted_rows:
            torch = dev.torch
            flags = torch.zeros(2, dtype=torch.int32, device='cuda')
            rc = lib.gp_csr_sort_rows(self.n, _p(self.indptr), _p(self.indices), _p(self.data),
                                      _p(self.ddata) if self.ddata is not None else None, _p(flags), dev.stream_ptr())
            check(rc, 'gp_csr_sort_rows')
            self.sorted_rows = True
        return self

    @property
    def shape(self):
        return (self.n, self.n)

    @property
    def nnz(self):
        return int(self.data.shape[0])

    @classmethod
    def from_scipy(cls, K):
        torch = dev.require_cuda()
        K = scipy.sparse.csr_matrix(K)
        K.sort_indices()
        if K.shape[0] != K.shape[1]:
            raise ValueError('K should be a square matrix.')
        return cls(K.shape[0], torch.from_numpy(K.indptr.astype(numpy.int32)).cuda(),
                   torch.from_numpy(K.indices.astype(numpy.int32)).cuda(),
                   torch.from_numpy(K.data.astype(numpy.float64)).cuda())

    def to_scipy(self):
        self.canonicalize()
        return scipy.sparse.csr_matrix((self.data.cpu().numpy(), self.indices.cpu().numpy(), self.indptr.cpu().numpy()),
                                       shape=(self.n, self.n))


class DeviceRowBlocks(object):
    """A sparse correlation matrix generated DIRECTLY as the operator the likelihood works on: 16-row blocks of the
    spatially ordered matrix (bptr, bidx, bvals[, bdvals] in the SpMM's fragment order, csrc/gp_sparse_la.cu), without a CSR.
    Rows [first_row, last_row) of the ordered operator are present (everything, or the slab of one GPU)."""

    R = 16

    def __init__(self, n, bptr, bidx, bvals, bdvals, order, inv_order, nnz, kernel_threshold, first_row, last_row,
                 row_slab=None):
        self.n = int(n)
        self.bptr, self.bidx, self.bvals, self.bdvals = bptr, bidx, bvals, bdvals
        self.ddata = bdvals                    # (engines ask `K.ddata is not None` for "carries dK/drho")
        self.order, self.inv_order = order, inv_order
        self.nnz = int(nnz)                    # entries in the pattern of the rows present
        self.kernel_threshold = kernel_threshold
        self.first_row, self.last_row = int(first_row), int(last_row)
        self.row_slab = row_slab
        self.sorted_rows = True
        self.encoded = None                    # set by the row-slab engine once the columns carry (owner, local row)
        self.dscale = None                     # (device points, scale, nu): dK/d scale[k] per dimension (anisotropic scale)
        self.bdvals_dims = None                # their d streams, computed by the first engine (before any column encoding)

    @property
    def shape(self):
        return (self.n, self.n)

    def to_scipy(self):
        """scipy.sparse.csr_matrix of the rows present, original row / column order (host reconstruction; rare path)"""
        if self.encoded is not None:
            raise ValueError('the columns of this operator were re-encoded for the row-slab engine')
        R = self.R
        bptr = self.bptr.cpu().numpy()
        bidx = self.bidx.cpu().numpy().astype(numpy.int64)
        vals = self.bvals.cpu().numpy().reshape(-1, 2, 8, 4)       # [group of 4 slots][fragment][row in fragment][slot in group]
        order = self.order.cpu().numpy().astype(numpy.int64)
        nrb = bptr.size - 1
        slot_block = numpy.repeat(numpy.arange(nrb), numpy.diff(bptr))
        v = vals.transpose(0, 3, 1, 2).reshape(-1, R)               # [slot][row of the block]
        rows_op = self.first_row + slot_block[:, None] * R + numpy.arange(R)[None, :]
        keep = (v != 0.0) & (rows_op < self.last_row)
        rows = order[numpy.minimum(rows_op, self.n - 1)][keep]
        cols = order[numpy.broadcast_to(bidx[:, None], v.shape)[keep]]
        M = scipy.sparse.csr_matrix((v[keep], (rows, cols)), shape=(self.n, self.n))
        M.sort_indices()
        return M


_POINTS_DEVICE_CACHE = []      # [(key, points array, device points, order, position)]


def _device_points(points):
    """(device copy, spatial order, position in the order) of a host point set. None of the three depends on the
    hyper-parameters, and an optimiser or a sweep generates K for the same points at every step: the last two point sets
    are kept (keyed by content, _device.host_key; arrays that cannot be written to are recognised without a digest).
    order = stable sort of the Hilbert / Z-order keys over the bounding box (own kernels, csrc/gp_index.cu): the
    deterministic, spatially local row order of the row-blocked operator; position = its inverse permutation."""
    torch = dev.torch
    key = dev.host_key(points)
    for ent in _POINTS_DEVICE_CACHE:
        if ent[0] == key:
            return ent[2], ent[3], ent[4]
    n, d = points.shape
    s = dev.stream_ptr()
    dpts = torch.from_numpy(numpy.array(points)).cuda()
    box = numpy.empty(2 * d)
    box_ws = torch.empty(148 * 2 * d + 2 * d, dtype=torch.float64, device='cuda')
    check(lib.gp_points_bbox(_p(dpts), n, d, dev.host_ptr(box), _p(box_ws), s), 'gp_points_bbox')
    lo, hi = dev.host_f64(box[:d]), dev.host_f64(box[d:])
    keys = torch.empty(n, dtype=torch.int64, device='cuda')
    check(lib.gp_spatial_keys(_p(dpts), n, d, dev.host_ptr(lo), dev.host_ptr(hi), _p(keys), s), 'gp_spatial_keys')
    order = torch.empty(n, dtype=torch.int32, device='cuda')
    sort_ws = torch.empty(lib.gp_sort_workspace_bytes(n) // 8 + 8, dtype=torch.float64, device='cuda')
    check(lib.gp_sort_keys_u64(_p(keys), n, 64, _p(order), _p(sort_ws), s), 'gp_sort_keys_u64')
    pos = torch.empty(n, dtype=torch.int32, device='cuda')
    check(lib.gp_inverse_permutation(_p(order), n, _p(pos), s), 'gp_inverse_permutation')
    _POINTS_DEVICE_CACHE.append((key, points, dpts, order, pos))
    del _POINTS_DEVICE_CACHE[:-2]
    return dpts, order, pos


def generate_sparse_correlation(points, correlation_scale, nu, density, verbose=False, device=False,
                                with_derivative=False, kernel_threshold=None, sort_rows=None, row_slab=None):
    """Device generator behind the reference's generate_sparse_correlation. Returns scipy.sparse.csr_matrix (or a
    DeviceCSR when ``device``). ``sort_rows``: canonical (column-sorted) rows right away; default: yes for the SciPy
    result, deferred (DeviceCSR.canonicalize) for a device handle.
    ``row_slab`` = (rank, world) (device handle only): generate only this rank's slab of rows of the spatially ordered
    operator (gaussian_proc/_slab.py); the other rows of the handle stay empty.
    ``with_derivative``: dK/drho on the pattern (``ddata``) for an isotropic scale; for an anisotropic one the device handle
    records (device points, scale, nu) instead and the engine builds dK/d scale[k] per dimension with its row blocks (the
    SciPy result cannot carry them: ValueError)."""
    sort_rows = (not device) if sort_rows is None else bool(sort_rows)
    torch = dev.require_cuda()
    points = numpy.ascontiguousarray(points, dtype=numpy.float64)
    scale = dev.host_f64(correlation_scale)
    n, d = points.shape
    tau = estimate_kernel_threshold(n, d, density, scale, nu) if kernel_threshold is None else float(kernel_threshold)
    per_dim = with_derivative and not numpy.all(scale == scale[0])
    if per_dim and not device:
        raise ValueError('d/d(correlation_scale) of an anisotropic correlation_scale needs device=True (the derivatives '
                         'are carried by the device operator).')
    if row_slab is not None and not device:
        raise ValueError('row_slab needs device=True (a slab is not a complete matrix).')
    s = dev.stream_ptr()
    dpts, order, pos = _device_points(points)
    rows = (None, 0, 0)              # (row filter, first, last): every row
    if row_slab is not None:
        from ._slab import slab_geometry
        rank, world = int(row_slab[0]), int(row_slab[1])
        _, first, last = slab_geometry(n, world, rank)
        rows = (_p(pos), first, last)
    ws = torch.empty(lib.gp_sparse_workspace_bytes(n, d) // 8 + 8, dtype=torch.float64, device='cuda')
    indptr = torch.empty(n + 1, dtype=torch.int32, device='cuda')
    nnz = ctypes.c_int64()
    check(lib.gp_matern_sparse_count(_p(dpts), dev.host_ptr(points), n, d, dev.host_ptr(scale), float(nu), tau, _p(ws),
                                     _p(indptr), ctypes.byref(nnz), *rows, s), 'gp_matern_sparse_count')
    indices = torch.empty(nnz.value, dtype=torch.int32, device='cuda')
    data = torch.empty(nnz.value, dtype=torch.float64, device='cuda')
    ddata = torch.empty(nnz.value, dtype=torch.float64, device='cuda') if with_derivative and not per_dim else None
    check(lib.gp_matern_sparse_fill(_p(dpts), dev.host_ptr(points), n, d, dev.host_ptr(scale), float(nu), tau, _p(ws),
                                    _p(indptr), _p(indices), _p(data), _p(ddata) if ddata is not None else None,
                                    1 if sort_rows else 0, *rows, s), 'gp_matern_sparse_fill')
    K = DeviceCSR(n, indptr, indices, data, ddata, kernel_threshold=tau, order=order, sorted_rows=sort_rows)
    K.inv_order = pos
    if per_dim:
        K.dscale = (dpts, scale, float(nu))
    if row_slab is not None:
        K.row_slab = (rank, world, first, last)       # only these rows of the ordered operator are present
    if verbose:
        print('Generated sparse correlation matrix using kernel threshold: %0.4f and sparse density: %0.2e.'
              % (tau, K.nnz / float(n) ** 2))
    return K if device else K.to_scipy()


def generate_sparse_operator(points, correlation_scale, nu, density, with_derivative=False, kernel_threshold=None,
                             row_slab=None, verbose=False):
    """The sparse correlation matrix of generate_sparse_correlation as a device OPERATOR for MixedCorrelation / SparseEngine:
    the row blocks are generated directly from the cell lists (csrc/gp_sparse.cu, sparse_blocks_kernel; same kernel
    arithmetic and pattern rule, no CSR in between), about half the time of CSR generation + block build. Falls back to that
    path (returns a DeviceCSR) for a matrix with entries inside the 8-ulp borderline band of the threshold, which the
    reference's rule decides in host arithmetic. ``row_slab`` = (rank, world): only this rank's slab (gaussian_proc/_slab.py).
    ``with_derivative`` with an anisotropic scale: per-dimension derivatives, as in generate_sparse_correlation."""
    torch = dev.require_cuda()
    points = numpy.ascontiguousarray(points, dtype=numpy.float64)
    scale = dev.host_f64(correlation_scale)
    n, d = points.shape
    tau = estimate_kernel_threshold(n, d, density, scale, nu) if kernel_threshold is None else float(kernel_threshold)
    per_dim = with_derivative and not numpy.all(scale == scale[0])
    s = dev.stream_ptr()
    dpts, order, pos = _device_points(points)
    first, last, slab = 0, n, None
    if row_slab is not None:
        from ._slab import slab_geometry
        rank, world = int(row_slab[0]), int(row_slab[1])
        _, first, last = slab_geometry(n, world, rank)
        slab = (rank, world, first, last)
    ws = torch.empty(lib.gp_sparse_workspace_bytes(n, d) // 8 + 8, dtype=torch.float64, device='cuda')
    nrb = (last - first + 15) // 16
    nblk = torch.empty(nrb, dtype=torch.int32, device='cuda')
    stats = (ctypes.c_int64 * 2)()
    rc = lib.gp_matern_blocks_count(_p(dpts), n, d, dev.host_ptr(scale), float(nu), tau, _p(ws), _p(order), _p(pos), first, last,
                                    _p(nblk), stats, s)
    if rc == 3:
        return generate_sparse_correlation(points, correlation_scale, nu, density, verbose=verbose, device=True,
                                           with_derivative=with_derivative, kernel_threshold=tau, row_slab=row_slab)
    check(rc, 'gp_matern_blocks_count')
    bptr = torch.empty(nrb + 1, dtype=torch.int64, device='cuda')
    check(lib.gp_scan_counts(_p(nblk), nrb, _p(bptr), s), 'gp_scan_counts')
    total = int(bptr[-1].item())
    bidx = torch.empty(total, dtype=torch.int32, device='cuda')
    bvals = torch.empty(total * 16, dtype=torch.float64, device='cuda')
    bdvals = torch.empty(total * 16, dtype=torch.float64, device='cuda') if with_derivative and not per_dim else None
    check(lib.gp_matern_blocks_fill(_p(dpts), n, d, dev.host_ptr(scale), float(nu), tau, _p(ws), _p(order), _p(pos), first, last,
                                    _p(bptr), _p(bidx), _p(bvals), _p(bdvals) if bdvals is not None else None, s),
          'gp_matern_blocks_fill')
    K = DeviceRowBlocks(n, bptr, bidx, bvals, bdvals, order, pos, stats[0], tau, first, last, row_slab=slab)
    if per_dim:
        K.dscale = (dpts, scale, float(nu))
    if verbose:
        print('Generated sparse correlation operator using kernel threshold: %0.4f and sparse density: %0.2e.'
              % (tau, K.nnz / float(n) / float(last - first)))
    return K


def lanczos_quadrature(alpha, beta, funcs, return_size=False):
    """Gauss quadrature of v^T f(A) v / ||v||^2 from the Lanczos tridiagonal: sum_k tau_k^2 f(theta_k) with theta the
    Ritz values and tau the first components of the Ritz vectors. A beta ~ 0 truncates the recurrence (invariant
    subspace reached)."""
    m = len(alpha)
    for j in range(m - 1):
        if not (beta[j] > 1e-12 * max(abs(alpha[0]), 1.0)):
            m = j + 1
            break
    theta, Y = scipy.linalg.eigh_tridiagonal(alpha[:m], beta[:m - 1]) if m > 1 else (alpha[:1], numpy.ones((1, 1)))
    w = Y[0, :] ** 2
    res = [float(numpy.sum(w * f(theta))) for f in funcs], float(theta.min())
    return res + (m,) if return_size else res


def lanczos_block_quadrature(alpha, beta, vnorm=None):
    """Batched host part of SLQ for a block of B Lanczos runs (alpha, beta: m x B): one stacked symmetric eigensolve of
    the B tridiagonals gives, per column, the Gauss quadratures of [log, 1/x, 1/x^2], the smallest Ritz value and - with
    ``vnorm`` (||v|| per column, or a scalar) - the coefficients of x = A^-1 v in the unnormalised Lanczos vectors
    (u_0 = v, u_j = beta_{j-1} q_j) together with the relative residual beta_m |y_m| of that Lanczos (= CG) solution.
    A column whose recurrence broke down (beta ~ 0: invariant subspace) is truncated there.
    Returns quad (B x 3), tmin (B), coef (m x B) or None, resid (B) or None."""
    m, B = alpha.shape
    ks = numpy.full(B, m, dtype=int)
    for c in range(B):
        small = numpy.nonzero(~(beta[:m - 1, c] > 1e-12 * max(abs(alpha[0, c]), 1.0)))[0]
        if small.size:
            ks[c] = small[0] + 1
    quad, tmin = numpy.empty((B, 3)), numpy.empty(B)
    want = vnorm is not None
    coef = numpy.zeros((m, B)) if want else None
    resid = numpy.zeros(B) if want else None
    vn = numpy.broadcast_to(numpy.asarray(vnorm, dtype=float), (B,)) if want else None
    for k in numpy.unique(ks):
        cols = numpy.nonzero(ks == k)[0]
        T = numpy.zeros((cols.size, k, k))
        idx = numpy.arange(k)
        T[:, idx, idx] = alpha[:k, cols].T
        if k > 1:
            T[:, idx[:-1], idx[1:]] = beta[:k - 1, cols].T
            T[:, idx[1:], idx[:-1]] = beta[:k - 1, cols].T
        theta, Y = numpy.linalg.eigh(T)
        w = Y[:, 0, :] ** 2
        with numpy.errstate(invalid='ignore', divide='ignore'):
            quad[cols, 0] = numpy.sum(w * numpy.log(theta), axis=1)
            quad[cols, 1] = numpy.sum(w / theta, axis=1)
            quad[cols, 2] = numpy.sum(w / theta ** 2, axis=1)
            tmin[cols] = theta.min(axis=1)
            if want:
                y = numpy.einsum('bij,bj->bi', Y, Y[:, 0, :] / theta)          # T^-1 e_1
                scale = numpy.empty((cols.size, k))
                scale[:, 0] = 1.0 / vn[cols]
                if k > 1:
                    scale[:, 1:] = 1.0 / beta[:k - 1, cols].T
                coef[:k, cols] = (vn[cols][:, None] * y * scale).T
                resid[cols] = numpy.abs(beta[k - 1, cols] * y[:, k - 1]) if k == m else 0.0
    return quad, tmin, coef, resid


class SparseEngine(object):
    """Stochastic logdet / traceinv and CG solves for K + eta I with K in device CSR or row blocks. On one GPU the engine
    works on every row; the row-slab engine (gaussian_proc/_slab.py) is this engine on one slab of rows with a peer."""

    peer = peer_side = None        # row-slab engine: this rank's PeerArena and the one of the prefetch stream

    def __init__(self, K, imate_method='slq', imate_options=None, probe_range=None):
        dev.require_cuda()
        if not isinstance(K, (DeviceCSR, DeviceRowBlocks)):
            K = DeviceCSR.from_scipy(K)
        self.K = K
        self.n = K.n
        if self.peer is None:      # one GPU: the rows [first_row, last_row) of the operator are all of them
            self.first_row, self.last_row = 0, K.n
        self.rows = self.last_row - self.first_row      # rows of the vectors this engine works on
        self.method = imate_method
        self.opt = dict(DEFAULTS)
        self.opt.update(imate_options or {})
        self._ws = {}
        self._krylov = {}          # shift-invariant Lanczos runs, see _probe_krylov / solve_rhs_block
        self._rhs_etas = {}
        self._slq_cache = {}
        self.last_info = {}
        # multi-GPU: (rank, world) -> this engine evaluates its slice of every round of probes; see _run_estimator
        self.probe_range = probe_range
        # A K with a spatial order (from the device generators) is worked on as the ROW-BLOCKED form of the symmetrically
        # permuted matrix P K P^T (rows in that order): 16 consecutive rows share one column list, so one gathered row of
        # the probe block serves 16 rows of K and four such block-columns are one DMMA.8x8x4 (csrc/gp_sparse_la.cu).
        # Results do not depend on the permutation: probes are hashed with ORIGINAL row ids. A K without an order (e.g.
        # from SciPy) stays plain CSR in the original order.
        self.order = self.inv_order = None
        self.R = 1                 # rows per block of the operator in use: 16 row-blocked, 1 plain CSR
        self.blocked = None
        self.dims = None           # (d, 16 * blocks) per-dimension derivative streams of an anisotropic scale
        self.last_dscale = None    # rows [tr(Kn^-1 dK_k), Q_k] of the last fused call (layout of DenseEngine.last_dscale)
        if K.order is not None:
            self._build_blocked(K)

    def _build_blocked(self, K):
        """The 16-row blocks of the rows [first_row, last_row) of the ordered operator: those of a DeviceRowBlocks as
        they are, else built from the CSR. With a peer the block-columns are encoded as (owner rank, row in its slab)."""
        torch = dev.torch
        n, r0, r1, R = self.n, self.first_row, self.last_row, 16
        s = dev.stream_ptr()
        my_rows = K.order[r0:r1]   # original ids of this engine's rows (contiguous int32 view)
        share = 1                  # 1 / the share of K's entries that lie in the rows built
        if isinstance(K, DeviceRowBlocks):         # generated as row blocks: nothing to build
            if self.peer is None and ((K.first_row, K.last_row) != (0, n) or K.encoded is not None):
                raise ValueError('this operator holds one slab of rows (or its columns were encoded for the row-slab engine): '
                                 'use the row-slab engine (row_slabs=True).')
            bptr, bidx, bvals, bdvals, inv, encoded = K.bptr, K.bidx, K.bvals, K.bdvals, K.inv_order, K.encoded
        else:
            inv = getattr(K, 'inv_order', None)
            if inv is None:
                inv = torch.empty(n, dtype=torch.int32, device='cuda')
                check(lib.gp_inverse_permutation(_p(K.order), n, _p(inv), s), 'gp_inverse_permutation')
            nrb = (self.rows + R - 1) // R
            nblk = torch.empty(nrb, dtype=torch.int32, device='cuda')
            flag = torch.zeros(1, dtype=torch.int32, device='cuda')
            check(lib.gp_bcsr_count(self.rows, _p(my_rows), _p(inv), _p(K.indptr), _p(K.indices), _p(nblk), _p(flag), s),
                  'gp_bcsr_count')
            if not K.sorted_rows and int(flag.item()) != 0:
                # some row block is too wide for the hash path: its binary-search fallback needs canonical rows
                K.canonicalize()
                check(lib.gp_bcsr_count(self.rows, _p(my_rows), _p(inv), _p(K.indptr), _p(K.indices), _p(nblk), _p(flag), s),
                      'gp_bcsr_count')
            bptr = torch.empty(nrb + 1, dtype=torch.int64, device='cuda')
            check(lib.gp_scan_counts(_p(nblk), nrb, _p(bptr), s), 'gp_scan_counts')
            total = int(bptr[-1].item())
            bidx = torch.empty(total, dtype=torch.int32, device='cuda')
            bvals = torch.empty(total * R, dtype=torch.float64, device='cuda')
            bdvals = torch.empty(total * R, dtype=torch.float64, device='cuda') if K.ddata is not None else None
            check(lib.gp_bcsr_fill(self.rows, _p(my_rows), _p(inv), _p(K.indptr), _p(K.indices), _p(K.data),
                                   _p(K.ddata) if K.ddata is not None else None, _p(bptr), total, _p(bidx), _p(bvals),
                                   _p(bdvals) if bdvals is not None else None, s), 'gp_bcsr_fill')
            encoded = None
            if self.peer is not None and getattr(K, 'row_slab', None) is None:
                share = self.world     # a handle with every row, of which this slab is built
        total = bidx.numel()
        if K.dscale is not None:
            # dK/d scale[k] on the blocks just built or generated, while the columns are still operator positions; a
            # generated handle keeps them, so a second engine on it (its columns possibly encoded since) reuses them
            dims = K.bdvals_dims if isinstance(K, DeviceRowBlocks) else None
            if dims is None:
                dpts, scale, nu = K.dscale
                d = scale.size
                dims = torch.empty((d, total * R), dtype=torch.float64, device='cuda')
                check(lib.gp_bcsr_dscale_fill(_p(bptr), _p(bidx), _p(bvals), total, r0, self.rows, _p(K.order), _p(dpts), n, d,
                                              dev.host_ptr(scale), nu, _p(dims), s), 'gp_bcsr_dscale_fill')
                if isinstance(K, DeviceRowBlocks):
                    K.bdvals_dims = dims
            self.dims = dims
        if self.peer is not None:
            if encoded is None:
                halo = (ctypes.c_int64 * 2)()   # block-columns whose row of X lives on another rank, and the distinct rows among them
                ws = torch.empty(2 + (n + 63) // 64 + 1, dtype=torch.int64, device='cuda')
                check(lib.gp_slab_encode_columns(_p(bidx), total, self.slab, self.rank, n, halo, _p(ws), s),
                      'gp_slab_encode_columns')
                encoded = (self.slab, self.rank, int(halo[0]), int(halo[1]))
                if isinstance(K, DeviceRowBlocks):
                    K.encoded = encoded        # its bidx now carries the encoding
            elif encoded[:2] != (self.slab, self.rank):
                raise ValueError('this operator was encoded for another slab geometry')
            self.halo_blocks, self.halo_rows, self.total_blocks = encoded[2], encoded[3], total
            self.halo_fraction = self.halo_blocks / float(max(total, 1))
        self.R = R
        self.blocked = (bptr, bidx, bvals, bdvals)
        self.fill_ratio = total * R / float(max(K.nnz, 1)) * share     # stored values per original nonzero (>= 1)
        self.order, self.inv_order = K.order, inv            # device int32 row maps of to_op / from_op
        self._my_rows = my_rows

    # ---- plumbing ----------------------------------------------------------------------------------------------
    def _workspace(self, B, side=False):
        """Krylov workspace for column blocks of width B; ``side``: the separate one of the prefetch stream (a Lanczos
        run there may overlap a CG / Lanczos run of the same width on the main stream)."""
        torch = dev.torch
        key = ('side', B) if side else B
        if key not in self._ws:
            self._ws[key] = torch.empty(lib.gp_krylov_workspace_bytes(self.rows, B) // 8 + 8, dtype=torch.float64, device='cuda')
        return self._ws[key]

    def _peer_ctx(self, side=False):
        """the peer argument of the row-blocked drivers: NULL on one GPU"""
        arena = self.peer_side if side else self.peer
        return arena.ctx if arena is not None else None

    def spmm(self, eta, X_dev, derivative=False, dim=None):
        """(K + eta I) X, (dK/drho + eta I) X with ``derivative``, or (dK/d scale[dim] + eta I) X with ``dim`` (an
        anisotropic scale's per-dimension streams), in OPERATOR space (rows in self.order when the operator is permuted)"""
        torch = dev.torch
        B = X_dev.shape[1]
        X_dev = X_dev.contiguous()
        Y = torch.empty_like(X_dev)
        if dim is not None:
            self._derivative_streams(required=True)
        if self.blocked is not None:
            bptr, bidx, bvals, bdvals = self.blocked
            vals = self.dims[dim] if dim is not None else (bdvals if derivative else bvals)
            check(lib.gp_bcsr_spmm(self._peer_ctx(), _p(bptr), _p(bidx), _p(vals), self.rows,
                                   float(eta), _p(X_dev), B, _p(Y), dev.stream_ptr()), 'gp_bcsr_spmm')
        else:
            K = self.K
            check(lib.gp_csr_spmm(_p(K.indptr), _p(K.indices), _p(K.ddata if derivative else K.data), self.n, float(eta),
                                  _p(X_dev), B, _p(Y), dev.stream_ptr()), 'gp_csr_spmm')
        return Y

    def _derivative_streams(self, required=False):
        """number of derivative operators K carries: 1 (dK/drho of an isotropic scale, K.ddata), d (dK/d scale[k] of an
        anisotropic one, self.dims) or 0; ``required``: ValueError instead of 0"""
        if self.K.dscale is not None:
            if self.dims is not None:
                return self.dims.shape[0]
            if required:
                raise ValueError('d/d(correlation_scale) per dimension needs the spatially ordered device operator of '
                                 'generate_sparse_operator / generate_sparse_correlation(..., device=True); a plain CSR '
                                 'or a SciPy matrix cannot carry it.')
            return 0
        if self.K.ddata is None:
            if required:
                raise ValueError('d/d(correlation_scale) needs a DeviceCSR generated with with_derivative=True')
            return 0
        return 1

    def _dk(self, X_dev, k):
        """dK_k X: the derivative operator k of _derivative_streams (k = 0 alone: dK/drho)"""
        if self.dims is not None:
            return self.spmm(0.0, X_dev, dim=k)
        return self.spmm(0.0, X_dev, derivative=True)

    def to_op(self, X_dev):
        """this engine's rows, in operator order, of an (n x B) block given in the caller's row order"""
        if self.order is None:
            return X_dev
        X_dev = X_dev.contiguous()
        B = X_dev.numel() // self.n
        Y = dev.torch.empty((self.rows, B), dtype=dev.torch.float64, device='cuda')
        check(lib.gp_gather_rows(_p(X_dev), _p(self._my_rows), self.rows, B, _p(Y), dev.stream_ptr()), 'gp_gather_rows')
        return Y

    def from_op(self, X_dev):
        """the (n x B) block in the caller's row order from operator order"""
        if self.order is None:
            return X_dev
        X_dev = X_dev.contiguous()
        Y = dev.torch.empty_like(X_dev)
        check(lib.gp_gather_rows(_p(X_dev), _p(self.inv_order), self.n, X_dev.numel() // self.n, _p(Y), dev.stream_ptr()),
              'gp_gather_rows')
        return Y

    def probes(self, first, B, out=None):
        torch = dev.torch
        V = torch.empty((self.rows, B), dtype=torch.float64, device='cuda') if out is None else out
        rmap = self._my_rows if self.order is not None else None
        check(lib.gp_rademacher(_p(V), self.rows, B, int(self.opt['seed']), int(first), _p(rmap) if rmap is not None else None,
                                dev.stream_ptr()), 'gp_rademacher')
        return V

    # ---- SLQ -----------------------------------------------------------------------------------------------------
    def _lanczos(self, eta, V, m, basis=None):
        alpha, beta = self._lanczos_launch(eta, V, m, basis)
        return alpha.cpu().numpy(), beta.cpu().numpy()

    def _lanczos_launch(self, eta, V, m, basis=None, alpha=None, beta=None, side=False):
        """enqueues the batched Lanczos run on torch's current stream; returns the device (alpha, beta)"""
        torch = dev.torch
        B = V.shape[1]
        alpha = torch.empty((m, B), dtype=torch.float64, device='cuda') if alpha is None else alpha
        beta = torch.empty((m, B), dtype=torch.float64, device='cuda') if beta is None else beta
        bp = _p(basis) if basis is not None else None
        if self.blocked is not None:
            bptr, bidx, bvals, _ = self.blocked
            check(lib.gp_bcsr_lanczos(self._peer_ctx(side), _p(bptr), _p(bidx), _p(bvals), self.rows, float(eta), _p(V), B, m,
                                      _p(alpha), _p(beta), bp, _p(self._workspace(B, side)), dev.stream_ptr()),
                  'gp_bcsr_lanczos')
        else:
            K = self.K
            check(lib.gp_lanczos(_p(K.indptr), _p(K.indices), _p(K.data), self.n, float(eta), _p(V), B, m, _p(alpha),
                                 _p(beta), bp, _p(self._workspace(B, side)), dev.stream_ptr()), 'gp_lanczos')
        return alpha, beta

    def _first_chunk(self):
        """(first probe id, width) of the first block of probes this rank evaluates in an estimator run"""
        o = self.opt
        B, hi = int(o['batch']), int(o['max_num_samples'])
        rank, world = self.probe_range if self.probe_range is not None else (0, 1)
        nb = min(B, hi)
        per = (nb + world - 1) // world
        my0 = rank * per
        chunks = self._chunks(my0, max(0, min(nb, my0 + per) - my0), B)
        return chunks[0] if chunks else None

    def prefetch_slq(self, eta):
        """Enqueues the first SLQ block of probes at `eta` on a side stream and returns at once, so that the batched CG
        for [X z] that follows on the main stream (HBM-bound, B = 8) overlaps the Lanczos run (L1-bound, B = 16).
        _slq_samples picks the result up."""
        torch = dev.torch
        if float(eta) in self._slq_cache or getattr(self, '_prefetched', None) is not None:
            return
        chunk = self._first_chunk()
        if chunk is None:
            return
        first, B = chunk
        if ('probes', first, B) in self._krylov and bool(self.opt.get('shift_reuse', True)):
            return                                 # already served by a kept Lanczos run
        m = int(self.opt['lanczos_degree'])
        with_dk = self._derivative_streams() > 0 and bool(self.opt.get('reuse_lanczos', True))
        if not hasattr(self, '_side_stream'):
            self._side_stream = torch.cuda.Stream()
        # every buffer is allocated on the main stream; the side stream only runs kernels on them
        V = torch.empty((self.rows, B), dtype=torch.float64, device='cuda')
        alpha = torch.empty((m, B), dtype=torch.float64, device='cuda')
        beta = torch.empty((m, B), dtype=torch.float64, device='cuda')
        basis = self._new_basis(m, B) if with_dk else None
        self._workspace(B, side=True)
        cur = torch.cuda.current_stream()
        self._side_stream.wait_stream(cur)
        with torch.cuda.stream(self._side_stream):
            self.probes(first, B, out=V)
            self._lanczos_launch(eta, V, m, basis, alpha, beta, side=True)
        self._prefetched = (float(eta), first, B, with_dk, V, alpha, beta, basis)

    # The Krylov space of K + eta I does not depend on eta and the Lanczos tridiagonal only shifts: T(eta) = T(eta_ref) +
    # (eta - eta_ref) I (the reference builds imate.AffineMatrixFunction(K) for this, mixed_correlation.py:44,141,207,266).
    # One batched Lanczos run per block of probes (and one per right-hand-side block) therefore serves EVERY eta asked of
    # this operator: new quadratures on the host, new solutions x(eta) = ||v|| Q (T + d I)^-1 e_1 by one pass over the kept
    # vectors. A root find or a sweep over eta at fixed rho pays the SpMMs once.
    KRYLOV_CACHE_BYTES = 32 << 30      # kept Lanczos vectors per operator (beyond it blocks are recomputed per eta)

    def _krylov_bytes(self):
        return sum(e['basis'].numel() * 8 for e in self._krylov.values() if e.get('basis') is not None)

    def _probe_krylov(self, eta, first, B, keep_basis):
        """(entry, shift) for the block of probes first .. first+B-1: the cached Lanczos run if there is one (shift =
        eta - eta_ref), else a new run at eta (picked up from the side-stream prefetch when it matches)."""
        torch = dev.torch
        m = int(self.opt['lanczos_degree'])
        key = ('probes', first, B)
        ent = self._krylov.get(key)
        if ent is not None and (ent['basis'] is not None or not keep_basis) and bool(self.opt.get('shift_reuse', True)):
            return ent, float(eta) - ent['eta_ref']
        pre = getattr(self, '_prefetched', None)
        self._prefetched = None
        if pre is not None and pre[:4] == (float(eta), first, B, keep_basis):
            V, alpha, beta, basis = pre[4:]
            torch.cuda.current_stream().wait_stream(self._side_stream)
            a, b = alpha.cpu().numpy(), beta.cpu().numpy()
        else:
            if pre is not None:
                self._side_stream.synchronize()        # an unused prefetch still owns the workspace
            V = self.probes(first, B)
            basis = self._new_basis(m, B) if keep_basis else None
            a, b = self._lanczos(eta, V, m, basis)
        ent = {'eta_ref': float(eta), 'a': a, 'b': b, 'basis': basis, 'V': V if keep_basis else None, 'Wd': None}
        if self._krylov_bytes() + (basis.numel() * 8 if basis is not None else 0) <= self.KRYLOV_CACHE_BYTES:
            self._krylov[key] = ent
        return ent, 0.0

    def _new_basis(self, m, B):
        return dev.torch.empty((m, self.rows, B), dtype=dev.torch.float64, device='cuda')

    def _slq_samples(self, eta, first, B, with_dk=0):
        """Per-probe quadratures [log, 1/x, 1/x^2] * n for probes first .. first+B-1. With ``with_dk`` derivative
        operators (_derivative_streams) one more column each: the Hutchinson sample v^T Kn^-1 dK_k v with Kn^-1 v taken
        from the SAME Lanczos run (x = ||v|| Q T^-1 e_1, the Lanczos form of CG) when its residual beta_k |y_k| meets the
        CG tolerance, else from a batched CG solve."""
        torch = dev.torch
        m = int(self.opt['lanczos_degree'])
        nd = int(with_dk)
        ent, shift = self._probe_krylov(eta, first, B, nd > 0)
        a, b = ent['a'] + shift, ent['b']
        out = numpy.empty((B, 3 + nd))
        vnorm = numpy.sqrt(float(self.n))          # Rademacher probes
        quad, tmin, coef, res = lanczos_block_quadrature(a, b, vnorm if nd else None)
        if not (tmin.min() > 0):
            raise numpy.linalg.LinAlgError(
                'K + eta*I (eta=%g) is not positive definite: Lanczos found a Ritz value %.3e. The thresholded '
                'Matern matrix is indefinite; use a larger eta (reference: _generate_sparse_correlation.pyx:516-523).'
                % (eta, tmin.min()))
        out[:, :3] = quad * self.n
        resid = float(res.max()) if nd else 0.0
        if nd:
            V = ent['V'] if ent['V'] is not None else self.probes(first, B)
            if ent['Wd'] is None:
                ent['Wd'] = [self._dk(V, k) for k in range(nd)]      # dK_k v does not depend on eta either
            if resid <= float(self.opt['cg_tol']):
                U = torch.empty_like(V)
                cd = torch.from_numpy(coef).cuda()
                check(lib.gp_block_combine(_p(ent['basis']), self.rows, B, m, _p(cd), _p(U), dev.stream_ptr()),
                      'gp_block_combine')
                self.last_dk_solver = 'lanczos'
            else:
                U = self.solve_dev(eta, V.clone())
                self.last_dk_solver = 'cg'
            for k in range(nd):
                out[:, 3 + k] = self.col_dot(U, ent['Wd'][k])
        return out

    def solve_rhs_block(self, eta, Rop, key, refs=None):
        """S = (K + eta I)^-1 R for the (cached) right-hand-side block of the likelihood, operator space. The first eta
        asked of this operator is solved by batched CG; from the second DISTINCT eta on (from the first with the option
        ``eager_rhs_basis``, which sweeps and the root finder set: they know more eta will follow), one batched Lanczos
        run on R (degree ~ twice the CG iteration count, 48 when unknown) is kept and every eta is served from it (shift
        invariance), falling back to CG for an eta whose Lanczos residual misses the CG tolerance."""
        torch = dev.torch
        eta = float(eta)
        if not bool(self.opt.get('shift_reuse', True)):
            return self.solve_dev(eta, Rop.clone())
        B = Rop.shape[1]
        ent = self._krylov.get(('rhs', key))
        if ent is None:
            seen = self._rhs_etas.setdefault(key, (set(), refs))[0]      # refs keep X, z alive: the ids stay unique
            seen.add(eta)
            if len(seen) < 2 and not bool(self.opt.get('eager_rhs_basis', False)):
                return self.solve_dev(eta, Rop.clone())
            m = int(self.opt.get('solve_degree') or min(128, max(int(self.opt['lanczos_degree']),
                                                                   2 * int(getattr(self, 'last_cg_iterations', 24)))))
            basis = self._new_basis(m, B)
            a, b = self._lanczos(eta, Rop, m, basis)
            norms = numpy.sqrt(numpy.maximum(self.col_dot(Rop, Rop), 0.0))
            ent = {'eta_ref': eta, 'a': a, 'b': b, 'basis': basis, 'norms': norms, 'm': m, 'refs': refs}
            if self._krylov_bytes() + basis.numel() * 8 <= self.KRYLOV_CACHE_BYTES:
                self._krylov[('rhs', key)] = ent
        a, b, m = ent['a'] + (eta - ent['eta_ref']), ent['b'], ent['m']
        live = numpy.nonzero(ent['norms'] > 0.0)[0]                 # zero (padding) columns stay zero
        coef = numpy.zeros((m, B))
        _, tmin, cf, res = lanczos_block_quadrature(a[:, live], b[:, live], ent['norms'][live])
        coef[:, live] = cf
        resid = float(res.max()) if (live.size and tmin.min() > 0) else numpy.inf
        if not (resid <= float(self.opt['cg_tol'])):
            self.last_rhs_solver = 'cg'
            return self.solve_dev(eta, Rop.clone())
        S = torch.empty_like(Rop)
        cd = torch.from_numpy(coef).cuda()
        check(lib.gp_block_combine(_p(ent['basis']), self.rows, B, m, _p(cd), _p(S), dev.stream_ptr()), 'gp_block_combine')
        self.last_rhs_solver = 'lanczos'
        return S

    @staticmethod
    def _chunks(first, count, batch):
        """split [first, first + count) into contiguous power-of-two blocks of width <= batch"""
        out = []
        while count > 0:
            w = 1
            while w * 2 <= min(count, batch):
                w *= 2
            out.append((first, w))
            first += w
            count -= w
        return out

    def _run_estimator(self, sample_fn, ncols, check_cols=None, state=None):
        """imate-style sampling loop: rounds of probes until every estimated quantity (the first ``check_cols`` columns)
        satisfies z * s / sqrt(N) <= max(atol, rtol |mean|) (after min_num_samples) or max_num_samples is reached.
        ``state`` = (samples, first) continues an earlier run (its convergence is tested before sampling more).
        Multi-GPU: each round's probe ids are cut into `world` contiguous slices, one per rank; the running
        (count, sum, sum of squares) are all-reduced, so every rank takes the same stopping decision. Probe ids, not
        ranks, seed the random signs: the union of the samples is the same set for any number of GPUs.
        Returns mean, half_width, N, (samples, first)."""
        o = self.opt
        B = int(o['batch'])
        zc = float(numpy.sqrt(2.0) * scipy.special.erfinv(float(o['confidence_level'])))
        lo, hi = int(o['min_num_samples']), int(o['max_num_samples'])
        rank, world = self.probe_range if self.probe_range is not None else (0, 1)
        cc = ncols if check_cols is None else check_cols
        samples, first = (numpy.empty((0, ncols)), 0) if state is None else state
        atol = o['error_atol'] if o['error_atol'] is not None else 0.0

        failure = []      # a breakdown on THIS rank (indefinite K + eta I: non-positive Ritz value / CG breakdown)

        def reduce_or_raise():
            """all-reduce of the running sums together with a 'some rank failed' flag: a local breakdown must not leave
            the other ranks blocked in the collective - every rank raises after it."""
            N, mean, sd, failed = self._reduce(samples, bool(failure))
            if failed:
                raise failure[0] if failure else numpy.linalg.LinAlgError(
                    'K + eta*I is not positive definite (breakdown reported by another rank of the probe split).')
            return N, mean, sd

        def converged():
            N, mean, sd = reduce_or_raise()
            if N < lo:
                return False
            half = zc * sd / numpy.sqrt(N)
            return bool(numpy.all(half[:cc] <= numpy.maximum(atol, o['error_rtol'] * numpy.abs(mean[:cc]))))

        done = (first > 0) and converged()
        while first < hi and not done:
            nb = min(B, hi - first)          # the round size does not depend on the rank count: same samples, same stopping decision
            per = (nb + world - 1) // world
            my0 = first + rank * per
            my1 = min(first + nb, my0 + per)
            for (f, w) in self._chunks(my0, max(0, my1 - my0), B):
                if failure:
                    break
                try:
                    samples = numpy.vstack([samples, sample_fn(f, w)])
                except numpy.linalg.LinAlgError as exc:
                    if world == 1:
                        raise
                    failure.append(exc)
            first += nb
            done = converged()
        N, mean, sd = reduce_or_raise()
        half = zc * sd / numpy.sqrt(max(N, 1))
        return mean, half, int(N), (samples, first)

    def _reduce(self, samples, failed=False):
        """(N, mean, unbiased std, any rank failed) over all ranks: all-reduce of (count, failure flag, sum, sum of
        squares) per quantity."""
        cnt = numpy.array([samples.shape[0], 1.0 if failed else 0.0], dtype=float)
        s1 = samples.sum(axis=0)
        s2 = (samples ** 2).sum(axis=0)
        if self.probe_range is not None and self.probe_range[1] > 1:
            from ._distributed import allreduce_sum
            packed = allreduce_sum(numpy.concatenate([cnt, s1, s2]))
            k = s1.size
            cnt, s1, s2 = packed[:2], packed[2:2 + k], packed[2 + k:]
        N = cnt[0]
        mean = s1 / max(N, 1)
        var = numpy.maximum(s2 - N * mean ** 2, 0.0) / max(N - 1, 1)
        return N, mean, numpy.sqrt(var), bool(cnt[1] > 0)

    def _slq(self, eta):
        """SLQ estimates [logdet, tr Kn^-1, tr Kn^-2] at eta (cached). When the matrix carries dK/drho (or dK/d scale[k]
        per dimension) the same Lanczos runs also yield the Hutchinson samples of tr(Kn^-1 dK_k) (kept for traceinv_dK;
        they do not influence the stopping decision here)."""
        key = float(eta)
        if key not in self._slq_cache:
            nd = self._derivative_streams() if bool(self.opt.get('reuse_lanczos', True)) else 0
            mean, half, N, state = self._run_estimator(
                lambda first, width: self._slq_samples(eta, first, width, nd), 3 + nd, check_cols=3)
            self._slq_cache = {key: (mean[:3], half[:3], N)}
            self._dk_state = {key: (state[0][:, 3:].copy(), state[1])} if nd else {}
        mean, half, N = self._slq_cache[key]
        self.last_info = {'num_samples': N, 'half_width': half, 'confidence_level': self.opt['confidence_level'],
                          'lanczos_degree': self.opt['lanczos_degree']}
        return mean

    def logdet(self, eta):
        """SLQ estimate of logdet(K + eta I) (also for method 'hutchinson', SURVEY Q6)."""
        return float(self._slq(eta)[0])

    def traceinv(self, eta, exponent=1):
        if exponent not in (1, 2):
            raise ValueError('traceinv on the sparse engine supports exponent 1 and 2.')
        if self.method == 'slq' or exponent == 2:
            return float(self._slq(eta)[exponent])

        def fn(first, width):   # hutchinson: v^T Kn^-1 v with CG solves
            V = self.probes(first, width)
            U = self.solve_dev(eta, V.clone())
            return self.col_dot(U, V).reshape(-1, 1)
        mean, half, N, _ = self._run_estimator(fn, 1)
        self.last_info = {'num_samples': N, 'half_width': half}
        return float(mean[0])

    def _dk_samples(self, eta, first, width):
        """Hutchinson samples (Kn^-1 v)^T (dK_k v) of probes first .. first+width-1, one column per derivative operator"""
        nd = self._derivative_streams(required=True)
        if bool(self.opt.get('reuse_lanczos', True)):
            # through the (kept, shift-invariant) Lanczos run of this probe block: reused for every later eta
            return self._slq_samples(eta, first, width, nd)[:, 3:]
        V = self.probes(first, width)
        U = self.solve_dev(eta, V.clone())
        return numpy.stack([self.col_dot(U, self._dk(V, k)) for k in range(nd)], axis=1)

    def traceinv_dK(self, eta):
        """Hutchinson estimate of tr((K + eta I)^-1 dK/d rho): mean over probes of (Kn^-1 v)^T (dK v); for an anisotropic
        scale the array of tr(Kn^-1 dK/d scale[k]), k < d, from the same probes. Samples that the SLQ run at this eta
        already produced (same probe ids, Kn^-1 v from its Lanczos basis) are used first; further rounds, if its own
        stopping rule (on every column) asks for them, go through the same kept-Lanczos path (CG when the Lanczos
        residual misses the tolerance or with reuse_lanczos=False)."""
        nd = self._derivative_streams(required=True)
        state = getattr(self, '_dk_state', {}).get(float(eta))
        mean, half, N, _ = self._run_estimator(lambda first, width: self._dk_samples(eta, first, width), nd, state=state)
        self.last_info = {'num_samples': N, 'half_width': half}
        return mean.copy() if self.dims is not None else float(mean[0])

    # ---- CG ------------------------------------------------------------------------------------------------------
    def col_dot(self, X, Y):
        torch = dev.torch
        B = X.shape[1]
        out = torch.empty(32, dtype=torch.float64, device='cuda')
        check(lib.gp_col_dot(self._peer_ctx(), _p(X), _p(Y), self.rows, B, _p(out), _p(self._workspace(B)), dev.stream_ptr()),
              'gp_col_dot')
        return out[:B].cpu().numpy()

    def solve_dev(self, eta, R_dev):
        """(K + eta I)^-1 R for a device block (n x B, B a power of two <= 32); R_dev is overwritten."""
        torch = dev.torch
        B = R_dev.shape[1]
        X = torch.empty_like(R_dev)
        it = ctypes.c_int64()
        if self.blocked is not None:
            bptr, bidx, bvals, _ = self.blocked
            rc = lib.gp_bcsr_cg_solve(self._peer_ctx(), _p(bptr), _p(bidx), _p(bvals), self.rows, float(eta), _p(R_dev), _p(X), B,
                                      float(self.opt['cg_tol']), int(self.opt['cg_maxiter']), ctypes.byref(it),
                                      _p(self._workspace(B)), dev.stream_ptr())
        else:
            K = self.K
            rc = lib.gp_cg_solve(_p(K.indptr), _p(K.indices), _p(K.data), self.n, float(eta), _p(R_dev), _p(X), B,
                                 float(self.opt['cg_tol']), int(self.opt['cg_maxiter']), ctypes.byref(it),
                                 _p(self._workspace(B)), dev.stream_ptr())
        check(rc, 'gp_cg_solve')
        self.last_cg_iterations = it.value
        if rc == 2:
            raise numpy.linalg.LinAlgError(
                'K + eta*I (eta=%g) is not positive definite (CG met p^T A p <= 0). The thresholded Matern matrix is '
                'indefinite; use a larger eta (reference: _generate_sparse_correlation.pyx:516-523).' % eta)
        if rc == 1:
            raise numpy.linalg.LinAlgError('CG did not converge in %d iterations (eta=%g)' % (it.value, eta))
        return X

    def _max_block(self):
        """widest column block handed to the SpMM: the 16 x 1 row-blocked kernel is tuned for B <= 16"""
        return 16 if self.blocked is not None else 32

    def solve(self, eta, Y):
        """mixed_correlation.py:280-299 for sparse K: CG per column with rtol 1e-6 (batched on the device)."""
        torch = dev.torch
        Y = numpy.asarray(Y, dtype=numpy.float64)
        vec = (Y.ndim == 1)
        Y2 = Y.reshape(self.n, -1)
        out = numpy.empty_like(Y2)
        k = Y2.shape[1]
        W = self._max_block()
        for c0 in range(0, k, W):
            blk = Y2[:, c0:c0 + W]
            B = 1
            while B < blk.shape[1]:
                B *= 2
            R = torch.zeros((self.n, B), dtype=torch.float64, device='cuda')
            R[:, :blk.shape[1]].copy_(torch.from_numpy(numpy.ascontiguousarray(blk)))
            X = self.from_op(self.solve_dev(eta, self.to_op(R)))
            out[:, c0:c0 + blk.shape[1]] = X[:, :blk.shape[1]].cpu().numpy()
        return out[:, 0] if vec else out

    def matmul(self, X):
        torch = dev.torch
        X = numpy.asarray(X, dtype=numpy.float64)
        vec = (X.ndim == 1)
        X2 = X.reshape(self.n, -1)
        k = X2.shape[1]
        B = 1
        while B < k:
            B *= 2
        W = self._max_block()
        if B > W:
            return numpy.hstack([self.matmul(X2[:, c:c + W]) for c in range(0, k, W)])
        Xd = torch.zeros((self.n, B), dtype=torch.float64, device='cuda')
        Xd[:, :k].copy_(torch.from_numpy(numpy.ascontiguousarray(X2)))
        res = self.from_op(self.spmm(0.0, self.to_op(Xd)))[:, :k].cpu().numpy()
        return res[:, 0] if vec else res

    # ---- fused likelihood ingredients -------------------------------------------------------------------------
    def gram(self, X_dev, Y_dev):
        """X^T Y (B x B, host) of two n x B device blocks (with a peer: summed over the ranks' slabs)."""
        torch = dev.torch
        B = X_dev.shape[1]
        if '_gram' not in self._ws:
            self._ws['_gram'] = torch.empty(lib.gp_gram_workspace_bytes(16) // 8, dtype=torch.float64, device='cuda')
        out = torch.empty(B * B, dtype=torch.float64, device='cuda')
        s = dev.stream_ptr()
        check(lib.gp_gram_skinny(_p(X_dev), _p(Y_dev), self.rows, B, _p(out), _p(self._ws['_gram']), s), 'gp_gram_skinny')
        if self.peer is not None:
            check(lib.gp_peer_allreduce(self.peer.ctx, _p(out), B * B, s), 'gp_peer_allreduce')
        return out.cpu().numpy().reshape(B, B)

    def _rhs_block(self, X, z, key=None):
        """[X z] as an operator-space device block, zero padded to a power-of-two width. The device copy in the original
        row order is cached per (X, z) objects across engines (an optimiser builds a new operator for every rho but
        keeps X and z); the operator-space permutation of it is cached per engine."""
        torch = dev.torch
        if key is None:
            key = (dev.host_key(X), dev.host_key(z))
        if getattr(self, '_rhs_cache', None) is not None and self._rhs_cache[0] == key:
            return self._rhs_cache[1]
        Rd = None
        for ent in _RHS_DEVICE_CACHE:
            if ent[0] == key and ent[1].shape[0] == self.n:
                Rd = ent[1]
        if Rd is None:
            X2 = numpy.asarray(X, dtype=float)
            p = X2.shape[1] + 1
            B = 1
            while B < p:
                B *= 2
            if B > 16:
                raise ValueError('the sparse likelihood evaluation supports at most 15 basis functions.')
            R = numpy.zeros((self.n, B))
            R[:, :p - 1] = X2
            R[:, p - 1] = numpy.asarray(z, dtype=float)
            Rd = torch.from_numpy(R).cuda()
            _RHS_DEVICE_CACHE.append((key, Rd, X, z))       # X, z kept alive so the ids stay unique
            del _RHS_DEVICE_CACHE[:-2]
        Rop = self.to_op(Rd)
        self._rhs_cache = (key, Rop, X, z)
        return Rop

    def fused(self, eta, X, z, traceinv=True, drho=True, cubic=False):
        """Everything log-likelihood + gradient need at one eta, in the layout of the dense evaluator's out[]
        (csrc/gp_loglik.cu): [logdet Kn, tr Kn^-1, tr Kn^-2, tr(Kn^-1 dK/drho), info, -, -, -, G, H, Q] with R = [X z],
        S = Kn^-1 R (batched CG, the reference's tol 1e-6), G = R^T S, H = S^T S, Q = S^T dK S; the traces are the
        stochastic estimates (SLQ / Hutchinson) of this engine. Reference formulas: _direct_likelihood.py:113-150,
        _profile_likelihood.py:104-130. For an anisotropic scale the d/d scale[k] pieces are the rows
        [tr(Kn^-1 dK_k), Q_k] of self.last_dscale (out[3] and Q stay 0), as DenseEngine does."""
        n, m = X.shape
        p = m + 1
        key = (dev.host_key(X), dev.host_key(z))          # ONE content fingerprint per evaluation
        Rd = self._rhs_block(X, z, key)
        if bool(self.opt.get('overlap', True)) and (self.method == 'slq' or drho):
            self.prefetch_slq(eta)
        S = self.solve_rhs_block(eta, Rd, key, refs=(X, z))
        out = numpy.zeros(8 + 4 * p * p)
        out[8:8 + p * p] = self.gram(Rd, S)[:p, :p].ravel()
        out[8 + p * p:8 + 2 * p * p] = self.gram(S, S)[:p, :p].ravel()
        self.last_dscale = None
        dscale = None
        if drho:
            nd = self._derivative_streams(required=True)
            if self.dims is not None:
                # anisotropic scale: rows [tr(Kn^-1 dK_k), Q_k = S^T dK_k S] per dimension, as DenseEngine.last_dscale
                dscale = numpy.zeros((nd, 1 + p * p))
                for k in range(nd):
                    dscale[k, 1:] = self.gram(S, self._dk(S, k))[:p, :p].ravel()
            else:
                D = self.spmm(0.0, S, derivative=True)
                out[8 + 2 * p * p:8 + 3 * p * p] = self.gram(S, D)[:p, :p].ravel()
        if cubic:
            # third moments T3 = S^T Kn^-1 S (Hessian / second eta-derivative): one more batched CG on S
            V2 = self.solve_dev(eta, S.clone())
            out[8 + 3 * p * p:8 + 4 * p * p] = self.gram(S, V2)[:p, :p].ravel()
        out[0] = self.logdet(eta)
        if traceinv or drho:
            out[1] = self.traceinv(eta)
            out[2] = self.traceinv(eta, exponent=2)
        if drho:
            if dscale is not None:
                dscale[:, 0] = self.traceinv_dK(eta)
                self.last_dscale = dscale
            else:
                out[3] = self.traceinv_dK(eta)
        return out

    def trace_K(self):
        """(tr K, tr K^2 = sum of squared entries) of the stored symmetric matrix (rare path: host reduction)."""
        Kh = self.K.to_scipy()
        return float(Kh.diagonal().sum()), float((Kh.data ** 2).sum())
