"""The log-likelihood gradient with respect to each entry of an anisotropic correlation scale on the sparse path: the
per-dimension derivative streams of the row-blocked operator (gp_bcsr_dscale_fill), the d Hutchinson columns of the
estimators, the rows [tr(Kn^-1 dK_k), Q_k] of SparseEngine.fused and the gradient arrays of the likelihoods.

The first two tests need no GPU (argument checks in a child process shown no device; a compile for sm_100a); the others
are marked gpu."""

import json
import os
import re
import shutil
import subprocess
import sys
import tempfile

import numpy
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'gaussian-process-param-estimation_b200')

CHILD = r'''
import ctypes, json, math, sys
sys.path.insert(0, %r)
from gaussian_proc import _device as dev
lib, null = dev.lib, ctypes.c_void_p(None)
a = ctypes.c_void_p(1 << 20)                       # a 16-byte aligned fake device pointer


def call(scale, nu, d=2, row_first=0, bptr=a, points=a):
    sc = (ctypes.c_double * 2)(*scale)
    return lib.gp_bcsr_dscale_fill(bptr, a, a, 100, row_first, 40, a, points, 1000, d, sc, nu, a, null)


good = [0.1, 0.2]                                   # anisotropic: accepted
r = {
    'zero': call([0.1, 0.0], 2.5), 'zero_first': call([0.0, 0.1], 0.5), 'negative': call([0.1, -0.1], 1.5),
    'nan': call([0.1, math.nan], 2.5), 'nan_general_nu': call([math.nan, 0.1], 0.7),
    'nu0': call(good, 0.0), 'nu_neg': call(good, -1.0),
    'null_bptr': call(good, 2.5, bptr=null), 'null_points': call(good, 2.5, points=null),
    'd9': call(good, 2.5, d=9), 'd0': call(good, 2.5, d=0), 'row_first8': call(good, 2.5, row_first=8),
}
r['launches'] = lib.gp_launch_count()
print(json.dumps(r))
''' % PKG


def test_dscale_fill_checks_its_arguments_before_any_work():
    res = subprocess.run([sys.executable, '-c', CHILD], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    r = json.loads(res.stdout.strip().splitlines()[-1])
    for k in ('zero', 'zero_first', 'negative', 'nan', 'nan_general_nu'):
        assert r[k] == -3, (k, r[k])
    assert r['nu0'] == -5 and r['nu_neg'] == -5
    for k in ('null_bptr', 'null_points', 'd9', 'd0', 'row_first8'):
        assert r[k] == -1, (k, r[k])
    assert r['launches'] == 0


def test_dscale_kernel_compiles_for_sm100a_without_spills():
    """Compile result (not a run): every instantiation of bcsr_dscale_kernel (five nu branches, d = 2 compiled in and d at
    run time) keeps its values in registers."""
    nvcc = os.environ.get('NVCC') or shutil.which('nvcc') or '/usr/local/cuda/bin/nvcc'
    src = os.path.join(PKG, 'csrc', 'gp_sparse.cu')
    with tempfile.TemporaryDirectory() as tmp:
        res = subprocess.run([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-std=c++17', '-Xcompiler', '-fPIC',
                              '-fmad=false', '-Xptxas', '-v', '-c', src, '-o', os.path.join(tmp, 'gp_sparse.o')],
                             capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stderr[-3000:]
    blocks = re.split(r"Compiling entry function '", res.stderr)
    ours = [b for b in blocks if b.startswith('_Z18bcsr_dscale_kernel')]
    assert len(ours) == 10, len(ours)
    for b in ours:
        m = re.search(r'(\d+) bytes spill stores, (\d+) bytes spill loads', b)
        assert m and m.group(1) == '0' and m.group(2) == '0', b[:400]


# ------------------------------------------------------------------------------------------------------ GPU helpers
def _unpack(t):
    """bvals-layout values (one 16-row block-column after the other) as [slot][row of the block]"""
    return t.cpu().numpy().reshape(-1, 2, 8, 4).transpose(0, 3, 1, 2).reshape(-1, 16)


def _dense_streams(eng):
    """(pattern, [dK_k]) of the engine's row blocks as dense n x n matrices in the original order, and whether every
    stream is exactly 0 where bvals is 0"""
    bptr, bidx, bvals, _ = eng.blocked
    n = eng.n
    bptr = bptr.cpu().numpy()
    bidx = bidx.cpu().numpy().astype(numpy.int64)
    kv = _unpack(bvals)
    order = eng.order.cpu().numpy().astype(numpy.int64)
    slot_block = numpy.repeat(numpy.arange(bptr.size - 1), numpy.diff(bptr))
    rows_op = eng.first_row + slot_block[:, None] * 16 + numpy.arange(16)[None, :]
    keep = (kv != 0.0) & (rows_op < eng.last_row)
    rows = order[numpy.minimum(rows_op, n - 1)][keep]
    cols = order[numpy.broadcast_to(bidx[:, None], kv.shape)[keep]]
    pattern = numpy.zeros((n, n), dtype=bool)
    pattern[rows, cols] = True
    streams, zeros_ok = [], True
    for k in range(eng.dims.shape[0]):
        v = _unpack(eng.dims[k])
        zeros_ok = zeros_ok and bool((v[kv == 0.0] == 0.0).all())
        M = numpy.zeros((n, n))
        M[rows, cols] = v[keep]
        streams.append(M)
    return pattern, streams, zeros_ok


def _check_streams(eng, pts, scale, nu, pattern_ref):
    from oracle import matern
    pattern, streams, zeros_ok = _dense_streams(eng)
    assert zeros_ok
    assert (pattern == pattern_ref).all()
    assert len(streams) == pts.shape[1]
    tol = 1e-11 if not (nu in (0.5, 1.5, 2.5) or nu >= 100) else 1e-14     # Bessel branch: the device K_nu
    for k, got in enumerate(streams):
        ref = numpy.where(pattern_ref, matern.matern_derivative_scale(pts, scale, nu, k), 0.0)
        assert numpy.max(numpy.abs(got - ref)) <= tol * numpy.max(numpy.abs(ref)), (k, nu)


def _problem(scale=(0.03, 0.05), nu=0.5):
    from oracle import data_utilities as du
    from gaussian_proc._sparse import generate_sparse_operator
    numpy.random.seed(1)
    pts = numpy.random.rand(3000, 2)
    K = generate_sparse_operator(pts, numpy.array(scale), nu, 0.01, with_derivative=True)
    return pts, du.generate_data(pts, 0.2), du.generate_basis_functions(pts, 2), K


@pytest.fixture(scope='module')
def aniso_problem():
    return _problem()


OPTS = {'seed': 0, 'lanczos_degree': 40, 'min_num_samples': 128, 'max_num_samples': 128, 'cg_tol': 1e-11}


# ------------------------------------------------------------------------------------------------------ 1. the streams
@pytest.mark.gpu
@pytest.mark.parametrize('d', [1, 2, 3])
@pytest.mark.parametrize('nu', [0.5, 1.5, 2.5, 0.7, 200.0])
def test_direct_operator_streams_equal_the_oracle(nu, d):
    from gaussian_proc._sparse import generate_sparse_operator, SparseEngine, DeviceRowBlocks, _device_points
    numpy.random.seed(10 * d + int(nu))
    n = 1203                                                   # not a multiple of 16
    pts = numpy.random.rand(n, d)
    scale = numpy.array([0.06, 0.1, 0.08][:d]) if d > 1 else numpy.array([0.01])
    K = generate_sparse_operator(pts, scale, nu, 0.05, with_derivative=True)
    assert isinstance(K, DeviceRowBlocks)
    if d == 1:
        # one entry is an isotropic scale (today's dK/drho in bdvals): the per-dimension path is forced
        assert K.dscale is None and K.bdvals is not None
        K.dscale = (_device_points(pts)[0], scale, float(nu))
    else:
        assert K.dscale is not None and K.ddata is None
    eng = SparseEngine(K)
    assert K.bdvals_dims is eng.dims
    _check_streams(eng, pts, scale, nu, K.to_scipy().toarray() != 0)


@pytest.mark.gpu
@pytest.mark.parametrize('nu', [0.5, 1.5])
def test_csr_fallback_streams_equal_the_oracle(nu):
    """grid points with the threshold on a lattice distance: exact ties, so the operator comes from the CSR generator and
    the engine builds the blocks (gp_bcsr_fill) - the same kernel writes the streams"""
    from gaussian_proc._sparse import generate_sparse_operator, SparseEngine, DeviceCSR
    from oracle import data_utilities as du, matern
    pts = du.generate_points(40, 2, grid=True)
    sc = numpy.array([0.03, 0.045])
    x = matern.scaled_distance_matrix(pts[[0, 2]], sc)[0, 1]
    tau = float(matern.matern_kernel(x, nu))
    K = generate_sparse_operator(pts, sc, nu, 0.01, kernel_threshold=tau, with_derivative=True)
    assert isinstance(K, DeviceCSR) and K.ddata is None and K.dscale is not None
    eng = SparseEngine(K)
    _check_streams(eng, pts, sc, nu, K.to_scipy().toarray() != 0)


@pytest.mark.gpu
def test_one_rank_slab_streams_equal_the_oracle(aniso_problem):
    from gaussian_proc._sparse import generate_sparse_operator
    from gaussian_proc._slab import SlabSparseEngine
    pts, _, _, K = aniso_problem
    Ks = generate_sparse_operator(pts, numpy.array([0.03, 0.05]), 0.5, 0.01, with_derivative=True, row_slab=(0, 1))
    eng = SlabSparseEngine(Ks, 'slq', {'overlap': False}, rank=0, world=1)
    _check_streams(eng, pts, numpy.array([0.03, 0.05]), 0.5, K.to_scipy().toarray() != 0)


# ------------------------------------------------------------------------------------------------------ 2. isotropic identity
@pytest.mark.gpu
@pytest.mark.parametrize('nu', [0.5, 2.5, 0.7])
def test_streams_of_an_isotropic_scale_sum_to_dK_drho(nu):
    import ctypes
    import torch
    from gaussian_proc import _device as dev
    from gaussian_proc._sparse import generate_sparse_operator, _device_points, SparseEngine
    numpy.random.seed(5)
    pts = numpy.random.rand(2000, 2)
    sc = numpy.array([0.03, 0.03])
    K = generate_sparse_operator(pts, sc, nu, 0.01, with_derivative=True)
    dpts = _device_points(pts)[0]
    total = K.bidx.numel()
    dims = torch.empty((2, 16 * total), dtype=torch.float64, device='cuda')
    P = lambda t: ctypes.c_void_p(t.data_ptr())       # noqa: E731
    assert dev.lib.gp_bcsr_dscale_fill(P(K.bptr), P(K.bidx), P(K.bvals), total, 0, K.n, P(K.order), P(dpts), K.n, 2,
                                       dev.host_ptr(sc), nu, P(dims), dev.stream_ptr()) == 0
    got = dims.sum(dim=0).cpu().numpy()
    ref = K.bdvals.cpu().numpy()
    assert ((got == 0.0) == (ref == 0.0)).all()
    assert numpy.max(numpy.abs(got - ref) / numpy.maximum(numpy.abs(ref), 1e-300)) <= 2e-15
    # engine level: the per-dimension Hutchinson samples summed over k = the isotropic samples of the same probes
    K2 = generate_sparse_operator(pts, sc, nu, 0.01, with_derivative=True)
    K2.dscale = (dpts, sc, float(nu))                          # forces the per-dimension path on an isotropic scale
    opts = {'seed': 7, 'lanczos_degree': 40, 'cg_tol': 1e-10}
    iso = SparseEngine(K, 'slq', dict(opts))._dk_samples(2.0, 0, 16)
    per = SparseEngine(K2, 'slq', dict(opts))._dk_samples(2.0, 0, 16)
    assert iso.shape == (16, 1) and per.shape == (16, 2)
    assert numpy.max(numpy.abs(per.sum(axis=1) - iso[:, 0])) <= 1e-12 * numpy.max(numpy.abs(iso))


# ------------------------------------------------------------------------------------------------------ 3. fused pieces
@pytest.mark.gpu
def test_fused_pieces_and_gradients_against_the_oracle(aniso_problem):
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood, DirectLikelihood, _fused
    from oracle import likelihood as L, matern
    pts, z, X, K = aniso_problem
    n, m = X.shape
    p = m + 1
    eta = 2.0
    scale = numpy.array([0.03, 0.05])
    Km = MixedCorrelation(K, imate_method='slq', imate_options=dict(OPTS))
    eng = Km.engine
    q = _fused.evaluate(z, X, Km, eta, traceinv=True, drho=True)
    rows = eng.last_dscale
    assert rows.shape == (2, 1 + p * p) and q.trace_MdK_dims.shape == (2,)
    Kh = K.to_scipy().toarray()
    dKh = [numpy.where(Kh != 0, matern.matern_derivative_scale(pts, scale, 0.5, k), 0.0) for k in range(2)]
    Kn = Kh + eta * numpy.eye(n)
    R = numpy.c_[X, z]
    S = numpy.linalg.solve(Kn, R)
    for k in range(2):
        ref = S.T @ dKh[k] @ S
        assert numpy.max(numpy.abs(rows[k, 1:].reshape(p, p) - ref)) <= 1e-8 * numpy.max(numpy.abs(ref))
    # per-probe samples against dense solves with the same probes
    V = eng.from_op(eng.probes(0, 16)).cpu().numpy()
    U = numpy.linalg.solve(Kn, V)
    got = eng._dk_samples(eta, 0, 16)
    for k in range(2):
        ref = numpy.sum(U * (dKh[k] @ V), axis=0)
        assert numpy.max(numpy.abs(got[:, k] - ref)) <= 1e-8 * numpy.max(numpy.abs(ref))
    # traces within 4 standard errors of the exact values
    Kninv = numpy.linalg.inv(Kn)
    tr = eng.traceinv_dK(eta)
    hwd = numpy.asarray(eng.last_info['half_width']) * 4.0 / 1.96
    assert eng.last_info['num_samples'] == 128 and hwd.shape == (2,)
    for k in range(2):
        assert abs(tr[k] - numpy.sum(Kninv * dKh[k])) <= hwd[k]
        assert tr[k] == rows[k, 0]
    # final numbers: the oracle's formulas per k on the dense matrices; error budget = half the trace errors
    Ko = L.MixedCorrelation(Kh, 'cholesky')
    _, _, drho = ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, eta)
    assert drho.shape == (2,)
    for k in range(2):
        ref = L.ProfileLikelihood.log_likelihood_der1_rho(z, X, Ko, dKh[k], eta)
        assert abs(drho[k] - ref) <= 0.5 * hwd[k] + 1e-7 * abs(ref), (k, drho, ref)
    sigma, sigma0 = 0.8, 0.8 * numpy.sqrt(eta)
    _, _, drho_d = DirectLikelihood.log_likelihood_and_gradient(z, X, Km, [sigma, sigma0])
    assert drho_d.shape == (2,)
    for k in range(2):
        ref = L.DirectLikelihood.log_likelihood_der1_rho(z, X, Ko, dKh[k], [sigma, sigma0])
        assert abs(drho_d[k] - ref) <= 0.5 * hwd[k] + 1e-7 * abs(ref), (k, drho_d, ref)


# ------------------------------------------------------------------------------------------------------ 4. - 6.
@pytest.mark.gpu
def test_loglik_and_eta_derivative_do_not_depend_on_the_gradient_request(aniso_problem):
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    pts, z, X, K = aniso_problem
    a = ProfileLikelihood.log_likelihood_and_gradient(z, X, MixedCorrelation(K, imate_method='slq', imate_options=dict(OPTS)), 2.0)
    b = ProfileLikelihood.log_likelihood_and_gradient(z, X, MixedCorrelation(K, imate_method='slq', imate_options=dict(OPTS)), 2.0,
                                                      with_rho=False)
    assert b[2] is None and a[2].shape == (2,)
    for x, y in zip(a[:2], b[:2]):
        assert abs(x - y) <= 1e-12 * max(abs(y), 1.0)


@pytest.mark.gpu
def test_a_second_eta_reuses_the_kept_krylov_runs(aniso_problem):
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    pts, z, X, K = aniso_problem
    opts = dict(OPTS, min_num_samples=32, max_num_samples=32, lanczos_degree=60, solve_degree=120)
    Km = MixedCorrelation(K, imate_method='slq', imate_options=opts)
    eng = Km.engine
    ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, 2.0)
    calls = []
    spmm = eng.spmm

    def counted(eta, X_dev, derivative=False, dim=None):
        calls.append((dim, X_dev.shape[1]))
        return spmm(eta, X_dev, derivative=derivative, dim=dim)
    eng.spmm = counted
    got = ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, 5.0)
    assert not [c for c in calls if c[0] is not None and c[1] == 16]       # no derivative SpMM of a probe block
    assert sorted(c[0] for c in calls if c[0] is not None) == [0, 1]       # the two Q_k
    assert eng.last_dk_solver == 'lanczos'
    fresh = MixedCorrelation(K, imate_method='slq', imate_options=opts)
    ref = ProfileLikelihood.log_likelihood_and_gradient(z, X, fresh, 5.0)
    fresh.engine.traceinv_dK(5.0)
    band = numpy.asarray(fresh.engine.last_info['half_width'])
    assert abs(got[0] - ref[0]) <= 1e-7 * abs(ref[0]) and abs(got[1] - ref[1]) <= 1e-7 * max(abs(ref[1]), 1.0)
    assert (numpy.abs(got[2] - ref[2]) <= band).all(), (got[2], ref[2], band)


@pytest.mark.gpu
def test_reuse_off_and_hutchinson_give_the_same_samples(aniso_problem):
    from gaussian_proc._sparse import SparseEngine
    pts, z, X, K = aniso_problem
    opts = {'seed': 2, 'lanczos_degree': 40, 'cg_tol': 1e-8}
    a = SparseEngine(K, 'slq', dict(opts))
    sa = a._dk_samples(2.0, 0, 16)
    assert a.last_dk_solver == 'lanczos' and sa.shape == (16, 2)
    for eng in (SparseEngine(K, 'slq', dict(opts, reuse_lanczos=False)), SparseEngine(K, 'hutchinson', dict(opts))):
        sb = eng._dk_samples(2.0, 0, 16)
        assert numpy.max(numpy.abs(sa - sb)) <= 1e-6 * numpy.max(numpy.abs(sa))


# ------------------------------------------------------------------------------------------------------ 7. one-rank slab
@pytest.mark.gpu
def test_one_rank_slab_engine_equals_the_sparse_engine(aniso_problem):
    from gaussian_proc._sparse import SparseEngine, generate_sparse_operator
    from gaussian_proc._slab import SlabSparseEngine
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    pts, z, X, K = aniso_problem
    opts = {'seed': 3, 'lanczos_degree': 40, 'overlap': False}
    one = SparseEngine(K, 'slq', dict(opts))
    f1 = one.fused(2.0, X, z)
    d1 = one.last_dscale.copy()
    Ks = generate_sparse_operator(pts, numpy.array([0.03, 0.05]), 0.5, 0.01, with_derivative=True, row_slab=(0, 1))
    for _ in range(2):                          # the second engine takes the already-encoded handle and its kept streams
        slab = SlabSparseEngine(Ks, 'slq', dict(opts), rank=0, world=1)
        f2 = slab.fused(2.0, X, z)
        assert numpy.max(numpy.abs(f1 - f2) / numpy.maximum(numpy.abs(f1), 1e-300)) <= 1e-12
        assert numpy.max(numpy.abs(d1 - slab.last_dscale) / numpy.maximum(numpy.abs(d1), 1e-300)) <= 1e-12
    assert Ks.encoded is not None and Ks.bdvals_dims is slab.dims
    a = ProfileLikelihood.log_likelihood_and_gradient(z, X, MixedCorrelation(K, imate_method='slq', imate_options=dict(opts)), 2.0)
    b = ProfileLikelihood.log_likelihood_and_gradient(z, X, MixedCorrelation(Ks, imate_method='slq', imate_options=dict(opts, row_slabs=True)),
                                                      2.0)
    # dl/deta and dl/d scale[k] are differences of pieces that agree to 1e-12: compared relative to those pieces
    assert abs(a[0] - b[0]) <= 1e-12 * abs(a[0])
    assert abs(a[1] - b[1]) <= 1e-12 * abs(f1[1])                                 # tr Kn^-1
    assert numpy.max(numpy.abs(a[2] - b[2])) <= 1e-12 * numpy.max(numpy.abs(d1[:, 0]))     # tr(Kn^-1 dK_k)


# ------------------------------------------------------------------------------------------------------ 8. errors
@pytest.mark.gpu
def test_operators_that_cannot_carry_per_dimension_derivatives_raise(aniso_problem):
    from gaussian_proc._sparse import generate_sparse_correlation, DeviceCSR
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    pts, z, X, _ = aniso_problem
    sc = numpy.array([0.03, 0.05])
    with pytest.raises(ValueError):
        generate_sparse_correlation(pts, sc, 0.5, 0.01, with_derivative=True)          # the SciPy result
    Kd = generate_sparse_correlation(pts, sc, 0.5, 0.01, device=True, with_derivative=True)
    assert Kd.ddata is None and Kd.dscale is not None
    plain = DeviceCSR(Kd.n, Kd.indptr, Kd.indices, Kd.data, None, kernel_threshold=Kd.kernel_threshold,
                      sorted_rows=Kd.sorted_rows)
    plain.dscale = Kd.dscale                                                             # no spatial order
    Km = MixedCorrelation(plain, imate_method='slq', imate_options={'min_num_samples': 16, 'max_num_samples': 16})
    with pytest.raises(ValueError):
        ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, 2.0)
    lp, deta, _ = ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, 2.0, with_rho=False)
    assert numpy.isfinite(lp) and numpy.isfinite(deta)
    # an isotropic scale keeps the scalar d/drho
    Ki = generate_sparse_correlation(pts, numpy.array([0.03, 0.03]), 0.5, 0.01, device=True, with_derivative=True)
    assert Ki.dscale is None
    drho = ProfileLikelihood.log_likelihood_and_gradient(z, X, MixedCorrelation(Ki, imate_method='slq'), 2.0)[2]
    assert isinstance(drho, float)


# ------------------------------------------------------------------------------------------------------ two or more GPUs
@pytest.mark.gpu
def test_anisotropic_gradient_on_row_slabs_equals_one_gpu():
    import torch
    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip('needs two GPUs')
    cmd = [sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr',
           '127.0.0.1', '--master-port', '29534', os.path.join(ROOT, 'tools', 'gpu_check_sparse_slab.py'), '65536', 'aniso']
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    out = [json.loads(line) for line in res.stdout.splitlines() if line.startswith('{')]
    an = [o for o in out if 'aniso' in o][0]['aniso']
    assert an['grad_rel_diff'] <= 1e-11 and an['dscale_rel_diff'] <= 1e-11 and an['peer_error'] == 0
