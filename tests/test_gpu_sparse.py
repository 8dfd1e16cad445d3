"""GPU parity tests (sparse path). Bar (BASELINE.json north_star): sparse pattern and CSR indices BIT-EXACT against the
reference's compiled generator; values within a few ulp; stochastic-trace outputs within the estimator's own stated
confidence band (at a fixed seed) around exact values from the CPU oracle."""

import numpy
import pytest
import scipy.sparse

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def gp():
    import gaussian_proc
    return gaussian_proc


def grid_points():
    from oracle import data_utilities as du
    return du.generate_points(40, 2, grid=True)


@pytest.mark.parametrize('tag', ['rand', 'grid'])
@pytest.mark.parametrize('nu', [0.5, 1.5, 2.5])
def test_sparse_csr_bit_exact_pattern(gp, golden_generate, tag, nu):
    pts = golden_generate['sparse_points'] if tag == 'rand' else grid_points()
    S = gp.generate_correlation(pts, numpy.array([0.03, 0.03]), nu, sparse=True, density=0.01)
    key = 'sparse_%s_nu%g_' % (tag, nu)
    assert scipy.sparse.isspmatrix_csr(S)
    assert S.indices.dtype == numpy.int32 and S.indptr.dtype == numpy.int32 and S.data.dtype == numpy.float64
    assert (S.indptr == golden_generate[key + 'indptr']).all()
    assert (S.indices == golden_generate[key + 'indices']).all()
    ref = golden_generate[key + 'data']
    assert numpy.max(numpy.abs(S.data - ref) / ref) <= 4 * 2.3e-16       # values: a few ulp (device exp)
    assert S.has_sorted_indices and (S.diagonal() == 1.0).all()


def test_kernel_threshold_bit_follows_reference():
    from gaussian_proc._sparse import estimate_kernel_threshold
    from oracle import matern
    for (n, d, density, scale, nu) in [(1500, 2, 0.01, [0.03, 0.03], 0.5), (1600, 2, 0.01, [0.03, 0.03], 2.5),
                                       (4000, 3, 0.005, [0.1, 0.2, 0.15], 1.5), (900, 1, 0.02, [0.05], 200.0),
                                       (2 ** 20, 2, 1e-3, [0.005, 0.005], 0.5)]:
        t = estimate_kernel_threshold(n, d, density, numpy.array(scale), nu)
        assert t == matern.estimate_kernel_threshold(n, d, density, numpy.array(scale), nu)
    with pytest.raises(ValueError):
        estimate_kernel_threshold(50, 2, 1e-3, numpy.array([0.1, 0.1]), 0.5)


def test_sparse_edge_cases(gp):
    from oracle import matern
    # 1-D and 3-D points, anisotropic scale, tiny n (single cell), explicit threshold
    for (n, d, scale, nu, dens) in [(300, 1, [0.02], 0.5, 0.05), (500, 3, [0.2, 0.3, 0.25], 1.5, 0.02),
                                    (64, 2, [0.5, 0.5], 2.5, 0.3), (700, 2, [0.02, 0.05], 1.5, 0.02),
                                    (2400, 2, [0.3, 0.3], 0.5, 0.9)]:     # rows of > 512 entries: CTA-wide sort path
        numpy.random.seed(n)
        pts = numpy.random.rand(n, d)
        S = gp.generate_correlation(pts, numpy.array(scale), nu, sparse=True, density=dens)
        R = matern.generate_sparse_correlation(pts, numpy.array(scale), nu, dens)
        assert (S.indptr == R.indptr).all() and (S.indices == R.indices).all()
        assert numpy.max(numpy.abs(S.data - R.data)) <= 1e-15
    # duplicate points (distance exactly zero off the diagonal)
    pts = numpy.random.rand(200, 2)
    pts[17] = pts[3]
    S = gp.generate_correlation(pts, 0.05, 0.5, sparse=True, density=0.05)
    assert S[17, 3] == 1.0 and S[3, 17] == 1.0


def test_sparse_device_handle_and_derivative(gp):
    from gaussian_proc._sparse import generate_sparse_correlation
    from oracle import matern
    numpy.random.seed(5)
    pts = numpy.random.rand(900, 2)
    Kd = generate_sparse_correlation(pts, numpy.array([0.04, 0.04]), 1.5, 0.02, device=True, with_derivative=True)
    S = Kd.to_scipy()
    dK = matern.matern_derivative_rho(pts, 0.04, 1.5)
    ref = dK[S.nonzero()]
    got = scipy.sparse.csr_matrix((Kd.ddata.cpu().numpy(), S.indices, S.indptr), shape=S.shape)[S.nonzero()]
    assert numpy.max(numpy.abs(numpy.asarray(got).ravel() - numpy.asarray(ref).ravel())) <= 1e-11


def test_full_size_pattern_properties(gp):
    """n = 2^20 (BASELINE configs[3]): sampled rows against the brute-force oracle row routine, plus symmetry of the
    pattern, sortedness and unit diagonal."""
    from gaussian_proc._sparse import generate_sparse_correlation
    from oracle import matern
    import ctypes
    n = 2 ** 20
    numpy.random.seed(0)
    pts = numpy.random.rand(n, 2)
    scale = numpy.array([0.005, 0.005])
    Kd = generate_sparse_correlation(pts, scale, 0.5, 1e-3, device=True)
    S = Kd.to_scipy()
    assert S.shape == (n, n) and S.indices.dtype == numpy.int32
    assert (numpy.diff(S.indptr) >= 1).all()
    lib = matern._c()
    tau = Kd.kernel_threshold
    rows = [0, 1, 12345, 500000, n - 1]
    for r in rows:
        cnt = numpy.zeros(n, dtype=numpy.int64)
        lib.oracle_sparse_rows(pts.ctypes.data, n, 2, scale.ctypes.data, 0.5, tau, 0, r, r + 1, cnt.ctypes.data, None, None, None)
        k = int(cnt[r])
        ip = numpy.zeros(n + 1, dtype=numpy.int64)
        idx = numpy.zeros(k, dtype=numpy.int32)
        dat = numpy.zeros(k)
        lib.oracle_sparse_rows(pts.ctypes.data, n, 2, scale.ctypes.data, 0.5, tau, 1, r, r + 1, None, ip.ctypes.data,
                               idx.ctypes.data, dat.ctypes.data)
        got = S.indices[S.indptr[r]:S.indptr[r + 1]]
        assert len(got) == k and (got == idx).all()
        assert numpy.max(numpy.abs(S.data[S.indptr[r]:S.indptr[r + 1]] - dat)) <= 1e-15
    sub = S[:20000]
    assert (numpy.diff(sub.indices) > 0)[numpy.diff(numpy.repeat(numpy.arange(20000), numpy.diff(sub.indptr))) == 0].all()
    # pattern symmetry on a block
    blk = S[:5000, :5000]
    assert (abs(blk - blk.T) > 0).nnz == 0


# --------------------------------------------------------------------------------------------- sparse operator
@pytest.fixture(scope='module')
def sparse_problem(gp):
    from oracle import data_utilities as du
    from gaussian_proc._sparse import generate_sparse_correlation
    numpy.random.seed(1)
    pts = numpy.random.rand(3000, 2)
    Kd = generate_sparse_correlation(pts, numpy.array([0.03, 0.03]), 0.5, 0.01, device=True, with_derivative=True)
    return pts, du.generate_data(pts, 0.2), du.generate_basis_functions(pts, 2), Kd


def _plain_csr(Kd):
    """the same matrix without a spatial order (its arrays shared): the engine keeps plain CSR in the original order"""
    from gaussian_proc._sparse import DeviceCSR
    return DeviceCSR(Kd.n, Kd.indptr, Kd.indices, Kd.data, Kd.ddata, kernel_threshold=Kd.kernel_threshold,
                     sorted_rows=Kd.sorted_rows)


def test_spmm_dot_solve(sparse_problem):
    from gaussian_proc._mixed_correlation import MixedCorrelation
    pts, z, X, Kd = sparse_problem
    S = Kd.to_scipy()
    Km = MixedCorrelation(Kd, imate_method='slq')
    assert Km.get_matrix_size() == 3000
    assert numpy.max(numpy.abs(Km.dot(0.7, z) - (S @ z + 0.7 * z))) <= 1e-12
    assert numpy.max(numpy.abs(Km.dot(0, X) - S @ X)) <= 1e-12
    eta = 2.0
    A = (S + eta * scipy.sparse.eye(3000)).toarray()
    ref = numpy.linalg.solve(A, numpy.c_[X, z])
    sol = Km.solve(eta, numpy.c_[X, z])
    # the reference's CG stops at ||r|| <= 1e-6 ||b|| (_linear_solver.py:24): same rule here
    r = A @ sol - numpy.c_[X, z]
    assert (numpy.linalg.norm(r, axis=0) <= 1e-6 * numpy.linalg.norm(numpy.c_[X, z], axis=0)).all()
    assert numpy.max(numpy.abs(sol - ref)) / numpy.max(numpy.abs(ref)) <= 1e-5
    assert abs(Km.trace(0.5) - (S.diagonal().sum() + 0.5 * 3000)) <= 1e-9


def test_slq_samples_equal_the_cpu_oracle_per_probe(sparse_problem):
    """Same seed -> same Rademacher probes (hash restated in oracle/slq.py) -> the device SLQ samples [log, 1/x, 1/x^2]
    equal an independent NumPy Lanczos + quadrature PER PROBE (not only in distribution)."""
    from gaussian_proc._sparse import SparseEngine
    from oracle import slq
    pts, z, X, Kd = sparse_problem
    eng = SparseEngine(_plain_csr(Kd), 'slq', {'seed': 11, 'lanczos_degree': 20})
    assert (eng.probes(4, 4).cpu().numpy() == slq.rademacher(eng.n, 4, 11, 4)).all()
    ref = slq.slq_samples(Kd.to_scipy(), 2.0, 11, 4, 4, 20)
    for K in (_plain_csr(Kd), Kd):
        e = SparseEngine(K, 'slq', {'seed': 11, 'lanczos_degree': 20})
        got = e._slq_samples(2.0, 4, 4)
        assert numpy.max(numpy.abs(got - ref) / numpy.abs(ref)) <= 1e-9, (e.blocked is not None, got, ref)


def test_probes_are_batching_invariant(sparse_problem):
    from gaussian_proc._sparse import SparseEngine
    eng = SparseEngine(sparse_problem[3])
    V8 = eng.probes(0, 8).cpu().numpy()
    V4 = eng.probes(4, 4).cpu().numpy()
    assert (V8[:, 4:] == V4).all() and set(numpy.unique(V8)) == {-1.0, 1.0}
    assert abs(V8.mean()) < 0.02


@pytest.mark.parametrize('method', ['slq', 'hutchinson'])
def test_stochastic_estimates_within_confidence_band(sparse_problem, method):
    from gaussian_proc._mixed_correlation import MixedCorrelation
    pts, z, X, Kd = sparse_problem
    S = Kd.to_scipy()
    n = S.shape[0]
    for eta in (1.0, 10.0):
        A = (S + eta * scipy.sparse.eye(n)).toarray()
        w = numpy.linalg.eigvalsh(A)
        assert w.min() > 0
        Km = MixedCorrelation(Kd, imate_method=method, imate_options={'seed': 0, 'lanczos_degree': 30})
        ld = Km.logdet(eta)
        band = Km.engine.last_info['half_width'][0]
        exact = numpy.sum(numpy.log(w))
        assert abs(ld - exact) <= max(band, 0.01 * abs(exact)) and band <= 0.011 * abs(exact) + 1e-9
        ti = Km.traceinv(eta)
        exact_ti = numpy.sum(1.0 / w)
        assert abs(ti - exact_ti) <= 0.012 * exact_ti
        # derivative trace (Hutchinson + CG), exact value from the dense inverse
        dS = scipy.sparse.csr_matrix((Kd.ddata.cpu().numpy(), S.indices, S.indptr), shape=S.shape).toarray()
        exact_d = numpy.sum(numpy.linalg.inv(A) * dS)
        est = Km.engine.traceinv_dK(eta)
        half = Km.engine.last_info['half_width'][0]
        assert abs(est - exact_d) <= max(2.0 * half, 0.02 * abs(exact_d))


def test_indefinite_matrix_is_reported(gp):
    """SURVEY Q11: hard-thresholded Matern is not positive definite; small eta must be reported, not silently used."""
    from gaussian_proc._mixed_correlation import MixedCorrelation
    numpy.random.seed(3)
    pts = numpy.random.rand(2000, 2)
    S = gp.generate_correlation(pts, 0.02, 2.5, sparse=True, density=5e-3)
    lam = scipy.sparse.linalg.eigsh(S, k=1, which='SA', return_eigenvectors=False)[0]
    assert lam < -0.05          # -0.665 for this seed (SURVEY Q11 probed -0.70 for the same settings): the check is unconditional
    Km = MixedCorrelation(S, imate_method='slq', imate_options={'lanczos_degree': 60})
    with pytest.raises(numpy.linalg.LinAlgError):
        Km.logdet(1e-3)
    assert numpy.isfinite(Km.logdet(1.0))      # eta above -lambda_min: fine


def test_slq_logdet_against_sparse_lu_n131072(gp):
    """n = 2^17: the SLQ log-determinant of K + eta I against the EXACT value from a sparse LU of the same matrix
    (scipy.sparse.linalg.splu, sum log |U_ii|; SURVEY 8c), inside the estimator's stated band (rtol 1e-2 at 95 %)."""
    import scipy.sparse.linalg
    from gaussian_proc._mixed_correlation import MixedCorrelation
    n = 2 ** 17
    numpy.random.seed(0)
    pts = numpy.random.rand(n, 2)
    S = gp.generate_correlation(pts, 0.0033, 0.5, sparse=True, density=9.6e-4)       # ~40 non-zeros per row
    assert 30 * n < S.nnz < 50 * n
    eta = 10.0
    lu = scipy.sparse.linalg.splu((S + eta * scipy.sparse.eye(n)).tocsc(), permc_spec='MMD_AT_PLUS_A',
                                  diag_pivot_thresh=0.0, options=dict(SymmetricMode=True))
    exact = float(numpy.sum(numpy.log(numpy.abs(lu.U.diagonal()))) + numpy.sum(numpy.log(numpy.abs(lu.L.diagonal()))))
    del lu
    Km = MixedCorrelation(S, imate_method='slq', imate_options={'seed': 0, 'lanczos_degree': 30})
    ld = Km.logdet(eta)
    band = Km.engine.last_info['half_width'][0]
    assert band <= 0.011 * abs(exact)
    assert abs(ld - exact) <= max(band, 0.01 * abs(exact)), (ld, exact, band)
    assert abs(ld - exact) <= 1e-3 * abs(exact)       # in fact far inside: K + 10 I is well conditioned


def test_cg_solve_residual_n1M(gp):
    """n = 2^20 (BASELINE configs[3]): the batched CG solve of (K + eta I) S = [X z] meets the reference's stopping rule
    ||r|| <= 1e-6 ||b|| (_linear_solver.py:24-73) in every column; the residual is formed with an independent product
    (SciPy CSR on the host) and M Kn M = M holds for the fused quantities."""
    from oracle import data_utilities as du
    from gaussian_proc._sparse import generate_sparse_correlation
    from gaussian_proc._mixed_correlation import MixedCorrelation
    n = 2 ** 20
    numpy.random.seed(0)
    pts = numpy.random.rand(n, 2)
    z, X = du.generate_data(pts, 0.2), du.generate_basis_functions(pts, 2)
    Kd = generate_sparse_correlation(pts, numpy.array([0.005, 0.005]), 0.5, 1e-3, device=True)
    Km = MixedCorrelation(Kd, imate_method='slq', imate_options={'seed': 0})
    eta = 10.0
    R = numpy.c_[X, z]
    sol = Km.solve(eta, R)
    S = Kd.to_scipy()
    r = S @ sol + eta * sol - R
    assert (numpy.linalg.norm(r, axis=0) <= 1.000001e-6 * numpy.linalg.norm(R, axis=0)).all()
    r_dev = Km.dot(eta, sol) - R                       # the device SpMM agrees with the host product
    assert numpy.max(numpy.abs(r_dev - r)) <= 1e-9 * numpy.max(numpy.abs(R))


def test_likelihood_through_sparse_operator(sparse_problem):
    """Q9: a sparse K can be trained through the Likelihood API (the reference cannot: eigh(sparse) raises)."""
    from gaussian_proc._likelihood import Likelihood
    pts, z, X, Kd = sparse_problem
    lk = Likelihood(X, Kd.to_scipy(), likelihood_method='profiled')
    assert lk.K_mixed.sparse and lk.K_mixed.imate_method == 'slq'
    # end to end: GaussianProcess.train on a sparse K (root of d l/d eta; the search interval starts above -lambda_min
    # of the hard-thresholded K) against the oracle's root finder on the densified matrix with exact traces
    from gaussian_proc import GaussianProcess
    from gaussian_proc._sparse import generate_sparse_correlation
    from oracle import likelihood as L, data_utilities as du
    numpy.random.seed(1)
    p2 = numpy.random.rand(1500, 2)
    z2, X2 = du.generate_data(p2, 0.2), du.generate_basis_functions(p2, 2)
    K2 = generate_sparse_correlation(p2, numpy.array([0.2, 0.2]), 0.5, 0.1, device=True)
    opts = {'seed': 0, 'lanczos_degree': 60, 'min_num_samples': 512, 'max_num_samples': 512, 'batch': 32, 'cg_tol': 1e-10}
    res = GaussianProcess(X2, K2, likelihood_method='profiled', imate_options=opts).train(z2, interval_eta=[8.0, 1e3])
    ref = L.ProfileLikelihood.find_log_likelihood_der1_zeros(z2, X2, L.MixedCorrelation(K2.to_scipy().toarray(), 'cholesky'),
                                                             [8.0, 1e3])
    assert res['success'] and ref['success']
    assert abs(numpy.log10(res['eta']) - numpy.log10(ref['eta'])) <= 0.15        # stochastic traces: 512 probes
    assert abs(res['sigma0'] - ref['sigma0']) <= 0.05 * ref['sigma0']
    with pytest.raises(numpy.linalg.LinAlgError):                                  # the reference's [1e-4, 1e3]: indefinite
        GaussianProcess(X2, K2, likelihood_method='profiled', imate_options={'min_num_samples': 16, 'max_num_samples': 16}).train(z2)


def test_sparse_loglik_and_gradient(sparse_problem):
    """The full profile log-likelihood + gradient through a sparse K (batched CG solves, skinny Gram matrices,
    SLQ / Hutchinson traces) against the oracle on the densified matrix: the deterministic ingredients G, H, Q to the
    CG tolerance, the final numbers within the estimators' confidence bands (fixed seed)."""
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood, _fused
    from oracle import likelihood as L
    pts, z, X, Kd = sparse_problem
    n, m = X.shape
    eta = 2.0
    Km = MixedCorrelation(Kd, imate_method='slq',
                          imate_options={'seed': 0, 'lanczos_degree': 40, 'min_num_samples': 128, 'max_num_samples': 128,
                                         'cg_tol': 1e-11})
    q = _fused.evaluate(z, X, Km, eta, traceinv=True, drho=True)
    Ks = Kd.to_scipy()
    Kh = Ks.toarray()
    dKh = scipy.sparse.csr_matrix((Kd.ddata.cpu().numpy(), Ks.indices, Ks.indptr), shape=Ks.shape).toarray()
    Kn = Kh + eta * numpy.eye(n)
    R = numpy.c_[X, z]
    S = numpy.linalg.solve(Kn, R)
    for got, ref in ((q.G, R.T @ S), (q.H, S.T @ S), (q.Q, S.T @ dKh @ S)):
        assert numpy.max(numpy.abs(got - ref)) <= 1e-8 * numpy.max(numpy.abs(ref))
    Kninv = numpy.linalg.inv(Kn)
    exact = {'logdet': numpy.linalg.slogdet(Kn)[1], 'ti': numpy.trace(Kninv), 'ti2': numpy.sum(Kninv * Kninv),
             'tdk': numpy.sum(Kninv * dKh)}
    # 128 probes: every estimate within 4 standard errors of the exact value (stated band: 1.96 standard errors)
    eng = Km.engine
    eng._slq_cache = {}
    eng.logdet(eta)
    hw = eng.last_info['half_width'] * 4.0 / 1.96
    assert abs(q.logdet_Kn - exact['logdet']) <= hw[0]
    assert abs(q.trace_Kninv - exact['ti']) <= hw[1]
    assert abs(q.trace_Kninv2 - exact['ti2']) <= hw[2]
    eng.traceinv_dK(eta)
    hwd = float(eng.last_info['half_width'][0]) * 4.0 / 1.96
    assert abs(q.trace_Kninv_dK - exact['tdk']) <= hwd
    # final numbers: the oracle's formulas on the dense matrices; error budget = half the trace errors
    Ko = L.MixedCorrelation(Kh, 'cholesky')
    sig = L.ProfileLikelihood.find_optimal_sigma(z, X, Ko, eta)
    ref = (L.ProfileLikelihood.log_likelihood(z, X, Ko, False, [sig, eta]),
           L.ProfileLikelihood.log_likelihood_der1_eta(z, X, Ko, numpy.log10(eta)),
           L.ProfileLikelihood.log_likelihood_der1_rho(z, X, Ko, dKh, eta))
    lp, deta, drho = ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, eta)
    assert abs(lp - ref[0]) <= 0.5 * hw[0] + 1e-7 * abs(ref[0])
    assert abs(deta - ref[1]) <= 0.5 * hw[1] + 1e-7 * abs(ref[1])
    assert abs(drho - ref[2]) <= 0.5 * hwd + 1e-7 * abs(ref[2])


def test_hutchinson_dk_reuses_the_lanczos_basis(sparse_problem):
    """tr(Kn^-1 dK): Kn^-1 v from the SLQ run's Lanczos vectors (x = ||v|| Q T^-1 e_1, residual checked against the CG
    tolerance) gives the same per-probe samples as separate batched CG solves."""
    from gaussian_proc._sparse import SparseEngine
    pts, z, X, Kd = sparse_problem
    opts = {'seed': 2, 'lanczos_degree': 40, 'min_num_samples': 32, 'max_num_samples': 32, 'cg_tol': 1e-8}
    a = SparseEngine(Kd, 'slq', dict(opts, reuse_lanczos=True))
    b = SparseEngine(Kd, 'slq', dict(opts, reuse_lanczos=False))
    a.logdet(2.0)
    assert a.last_dk_solver == 'lanczos' and a._dk_state[2.0][0].shape == (32, 1)
    ta, tb = a.traceinv_dK(2.0), b.traceinv_dK(2.0)
    assert a.last_info['num_samples'] == b.last_info['num_samples'] == 32
    assert abs(ta - tb) <= 1e-6 * abs(tb)
    # 6 Lanczos steps cannot reach the tolerance at a small shift (lambda_min(K) ~ -0.5) -> fall back to CG
    c = SparseEngine(Kd, 'slq', dict(opts, lanczos_degree=6, reuse_lanczos=True))
    c.logdet(0.8)
    assert c.last_dk_solver == 'cg'
    assert abs(c.traceinv_dK(0.8) - SparseEngine(Kd, 'slq', dict(opts, reuse_lanczos=False)).traceinv_dK(0.8)) \
        <= 1e-6 * abs(c.traceinv_dK(0.8))


def test_krylov_runs_are_reused_across_eta(sparse_problem):
    """Shift invariance (the reference's imate.AffineMatrixFunction, mixed_correlation.py:44): one kept Lanczos run per
    probe block and one per right-hand-side block serve every eta of an operator. The numbers equal those of operators
    that recompute everything per eta (same probes; the solves agree to the CG tolerance)."""
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    pts, z, X, Kd = sparse_problem
    opts = {'seed': 4, 'lanczos_degree': 60, 'min_num_samples': 16, 'max_num_samples': 16, 'cg_tol': 1e-11,
            'solve_degree': 120}
    Ka = MixedCorrelation(Kd, imate_method='slq', imate_options=dict(opts, shift_reuse=True))
    etas = [2.0, 5.0, 40.0, 1.5]
    got = [ProfileLikelihood.log_likelihood_and_gradient(z, X, Ka, eta) for eta in etas]
    eng = Ka.engine
    assert ('probes', 0, 16) in eng._krylov and any(k[0] == 'rhs' for k in eng._krylov)
    assert eng.last_rhs_solver == 'lanczos' and eng.last_dk_solver == 'lanczos'
    launches_before = None
    for eta, g in zip(etas, got):
        Kb = MixedCorrelation(Kd, imate_method='slq', imate_options=dict(opts, shift_reuse=False))
        ref = ProfileLikelihood.log_likelihood_and_gradient(z, X, Kb, eta)
        for a, b in zip(g, ref):
            assert abs(a - b) <= 1e-7 * max(abs(b), 1.0), (eta, g, ref)
    # an eta below -lambda_min is still reported as not positive definite from the kept run
    with pytest.raises(numpy.linalg.LinAlgError):
        ProfileLikelihood.log_likelihood_and_gradient(z, X, Ka, 0.05)


def test_sparse_loglik_wide_basis(sparse_problem):
    """m + 1 > 8 right-hand sides: the [X z] block is 16 columns wide, the same width as the probe block whose Lanczos
    run overlaps its solve on the side stream (separate workspaces). Deterministic ingredients against dense solves."""
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import _fused
    pts, z, X, Kd = sparse_problem
    x, y = pts[:, 0], pts[:, 1]
    X10 = numpy.stack([numpy.ones_like(x), x, y, x * x, x * y, y * y, x ** 3, x * x * y, x * y * y, y ** 3], axis=1)
    eta = 2.0
    Km = MixedCorrelation(Kd, imate_method='slq', imate_options={'seed': 0, 'lanczos_degree': 40, 'cg_tol': 1e-11})
    q1 = _fused.evaluate(z, X10, Km, eta, traceinv=True, drho=True)
    q2 = _fused.evaluate(z, X10, Km, 5.0, traceinv=True, drho=True)          # second eta: kept Krylov runs
    Ks = Kd.to_scipy().toarray()
    R = numpy.c_[X10, z]
    for q, e in ((q1, eta), (q2, 5.0)):
        S = numpy.linalg.solve(Ks + e * numpy.eye(Ks.shape[0]), R)
        assert numpy.max(numpy.abs(q.G - R.T @ S)) <= 1e-8 * numpy.max(numpy.abs(R.T @ S))
        assert numpy.max(numpy.abs(q.H - S.T @ S)) <= 1e-8 * numpy.max(numpy.abs(S.T @ S))
        exact = numpy.linalg.slogdet(Ks + e * numpy.eye(Ks.shape[0]))[1]
        assert abs(q.logdet_Kn - exact) <= 2e-2 * abs(exact)          # the estimator stops at a 1 % half width


def test_row_blocked_operator_equals_csr(gp):
    """The row-blocked operator (16 x 1 blocks of the curve-ordered matrix, zero filled, DMMA SpMM) is the same linear map as
    the canonical CSR: products against the SciPy matrix to rounding, for K and for dK/drho, n not a multiple of 16."""
    import torch
    from gaussian_proc._sparse import SparseEngine, generate_sparse_correlation
    numpy.random.seed(5)
    n = 3001
    pts = numpy.random.rand(n, 2)
    Kd = generate_sparse_correlation(pts, numpy.array([0.03, 0.03]), 1.5, 0.01, device=True, with_derivative=True)
    order = Kd.order.cpu().numpy()
    assert sorted(order.tolist()) == list(range(n))
    eng = SparseEngine(Kd, 'slq', {})
    R = 16
    assert eng.R == R and eng.blocked is not None and 1.0 <= eng.fill_ratio <= R
    Ks = Kd.to_scipy()
    dKs = scipy.sparse.csr_matrix((Kd.ddata.cpu().numpy(), Ks.indices, Ks.indptr), shape=Ks.shape)
    for B in (1, 2, 4, 8, 16, 32):
        Xh = numpy.random.randn(n, B)
        Xd = torch.from_numpy(Xh).cuda()
        Y = eng.from_op(eng.spmm(0.75, eng.to_op(Xd))).cpu().numpy()
        ref = Ks @ Xh + 0.75 * Xh
        assert numpy.max(numpy.abs(Y - ref)) <= 1e-12 * numpy.max(numpy.abs(ref))
        Yd = eng.from_op(eng.spmm(0.0, eng.to_op(Xd), derivative=True)).cpu().numpy()
        refd = dKs @ Xh
        assert numpy.max(numpy.abs(Yd - refd)) <= 1e-12 * numpy.max(numpy.abs(refd))
    # the stored block-columns are exactly the union of the rows' patterns: value count = R * (number of block-columns)
    bptr, bidx, bvals, _ = eng.blocked
    assert int(bptr[-1]) == bidx.numel() and bvals.numel() == R * bidx.numel()
    assert int(((bptr[1:] - bptr[:-1]) % 4).abs().sum()) == 0        # padded to whole DMMA k-steps
    assert int((bvals != 0).sum()) == Ks.nnz


@pytest.mark.parametrize('n', [3, 8, 13, 70])
def test_row_blocked_operator_tiny_sizes(n):
    """fewer rows than one block, exactly one block, a ragged last block: products, solves and the estimators still
    agree with the dense matrix"""
    import torch
    from gaussian_proc._sparse import SparseEngine, generate_sparse_correlation
    numpy.random.seed(n)
    pts = numpy.random.rand(n, 2)
    Kd = generate_sparse_correlation(pts, numpy.array([0.3, 0.3]), 0.5, 0.6, device=True, with_derivative=True)
    eng = SparseEngine(Kd, 'slq', {'min_num_samples': 64, 'max_num_samples': 64, 'lanczos_degree': min(n, 20)})
    Ks = Kd.to_scipy().toarray()
    Xh = numpy.random.randn(n, 4)
    Y = eng.from_op(eng.spmm(0.5, eng.to_op(torch.from_numpy(Xh).cuda()))).cpu().numpy()
    assert numpy.max(numpy.abs(Y - (Ks @ Xh + 0.5 * Xh))) <= 1e-13
    eta = 3.0
    sol = eng.solve(eta, Xh[:, 0])
    assert numpy.max(numpy.abs(sol - numpy.linalg.solve(Ks + eta * numpy.eye(n), Xh[:, 0]))) <= 1e-6
    exact = numpy.linalg.slogdet(Ks + eta * numpy.eye(n))[1]
    assert abs(eng.logdet(eta) - exact) <= max(4.0 / 1.96 * eng.last_info['half_width'][0], 1e-9 * abs(exact))


@pytest.mark.parametrize('d,scale,nu,dens', [(1, [0.02], 1.5, 0.05), (3, [0.2, 0.3, 0.25], 2.5, 0.02), (2, [0.02, 0.05], 3.3, 0.02)])
def test_row_blocked_operator_other_dimensions(d, scale, nu, dens):
    """1-D and 3-D points (Z-order keys), anisotropic scale, general nu: the operator equals the canonical CSR"""
    import torch
    from gaussian_proc._sparse import SparseEngine, generate_sparse_correlation
    numpy.random.seed(17 + d)
    n = 1234
    pts = numpy.random.rand(n, d)
    Kd = generate_sparse_correlation(pts, numpy.array(scale), nu, dens, device=True)
    eng = SparseEngine(Kd, 'slq', {})
    assert eng.R == 16
    Ks = Kd.to_scipy()
    Xh = numpy.random.randn(n, 8)
    Y = eng.from_op(eng.spmm(1.0, eng.to_op(torch.from_numpy(Xh).cuda()))).cpu().numpy()
    ref = Ks @ Xh + Xh
    assert numpy.max(numpy.abs(Y - ref)) <= 1e-12 * numpy.max(numpy.abs(ref))


def test_row_blocked_build_search_fallback():
    """Row blocks with more distinct columns than the shared-memory hash table holds are built by the binary-search
    path: an unstructured random symmetric matrix (8 rows share almost nothing) with the identity as row order."""
    import torch
    from gaussian_proc._sparse import SparseEngine, DeviceCSR
    rng = numpy.random.RandomState(7)
    n = 3003
    A = scipy.sparse.random(n, n, density=0.08, random_state=rng, format='csr')
    A = (A + A.T + scipy.sparse.identity(n)).tocsr()
    A.sort_indices()
    Kd = DeviceCSR.from_scipy(A)
    Kd.order = torch.arange(n, dtype=torch.int32, device='cuda')
    eng = SparseEngine(Kd, 'slq', {})
    assert eng.R == 16 and eng.fill_ratio > 4.0         # ~ 16 x 480 distinct columns per block: above the hash capacity
    Xh = rng.randn(n, 16)
    Y = eng.from_op(eng.spmm(0.0, eng.to_op(torch.from_numpy(Xh).cuda()))).cpu().numpy()
    ref = A @ Xh
    assert numpy.max(numpy.abs(Y - ref)) <= 1e-12 * numpy.max(numpy.abs(ref))
    assert int((eng.blocked[2] != 0).sum()) == A.nnz


def test_internal_permutation_does_not_change_results(sparse_problem):
    """The operator works on a Z-order permuted, row-blocked copy of the CSR matrix; probes are hashed with original row
    ids, so every output must agree with the unpermuted plain-CSR operator up to summation order. The order is a
    stable sort, so two builds give bit-identical results."""
    from gaussian_proc._sparse import SparseEngine
    pts, z, X, Kd = sparse_problem
    opts = {'seed': 3, 'lanczos_degree': 25, 'min_num_samples': 16, 'max_num_samples': 16}
    a = SparseEngine(Kd, 'slq', dict(opts))
    b = SparseEngine(_plain_csr(Kd), 'slq', dict(opts))
    a2 = SparseEngine(Kd, 'slq', dict(opts))
    assert a.order is not None and b.order is None
    assert a.logdet(2.0) == a2.logdet(2.0)
    assert abs(a.logdet(2.0) - b.logdet(2.0)) <= 1e-10 * abs(b.logdet(2.0))
    assert abs(a.traceinv(2.0) - b.traceinv(2.0)) <= 1e-10 * abs(b.traceinv(2.0))
    assert abs(a.traceinv_dK(2.0) - b.traceinv_dK(2.0)) <= 1e-7 * abs(b.traceinv_dK(2.0))    # CG stops at rtol 1e-6
    assert numpy.max(numpy.abs(a.solve(2.0, z) - b.solve(2.0, z))) <= 1e-6 * numpy.max(numpy.abs(b.solve(2.0, z)))
    assert numpy.max(numpy.abs(a.matmul(X) - b.matmul(X))) <= 1e-12
    wide = numpy.random.RandomState(0).randn(a.n, 37)               # more columns than one SpMM block
    assert numpy.max(numpy.abs(a.matmul(wide) - b.matmul(wide))) <= 1e-11
    sw = a.solve(2.0, wide[:, :20])
    assert numpy.max(numpy.abs((Kd.to_scipy() @ sw + 2.0 * sw) - wide[:, :20])) <= 1e-5 * numpy.max(numpy.abs(wide))
    Va = a.from_op(a.probes(0, 4)).cpu().numpy()
    assert (Va == b.probes(0, 4).cpu().numpy()).all()


def test_sparse_grid_sweep(sparse_problem):
    """likelihood_grid(sparse=True): every cell equals the direct public-API evaluation at the same seed (within a row the
    eta cells share the operator's kept Krylov runs, so the agreement is at the level of the solver tolerance)."""
    from gaussian_proc.sweep import likelihood_grid
    from gaussian_proc._sparse import generate_sparse_correlation
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    pts, z, X, _ = sparse_problem
    opts = {'seed': 1, 'lanczos_degree': 60, 'min_num_samples': 16, 'max_num_samples': 16, 'cg_tol': 1e-11,
            'solve_degree': 120}
    rhos, etas = [0.025, 0.03], [2.0, 20.0]
    G = likelihood_grid(pts, z, X, 0.5, rhos, etas, sparse=True, density=0.01, imate_options=opts)
    assert G.shape == (2, 2, 3) and numpy.isfinite(G).all()
    K = generate_sparse_correlation(pts, numpy.array([0.03, 0.03]), 0.5, 0.01, device=True, with_derivative=True)
    ref = ProfileLikelihood.log_likelihood_and_gradient(z, X, MixedCorrelation(K, imate_method='slq', imate_options=opts), 20.0)
    assert numpy.allclose(G[1, 1], ref, rtol=1e-7, atol=0)


@pytest.mark.parametrize('n,bits', [(1, 64), (31, 8), (1024, 62), (1025, 63), (5000, 20), (300001, 64), (1 << 20, 62),
                                    (70000, 5)])
def test_index_kernels_match_numpy(n, bits):
    """csrc/gp_index.cu against numpy: stable radix argsort of 64-bit keys (odd and even pass counts, heavy duplicates),
    inverse permutation, count scan, row gather, bounding box - all bit-exact (integer / copy / min-max work)."""
    import ctypes
    from gaussian_proc import _device as dev
    torch = dev.require_cuda()
    lib = dev.lib
    P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
    rng = numpy.random.RandomState(n % 9973 + bits)
    keys = rng.randint(0, 1 << 62, size=n, dtype=numpy.int64).astype(numpy.uint64)
    if bits < 64:
        keys &= numpy.uint64((1 << bits) - 1)
    if n > 4096:
        keys[rng.randint(0, n, n // 3)] = keys[rng.randint(0, n, n // 3)]          # duplicates: stability matters
    dkeys = torch.from_numpy(keys.view(numpy.int64).copy()).cuda()
    order = torch.empty(n, dtype=torch.int32, device='cuda')
    ws = torch.empty(lib.gp_sort_workspace_bytes(n) // 8 + 8, dtype=torch.float64, device='cuda')
    s = dev.stream_ptr()
    assert lib.gp_sort_keys_u64(P(dkeys), n, bits, P(order), P(ws), s) == 0
    want = numpy.argsort(keys, kind='stable').astype(numpy.int32)
    got = order.cpu().numpy()
    assert (got == want).all()

    inv = torch.empty(n, dtype=torch.int32, device='cuda')
    assert lib.gp_inverse_permutation(P(order), n, P(inv), s) == 0
    inv_want = numpy.empty(n, dtype=numpy.int32)
    inv_want[want] = numpy.arange(n, dtype=numpy.int32)
    assert (inv.cpu().numpy() == inv_want).all()

    counts = rng.randint(0, 4000, size=n).astype(numpy.int32)
    offs = torch.empty(n + 1, dtype=torch.int64, device='cuda')
    assert lib.gp_scan_counts(P(torch.from_numpy(counts).cuda()), n, P(offs), s) == 0
    assert (offs.cpu().numpy() == numpy.concatenate([[0], numpy.cumsum(counts, dtype=numpy.int64)])).all()

    for B in (1, 7, 16):
        X = rng.randn(n, B)
        dX = torch.from_numpy(X).cuda()
        Y = torch.empty_like(dX)
        assert lib.gp_gather_rows(P(dX), P(order), n, B, P(Y), s) == 0
        assert (Y.cpu().numpy() == X[want]).all()
    assert lib.gp_gather_rows(P(dX), P(order), n, B, P(dX), s) == -1               # in place is refused

    for d in (1, 2, 3, 8):
        pts = rng.randn(n, d)
        box = numpy.empty(2 * d)
        bws = torch.empty(148 * 2 * d + 2 * d, dtype=torch.float64, device='cuda')
        assert lib.gp_points_bbox(P(torch.from_numpy(pts).cuda()), n, d, dev.host_ptr(box), P(bws), s) == 0
        assert (box[:d] == pts.min(axis=0)).all() and (box[d:] == pts.max(axis=0)).all()


def test_row_slab_engine_on_one_rank_equals_sparse_engine(sparse_problem):
    """gaussian_proc/_slab.py with a group of one: the peer-gather SpMM (owner-encoded block columns, exchange vectors in the
    arena), the slab Lanczos / CG drivers and the Gram all-reduce entry run on this GPU and must reproduce SparseEngine
    (same kernels apart from the gather address; the multi-rank check is tools/gpu_check_sparse_slab.py under torchrun)."""
    from gaussian_proc._sparse import SparseEngine
    from gaussian_proc._slab import SlabSparseEngine, slab_geometry
    pts, z, X, K = sparse_problem
    opts = {'seed': 3, 'lanczos_degree': 40, 'overlap': False}
    one = SparseEngine(K, 'slq', dict(opts))
    slab = SlabSparseEngine(K, 'slq', dict(opts), rank=0, world=1)
    assert slab.rows == K.n and slab.halo_fraction == 0.0
    assert slab_geometry(K.n, 1, 0)[1:] == (0, K.n)
    f1 = one.fused(2.0, X, z, cubic=True)
    f2 = slab.fused(2.0, X, z, cubic=True)
    assert numpy.max(numpy.abs(f1 - f2) / numpy.maximum(numpy.abs(f1), 1e-300)) <= 1e-12
    y = numpy.random.RandomState(0).randn(K.n, 3)
    assert numpy.max(numpy.abs(one.solve(2.0, y) - slab.solve(2.0, y))) <= 1e-12 * numpy.abs(y).max()
    assert numpy.max(numpy.abs(one.matmul(y) - slab.matmul(y))) <= 1e-12 * numpy.abs(y).max()


@pytest.mark.parametrize('n,d,scale,nu,dens', [(3000, 2, [0.03, 0.03], 0.5, 0.01), (3000, 2, [0.03, 0.03], 2.5, 0.01),
                                               (1000, 3, [0.2, 0.3, 0.25], 1.5, 0.02), (700, 2, [0.02, 0.05], 1.5, 0.02),
                                               (300, 1, [0.02], 0.5, 0.05), (13, 2, [0.5, 0.5], 2.5, 0.5),
                                               (2400, 2, [0.3, 0.3], 0.5, 0.9), (20011, 2, [0.02, 0.02], 0.5, 0.003)])
def test_direct_row_block_generation_equals_the_csr_generator(gp, n, d, scale, nu, dens):
    """generate_sparse_operator (row blocks straight from the cell lists, csrc/gp_sparse.cu sparse_blocks_kernel) holds exactly
    the matrix of the CSR generator - which the tests above pin bit-for-bit to the reference: same pattern, same values
    (same device arithmetic per entry), same dK/drho values where the scale is isotropic; nnz is counted by the count pass."""
    from gaussian_proc._sparse import generate_sparse_operator, generate_sparse_correlation, DeviceRowBlocks
    numpy.random.seed(n + d)
    pts = numpy.random.rand(n, d)
    iso = len(set(scale)) == 1
    Kd = generate_sparse_correlation(pts, numpy.array(scale), nu, dens, device=True, with_derivative=iso)
    S = Kd.to_scipy()
    Kb = generate_sparse_operator(pts, numpy.array(scale), nu, dens, with_derivative=iso)
    assert isinstance(Kb, DeviceRowBlocks) and Kb.nnz == S.nnz
    assert Kb.kernel_threshold == Kd.kernel_threshold
    B = Kb.to_scipy()
    assert (B.indptr == S.indptr).all() and (B.indices == S.indices).all()
    assert (B.data == S.data).all()
    assert (numpy.diff(Kb.bptr.cpu().numpy()) % 4 == 0).all()
    if iso:
        Kd.canonicalize()
        vals, Kb.bvals = Kb.bvals, Kb.bdvals          # the same reconstruction on the derivative values
        D = Kb.to_scipy()
        Kb.bvals = vals
        ref = scipy.sparse.csr_matrix((Kd.ddata.cpu().numpy(), Kd.indices.cpu().numpy(), Kd.indptr.cpu().numpy()), shape=S.shape)
        ref.eliminate_zeros()                         # (the diagonal and duplicate points have derivative exactly 0)
        assert (D.indptr == ref.indptr).all() and (D.indices == ref.indices).all() and (D.data == ref.data).all()


def test_direct_row_block_generation_falls_back_on_exact_ties_and_feeds_the_engine(gp, sparse_problem):
    from gaussian_proc._sparse import generate_sparse_operator, SparseEngine, DeviceCSR, DeviceRowBlocks
    from gaussian_proc._mixed_correlation import MixedCorrelation
    # a regular grid with the threshold placed exactly on a lattice distance: those pairs sit inside the 8-ulp band, which
    # the reference's rule decides in host arithmetic -> the CSR path
    from oracle import matern
    pts = grid_points()
    sc = numpy.array([0.03, 0.03])
    x = matern.scaled_distance_matrix(pts[[0, 2]], sc)[0, 1]
    tau = float(matern.matern_kernel(x, 0.5))                 # the kernel value of a lattice distance, to the last bit
    K = generate_sparse_operator(pts, sc, 0.5, 0.01, kernel_threshold=tau)
    assert isinstance(K, DeviceCSR)
    R = matern.generate_sparse_correlation(pts, sc, 0.5, 0.01, kernel_threshold=tau)
    S = K.to_scipy()
    assert (S.indptr == R.indptr).all() and (S.indices == R.indices).all()
    # the engine on the directly generated operator = the engine on the CSR-built one
    p, z, X, Kd = sparse_problem
    Kb = generate_sparse_operator(p, numpy.array([0.03, 0.03]), 0.5, 0.01, with_derivative=True)
    assert isinstance(Kb, DeviceRowBlocks)
    opts = {'seed': 3, 'lanczos_degree': 40}
    f1 = SparseEngine(Kd, 'slq', dict(opts)).fused(2.0, X, z)
    f2 = SparseEngine(Kb, 'slq', dict(opts)).fused(2.0, X, z)
    assert numpy.max(numpy.abs(f1 - f2) / numpy.maximum(numpy.abs(f1), 1e-300)) <= 1e-11
    Km = MixedCorrelation(Kb, imate_method='slq', imate_options=opts)
    y = numpy.random.RandomState(1).randn(Kb.n)
    assert numpy.max(numpy.abs(Km.dot(0.0, y) - Kd.to_scipy() @ y)) <= 1e-12 * numpy.abs(y).max() * 50
    from gaussian_proc._slab import SlabSparseEngine
    Ks = generate_sparse_operator(p, numpy.array([0.03, 0.03]), 0.5, 0.01, with_derivative=True, row_slab=(0, 1))
    f3 = SlabSparseEngine(Ks, 'slq', dict(opts), rank=0, world=1).fused(2.0, X, z)
    assert numpy.max(numpy.abs(f1 - f3) / numpy.maximum(numpy.abs(f1), 1e-300)) <= 1e-11
