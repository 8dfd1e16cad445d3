"""CPU tests that PIN the oracle: the restatement in oracle/ against
  (A) numbers from the reference's shipped pickles (tests/golden/golden_pickles.npz),
  (B) vectors produced by the reference's own Python modules (tests/golden/golden_likelihood.npz),
  (C) matrices produced by the reference's compiled Cython generators (tests/golden/golden_generate.npz)."""

import os

import numpy
import pytest

from oracle import data_utilities as du
from oracle import likelihood as L
from oracle import matern


def rel(a, b):
    a, b = numpy.asarray(a, dtype=float), numpy.asarray(b, dtype=float)
    return float(numpy.max(numpy.abs(a - b)) / max(numpy.max(numpy.abs(b)), 1e-300))


# ---- (C) generators -----------------------------------------------------------------------------------------
@pytest.mark.parametrize('nu', [0.5, 1.5, 2.5, 200.0])
def test_dense_closed_form_bit_identical(golden_generate, nu):
    K = matern.generate_dense_correlation(golden_generate['points2d'], numpy.array([0.1, 0.17]), nu)
    assert (K == golden_generate['dense_nu%g' % nu]).all()


@pytest.mark.parametrize('nu', [3.3, 0.8])
def test_dense_bessel_branch(golden_generate, nu):
    K = matern.generate_dense_correlation(golden_generate['points2d'], numpy.array([0.1, 0.17]), nu)
    assert numpy.max(numpy.abs(K - golden_generate['dense_nu%g' % nu])) <= 1e-14


def test_dense_3d(golden_generate):
    K = matern.generate_dense_correlation(golden_generate['points3d'], numpy.array([0.2, 0.3, 0.25]), 1.5)
    assert (K == golden_generate['dense3d_nu1.5']).all()


@pytest.mark.parametrize('tag', ['rand', 'grid'])
@pytest.mark.parametrize('nu', [0.5, 1.5, 2.5])
def test_sparse_csr_bit_identical(golden_generate, tag, nu):
    pts = golden_generate['sparse_points'] if tag == 'rand' else du.generate_points(40, 2, grid=True)
    S = matern.generate_sparse_correlation(pts, numpy.array([0.03, 0.03]), nu, 0.01)
    key = 'sparse_%s_nu%g_' % (tag, nu)
    assert S.indices.dtype == numpy.int32 and S.indptr.dtype == numpy.int32
    assert (S.indptr == golden_generate[key + 'indptr']).all()
    assert (S.indices == golden_generate[key + 'indices']).all()
    assert (S.data == golden_generate[key + 'data']).all()


def test_sparse_density_too_small_raises():
    with pytest.raises(ValueError):
        matern.generate_sparse_correlation(numpy.random.rand(50, 2), 0.1, 0.5, 1e-3)   # density * n < 1


# ---- (B) likelihood vectors from the reference's own Python ---------------------------------------------------
@pytest.mark.parametrize('case', [0, 1, 2, 3, 4])
@pytest.mark.parametrize('method', ['eigenvalue', 'cholesky'])
def test_oracle_likelihood_equals_reference(golden_likelihood, case, method):
    g = golden_likelihood
    nu, rho = g['cases'][case]
    pts, z, X = g['points'], g['z'], g['X']
    K = matern.generate_dense_correlation(pts, numpy.array([rho, rho]), nu)
    Km = L.MixedCorrelation(K, method)
    tag = 'c%d_%s_' % (case, method)
    t = 1e-12 if case != 4 else 1e-6     # case 4 = Gaussian kernel, condition number ~1e12+
    for i, h in enumerate(g['hyper_direct']):
        assert rel(L.DirectLikelihood.log_likelihood(z, X, Km, False, list(h)), g[tag + 'direct_ll'][i]) <= t
        assert rel(L.DirectLikelihood.log_likelihood_jacobian(z, X, Km, False, list(h)), g[tag + 'direct_jac'][i]) <= t * 1e3
        assert rel(L.DirectLikelihood.log_likelihood_hessian(z, X, Km, False, list(h)), g[tag + 'direct_hess'][i]) <= t * 1e4
    for i, h in enumerate(g['hyper_profile']):
        assert rel(L.ProfileLikelihood.log_likelihood(z, X, Km, False, list(h)), g[tag + 'profile_ll'][i]) <= t
    for i, le in enumerate(g['log_etas']):
        assert rel(L.ProfileLikelihood.log_likelihood_der1_eta(z, X, Km, le), g[tag + 'profile_der1'][i]) <= t * 1e3
        assert rel(Km.logdet(10.0 ** le), g[tag + 'logdet'][i]) <= 1e-12
        assert rel(Km.traceinv(10.0 ** le), g[tag + 'traceinv'][i]) <= t * 1e3
    if method == 'eigenvalue' and not numpy.isnan(g[tag + 'root']).any():
        r = L.ProfileLikelihood.find_log_likelihood_der1_zeros(z, X, Km, [1e-4, 1e3])
        assert rel([r['sigma'], r['sigma0'], r['eta']], g[tag + 'root']) <= 1e-9


def test_identities_the_reference_satisfies(golden_likelihood):
    """SURVEY 8c: jacobian == FD of l in (sigma^2, sigma0^2); der1_eta == FD of profiled l in eta;
    direct - profile == -1/2 (n - m) log 2 pi."""
    g = golden_likelihood
    pts, z, X = g['points'], g['z'], g['X']
    n, m = X.shape
    Km = L.MixedCorrelation(matern.generate_dense_correlation(pts, 0.1, 1.5), 'cholesky')
    s, s0 = 0.3, 0.2
    jac = L.DirectLikelihood.log_likelihood_jacobian(z, X, Km, False, [s, s0])
    h = 1e-6
    f = lambda v, v0: L.DirectLikelihood.log_likelihood(z, X, Km, False, [numpy.sqrt(v), numpy.sqrt(v0)])  # noqa: E731
    fd = [(f(s * s + h, s0 * s0) - f(s * s - h, s0 * s0)) / (2 * h), (f(s * s, s0 * s0 + h) - f(s * s, s0 * s0 - h)) / (2 * h)]
    assert rel(jac, fd) <= 1e-6
    eta = (s0 / s) ** 2
    d = L.DirectLikelihood.log_likelihood(z, X, Km, False, [s, s0]) - L.ProfileLikelihood.log_likelihood(z, X, Km, False, [s, eta])
    assert abs(d - (-0.5 * (n - m) * numpy.log(2 * numpy.pi))) <= 1e-9

    def prof(e):
        sig = L.ProfileLikelihood.find_optimal_sigma(z, X, Km, e)
        return L.ProfileLikelihood.log_likelihood(z, X, Km, False, [sig, e])
    he = 1e-5
    fd_eta = (prof(eta + he) - prof(eta - he)) / (2 * he)
    assert rel(L.ProfileLikelihood.log_likelihood_der1_eta(z, X, Km, numpy.log10(eta)), fd_eta) <= 1e-6


def test_drho_extension_pinned_by_finite_differences(golden_likelihood):
    """The reference has no d/d rho (parity unpinned by the reference); pin the oracle's analytic formula to a
    Richardson-extrapolated central difference of the pinned log-likelihoods."""
    g = golden_likelihood
    pts, z, X = g['points'], g['z'], g['X']
    for nu in (0.5, 1.5, 2.5, 3.3):
        rho = 0.1

        def direct(r):
            return L.DirectLikelihood.log_likelihood(z, X, L.MixedCorrelation(matern.generate_dense_correlation(pts, r, nu)), False, [0.3, 0.2])

        def prof(r):
            Km = L.MixedCorrelation(matern.generate_dense_correlation(pts, r, nu))
            return L.ProfileLikelihood.log_likelihood(z, X, Km, False, [L.ProfileLikelihood.find_optimal_sigma(z, X, Km, 0.5), 0.5])
        Km = L.MixedCorrelation(matern.generate_dense_correlation(pts, rho, nu))
        dK = matern.matern_derivative_rho(pts, rho, nu)
        for fn, an in ((direct, L.DirectLikelihood.log_likelihood_der1_rho(z, X, Km, dK, [0.3, 0.2])),
                       (prof, L.ProfileLikelihood.log_likelihood_der1_rho(z, X, Km, dK, 0.5))):
            h = 1e-3
            d1 = (fn(rho + h) - fn(rho - h)) / (2 * h)
            d2 = (fn(rho + h / 2) - fn(rho - h / 2)) / h
            fd = (4 * d2 - d1) / 3
            assert rel(an, fd) <= 2e-7, (nu, an, fd)


def test_anisotropic_scale_derivative_pinned_by_finite_differences():
    """EXTENSION (anisotropic d/d correlation_scale[k]): the analytic per-dimension derivative equals Richardson finite
    differences of the pinned generator, and the per-dimension derivatives of an isotropic scale sum to d/d rho."""
    numpy.random.seed(8)
    pts = numpy.random.rand(60, 2)
    scale = numpy.array([0.12, 0.2])
    for nu in (0.5, 1.5, 2.5, 200.0, 3.3):
        for k in (0, 1):
            def Kof(h):
                s2 = scale.copy()
                s2[k] += h
                return matern.generate_dense_correlation(pts, s2, nu)
            h = 1e-4
            d1 = (Kof(h) - Kof(-h)) / (2 * h)
            d2 = (Kof(h / 2) - Kof(-h / 2)) / h
            fd = (4 * d2 - d1) / 3
            an = matern.matern_derivative_scale(pts, scale, nu, k)
            assert numpy.max(numpy.abs(an - fd)) <= 2e-8 * max(numpy.max(numpy.abs(an)), 1.0), (nu, k)
        iso = numpy.array([0.15, 0.15])
        tot = matern.matern_derivative_scale(pts, iso, nu, 0) + matern.matern_derivative_scale(pts, iso, nu, 1)
        assert numpy.max(numpy.abs(tot - matern.matern_derivative_rho(pts, 0.15, nu))) <= 1e-12 * numpy.max(numpy.abs(tot))


# ---- (A) shipped pickles -------------------------------------------------------------------------------------
def test_golden_pickle_cells(golden_pickles):
    pts = du.generate_points(30, 2, grid=True)
    z = du.generate_data(pts, 0.2)
    X = du.generate_basis_functions(pts, 2)
    assert X.shape == (900, 6)
    rng = numpy.random.RandomState(5)
    cells = [(0, 0), (60, 59), (0, 59), (60, 0)] + [(int(rng.randint(61)), int(rng.randint(60))) for _ in range(6)]
    for (i, j) in cells:
        rho, nu = golden_pickles['rho'][i], golden_pickles['nu'][j]
        Km = L.MixedCorrelation(matern.generate_dense_correlation(pts, rho, nu), 'eigenvalue')
        r = L.ProfileLikelihood.find_log_likelihood_der1_zeros(z, X, Km, [1e-3, 1e3])
        lp = L.ProfileLikelihood.log_likelihood(z, X, Km, False, [r['sigma'], r['eta']])
        assert abs(lp - golden_pickles['Lp_noprior'][i, j]) <= 5e-10
        prior = -2.0 * numpy.log(1.0 + rho) - 2.0 * numpy.log(1.0 + nu / 25.0)
        assert abs(lp + prior - golden_pickles['Lp_prior'][i, j]) <= 5e-9


def test_golden_noise_level_results(golden_pickles):
    pts = du.generate_points(50, 2, grid=True)
    X = du.generate_basis_functions(pts, 2)
    Km = L.MixedCorrelation(matern.generate_dense_correlation(pts, 0.1, 0.5), 'eigenvalue')
    for idx in (50, 120):   # finite-eta rows (row 199 is the eta -> inf fallback branch)
        noise = golden_pickles['noise_NoiseMagnitude'][idx]
        z = du.generate_data(pts, noise)
        r = L.ProfileLikelihood.find_log_likelihood_der1_zeros(z, X, Km, [1e-4, 1e3])
        got = numpy.array([r['sigma'], r['sigma0'], r['eta']])
        ref = numpy.array([golden_pickles['noise_sigma'][idx], golden_pickles['noise_sigma0'][idx], golden_pickles['noise_eta'][idx]])
        assert rel(got, ref) <= 1e-6


def test_slq_oracle_estimates_exact_traces():
    """oracle/slq.py (CPU restatement of the stochastic Lanczos quadrature, parity unpinned: imate absent): the mean over
    64 Rademacher probes lands within 3 standard errors of the exact logdet / trace of the inverse."""
    from oracle import slq, matern
    numpy.random.seed(1)
    pts = numpy.random.rand(400, 2)
    K = matern.generate_sparse_correlation(pts, numpy.array([0.05, 0.05]), 0.5, 0.05)
    eta = 2.0
    S = slq.slq_samples(K, eta, 0, 0, 64, 30)
    Kn = K.toarray() + eta * numpy.eye(400)
    Kinv = numpy.linalg.inv(Kn)
    exact = [numpy.linalg.slogdet(Kn)[1], numpy.trace(Kinv), numpy.sum(Kinv * Kinv)]
    for c in range(3):
        assert abs(S[:, c].mean() - exact[c]) <= 3.0 * S[:, c].std(ddof=1) / 8.0
    V = slq.rademacher(6, 2, 5, 3)
    assert set(numpy.unique(V)) <= {-1.0, 1.0} and V.shape == (6, 2)
