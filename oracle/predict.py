"""TEST INFRASTRUCTURE. CPU reference for prediction at new points (kriging), the model of gaussian_proc/_predict.py:
z ~ N(X beta, sigma^2 (K + eta I)), beta by generalised least squares. SciPy Cholesky formulas on K, the cross block P and
K** built from the oracle's Matern kernel (oracle/matern.py)."""

import numpy
import scipy.linalg

from . import matern

__all__ = ['cross_correlation', 'predict', 'bordered_predict']


def cross_correlation(points, test_points, correlation_scale, nu):
    """P[i][j] = matern(||(p_i - q_j) / scale||, nu): the off-diagonal block of the correlation of the stacked point set
    (the oracle's dense generator, same k-ordered distance)."""
    n = points.shape[0]
    Kall = matern.generate_dense_correlation(numpy.r_[points, test_points], correlation_scale, nu)
    return numpy.ascontiguousarray(Kall[:n, n:])


def predict(points, z, X, test_points, X_test, correlation_scale, nu, eta, sigma=None, noise=False):
    """(mean, var, cov, sigma) at the test points. sigma=None: the profiled sigma^2 = z^T M z / (n - m)."""
    n, m = X.shape
    K = matern.generate_dense_correlation(points, correlation_scale, nu)
    P = cross_correlation(points, test_points, correlation_scale, nu)
    Kss = matern.generate_dense_correlation(test_points, correlation_scale, nu)
    c = scipy.linalg.cho_factor(K + eta * numpy.eye(n), lower=True)
    KiX = scipy.linalg.cho_solve(c, X)
    B = X.T @ KiX
    beta = numpy.linalg.solve(B, KiX.T @ z)
    alpha = scipy.linalg.cho_solve(c, z - X @ beta)
    if sigma is None:
        sigma = numpy.sqrt(z @ alpha / (n - m))
    mean = X_test @ beta + P.T @ alpha
    L = numpy.tril(c[0])
    v = scipy.linalg.solve_triangular(L, P, lower=True)
    r = X_test.T - KiX.T @ P
    Br = numpy.linalg.solve(B, r)
    nugget = sigma ** 2 * eta if noise else 0.0
    var = sigma ** 2 * (1.0 - numpy.sum(v * v, axis=0) + numpy.sum(r * Br, axis=0)) + nugget
    cov = sigma ** 2 * (Kss - v.T @ v + r.T @ Br) + nugget * numpy.eye(len(mean))
    return mean, var, cov, sigma


def bordered_predict(K, P, X, z, X_test, eta):
    """An independent formulation: the bordered kriging system [[Kn, X], [X^T, 0]] [w; lam] = [k*; x*] gives
    mean = w^T z and var / sigma^2 = 1 - w^T k* - lam^T x* (unit diagonal K)."""
    n, m = X.shape
    A = numpy.block([[K + eta * numpy.eye(n), X], [X.T, numpy.zeros((m, m))]])
    sol = numpy.linalg.solve(A, numpy.r_[P, X_test.T])
    w, lam = sol[:n], sol[n:]
    return w.T @ z, 1.0 - numpy.sum(w * P, axis=0) - numpy.sum(lam * X_test.T, axis=0)
