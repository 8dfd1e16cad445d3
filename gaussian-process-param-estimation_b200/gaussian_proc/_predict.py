"""
Prediction at new points (kriging) on the dense device path, for the model the package fits:
z ~ N(X beta, sigma^2 K + sigma0^2 I), eta = sigma0^2 / sigma^2, Kn = K + eta I, beta by generalised least squares.

For a test point with correlation vector k* (against the training points) and basis row x*:
    B = X^T Kn^-1 X,  beta^ = B^-1 X^T Kn^-1 z,  alpha = Kn^-1 (z - X beta^)
    mean  = x*^T beta^ + k*^T alpha
    var   = sigma^2 (1 - ||L^-1 k*||^2 + r^T B^-1 r),  r = x* - X^T Kn^-1 k*       (+ sigma0^2 with noise=True)
    cov   = sigma^2 (K** - V^T V + R^T B^-1 R),        V = L^-1 [k*_1 ...],  R = [r_1 ...]

Device work per chunk of test points (csrc/gp_matern.cu, csrc/gp_predict.cu): the cross block P is generated, V = W P with
W = inv(L) (cached by the DenseEngine), and one pass reduces P^T S (S = Kn^-1 [X z]) and the column norms of V. The m x m
algebra runs on the host from that small result. The covariance adds two GEMMs over the whole test set.
"""

import ctypes
import math

import numpy

from . import _device as dev
from ._device import lib, check

__all__ = ['Predictor']

_KR_FULL, _TM_LOWER = 0, 1          # csrc/gp_internal.h


def _p(t, offset=0):
    return ctypes.c_void_p(t.data_ptr() + 8 * offset)


class Predictor(object):
    """Kriging predictor on the dense ``DeviceCorrelation`` of a ``MixedCorrelation`` at fixed ``eta``.

    ``sigma=None`` uses the profiled sigma^ = sqrt(z^T M z / (n - m)). The factor of K + eta I and its triangular inverse
    are the engine's cached ones (``DenseEngine.factor`` / ``_trtri``)."""

    def __init__(self, K_mixed, X, z, eta, sigma=None):
        if getattr(K_mixed, 'sparse', False):
            raise NotImplementedError('prediction is available for a dense correlation matrix only (a sparse K would '
                                      'need one Krylov solve per test point).')
        K = K_mixed.K
        if not K.has_kernel():
            raise ValueError('prediction needs the points, correlation_scale and nu behind K: generate K with '
                             'generate_correlation(..., device=True), or call MixedCorrelation.set_kernel(points, '
                             'correlation_scale, nu) on the operator built from a plain array.')
        eta = float(eta)
        if not (math.isfinite(eta) and eta >= 0.0):
            raise ValueError('eta must be finite and non-negative for prediction, got %r.' % eta)
        X = numpy.asarray(X, dtype=numpy.float64)
        z = numpy.asarray(z, dtype=numpy.float64).reshape(-1)
        n = K.n
        if X.ndim != 2 or X.shape[0] != n or z.shape[0] != n:
            raise ValueError('X must be (n, m) and z (n,) with n = %d training points.' % n)
        m = X.shape[1]
        p = m + 1
        if p > 16:
            raise ValueError('at most 15 basis functions are supported, got %d.' % m)
        torch = dev.torch
        self.K_mixed, self.K, self.engine = K_mixed, K, K_mixed.engine
        self.n, self.npad, self.m, self.p, self.eta = n, K.npad, m, p, eta
        self.d = int(K.points.shape[1])

        # S = Kn^-1 [X z] and G = [X z]^T S: B, beta^ and z^T M z
        eng = self.engine
        eng.factor(eta)
        R, _ = eng.pad_rhs(numpy.c_[X, z])
        S = R.clone()
        s = dev.stream_ptr()
        check(lib.gp_potrs_f64(_p(eng.A), self.npad, _p(eng.potrf_ws), _p(S), p, p, s), 'gp_potrs_f64')
        G = torch.empty(p * p, dtype=torch.float64, device='cuda')
        gws = torch.empty(lib.gp_gram_workspace_bytes(16) // 8, dtype=torch.float64, device='cuda')
        check(lib.gp_gram_skinny(_p(R), _p(S), n, p, _p(G), _p(gws), s), 'gp_gram_skinny')
        G = G.cpu().numpy().reshape(p, p)
        self.S = S
        self.B = G[:m, :m]
        self.beta = numpy.linalg.solve(self.B, G[:m, m])
        zMz = float(G[m, m] - G[:m, m] @ self.beta)
        self.sigma = math.sqrt(zMz / (n - m)) if sigma is None else float(sigma)

    def predict(self, test_points, X_test, return_var=True, return_cov=False, noise=False, chunk_size=8192):
        """Mean at the test points (rows of ``test_points``, basis rows ``X_test``), plus the variance and the covariance
        when asked: returns ``mean``, ``(mean, var)``, ``(mean, cov)`` or ``(mean, var, cov)``. ``noise=True`` adds the
        nugget sigma0^2 = sigma^2 eta (the variance of a new observation rather than of the latent value). Test points
        are processed ``chunk_size`` at a time; the results do not depend on it. The covariance is formed over the whole
        test set in one pass. A variance that cancellation pushed below zero is returned as 0."""
        torch = dev.torch
        K, eng = self.K, self.engine
        n, npad, m, p, d = self.n, self.npad, self.m, self.p, self.d
        tp = numpy.ascontiguousarray(test_points, dtype=numpy.float64)
        Xs = numpy.asarray(X_test, dtype=numpy.float64)
        if tp.ndim != 2 or tp.shape[1] != d:
            raise ValueError('test_points must be (m*, %d) like the training points, got shape %s.' % (d, tp.shape))
        ms = tp.shape[0]
        if Xs.ndim != 2 or Xs.shape != (ms, m):
            raise ValueError('X_test must be (%d, %d): one row per test point, one column per basis function; got %s.'
                             % (ms, m, Xs.shape))
        if ms == 0:
            raise ValueError('no test points.')
        if int(chunk_size) < 1:
            raise ValueError('chunk_size must be positive.')
        chunk = ms if return_cov else min(int(chunk_size), ms)
        mcpad = dev.padded_size(chunk)
        s = dev.stream_ptr()
        eng._trtri(self.eta)              # factor of K + eta I and W = inv(L), cached per eta
        f64 = torch.float64
        qd = torch.from_numpy(tp).cuda()
        P = torch.empty((npad, mcpad), dtype=f64, device='cuda')
        V = torch.empty((npad, mcpad), dtype=f64, device='cuda')
        ws = torch.empty(lib.gp_predict_workspace_bytes(npad, chunk, p) // 8, dtype=f64, device='cuda')
        out = torch.empty(chunk * (p + 1), dtype=f64, device='cuda')
        scale, nu = K.correlation_scale, float(K.nu)
        o = numpy.empty((ms, p + 1))
        for c0 in range(0, ms, chunk):
            mc = min(chunk, ms - c0)
            check(lib.gp_matern_cross_points(_p(K.points), n, _p(qd, c0 * d), mc, d, dev.host_ptr(scale), nu, _p(P), mcpad,
                                             s), 'gp_matern_cross_points')
            check(lib.gp_predict_dense(_p(eng.W), n, npad, _p(self.S), p, _p(P), mc, mcpad, _p(V), mcpad, _p(out), _p(ws),
                                       s), 'gp_predict_dense')
            o[c0:c0 + mc] = out[:mc * (p + 1)].cpu().numpy().reshape(mc, p + 1)

        kS = o[:, :m]                                 # (X^T Kn^-1 k*)^T
        mean = Xs @ self.beta + (o[:, m] - kS @ self.beta)
        r = Xs - kS                                   # rows r^T
        Br = numpy.linalg.solve(self.B, r.T)          # B^-1 r, one column per test point
        sigma2 = self.sigma ** 2
        nugget = sigma2 * self.eta if noise else 0.0
        res = [mean]
        if return_var:
            var = sigma2 * (1.0 - o[:, p] + numpy.einsum('ij,ji->i', r, Br)) + nugget
            res.append(numpy.maximum(var, 0.0))
        if return_cov:
            C = torch.empty((mcpad, mcpad), dtype=f64, device='cuda')
            check(lib.gp_matern_dense(_p(qd), ms, d, dev.host_ptr(scale), nu, _p(C), mcpad, None, s), 'gp_matern_dense')
            check(lib.gp_dgemm_f64(1, 1, _p(C), mcpad, _p(V), mcpad, _p(V), mcpad, mcpad, mcpad, npad, -1.0, 1.0, _KR_FULL,
                                   _TM_LOWER, s), 'gp_dgemm_f64')
            Rt = torch.zeros((32, mcpad), dtype=f64, device='cuda')
            BRt = torch.zeros((32, mcpad), dtype=f64, device='cuda')
            Rt[:m, :ms] = torch.from_numpy(numpy.ascontiguousarray(r.T))
            BRt[:m, :ms] = torch.from_numpy(numpy.ascontiguousarray(Br))
            check(lib.gp_dgemm_f64(1, 1, _p(C), mcpad, _p(Rt), mcpad, _p(BRt), mcpad, mcpad, mcpad, 32, 1.0, 1.0, _KR_FULL,
                                   _TM_LOWER, s), 'gp_dgemm_f64')
            Cl = torch.tril(C[:ms, :ms])
            cov = (Cl + torch.tril(Cl, -1).T) * sigma2
            if noise:
                cov.diagonal().add_(nugget)
            res.append(cov.cpu().numpy())
        return res[0] if len(res) == 1 else tuple(res)
