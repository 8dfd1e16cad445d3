"""
Host-side (m+1)x(m+1) algebra on top of the fused device evaluator (dense: csrc/gp_loglik.cu, `gp_loglik_dense`;
sparse: `SparseEngine.fused`, batched CG + skinny Gram matrices + stochastic traces, same out[] layout).

With R = [X z], S = Kn^-1 R and the device outputs G = R^T S, H = S^T S, Q = S^T dK S the quantities of the reference
formulas follow without touching n-sized data again (M = Kn^-1 - Kn^-1 X (X^T Kn^-1 X)^-1 X^T Kn^-1, c = [-beta; 1]):
    B = G[:m,:m]            beta = B^-1 G[:m,m]          z^T M z   = G[m,m] - G[:m,m].beta
    z^T M^2 z = c^T H c     z^T M K M z = c^T (G - eta H) c          z^T M dK M z = c^T Q c
    tr M = tr Kn^-1 - tr(B^-1 H[:m,:m])                  tr(M dK) = tr(Kn^-1 dK) - tr(B^-1 Q[:m,:m])
(reference: _direct_likelihood.py:113-150, _profile_likelihood.py:104-130.)
"""

import numpy

from .. import _device as dev
from .._dense import FLAG_TRACEINV, FLAG_INVERSE, FLAG_DRHO, FLAG_CUBIC

__all__ = ['FusedQuantities', 'evaluate', 'evaluate_async', 'finish']


class FusedQuantities(object):
    """Unpacked result of one fused evaluation at a given eta (all host floats / small arrays)."""

    def __init__(self, out, n, m, eta, flags, dscale=None):
        p = m + 1
        self.n, self.m, self.eta, self.flags = n, m, eta, flags
        self.logdet_Kn = float(out[0])
        self.trace_Kninv = float(out[1])
        self.trace_Kninv2 = float(out[2])
        self.trace_Kninv_dK = float(out[3])
        self.info = int(out[4])
        G = out[8:8 + p * p].reshape(p, p)
        H = out[8 + p * p:8 + 2 * p * p].reshape(p, p)
        Q = out[8 + 2 * p * p:8 + 3 * p * p].reshape(p, p)
        self.G, self.H, self.Q = G, H, Q
        self.B = G[:m, :m]
        self.Binv = numpy.linalg.inv(self.B)
        self.beta = self.Binv @ G[:m, m]
        self.c = numpy.append(-self.beta, 1.0)
        self.zMz = float(G[m, m] - G[:m, m] @ self.beta)
        self.zM2z = float(self.c @ H @ self.c)
        self.zMKMz = float(self.c @ (G - eta * H) @ self.c)
        self.zMdKMz = float(self.c @ Q @ self.c)
        self.trace_M = self.trace_Kninv - float(numpy.trace(self.Binv @ H[:m, :m]))
        self.trace_MdK = self.trace_Kninv_dK - float(numpy.trace(self.Binv @ Q[:m, :m]))
        # anisotropic correlation scale: per-dimension tr(M dK_k) and z^T M dK_k M z (rows of `dscale`: [trace, Q_k])
        self.trace_MdK_dims = self.zMdKMz_dims = None
        if dscale is not None:
            self.trace_MdK_dims = numpy.array([row[0] - numpy.trace(self.Binv @ row[1:].reshape(p, p)[:m, :m]) for row in dscale])
            self.zMdKMz_dims = numpy.array([self.c @ row[1:].reshape(p, p) @ self.c for row in dscale])
        # third moments (flag CUBIC): T3 = R^T Kn^-3 R. With u = M z = S c:  M u = Kn^-1 u - S_X B^-1 (S_X^T u), hence
        #   z^T M^3 z = c^T T3 c - (H_x c)^T B^-1 (H_x c),   tr M^2 = tr Kn^-2 - 2 tr(B^-1 T3_xx) + tr((B^-1 H_xx)^2)
        self.zM3z = self.trace_M2 = None
        if out.shape[0] >= 8 + 4 * p * p and (flags == -1 or (flags >= 0 and (flags & FLAG_CUBIC))):
            T3 = out[8 + 3 * p * p:8 + 4 * p * p].reshape(p, p)
            self.T3 = T3
            hx = H[:m, :] @ self.c
            self.zM3z = float(self.c @ T3 @ self.c - hx @ self.Binv @ hx)
            BH = self.Binv @ H[:m, :m]
            self.trace_M2 = self.trace_Kninv2 - 2.0 * float(numpy.trace(self.Binv @ T3[:m, :m])) + float(numpy.trace(BH @ BH))

    def moments(self):
        """(t, s): t[k] = tr M^k (k = 1, 2), s[k] = z^T M^k z (k = 1, 2, 3) of the projected precision
        M = Kn^-1 - Kn^-1 X B^-1 X^T Kn^-1 at this eta (index 0 unused) - what every derivative up to second order is
        made of (_direct_likelihood.py:163-270, _profile_likelihood.py:138-192)."""
        if self.zM3z is None:
            raise ValueError('third moments were not requested (cubic=True)')
        return (None, self.trace_M, self.trace_M2), (None, self.zMz, self.zM2z, self.zM3z)

    def set_trace_Kninv(self, value):
        """tr Kn^-1 supplied from outside (the interpolated trace of a MixedCorrelation(interpolate=True))"""
        self.trace_Kninv = float(value)
        self.trace_M = self.trace_Kninv - float(numpy.trace(self.Binv @ self.H[:self.m, :self.m]))


def _rhs_device(K_mixed, X, z):
    """[X z] zero-padded on the device, cached on the operator while X and z are the same objects."""
    key = (dev.host_key(X), dev.host_key(z))
    cache = getattr(K_mixed, '_rhs_cache', None)
    if cache is not None and cache[0] == key:
        return cache[1]
    R = numpy.c_[numpy.asarray(X, dtype=float), numpy.asarray(z, dtype=float)]
    Rd, _ = K_mixed.engine.pad_rhs(R)
    K_mixed._rhs_cache = (key, Rd, X, z)  # keep X, z alive so the ids stay unique
    return Rd


def evaluate_async(z, X, K_mixed, eta, traceinv=False, inverse=False, drho=False, cubic=False):
    """Enqueues one fused evaluation on torch's current stream and returns a handle without synchronising; several
    evaluations on different streams / operators can be in flight (see sweep.py). Complete it with finish()."""
    n, m = X.shape
    if K_mixed.sparse:
        # sparse K: batched CG solves + skinny Gram matrices + the engine's stochastic traces (synchronous)
        out = K_mixed.engine.fused(float(eta), X, z, traceinv=traceinv or inverse or cubic, drho=drho, cubic=cubic)
        return (out, n, m, float(eta), -1 if cubic else -2, None, K_mixed.engine.last_dscale)
    flags = 0
    if traceinv:
        flags |= FLAG_TRACEINV
    if inverse or drho:
        flags |= FLAG_INVERSE
    if drho:
        flags |= FLAG_DRHO
    if cubic:
        flags |= FLAG_CUBIC | FLAG_INVERSE         # tr Kn^-2 comes with the explicit inverse
    Rd = _rhs_device(K_mixed, X, z)
    dscale = None
    if getattr(K_mixed, 'imate_method', None) == 'eigenvalue':
        # one eigendecomposition per matrix, O(n^2 p) per eta (the reference's default method, likelihood.py:41)
        out = K_mixed.eigen_engine().fused(float(eta), Rd, m + 1, flags)
    else:
        out = K_mixed.engine.fused(float(eta), Rd, m + 1, flags)
        dscale = K_mixed.engine.last_dscale
    return (out, n, m, float(eta), flags, dev.torch.cuda.current_stream(), dscale)


def finish(handle):
    """Waits for the evaluation's stream, reads out[] back (one small D2H) and does the host algebra; raises
    numpy.linalg.LinAlgError if K + eta I was not positive definite."""
    out, n, m, eta, flags, stream, dscale = handle
    if stream is None:       # sparse engine: already complete, breakdowns raised there; dscale a host array
        return FusedQuantities(out, n, m, eta, flags, dscale)
    stream.synchronize()
    q = FusedQuantities(out.cpu().numpy(), n, m, eta, flags, None if dscale is None else dscale.cpu().numpy())
    if q.info != 0:
        raise numpy.linalg.LinAlgError(
            '%d-th leading minor of K + eta*I (eta=%g) is not positive definite.' % (q.info, eta))
    return q


def evaluate(z, X, K_mixed, eta, traceinv=False, inverse=False, drho=False, cubic=False):
    """Runs the fused evaluator once; raises numpy.linalg.LinAlgError if K + eta I is not positive definite.
    With MixedCorrelation(interpolate=True) the trace of the inverse is the interpolated one
    (mixed_correlation.py:167-170) and the evaluation skips the inverse it would otherwise need for it."""
    if traceinv and getattr(K_mixed, 'interpolate', False) and not (inverse or drho or cubic):
        q = finish(evaluate_async(z, X, K_mixed, eta, traceinv=False))
        q.set_trace_Kninv(K_mixed.traceinv(eta))
        return q
    return finish(evaluate_async(z, X, K_mixed, eta, traceinv=traceinv, inverse=inverse, drho=drho, cubic=cubic))
