"""TEST INFRASTRUCTURE: NumPy implementation of the `ops` interface of gaussian_proc/_blockcyclic.py so that the
distributed algorithm (ownership, look-ahead order, broadcasts, staircase k ranges, reductions) can be exercised on CPU
with the gloo backend. Storage = torch CPU float64 tensors (gloo collectives work on them); streams / events are no-ops."""

import contextlib

import numpy
import torch


def _matern(x, nu, inv_rho=None):
    if nu == 0.5:
        K = numpy.exp(-x)
        dK = None if inv_rho is None else x * inv_rho * numpy.exp(-x)
    elif nu == 1.5:
        s3 = numpy.sqrt(3.0)
        K = (1 + s3 * x) * numpy.exp(-s3 * x)
        dK = None if inv_rho is None else 3.0 * x * x * inv_rho * numpy.exp(-s3 * x)
    else:
        s5 = numpy.sqrt(5.0)
        K = (1 + s5 * x + 5.0 / 3.0 * x ** 2) * numpy.exp(-s5 * x)
        dK = None if inv_rho is None else (5.0 / 3.0) * x * x * (1 + s5 * x) * inv_rho * numpy.exp(-s5 * x)
    return K, dK


class NumpyOps(object):
    def empty(self, shape):
        return torch.zeros(shape, dtype=torch.float64)

    zeros = empty

    def from_host(self, a, dtype=None):
        return torch.from_numpy(numpy.ascontiguousarray(a).copy())

    def int_tensor(self, values):
        return torch.tensor(list(values), dtype=torch.int32)

    def to_host(self, t):
        return t.numpy().copy()

    # streams / events: everything runs in program order on the CPU
    def new_stream(self):
        return None

    def use(self, stream):
        return contextlib.nullcontext()

    def event(self, stream=None, timing=False):
        return None

    def wait(self, stream, event):
        pass

    def elapsed_s(self, e0, e1):
        return 0.0

    def synchronize(self):
        pass

    def _dist(self, prow, pcol, scale):
        pr, pc = prow.numpy(), pcol.numpy()
        return numpy.sqrt((((pr[:, None, :] - pc[None, :, :]) / scale) ** 2).sum(-1))

    def generate(self, prow, pcol, rg, cg, n, scale, nu, eta, out):
        K = _matern(self._dist(prow, pcol, scale), nu)[0]
        gi, gj = rg.numpy()[:, None], cg.numpy()[None, :]
        K = numpy.where(gi == gj, 1.0 + eta, K)
        pad = (gi >= n) | (gj >= n)
        K = numpy.where(pad, (gi == gj).astype(float), K)
        out.copy_(torch.from_numpy(K))

    def generate_dk(self, prow, pcol, rg, cg, n, scale, nu, out):
        dK = _matern(self._dist(prow, pcol, scale), nu, 1.0 / scale[0])[1]
        gi, gj = rg.numpy()[:, None], cg.numpy()[None, :]
        dK = numpy.where((gi == gj) | (gi >= n) | (gj >= n), 0.0, dK)
        out.copy_(torch.from_numpy(dK))

    def potrf_inv(self, D, nvalid, Linv):
        try:
            L = numpy.linalg.cholesky(D.numpy())
        except numpy.linalg.LinAlgError:
            Linv.zero_()
            return torch.ones(1, dtype=torch.int32)
        D.copy_(torch.from_numpy(L))
        Linv.copy_(torch.from_numpy(numpy.linalg.inv(L)))
        return torch.zeros(1, dtype=torch.int32)

    def gemm(self, C, A, B, alpha, beta, at=0, bt=0, kbeg=None, kend=None):
        Am = A.numpy() if at == 0 else A.numpy().T          # M x K
        Bm = B.numpy().T if bt == 0 else B.numpy()          # K x N
        M, K = Am.shape
        assert M % 128 == 0 and C.shape[1] % 128 == 0 and K % 32 == 0 and Bm.shape == (K, C.shape[1])
        # gp_dgemm_ktab_f64 takes table entries that are multiples of its 16-wide k-slab (include/gpgp.h)
        for tab in (kbeg, kend):
            assert tab is None or all(int(v) % 16 == 0 for v in tab), 'k tables must hold multiples of 16'
        prod = numpy.zeros((M, C.shape[1]))
        for t in range(M // 128):
            kb = 0 if kbeg is None else min(int(kbeg[t]), K)
            ke = K if kend is None else min(int(kend[t]), K)
            if ke > kb:
                prod[128 * t:128 * t + 128] = Am[128 * t:128 * t + 128, kb:ke] @ Bm[kb:ke]
        C.copy_(torch.from_numpy(beta * C.numpy() + alpha * prod))

    def logdet_chol(self, D, nvalid, out):
        out[0] = float(2.0 * numpy.sum(numpy.log(numpy.diag(D.numpy())[:nvalid])))

    def rect_apply(self, X, R, Y, alpha=1.0, beta=0.0):
        Y.copy_(torch.from_numpy(alpha * (X.numpy() @ R.numpy()) + beta * Y.numpy()))

    def rect_apply_t(self, X, Y, S, alpha=1.0, beta=0.0):
        S.copy_(torch.from_numpy(alpha * (X.numpy().T @ Y.numpy()) + beta * S.numpy()))

    def pair_dot(self, A, B, rows_w1, w_rest, accum):
        a, b = A.numpy(), B.numpy()
        accum[0] += float(numpy.sum(a[:rows_w1] * b[:rows_w1]) + w_rest * numpy.sum(a[rows_w1:] * b[rows_w1:]))

    def dk_apply(self, points, n, scale, nu, S, V):
        dK = _matern(self._dist(points, points, scale), nu, 1.0 / scale[0])[1]
        numpy.fill_diagonal(dK, 0.0)
        V.zero_()
        V[:n] = torch.from_numpy(dK @ S.numpy()[:n])
