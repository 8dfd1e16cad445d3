"""Gradients of the kriging mean and variance with respect to the test-point coordinates: the device reduction
gp_predict_grad_dense on its own, and Predictor.predict_gradient / GaussianProcess.predict_gradient against a NumPy/SciPy
reference written out below (grad_reference) and against central differences of predict().

The unmarked tests run without a GPU: the reference against central differences of oracle.predict, its far-point
identities, the basis Jacobian, and argument validation of the new C entry points. The tests marked gpu need a CUDA
device."""

import ctypes
import json
import math
import os
import subprocess
import sys

import numpy
import pytest
import scipy.linalg
import scipy.special

gpu = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'gaussian-process-param-estimation_b200')
EPS = numpy.finfo(numpy.float64).eps
SENTINEL = numpy.array([0x7ff8dead0000beef], dtype=numpy.uint64).view(numpy.float64)[0]   # a NaN with a payload


def padded(n):
    return (n + 127) // 128 * 128


def problem(n, seed=0, d=2):
    from oracle import data_utilities as du
    rng = numpy.random.RandomState(seed)
    pts = rng.rand(n, d)
    return pts, du.generate_data(pts, 0.2), du.generate_basis_functions(pts, 2)


# ------------------------------------------------------------------------------------------------- host reference
def basis_jacobian(tp, degree=2):
    """d X[j] / d tp[j, k] (m*, d, m) of oracle.data_utilities.generate_basis_functions(tp, degree): the monomial
    prod_i q_i^e_i differentiates to e_k q_k^(e_k - 1) prod_{i != k} q_i^e_i (same column order as the generator)."""
    ms, dim = tp.shape
    grids = numpy.meshgrid(*([numpy.arange(degree + 1)] * dim))
    powers = numpy.array([g.ravel() for g in grids])
    powers = powers[:, powers.sum(axis=0) <= degree]
    J = numpy.zeros((ms, dim, powers.shape[1]))
    for c in range(powers.shape[1]):
        for k in range(dim):
            e = powers[k, c]
            if e == 0:
                continue
            t = e * tp[:, k] ** (e - 1)
            for i in range(dim):
                if i != k:
                    t = t * tp[:, i] ** powers[i, c]
            J[:, k, c] = t
    return J


def h_of_x(x, nu):
    """h(x) = -K'(x) / x of the Matern correlation K (the matern_mode_of branches), 0 at x == 0. General nu:
    coef 2 nu y^(nu-1) K_{nu-1}(y), y = sqrt(2 nu) x, with scipy.special.kv."""
    x = numpy.asarray(x, dtype=numpy.float64)
    h = numpy.zeros_like(x)
    nz = x > 0
    t = x[nz]
    if nu == 0.5:
        h[nz] = numpy.exp(-t) / t
    elif nu == 1.5:
        h[nz] = 3.0 * numpy.exp(-math.sqrt(3.0) * t)
    elif nu == 2.5:
        h[nz] = 5.0 / 3.0 * (1.0 + math.sqrt(5.0) * t) * numpy.exp(-math.sqrt(5.0) * t)
    elif nu >= 100:
        h[nz] = numpy.exp(-0.5 * t * t)
    else:
        y = math.sqrt(2.0 * nu) * t
        coef = 2.0 ** (1.0 - nu) / scipy.special.gamma(nu)
        h[nz] = coef * 2.0 * nu * y ** (nu - 1.0) * scipy.special.kv(nu - 1.0, y)
    return h


def cross_gradient(points, test_points, scale, nu):
    """G (d, n, m*): G[k][i, j] = dK(p_i, q_j) / dq_jk = h(x) (p_ik - q_jk) / scale_k^2; 0 for a pair at distance 0"""
    d = points.shape[1]
    scale = numpy.broadcast_to(numpy.asarray(scale, dtype=numpy.float64), (d,))
    diff = points[None, :, :] - test_points[:, None, :]                     # (m*, n, d): p_i - q_j
    x = numpy.sqrt(numpy.sum((diff / scale) ** 2, axis=2))
    h = h_of_x(x, nu)
    return numpy.transpose(h[:, :, None] * diff / scale ** 2, (2, 1, 0))


def grad_reference(points, z, X, test_points, X_test, X_test_grad, scale, nu, eta, sigma=None):
    """(mean_grad, var_grad, parts) of the model of oracle/predict.py, SciPy Cholesky on K + eta I:
        d mean / dq_k = (dx*/dq_k)^T beta + G_k^T alpha
        d var / dq_k  = sigma^2 (-2 (Kn^-1 k*)^T G_k + 2 (B^-1 r)^T (dx*/dq_k - X^T Kn^-1 G_k))
    parts carries the quantities the tolerances below are built from."""
    from oracle import matern, predict as op
    n, m = X.shape
    K = matern.generate_dense_correlation(points, scale, nu)
    P = op.cross_correlation(points, test_points, scale, nu)
    c = scipy.linalg.cho_factor(K + eta * numpy.eye(n), lower=True)
    KiX = scipy.linalg.cho_solve(c, X)
    Kiz = scipy.linalg.cho_solve(c, z)
    B = X.T @ KiX
    beta = numpy.linalg.solve(B, KiX.T @ z)
    alpha = scipy.linalg.cho_solve(c, z - X @ beta)
    if sigma is None:
        sigma = numpy.sqrt(z @ alpha / (n - m))
    U = scipy.linalg.cho_solve(c, P)
    r = X_test.T - KiX.T @ P
    Br = numpy.linalg.solve(B, r)
    G = cross_gradient(points, test_points, scale, nu)
    mean_grad = numpy.einsum('jkc,c->jk', X_test_grad, beta) + numpy.einsum('kij,i->jk', G, alpha)
    uG = numpy.einsum('kij,ij->jk', G, U)
    DX = numpy.einsum('kij,ic->jkc', G, KiX)
    var_grad = sigma ** 2 * (-2.0 * uG + 2.0 * numpy.einsum('jkc,cj->jk', X_test_grad - DX, Br))
    aG = numpy.abs(G)
    parts = {'sigma': sigma, 'beta': beta, 'B': B,
             # sum_i |G| (|Kn^-1 z| + |Kn^-1 X| |beta|): the size of the terms the mean gradient sums
             'mean_scale': numpy.einsum('kij,i->jk', aG, numpy.abs(Kiz) + numpy.abs(KiX) @ numpy.abs(beta)),
             # the same for the variance gradient's terms
             'var_scale': sigma ** 2 * (2.0 * numpy.einsum('kij,ij->jk', aG, numpy.abs(U)) + 2.0 * numpy.einsum(
                 'jkc,cj->jk', numpy.abs(X_test_grad) + numpy.einsum('kij,ic->jkc', aG, numpy.abs(KiX)), numpy.abs(Br)))}
    return mean_grad, var_grad, parts


def _grad_tol(n, eta):
    # like _var_tol of the prediction tests: S, U = Kn^-1 [...] carry about cond(Kn) eps <= (n / eta) eps of relative
    # rounding, which the sums over the training points pass on (relative to the size of their terms); never below 1e-9
    return max(1e-9, 10.0 * n / eta * EPS)


def central_difference(f, q, step):
    """(f(q + step e_k) - f(q - step e_k)) / (2 step) for every test point and dimension: (m*, d) per output of f"""
    ms, d = q.shape
    outs = None
    for k in range(d):
        e = numpy.zeros_like(q)
        e[:, k] = step
        fp, fm = f(q + e), f(q - e)
        cols = [(a - b) / (2.0 * step) for a, b in zip(fp, fm)]
        if outs is None:
            outs = [numpy.empty((ms, d)) for _ in cols]
        for o, c in zip(outs, cols):
            o[:, k] = c
    return outs


def fd_bound(f, q, step, rounding):
    """central differences at `step` and the bound on their distance from the derivative: the O(step^2) truncation term,
    step^2 f'''/6, is estimated by Richardson from the difference at 2 step (FD_2h - FD_h = 3 c h^2 + O(h^4)) and
    counted twice; `rounding` (per output, an absolute bound on one evaluation's error) adds rounding / step."""
    fd1 = central_difference(f, q, step)
    fd2 = central_difference(f, q, 2.0 * step)
    return [(a, 2.0 * numpy.abs(b - a) / 3.0 + r / step) for a, b, r in zip(fd1, fd2, rounding)]


# ----------------------------------------------------------------------------------------------------- CPU tests
def test_basis_jacobian_matches_central_differences():
    from oracle import data_utilities as du
    tp = numpy.random.RandomState(5).rand(40, 3)
    J = basis_jacobian(tp)
    step = 1e-6
    for k in range(3):
        e = numpy.zeros_like(tp)
        e[:, k] = step
        fd = (du.generate_basis_functions(tp + e, 2) - du.generate_basis_functions(tp - e, 2)) / (2 * step)
        # degree 2: the central difference of a quadratic is exact up to rounding (|X| <= 1 here: eps / step)
        assert numpy.max(numpy.abs(fd - J[:, k, :])) <= 10 * EPS / step


@pytest.mark.parametrize('nu,scale', [(1.5, 0.2), (2.5, (0.15, 0.25)), (0.7, 0.2), (200.0, (0.2, 0.3)), (0.5, 0.2)])
def test_reference_matches_central_differences_of_oracle(nu, scale):
    from oracle import data_utilities as du, predict as op
    pts, z, X = problem(200, seed=2)
    eta = 0.5
    tp = 0.1 + 0.8 * numpy.random.RandomState(3).rand(15, 2)
    Xs, Xg = du.generate_basis_functions(tp, 2), basis_jacobian(tp)
    mg, vg, parts = grad_reference(pts, z, X, tp, Xs, Xg, scale, nu, eta)

    def f(q):
        mean, var, _, _ = op.predict(pts, z, X, q, du.generate_basis_functions(q, 2), scale, nu, eta, sigma=parts['sigma'])
        return mean, var

    # one oracle evaluation rounds at about cond(Kn) eps <= (n / eta) eps relative to its terms (|z|, sigma^2)
    rnd = 10.0 * 200 / eta * EPS
    (fdm, bm), (fdv, bv) = fd_bound(f, tp, 1e-4, [rnd * numpy.max(numpy.abs(z)), rnd * parts['sigma'] ** 2])
    assert (numpy.abs(fdm - mg) <= bm).all(), numpy.max(numpy.abs(fdm - mg) - bm)
    assert (numpy.abs(fdv - vg) <= bv).all(), numpy.max(numpy.abs(fdv - vg) - bv)


def test_reference_at_a_training_point_matches_central_differences():
    """nu = 5/2 at q = p_i: the pair at distance 0 contributes 0, which is the derivative's limit (K is smooth there)"""
    from oracle import data_utilities as du, predict as op
    pts, z, X = problem(200, seed=4)
    eta, scale, nu = 0.5, 0.2, 2.5
    tp = pts[[3, 50, 120]]
    Xs, Xg = du.generate_basis_functions(tp, 2), basis_jacobian(tp)
    mg, vg, parts = grad_reference(pts, z, X, tp, Xs, Xg, scale, nu, eta)

    def f(q):
        mean, var, _, _ = op.predict(pts, z, X, q, du.generate_basis_functions(q, 2), scale, nu, eta, sigma=parts['sigma'])
        return mean, var

    rnd = 10.0 * 200 / eta * EPS
    (fdm, bm), (fdv, bv) = fd_bound(f, tp, 1e-4, [rnd * numpy.max(numpy.abs(z)), rnd * parts['sigma'] ** 2])
    assert (numpy.abs(fdm - mg) <= bm).all()
    assert (numpy.abs(fdv - vg) <= bv).all()


def test_reference_far_point_identities():
    """far from every training point (P == 0): d mean = (dx*)^T beta and d var = 2 sigma^2 (B^-1 x*)^T dx*"""
    from oracle import data_utilities as du, predict as op
    pts, z, X = problem(250, seed=3)
    rho, eta = 0.1, 0.1
    tp = 100.0 + numpy.random.RandomState(4).rand(30, 2)
    Xs, Xg = du.generate_basis_functions(tp, 2), basis_jacobian(tp)
    assert not op.cross_correlation(pts, tp, rho, 0.5).any()
    mg, vg, parts = grad_reference(pts, z, X, tp, Xs, Xg, rho, 0.5, eta)
    ref_m = numpy.einsum('jkc,c->jk', Xg, parts['beta'])
    ref_v = 2.0 * parts['sigma'] ** 2 * numpy.einsum('jkc,cj->jk', Xg, numpy.linalg.solve(parts['B'], Xs.T))
    assert (mg == ref_m).all()
    # B^-1 x* ~ |x*| / lambda_min(B): cond(B) eps of relative rounding between the two solves
    assert numpy.max(numpy.abs(vg - ref_v) / numpy.abs(ref_v)) <= 1e-9


def test_new_entry_points_reject_bad_arguments_without_a_device():
    """Each call gets one bad argument; the status must come back before any launch. The calls run in a child process that
    is shown no CUDA device, so a check that let a call through could not reach a GPU."""
    code = r'''
import ctypes, json, sys
sys.path.insert(0, %r)
from gaussian_proc import _device as dev
lib, null = dev.lib, ctypes.c_void_p(None)
a = ctypes.c_void_p(1 << 20)                       # never dereferenced: every call below fails validation first
sc = (ctypes.c_double * 2)(0.1, 0.1)
bad = (ctypes.c_double * 2)(0.1, 0.0)
args = lambda **k: [k.get('pts', a), k.get('n', 10), k.get('q', a), k.get('mc', 5), k.get('d', 2), k.get('sc', sc),
                    k.get('nu', 2.5), k.get('S', a), k.get('p', 7), k.get('U', a), k.get('ldu', 128), k.get('out', a),
                    k.get('ws', a), null]
r = {}
r['null_pts'] = lib.gp_predict_grad_dense(*args(pts=null))
r['null_q'] = lib.gp_predict_grad_dense(*args(q=null))
r['null_S'] = lib.gp_predict_grad_dense(*args(S=null))
r['null_out'] = lib.gp_predict_grad_dense(*args(out=null))
r['null_ws'] = lib.gp_predict_grad_dense(*args(ws=null))
r['null_scale'] = lib.gp_predict_grad_dense(*args(sc=null))
r['n0'] = lib.gp_predict_grad_dense(*args(n=0))
r['mc0'] = lib.gp_predict_grad_dense(*args(mc=0))
r['d0'] = lib.gp_predict_grad_dense(*args(d=0))
r['d9'] = lib.gp_predict_grad_dense(*args(d=9))
r['p0'] = lib.gp_predict_grad_dense(*args(p=0))
r['p17'] = lib.gp_predict_grad_dense(*args(p=17))
r['ldu'] = lib.gp_predict_grad_dense(*args(mc=200, ldu=128))
r['scale'] = lib.gp_predict_grad_dense(*args(sc=bad))
r['nu'] = lib.gp_predict_grad_dense(*args(nu=-1.0))
r['nu0'] = lib.gp_predict_grad_dense(*args(nu=0.0))
r['ws_ok'] = lib.gp_predict_grad_workspace_bytes(4097, 1000, 2, 7)
r['ws_p17'] = lib.gp_predict_grad_workspace_bytes(4097, 1000, 2, 17)
r['ws_d9'] = lib.gp_predict_grad_workspace_bytes(4097, 1000, 9, 7)
r['ws_mc0'] = lib.gp_predict_grad_workspace_bytes(4097, 0, 2, 7)
r['ws_n0'] = lib.gp_predict_grad_workspace_bytes(0, 1000, 2, 7)
r['launches'] = lib.gp_launch_count()
print(json.dumps(r))
''' % PKG
    res = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    r = json.loads(res.stdout.strip().splitlines()[-1])
    assert r.pop('launches') == 0
    assert r.pop('ws_ok') == 8 * 3 * 1000 * 2 * 8        # 3 chunks of 2048 rows x 1000 columns x d x (p + 1)
    for k in ('ws_p17', 'ws_d9', 'ws_mc0', 'ws_n0'):
        assert r.pop(k) == -1, k
    assert r['ldu'] == -2 and r['scale'] == -3 and r['nu'] == -5 and r['nu0'] == -5
    for k, v in r.items():
        assert v == -1 if k not in ('ldu', 'scale', 'nu', 'nu0') else v < 0, (k, v)


# ---------------------------------------------------------------------------------------------------- device plumbing
def _torch():
    import torch
    return torch


def dptr(t, offset=0):
    return ctypes.c_void_p(t.data_ptr() + 8 * offset)


@pytest.fixture(scope='module')
def cu():
    from gaussian_proc import _device as dev
    dev.require_cuda()
    return dev


def grad_on_device(cu, pts, tp, scale, nu, S, U):
    """gp_predict_grad_dense with the points, S and U in buffers whose rows >= n are NaN, U's columns >= mc NaN and a
    sentinel after the last output. Returns out (mc, d, p + 1) and the bits after it."""
    torch = _torch()
    n, d = pts.shape
    mc, p = tp.shape[0], S.shape[1]
    npad, ldu = padded(n), padded(mc) + 64
    pb = numpy.full((npad, d), numpy.nan)
    pb[:n] = pts
    Sb = numpy.full((npad, p), numpy.nan)
    Sb[:n] = S
    pd, qd, Sd = (torch.from_numpy(numpy.ascontiguousarray(a)).cuda() for a in (pb, tp, Sb))
    Ud = None
    if U is not None:
        Ub = numpy.full((npad, ldu), numpy.nan)
        Ub[:n, :mc] = U
        Ud = torch.from_numpy(Ub).cuda()
    w = mc * d * (p + 1)
    out = torch.full((w + 64,), SENTINEL, dtype=torch.float64, device='cuda')
    ws = torch.empty(cu.lib.gp_predict_grad_workspace_bytes(n, mc, d, p) // 8, dtype=torch.float64, device='cuda')
    sc = numpy.ascontiguousarray(numpy.broadcast_to(numpy.asarray(scale, dtype=numpy.float64), (d,)))
    rc = cu.lib.gp_predict_grad_dense(dptr(pd), n, dptr(qd), mc, d, cu.host_ptr(sc), float(nu), dptr(Sd), p,
                                      dptr(Ud) if Ud is not None else None, ldu, dptr(out), dptr(ws), cu.stream_ptr())
    assert rc == 0
    o = out.cpu().numpy()
    return o[:w].reshape(mc, d, p + 1), o[w:]


def h_error_bound(x, nu):
    """bound on the device's error in h(x): a few ulp for the closed forms; for general nu the device forms
    K_{nu-1} = K_{nu+1} - (2 nu / y) K_nu from Bessel values good to about 1e-13, so the bound scales with those terms"""
    if nu in (0.5, 1.5, 2.5) or nu >= 100:
        return 8 * EPS * h_of_x(x, nu)
    t = numpy.where(x > 0, x, 1.0)
    y = math.sqrt(2.0 * nu) * t
    coef = 2.0 ** (1.0 - nu) / scipy.special.gamma(nu)
    terms = coef * 2.0 * nu * y ** (nu - 1.0) * (scipy.special.kv(nu + 1.0, y) + 2.0 * nu / y * scipy.special.kv(nu, y))
    return numpy.where(x > 0, 1e-13 * terms + 8 * EPS * h_of_x(x, nu), 0.0)


# --------------------------------------------------------------------------------------- GPU: the kernel on its own
@gpu
@pytest.mark.parametrize('d', [1, 2, 3, 8])
@pytest.mark.parametrize('nu', [0.5, 1.5, 2.5, 0.7, 200.0])
def test_grad_kernel_matches_host_reference(cu, nu, d):
    """n = 2177 (two row chunks, the second partial), mc = 300, p in {1, 8, 9, 16} (both templates, full and partial),
    with U and without. The first five test points are training points (a pair at distance 0 contributes exactly 0).
    Rows >= n of the points, S and U and U's columns >= mc are NaN; the words after the output hold a sentinel."""
    n, mc = 2177, 300
    rng = numpy.random.RandomState(10 * d + int(nu * 10) % 7)
    pts, tp = rng.rand(n, d), rng.rand(mc, d)
    tp[:5] = pts[[0, 7, 2100, 2176, 1000]]
    for t, p in enumerate((1, 8, 9, 16)):
        scale = numpy.full(d, 0.2) if t % 2 == 0 else 0.15 + 0.05 * numpy.arange(d)    # isotropic / anisotropic
        if d == 8:
            scale = scale * 3.0                                                           # keep P away from underflow
        S, U = rng.randn(n, p), rng.randn(n, mc)
        G = cross_gradient(pts, tp, scale, nu)                                            # (d, n, mc)
        dist = numpy.sqrt(numpy.sum(((pts[None, :, :] - tp[:, None, :]) / scale) ** 2, axis=2)).T      # (n, mc)
        eG = h_error_bound(dist, nu)[None] * numpy.abs((pts.T[:, :, None] - tp.T[:, None, :])) / (scale ** 2)[:, None, None]
        ref = numpy.concatenate([numpy.einsum('kij,ic->jkc', G, S), numpy.einsum('kij,ij->jk', G, U)[:, :, None]], axis=2)
        aSU = [numpy.einsum('kij,ic->jkc', A, numpy.abs(S)) for A in (numpy.abs(G), eG)]
        aUU = [numpy.einsum('kij,ij->jk', A, numpy.abs(U)) for A in (numpy.abs(G), eG)]
        # sums of up to 2048 + ceil(n / 2048) terms: gamma_k = k eps of the sum of |terms|, plus the error of h
        gam = (2048 + 2 + 8) * EPS
        tol = numpy.concatenate([gam * aSU[0] + aSU[1], (gam * aUU[0] + aUU[1])[:, :, None]], axis=2)
        for with_u in (True, False):
            got, tail = grad_on_device(cu, pts, tp, scale, nu, S, U if with_u else None)
            assert numpy.isfinite(got).all(), (p, with_u)
            assert (tail.view(numpy.uint64) == SENTINEL.view(numpy.uint64)).all(), (p, with_u)
            assert (numpy.abs(got[:, :, :p] - ref[:, :, :p]) <= tol[:, :, :p]).all(), (p, with_u)
            if with_u:
                assert (numpy.abs(got[:, :, p] - ref[:, :, p]) <= tol[:, :, p]).all(), p
            else:
                assert (got[:, :, p] == 0.0).all()


@gpu
@pytest.mark.parametrize('nu', [0.5, 1.5, 0.7])
def test_grad_kernel_coincident_pair_contributes_zero(cu, nu):
    """A test point equal to one training point: the result equals the one for the same data with that training point's
    row of S and U set to 0, bit for bit (the pair contributes exactly 0, even where h(0) is infinite)."""
    rng = numpy.random.RandomState(21)
    n, mc, d, p = 1000, 130, 2, 5
    pts, tp = rng.rand(n, d), rng.rand(mc, d)
    tp[:] = tp[0]                                          # every column the same point ...
    pts[417] = tp[0]                                       # ... which is also training point 417
    S, U = rng.randn(n, p), rng.randn(n, mc)
    got, _ = grad_on_device(cu, pts, tp, 0.2, nu, S, U)
    S0, U0 = S.copy(), U.copy()
    S0[417], U0[417] = 0.0, 0.0
    ref, _ = grad_on_device(cu, pts, tp, 0.2, nu, S0, U0)
    assert numpy.isfinite(got).all()
    assert (got.view(numpy.uint64) == ref.view(numpy.uint64)).all()


# ------------------------------------------------------------------------------------------------- GPU: public API
def _device_problem(n, scale, nu=2.5, seed=0):
    import gaussian_proc
    from gaussian_proc._mixed_correlation import MixedCorrelation
    pts, z, X = problem(n, seed)
    K = gaussian_proc.generate_correlation(pts, scale, nu, device=True)
    return pts, z, X, MixedCorrelation(K)


def _test_set(ms, seed=11):
    from oracle import data_utilities as du
    tp = numpy.random.RandomState(seed).rand(ms, 2) * 1.1 - 0.05         # inside and a little outside the data's square
    return tp, du.generate_basis_functions(tp, 2), basis_jacobian(tp)


@gpu
def test_gradient_chunk_size_does_not_change_the_bits(cu):
    from gaussian_proc._predict import Predictor
    pts, z, X, Km = _device_problem(1000, 0.1)
    tp, Xs, Xg = _test_set(3000)
    pr = Predictor(Km, X, z, 0.1)
    res = [pr.predict_gradient(tp, Xs, Xg, chunk_size=c) for c in (128, 1000, 8192)]
    for r in res[1:]:
        for a, b in zip(r, res[0]):
            assert (a.view(numpy.uint64) == b.view(numpy.uint64)).all()
    res = [pr.predict_gradient(tp, Xs, Xg, return_var=False, chunk_size=c) for c in (128, 8192)]
    for a, b in zip(res[1], res[0]):
        assert (a.view(numpy.uint64) == b.view(numpy.uint64)).all()


@gpu
@pytest.mark.parametrize('noise', [False, True])
def test_gradient_mean_and_var_are_the_bits_of_predict(cu, noise):
    from gaussian_proc._predict import Predictor
    pts, z, X, Km = _device_problem(2177, 0.1)
    tp, Xs, Xg = _test_set(1500)
    pr = Predictor(Km, X, z, 0.1)
    for chunk in (1000, 8192):
        mean, var = pr.predict(tp, Xs, noise=noise, chunk_size=chunk)
        gm, gv, mg, vg = pr.predict_gradient(tp, Xs, Xg, noise=noise, chunk_size=chunk)
        assert (gm.view(numpy.uint64) == mean.view(numpy.uint64)).all()
        assert (gv.view(numpy.uint64) == var.view(numpy.uint64)).all()
        gm2, mg2 = pr.predict_gradient(tp, Xs, Xg, return_var=False, noise=noise, chunk_size=chunk)
        assert (gm2.view(numpy.uint64) == mean.view(numpy.uint64)).all()
        assert (mg2.view(numpy.uint64) == mg.view(numpy.uint64)).all()       # the U GEMM does not touch the mean
    # the nugget is constant: it does not change the gradients
    _, _, mg0, vg0 = pr.predict_gradient(tp, Xs, Xg, noise=not noise)
    assert (mg0 == mg).all() and (vg0 == vg).all()


@gpu
@pytest.mark.parametrize('n,eta,ms', [(1000, 1e-2, 300), (1000, 10.0, 1), (1000, 0.1, 2100), (2177, 0.1, 300),
                                      (2177, 1.0, 1000), (2177, 1e-2, 7)])
def test_predict_gradient_matches_reference(cu, n, eta, ms):
    from gaussian_proc._predict import Predictor
    pts, z, X, Km = _device_problem(n, 0.1)
    tp, Xs, Xg = _test_set(ms)
    tp[0] = pts[5]                                             # one test point on a training point
    Xs[0], Xg[0] = X[5], basis_jacobian(tp[:1])[0]
    pr = Predictor(Km, X, z, eta)
    mean, var, mg, vg = pr.predict_gradient(tp, Xs, Xg)
    rmg, rvg, parts = grad_reference(pts, z, X, tp, Xs, Xg, 0.1, 2.5, eta, sigma=pr.sigma)
    tol = _grad_tol(n, eta)
    assert (numpy.abs(mg - rmg) <= tol * parts['mean_scale']).all(), numpy.max(numpy.abs(mg - rmg) / parts['mean_scale'])
    assert (numpy.abs(vg - rvg) <= tol * parts['var_scale']).all(), numpy.max(numpy.abs(vg - rvg) / parts['var_scale'])


@gpu
@pytest.mark.parametrize('nu', [0.5, 1.5, 0.7])
def test_predict_gradient_at_training_points_matches_reference(cu, nu):
    """test points on training points: finite, and equal to the reference in which the coincident pair contributes 0
    (the limit of the derivative for nu > 1/2, the symmetric derivative for nu = 1/2)"""
    from gaussian_proc._predict import Predictor
    n, eta = 1000, 0.1
    pts, z, X, Km = _device_problem(n, 0.1, nu=nu, seed=8)
    idx = numpy.arange(0, n, 7)
    tp, Xs, Xg = pts[idx], X[idx], basis_jacobian(pts[idx])
    pr = Predictor(Km, X, z, eta)
    mean, var, mg, vg = pr.predict_gradient(tp, Xs, Xg)
    assert numpy.isfinite(mg).all() and numpy.isfinite(vg).all()
    rmg, rvg, parts = grad_reference(pts, z, X, tp, Xs, Xg, 0.1, nu, eta, sigma=pr.sigma)
    # the Bessel branch (nu = 0.7) adds the device's K_nu error (1e-13 relative) to the cond(Kn) eps of _grad_tol
    tol = _grad_tol(n, eta) + (1e-12 if nu == 0.7 else 0.0)
    assert (numpy.abs(mg - rmg) <= tol * parts['mean_scale']).all()
    assert (numpy.abs(vg - rvg) <= tol * parts['var_scale']).all()


@gpu
@pytest.mark.parametrize('nu', [1.5, 2.5, 0.7])
def test_predict_gradient_matches_central_differences_of_predict(cu, nu):
    """independent of the reference: central differences of the device predict() at test points at least 0.3 rho from
    every training point"""
    from oracle import data_utilities as du
    from gaussian_proc._predict import Predictor
    n, eta, rho = 400, 0.5, 0.1
    pts, z, X, Km = _device_problem(n, rho, nu=nu, seed=9)
    cand = numpy.random.RandomState(12).rand(400, 2)
    far = numpy.min(numpy.linalg.norm(cand[:, None, :] - pts[None, :, :], axis=2), axis=1) >= 0.3 * rho
    tp = cand[far][:40]
    assert tp.shape[0] == 40
    pr = Predictor(Km, X, z, eta)
    mean, var, mg, vg = pr.predict_gradient(tp, du.generate_basis_functions(tp, 2), basis_jacobian(tp))

    def f(q):
        return pr.predict(q, du.generate_basis_functions(q, 2))

    # one device evaluation rounds at about cond(Kn) eps <= (n / eta) eps relative to |z| (mean) and sigma^2 (var)
    rnd = 10.0 * n / eta * EPS
    (fdm, bm), (fdv, bv) = fd_bound(f, tp, 1e-4, [rnd * numpy.max(numpy.abs(z)), rnd * pr.sigma ** 2])
    assert (numpy.abs(fdm - mg) <= bm).all(), numpy.max(numpy.abs(fdm - mg) - bm)
    assert (numpy.abs(fdv - vg) <= bv).all(), numpy.max(numpy.abs(fdv - vg) - bv)


@gpu
@pytest.mark.parametrize('method,imate', [('direct', None), ('profiled', None), ('profiled', 'eigenvalue')])
def test_train_then_predict_gradient_matches_reference(cu, method, imate):
    import gaussian_proc
    n, scale = 1000, numpy.array([0.1, 0.13])
    pts, z, X = problem(n, seed=5)
    K = gaussian_proc.generate_correlation(pts, scale, 2.5, device=True)
    gpr = gaussian_proc.GaussianProcess(X, K, likelihood_method=method, imate_method=imate)
    res = gpr.train(z)
    tp, Xs, Xg = _test_set(500)
    mean, var, mg, vg = gpr.predict_gradient(tp, Xs, Xg)
    pm, pv = gpr.predict(tp, Xs)
    assert (mean == pm).all() and (var == pv).all()
    eta, sigma = float(res['eta']), float(res['sigma'])
    rmg, rvg, parts = grad_reference(pts, z, X, tp, Xs, Xg, scale, 2.5, eta, sigma=sigma)
    tol = _grad_tol(n, eta)
    assert (numpy.abs(mg - rmg) <= tol * parts['mean_scale']).all()
    assert (numpy.abs(vg - rvg) <= tol * parts['var_scale']).all()
    mean2, mg2 = gpr.predict_gradient(tp, Xs, Xg, return_var=False)
    assert (mean2 == mean).all() and (mg2 == mg).all()


@gpu
def test_predict_gradient_error_cases(cu):
    import gaussian_proc
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._predict import Predictor
    pts, z, X = problem(300)
    tp, Xs, Xg = _test_set(10)
    gpr = gaussian_proc.GaussianProcess(X, gaussian_proc.generate_correlation(pts, 0.1, 2.5, device=True))
    with pytest.raises(RuntimeError):
        gpr.predict_gradient(tp, Xs, Xg)
    Km = MixedCorrelation(gaussian_proc.generate_correlation(pts, 0.1, 2.5))      # a NumPy K: no points / scale / nu
    with pytest.raises(ValueError, match='set_kernel'):
        Predictor(Km, X, z, 0.1)
    Ks = gaussian_proc.generate_correlation(pts, 0.1, 0.5, sparse=True, density=0.05)
    with pytest.raises(NotImplementedError):
        Predictor(MixedCorrelation(Ks, imate_method='slq'), X, z, 0.1)
    pr = Predictor(MixedCorrelation(gaussian_proc.generate_correlation(pts, 0.1, 2.5, device=True)), X, z, 0.1)
    for bad in (Xg[:, :1], Xg[:-1], Xg[:, :, :-1], Xg[0]):
        with pytest.raises(ValueError, match='X_test_grad'):
            pr.predict_gradient(tp, Xs, bad)
    with pytest.raises(ValueError):
        pr.predict_gradient(tp, Xs[:, :-1], Xg)
    with pytest.raises(ValueError):
        pr.predict_gradient(numpy.c_[tp, tp[:, :1]], Xs, Xg)
    with pytest.raises(ValueError):
        pr.predict_gradient(tp, Xs, Xg, chunk_size=0)
    gpr.results = {'sigma': 1.0, 'eta': math.inf, 'sigma0': math.inf}       # what the root finder reports at the bracket end
    gpr.z = z
    with pytest.raises(ValueError):
        gpr.predict_gradient(tp, Xs, Xg)


@gpu
def test_n20k_identities_and_central_differences(cu):
    """n = 20 000 (nu = 2.5, rho = 0.1): far from every training point (P == 0) the gradients are (dx*)^T beta and
    2 sigma^2 (B^-1 x*)^T dx*; at a few points inside the data the gradients match central differences of predict()."""
    from oracle import data_utilities as du
    from gaussian_proc._predict import Predictor
    n, eta = 20000, 0.1
    pts, z, X, Km = _device_problem(n, 0.1)
    pr = Predictor(Km, X, z, eta)
    tp = 100.0 + numpy.random.RandomState(3).rand(1000, 2)
    Xs, Xg = du.generate_basis_functions(tp, 2), basis_jacobian(tp)
    mean, var, mg, vg = pr.predict_gradient(tp, Xs, Xg)
    assert (mg == Xg @ pr.beta).all()
    ref = pr.sigma ** 2 * (2.0 * numpy.einsum('jkc,cj->jk', Xg, numpy.linalg.solve(pr.B, Xs.T)))
    assert numpy.max(numpy.abs(vg - ref) / numpy.abs(ref)) <= 4 * EPS
    tp = 0.2 + 0.6 * numpy.random.RandomState(4).rand(6, 2)
    mean, var, mg, vg = pr.predict_gradient(tp, du.generate_basis_functions(tp, 2), basis_jacobian(tp))

    def f(q):
        return pr.predict(q, du.generate_basis_functions(q, 2))

    rnd = 10.0 * n / eta * EPS
    (fdm, bm), (fdv, bv) = fd_bound(f, tp, 1e-4, [rnd * numpy.max(numpy.abs(z)), rnd * pr.sigma ** 2])
    assert (numpy.abs(fdm - mg) <= bm).all(), numpy.max(numpy.abs(fdm - mg) - bm)
    assert (numpy.abs(fdv - vg) <= bv).all(), numpy.max(numpy.abs(fdv - vg) - bv)
