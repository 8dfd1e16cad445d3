"""Prediction at new points (kriging): the cross-correlation generator, the device reduction gp_predict_dense, and the
public GaussianProcess.predict / Predictor against the CPU oracle (oracle/predict.py).

The unmarked tests run without a GPU: the oracle against an independent formulation (the bordered kriging system), two
identities of the oracle, and argument validation of the new C entry points. The tests marked gpu need a CUDA device."""

import ctypes
import json
import math
import os
import subprocess
import sys

import numpy
import pytest

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


def gls(K, X, z, eta):
    """beta^, alpha = Kn^-1 (z - X beta^), B = X^T Kn^-1 X (dense solves, independent of oracle/predict.py)"""
    Kn = K + eta * numpy.eye(K.shape[0])
    KiX = numpy.linalg.solve(Kn, X)
    B = X.T @ KiX
    beta = numpy.linalg.solve(B, KiX.T @ z)
    return beta, numpy.linalg.solve(Kn, z - X @ beta), B


# ------------------------------------------------------------------------------------------------------- CPU: oracle
def test_oracle_matches_bordered_kriging_system():
    from oracle import data_utilities as du, matern, predict as op
    pts, z, X = problem(300)
    tp = numpy.random.RandomState(1).rand(70, 2)
    Xs = du.generate_basis_functions(tp, 2)
    eta, rho, nu = 0.05, 0.1, 2.5
    mean, var, cov, sigma = op.predict(pts, z, X, tp, Xs, rho, nu, eta)
    K = matern.generate_dense_correlation(pts, rho, nu)
    P = op.cross_correlation(pts, tp, rho, nu)
    bmean, bvar = op.bordered_predict(K, P, X, z, Xs, eta)
    assert numpy.max(numpy.abs(mean - bmean)) <= 1e-12 * numpy.max(numpy.abs(bmean))
    assert numpy.max(numpy.abs(var / sigma ** 2 - bvar)) <= 1e-12
    assert numpy.max(numpy.abs(numpy.diag(cov) - var)) <= 1e-12 * sigma ** 2


def test_oracle_identities_at_training_and_far_points():
    from oracle import matern, predict as op
    from oracle import data_utilities as du
    pts, z, X = problem(250, seed=3)
    rho, eta = 0.1, 0.1
    # test points = training points: mean = x^T beta + K alpha = z - eta alpha
    mean, var, _, _ = op.predict(pts, z, X, pts, X, rho, 0.5, eta)
    beta, alpha, B = gls(matern.generate_dense_correlation(pts, rho, 0.5), X, z, eta)
    assert numpy.max(numpy.abs(mean - (z - eta * alpha))) <= 1e-11 * numpy.max(numpy.abs(z))
    # far points (distance > 800 rho, nu = 1/2: exp(-800) underflows, P == 0): mean = X* beta, var = sigma^2 (1 + x*^T B^-1 x*)
    tp = 100.0 + numpy.random.RandomState(4).rand(30, 2)
    Xs = du.generate_basis_functions(tp, 2)
    assert not op.cross_correlation(pts, tp, rho, 0.5).any()
    mean, var, _, sigma = op.predict(pts, z, X, tp, Xs, rho, 0.5, eta)
    assert numpy.max(numpy.abs(mean - Xs @ beta)) <= 1e-11 * numpy.max(numpy.abs(Xs @ beta))
    ref = sigma ** 2 * (1.0 + numpy.sum(Xs.T * numpy.linalg.solve(B, Xs.T), axis=0))
    assert numpy.max(numpy.abs(var - ref) / ref) <= 1e-9      # x*^T B^-1 x* ~ |x*|^2 / lambda_min(B): cond(B) eps


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
r = {}
r['cross_null'] = lib.gp_matern_cross_points(null, 10, a, 5, 2, sc, 2.5, a, 128, null)
r['cross_d'] = lib.gp_matern_cross_points(a, 10, a, 5, 9, sc, 2.5, a, 128, null)
r['cross_m0'] = lib.gp_matern_cross_points(a, 10, a, 0, 2, sc, 2.5, a, 128, null)
r['cross_ld'] = lib.gp_matern_cross_points(a, 10, a, 200, 2, sc, 2.5, a, 128, null)
r['cross_ld_odd'] = lib.gp_matern_cross_points(a, 10, a, 5, 2, sc, 2.5, a, 129, null)
r['cross_align'] = lib.gp_matern_cross_points(a, 10, a, 5, 2, sc, 2.5, ctypes.c_void_p((1 << 20) + 8), 128, null)
r['cross_scale'] = lib.gp_matern_cross_points(a, 10, a, 5, 2, bad, 2.5, a, 128, null)
r['cross_nu'] = lib.gp_matern_cross_points(a, 10, a, 5, 2, sc, -1.0, a, 128, null)
args = lambda **k: [k.get('W', a), k.get('n', 10), k.get('npad', 128), k.get('S', a), k.get('p', 7), k.get('P', a),
                    k.get('mc', 5), k.get('ldp', 128), k.get('V', a), k.get('ldv', 128), k.get('out', a), k.get('ws', a), null]
r['pred_null_W'] = lib.gp_predict_dense(*args(W=null))
r['pred_null_ws'] = lib.gp_predict_dense(*args(ws=null))
r['pred_null_out'] = lib.gp_predict_dense(*args(out=null))
r['pred_p17'] = lib.gp_predict_dense(*args(p=17))
r['pred_p0'] = lib.gp_predict_dense(*args(p=0))
r['pred_mc0'] = lib.gp_predict_dense(*args(mc=0))
r['pred_npad'] = lib.gp_predict_dense(*args(npad=256))
r['pred_ldp'] = lib.gp_predict_dense(*args(mc=129))
r['pred_ldv'] = lib.gp_predict_dense(*args(ldv=126))
r['pred_ld_odd'] = lib.gp_predict_dense(*args(ldp=129))
r['pred_align'] = lib.gp_predict_dense(*args(V=ctypes.c_void_p((1 << 20) + 8)))
r['ws_ok'] = lib.gp_predict_workspace_bytes(4096, 1000, 7)
r['ws_p17'] = lib.gp_predict_workspace_bytes(4096, 1000, 17)
r['ws_mc0'] = lib.gp_predict_workspace_bytes(4096, 0, 7)
r['launches'] = lib.gp_launch_count()
print(json.dumps(r))
''' % PKG
    res = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    r = json.loads(res.stdout.strip().splitlines()[-1])
    assert r.pop('launches') == 0
    assert r.pop('ws_ok') == 8 * 2 * 1024 * 8           # 2 chunks of 2048 rows x 1024 padded columns x (p + 1)
    assert r.pop('ws_p17') == -1 and r.pop('ws_mc0') == -1
    assert r['cross_ld'] == -2 and r['cross_ld_odd'] == -2 and r['cross_align'] == -2
    assert r['cross_scale'] == -3 and r['cross_nu'] == -5
    assert r['pred_ldp'] == -2 and r['pred_ldv'] == -2 and r['pred_ld_odd'] == -2 and r['pred_align'] == -3
    for k, v in r.items():
        assert v < 0, (k, v)


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


def cross_on_device(cu, pts, tp, scale, nu, ldp=None, fill=numpy.nan):
    torch = _torch()
    n, m, d = pts.shape[0], tp.shape[0], pts.shape[1]
    npad, mpad = padded(n), padded(m)
    ldp = ldp or mpad
    P = torch.full((npad, ldp), fill, dtype=torch.float64, device='cuda')
    p_d, q_d = torch.from_numpy(pts).cuda(), torch.from_numpy(tp).cuda()
    sc = numpy.ascontiguousarray(scale, dtype=numpy.float64)
    rc = cu.lib.gp_matern_cross_points(dptr(p_d), n, dptr(q_d), m, d, cu.host_ptr(sc), float(nu), dptr(P), ldp,
                                       cu.stream_ptr())
    assert rc == 0
    return P.cpu().numpy()


# ------------------------------------------------------------------------------------------------ GPU: cross generator
@gpu
@pytest.mark.parametrize('d', [1, 2, 3])
@pytest.mark.parametrize('nu', [0.5, 1.5, 2.5, 0.7, 200.0])
def test_cross_generator_matches_oracle(cu, nu, d):
    from oracle import predict as op
    # Closed forms: a few ulp of 1. The device scales the distance by 1 / scale, the oracle divides by scale (1 ulp of x),
    # and exp differs by an ulp; nu = 2.5 reaches 2 ulp of 1 (4.4e-16) on these points. The dense generator does the same
    # on them: P equals its off-diagonal block bit for bit (next test). Bessel branch (nu = 0.7): the device K_nu, the
    # dense generator's bar.
    tol = 4 * EPS if nu in (0.5, 1.5, 2.5, 200.0) else 2e-13
    sizes = [(1, 1), (127, 129), (129, 1000), (1000, 127), (1000, 1000), (1, 1000)]
    for t, (n, m) in enumerate(sizes):
        rng = numpy.random.RandomState(100 * d + t)
        pts, tp = rng.rand(n, d), rng.rand(m, d)
        scale = numpy.full(d, 0.2) if t % 2 == 0 else 0.1 + 0.1 * numpy.arange(d)      # isotropic / anisotropic
        P = cross_on_device(cu, pts, tp, scale, nu, ldp=padded(m) + (64 if t % 3 == 0 else 0))
        ref = op.cross_correlation(pts, tp, scale, nu)
        assert numpy.max(numpy.abs(P[:n, :m] - ref)) <= tol, (n, m)
        assert (P[n:, :padded(m)] == 0.0).all() and (P[:, m:padded(m)] == 0.0).all()      # padding exactly 0 (no NaN left)
        assert numpy.isnan(P[:, padded(m):]).all()                                         # beyond mpad: not written


@gpu
@pytest.mark.parametrize('nu', [0.5, 2.5, 0.7])
def test_cross_generator_self_block_equals_dense_generator(cu, nu):
    """P(points, points) == gp_matern_dense's K bit for bit, P(p, q) == the off-diagonal block of gp_matern_dense on the
    stacked points bit for bit, and a duplicated point gives exactly 1."""
    torch = _torch()

    def dense(pts, scale):
        n, npad = pts.shape[0], padded(pts.shape[0])
        K = torch.empty((npad, npad), dtype=torch.float64, device='cuda')
        p_d = torch.from_numpy(numpy.ascontiguousarray(pts)).cuda()
        assert cu.lib.gp_matern_dense(dptr(p_d), n, pts.shape[1], cu.host_ptr(scale), nu, dptr(K), npad, None,
                                      cu.stream_ptr()) == 0
        return K.cpu().numpy()[:n, :n]

    rng = numpy.random.RandomState(7)
    pts = rng.rand(333, 3)
    pts[17] = pts[200]
    scale = numpy.array([0.1, 0.25, 0.17])
    n = pts.shape[0]
    P = cross_on_device(cu, pts, pts, scale, nu)
    assert (P[:n, :n].view(numpy.uint64) == dense(pts, scale).view(numpy.uint64)).all()
    assert P[17, 200] == 1.0 and P[200, 17] == 1.0 and (numpy.diag(P)[:n] == 1.0).all()
    tp = rng.rand(290, 3)
    tp[3] = pts[5]
    P2 = cross_on_device(cu, pts, tp, scale, nu)
    assert P2[5, 3] == 1.0
    Kall = dense(numpy.r_[pts, tp], scale)
    assert (P2[:n, :290].view(numpy.uint64) == Kall[:n, n:].view(numpy.uint64)).all()


# ----------------------------------------------------------------------------------- GPU: gp_predict_dense, exact inputs
def dyadic_inverse_factor(n, rng):
    """lower W (npad x npad): unit diagonal, strictly lower entries in {-2..2} / 16 at density 1/8, identity padding;
    NaN above the 128-block diagonal (never read: k < m0 + 128), zero above the diagonal inside the diagonal blocks"""
    npad = padded(n)
    W = numpy.tril(rng.integers(-2, 3, size=(npad, npad)) * (rng.random((npad, npad)) < 0.125) / 16.0, -1)
    W[range(npad), range(npad)] = 1.0
    W[n:, :] = 0.0
    W[:, n:] = 0.0
    W[range(n, npad), range(n, npad)] = 1.0
    for b in range(0, npad, 128):
        W[b:b + 128, b + 128:] = numpy.nan
    return W


@gpu
@pytest.mark.parametrize('n,mc,p', [(129, 1, 3), (1000, 200, 7), (2177, 1000, 16), (2048, 128, 9), (300, 129, 8)])
def test_predict_dense_exact_on_dyadic_inputs(cu, n, mc, p):
    """Integer P and S and a dyadic W: V = W P, P^T S and ||V[:, j]||^2 are exact in any summation order (|entries| stay far
    below 2^53 / 256), so the result is checked bit for bit. P's columns beyond mcpad are NaN (must not be read), V's beyond
    mcpad and out[] beyond mc (p + 1) hold a sentinel (must not be written)."""
    torch = _torch()
    rng = numpy.random.default_rng(n + mc + p)
    npad, mcpad = padded(n), padded(mc)
    ld = mcpad + 64
    W = dyadic_inverse_factor(n, rng)
    P = numpy.full((npad, ld), numpy.nan)
    P[:, :mcpad] = 0.0
    P[:n, :mc] = rng.integers(-4, 5, size=(n, mc))
    S = numpy.zeros((npad, p))
    S[:n] = rng.integers(-4, 5, size=(n, p))
    Wd, Pd, Sd = (torch.from_numpy(a).cuda() for a in (W, P, S))
    Vd = torch.full((npad, ld), SENTINEL, dtype=torch.float64, device='cuda')
    out = torch.full((mc * (p + 1) + 64,), SENTINEL, dtype=torch.float64, device='cuda')
    ws = torch.empty(cu.lib.gp_predict_workspace_bytes(npad, mc, p) // 8, dtype=torch.float64, device='cuda')
    rc = cu.lib.gp_predict_dense(dptr(Wd), n, npad, dptr(Sd), p, dptr(Pd), mc, ld, dptr(Vd), ld, dptr(out), dptr(ws),
                                 cu.stream_ptr())
    assert rc == 0
    Wz = numpy.nan_to_num(W, nan=0.0)
    Pz = P[:, :mcpad]
    Vref = Wz @ Pz
    V = Vd.cpu().numpy()
    assert (V[:, :mcpad] == Vref).all()
    assert (V[:, mcpad:].view(numpy.uint64) == numpy.uint64(SENTINEL.view(numpy.uint64))).all()
    o = out.cpu().numpy()
    got = o[:mc * (p + 1)].reshape(mc, p + 1)
    assert (got[:, :p] == Pz[:, :mc].T @ S).all()
    assert (got[:, p] == numpy.sum(Vref[:, :mc] ** 2, axis=0)).all()
    assert (o[mc * (p + 1):].view(numpy.uint64) == numpy.uint64(SENTINEL.view(numpy.uint64))).all()


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
    return tp, du.generate_basis_functions(tp, 2)


def _var_tol(n, eta):
    # the variance 1 - ||L^-1 k*||^2 + r^T B^-1 r cancels: its rounding is bounded by about cond(Kn) eps <= (n / eta) eps;
    # never tighter than 1e-9 (relative to sigma^2)
    return max(1e-9, 10.0 * n / eta * EPS)


@gpu
def test_chunk_size_does_not_change_the_bits(cu):
    from gaussian_proc._predict import Predictor
    pts, z, X, Km = _device_problem(1000, 0.1)
    tp, Xs = _test_set(3000)
    pr = Predictor(Km, X, z, 0.1)
    res = [pr.predict(tp, Xs, chunk_size=c) for c in (128, 1000, 8192)]
    for mean, var in res[1:]:
        assert (mean.view(numpy.uint64) == res[0][0].view(numpy.uint64)).all()
        assert (var.view(numpy.uint64) == res[0][1].view(numpy.uint64)).all()


@gpu
@pytest.mark.parametrize('n,eta,ms', [(1000, 1e-2, 300), (1000, 10.0, 1), (1000, 0.1, 4099), (2177, 0.1, 300),
                                      (2177, 1.0, 4099), (2177, 1e-2, 1)])
def test_predictor_matches_oracle(cu, n, eta, ms):
    from gaussian_proc._predict import Predictor
    from oracle import predict as op
    pts, z, X, Km = _device_problem(n, 0.1)
    tp, Xs = _test_set(ms)
    pr = Predictor(Km, X, z, eta)
    mean, var, cov = pr.predict(tp, Xs, return_cov=True)
    rmean, rvar, rcov, sigma = op.predict(pts, z, X, tp, Xs, 0.1, 2.5, eta)
    assert abs(pr.sigma - sigma) <= 1e-10 * sigma
    assert numpy.max(numpy.abs(mean - rmean)) <= 1e-10 * numpy.max(numpy.abs(rmean))
    tol = _var_tol(n, eta) * sigma ** 2
    assert numpy.max(numpy.abs(var - numpy.maximum(rvar, 0.0))) <= tol
    assert numpy.max(numpy.abs(cov - rcov)) <= tol
    assert (cov == cov.T).all()
    # the nugget: observation variance = latent variance + sigma^2 eta
    mean2, var2, cov2 = pr.predict(tp, Xs, return_cov=True, noise=True)
    assert (mean2 == mean).all()
    assert numpy.max(numpy.abs(var2 - (rvar + sigma ** 2 * eta))) <= tol
    assert numpy.max(numpy.abs(numpy.diag(cov2) - numpy.diag(cov) - sigma ** 2 * eta)) <= tol
    only_mean = pr.predict(tp, Xs, return_var=False)
    assert (only_mean == mean).all()


@gpu
@pytest.mark.parametrize('method,imate', [('direct', None), ('profiled', None), ('profiled', 'eigenvalue')])
def test_train_then_predict_matches_oracle(cu, method, imate):
    import gaussian_proc
    from oracle import predict as op
    n, scale = 1000, numpy.array([0.1, 0.13])
    pts, z, X = problem(n, seed=5)
    K = gaussian_proc.generate_correlation(pts, scale, 2.5, device=True)
    gpr = gaussian_proc.GaussianProcess(X, K, likelihood_method=method, imate_method=imate)
    res = gpr.train(z)
    tp, Xs = _test_set(500)
    mean, var = gpr.predict(tp, Xs)
    eta, sigma = float(res['eta']), float(res['sigma'])
    rmean, rvar, _, _ = op.predict(pts, z, X, tp, Xs, scale, 2.5, eta, sigma=sigma)
    assert numpy.max(numpy.abs(mean - rmean)) <= 1e-10 * numpy.max(numpy.abs(rmean))
    assert numpy.max(numpy.abs(var - numpy.maximum(rvar, 0.0))) <= _var_tol(n, eta) * sigma ** 2


@gpu
def test_prediction_error_cases(cu):
    import gaussian_proc
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._predict import Predictor
    pts, z, X = problem(300)
    tp, Xs = _test_set(10)
    gpr = gaussian_proc.GaussianProcess(X, gaussian_proc.generate_correlation(pts, 0.1, 2.5, device=True))
    with pytest.raises(RuntimeError):
        gpr.predict(tp, Xs)
    Kh = gaussian_proc.generate_correlation(pts, 0.1, 2.5)                    # a NumPy K: no points / scale / nu
    Km = MixedCorrelation(Kh)
    with pytest.raises(ValueError, match='set_kernel'):
        Predictor(Km, X, z, 0.1)
    Km.set_kernel(pts, 0.1, 2.5)
    Predictor(Km, X, z, 0.1).predict(tp, Xs)
    Ks = gaussian_proc.generate_correlation(pts, 0.1, 0.5, sparse=True, density=0.05)
    with pytest.raises(NotImplementedError):
        Predictor(MixedCorrelation(Ks, imate_method='slq'), X, z, 0.1)
    Kd = MixedCorrelation(gaussian_proc.generate_correlation(pts, 0.1, 2.5, device=True))
    for eta in (math.inf, -0.1, math.nan):
        with pytest.raises(ValueError):
            Predictor(Kd, X, z, eta)
    pr = Predictor(Kd, X, z, 0.1)
    with pytest.raises(ValueError):
        pr.predict(tp, Xs[:, :-1])
    with pytest.raises(ValueError):
        pr.predict(numpy.c_[tp, tp[:, :1]], Xs)
    gpr.results = {'sigma': 1.0, 'eta': math.inf, 'sigma0': math.inf}       # what the root finder reports at the bracket end
    gpr.z = z
    with pytest.raises(ValueError):
        gpr.predict(tp, Xs)


@gpu
def test_n20k_identities(cu):
    """n = 20 000 (nu = 2.5, rho = 0.1), where the CPU is too slow to compare against: at training points used as test
    points the mean is z - eta alpha; far from every training point (P == 0) it is X* beta with variance
    sigma^2 (1 + x*^T B^-1 x*)."""
    from oracle import data_utilities as du
    from gaussian_proc._predict import Predictor
    n, eta = 20000, 0.1
    pts, z, X, Km = _device_problem(n, 0.1)
    pr = Predictor(Km, X, z, eta)
    idx = numpy.random.RandomState(2).choice(n, 4096, replace=False)
    mean, var = pr.predict(pts[idx], X[idx])
    alpha = Km.solve(eta, z - X @ pr.beta)
    # the solve and the prediction each round at about cond(Kn) eps <= (n / eta) eps relative to |z|
    assert numpy.max(numpy.abs(mean - (z[idx] - eta * alpha[idx]))) <= 10.0 * n / eta * EPS * numpy.max(numpy.abs(z))
    assert (var >= 0.0).all() and (var < pr.sigma ** 2).all()
    tp = 100.0 + numpy.random.RandomState(3).rand(1000, 2)
    Xs = du.generate_basis_functions(tp, 2)
    mean, var = pr.predict(tp, Xs)
    assert (mean == Xs @ pr.beta).all()
    ref = pr.sigma ** 2 * (1.0 + numpy.einsum('ij,ji->i', Xs, numpy.linalg.solve(pr.B, Xs.T)))
    assert (var == ref).all()
