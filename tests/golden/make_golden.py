"""Generates the committed golden fixtures in tests/golden/ from the REFERENCE ITSELF (run in the build container,
where /root/reference exists; the GPU box only reads the committed .npz files).

Sources of truth:
  A. the reference's shipped result pickles (data/OptimalCovariance_With{,out}Prior.pickle,
     data/NoiseLevelResults.pickle) -> golden_pickles.npz   (numbers copied, pickles are data not source)
  B. the reference's own Python likelihood modules imported unmodified through oracle/ref_loader.py (imate shim,
     eigenvalue and cholesky methods) -> golden_likelihood.npz
  C. the reference's compiled Cython generators (oracle/_ref, built by oracle/build_ref.py) -> golden_generate.npz

Usage: python tests/golden/make_golden.py
"""

import contextlib
import io
import os
import pickle
import sys

import numpy

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle import data_utilities as du  # noqa: E402
from oracle import ref_loader  # noqa: E402

REF = ref_loader.REF


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def pickles():
    out = {}
    for tag, name in (('noprior', 'OptimalCovariance_WithoutPrior.pickle'), ('prior', 'OptimalCovariance_WithPrior.pickle')):
        g = pickle.load(open(os.path.join(REF, 'data', name), 'rb'))
        out['rho'] = numpy.asarray(g['DecorrelationScale'], dtype=float)
        out['nu'] = numpy.asarray(g['nu'], dtype=float)
        out['Lp_' + tag] = numpy.asarray(g['Lp'], dtype=float)
    g = pickle.load(open(os.path.join(REF, 'data', 'NoiseLevelResults.pickle'), 'rb'))[1]  # Poly-2 basis
    for k in ('NoiseMagnitude', 'sigma', 'sigma0', 'eta'):
        out['noise_' + k] = numpy.asarray(g[k], dtype=float)
    numpy.savez_compressed(os.path.join(HERE, 'golden_pickles.npz'), **out)
    print('golden_pickles.npz', {k: v.shape for k, v in out.items()})


def likelihood():
    ref = ref_loader.load()
    cy = ref_loader.load_cython()
    out = {}
    cases = []
    n = 300
    numpy.random.seed(0)
    pts = numpy.random.rand(n, 2)
    z = du.generate_data(pts, 0.2)
    X = du.generate_basis_functions(pts, 2)
    out['points'], out['z'], out['X'] = pts, z, X
    hyper_direct = [(0.3, 0.2), (0.12, 0.25), (1.0, 0.05), (0.05, 0.5)]
    hyper_profile = [(0.3, 0.5), (0.2, 0.01), (1.0, 10.0)]
    log_etas = [-2.0, -1.0, 0.0, 1.0, 2.0]
    for ci, (nu, rho) in enumerate([(0.5, 0.1), (1.5, 0.1), (2.5, 0.1), (2.5, 0.3), (200.0, 0.05)]):
        K = cy.generate_dense_correlation(pts, numpy.array([rho, rho]), nu, False)
        for method in ('eigenvalue', 'cholesky'):
            Km = ref.MixedCorrelation(K, imate_method=method)
            tag = 'c%d_%s_' % (ci, method)
            out[tag + 'direct_ll'] = numpy.array([ref.DirectLikelihood.log_likelihood(z, X, Km, False, list(h)) for h in hyper_direct])
            out[tag + 'direct_jac'] = numpy.array([ref.DirectLikelihood.log_likelihood_jacobian(z, X, Km, False, list(h)) for h in hyper_direct])
            out[tag + 'direct_hess'] = numpy.array([ref.DirectLikelihood.log_likelihood_hessian(z, X, Km, False, list(h)) for h in hyper_direct])
            out[tag + 'profile_ll'] = numpy.array([ref.ProfileLikelihood.log_likelihood(z, X, Km, False, list(h)) for h in hyper_profile])
            out[tag + 'profile_der1'] = numpy.array([ref.ProfileLikelihood.log_likelihood_der1_eta(z, X, Km, t) for t in log_etas])
            out[tag + 'logdet'] = numpy.array([Km.logdet(10.0 ** t) for t in log_etas])
            out[tag + 'traceinv'] = numpy.array([Km.traceinv(10.0 ** t) for t in log_etas])
            out[tag + 'traceinv2'] = numpy.array([Km.traceinv(10.0 ** t, exponent=2) for t in log_etas])
            if method == 'eigenvalue':
                try:
                    r = quiet(ref.ProfileLikelihood.find_log_likelihood_der1_zeros, z, X, Km, [1e-4, 1e3])
                    out[tag + 'root'] = numpy.array([r['sigma'], r['sigma0'], r['eta']])
                except Exception as e:  # noqa: BLE001 -- (e.g. no sign change -> der2 fallback) recorded as NaN
                    print('root find failed for case', ci, repr(e)[:80])
                    out[tag + 'root'] = numpy.full(3, numpy.nan)
        sol = ref.MixedCorrelation(K, imate_method='cholesky').solve(0.1, numpy.c_[X, z])
        out['c%d_solve_eta0.1' % ci] = sol
        cases.append((nu, rho))
    out['cases'] = numpy.array(cases)
    out['hyper_direct'] = numpy.array(hyper_direct)
    out['hyper_profile'] = numpy.array(hyper_profile)
    out['log_etas'] = numpy.array(log_etas)
    numpy.savez_compressed(os.path.join(HERE, 'golden_likelihood.npz'), **out)
    print('golden_likelihood.npz', len(out), 'arrays')


def generate():
    cy = ref_loader.load_cython()
    out = {}
    numpy.random.seed(7)
    pts = numpy.random.rand(160, 2)
    out['points2d'] = pts
    for nu in (0.5, 1.5, 2.5, 200.0, 3.3, 0.8):
        out['dense_nu%g' % nu] = cy.generate_dense_correlation(pts, numpy.array([0.1, 0.17]), nu, False)
    pts3 = numpy.random.rand(90, 3)
    out['points3d'] = pts3
    out['dense3d_nu1.5'] = cy.generate_dense_correlation(pts3, numpy.array([0.2, 0.3, 0.25]), 1.5, False)
    # sparse: random points and a structured grid (exact ties at the taper radius)
    numpy.random.seed(11)
    ps = numpy.random.rand(1500, 2)
    out['sparse_points'] = ps
    grid = du.generate_points(40, 2, grid=True)
    for tag, p in (('rand', ps), ('grid', grid)):
        for nu in (0.5, 1.5, 2.5):
            S = quiet(cy.generate_sparse_correlation, p, numpy.array([0.03, 0.03]), nu, 0.01, False)
            key = 'sparse_%s_nu%g_' % (tag, nu)
            out[key + 'indptr'], out[key + 'indices'], out[key + 'data'] = S.indptr, S.indices, S.data
    # the dense matrices are exactly symmetric: keep the packed lower triangles (tests/conftest.py mirrors them back)
    for key in [k for k in out if k.startswith('dense')]:
        K = out.pop(key)
        assert (K == K.T).all()
        out[key + '_tril'] = K[numpy.tril_indices(K.shape[0])]
    numpy.savez_compressed(os.path.join(HERE, 'golden_generate.npz'), **out)
    print('golden_generate.npz', len(out), 'arrays')


if __name__ == '__main__':
    if not ref_loader.available():
        sys.exit('reference tree not available; fixtures can only be regenerated in the build container')
    pickles()
    likelihood()
    generate()
