"""The Matern parameter checks shared by every entry point that takes a correlation scale and nu (include/gpgp.h,
conventions): -3 for a scale entry that is not > 0, -4 for an anisotropic scale where a d/drho is requested, -5 for a
general-branch nu that is not > 0, all returned before anything is enqueued.

The calls run in a child process that is shown no CUDA device, with fake device pointers that are never dereferenced: a
call that got past its checks would launch (gp_launch_count) or fail with a CUDA error instead of the expected status."""

import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'gaussian-process-param-estimation_b200')

# entry point -> the derivative settings checked (True: the derivative output or flag is given, which requires an isotropic
# scale). gp_loglik_dense reads the scale and nu only with flag 4.
DERIVATIVE = {
    'gp_matern_dense': (False, True), 'gp_matern_cross': (False,), 'gp_matern_cross_dk': (True,),
    'gp_matern_cross_points': (False,), 'gp_predict_grad_dense': (False,), 'gp_dk_apply': (True,),
    'gp_loglik_dense': (True,), 'gp_loglik_dense_dscale': (False,), 'gp_matern_sparse_count': (False,),
    'gp_matern_sparse_fill': (False, True), 'gp_matern_blocks_count': (False,), 'gp_matern_blocks_fill': (False, True),
    'gp_kernel_threshold': (False,),
}

BAD_SCALES = {'zero': [0.1, 0.0], 'zero_first': [0.0, 0.1], 'negative': [0.1, -0.1], 'nan': [0.1, math.nan]}
BAD_NUS = {'nu0': 0.0, 'nu_neg': -1.0}
GOOD = [0.1, 0.1]

CHILD = r'''
import ctypes, json, math, sys
sys.path.insert(0, %r)
from gaussian_proc import _device as dev
lib, null = dev.lib, ctypes.c_void_p(None)
a = ctypes.c_void_p(1 << 20)                       # a 16-byte aligned fake device pointer
ph = (ctypes.c_double * 20)()                      # real host memory for the host-pointer arguments
i64 = (ctypes.c_int64 * 2)()
tau = ctypes.c_double(-7.0)


def call(name, scale, nu, deriv):
    sc = (ctypes.c_double * 2)(*scale)
    dv = a if deriv else null
    if name == 'gp_matern_dense':
        return lib.gp_matern_dense(a, 10, 2, sc, nu, a, 128, dv, null)
    if name == 'gp_matern_cross':
        return lib.gp_matern_cross(a, a, a, a, 64, 128, 100, 2, sc, nu, 0.1, a, 128, null)
    if name == 'gp_matern_cross_dk':
        return lib.gp_matern_cross_dk(a, a, a, a, 64, 128, 100, 2, sc, nu, a, 128, null)
    if name == 'gp_matern_cross_points':
        return lib.gp_matern_cross_points(a, 10, a, 5, 2, sc, nu, a, 128, null)
    if name == 'gp_predict_grad_dense':
        return lib.gp_predict_grad_dense(a, 10, a, 5, 2, sc, nu, a, 7, a, 128, a, a, null)
    if name == 'gp_dk_apply':
        return lib.gp_dk_apply(a, 10, 2, sc, nu, a, 7, 7, a, null)
    if name == 'gp_loglik_dense':
        return lib.gp_loglik_dense(a, 10, 128, a, 7, 0.1, 1 | 2 | (4 if deriv else 0), a, 2, sc, nu, a, a, a, a, a, null)
    if name == 'gp_loglik_dense_dscale':
        return lib.gp_loglik_dense_dscale(a, 10, 128, 7, a, 2, sc, nu, 1, a, a, null)
    if name == 'gp_matern_sparse_count':
        return lib.gp_matern_sparse_count(a, ph, 10, 2, sc, nu, 0.1, a, a, i64, null, 0, 0, null)
    if name == 'gp_matern_sparse_fill':
        return lib.gp_matern_sparse_fill(a, ph, 10, 2, sc, nu, 0.1, a, a, a, a, dv, 1, null, 0, 0, null)
    if name == 'gp_matern_blocks_count':
        return lib.gp_matern_blocks_count(a, 10, 2, sc, nu, 0.1, a, a, a, 0, 10, a, i64, null)
    if name == 'gp_matern_blocks_fill':
        return lib.gp_matern_blocks_fill(a, 10, 2, sc, nu, 0.1, a, a, a, 0, 10, a, a, a, dv, null)
    if name == 'gp_kernel_threshold':
        return lib.gp_kernel_threshold(10000, 2, 1e-3, sc, nu, ctypes.byref(tau))
    raise KeyError(name)


cases = json.loads(sys.argv[1])
r = {key: call(*args) for key, args in cases.items()}
sc = (ctypes.c_double * 2)(0.1, 0.1)
bad = (ctypes.c_double * 2)(0.1, 0.0)
r['loglik_dk_without_inverse'] = lib.gp_loglik_dense(a, 10, 128, a, 7, 0.1, 1 | 4, a, 2, sc, 2.5, a, a, a, a, a, null)
r['loglik_dk_without_points'] = lib.gp_loglik_dense(a, 10, 128, a, 7, 0.1, 2 | 4, null, 2, sc, 2.5, a, a, a, a, a, null)
r['loglik_dk_without_scale'] = lib.gp_loglik_dense(a, 10, 128, a, 7, 0.1, 2 | 4, a, 2, null, 2.5, a, a, a, a, a, null)
r['loglik_dk_d9'] = lib.gp_loglik_dense(a, 10, 128, a, 7, 0.1, 2 | 4, a, 9, sc, 2.5, a, a, a, a, a, null)
r['loglik_cubic_without_inverse'] = lib.gp_loglik_dense(a, 10, 128, a, 7, 0.1, 8, a, 2, sc, 2.5, a, a, a, a, a, null)
r['threshold_density'] = lib.gp_kernel_threshold(10, 2, 1e-3, sc, 2.5, ctypes.byref(tau))
r['threshold_density_bad_scale'] = lib.gp_kernel_threshold(10, 2, 1e-3, bad, 2.5, ctypes.byref(tau))
r['threshold_density_bad_nu'] = lib.gp_kernel_threshold(10, 2, 1e-3, sc, -1.0, ctypes.byref(tau))
r['tau_untouched'] = tau.value == -7.0
r['launches'] = lib.gp_launch_count()
print(json.dumps(r))
''' % PKG


def expected_cases():
    """key -> ((entry point, scale, nu, derivative requested), expected status)"""
    cases = {}
    for name, derivs in DERIVATIVE.items():
        for deriv in derivs:
            tag = '%s/%s' % (name, 'deriv' if deriv else 'plain')
            for k, scale in BAD_SCALES.items():
                cases['%s/%s' % (tag, k)] = ((name, scale, 2.5, deriv), -3)
                cases['%s/%s_general_nu' % (tag, k)] = ((name, scale, 0.7, deriv), -3)
            for k, nu in BAD_NUS.items():
                cases['%s/%s' % (tag, k)] = ((name, GOOD, nu, deriv), -5)
            if deriv:
                cases['%s/anisotropic' % tag] = ((name, [0.1, 0.2], 2.5, deriv), -4)
                cases['%s/anisotropic_general_nu' % tag] = ((name, [0.1, 0.2], 0.7, deriv), -4)
    return cases


def test_every_entry_point_checks_the_matern_parameters_before_any_work():
    cases = expected_cases()
    arg = json.dumps({k: v[0] for k, v in cases.items()})
    res = subprocess.run([sys.executable, '-c', CHILD, arg], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    r = json.loads(res.stdout.strip().splitlines()[-1])
    # each of the 13 entry points is covered, with an anisotropic case on those that take a derivative
    assert {k.split('/')[0] for k in cases} == set(DERIVATIVE)
    assert sum(k.endswith('/anisotropic') for k in cases) == 6
    wrong = {k: (r[k], want) for k, (_, want) in cases.items() if r[k] != want}
    assert not wrong, wrong
    assert r['launches'] == 0
    assert r['tau_untouched']
    # gp_loglik_dense's own flag checks
    assert r['loglik_dk_without_inverse'] == -8
    assert r['loglik_dk_without_points'] == -8
    assert r['loglik_dk_without_scale'] == -8
    assert r['loglik_dk_d9'] == -8
    assert r['loglik_cubic_without_inverse'] == -9
    # the density check (-10) comes after the parameter checks
    assert r['threshold_density'] == -10
    assert r['threshold_density_bad_scale'] == -3
    assert r['threshold_density_bad_nu'] == -5
