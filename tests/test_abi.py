"""CPU tests of the drop-in boundary: libgpgp.so loads without a GPU, exports every symbol include/gpgp.h declares,
the ctypes table covers exactly that set, and argument validation answers without touching a device."""

import ctypes
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def header_symbols():
    text = open(os.path.join(ROOT, 'include', 'gpgp.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(gp_[a-z0-9_]+)\s*\(', text)))


def test_header_declares_expected_surface():
    syms = header_symbols()
    for must in ('gp_matern_dense', 'gp_potrf_f64', 'gp_potrs_f64', 'gp_potri_f64', 'gp_loglik_dense',
                 'gp_logdet_from_chol', 'gp_dgemm_f64', 'gp_shift_copy'):
        assert must in syms


def test_library_exports_every_declared_symbol():
    from gaussian_proc import _device as dev
    for s in header_symbols():
        assert hasattr(dev.lib, s), 'libgpgp.so does not export %s' % s


def test_ctypes_table_matches_header():
    from gaussian_proc import _device as dev
    assert sorted(dev.SIGNATURES) == header_symbols()


def test_no_gpu_calls_are_pure():
    from gaussian_proc import _device as dev
    assert dev.lib.gp_abi_version() == 100
    assert dev.padded_size(1) == 128 and dev.padded_size(128) == 128 and dev.padded_size(129) == 256
    assert dev.padded_size(20000) == 20096 and dev.padded_size(0) == 0
    assert dev.lib.gp_potrf_workspace_bytes(256) == 2 * 128 * 128 * 8
    assert dev.lib.gp_loglik_out_len(7) == 8 + 4 * 49          # G, H, Q, T3
    assert dev.lib.gp_launch_count() == 0


def test_bad_arguments_are_rejected_before_any_launch():
    from gaussian_proc import _device as dev
    lib = dev.lib
    null = ctypes.c_void_p(None)
    assert lib.gp_matern_dense(null, 10, 2, null, 0.5, null, 128, null, null) < 0
    assert lib.gp_potrf_f64(null, 10, 128, null, null, null) < 0
    assert lib.gp_dgemm_f64(0, 0, null, 128, null, 128, null, 128, 100, 128, 16, 1.0, 0.0, 0, 0, null) == -1   # M % 128
    assert lib.gp_potrs_f64(null, 128, null, null, 3, 3, null) < 0
    assert lib.gp_loglik_dense(null, 10, 128, null, 7, 0.1, 0, null, 2, null, 2.5, null, null, null, null, null,
                               null) < 0
    with pytest.raises(dev.GpgpError):
        dev.check(-3, 'x')
    with pytest.raises(dev.GpgpError):
        dev.check(-1001, 'x')
    assert dev.check(5, 'x') == 5


def test_no_cpu_fallback():
    """The product must fail loudly without a CUDA device (and must never import the oracle). The call runs in a child
    process that is shown no device, so that the check holds on a machine with a GPU as well."""
    import subprocess
    import sys
    pkg = os.path.join(ROOT, 'gaussian-process-param-estimation_b200')
    code = ('import sys\n'
            'sys.path.insert(0, %r)\n'
            'import numpy\n'
            'import gaussian_proc\n'
            'from gaussian_proc import _device as dev\n'
            'try:\n'
            '    gaussian_proc.generate_correlation(numpy.random.rand(10, 2))\n'
            'except dev.GpgpError:\n'
            '    sys.exit(0)\n'
            'sys.exit("generate_correlation ran without a CUDA device")\n' % pkg)
    res = subprocess.run([sys.executable, '-c', code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=''),
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    for base, _, files in os.walk(pkg):
        for f in files:
            if f.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(base, f)).read()
                assert 'import oracle' not in src and 'from oracle' not in src, f
