"""
ctypes binding of ``libgpgp.so`` (the C ABI declared in ``include/gpgp.h``) and the small amount of device-buffer
plumbing shared by the package. PyTorch is used only to own device memory and streams.

There is deliberately NO CPU fallback: importing the library or calling any compute entry point without the
CUDA extension / a CUDA device raises.
"""

import ctypes
import os

import numpy

__all__ = ['lib', 'check', 'GpgpError', 'padded_size', 'stream_ptr', 'torch', 'require_cuda']

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, 'libgpgp.so')


class GpgpError(RuntimeError):
    """Raised when a libgpgp entry point reports a bad argument or a CUDA error (negative status)."""


def _load():
    if not os.path.exists(_LIB_PATH):
        raise ImportError(
            'libgpgp.so not found at %s. Build it with `python __graft_entry__.py build` (nvcc, sm_100a). '
            'This package has no CPU fallback.' % _LIB_PATH)
    return ctypes.CDLL(_LIB_PATH)


lib = _load()

_vp = ctypes.c_void_p
_i64 = ctypes.c_int64
_f64 = ctypes.c_double
_int = ctypes.c_int

# name -> (restype, argtypes); must list every symbol of include/gpgp.h (tests/test_abi.py checks that)
SIGNATURES = {
    'gp_abi_version': (_int, []),
    'gp_padded_size': (_i64, [_i64]),
    'gp_launch_count': (ctypes.c_ulonglong, []),
    'gp_gemm_profile_enable': (_int, [_int]),
    'gp_gemm_profile_read': (_int, [_vp, _vp, _vp, _vp]),
    'gp_matern_dense': (_int, [_vp, _i64, _i64, _vp, _f64, _vp, _i64, _vp, _vp]),
    'gp_matern_cross': (_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _f64, _f64, _vp, _i64, _vp]),
    'gp_matern_cross_points': (_int, [_vp, _i64, _vp, _i64, _i64, _vp, _f64, _vp, _i64, _vp]),
    'gp_predict_workspace_bytes': (_i64, [_i64, _i64, _i64]),
    'gp_predict_dense': (_int, [_vp, _i64, _i64, _vp, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp]),
    'gp_kernel_threshold': (_int, [_i64, _i64, _f64, _vp, _f64, _vp]),
    'gp_sparse_workspace_bytes': (_i64, [_i64, _i64]),
    'gp_matern_sparse_count': (_int, [_vp, _vp, _i64, _i64, _vp, _f64, _f64, _vp, _vp, _vp, _vp]),
    'gp_matern_sparse_fill': (_int, [_vp, _vp, _i64, _i64, _vp, _f64, _f64, _vp, _vp, _vp, _vp, _vp, _int, _vp]),
    'gp_matern_sparse_count_rows': (_int, [_vp, _vp, _i64, _i64, _vp, _f64, _f64, _vp, _vp, _vp, _vp, _i64, _i64, _vp]),
    'gp_matern_sparse_fill_rows': (_int, [_vp, _vp, _i64, _i64, _vp, _f64, _f64, _vp, _vp, _vp, _vp, _vp, _int, _vp, _i64, _i64,
                                          _vp]),
    'gp_csr_sort_rows': (_int, [_i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    'gp_csr_spmm': (_int, [_vp, _vp, _vp, _i64, _f64, _vp, _i64, _vp, _vp]),
    'gp_rademacher': (_int, [_vp, _i64, _i64, ctypes.c_uint64, _i64, _vp, _vp]),
    'gp_spatial_keys': (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp]),
    'gp_bcsr_count': (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    'gp_bcsr_fill': (_int, [_i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i64, _vp, _vp, _vp, _vp]),
    'gp_bcsr_spmm': (_int, [_i64, _vp, _vp, _vp, _i64, _f64, _vp, _i64, _vp, _vp]),
    'gp_gram_workspace_bytes': (_i64, [_i64]),
    'gp_gram_skinny': (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    'gp_bcsr_lanczos': (_int, [_i64, _vp, _vp, _vp, _i64, _f64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    'gp_bcsr_cg_solve': (_int, [_i64, _vp, _vp, _vp, _i64, _f64, _vp, _vp, _i64, _f64, _i64, _vp, _vp, _vp]),
    'gp_krylov_workspace_bytes': (_i64, [_i64, _i64]),
    'gp_col_dot': (_int, [_vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    'gp_lanczos': (_int, [_vp, _vp, _vp, _i64, _f64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    'gp_block_combine': (_int, [_vp, _i64, _i64, _i64, _vp, _vp, _vp]),
    'gp_cg_solve': (_int, [_vp, _vp, _vp, _i64, _f64, _vp, _vp, _i64, _f64, _i64, _vp, _vp, _vp]),
    'gp_dgemm_f64': (_int, [_int, _int, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _i64, _f64, _f64, _int, _int,
                            _vp]),
    'gp_dgemm_ktab_f64': (_int, [_int, _int, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i64, _i64, _f64, _f64, _vp, _vp, _vp]),
    'gp_matern_cross_dk': (_int, [_vp, _vp, _vp, _vp, _i64, _i64, _i64, _i64, _vp, _f64, _vp, _i64, _vp]),
    'gp_rect_apply': (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _f64, _f64, _vp]),
    'gp_rect_workspace_bytes': (_i64, [_i64, _i64, _i64]),
    'gp_rect_apply_t': (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _i64, _vp, _i64, _f64, _f64, _vp, _vp]),
    'gp_pair_dot': (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _i64, _f64, _vp, _vp, _vp]),
    'gp_dk_apply': (_int, [_vp, _i64, _i64, _vp, _f64, _vp, _i64, _i64, _vp, _vp]),
    'gp_points_bbox': (_int, [_vp, _i64, _i64, _vp, _vp, _vp]),
    'gp_sort_workspace_bytes': (_i64, [_i64]),
    'gp_sort_keys_u64': (_int, [_vp, _i64, _int, _vp, _vp, _vp]),
    'gp_inverse_permutation': (_int, [_vp, _i64, _vp, _vp]),
    'gp_scan_counts': (_int, [_vp, _i64, _vp, _vp]),
    'gp_scan_counts_i32': (_int, [_vp, _i64, _vp, _vp]),
    'gp_gather_rows': (_int, [_vp, _vp, _i64, _i64, _vp, _vp]),
    'gp_matern_blocks_count': (_int, [_vp, _i64, _i64, _vp, _f64, _f64, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    'gp_matern_blocks_fill': (_int, [_vp, _i64, _i64, _vp, _f64, _f64, _vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    'gp_peer_handle_bytes': (_i64, []),
    'gp_peer_create': (_vp, [_i64, _i64, _i64]),
    'gp_peer_handle': (_int, [_vp, _vp]),
    'gp_peer_connect': (_int, [_vp, _vp]),
    'gp_peer_destroy': (_int, [_vp]),
    'gp_peer_vec': (_vp, [_vp, _i64]),
    'gp_peer_barrier': (_int, [_vp, _vp]),
    'gp_peer_allreduce': (_int, [_vp, _vp, _i64, _vp]),
    'gp_peer_error': (_int, [_vp, _vp]),
    'gp_slab_encode_columns': (_int, [_vp, _i64, _i64, _i64, _i64, _vp, _vp, _vp]),
    'gp_slab_spmm': (_int, [_vp, _vp, _vp, _vp, _i64, _f64, _vp, _i64, _vp, _vp]),
    'gp_slab_col_dot': (_int, [_vp, _vp, _vp, _i64, _i64, _vp, _vp, _vp]),
    'gp_slab_lanczos': (_int, [_vp, _vp, _vp, _vp, _i64, _f64, _vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    'gp_slab_cg_solve': (_int, [_vp, _vp, _vp, _vp, _i64, _f64, _vp, _vp, _i64, _f64, _i64, _vp, _vp, _vp]),
    'gp_sytrd_workspace_bytes': (_i64, [_i64]),
    'gp_sytrd_f64': (_int, [_vp, _i64, _i64, _vp, _vp, _vp, _vp, _vp]),
    'gp_stebz_f64': (_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    'gp_ormtr_skinny': (_int, [_vp, _i64, _i64, _vp, _int, _vp, _i64, _i64, _vp]),
    'gp_tridiag_solve': (_int, [_vp, _vp, _i64, _f64, _vp, _i64, _i64, _vp, _i64, _vp, _vp, _vp]),
    'gp_eig_reduce': (_int, [_vp, _i64, _f64, _vp, _vp]),
    'gp_shift_copy': (_int, [_vp, _i64, _i64, _f64, _vp, _vp]),
    'gp_potrf_workspace_bytes': (_i64, [_i64]),
    'gp_potrf_f64': (_int, [_vp, _i64, _i64, _vp, _vp, _vp]),
    'gp_logdet_from_chol': (_int, [_vp, _i64, _i64, _vp, _vp]),
    'gp_potrs_f64': (_int, [_vp, _i64, _vp, _vp, _i64, _i64, _vp]),
    'gp_potri_workspace_bytes': (_i64, [_i64]),
    'gp_potri_f64': (_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    'gp_trtri_f64': (_int, [_vp, _vp, _i64, _vp, _vp, _vp]),
    'gp_lauum_f64': (_int, [_vp, _vp, _i64, _vp]),
    'gp_traces_workspace_bytes': (_i64, [_i64]),
    'gp_inverse_traces': (_int, [_vp, _i64, _i64, _int, _vp, _vp, _vp]),
    'gp_symm_skinny': (_int, [_vp, _i64, _i64, _vp, _i64, _vp, _vp]),
    'gp_loglik_dense_dscale': (_int, [_vp, _i64, _i64, _i64, _vp, _i64, _vp, _f64, _i64, _vp, _vp, _vp]),
    'gp_loglik_workspace_bytes': (_i64, [_i64]),
    'gp_loglik_out_len': (_i64, [_i64]),
    'gp_loglik_dense': (_int, [_vp, _i64, _i64, _vp, _i64, _f64, _int, _vp, _i64, _vp, _f64, _vp, _vp, _vp, _vp, _vp,
                               _vp]),
}

for _name, (_res, _args) in SIGNATURES.items():
    _fn = getattr(lib, _name)
    _fn.restype = _res
    _fn.argtypes = _args


def check(status, what):
    """Map a negative libgpgp status to an exception; non-negative values (LAPACK-style info) are returned."""
    if status < 0:
        if status <= -1000:
            raise GpgpError('%s: CUDA error %d' % (what, -status - 1000))
        raise GpgpError('%s: invalid argument (status %d)' % (what, status))
    return status


def padded_size(n):
    return int(lib.gp_padded_size(int(n)))


_torch = None


def _get_torch():
    global _torch
    if _torch is None:
        import torch as _t
        _torch = _t
    return _torch


class _TorchProxy(object):
    def __getattr__(self, name):
        return getattr(_get_torch(), name)


torch = _TorchProxy()


def require_cuda():
    t = _get_torch()
    if not t.cuda.is_available():
        raise GpgpError('gaussian_proc (B200 build) needs a CUDA device; there is no CPU fallback.')
    return t


def stream_ptr():
    """cudaStream_t of torch's current stream as an integer (0 = legacy default stream)."""
    t = _get_torch()
    return ctypes.c_void_p(t.cuda.current_stream().cuda_stream)


def host_f64(a):
    """C-contiguous float64 view/copy of a host array."""
    return numpy.ascontiguousarray(a, dtype=numpy.float64)


def host_ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p)


_READ_ONLY_KEYS = []      # [(array, key)] of arrays that cannot be written to (kept alive: their ids stay unique); small LRU


def _digest(arr):
    """Content digest of a host array in two streaming passes at memory speed: the 64-bit words are laid out as rows of 4096
    and both the row sums and the column sums (wrap-around integer arithmetic) are hashed. Any single edited entry and any
    exchange of two entries changes it (an entry moves to another row or another column). BLAKE2b over all bytes costs
    140 ms for the 56 MB of [X z] at n = 2^20 - longer than a sparse evaluation; this takes about 15 ms."""
    import hashlib
    raw = numpy.ascontiguousarray(arr)
    h = hashlib.blake2b(digest_size=16)
    h.update(repr((raw.shape, raw.dtype.str)).encode())
    if raw.nbytes < (1 << 16) or raw.dtype.itemsize != 8:
        h.update(raw.view(numpy.uint8).reshape(-1))
        return h.digest()
    v = raw.view(numpy.uint64).reshape(-1)
    cut = (v.size // 4096) * 4096
    m = v[:cut].reshape(-1, 4096)
    h.update(m.sum(axis=1, dtype=numpy.uint64).tobytes())
    h.update(m.sum(axis=0, dtype=numpy.uint64).tobytes())
    h.update(v[cut:].tobytes())
    return h.digest()


def host_key(a):
    """Content fingerprint of a host array used as the cache key of its device copy (and of Krylov runs started from
    it): shape, dtype and a digest of ALL entries, so that an in-place edit between two evaluations is noticed (the
    reference re-reads z and X on every call). Arrays that own their data and are marked read-only
    (``a.setflags(write=False)``; the sweeps do that with their copies of X and z) are fingerprinted once."""
    arr = numpy.asarray(a)
    frozen = (not arr.flags.writeable) and arr.flags.owndata
    if frozen:
        for ent in _READ_ONLY_KEYS:
            if ent[0] is arr:
                return ent[1]
    key = (arr.shape, arr.dtype.str, _digest(arr))
    if frozen:
        _READ_ONLY_KEYS.append((arr, key))
        del _READ_ONLY_KEYS[:-8]
    return key
