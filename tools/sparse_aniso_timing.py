"""Timing of the anisotropic sparse gradient (dl/d scale[k] per dimension) against the isotropic dl/drho at n = 2^20, d = 2,
density 1e-3, nu = 0.5 and 1.5; scales (0.005, 0.005) and (0.004, 0.00625) (same geometric mean, so a similar nnz).

Per (nu, scale): generation + engine build with the derivatives (gp_matern_blocks_fill, plus gp_bcsr_dscale_fill for the
anisotropic scale), one l^ + gradient at eta = 10 on the fresh operator (a new-rho step), a further eta (5) on the same
operator; best of three, host clock around synchronised work. For the anisotropic operator also the kernel
gp_bcsr_dscale_fill alone (CUDA events, warmed, mean of 10 launches) with its byte floor from the shapes (reads 16 * 8 + 4 B
per block-column, writes d * 16 * 8 B) at the HBM3e bandwidth of one B200 (7.7 TB/s), and the derivative SpMMs of one
evaluation (count and CUDA-event time per width). Prints one JSON line (GPU name and power limit included); --out also
writes it to a file."""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'gaussian-process-param-estimation_b200'))
import torch  # noqa: E402
from gaussian_proc import _device as dev  # noqa: E402
from gaussian_proc._sparse import generate_sparse_operator, _device_points  # noqa: E402
from gaussian_proc._mixed_correlation import MixedCorrelation  # noqa: E402
from gaussian_proc._likelihood import ProfileLikelihood  # noqa: E402

HBM_BYTES_PER_S = 7.7e12
P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731


def sync_time():
    torch.cuda.synchronize()
    return time.perf_counter()


def event_ms(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def gpu_info():
    info = {'gpu': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=60)
        info['power_limit_and_max_sm_clock'] = q.stdout.strip()
    except OSError as exc:
        info['power_limit_and_max_sm_clock'] = 'nvidia-smi not available: %s' % exc
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--n', type=int, default=1 << 20)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('needs a CUDA device')
    n, dens = args.n, 1e-3
    numpy.random.seed(0)
    pts = numpy.random.rand(n, 2)
    z = numpy.sin(pts[:, 0] * 7) + numpy.cos(pts[:, 1] * 5) + 0.1 * numpy.random.randn(n)
    X = numpy.stack([numpy.ones(n), pts[:, 0], pts[:, 1], pts[:, 0] ** 2, pts[:, 0] * pts[:, 1], pts[:, 1] ** 2], axis=1)
    for arr in (pts, z, X):
        arr.setflags(write=False)
    opts = {'seed': 0, 'lanczos_degree': 20}
    res = dict(gpu_info(), n=n, d=2, density=dens, eta=10.0, further_eta=5.0, options=opts, runs=[])
    for nu in (0.5, 1.5):
        for label, scale in (('isotropic', [0.005, 0.005]), ('anisotropic', [0.004, 0.00625])):
            scale = numpy.array(scale)
            best = None
            for rep in range(args.reps + 1):          # the first pass warms every shape
                t0 = sync_time()
                K = generate_sparse_operator(pts, scale, nu, dens, with_derivative=True)
                t1 = sync_time()
                Km = MixedCorrelation(K, imate_method='slq', imate_options=dict(opts))
                t2 = sync_time()
                g = ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, 10.0)
                t3 = sync_time()
                g2 = ProfileLikelihood.log_likelihood_and_gradient(z, X, Km, 5.0)
                t4 = sync_time()
                row = {'generate_s': t1 - t0, 'build_s': t2 - t1, 'loglik_grad_s': t3 - t2, 'further_eta_s': t4 - t3}
                if rep > 0 and (best is None or row['generate_s'] + row['build_s'] + row['loglik_grad_s']
                                < best['generate_s'] + best['build_s'] + best['loglik_grad_s']):
                    best = row
                if rep < args.reps:
                    del Km, K
                    torch.cuda.empty_cache()
            eng = Km.engine
            total = int(eng.blocked[1].numel())
            run = dict(best, nu=nu, scale=scale.tolist(), kind=label, nnz=int(K.nnz), block_columns=total,
                       fill_ratio=eng.fill_ratio, samples=int(eng.last_info['num_samples']),
                       loglik=g[0], dloglik_deta=g[1], dloglik_dscale=numpy.atleast_1d(g[2]).tolist(),
                       further_eta_gradient=numpy.atleast_1d(g2[2]).tolist())
            # derivative SpMMs of one evaluation at a new eta on this operator (fresh engine: nothing kept yet)
            Kc = MixedCorrelation(K, imate_method='slq', imate_options=dict(opts))
            widths = {}
            spmm = Kc.engine.spmm

            def counted(eta, X_dev, derivative=False, dim=None, spmm=spmm):
                if derivative or dim is not None:
                    widths[X_dev.shape[1]] = widths.get(X_dev.shape[1], 0) + 1
                return spmm(eta, X_dev, derivative=derivative, dim=dim)
            Kc.engine.spmm = counted
            ProfileLikelihood.log_likelihood_and_gradient(z, X, Kc, 10.0)
            dk = {}
            for B, cnt in sorted(widths.items()):
                V = torch.randn((n, B), dtype=torch.float64, device='cuda')
                if label == 'anisotropic':
                    ms = event_ms(lambda: spmm(0.0, V, dim=0), 10)
                else:
                    ms = event_ms(lambda: spmm(0.0, V, derivative=True), 10)
                dk['B%d' % B] = {'calls': cnt, 'ms_each': ms}
            run['derivative_spmms_per_evaluation'] = dk
            run['derivative_spmm_ms_per_evaluation'] = sum(v['calls'] * v['ms_each'] for v in dk.values())
            del Kc
            if label == 'anisotropic':
                dpts = _device_points(pts)[0]
                dims = torch.empty((2, 16 * total), dtype=torch.float64, device='cuda')
                bptr, bidx, bvals, _ = eng.blocked
                lib, s = dev.lib, dev.stream_ptr()

                def fill():
                    dev.check(lib.gp_bcsr_dscale_fill(P(bptr), P(bidx), P(bvals), total, 0, n, P(K.order), P(dpts), n, 2,
                                                      dev.host_ptr(scale), nu, P(dims), s), 'gp_bcsr_dscale_fill')
                ms = event_ms(fill, 10)
                assert torch.equal(dims, eng.dims)
                nbytes = total * (16 * 8 + 4) + 2 * 16 * 8 * total
                run['dscale_fill'] = {'ms': ms, 'bytes': nbytes, 'floor_ms_at_7.7TBps': nbytes / HBM_BYTES_PER_S * 1e3,
                                      'achieved_TBps': nbytes / (ms * 1e-3) / 1e12}
                del dims
            res['runs'].append(run)
            del Km, K, eng
            torch.cuda.empty_cache()
            print(json.dumps({'progress': [nu, label]}), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
