#!/usr/bin/env python
"""
bench.py -- headline benchmark of the GP log-likelihood hot path on B200.

Metric (BASELINE.json): log-likelihood + gradient evaluations per second, dense Matern nu = 2.5, n = 20 000 random 2-D
points (configs[1]), FP64. One STEP = one evaluation at a new (eta, rho): Matern correlation generation for that rho,
one blocked Cholesky of K + eta I, the solves for [X z], the inverse for the traces, and every reduction needed for
l^, d l^/d eta and d l^/d rho (n^3 flop, SURVEY 8d). --cells-in-flight (default 2) independent evaluations are in
flight per GPU, each with its own buffers and CUDA stream; exactly K steps complete inside the timed region.

  python bench.py [--gpus N] [--steps K] [--warmup W]          our CUDA path (under torchrun for N > 1: one rank per
                                                                GPU, independent (eta, rho) cells per rank, weak scaling,
                                                                no data-path collective; results all-gathered at the end)
  python bench.py --impl reference [...]                        the reference's CPU algorithm (oracle port; the
                                                                reference's likelihood code is Python + imate and cannot
                                                                travel, see DESIGN.md) on the host cores, bounded sample
Prints ONE JSON line on rank 0.
"""

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import threading
import time

# torchrun exports OMP_NUM_THREADS=1 to its workers; the CPU legs (cpu_baseline, --impl reference) must run on all host
# cores, so the BLAS / OpenMP pools are sized before numpy loads them (pin_host_threads() re-asserts it at run time)
if os.environ.get('GP_BENCH_KEEP_THREADS', '0') == '0':
    try:
        _ncpu = len(os.sched_getaffinity(0))
    except AttributeError:
        _ncpu = os.cpu_count() or 1
    for _v in ('OMP_NUM_THREADS', 'OPENBLAS_NUM_THREADS', 'MKL_NUM_THREADS'):
        os.environ[_v] = str(_ncpu)

import numpy  # noqa: E402

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'gaussian-process-param-estimation_b200'))

METRIC = 'loglik+grad evals/s (Matern nu=2.5 dense n=20k, FP64)'
UNIT = 'evals/s'
NU = 2.5
ETAS = [1e-2, 1e-1, 1.0, 10.0]          # SURVEY 8d C2


def cell(idx):
    """(eta, rho) of the idx-th evaluation: eta cycles over the C2 set, rho moves every step so that the correlation
    matrix really is regenerated each time."""
    return ETAS[idx % 4], 0.1 * (1.0 + 0.01 * (idx % 11))


def make_inputs(n):
    """SURVEY 8d synthetic inputs: points = rand(n, 2) with seed 0; z = sin(pi x) + sin(pi y) + 0.2 randn with seed 31
    (examples/_utilities/data_utilities.py:93-101); X = monomials of total degree <= 2 (m = 6, :150-173)."""
    numpy.random.seed(0)
    pts = numpy.random.rand(n, 2)
    z = numpy.sin(numpy.pi * pts[:, 0]) + numpy.sin(numpy.pi * pts[:, 1])
    numpy.random.seed(31)
    z = z + 0.2 * numpy.random.randn(n)
    x, y = pts[:, 0], pts[:, 1]
    X = numpy.stack([numpy.ones(n), x, x * x, y, x * y, y * y], axis=1)
    for a in (pts, z, X):
        a.setflags(write=False)      # read-only inputs: the library fingerprints their content once, not per evaluation
    return pts, z, X


# ------------------------------------------------------------------------------------------------- clocks sampler
class ClockSampler(object):
    Q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
        'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for k, name in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'power_w_max': max(pw) if pw else None, 'samples': len(sm), 'reasons': sorted(reasons)}


# --------------------------------------------------------------------------------------------------- CPU baseline
WORKLOAD = ('configs[1]: dense Matern nu=2.5, n=%d random 2-D points (seed 0), m=6 (Poly-2 basis), '
            'one (eta, rho) cell per step per GPU, eta in {1e-2,1e-1,1,10}, rho ~ 0.1')


def bench_config(n, npad, C):
    """The `config` object of the JSON line - identical in both arms (same workload, same keys)."""
    return {'workload': WORKLOAD % n,
            'l2': 'inputs larger than L2 (K = %.1f GB per evaluation)' % (npad * npad * 8e-9),
            'parallelism': 'independent cells per GPU (replicas), results all-gathered',
            'cells_in_flight': C}


def host_threads():
    """Host cores this process may use (torchrun exports OMP_NUM_THREADS=1; the CPU arm must not inherit that)."""
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


_THREAD_LIMIT = []


def pin_host_threads():
    """BLAS / OpenMP pools of this process -> all host cores, whatever the launcher exported."""
    nthr = host_threads()
    try:
        from threadpoolctl import threadpool_limits, threadpool_info
        _THREAD_LIMIT.append(threadpool_limits(limits=nthr))
        blas = [i.get('num_threads') for i in threadpool_info() if i.get('user_api') == 'blas']
        return max(blas) if blas else nthr
    except Exception:  # noqa: BLE001
        return nthr


def cpu_evaluation(n, method='cholesky', idx=0):
    """ONE loglik+grad evaluation of the reference's CPU algorithm at n points, timed (BASELINE.md section 4): Matern
    generation (compiled reference Cython when oracle/_ref is there, else the oracle's C restatement) +
    DirectLikelihood.log_likelihood + log_likelihood_jacobian (_direct_likelihood.py:31-157: 4 dposv solves, one logdet,
    one trace of the inverse; `method` = the imate method behind logdet / traceinv: 'cholesky', or 'eigenvalue' - the one
    likelihood.py:41 hard-codes - which adds one eigvalsh per correlation matrix). Returns (seconds_generation,
    seconds_likelihood, kind)."""
    from oracle import likelihood as L
    from oracle import matern
    pts, z, X = make_inputs(n)
    eta, rho = cell(idx)
    scale = numpy.array([rho, rho])
    kind = 'port'
    gen = lambda: matern.generate_dense_correlation(pts, scale, NU)   # noqa: E731
    try:
        from oracle import ref_loader
        cy = ref_loader.load_cython()
        gen = lambda: cy.generate_dense_correlation(pts, scale, NU, False)  # noqa: E731
        kind = 'port (likelihood) + reference (compiled Cython generator)'
    except Exception:  # noqa: BLE001
        pass
    sigma = 0.3
    hyper = [sigma, sigma * numpy.sqrt(eta)]
    t0 = time.perf_counter()
    K = gen()
    t1 = time.perf_counter()
    Km = L.MixedCorrelation(K, method)
    L.DirectLikelihood.log_likelihood(z, X, Km, False, hyper)
    L.DirectLikelihood.log_likelihood_jacobian(z, X, Km, False, hyper)
    t2 = time.perf_counter()
    return t1 - t0, t2 - t1, kind


def cpu_sample(n_full, sizes=(4000, 8000), repeats=(2, 1), full=True, eigen_n=4000):
    """The reference's CPU path on this box's host cores: best of `repeats` at each n in `sizes`, the fitted exponent,
    and (full=True) ONE measured evaluation at n_full - the value is then a measurement, not an extrapolation."""
    cores = pin_host_threads()
    rows, kind = [], 'port'
    for ns, reps in zip(sizes, repeats):
        best = None
        for r in range(reps):
            tg, tl, kind = cpu_evaluation(ns, 'cholesky', r)
            best = (tg, tl) if best is None or tg + tl < sum(best) else best
        rows.append({'n': ns, 'generation_s': best[0], 'likelihood_s': best[1], 'seconds': sum(best)})
    exponent = None
    if len(rows) >= 2:
        exponent = float(numpy.log(rows[-1]['seconds'] / rows[0]['seconds']) / numpy.log(rows[-1]['n'] / float(rows[0]['n'])))
    s = n_full / float(rows[-1]['n'])
    t_fit = rows[-1]['generation_s'] * s ** 2 + rows[-1]['likelihood_s'] * s ** 3
    out = {'unit': UNIT, 'cores': cores, 'kind': kind, 'samples': rows, 'fitted_exponent': exponent,
           'seconds_per_eval_n3_fit_from_largest_sample': t_fit}
    if eigen_n:
        ns = eigen_n
        tg, tl, _ = cpu_evaluation(ns, 'eigenvalue', 0)
        out['eigenvalue_method'] = {'n': ns, 'generation_s': tg, 'likelihood_s': tl,
                                    'note': "imate_method='eigenvalue' (likelihood.py:41): one eigvalsh per matrix + the same 4 dposv"}
    if full:
        tg, tl, _ = cpu_evaluation(n_full, 'cholesky', 0)
        out.update({'value': 1.0 / (tg + tl), 'extrapolated': False, 'seconds_per_eval': tg + tl,
                    'sample': 'ONE measured evaluation at n=%d (Matern generation %.1fs + DirectLikelihood l and jacobian '
                              '%.1fs, Cholesky method, %d threads); smaller n (best of %s): %s'
                              % (n_full, tg, tl, cores, list(repeats),
                                 ', '.join('n=%d %.2fs' % (r_['n'], r_['seconds']) for r_ in rows))})
    else:
        out.update({'value': 1.0 / t_fit, 'extrapolated': True, 'seconds_per_eval': t_fit,
                    'sample': 'best of %d at n=%d (generation %.2fs + likelihood %.2fs), scaled with n^2 / n^3 to n=%d'
                              % (repeats[-1], rows[-1]['n'], rows[-1]['generation_s'], rows[-1]['likelihood_s'], n_full)})
    return out


def run_reference(args):
    """The CPU arm. value = 1 / (measured seconds of ONE n = 20 000 evaluation on all host cores); every --steps step is
    a bounded sample (one whole evaluation at n = GP_BENCH_CPU_N, default 4000) whose wall time is ms_per_step."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n = int(os.environ.get('GP_BENCH_N', '20000'))
    ns = int(os.environ.get('GP_BENCH_CPU_N', '4000'))
    full = os.environ.get('GP_BENCH_CPU_FULL', '1') != '0'
    cores = pin_host_threads()
    for w in range(args.warmup):
        cpu_evaluation(min(ns, 2000), 'cholesky', w)
    t0 = time.perf_counter()
    steps = [cpu_evaluation(ns, 'cholesky', s_) for s_ in range(args.steps)]
    wall = time.perf_counter() - t0
    base = cpu_sample(n, sizes=(ns, 2 * ns), repeats=(1, 1), full=full, eigen_n=2 * ns)
    base['step_sample'] = {'n': ns, 'steps': args.steps, 'mean_s': wall / max(args.steps, 1),
                           'min_s': min(a + b for a, b, _ in steps), 'max_s': max(a + b for a, b, _ in steps)}
    base['cores'] = cores
    v = base['value']
    line = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * wall / max(args.steps, 1), 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': bench_config(n, -(-n // 128) * 128, 2),
            'step_definition': 'a step is a bounded sample: one whole reference evaluation at n=%d; value = 1 / seconds of '
                               'the one evaluation measured at n=%d in this run (extrapolated: %s); the CPU arm does not '
                               'scale with --gpus (one host)' % (ns, n, base['extrapolated']),
            'cpu_baseline': base,
            'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# ------------------------------------------------------------------- secondary workloads (reported, not the metric)
def secondary_measurements():
    """Bounded (~20 s) measurements of the other BASELINE.json configs on one GPU: configs[2] grid sweep at n = 8000
    (cells/s for one rho group) and configs[3] sparse n = 2^20 (generation, SpMM bandwidth, SLQ logdet + Hutchinson
    tr(Kn^-1 dK) evaluation). HBM roofline fractions use MEASURED_PEAKS.json's hbm_gbs when present."""
    import torch
    from gaussian_proc.sweep import likelihood_grid
    from gaussian_proc._sparse import generate_sparse_correlation, SparseEngine
    hbm = 6536.7
    try:
        hbm = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs']
    except Exception:  # noqa: BLE001
        pass
    out = {}
    # configs[2]: one rho group (K generated once) x 8 eta values at n = 8000
    pts, z, X = make_inputs(8000)
    etas = numpy.logspace(-2, 2, 16)
    likelihood_grid(pts, z, X, NU, [0.1, 0.2], etas[:4])      # same shapes: allocator and kernel attributes warm
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    G = likelihood_grid(pts, z, X, NU, [0.1, 0.15, 0.2], etas)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    out['sweep_n8k'] = {'cells': int(G.shape[0] * G.shape[1]), 'cells_per_s': G.shape[0] * G.shape[1] / dt,
                        'workload': 'configs[2] slice: n=8000, 3 rho x 16 eta, l^ + d/d eta + d/d rho per cell',
                        'tflops': G.shape[0] * G.shape[1] * 8000.0 ** 3 / dt * 1e-12}
    # the same rows through imate_method='eigenvalue' (the reference's default) on the library's own kernels: one Householder
    # tridiagonalisation + bisection per rho (csrc/gp_eig.cu), then O(n p) per eta for l^ and d l^/d eta
    etas64 = numpy.logspace(-2, 2, 64)
    likelihood_grid(pts, z, X, NU, [0.1], etas64[:2], method='eigenvalue', with_rho=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Ge = likelihood_grid(pts, z, X, NU, [0.1, 0.2], etas64, method='eigenvalue', with_rho=False)
    torch.cuda.synchronize()
    dte = time.perf_counter() - t0
    out['sweep_n8k_eigenvalue'] = {'cells': int(Ge.shape[0] * Ge.shape[1]), 'cells_per_s': Ge.shape[0] * Ge.shape[1] / dte,
                                   'seconds_per_rho': dte / Ge.shape[0],
                                   'workload': 'configs[2] rows: n=8000, 2 rho x 64 eta (l^ and d/d eta), one tridiagonalisation + '
                                               'bisection per rho on own kernels (gp_sytrd_f64, gp_stebz_f64), no library eigensolver'}
    # configs[3]: sparse n = 2^20, nu = 0.5, rho = 0.005, density 1e-3
    n = 2 ** 20
    numpy.random.seed(0)
    sp = numpy.random.rand(n, 2)
    sp.setflags(write=False)       # (content keys of read-only arrays are cached: no digest per generation)
    scale = numpy.array([0.005, 0.005])
    opts = {'seed': 0, 'lanczos_degree': 30}

    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    _, zs, Xs = make_inputs(n)      # same seed 0 points as sp

    def build():
        Kc = generate_sparse_correlation(sp, scale, 0.5, 1e-3, device=True, with_derivative=True)
        return Kc, SparseEngine(Kc, 'slq', opts)

    def loglik_grad():
        """the public call: generate_correlation(sparse) -> MixedCorrelation -> ProfileLikelihood (l^, d/d eta, d/d rho)"""
        Kc = generate_sparse_correlation(sp, scale, 0.5, 1e-3, device=True, with_derivative=True)
        Km = MixedCorrelation(Kc, imate_method='slq', imate_options=opts)
        return ProfileLikelihood.log_likelihood_and_gradient(zs, Xs, Km, 10.0)

    build()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    K = generate_sparse_correlation(sp, scale, 0.5, 1e-3, device=True, with_derivative=True)
    torch.cuda.synchronize()
    tg = time.perf_counter() - t0
    eng = SparseEngine(K, 'slq', opts)
    torch.cuda.synchronize()
    tb = time.perf_counter() - t0 - tg
    spm = {}
    for B in (1, 16):
        V = eng.probes(0, B)
        eng.spmm(1.0, V)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            eng.spmm(1.0, V)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / 10
        gbs = (12.0 * K.nnz + 4.0 * (n + 1) + 16.0 * n * B) / ms * 1e-6
        spm['B%d' % B] = {'ms': ms, 'algorithmic_GBs': gbs, 'frac_of_measured_hbm': gbs / hbm,
                          'useful_GFLOPs': 2.0 * K.nnz * B / ms * 1e-6}
    eta = 10.0     # lambda_min(K) ~ -1.2 for this hard-thresholded matrix: eta = 1 is indefinite (SURVEY Q11)

    def evaluate(e, eta_):
        e._slq_cache = {}
        ld_ = e.logdet(eta_)
        info_ = dict(e.last_info)
        ti_ = e.traceinv(eta_)
        tr_ = e.traceinv_dK(eta_)
        return ld_, info_, ti_, tr_

    evaluate(eng, eta)                                 # warm (allocations, kernel attributes)
    eng_f = SparseEngine(K, 'slq', opts)               # a fresh operator on the same matrix: no kept Krylov runs yet
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    ld, info, ti, tr = evaluate(eng_f, eta)            # first eta of an operator: pays the Lanczos run
    torch.cuda.synchronize()
    te = time.perf_counter() - t0
    t0 = time.perf_counter()
    evaluate(eng_f, 2.0 * eta)                         # a further eta: served from the kept (shift-invariant) runs
    torch.cuda.synchronize()
    te2 = time.perf_counter() - t0
    del eng_f
    # the same evaluation at a NEW rho: canonical CSR generation + row-blocked build + estimators (the previous
    # operator is released first, as an optimiser loop would: its buffers go back to the caching allocator)
    nnz, fill = K.nnz, eng.fill_ratio
    del K, eng, V
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    K2, eng2 = build()
    evaluate(eng2, eta)
    torch.cuda.synchronize()
    tn = time.perf_counter() - t0
    del K2, eng2
    loglik_grad()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    lgr = loglik_grad()
    torch.cuda.synchronize()
    tl = time.perf_counter() - t0

    # the same evaluation with the operator generated DIRECTLY as row blocks (generate_sparse_operator: no CSR, no block
    # build) - what sweeps and optimisers over rho use
    from gaussian_proc._sparse import generate_sparse_operator

    def loglik_grad_direct():
        Kb = generate_sparse_operator(sp, scale, 0.5, 1e-3, with_derivative=True)
        Km = MixedCorrelation(Kb, imate_method='slq', imate_options=opts)
        return ProfileLikelihood.log_likelihood_and_gradient(zs, Xs, Km, 10.0)

    loglik_grad_direct()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    Kb = generate_sparse_operator(sp, scale, 0.5, 1e-3, with_derivative=True)
    torch.cuda.synchronize()
    tgd = time.perf_counter() - t0
    direct_kind = type(Kb).__name__
    del Kb
    t0 = time.perf_counter()
    lgd = loglik_grad_direct()
    torch.cuda.synchronize()
    tld = time.perf_counter() - t0
    # the reference's headline driver on this matrix: maximum profile likelihood by the root of d l^/d eta
    # (_profile_likelihood.py:244-415); the kept Krylov runs of the operator serve every eta of the root find
    import contextlib
    import io
    t0 = time.perf_counter()
    Kr = generate_sparse_operator(sp, scale, 0.5, 1e-3)
    Kmr = MixedCorrelation(Kr, imate_method='slq', imate_options=opts)
    with contextlib.redirect_stdout(io.StringIO()):
        root = ProfileLikelihood.find_log_likelihood_der1_zeros(zs, Xs, Kmr, [10.0, 1e3])
    torch.cuda.synchronize()
    tr_ = time.perf_counter() - t0
    del Kr, Kmr
    # CPU comparator for the sparse leg, bounded (~15 s): the reference's compiled brute-force generator (O(n^2)) at
    # n = 2^13 extrapolated with n^2, and the operation its SLQ / CG estimators are built on - SciPy's CSR x dense-block
    # product with the same number of non-zeros per row - at n = 2^17 extrapolated linearly in nnz.
    cpu = {}
    try:
        from oracle import matern as omat
        ns = 2 ** 13
        fac = float(n) / ns
        psub = sp[:ns] * 1.0
        args_s = (numpy.array([0.005, 0.005]) * numpy.sqrt(fac), 0.5, 1e-3 * fac)
        kind = 'port (oracle/cmatern.c)'
        gen = lambda: omat.generate_sparse_correlation(psub, *args_s)   # noqa: E731
        try:
            from oracle import ref_loader
            cy = ref_loader.load_cython()
            gen = lambda: cy.generate_sparse_correlation(psub, args_s[0], args_s[1], args_s[2], False)   # noqa: E731
            kind = 'reference (compiled Cython generator)'
        except Exception:  # noqa: BLE001
            pass
        t0 = time.perf_counter()
        Ks = gen()
        tgs = time.perf_counter() - t0
        nm = 2 ** 17
        fm = float(n) / nm
        Km_host = generate_sparse_correlation(sp[:nm] * 1.0, numpy.array([0.005, 0.005]) * numpy.sqrt(fm), 0.5, 1e-3 * fm)
        Vh = numpy.random.randn(nm, 16)
        Km_host @ Vh
        t0 = time.perf_counter()
        for _ in range(3):
            Km_host @ Vh
        tsp = (time.perf_counter() - t0) / 3 * (nnz / float(Km_host.nnz))
        n_spmm16, n_spmm8 = 31, 25
        cpu = {'kind': kind, 'cores': os.cpu_count(),
               'generate_s_extrapolated': tgs * fac ** 2, 'generate_sample': 'n=%d in %.2f s, x (n/ns)^2' % (ns, tgs),
               'spmm_B16_s_extrapolated': tsp, 'spmm_sample': 'scipy CSR @ (n x 16) at n=%d, nnz=%d, x nnz ratio' % (nm, Km_host.nnz),
               'loglik_grad_s_new_rho_extrapolated': tgs * fac ** 2 + (n_spmm16 + 0.5 * n_spmm8) * tsp,
               'note': 'the reference has no working sparse likelihood path (SURVEY Q6, Q8, Q9); this is its generator '
                       'plus %d B=16 and %d B=8 SciPy products, the SpMM count of one evaluation here' % (n_spmm16, n_spmm8)}
    except Exception as exc:  # noqa: BLE001
        cpu = {'unavailable': repr(exc)[:200]}
    out['sparse_n1M'] = {'workload': 'configs[3]: n=2^20 random 2-D points, nu=0.5, rho=0.005, density=1e-3, eta=10',
                         'nnz': nnz, 'generate_s': tg, 'generate_GBs': (20.0 * nnz + 4.0 * (n + 1)) / tg * 1e-9,
                         'row_blocked_build_s': tb, 'row_blocked_fill_ratio': fill,
                         'spmm': spm, 'spmm_kernel': 'gp::bcsr8_spmm_dmma_kernel<B, DOT, 2> (16x1 row blocks, two DMMA.8x8x4 per gathered fragment)',
                         # the sparse hot kernel against the HBM roofline (B = 16, the estimators' batch): algorithmic bytes =
                         # 12 nnz + 4 (n + 1) + 16 n B; traffic = dram read + write of one launch from the ncu --set full capture
                         # in profiles/r01_spmm_ncu_summary.md (16 x 1 blocks: DRAM 77 % of peak, L1 data pipe 70 % at B = 16)
                         'spmm_roofline': {'bound': 'hbm', 'achieved': spm['B16']['algorithmic_GBs'], 'peak': hbm, 'unit': 'GB/s',
                                           'frac': spm['B16']['frac_of_measured_hbm'], 'traffic': 4.491e9,
                                           'algorithmic_bytes': 12.0 * nnz + 4.0 * (n + 1) + 16.0 * n * 16},
                         'evals_per_s': 1.0 / te, 'evals_per_s_further_eta': 1.0 / te2, 'evals_per_s_new_rho': 1.0 / tn,
                         'loglik_grad_evals_per_s_new_rho': 1.0 / tl, 'loglik_grad': [float(v) for v in lgr],
                         'direct_operator': {'what': 'generate_sparse_operator: the 16-row blocks straight from the cell lists '
                                                     '(replaces CSR generation + row-blocked build)', 'handle': direct_kind,
                                             'generate_s': tgd, 'loglik_grad_evals_per_s_new_rho': 1.0 / tld,
                                             'loglik_grad': [float(v) for v in lgd],
                                             'rel_diff_vs_csr_path': [abs(a - b) / max(abs(b), 1e-300) for a, b in zip(lgd, lgr)]},
                         'mle_root_find_s': tr_, 'mle_root': {k: float(v) for k, v in root.items()},
                         'eval': 'SLQ logdet + traceinv (degree 30, <= 50 Rademacher probes, batch 16, rtol 1e-2 @ 95 %) + '
                                 'Hutchinson tr(Kn^-1 dK/drho) at the first eta of an operator; further_eta = another eta served from the kept '
                                 'Krylov runs; new_rho adds CSR generation and the row-blocked build; loglik_grad = the '
                                 'whole profile likelihood + gradient through the public API (adds the CG solves for [X z], m = 6)',
                         'logdet': ld, 'logdet_half_width': float(info['half_width'][0]), 'num_samples': info['num_samples'],
                         'traceinv': ti, 'trace_Kninv_dK': tr, 'cpu_comparator': cpu}
    return out


def _timed_max_ms(fn, world):
    """Runs fn() between a barrier + synchronize on both sides, timed with CUDA events on the current stream (everything
    the library enqueues is ordered after / joined into it); returns (result, milliseconds as the MAX over ranks)."""
    import torch
    import torch.distributed as dist
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    res = fn()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return res, float(ms.item())


def sharded_measurements(world, rank):
    """The workloads of BASELINE.json that SHARD across GPUs, run by every rank at every --gpus N (N = 1 included, as the
    base of the scaling curve), each a FIXED total amount of work (strong scaling):
      C3  configs[2]: (rho x eta) grid of cells at n = 8000, contiguous rho groups per rank, results all-gathered;
      C4  configs[3]: ONE sparse n = 2^20 loglik + gradient with the Hutchinson / SLQ probes split over the ranks
                      (all-reduce of count / sum / sum of squares), and a sparse (rho x eta) sweep;
      C5  configs[4]: dense n = 100 000, block-cyclic distributed Cholesky with NCCL panel broadcasts, l^ + gradient.
    Collective per workload (the limiting one is named in DESIGN.md section 6)."""
    import torch
    from gaussian_proc.sweep import likelihood_grid
    from gaussian_proc._sparse import generate_sparse_operator
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    out = {}

    # ---- C3: 32 rho x 16 eta = 512 cells at n = 8000 (one eighth of the 64 x 64 grid; the same cells at every N)
    pts, z, X = make_inputs(8000)
    rhos, etas = numpy.linspace(0.05, 0.3, 32), numpy.logspace(-2, 2, 16)
    likelihood_grid(pts, z, X, NU, rhos[:world], etas[:4])                      # warm: allocator, kernel attributes
    G, ms = _timed_max_ms(lambda: likelihood_grid(pts, z, X, NU, rhos, etas), world)
    cells = G.shape[0] * G.shape[1]
    out['C3_sweep_n8k'] = {'workload': 'configs[2] slice: n=8000, 32 rho x 16 eta = 512 cells (l^, d/d eta, d/d rho each)',
                           'scaling': 'strong', 'cells': int(cells), 'seconds': ms * 1e-3, 'cells_per_s': cells / (ms * 1e-3),
                           'tflops_per_gpu': cells * 8000.0 ** 3 / (ms * 1e-3) / world * 1e-12,
                           'collective': 'one all_gather of 5 doubles per cell at the end',
                           'checksum': float(numpy.sum(G[:, :, 0]))}
    del G
    torch.cuda.empty_cache()

    # ---- C4: sparse n = 2^20
    n = 2 ** 20
    sp, zs, Xs = make_inputs(n)
    scale = numpy.array([0.005, 0.005])
    opts = {'seed': 0, 'lanczos_degree': 30}

    def sparse_eval(split):
        Kc = generate_sparse_operator(sp, scale, 0.5, 1e-3, with_derivative=True)
        o = dict(opts)
        o['probe_split'] = bool(split)
        Km = MixedCorrelation(Kc, imate_method='slq', imate_options=o)
        r = ProfileLikelihood.log_likelihood_and_gradient(zs, Xs, Km, 10.0)
        return [float(v) for v in r], int(Km.engine.last_info.get('num_samples', 0))

    sparse_eval(True)
    sparse_eval(False)          # (warm both variants: the unsplit one keeps twice the Lanczos vectors - allocator growth)
    (r_split, ns_split), ms_split = _timed_max_ms(lambda: sparse_eval(True), world)
    (r_single, ns_single), ms_single = _timed_max_ms(lambda: sparse_eval(False), world)
    out['C4_sparse_n1M_probe_split'] = {
        'workload': 'configs[3]: ONE loglik+grad at n=2^20 (nu=0.5, rho=0.005, density=1e-3, eta=10): CSR generation + '
                    'row-blocked build + CG for [X z] (replicated) + SLQ / Hutchinson probes split over the ranks',
        'scaling': 'strong', 'seconds': ms_split * 1e-3, 'evals_per_s': 1e3 / ms_split,
        'seconds_unsplit_same_run': ms_single * 1e-3, 'speedup_vs_unsplit': ms_single / ms_split,
        'num_samples': ns_split, 'loglik_grad': r_split,
        'rel_diff_vs_unsplit': [abs(a - b) / max(abs(b), 1e-300) for a, b in zip(r_split, r_single)],
        'collective': 'all_reduce of (count, failed, sum, sum of squares) per estimator round'}
    # the same evaluation with the ROWS of the operator cut into one slab per GPU (gaussian_proc/_slab.py): generation, build
    # and every Krylov vector are 1/N per rank; halo rows of the SpMM input are loaded from the owner's memory over NVLink and
    # the Lanczos / CG reductions are summed inside the reduction kernels through peer mailboxes (no library collective)
    def slab_eval():
        Kc = generate_sparse_operator(sp, scale, 0.5, 1e-3, with_derivative=True, row_slab=(rank, world))
        o = dict(opts)
        o['row_slabs'] = True
        Km = MixedCorrelation(Kc, imate_method='slq', imate_options=o)
        r = ProfileLikelihood.log_likelihood_and_gradient(zs, Xs, Km, 10.0)
        e = Km.engine
        return [float(v) for v in r], (e.halo_blocks, e.halo_rows, e.total_blocks, e.rows)

    def slab_root_find(slabs):
        # the reference's MLE driver (root of d l^/d eta, _profile_likelihood.py:244-415) on the row-slab operator: every
        # rank runs the same bracketing + Chandrupatla iterations on identical numbers
        import contextlib
        import io
        Kc = generate_sparse_operator(sp, scale, 0.5, 1e-3, row_slab=(rank, world) if slabs else None)
        o = dict(opts)
        o['row_slabs'] = bool(slabs)
        Km = MixedCorrelation(Kc, imate_method='slq', imate_options=o)
        with contextlib.redirect_stdout(io.StringIO()):
            return ProfileLikelihood.find_log_likelihood_der1_zeros(zs, Xs, Km, [10.0, 1e3])

    try:
        if world < 2:
            raise RuntimeError('one slab = the single-GPU evaluation above; measured for --gpus >= 2')
        slab_eval()
        (r_slab, halo), ms_slab = _timed_max_ms(slab_eval, world)
        slab_root_find(True)
        root_slab, ms_root_slab = _timed_max_ms(lambda: slab_root_find(True), world)
        slab_root_find(False)
        root_one, ms_root_one = _timed_max_ms(lambda: slab_root_find(False), world)
        out['C4_sparse_n1M_row_slabs'] = {
            'workload': 'configs[3]: ONE loglik+grad at n=2^20 (nu=0.5, rho=0.005, density=1e-3, eta=10) with the operator '
                        'rows in %d slabs, one per GPU: slab generation + slab build + CG for [X z] + SLQ / Hutchinson' % world,
            'scaling': 'strong', 'seconds': ms_slab * 1e-3, 'evals_per_s': 1e3 / ms_slab,
            'seconds_one_gpu_same_run': ms_single * 1e-3, 'speedup_vs_one_gpu': ms_single / ms_slab,
            'loglik_grad': r_slab,
            'rel_diff_vs_one_gpu': [abs(a - b) / max(abs(b), 1e-300) for a, b in zip(r_slab, r_single)],
            'rows_per_gpu': int(halo[3]), 'halo_fraction_of_block_columns': halo[0] / float(max(halo[2], 1)),
            'mle_root_find_s': ms_root_slab * 1e-3, 'mle_root_find_s_one_gpu_same_run': ms_root_one * 1e-3,
            'mle_root': {k: float(v) for k, v in root_slab.items()},
            'mle_root_rel_diff_vs_one_gpu': abs(root_slab['eta'] - root_one['eta']) / abs(root_one['eta']),
            'nvlink_bytes_per_spmm_B16_rank0': int(halo[0]) * 16 * 8,
            'halo_algorithmic_bytes_B16_rank0': int(halo[1]) * 16 * 8,
            'exchange': 'halo rows: loads from the owner GPU inside the SpMM kernel (CUDA IPC mapping, NVLink); reductions: '
                        'in-kernel sum through per-rank mailboxes, 2 per Lanczos step / 3 per CG iteration'}
    except Exception as e:  # noqa: BLE001 -- the other legs must still print
        out['C4_sparse_n1M_row_slabs'] = {'skipped' if world < 2 else 'error': repr(e)[:300]}
    rh, et = numpy.linspace(0.004, 0.006, 8), numpy.logspace(1, 3, 16)
    Gs, ms = _timed_max_ms(lambda: likelihood_grid(sp, zs, Xs, 0.5, rh, et, sparse=True, density=1e-3, imate_options=opts), world)
    out['C4_sparse_sweep_n1M'] = {'workload': 'configs[3] sweep: n=2^20, 8 rho x 16 eta = 128 cells, one CSR + operator per rho',
                                  'scaling': 'strong', 'cells': 128, 'seconds': ms * 1e-3, 'cells_per_s': 128 / (ms * 1e-3),
                                  'collective': 'one all_gather of 5 doubles per cell at the end',
                                  'checksum': float(numpy.sum(Gs[:, :, 0]))}
    del Gs
    torch.cuda.empty_cache()

    # ---- C5: dense n = 100 000 distributed Cholesky (needs >= 2 GPUs for the memory: 80 GB of K + the replicated factor)
    nbig = int(os.environ.get('GP_BENCH_C5_N', '100000' if world >= 2 else '40000'))
    try:
        out['C5_blockcyclic'] = blockcyclic_measurement(nbig, world, rank)
    except Exception as e:  # noqa: BLE001 -- the other legs must still print
        out['C5_blockcyclic'] = {'error': repr(e)[:300]}
    return out


def blockcyclic_measurement(n, world, rank):
    import torch
    from gaussian_proc._blockcyclic import BlockCyclicCholesky
    pts, z, X = make_inputs(n)
    nb = int(os.environ.get('GP_BENCH_C5_NB', '512'))
    bc = BlockCyclicCholesky(pts, 0.1, NU, nb=nb)
    res, ms = _timed_max_ms(lambda: bc.profile_log_likelihood_and_gradient(z, X, 0.1), world)
    st = dict(bc.stats)
    fl_factor = n ** 3 / 3.0
    out = {'workload': 'configs[4]: dense Matern nu=2.5, n=%d, eta=0.1, nb=%d, %d x %d process grid: generation in place, '
                       'distributed Cholesky, l^ + d/d eta + d/d rho' % (n, nb, bc.P_r, bc.P_c),
           'scaling': 'strong', 'seconds_total': ms * 1e-3, 'loglik_grad': [float(v) for v in res],
           'seconds_generate_factor': st.get('factor_s'), 'factor_tflops_total': fl_factor / st['factor_s'] * 1e-12 if st.get('factor_s') else None,
           'factor_tflops_per_gpu': fl_factor / st['factor_s'] / world * 1e-12 if st.get('factor_s') else None,
           'seconds_inverse_rows': st.get('inverse_rows_s'), 'seconds_traces': st.get('traces_s'), 'seconds_solves': st.get('solve_s'),
           'total_tflops_per_gpu': float(n) ** 3 / (ms * 1e-3) / world * 1e-12,
           'bytes_received_per_rank': st.get('bytes_received'), 'nccl_seconds_on_comm_stream': st.get('comm_s'),
           'nccl_fraction_of_factor_time': (st['comm_s'] / st['factor_s']) if st.get('comm_s') is not None and st.get('factor_s') else None,
           'collective': 'panel broadcast (NCCL, side stream, look-ahead 1) per block column; all_reduce of the trace partials'}
    del bc
    torch.cuda.empty_cache()
    return out


DUMP_SAMPLES = 1 << 20


def dump_outputs(directory, out, Kbuf, n, m, eta, flags):
    """Writes what the last timed step of this rank computed as DIR/<name>.npy (float64), so that two builds can be
    compared output for output. run_ours calls it on rank 0 only: under torchrun the files hold rank 0's last cell and
    nothing from the other ranks. fused_out = the evaluator's out[] (logdet, traces, Gram matrices; include/gpgp.h), loglik_grad = the
    (l^, d l^/d eta, d l^/d rho) a caller of ProfileLikelihood.log_likelihood_and_gradient gets from it, and
    correlation_sample = the generated K at DUMP_SAMPLES (row, column) pairs drawn with numpy.random.RandomState(0)."""
    import torch
    from gaussian_proc._likelihood import ProfileLikelihood, _fused
    os.makedirs(directory, exist_ok=True)
    q = _fused.FusedQuantities(out, n, m, eta, flags)
    ij = torch.from_numpy(numpy.random.RandomState(0).randint(0, n, size=(2, DUMP_SAMPLES))).cuda()
    arrays = {'fused_out': out, 'loglik_grad': numpy.array(ProfileLikelihood._gradient_from(q, (n, m), True)),
              'correlation_sample': Kbuf[ij[0], ij[1]].cpu().numpy()}
    for name, a in arrays.items():
        numpy.save(os.path.join(directory, name + '.npy'), numpy.ascontiguousarray(a, dtype=numpy.float64))


# ---------------------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (there is no CPU fallback; use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))

    from gaussian_proc import _device as dev
    from gaussian_proc import generate_correlation
    from gaussian_proc._dense import DeviceCorrelation, DenseEngine, FLAG_TRACEINV, FLAG_INVERSE, FLAG_DRHO
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    lib = dev.lib

    n = int(os.environ.get('GP_BENCH_N', '20000'))
    pts, z, X = make_inputs(n)
    m = X.shape[1]
    p = m + 1
    npad = dev.padded_size(n)
    P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731

    # ---- resident inputs -------------------------------------------------------------------------------------
    # `cells_in_flight` independent evaluations are kept in flight per GPU, each with its own K buffer / scratch and its
    # own CUDA stream (the latency-bound phases of one evaluation - diagonal blocks, small recursion levels, the
    # HBM-bound reductions - are filled by the GEMMs of another; the grid sweep does the same, gaussian_proc/sweep.py)
    dpts = torch.from_numpy(numpy.array(pts)).cuda()         # (pts is a read-only array: copy before wrapping)
    C = max(1, int(args.cells_in_flight))
    slots = []
    for c in range(C):
        Kbuf = torch.empty((npad, npad), dtype=torch.float64, device='cuda')
        Kdev = DeviceCorrelation(n, Kbuf, points=dpts, correlation_scale=numpy.array([0.1, 0.1]), nu=NU)
        slots.append({'Kbuf': Kbuf, 'Kdev': Kdev, 'eng': DenseEngine(Kdev), 'stream': torch.cuda.Stream()})
    R, _ = slots[0]['eng'].pad_rhs(numpy.c_[X, z])
    flags = FLAG_TRACEINV | FLAG_INVERSE | FLAG_DRHO
    results = []
    counter = [0]

    def step(idx):
        eta, rho = cell(idx)
        scale = numpy.array([rho, rho])
        sl = slots[counter[0] % C]
        counter[0] += 1
        with torch.cuda.stream(sl['stream']):
            sl['Kdev'].correlation_scale = scale
            dev.check(lib.gp_matern_dense(P(dpts), n, 2, dev.host_ptr(scale), NU, P(sl['Kbuf']), npad, None,
                                          dev.stream_ptr()), 'gp_matern_dense')
            results.append(sl['eng'].fused(eta, R, p, flags))

    def fork():
        cur = torch.cuda.current_stream()
        for sl in slots:
            sl['stream'].wait_stream(cur)

    def join():
        cur = torch.cuda.current_stream()
        for sl in slots:
            cur.wait_stream(sl['stream'])

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    fork()
    for w in range(max(args.warmup, C)):
        step(w * world + rank)
    join()
    torch.cuda.synchronize()
    results.clear()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    lib.gp_gemm_profile_enable(1)
    launches0 = lib.gp_launch_count()
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fork()
    for s in range(args.steps):
        step((args.warmup + s) * world + rank)
    join()
    stacked = torch.stack(results)
    if world > 1:
        gathered = [torch.empty_like(stacked) for _ in range(world)]
        dist.all_gather(gathered, stacked)        # the only collective: the per-cell results
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    launches = int(lib.gp_launch_count() - launches0)
    gm, gu, gf, gl = ctypes.c_double(), ctypes.c_double(), ctypes.c_double(), ctypes.c_longlong()
    lib.gp_gemm_profile_read(ctypes.byref(gm), ctypes.byref(gu), ctypes.byref(gf), ctypes.byref(gl))
    lib.gp_gemm_profile_enable(0)
    clocks = sampler.stop() if rank == 0 else None
    host = stacked.cpu().numpy()
    if not numpy.isfinite(host[:, :4]).all() or (host[:, 4] != 0).any():
        raise SystemExit('bench.py: non-finite result or Cholesky breakdown in the timed region')
    if args.dump_outputs and rank == 0:
        eta_last = cell((args.warmup + args.steps - 1) * world + rank)[0]
        dump_outputs(args.dump_outputs, host[-1], slots[(counter[0] - 1) % C]['Kbuf'], n, m, eta_last, flags)

    value = args.steps * world / (ms * 1e-3)

    # ---- FP64 GEMM ceiling measured in-run (MEASURED_PEAKS.json carries no FP64 entry) --------------------------
    a = torch.randn(8192, 8192, dtype=torch.float64, device='cuda')
    b = torch.randn(8192, 8192, dtype=torch.float64, device='cuda')
    torch.matmul(a, b)
    best = 1e30
    for _ in range(3):
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record(); torch.matmul(a, b); t1.record(); torch.cuda.synchronize()
        best = min(best, t0.elapsed_time(t1))
    peak_tflops = 2 * 8192.0 ** 3 / best * 1e-9
    del a, b

    # launches on the look-ahead / recursion helper streams overlap: the kernel's busy time is the UNION of the
    # per-launch [start, stop] event intervals, not their sum
    gemm_ms_per_step = gu.value / args.steps
    alg_flops = float(n) ** 3
    achieved = alg_flops / (gemm_ms_per_step * 1e-3) * 1e-12
    roofline = {'bound': 'tensor', 'kernel': 'gp::dgemm_tma_kernel (TMA + mbarrier ring, DMMA.8x8x4 on the FP64 tensor pipe)',
                'achieved': achieved, 'peak': peak_tflops, 'unit': 'TFLOP/s', 'frac': achieved / peak_tflops,
                # dram__bytes_read.sum + dram__bytes_write.sum of the dominant launch (potrf trailing update, 19456^2 lower
                # tiles, K = 512) from the ncu --set full capture summarised in profiles/r02_gemm_tma_ncu_summary.md (2.21 GB read + 1.42 GB written);
                # algorithmic bytes of that launch: 3.12e9 (lower triangle of C read + written, plus the panel)
                'traffic': 3.63e9,
                'peak_source': 'in-run cuBLAS DGEMM 8192^3 (torch.matmul f64, best of 3); MEASURED_PEAKS.json has no FP64 '
                               'entry; raw DMMA issue peak measured by tools/microbench.cu = 37.1 TFLOP/s',
                'algorithmic_flops_per_step': alg_flops,
                'executed_tile_tflops': gf.value / (gu.value * 1e-3) * 1e-12,
                'gemm_ms_per_step_summed_over_streams': gm.value / args.steps,
                'gemm_launches_per_step': gl.value / args.steps,
                'gemm_ms_per_step': gemm_ms_per_step, 'gemm_share_of_step': gemm_ms_per_step / (ms / args.steps),
                'step_tflops': alg_flops / (ms / args.steps * 1e-3) * 1e-12}

    # ---- end-to-end through the public API with host (pinned) buffers ----------------------------------------------
    del slots, results, stacked, Kbuf, Kdev
    torch.cuda.empty_cache()
    pin = lambda a: torch.from_numpy(numpy.ascontiguousarray(a)).pin_memory().numpy()  # noqa: E731
    hp, hz, hX = pin(pts), pin(z), pin(X)
    e2e_steps = max(2 * C, min(args.steps, 6))
    streams = [torch.cuda.Stream() for _ in range(C)]

    def e2e_run(first, count):
        """`count` evaluations through the public API, C in flight (log_likelihood_and_gradient_async returns a
        completion callable; its result is read back - D2H of out[] - when the slot is needed again)"""
        pending, last = [], None
        for k in range(count):
            eta, rho = cell((first + k) * world + rank)
            if len(pending) >= C:
                last = pending.pop(0)()
            with torch.cuda.stream(streams[k % C]):
                K = generate_correlation(hp, rho, NU, device=True)                 # H2D: points
                Km = MixedCorrelation(K)
                pending.append(ProfileLikelihood.log_likelihood_and_gradient_async(hz, hX, Km, eta))   # H2D: [X z]
        for fin in pending:
            last = fin()                                                           # D2H: out[]
        return last
    e2e_run(0, C)
    sync_all()
    t0 = time.perf_counter()
    r = e2e_run(C, e2e_steps)
    sync_all()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e = {'value': e2e_steps * world / float(e2e_s.item()), 'unit': UNIT, 'steps': e2e_steps,
           'h2d_bytes_per_step': int(hp.nbytes + npad * p * 8), 'd2h_bytes_per_step': int((8 + 3 * p * p) * 8),
           'cells_in_flight': C,
           'api': 'generate_correlation(points, rho, nu, device=True) -> MixedCorrelation(K) -> '
                  'ProfileLikelihood.log_likelihood_and_gradient_async(z, X, K_mixed, eta)() ',
           'last_result': [float(v) for v in r]}

    # ---- the headline line is complete here; everything below is reported alongside it -------------------------------------
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': bench_config(n, npad, C),
            'gpu_launches': launches, 'clocks': clocks, 'roofline': roofline, 'e2e': e2e}
    printed = threading.Lock()

    def emit(extra):
        """prints the ONE JSON line (rank 0), exactly once"""
        if printed.acquire(blocking=False):
            if rank == 0:
                out = dict(line)
                out.update(extra)
                print(json.dumps(out), flush=True)

    # Watchdog: the secondary legs contain collectives; if one rank fails inside them the others would wait forever and the
    # headline would never be printed. After the deadline rank 0 prints the line without the unfinished legs and every
    # rank leaves.
    deadline = float(os.environ.get('GP_BENCH_SECONDARY_TIMEOUT', '600'))

    def watchdog():
        emit({'secondary': {'error': 'secondary measurements did not finish within %.0f s' % deadline}})
        sys.stdout.flush()
        os._exit(0)
    timer = threading.Timer(deadline, watchdog)
    timer.daemon = True
    extra = {}
    if not args.no_secondary:
        timer.start()
        del hp, hz, hX
        torch.cuda.empty_cache()
        try:
            sharded = sharded_measurements(world, rank)
        except Exception as e:  # noqa: BLE001 -- the headline must still print
            sharded = {'error': repr(e)[:300]}
        extra['secondary'] = {'sharded': sharded}
        if world == 1 and rank == 0:
            try:
                extra['secondary'].update(secondary_measurements())
            except Exception as e:  # noqa: BLE001 -- the headline must still print
                extra['secondary']['error'] = repr(e)[:300]
    if world == 1 and rank == 0 and not args.no_cpu:
        # bounded (~30 s): n = 4000 and 8000 measured, n = 20 000 from the n^2 / n^3 fit (flagged); the measured
        # n = 20 000 evaluation is the reference arm's (`bench.py --impl reference`)
        try:
            extra['cpu_baseline'] = cpu_sample(n, full=os.environ.get('GP_BENCH_CPU_FULL', '0') != '0')
        except Exception as e:  # noqa: BLE001
            extra['cpu_baseline'] = {'error': repr(e)[:300]}
    timer.cancel()
    emit(extra)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=8)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--cells-in-flight', type=int, default=2,
                    help='independent evaluations kept in flight per GPU (own buffers and stream each)')
    ap.add_argument('--no-cpu', action='store_true', help='skip the cpu_baseline leg')
    ap.add_argument('--no-secondary', action='store_true', help='skip the sparse / sweep secondary measurements')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the last timed step computed to DIR/<name>.npy (float64, about 8 MB in all); under '
                         'torchrun only rank 0 writes, so the files hold rank 0\'s last cell')
    args = ap.parse_args()
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of the CUDA path (--impl ours)')
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
