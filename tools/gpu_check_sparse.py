"""Developer timing (GPU): sparse n = 2^20 path (BASELINE configs[3]): generation, SpMM bandwidth, SLQ, Hutchinson."""
import ctypes, json, os, sys, time
import numpy
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'gaussian-process-param-estimation_b200'))
import torch
from gaussian_proc import _device as dev
from gaussian_proc._sparse import generate_sparse_correlation, SparseEngine, DeviceCSR

def timed(fn, reps=1):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(reps): r = fn()
    torch.cuda.synchronize(); return (time.perf_counter() - t0) / reps, r

n = int(sys.argv[1]) if len(sys.argv) > 1 else 2 ** 20
nu = float(sys.argv[2]) if len(sys.argv) > 2 else 0.5
numpy.random.seed(0)
pts = numpy.random.rand(n, 2)
out = {'n': n, 'nu': nu}
gen = lambda: generate_sparse_correlation(pts, numpy.array([0.005, 0.005]), nu, 1e-3, device=True, with_derivative=True)
gen()
out['t_generate_s'], K = timed(gen)
out['nnz'] = K.nnz
out['generate_GBs'] = (20.0 * K.nnz + 4.0 * (n + 1)) / out['t_generate_s'] * 1e-9
# plain CSR (the same matrix without its spatial order) against the 16-row blocks
Kcsr = DeviceCSR(n, K.indptr, K.indices, K.data, K.ddata, kernel_threshold=K.kernel_threshold, sorted_rows=K.sorted_rows)
for name, Kop in (('R1', Kcsr), ('R16', K)):
    SparseEngine(Kop, 'slq', {})
    t, e = timed(lambda: SparseEngine(Kop, 'slq', {}))
    out[name] = {'build_s': t, 'fill_ratio': getattr(e, 'fill_ratio', 1.0)}
    for B in (1, 8, 16, 32):
        V = e.probes(0, B)
        e.spmm(1.0, V)
        t, _ = timed(lambda: e.spmm(1.0, V), 10)
        out[name]['spmm_B%d_ms' % B] = t * 1e3
        out[name]['spmm_B%d_algGBs' % B] = (12.0 * K.nnz + 4.0 * (n + 1) + 16.0 * n * B) / t * 1e-9
    del e
    torch.cuda.empty_cache()
eng = SparseEngine(K, 'slq', {'seed': 0, 'lanczos_degree': 30})
# extreme Ritz values of K itself (eta = 0) from one 60-step Lanczos run: tells which eta keep K + eta I positive
from gaussian_proc._sparse import lanczos_quadrature
import torch as _t
Vp = eng.probes(0, 1)
al = _t.empty((60, 1), dtype=_t.float64, device='cuda'); be = _t.empty((60, 1), dtype=_t.float64, device='cuda')
P = lambda t: ctypes.c_void_p(t.data_ptr())
dev.lib.gp_lanczos(P(K.indptr), P(K.indices), P(K.data), n, 0.0, P(Vp), 1, 60, P(al), P(be), None, P(eng._workspace(1)), dev.stream_ptr())
import scipy.linalg
th = scipy.linalg.eigh_tridiagonal(al.cpu().numpy()[:, 0], be.cpu().numpy()[:59, 0], eigvals_only=True)
out['ritz_min_max_of_K'] = [float(th.min()), float(th.max())]
etas = [e for e in (1.0, 10.0, 100.0) if e + th.min() > 0.05]
out['etas_used'] = etas
for eta in etas:
    for rep in range(2):      # second pass = warm
        eng._slq_cache = {}
        t, ld = timed(lambda: eng.logdet(eta))
        t2, tr = timed(lambda: eng.traceinv_dK(eta))
    out['slq_eta%g' % eta] = {'t_s': t, 'logdet': ld, 'info': {k: (v.tolist() if hasattr(v, 'tolist') else v) for k, v in eng.last_info.items()}}
    out['hutch_dK_eta%g' % eta] = {'t_s': t2, 'value': tr, 'cg_iters': getattr(eng, 'last_cg_iterations', None), 'dk_solver': getattr(eng, 'last_dk_solver', None), 'samples': eng.last_info['num_samples']}
    out['evals_per_s_eta%g' % eta] = 1.0 / (t + t2)
# raw driver timings (CUDA events): one 30-step Lanczos and one CG solve at B = 16
V = eng.probes(0, 16)
import ctypes as _c
bptr, bidx, bvals, _ = eng.blocked
al = torch.empty((30, 16), dtype=torch.float64, device='cuda'); be = torch.empty((30, 16), dtype=torch.float64, device='cuda')
ws = eng._workspace(16)
def lz():
    dev.lib.gp_bcsr_lanczos(None, P(bptr), P(bidx), P(bvals), n, 10.0, P(V), 16, 30, P(al), P(be), None, P(ws), dev.stream_ptr())
lz()
t, _ = timed(lz, 3)
out['lanczos30_B16_ms'] = t * 1e3
def cg():
    eng.solve_dev(10.0, V.clone())
cg()
t, _ = timed(cg, 3)
out['cg_B16_ms'] = t * 1e3
out['cg_iters'] = eng.last_cg_iterations
print(json.dumps(out))
