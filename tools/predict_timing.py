"""Developer timing of prediction at new points (gaussian_proc/_predict.py) at n = m* = 20 000 (nu = 2.5, rho = 0.1), in
chunks of 8192 test points: factor + triangular inverse, cross-correlation generation, the V = W P GEMM and the reduction
pass, each timed with CUDA events around the library calls the predictor makes (the reduction is gp_predict_dense minus the
same GEMM timed on its own), plus the end-to-end predict() and the covariance GEMM at m* = 8192. Prints one JSON line.
Usage: python tools/predict_timing.py [n] [m*]"""
import ctypes, json, os, subprocess, sys, time
import numpy
ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, 'gaussian-process-param-estimation_b200'))
import torch
import bench, gaussian_proc
from gaussian_proc import _device as dev
from gaussian_proc._mixed_correlation import MixedCorrelation
from gaussian_proc._predict import Predictor
from oracle import data_utilities as du

n = int(sys.argv[1]) if len(sys.argv) > 1 else 20000
ms = int(sys.argv[2]) if len(sys.argv) > 2 else 20000
chunk, eta, rho, nu = 8192, 0.1, 0.1, 2.5
lib, s = dev.lib, dev.stream_ptr()
P_ = lambda t, off=0: ctypes.c_void_p(t.data_ptr() + 8 * off)


def timed(fn, reps=1):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3 / reps


pts, z, X = bench.make_inputs(n)
tp = numpy.random.RandomState(1).rand(ms, 2)
Xs = du.generate_basis_functions(tp, 2)
Km = MixedCorrelation(gaussian_proc.generate_correlation(pts, rho, nu, device=True))
pr = Predictor(Km, X, z, eta)
eng, K = Km.engine, Km.K
npad, p, d = K.npad, pr.p, 2
out = {'gpu': torch.cuda.get_device_name(0), 'n': n, 'm_star': ms, 'chunk': chunk, 'nu': nu, 'rho': rho, 'eta': eta}
try:
    out['power_limit'] = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                                        capture_output=True, text=True).stdout.strip()
except OSError:
    out['power_limit'] = None


def factor_trtri():
    eng.invalidate()
    eng._trtri(eta)


factor_trtri()
out['factor_trtri_s'] = timed(factor_trtri)

# the predictor's chunk loop, one library call at a time
mcpad = dev.padded_size(chunk)
qd = torch.from_numpy(numpy.ascontiguousarray(tp)).cuda()
Pb = torch.empty((npad, mcpad), dtype=torch.float64, device='cuda')
Vb = torch.empty((npad, mcpad), dtype=torch.float64, device='cuda')
ws = torch.empty(lib.gp_predict_workspace_bytes(npad, chunk, p) // 8, dtype=torch.float64, device='cuda')
ob = torch.empty(chunk * (p + 1), dtype=torch.float64, device='cuda')
scale = K.correlation_scale
t_cross = t_gemm = t_pred = 0.0
bytes_cross = flops_gemm = 0.0
for c0 in range(0, ms, chunk):
    mc = min(chunk, ms - c0)
    mp = dev.padded_size(mc)
    cross = lambda: dev.check(lib.gp_matern_cross_points(P_(K.points), n, P_(qd, c0 * d), mc, d, dev.host_ptr(scale), nu,
                                                         P_(Pb), mcpad, s), 'cross')
    gemm = lambda: dev.check(lib.gp_dgemm_f64(0, 1, P_(Vb), mcpad, P_(eng.W), npad, P_(Pb), mcpad, npad, mp, npad, 1.0, 0.0,
                                              1, 0, s), 'gemm')
    pred = lambda: dev.check(lib.gp_predict_dense(P_(eng.W), n, npad, P_(pr.S), p, P_(Pb), mc, mcpad, P_(Vb), mcpad, P_(ob),
                                                  P_(ws), s), 'predict')
    for f in (cross, gemm, pred):          # warm-up of every shape
        f()
    t_cross += timed(cross, 3)
    t_gemm += timed(gemm, 3)
    t_pred += timed(pred, 3)
    bytes_cross += 8.0 * npad * mp
    flops_gemm += float(n) * n * mc
out['cross_s'] = t_cross
out['cross_GBs'] = bytes_cross / t_cross * 1e-9
out['v_gemm_s'] = t_gemm
out['v_gemm_TFLOPs'] = flops_gemm / t_gemm * 1e-12          # n^2 m* flop for the triangular product
out['reduction_s'] = t_pred - t_gemm
pr.predict(tp, Xs, chunk_size=chunk)
torch.cuda.synchronize(); t0 = time.perf_counter()
pr.predict(tp, Xs, chunk_size=chunk)
torch.cuda.synchronize(); out['predict_mean_var_s'] = time.perf_counter() - t0
del Pb, Vb

# covariance at m* = 8192: C = K** - V^T V (lower), one pass over the whole test set
mc = min(8192, ms)
mp = dev.padded_size(mc)
Vc = torch.empty((npad, mp), dtype=torch.float64, device='cuda')
C = torch.empty((mp, mp), dtype=torch.float64, device='cuda')
Vc.normal_()
cov = lambda: dev.check(lib.gp_dgemm_f64(1, 1, P_(C), mp, P_(Vc), mp, P_(Vc), mp, mp, mp, npad, -1.0, 1.0, 0, 1, s), 'cov')
cov()
out['cov_m_star'] = mc
out['cov_gemm_s'] = timed(cov, 3)
out['cov_gemm_TFLOPs'] = float(n) * mc * mc / out['cov_gemm_s'] * 1e-12  # lower triangle of V^T V: n m*^2 flop
del Vc, C
pr.predict(tp[:mc], Xs[:mc], return_cov=True)
torch.cuda.synchronize(); t0 = time.perf_counter()
pr.predict(tp[:mc], Xs[:mc], return_cov=True)
torch.cuda.synchronize(); out['predict_with_cov_s'] = time.perf_counter() - t0
print(json.dumps(out), flush=True)
