"""Developer timing of the gradients of the prediction (Predictor.predict_gradient, gaussian_proc/_predict.py) at
n = m* = 20 000 (nu = 2.5, rho = 0.1, d = 2), in chunks of 8192 test points: the U = W^T V GEMM (gp_dgemm_ktab_f64,
W^T upper) and the gradient pass gp_predict_grad_dense, each timed with CUDA events around the library calls the predictor
makes, plus predict() and predict_gradient() end to end. Prints one JSON line with the card name and power limit.
Usage: python tools/predict_grad_timing.py [n] [m*]"""
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


def wall(fn):
    torch.cuda.synchronize(); t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0


pts, z, X = bench.make_inputs(n)
tp = numpy.random.RandomState(1).rand(ms, 2)
Xs = du.generate_basis_functions(tp, 2)
# Jacobian of the degree-2 monomials, in generate_basis_functions' column order (meshgrid of the powers, filtered by sum)
powers = numpy.array([g.ravel() for g in numpy.meshgrid(numpy.arange(3), numpy.arange(3))])
powers = powers[:, powers.sum(axis=0) <= 2].T
Xg = numpy.zeros((ms, 2, Xs.shape[1]))
for c, (ex, ey) in enumerate(powers):
    if ex:
        Xg[:, 0, c] = ex * tp[:, 0] ** (ex - 1) * tp[:, 1] ** ey
    if ey:
        Xg[:, 1, c] = ey * tp[:, 1] ** (ey - 1) * tp[:, 0] ** ex
assert numpy.allclose(Xs, numpy.stack([tp[:, 0] ** ex * tp[:, 1] ** ey for ex, ey in powers], axis=1))
Km = MixedCorrelation(gaussian_proc.generate_correlation(pts, rho, nu, device=True))
pr = Predictor(Km, X, z, eta)
eng, K = Km.engine, Km.K
npad, p, d = K.npad, pr.p, 2
out = {'gpu': torch.cuda.get_device_name(0), 'n': n, 'm_star': ms, 'chunk': chunk, 'nu': nu, 'rho': rho, 'eta': eta, 'd': d}
try:
    out['power_limit'] = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                                        capture_output=True, text=True).stdout.strip()
except OSError:
    out['power_limit'] = None
eng._trtri(eta)

# the predictor's chunk loop, one library call at a time
mcpad = dev.padded_size(chunk)
qd = torch.from_numpy(numpy.ascontiguousarray(tp)).cuda()
Pb = torch.empty((npad, mcpad), dtype=torch.float64, device='cuda')
Vb = torch.empty((npad, mcpad), dtype=torch.float64, device='cuda')
ws = torch.empty(lib.gp_predict_workspace_bytes(npad, chunk, p) // 8, dtype=torch.float64, device='cuda')
gws = torch.empty(lib.gp_predict_grad_workspace_bytes(n, chunk, d, p) // 8, dtype=torch.float64, device='cuda')
ob = torch.empty(chunk * (p + 1) * (1 + d), dtype=torch.float64, device='cuda')
kbeg = torch.arange(0, npad, 128, dtype=torch.int32, device='cuda')
scale = K.correlation_scale
t_v = t_u = t_grad = 0.0
flops = 0.0
for c0 in range(0, ms, chunk):
    mc = min(chunk, ms - c0)
    mp = dev.padded_size(mc)
    dev.check(lib.gp_matern_cross_points(P_(K.points), n, P_(qd, c0 * d), mc, d, dev.host_ptr(scale), nu, P_(Pb), mcpad, s),
              'cross')
    vgemm = lambda: dev.check(lib.gp_dgemm_f64(0, 1, P_(Vb), mcpad, P_(eng.W), npad, P_(Pb), mcpad, npad, mp, npad, 1.0,
                                               0.0, 1, 0, s), 'v gemm')
    vgemm()
    t_v += timed(vgemm, 3)
    # U overwrites P, as in the predictor; V is not changed by the repeats
    ugemm = lambda: dev.check(lib.gp_dgemm_ktab_f64(1, 1, P_(Pb), mcpad, P_(eng.W), npad, P_(Vb), mcpad, npad, mp, npad,
                                                    1.0, 0.0, P_(kbeg), None, s), 'u gemm')
    grad = lambda: dev.check(lib.gp_predict_grad_dense(P_(K.points), n, P_(qd, c0 * d), mc, d, dev.host_ptr(scale), nu,
                                                       P_(pr.S), p, P_(Pb), mcpad, P_(ob), P_(gws), s), 'grad')
    ugemm(); grad()                         # warm-up of every shape
    t_u += timed(ugemm, 3)
    t_grad += timed(grad, 3)
    flops += float(n) * n * mc
out['v_gemm_s'] = t_v
out['u_gemm_s'] = t_u
out['u_gemm_TFLOPs'] = flops / t_u * 1e-12          # n^2 m* flop for the triangular product, as for V
out['grad_kernel_s'] = t_grad
del Pb, Vb
pr.predict(tp, Xs, chunk_size=chunk)
pr.predict_gradient(tp, Xs, Xg, chunk_size=chunk)
out['predict_s'] = wall(lambda: pr.predict(tp, Xs, chunk_size=chunk))
out['predict_gradient_s'] = wall(lambda: pr.predict_gradient(tp, Xs, Xg, chunk_size=chunk))
out['predict_gradient_mean_only_s'] = wall(lambda: pr.predict_gradient(tp, Xs, Xg, return_var=False, chunk_size=chunk))
print(json.dumps(out), flush=True)
