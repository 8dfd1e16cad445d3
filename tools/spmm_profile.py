"""Developer profile target: a few SpMMs of the row-blocked operator at n = 2^20 (use under ncu -k regex:spmm)."""
import os, sys
import numpy
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'gaussian-process-param-estimation_b200'))
import torch
from gaussian_proc._sparse import generate_sparse_correlation, SparseEngine

n = int(sys.argv[1]) if len(sys.argv) > 1 else 2 ** 20
B = int(sys.argv[2]) if len(sys.argv) > 2 else 16
numpy.random.seed(0)
pts = numpy.random.rand(n, 2)
K = generate_sparse_correlation(pts, numpy.array([0.005, 0.005]), 0.5, 1e-3, device=True)
e = SparseEngine(K, 'slq', {})
V = e.probes(0, B)
for _ in range(3):
    Y = e.spmm(1.0, V)
torch.cuda.synchronize()
print('ok', float(Y[0, 0]))
