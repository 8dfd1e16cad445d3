"""Developer check (torchrun, one rank per GPU): the row-slab sparse engine (gaussian_proc/_slab.py) against the single-GPU
engine on the same matrix: peer all-reduce, SpMM, CG, then the whole loglik + gradient; timing of a new-rho evaluation.
Arguments: [n] [aniso]. With `aniso` the run compares the per-dimension gradient of an anisotropic scale after the
operator pieces and stops there."""
import ctypes, json, os, sys, time
import numpy
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', 'gaussian-process-param-estimation_b200'))
import torch
import torch.distributed as dist
world = int(os.environ.get('WORLD_SIZE', '1')); rank = int(os.environ.get('RANK', '0')); local = int(os.environ.get('LOCAL_RANK', '0'))
torch.cuda.set_device(local)
if world > 1:
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    dist.init_process_group('nccl', device_id=torch.device('cuda', local))
from gaussian_proc import _device as dev
from gaussian_proc._sparse import generate_sparse_correlation, generate_sparse_operator, SparseEngine
DIRECT = os.environ.get('GP_SLAB_DIRECT', '1') != '0'     # operators generated directly as row blocks (default) or via CSR
from gaussian_proc._slab import SlabSparseEngine, PeerArena
lib = dev.lib
P = lambda t: ctypes.c_void_p(t.data_ptr())  # noqa: E731
n = int(sys.argv[1]) if len(sys.argv) > 1 else 2 ** 17
out = {'world': world, 'n': n}

# ---- 1. in-kernel all-reduce: 300 exchanges back to back, rank-dependent values
arena = PeerArena.get(rank, world, 4096)
v = torch.arange(256, dtype=torch.float64, device='cuda') * (rank + 1)
ok = True
for it in range(300):
    w = v + it
    lib.gp_peer_allreduce(arena.ctx, P(w), 256, dev.stream_ptr())
    want = torch.arange(256, dtype=torch.float64, device='cuda') * (world * (world + 1) / 2) + it * world
    ok = ok and bool((w == want).all().item())
torch.cuda.synchronize()
t0 = time.perf_counter()
for it in range(1000):
    lib.gp_peer_allreduce(arena.ctx, P(v), 32, dev.stream_ptr())
torch.cuda.synchronize()
out['allreduce_ok'] = ok
out['allreduce_us'] = (time.perf_counter() - t0) * 1e3
out['peer_error'] = lib.gp_peer_error(arena.ctx, dev.stream_ptr())
if rank == 0:
    print(json.dumps(out), flush=True)

# ---- 2. operator pieces on a mid-size matrix
numpy.random.seed(0)
pts = numpy.random.rand(n, 2)
rho = 0.005 * numpy.sqrt(2 ** 20 / n)
dens = min(0.05, 1e-3 * 2 ** 20 / n)
z = numpy.sin(pts[:, 0] * 7) + numpy.cos(pts[:, 1] * 5) + 0.1 * numpy.random.randn(n)
X = numpy.stack([numpy.ones(n), pts[:, 0], pts[:, 1], pts[:, 0] ** 2, pts[:, 0] * pts[:, 1], pts[:, 1] ** 2], axis=1)
for arr in (pts, z, X):
    arr.setflags(write=False)      # (content keys of read-only arrays are cached: no digest per evaluation)
K = generate_sparse_correlation(pts, numpy.array([rho, rho]), 0.5, dens, device=True, with_derivative=True)
opts = {'seed': 0, 'lanczos_degree': 30}
one = SparseEngine(K, 'slq', dict(opts, overlap=False))
slab = SlabSparseEngine(K, 'slq', opts)
out.update({'nnz': K.nnz, 'halo_fraction': slab.halo_fraction, 'rows': slab.rows})
Vfull = torch.from_numpy(numpy.random.randn(n, 8)).cuda()
Y1 = one.from_op(one.spmm(0.5, one.to_op(Vfull)))
Y2 = slab.from_op(slab.spmm(0.5, slab.to_op(Vfull)))
out['spmm_max_abs_diff'] = float((Y1 - Y2).abs().max().item())
D1 = one.from_op(one.spmm(0.0, one.to_op(Vfull), derivative=True))
D2 = slab.from_op(slab.spmm(0.0, slab.to_op(Vfull), derivative=True))
out['dspmm_max_abs_diff'] = float((D1 - D2).abs().max().item())
S1 = one.from_op(one.solve_dev(10.0, one.to_op(Vfull)))
S2 = slab.from_op(slab.solve_dev(10.0, slab.to_op(Vfull)))
out['cg_rel_diff'] = float(((S1 - S2).abs().max() / S1.abs().max()).item())
out['cg_iters'] = [one.last_cg_iterations, slab.last_cg_iterations]
f1 = one.fused(10.0, X, z)
f2 = slab.fused(10.0, X, z)
out['fused_rel_diff'] = float(numpy.max(numpy.abs(f1 - f2) / numpy.maximum(numpy.abs(f1), 1e-300)))
out['fused_head'] = [f1[:4].tolist(), f2[:4].tolist()]
out['peer_error_after'] = lib.gp_peer_error(slab.peer.ctx, dev.stream_ptr())
if rank == 0:
    print(json.dumps(out), flush=True)

if len(sys.argv) > 2 and sys.argv[2] == 'aniso':
    # ---- anisotropic scale: the per-dimension gradient (d/d scale[k]) on row slabs against one GPU, then stop
    from gaussian_proc._mixed_correlation import MixedCorrelation
    from gaussian_proc._likelihood import ProfileLikelihood
    Ka = generate_sparse_correlation(pts, numpy.array([rho, 1.6 * rho]), 0.5, dens, device=True, with_derivative=True)
    Ms = MixedCorrelation(Ka, imate_method='slq', imate_options=dict(opts, row_slabs=True))
    Mo = MixedCorrelation(Ka, imate_method='slq', imate_options=dict(opts, overlap=False))
    gs = ProfileLikelihood.log_likelihood_and_gradient(z, X, Ms, 10.0)
    go = ProfileLikelihood.log_likelihood_and_gradient(z, X, Mo, 10.0)
    rel = lambda a, b: float(numpy.max(numpy.abs(numpy.asarray(a) - b)) / numpy.max(numpy.abs(b)))   # noqa: E731
    an = {'grad': [gs[0], gs[1], list(gs[2])], 'grad_one_gpu': [go[0], go[1], list(go[2])],
          'grad_rel_diff': max(rel(gs[0], go[0]), rel(gs[1], go[1]), rel(gs[2], go[2])),
          'dscale_rel_diff': rel(Ms.engine.last_dscale, Mo.engine.last_dscale),
          'peer_error': lib.gp_peer_error(Ms.engine.peer.ctx, dev.stream_ptr())}
    if rank == 0:
        print(json.dumps({'aniso': an}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.exit(0)

# ---- 3. timing: fresh operator + evaluation (a new-rho step of an optimiser), slabs against one GPU
def evaluate(cls, phases=None):
    slabbed = issubclass(cls, SlabSparseEngine)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    gen = generate_sparse_operator if DIRECT else (lambda *a, **k: generate_sparse_correlation(*a, device=True, **k))
    Kc = gen(pts, numpy.array([rho, rho]), 0.5, dens, with_derivative=True, row_slab=(rank, world) if slabbed else None)
    torch.cuda.synchronize(); ta = time.perf_counter()
    eng = cls(Kc, 'slq', dict(opts))
    torch.cuda.synchronize(); tb = time.perf_counter()
    if phases is not None:
        for name in ('_rhs_block', 'solve_rhs_block', 'gram', 'spmm', '_slq', 'traceinv_dK'):
            def wrap(fn, name=name):
                def timed(*a, **k):
                    torch.cuda.synchronize(); t = time.perf_counter()
                    r = fn(*a, **k)
                    torch.cuda.synchronize(); phases[name] = phases.get(name, 0.0) + time.perf_counter() - t
                    return r
                return timed
            setattr(eng, name, wrap(getattr(eng, name)))
    r = eng.fused(10.0, X, z)
    torch.cuda.synchronize(); tc = time.perf_counter()
    return r, ta - t0, tb - ta, tc - tb

tm = {}
res = {}
class SlabNoOverlap(SlabSparseEngine):
    def __init__(self, K, method, o):
        SlabSparseEngine.__init__(self, K, method, dict(o, overlap=False))

for name, cls in (('one_gpu', SparseEngine), ('slabs', SlabSparseEngine), ('slabs_no_overlap', SlabNoOverlap)):
    evaluate(cls)
    best = None
    for rep in range(3):
        if world > 1:
            dist.barrier()
        r, tgen, tbuild, tfused = evaluate(cls)
        t = tgen + tbuild + tfused
        if best is None or t < best[0]:
            best = (t, tgen, tbuild, tfused)
    res[name] = r
    ph = {}
    evaluate(cls, ph)
    tm[name] = {'total_s': best[0], 'generate_s': best[1], 'build_s': best[2], 'fused_s': best[3],
                'phases_ms_with_syncs': {k: round(v * 1e3, 3) for k, v in ph.items()}}
tm['speedup_total'] = tm['one_gpu']['total_s'] / tm['slabs']['total_s']
tm['speedup_fused'] = tm['one_gpu']['fused_s'] / tm['slabs']['fused_s']
tm['rel_diff'] = float(numpy.max(numpy.abs(res['one_gpu'] - res['slabs']) / numpy.maximum(numpy.abs(res['one_gpu']), 1e-300)))
if rank == 0:
    print(json.dumps({'timing': tm}), flush=True)
# ---- 4. the Krylov drivers alone (CUDA events): Lanczos m = 30 on 16 probes with / without kept vectors, CG on 8 columns
def ev_ms(fn, reps=3):
    best = 1e30
    for _ in range(reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record(); torch.cuda.synchronize()
        best = min(best, a.elapsed_time(b))
    return best

kr = {}
Kfull = generate_sparse_correlation(pts, numpy.array([rho, rho]), 0.5, dens, device=True, with_derivative=True)
for name, eng in (('one_gpu', SparseEngine(Kfull, 'slq', dict(opts, overlap=False))), ('slabs', SlabSparseEngine(Kfull, 'slq', dict(opts)))):
    V16 = eng.probes(0, 16)
    V8 = eng.probes(0, 8)
    basis = eng._new_basis(30, 16)
    kr[name] = {
        'lanczos_m30_B16_ms': ev_ms(lambda: eng._lanczos_launch(10.0, V16, 30)),
        'lanczos_m30_B16_kept_ms': ev_ms(lambda: eng._lanczos_launch(10.0, V16, 30, basis)),
        'cg_B8_ms': ev_ms(lambda: eng.solve_dev(10.0, V8.clone())),
        'spmm_B16_ms': ev_ms(lambda: eng.spmm(10.0, V16)),
        'spmm_B8_ms': ev_ms(lambda: eng.spmm(10.0, V8)),
    }
    del basis
if rank == 0:
    print(json.dumps({'krylov': kr}), flush=True)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
