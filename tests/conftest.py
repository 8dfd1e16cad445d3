import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, 'gaussian-process-param-estimation_b200')
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


@pytest.fixture(scope='session')
def golden_likelihood():
    import numpy
    return numpy.load(os.path.join(GOLDEN, 'golden_likelihood.npz'))


@pytest.fixture(scope='session')
def golden_generate():
    """The dense matrices are exactly symmetric and stored as their packed lower triangles (`<key>_tril`, row-major
    numpy.tril_indices order) to keep the file small; they are mirrored back to the full matrices here, bit for bit."""
    import numpy
    g = dict(numpy.load(os.path.join(GOLDEN, 'golden_generate.npz')))
    for key in [k for k in g if k.endswith('_tril')]:
        v = g.pop(key)
        n = int(round((numpy.sqrt(8.0 * v.size + 1.0) - 1.0) / 2.0))
        K = numpy.zeros((n, n))
        K[numpy.tril_indices(n)] = v
        K.T[numpy.tril_indices(n)] = v
        g[key[:-len('_tril')]] = K
    return g


@pytest.fixture(scope='session')
def golden_pickles():
    import numpy
    return numpy.load(os.path.join(GOLDEN, 'golden_pickles.npz'))


class RankResults(object):
    """Results of spawned ranks, exchanged through pickle files in a temporary directory. (A multiprocessing.Manager would
    fork() the test process; a fork after the multi-threaded OpenBLAS pool has been used leaves later BLAS calls of the
    parent hanging in this image.)"""

    def __init__(self):
        import tempfile
        self.dir = tempfile.mkdtemp(prefix='gp_ranks_')

    def __setitem__(self, rank, value):
        import os
        import pickle
        tmp = os.path.join(self.dir, '%d.tmp' % rank)
        with open(tmp, 'wb') as f:
            pickle.dump(value, f)
        os.replace(tmp, os.path.join(self.dir, '%d.pkl' % rank))

    def __getitem__(self, rank):
        import os
        import pickle
        with open(os.path.join(self.dir, '%d.pkl' % rank), 'rb') as f:
            return pickle.load(f)
