"""Worker of tests/test_oracle_fi_block2.py: one rank of a world_size-N gloo group running NNAL.CNN_query(..., 'fi') with
fi_mode='block-greedy' and fi_layers=2 on a c = 3 net over the NumPy fake engine, whose block-FI entry points are backed by
the float64 oracle.  Writes its results to <out>/rank<r>.npz."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, B, DELTA = 6, 25, 1e-4


def make_case(c=3):
    import oracle as O
    layers = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [12, 'fc']), ('fc2', [8, 'fc']),
              ('fc3', [c, 'fc'])]
    w = O.he_init_weights(layers, (5, 5, 2), 11, bias_scale=0.1)
    x = np.random.RandomState(7).rand(70, 5, 5, 2).astype(np.float32)
    return layers, w, x


def block2_fake_engine():
    from tests import fi_block2_oracle as FB2
    from tests.fake_engine import FakeEngine

    f32 = lambda a: np.asarray(a, dtype=np.float32)

    class Block2FakeEngine(FakeEngine):
        """Adds the one- and two-layer block-form FI entry points, computed by the float64 oracle on float32 factors like
        the device's."""

        def pool_prev_rows(self, pos):
            return f32(self.prev[np.asarray(pos, dtype=np.int64)])

        def fi_block_set_candidates(self, cand=None, n_layers=1):
            rows = np.arange(self._pool_n) if cand is None else np.asarray(cand, dtype=np.int64)
            self.fib_post, self.fib_U = f32(self.post[:, rows]), f32(self.feat[rows])
            self.fib_A = f32(self.prev[rows]) if n_layers == 2 else None
            self.fib_W = f32(self.weights[self.layers[-1][0]][0]) if n_layers == 2 else None

        def fi_block_set_factors(self, post, U, A_prev=None, w_last=None):
            post, U = f32(post), f32(U)
            if post.ndim != 2 or U.ndim != 2 or post.shape[1] != U.shape[0]:
                raise ValueError('post must be [c,n] and U [n,d] for the same n')
            if (A_prev is None) != (w_last is None):
                raise ValueError('two-layer FI needs both A_prev and w_last')
            self.fib_post, self.fib_U = post, U
            self.fib_A = None if A_prev is None else f32(A_prev)
            self.fib_W = None if w_last is None else f32(w_last)

        def fi_block_greedy(self, k, delta):
            assert self.fib_A is not None, 'the one-layer path is covered by tests/_fi_block_dist_worker.py'
            f64 = lambda a: a.astype(np.float64)
            return FB2.greedy_fi_block2(f64(self.fib_post), f64(self.fib_U).T, f64(self.fib_A).T, f64(self.fib_W), delta, k)

    return Block2FakeEngine()


def run(rank, world, out):
    import torch.distributed as td
    if world > 1:
        td.init_process_group('gloo', rank=rank, world_size=world)
    from collections import OrderedDict
    import nnal_b200
    from nnal_b200 import engine
    engine._engine = block2_fake_engine()
    layers, w, x = make_case()
    model = nnal_b200.NN.CNN((5, 5, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)

    class Expr(object):
        pass

    expr = Expr()
    expr.pars = dict(k=K, B=B, lambda_=0., batch_size=32, fi_mode='block-greedy', fi_layers=2, fi_diag_load=DELTA)
    expr.pool_images = x
    res = {}
    res['q_pre'] = nnal_b200.NNAL.CNN_query(model, expr, np.arange(len(x)), 'fi', None)
    _, _, res['red_pre'] = nnal_b200.fi.query_whole_block(model, expr, np.arange(len(x)), None, return_objective='reduced')
    expr.pars['B'] = 10 ** 6
    res['q_all'] = nnal_b200.NNAL.CNN_query(model, expr, np.arange(len(x)), 'fi', None)
    np.savez(os.path.join(out, 'rank%d.npz' % rank), **res)
    if world > 1:
        td.barrier()
        td.destroy_process_group()


if __name__ == '__main__':
    run(int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), sys.argv[1])
