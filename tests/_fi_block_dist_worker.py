"""Worker of tests/test_oracle_fi_block.py: one rank of a world_size-N gloo group running NNAL.CNN_query(..., 'fi') with
fi_mode='block-greedy' on a c = 3 net over the NumPy fake engine, whose block-FI entry points are backed by the float64
oracle.  Writes its results to <out>/rank<r>.npz."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, B, DELTA = 6, 25, 1e-4


def make_case():
    import oracle as O
    layers = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [12, 'fc']), ('fc2', [8, 'fc']),
              ('fc3', [3, 'fc'])]
    w = O.he_init_weights(layers, (5, 5, 2), 11, bias_scale=0.1)
    x = np.random.RandomState(7).rand(70, 5, 5, 2).astype(np.float32)
    return layers, w, x


def block_fake_engine():
    from tests import fi_block_oracle as FB
    from tests.fake_engine import FakeEngine

    class BlockFakeEngine(FakeEngine):
        """Adds the block-form FI entry points, computed by the float64 oracle on float32 factors like the device's."""

        def fi_block_set_candidates(self, cand=None):
            rows = np.arange(self._pool_n) if cand is None else np.asarray(cand, dtype=np.int64)
            self.fib_post = self.post[:, rows].astype(np.float32)
            self.fib_U = self.feat[rows].astype(np.float32)

        def fi_block_set_factors(self, post, U):
            post, U = np.asarray(post, dtype=np.float32), np.asarray(U, dtype=np.float32)
            if post.ndim != 2 or U.ndim != 2 or post.shape[1] != U.shape[0]:
                raise ValueError('post must be [c,n] and U [n,d] for the same n')
            self.fib_post, self.fib_U = post, U

        def fi_block_greedy(self, k, delta):
            return FB.greedy_fi_block(self.fib_post.astype(np.float64), self.fib_U.T.astype(np.float64), delta, k)

    return BlockFakeEngine()


def run(rank, world, out):
    import torch.distributed as td
    if world > 1:
        td.init_process_group('gloo', rank=rank, world_size=world)
    from collections import OrderedDict
    import nnal_b200
    from nnal_b200 import engine
    engine._engine = block_fake_engine()
    layers, w, x = make_case()
    model = nnal_b200.NN.CNN((5, 5, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)

    class Expr(object):
        pass

    expr = Expr()
    expr.pars = dict(k=K, B=B, lambda_=0., batch_size=32, fi_mode='block-greedy', fi_diag_load=DELTA)
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
