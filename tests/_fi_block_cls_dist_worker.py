"""Worker of tests/test_oracle_fi_block_classes.py: one rank of a world_size-N gloo group running NNAL.CNN_query(..., 'fi')
with fi_mode='block-greedy' and fi_classes on a c = 40 net over the NumPy fake engine, whose class-capped block-FI entry
points are backed by the float64 oracle.  Writes its results to <out>/rank<r>.npz."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, B, DELTA, C, R = 6, 25, 1e-4, 40, 5


def make_case():
    import oracle as O
    layers = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [12, 'fc']), ('fc2', [8, 'fc']),
              ('fc3', [C, 'fc'])]
    w = O.he_init_weights(layers, (5, 5, 2), 13, bias_scale=0.1)
    w['fc3'] = (w['fc3'][0] * np.float32(3.), w['fc3'][1])
    x = np.random.RandomState(8).rand(70, 5, 5, 2).astype(np.float32)
    return layers, w, x


def cls_fake_engine():
    from tests import fi_block_cls_oracle as FC
    from tests.fake_engine import FakeEngine

    class ClsFakeEngine(FakeEngine):
        """Adds the class-capped block-FI entry points, computed by the float64 oracle on float32 factors like the
        device's."""

        def pool_top_classes(self, rows, r):
            return FC.top_classes(self.post[:, np.asarray(rows, dtype=np.int64)].astype(np.float32), r)

        def fi_block_set_candidates_cls(self, cand, r):
            rows = np.arange(self._pool_n) if cand is None else np.asarray(cand, dtype=np.int64)
            self.fib = self.pool_top_classes(rows, r) + (self.feat[rows].astype(np.float32), self.n_class)

        def fi_block_set_factors_cls(self, cls, p, U, c):
            cls, p, U = np.asarray(cls), np.asarray(p, dtype=np.float32), np.asarray(U, dtype=np.float32)
            assert cls.shape == p.shape and U.shape[0] == cls.shape[0]
            self.fib = (cls, p, U, int(c))

        def fi_block_greedy(self, k, delta):
            cls, p, U, c = self.fib
            return FC.greedy_fi_block_cls(cls, p, U.T.astype(np.float64), c, delta, k)

    return ClsFakeEngine()


def run(rank, world, out):
    import torch.distributed as td
    if world > 1:
        td.init_process_group('gloo', rank=rank, world_size=world)
    from collections import OrderedDict
    import nnal_b200
    from nnal_b200 import engine
    engine._engine = cls_fake_engine()
    layers, w, x = make_case()
    model = nnal_b200.NN.CNN((5, 5, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)

    class Expr(object):
        pass

    expr = Expr()
    expr.pars = dict(k=K, B=B, lambda_=0., batch_size=32, fi_mode='block-greedy', fi_diag_load=DELTA, fi_classes=R)
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
