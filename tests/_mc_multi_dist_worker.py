"""Worker of tests/test_oracle_mc_multi.py: one rank of a world_size-N gloo group running NNAL.CNN_query with 'MC-entropy',
'BALD', 'ensemble' and 'QBC-JS' on c = 2 and c = 5 nets over the NumPy fake engine, whose multi-class MC entry points are
backed by the float64 reference (tests/mc_multi_oracle.py).  Writes its results to <out>/rank<r>.npz."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

K, T, KEEP, SEED, FIRST_PASS = 9, 4, 0.6, 0x5eed2024, 3
DROPOUT_LAYERS = [2, 3, 4]
METHODS = ('MC-entropy', 'BALD', 'ensemble', 'QBC-JS')
CLASSES = (2, 5)
N_MEMBERS = 3


def make_layers(c):
    return [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [12, 'fc']), ('fc2', [8, 'fc']),
            ('fc3', [c, 'fc'])]


def make_case(c):
    """Layers, the model's weights, the committee's weight sets and the pool images [70,5,5,2]."""
    import oracle as O
    layers = make_layers(c)
    w = O.he_init_weights(layers, (5, 5, 2), 11 + c, bias_scale=0.3)
    members = [O.he_init_weights(layers, (5, 5, 2), 40 + 7 * i + c, bias_scale=0.3) for i in range(N_MEMBERS)]
    x = np.random.RandomState(7 + c).rand(70, 5, 5, 2).astype(np.float32)
    return layers, w, members, x


def mc_multi_fake_engine():
    from tests import mc_multi_oracle as MM
    from tests.fake_engine import FakeEngine

    class MCMultiFakeEngine(FakeEngine):
        """Adds the c-class MC-dropout / committee statistics and score kinds 12 / 13.  c = 2 keeps the base class's binary
        statistics, as the device does."""

        def pool_begin(self, n, keep=0):
            FakeEngine.pool_begin(self, n, keep)
            if self._mc is not None and self.n_class > 2:
                self.av_post = np.zeros((self.n_class, n))

        def _forward_mc(self, x, offset):
            if self.n_class == 2:
                return FakeEngine._forward_mc(self, x, offset)
            T_, keep, layers, pos0, first = self._mc
            n = x.shape[0]
            passes = MM.mc_passes(self.layers, self.weights, x, pos0 + offset + np.arange(n), T_, keep, layers,
                                  self.dropout_seed, first)
            av_p, av_e = MM.class_running_means(passes)
            self.av_post[:, offset:offset + n] = av_p
            self.av_ent[offset:offset + n] = av_e
            self.post[:, offset:offset + n] = passes[-1]

        def pool_ensemble_accumulate(self, t):
            if self.n_class == 2:
                return FakeEngine.pool_ensemble_accumulate(self, t)
            p = self.post.astype(np.float32).astype(np.float64)
            if t == 0:
                self.av_post, self.av_ent = np.zeros_like(p), np.zeros(self._pool_n)
            self.av_post = (p + t * self.av_post) / (t + 1)
            self.av_ent = (MM.class_entropy_bumped(p) + t * self.av_ent) / (t + 1)

        def pool_mc_class_means(self):
            if self.n_class == 2:
                return np.stack([1 - self.av_post, self.av_post]), self.av_ent.copy()
            return self.av_post.copy(), self.av_ent.copy()

        def pool_score(self, kind, eps=0.0):
            if kind in (12, 13):
                self.score = (MM.scores_from_binary(self.av_post, self.av_ent, kind) if self.n_class == 2
                              else MM.scores(self.av_post, self.av_ent, kind))
            else:
                FakeEngine.pool_score(self, kind, eps)

    return MCMultiFakeEngine()


def run(rank, world, out):
    import torch.distributed as td
    if world > 1:
        td.init_process_group('gloo', rank=rank, world_size=world)
    from collections import OrderedDict
    import nnal_b200
    from nnal_b200 import engine
    eng = engine._engine = mc_multi_fake_engine()

    class Expr(object):
        pass

    res = {}
    for c in CLASSES:
        layers, w, members, x = make_case(c)
        model = nnal_b200.NN.CNN((5, 5, 2), OrderedDict(layers), feature_layer=len(layers) - 2,
                                 dropout=[DROPOUT_LAYERS, KEEP])
        model.set_weights(w)
        holder = nnal_b200.NN.CNN((5, 5, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
        paths = []
        for i, m in enumerate(members):
            holder.set_weights(m)
            paths.append(os.path.join(out, 'c%d_member%d_rank%d.npz' % (c, i, rank)))
            holder.save_weights(paths[-1])
        expr = Expr()
        expr.pars = dict(k=K, MC_iters=T)
        expr.pool_images = x
        expr.model_holder = holder
        expr.pretrained_paths = paths
        for method in METHODS:
            eng.set_dropout_seed(SEED, first_pass=FIRST_PASS)
            res['c%d_%s' % (c, method)] = nnal_b200.NNAL.CNN_query(model, expr, np.arange(len(x)), method, None)
    np.savez(os.path.join(out, 'rank%d.npz' % rank), **res)
    if world > 1:
        td.barrier()
        td.destroy_process_group()


if __name__ == '__main__':
    run(int(os.environ['RANK']), int(os.environ['WORLD_SIZE']), sys.argv[1])
