"""Seeded outputs of the uncapped block-form greedy FI (no ``fi_classes``) for comparing two builds byte for byte:
c = 3, 10, 32 over one and two FC layers, from host factors (Engine.fi_block_set_factors) and in place through
fi.query_whole_block on a small conv net.
usage: python scripts/fi_block_parity.py --root TREE --out FILE.npz      (outputs of the package in TREE)
       python scripts/fi_block_parity.py --compare A.npz B.npz            (exit 1 unless every array is byte-identical)"""
import argparse
import os
import sys
from collections import OrderedDict

import numpy as np


class Expr(object):
    def __init__(self, **pars):
        self.pars = pars


def run(root, out):
    sys.path.insert(0, os.path.abspath(root))
    import nnal_b200 as nb
    import oracle as O
    res = {}
    eng = nb.get_engine()
    for c in (3, 10, 32):
        rs = np.random.RandomState(c)
        n, d, dp = 2000, 256, 128
        post = rs.dirichlet(np.ones(c) * 0.5, n).T.astype(np.float32)
        post[:, ::17] = 0.
        post[c - 1, ::17] = 1.
        U = np.maximum(rs.randn(n, d), 0).astype(np.float32)
        A = np.maximum(rs.randn(n, dp), 0).astype(np.float32)
        W = (rs.randn(c, d) / np.sqrt(d)).astype(np.float32)
        k = min(60, 4096 // (c - 1))
        for nl in (1, 2):
            if nl == 1:
                eng.fi_block_set_factors(post, U)
            else:
                eng.fi_block_set_factors(post, U, A, W)
            for key, v in zip(('sel', 'obj', 'red'), eng.fi_block_greedy(k, 1e-4)):
                res['host_c%d_l%d_%s' % (c, nl, key)] = v
        layers = [('conv1', [6, 'conv', [3, 3]]), ('conv2', [5, 'conv', [5, 5]]), ('max1', [[2, 2], 'pool']),
                  ('conv3', [8, 'conv', [3, 3]]), ('max2', [[2, 2], 'pool']), ('fc1', [40, 'fc']), ('fc2', [24, 'fc']),
                  ('fc3', [c, 'fc'])]
        w = O.he_init_weights(layers, (9, 7, 2), 70 + c, bias_scale=0.1)
        model = nb.NN.CNN((9, 7, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
        model.set_weights(w)
        x = np.random.RandomState(71).rand(600, 9, 7, 2).astype(np.float32)
        for nl in (1, 2):
            expr = Expr(k=20, B=200, lambda_=0., batch_size=128, fi_mode='block-greedy', fi_layers=nl)
            expr.pool_images = x
            for key, v in zip(('q', 'obj', 'red'), nb.fi.query_whole_block(model, expr, np.arange(600), None,
                                                                         return_objective='reduced')):
                res['query_c%d_l%d_%s' % (c, nl, key)] = v
    np.savez(out, **res)
    print('%s: %d arrays' % (out, len(res)))


def compare(a, b):
    A, B = np.load(a), np.load(b)
    assert sorted(A.files) == sorted(B.files), set(A.files) ^ set(B.files)
    bad = [f for f in A.files if A[f].dtype != B[f].dtype or A[f].tobytes() != B[f].tobytes()]
    print('%d arrays compared, %d differ%s' % (len(A.files), len(bad), (': ' + ', '.join(bad)) if bad else ''))
    return 1 if bad else 0


if __name__ == '__main__':
    ap = argparse.ArgumentParser()
    ap.add_argument('--root', default=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    ap.add_argument('--out')
    ap.add_argument('--compare', nargs=2)
    a = ap.parse_args()
    sys.exit(compare(*a.compare) if a.compare else run(a.root, a.out))
