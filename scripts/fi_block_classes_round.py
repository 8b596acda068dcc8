"""Timing of the block-form greedy FI with a class cap (``fi_classes``, csrc/fi_block.cu kept classes).  Prints one JSON
line (and writes it to --out):
  * the GPU's name and power limit, read in the same run;
  * ms per Engine.fi_block_greedy at B = 10,000 candidates, d = 4,096, k = 100 with r = 10 classes kept, for c = 10, 100 and
    1,000 (Dirichlet(0.1) posteriors, kept classes selected on the host), the uncapped c = 10 greedy beside it, and the
    split between the per-step system (K_SS row, inversion, Z, tr C), the candidate evaluation and the winner's column
    from CUDA events in a separate profiled run;
  * one NNAL.CNN_query(..., 'fi') round with fi_mode = 'block-greedy', fi_classes = 10 at the config-1 shape (PW1 layer
    dict on 28x28x1) with a 1,000-class head over a 100,000-image pool, B = 10,000, k = 100.
usage: python scripts/fi_block_classes_round.py [--reps 5] [--out FILE]"""
import argparse
import json
import os
import sys
import time
from collections import OrderedDict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'scripts'))


class Expr(object):
    def __init__(self, **pars):
        self.pars = pars


def time_greedy(eng, k, reps):
    eng.fi_block_greedy(k, 1e-5)                                       # warm-up: buffers at full size
    ts = []
    for _ in range(reps):
        eng.synchronize()
        t0 = time.perf_counter()
        sel, obj, red = eng.fi_block_greedy(k, 1e-5)                   # returns host results: ends in a device synchronise
        ts.append((time.perf_counter() - t0) * 1e3)
    eng.profile(True)
    eng.fi_block_greedy(k, 1e-5)
    split = {}
    for key, cls in (('system', 114), ('eval', 115), ('column', 116)):
        t, n = eng.profile_read(cls)
        split[key + '_ms'] = round(t, 3)
    eng.profile(False)
    ms = float(np.median(ts))
    return {'greedy_ms': round(ms, 3), 'greedy_ms_reps': [round(t, 3) for t in ts], 'us_per_step': round(1e3 * ms / k, 2),
            'final_red': float(red[-1]), 'split_profiled': split}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--pool', type=int, default=100000)
    ap.add_argument('--out')
    a = ap.parse_args()
    import nnal_b200 as nb
    import oracle as O
    from fi_block_round import gpu_info
    from tests.fi_block_cls_oracle import top_classes
    name, power = gpu_info()
    res = {'gpu': name, 'power_limit': power}
    B, d, k, r = 10000, 4096, 100, 10
    rs = np.random.RandomState(1)
    U = np.maximum(rs.randn(B, d), 0).astype(np.float32)
    eng = nb.get_engine()
    res['synthetic'] = {'B': B, 'd': d, 'k': k, 'fi_classes': r, 'posteriors': 'Dirichlet(0.1)'}
    for c in (10, 100, 1000):
        post = rs.dirichlet(np.ones(c) * 0.1, B).T.astype(np.float32)
        if c == 10:
            eng.fi_block_set_factors(post, U)
            res['synthetic']['c10_uncapped'] = time_greedy(eng, k, a.reps)
        cls, p = top_classes(post, r)
        eng.fi_block_set_factors_cls(cls, p, U, c)
        res['synthetic']['c%d_r%d' % (c, r)] = time_greedy(eng, k, a.reps)
    layers = O.pw1_layers(1000)
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    x = np.random.RandomState(0).rand(a.pool, 28, 28, 1).astype(np.float32)
    model = nb.NN.CNN((28, 28, 1), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)
    expr = Expr(k=k, B=B, lambda_=0., batch_size=500, fi_mode='block-greedy', fi_classes=r)
    expr.pool_images = x
    nb.NNAL.CNN_query(model, expr, np.arange(a.pool), 'fi', None)       # warm-up: module load, buffers
    ts = []
    for _ in range(max(1, a.reps // 2)):
        t0 = time.perf_counter()
        nb.NNAL.CNN_query(model, expr, np.arange(a.pool), 'fi', None)    # returns host results: ends in a device synchronise
        ts.append((time.perf_counter() - t0) * 1e3)
    res['config1_c1000_query'] = {'pool': a.pool, 'B': B, 'k': k, 'fi_classes': r, 'ms': round(float(np.median(ts)), 1),
                                  'ms_reps': [round(t, 1) for t in ts]}
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
