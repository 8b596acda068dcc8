"""Timing of the multi-class block-form greedy FI selection (csrc/fi_block.cu).  Prints one JSON line:
  * the GPU's name and power limit, read in the same run;
  * ms per NNAL.CNN_query(..., 'fi') at the config-1 shape (PW1 layer dict on 28x28x1, c = 10, 2,000-image pool, B = 100,
    k = 10) with fi_mode='block-greedy', and with the default (trace top-k) side by side;
  * ms and us per step of Engine.fi_block_greedy on synthetic factors at B = 10,000 candidates, d = 4096, c = 10, k = 100
    (largest system 900 x 900), and the split between the per-step system (K_SS row, inversion, Z, tr C), the candidate
    evaluation and the winner's column, from CUDA events in a separate profiled run.
usage: python scripts/fi_block_round.py [--reps 5]"""
import argparse
import json
import os
import subprocess
import sys
import time
from collections import OrderedDict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


class Expr(object):
    def __init__(self, **pars):
        self.pars = pars


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i', '0'],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=60).stdout.decode().strip()
    except Exception as e:          # the number is reported as missing rather than guessed
        out = 'unavailable (%s)' % e
    return name, out


def time_query(nb, model, expr, n, reps):
    nb.NNAL.CNN_query(model, expr, np.arange(n), 'fi', None)          # warm-up: module load, buffers
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        nb.NNAL.CNN_query(model, expr, np.arange(n), 'fi', None)       # returns host results: ends in a device synchronise
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 3) for t in ts]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    a = ap.parse_args()
    import nnal_b200 as nb
    import oracle as O
    name, power = gpu_info()
    res = {'gpu': name, 'power_limit': power}
    # config-1 shape
    layers = O.pw1_layers(10)
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    x = np.random.RandomState(0).rand(2000, 28, 28, 1).astype(np.float32)
    model = nb.NN.CNN((28, 28, 1), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)
    for mode in ('block-greedy', 'default'):
        expr = Expr(k=10, B=100, lambda_=0., batch_size=500)
        if mode != 'default':
            expr.pars['fi_mode'] = mode
        expr.pool_images = x
        med, ts = time_query(nb, model, expr, 2000, a.reps)
        res['config1_query_ms_%s' % mode] = round(med, 3)
        res['config1_query_ms_%s_reps' % mode] = ts
    # synthetic factors
    B, d, c, k = 10000, 4096, 10, 100
    rs = np.random.RandomState(1)
    post = rs.dirichlet(np.ones(c), B).T.astype(np.float32)
    U = np.maximum(rs.randn(B, d), 0).astype(np.float32)
    eng = nb.get_engine()
    eng.fi_block_set_factors(post, U)
    eng.fi_block_greedy(k, 1e-5)                                       # warm-up: buffers at full size
    ts = []
    for _ in range(a.reps):
        eng.synchronize()
        t0 = time.perf_counter()
        sel, obj, red = eng.fi_block_greedy(k, 1e-5)
        ts.append((time.perf_counter() - t0) * 1e3)
    ms = float(np.median(ts))
    res.update({'synthetic': {'B': B, 'd': d, 'c': c, 'k': k, 'max_system': k * (c - 1)},
                'synthetic_greedy_ms': round(ms, 3), 'synthetic_greedy_ms_reps': [round(t, 3) for t in ts],
                'synthetic_us_per_step': round(1e3 * ms / k, 2), 'synthetic_final_red': float(red[-1])})
    eng.profile(True)
    eng.fi_block_greedy(k, 1e-5)
    split = {}
    for key, cls in (('system', 114), ('eval', 115), ('column', 116)):
        t, n = eng.profile_read(cls)
        split[key + '_ms'] = round(t, 3)
        split[key + '_launch_groups'] = n
    eng.profile(False)
    res['synthetic_split_profiled'] = split
    print(json.dumps(res))


if __name__ == '__main__':
    main()
