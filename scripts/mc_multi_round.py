"""Timing of the multi-class MC-dropout queries of NNAL.CNN_query ('BALD', 'MC-entropy').  Prints one JSON line:
  * the GPU's name and power limit, read in the same run;
  * ms per query through the API (median of --reps, after a warm-up query) at the config-1 shape (PW1 layer dict on
    28x28x1, c = 10, dropout on fc1, fc2 and the logits, T = MC_iters = 10, k = 10) over a 2,000-image pool and over a
    100,000-image pool; the deterministic 'entropy' query beside them;
  * from CUDA events in a separate profiled query per pool size: ms per stochastic pass (the FC tail and the
    running-mean update, summed over the pool's chunks), and the share of the running-mean kernel in the passes.
usage: python scripts/mc_multi_round.py [--reps 5] [--pools 2000 100000] [--T 10]"""
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

PROF_MC_ACCUM = 103          # NNAL_PROF_MC_ACCUM (csrc/nnal_common.cuh)


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


def time_query(nb, model, expr, n, method, reps):
    nb.NNAL.CNN_query(model, expr, np.arange(n), method, None)          # warm-up: module load, buffers at full size
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        nb.NNAL.CNN_query(model, expr, np.arange(n), method, None)       # returns host results: ends in a device synchronise
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 3) for t in ts]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--pools', type=int, nargs='+', default=[2000, 100000])
    ap.add_argument('--T', type=int, default=10)
    a = ap.parse_args()
    import nnal_b200 as nb
    import oracle as O
    name, power = gpu_info()
    res = {'gpu': name, 'power_limit': power, 'T': a.T, 'classes': 10, 'k': 10}
    layers = O.pw1_layers(10)
    sites = [6, 7, 8]
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    model = nb.NN.CNN((28, 28, 1), OrderedDict(layers), feature_layer=len(layers) - 2, dropout=[sites, 0.5])
    model.set_weights(w)
    eng = nb.get_engine()
    eng.set_dropout_seed(2024)
    for n in a.pools:
        x = np.random.RandomState(0).rand(n, 28, 28, 1).astype(np.float32)
        expr = Expr(k=10, MC_iters=a.T)
        expr.pool_images = x
        for method in ('BALD', 'MC-entropy', 'entropy'):
            med, ts = time_query(nb, model, expr, n, method, a.reps)
            res['query_ms_%s_%d' % (method, n)] = round(med, 3)
            res['query_ms_%s_%d_reps' % (method, n)] = ts
        eng.profile(True)
        nb.NNAL.CNN_query(model, expr, np.arange(n), 'BALD', None)
        tail = sum(eng.profile_read(j)[0] for j in sites)
        acc, groups = eng.profile_read(PROF_MC_ACCUM)
        eng.profile(False)
        res['profiled_%d' % n] = {'ms_per_pass': round((tail + acc) / a.T, 4), 'fc_tail_ms_per_pass': round(tail / a.T, 4),
                                  'accum_ms_per_pass': round(acc / a.T, 4), 'accum_share_of_passes': round(acc / (tail + acc), 4),
                                  'accum_launches': groups,
                                  'accum_bytes_per_pass': n * (20 * 10 + 16)}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
