"""Whole-image queries with wide classifier heads: the config-1 shape (PW1 layer dict on 28x28x1) with c = 10 (fused head),
100 and 1,000 classes (wide head: FC GEMM for the logits, then wide_softmax_kernel).  Prints one JSON line:
  * the GPU's name, power limit and maximum SM clock, read in the same run;
  * ms per query through NNAL.CNN_query ('entropy', 'fi', 'BALD' with T = MC_iters = 10; median of --reps after a warm-up);
  * from the per-layer profile classes (CUDA events) of one profiled 'entropy' query: the pool pass and the head's share of
    it (GEMM and softmax together; at c = 10 the fused head kernel);
  * from torch.profiler in a separate 'entropy' query: the softmax kernel alone, against 7.7 TB/s for 8c bytes per sample
    (logits read once, posteriors written once; the second logits read comes from L2);
  * the head GEMM (head class minus the softmax) against its MMA-issue bound, DESIGN §8's tile arithmetic at the maximum
    SM clock: per chunk ceil(pair tiles / pairs) x k-blocks x 12 MMAs x 128 cycles, 74 CTA pairs.
usage: python scripts/wide_head_round.py [--reps 3] [--n 100000] [--classes 10 100 1000] [--T 10] [--out FILE]"""
import argparse
import json
import math
import os
import subprocess
import sys
import time
from collections import OrderedDict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CHUNK = 16384                # DEFAULT_CHUNK (csrc/capi.cu)
PAIRS = 74                   # CTA pairs of fc_tc_pair_kernel with all 148 SMs paired
HBM_TBS = 7.7


class Expr(object):
    def __init__(self, **pars):
        self.pars = pars


def gpu_info():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader', '-i', '0'],
                             stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=60).stdout.decode().strip()
        power, clk = [s.strip() for s in out.split(',')]
        mhz = float(clk.split()[0])
    except Exception as e:          # reported as missing rather than guessed
        power, mhz = 'unavailable (%s)' % e, None
    return name, power, mhz


def time_query(nb, model, expr, n, method, reps):
    nb.NNAL.CNN_query(model, expr, np.arange(n), method, None)          # warm-up: module load, buffers at full size
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        nb.NNAL.CNN_query(model, expr, np.arange(n), method, None)       # returns host results: ends in a device synchronise
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), [round(t, 3) for t in ts]


def head_gemm_bound_cycles(n, c, K):
    cyc = 0
    for o in range(0, n, CHUNK):
        nb_ = min(CHUNK, n - o)
        tiles = math.ceil(nb_ / 256) * math.ceil(c / 256)
        cyc += math.ceil(tiles / PAIRS) * math.ceil(K / 64) * 12 * 128
    return cyc


def softmax_profiled_ms(nb, model, expr, n):
    import torch
    from torch.profiler import profile, ProfilerActivity
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        nb.NNAL.CNN_query(model, expr, np.arange(n), 'entropy', None)
        torch.cuda.synchronize()
    us, cnt = 0.0, 0
    for e in prof.events():
        if 'wide_softmax_kernel' in e.name and e.device_type == torch.autograd.DeviceType.CUDA:
            us += e.device_time if hasattr(e, 'device_time') else e.cuda_time
            cnt += 1
    return us / 1e3, cnt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--n', type=int, default=100000)
    ap.add_argument('--classes', type=int, nargs='+', default=[10, 100, 1000])
    ap.add_argument('--T', type=int, default=10)
    ap.add_argument('--out', default=None)
    a = ap.parse_args()
    import nnal_b200 as nb
    import oracle as O
    name, power, mhz = gpu_info()
    res = {'gpu': name, 'power_limit': power, 'max_sm_clock_mhz': mhz, 'n': a.n, 'T': a.T, 'k': 10,
           'shape': 'PW1 layer dict on 28x28x1'}
    x = np.random.RandomState(0).rand(a.n, 28, 28, 1).astype(np.float32)
    eng = nb.get_engine()
    eng.set_dropout_seed(2024)
    for c in a.classes:
        layers = O.pw1_layers(c)
        head = len(layers) - 1
        K = layers[head - 1][1][0]
        w = O.he_init_weights(layers, (28, 28, 1), 1)
        model = nb.NN.CNN((28, 28, 1), OrderedDict(layers), feature_layer=len(layers) - 2, dropout=[[6, 7, 8], 0.5])
        model.set_weights(w)
        expr = Expr(k=10, B=100, MC_iters=a.T)
        expr.pool_images = x
        r = {}
        for method in ('entropy', 'fi', 'BALD'):
            med, ts = time_query(nb, model, expr, a.n, method, a.reps)
            r['query_ms_%s' % method] = round(med, 3)
            r['query_ms_%s_reps' % method] = ts
        eng.profile(True)
        nb.NNAL.CNN_query(model, expr, np.arange(a.n), 'entropy', None)
        per_layer = [eng.profile_read(i)[0] for i in range(len(layers))]
        eng.profile(False)
        head_ms = per_layer[head]
        r['pass_ms_layers'] = round(sum(per_layer), 4)
        r['head_ms'] = round(head_ms, 4)
        r['head_share_of_layers'] = round(head_ms / sum(per_layer), 4)
        r['head_uses_tc'] = eng.layer_info(head)[2]
        if c >= 64:
            sm_ms, launches = softmax_profiled_ms(nb, model, expr, a.n)
            byts = 8.0 * c * a.n
            r['softmax_ms_profiler'] = round(sm_ms, 4)
            r['softmax_launches'] = launches
            r['softmax_bytes'] = byts
            r['softmax_share_of_hbm_bound'] = round(byts / (HBM_TBS * 1e12) * 1e3 / sm_ms, 4) if sm_ms > 0 else None
            gemm_ms = head_ms - sm_ms
            cyc = head_gemm_bound_cycles(a.n, c, K)
            r['head_gemm_ms'] = round(gemm_ms, 4)
            r['head_gemm_issue_bound_cycles'] = cyc
            if mhz:
                bound_ms = cyc / (mhz * 1e6) * 1e3
                r['head_gemm_issue_bound_ms'] = round(bound_ms, 4)
                r['head_gemm_share_of_issue_bound'] = round(bound_ms / gemm_ms, 4) if gemm_ms > 0 else None
            r['head_gemm_tflops_algorithmic'] = round(2.0 * a.n * c * K / (gemm_ms * 1e-3) / 1e12, 1) if gemm_ms > 0 else None
        res['c%d' % c] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
