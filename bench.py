#!/usr/bin/env python
"""bench.py -- headline benchmark of the query-scoring hot path (BASELINE.json metric: pool samples scored per
second for an entropy + Fisher-information query round; config 2 of BASELINE.json at N=1).

A "step" is ONE query round over one synthetic pool (SURVEY.md 8d): gather 25x25x3 patches around `--pool` voxels of
3 synthetic 256x256x180 volumes -> PW1 patch-CNN forward (c=2), keeping the factors of the last two FC layers ->
|P(class1)-0.5| -> top-k (the 'entropy' answer, k=100) AND uncertainty pre-filter to B=10,000 -> factored FI of the
last two FC layers -> greedy selection of k=100 (the 'fi' answer) -> both index sets on the host.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

`--dump-outputs DIR` also writes what the timed path computed in its last step as DIR/<name>.npy (float32 / float64;
indices as float64): the inputs are seeded, so two builds can be compared array by array.

Prints ONE JSON line (rank 0).  `value` = whole-job samples/s with volumes, weights and pool indices resident in
HBM; `e2e` = the same round through the reference-facing API (nnal_b200.PW_NNAL.CNN_query(..., 'entropy+fi') with
HOST arrays: volumes + indices copied host->device from pinned memory and the selected indices read back, every
step).  `--impl reference` times the restated reference CPU path (oracle port: NumPy gather + float32 torch-CPU
forward + NumPy scoring + NumPy FI greedy) on the host cores, on a bounded sample of the same workload.

Extra keys (stage evidence): `stage_ms_per_step`, `entropy_round` (the round-1 headline: entropy query alone),
`fi_round` (FI stages + the Gram all-reduce), `mc_round`, `fi_sdp_round`, `config4` (memory-bound gather / entropy map)
and `strong_scaling` (BASELINE config 3: a FIXED 1 M-patch pool of 8 subjects through query_multimg at any N, with a hash
of the selected indices that must not depend on N, the NCCL Gram all-reduce and the primal-vs-dual objective check).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

VOL_SHAPE = (256, 256, 180)
PATCH = (25, 25, 1)
N_MOD = 3
METRIC = 'pool samples scored/sec (entropy+FI query round: gather + PW1 forward + |p-0.5| top-k + FI pre-filter B + greedy k)'
UNIT = 'samples/s'
PW1_MFLOP = 117.05          # per patch, SURVEY.md 8a row 5
K_QUERY = 100
FI_DELTA = 1e-5             # diag_load of the single-volume 'fi' branch (PW_NNAL.py:738-745)


class Expr(object):
    pass


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return {'hbm_gbs': d.get('hbm_gbs', 6650.0), 'bf16_burst': d.get('bf16_tflops', 1590.0),
                'bf16_sustained': d.get('bf16_tflops_sustained', 1400.0), 'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_burst': 1590.0, 'bf16_sustained': 1400.0, 'source': 'fallback'}


def _host_buffer(shape, dtype, pinned):
    if pinned:
        import torch
        return torch.zeros(shape, dtype=getattr(torch, np.dtype(dtype).name)).pin_memory().numpy()
    return np.zeros(shape, dtype=dtype)


def make_workload(pool_total, seed_pool=3, pinned=False):
    """config 2 of BASELINE.json / SURVEY.md 8d: m=3 volumes 256x256x180 float32 clip(N(100,30^2),0,inf),
    zero-padded by (12,12,0); stats = (mean,std) of the unpadded volume; pool = distinct raveled voxel ids."""
    g = np.random.Generator(np.random.PCG64(2))
    imgs, stats = [], []
    for j in range(N_MOD):
        v = g.standard_normal(VOL_SHAPE, dtype=np.float32)
        v *= 30.
        v += 100.
        np.maximum(v, 0, out=v)
        stats.append([float(v.mean(dtype=np.float64)), float(v.std(dtype=np.float64))])
        imgs.append(v)
    r = [(p - 1) // 2 for p in PATCH]
    padded = []
    for v in imgs:
        shp = tuple(v.shape[i] + 2 * r[i] for i in range(3))
        buf = _host_buffer(shp, np.float32, pinned)
        buf[r[0]:r[0] + v.shape[0], r[1]:r[1] + v.shape[1], r[2]:r[2] + v.shape[2]] = v
        padded.append(buf)
    nvox = int(np.prod(VOL_SHAPE))
    rs = np.random.RandomState(seed_pool)
    pool = rs.choice(nvox, pool_total, replace=False).astype(np.int64) if pool_total <= nvox else \
        rs.randint(0, nvox, pool_total).astype(np.int64)
    if pinned:
        pb = _host_buffer((pool_total,), np.int64, True)
        pb[:] = pool
        pool = pb
    return padded, stats, pool


def workload_config(args, world):
    return {'workload': 'config2: PW1 2-class CNN, 3x 256x256x180 f32 volumes, 25x25x3 patches, %d-patch pool per GPU, '
                        'one query round = entropy query k=%d + FI query (pre-filter B=%d, last two FC layers, greedy k=%d)'
                        % (args.pool, K_QUERY, args.fi_B, K_QUERY),
            'pool_per_gpu': args.pool, 'k': K_QUERY, 'fi_B': args.fi_B, 'parallelism': 'pool sharded x%d' % world,
            'l2': 'inputs larger than L2 (volumes 169 MB + >600 MB activations per chunk)',
            'forward_gflop_per_step_per_gpu': PW1_MFLOP * args.pool / 1e3}


def load_traffic():
    """DRAM bytes per sample of each kernel class, from the committed ncu --set full captures
    (profiles/r*_traffic.json, written by scripts/summarize_ncu.py traffic); the newest round wins."""
    out = {}
    for name in ('r1_traffic.json', 'r2_traffic.json'):
        p = os.path.join(ROOT, 'profiles', name)
        if os.path.exists(p):
            out.update(json.load(open(p)))
    return out


def make_model():
    """PW1 (NN.create_PW1, NN.py:1319-1359) with He-normal weights (NN.py:1430-1470), RandomState(4): product-side workload
    generation -- oracle.he_init_weights(pw1_layers(2), (25,25,3), 4) draws the same stream for the reference arm."""
    import nnal_b200
    model = nnal_b200.NN.create_PW1(2)
    model.initialize(4)
    return model


DUMP_MAX_BYTES = 64 * 10 ** 6      # all files of one --dump-outputs together
NPY_HEADER_BYTES = 1024            # allowance per file for the .npy header (128 bytes for these shapes)


def _dump_float(a):
    a = np.asarray(a)
    return a if a.dtype == np.float32 else a.astype(np.float64)


def dump_outputs(out_dir, arrays, posteriors=None, posteriors_name='pool_posteriors', lo=0):
    """Writes each array as out_dir/<name>.npy: float32 stays float32, everything else (indices included) becomes float64.
    ``posteriors`` [..., n] (one column per pool sample, global positions lo..lo+n-1) is written as ``posteriors_name``
    next to ``pool_positions``: all n columns, or a fixed seeded sample of as many as the byte budget leaves after the
    other arrays and the file headers (each sampled column costs its posterior rows plus one float64 position)."""
    conv = {name: _dump_float(a) for name, a in arrays.items()}
    if posteriors is not None:
        post = _dump_float(posteriors)
        n = post.shape[-1]
        per_col = 8 + post.dtype.itemsize * int(np.prod(post.shape[:-1]))
        left = DUMP_MAX_BYTES - sum(a.nbytes for a in conv.values()) - NPY_HEADER_BYTES * (len(conv) + 2)
        m = max(0, min(n, left // per_col))
        cols = np.arange(n) if m == n else np.sort(np.random.RandomState(0).choice(n, m, replace=False))
        conv['pool_positions'] = (cols + lo).astype(np.float64)
        conv[posteriors_name] = np.ascontiguousarray(post[..., cols])
    if sum(a.nbytes for a in conv.values()) + NPY_HEADER_BYTES * len(conv) > DUMP_MAX_BYTES:
        raise ValueError('outputs do not fit the %d-byte dump budget' % DUMP_MAX_BYTES)
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in conv.items():
        path = os.path.join(out_dir, name + '.npy')
        np.save(path, a)
        total += os.path.getsize(path)
    sys.stderr.write('bench.py: wrote %d arrays (%d bytes) to %s\n' % (len(conv), total, out_dir))


def digest(*arrays):
    h = hashlib.sha1()
    for a in arrays:
        h.update(np.ascontiguousarray(a, dtype=np.int64).tobytes())
        h.update(b'|')
    return h.hexdigest()[:16]


class ClockSampler(threading.Thread):
    """Samples nvidia-smi clocks and throttle reasons DURING the timed region."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,' \
        'clocks_event_reasons.sw_power_cap'

    def __init__(self, gpu_index):
        threading.Thread.__init__(self)
        self.daemon = True
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def run(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.gpu), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '100'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(',')])
        except Exception:
            pass

    def stop(self):
        if self.proc:
            try:
                self.proc.terminate()
            except Exception:
                pass
        self.join(timeout=2)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'], r[4:8]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        return {'sm_mhz': float(np.median(sm)), 'sm_max_mhz': float(max(mx)), 'reasons': sorted(reasons),
                'samples': len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the restated reference CPU path (oracle port; the only place bench.py touches oracle/)
# ----------------------------------------------------------------------------------------------------------------------
class _TorchFactors(object):
    """float32 torch-CPU forward that also returns the input of the feature layer's FC (the 'a' factor of the two-layer FI)."""

    def __init__(self, layers, w, threads):
        from oracle.torch_fp32 import TorchForward
        self.fwd = TorchForward(layers, w, feature_layer=len(layers) - 2, threads=threads)
        self.prev = TorchForward(layers, w, feature_layer=len(layers) - 3, threads=threads)

    def factors(self, x):
        r = self.fwd(x)
        a = self.prev(x)['feature_layer']
        return r['posteriors'][1].astype(np.float64), r['feature_layer'].astype(np.float64), a.astype(np.float64)


def cpu_reference_round(sample, fi_B, threads=None):
    """Restated reference CPU path on a bounded sample (oracle port; TF 1.x cannot be installed), ONE query round:
    NumPy gather (as patch_utils.get_patches) + float64 normalise + float32 torch-CPU forward + NumPy |p-0.5| argsort (the
    'entropy' answer), then the FI half on the B most uncertain samples: re-gather, forward keeping the last-two-layer
    factors, kernel of the factored conditional FIs, NumPy greedy k (oracle.greedy_fi_rank1).  The FI half is scaled with
    the sample: B = fi_B * sample / pool.  Returns (seconds, samples, threads, stage seconds)."""
    import torch
    import oracle as O
    from oracle.torch_fp32 import TorchForward
    threads = threads or os.cpu_count()
    torch.set_num_threads(threads)
    padded, stats, pool = make_workload(sample)
    layers = O.pw1_layers(2)
    w = O.he_init_weights(layers, (25, 25, 3), 4)
    fwd = TorchForward(layers, w, feature_layer=len(layers) - 2, threads=threads)
    fac = _TorchFactors(layers, w, threads)
    t0 = time.perf_counter()
    posts = O.batch_eval(layers, w, padded, pool, PATCH, 1000, stats, 'posteriors', fwd=fwd)[0]
    order = O.stable_topk(np.abs(posts - .5), max(fi_B, K_QUERY))
    q_ent = order[:K_QUERY]
    t1 = time.perf_counter()
    sel = order[:fi_B]
    x = O.normalize_batch_eval(O.get_patches(padded, pool[sel], PATCH), stats).astype(np.float32)
    p1, U, A = fac.factors(x)
    Kt = O.last_layers_kernel(p1, U, A, w[layers[-1][0]][0].astype(np.float64))
    D = O.last_layers_dim(2, U.shape[0], A.shape[0])
    S, _ = O.greedy_fi_rank1(Kt, D, FI_DELTA, min(K_QUERY, fi_B))
    t2 = time.perf_counter()
    return t2 - t0, sample, threads, {'entropy_half_s': t1 - t0, 'fi_half_s': t2 - t1, 'q_ent': q_ent, 'q_fi': sel[S],
                                      'posts': posts}


def _cpu_desc(sample, fi_B, pool):
    return ('%d-patch sample of the %d-patch pool per round, FI pre-filter scaled to B=%d: NumPy gather + fp32 torch-CPU PW1 '
            'forward + NumPy argsort, then NumPy/torch factored FI + greedy k=%d on the B candidates; restated reference CPU '
            'path (TF 1.x unavailable)' % (sample, pool, fi_B, min(K_QUERY, fi_B)))


def run_reference(args, rank, world):
    if rank != 0:
        return
    sample = args.cpu_sample
    fi_B = max(K_QUERY, int(round(args.fi_B * sample / float(args.pool))))
    times = []
    threads = os.cpu_count()
    for i in range(args.warmup + args.steps):
        dt, n, threads, det = cpu_reference_round(sample, fi_B)
        if i >= args.warmup:
            times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'entropy_query': det['q_ent'], 'fi_query': det['q_fi']}, det['posts'],
                     'pool_posteriors_class1')
    total = sum(times)
    value = sample * len(times) / total
    line = {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / len(times),
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args, world),
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'sample': _cpu_desc(sample, fi_B, args.pool)},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------------
KERNEL_OF = {0: None, 1: None, 2: 'conv_wt_kernel'}


def run_ours(args, rank, world):
    import torch
    import nnal_b200
    from nnal_b200 import _lib as L
    from nnal_b200 import dist, fi as fimod
    if args.no_p2p:
        fimod.p2p_enabled = False

    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    peaks = load_peaks()
    pool_total = args.pool * world
    padded, stats, pool = make_workload(pool_total, pinned=True)
    model = make_model()
    layer_names = list(model.layer_dict.keys())
    eng = nnal_b200.get_engine()
    eng.set_model(model)
    b = dist.shard_bounds(pool_total, world)
    lo, hi = int(b[rank]), int(b[rank + 1])
    n_local = hi - lo
    k = K_QUERY
    B = min(args.fi_B, pool_total)
    st = np.array(stats, dtype=np.float64)
    stream = torch.cuda.ExternalStream(eng.stream)
    d_inds = torch.from_numpy(np.ascontiguousarray(pool[lo:hi])).cuda()
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        eng.synchronize()
        torch.cuda.synchronize()

    # ---------------- device-resident leg (value) ----------------
    eng.upload(0, padded)
    ev_stage = None

    def step_resident(mark=None):
        """One query round on resident inputs; the host logic is fi.query_single's (one pool pass, candidates indexed in place)."""
        eng.pool_begin(n_local, 2)
        eng.pool_eval_device(0, d_inds.data_ptr(), n_local, 0, PATCH, st)
        eng.pool_score(L.SCORE_BINARY)
        if mark:
            mark(0)
        top, _ = dist.topk_global(eng, max(B, k), lo, pool_total)
        q_ent, sel = top[:k], top[:B]
        if mark:
            mark(1)
        own = (sel >= lo) & (sel < hi)
        eng.fi_set_candidates(sel[own] - lo, 2)
        if mark:
            mark(2)
        chosen, obj, red = fimod.greedy_select(eng, min(k, len(sel)), FI_DELTA, np.nonzero(own)[0].astype(np.int64))
        if mark:
            mark(3)
        return q_ent, sel[chosen], red, obj

    # The interpreter's cyclic collector walks every tracked object of the process (torch, NumPy, this harness: millions) whenever
    # a generation-2 collection triggers -- 20-80 ms pauses at random steps of the host-timed e2e leg.  Objects alive now are
    # moved to the permanent generation (they are never garbage); objects created later are collected as usual.
    import gc
    gc.collect()
    gc.freeze()
    # untimed: the API path of the e2e leg once through as well (a fresh box pages the Python / NumPy / library code of that
    # path in from the image on first use; the timed e2e steps further down come W more untimed steps later)
    expr0 = Expr()
    expr0.pars = dict(k=k, B=B, lambda_=0., patch_shape=PATCH, ntb=10000, stats=stats, fi_layers=2, fi_diag_load=FI_DELTA)
    for _ in range(args.warmup):
        nnal_b200.PW_NNAL.CNN_query(expr0, model, None, padded, pool, None, 'entropy+fi')
    for _ in range(args.warmup):
        q_res = step_resident()
    barrier()
    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
        time.sleep(0.25)
    eng.profile(True)
    launches0 = eng.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = []

    def mark(i):
        e = torch.cuda.Event(enable_timing=True)
        e.record(stream)
        marks.append((i, e))
    barrier()
    ev0.record(stream)
    for _ in range(args.steps):
        mark(-1)
        q_res = step_resident(mark)
    ev1.record(stream)
    ev1.synchronize()
    barrier()
    dev_ms = ev0.elapsed_time(ev1)
    launches = eng.launches - launches0
    clocks = sampler.stop() if sampler else None
    # stage times between the marks (device time on the library's stream)
    stage_names = ['pool_pass(gather+forward+score)', 'topk+merge(entropy answer, FI pre-filter)', 'fi_factors_setup', 'fi_greedy']
    stage_acc = np.zeros(4)
    for j in range(len(marks) - 1):
        i0, e0 = marks[j]
        i1, e1 = marks[j + 1]
        if i1 >= 0:
            stage_acc[i1] += e0.elapsed_time(e1)
    # per kernel-class times measured over the same timed region
    classes = {}
    for i, name in enumerate(layer_names):
        t, c = eng.profile_read(i)
        ty, macs, tc = eng.layer_info(i)
        classes[name] = {'ms': t, 'launches': c, 'macs_per_sample': macs, 'tc': tc, 'type': ty}
    for name, cid in (('gather', 100), ('score', 101), ('topk', 102), ('fi_setup', 110), ('fi_greedy', 112)):
        t, c = eng.profile_read(cid)
        classes[name] = {'ms': t, 'launches': c, 'macs_per_sample': 0, 'tc': 0, 'type': -1}
    eng.profile(False)
    if args.dump_outputs and rank == 0:
        # the last timed step's answers and its pool posteriors (still in the pool buffers: the e2e leg below reuses them);
        # with several ranks, the posteriors are rank 0's shard
        dump_outputs(args.dump_outputs, {'entropy_query': q_res[0], 'fi_query': q_res[1], 'fi_reduced_objective': q_res[2],
                                         'fi_objective': q_res[3]}, eng.pool_posteriors(), 'pool_posteriors', lo)
    if world > 1:
        tms = torch.tensor([dev_ms] + list(stage_acc), dtype=torch.float64, device='cuda')
        torch.distributed.all_reduce(tms, op=torch.distributed.ReduceOp.MAX)
        dev_ms = float(tms[0].item())
        stage_acc = tms[1:].cpu().numpy()
    value = pool_total * args.steps / (dev_ms * 1e-3)

    # ---------------- end-to-end leg through the reference-facing API ----------------
    # (right after the resident leg, so that both legs of the headline see the chip in the same thermal / power state;
    # the stage evidence below runs minutes of other work)
    expr = Expr()
    expr.pars = dict(k=k, B=B, lambda_=0., patch_shape=PATCH, ntb=10000, stats=stats, fi_layers=2, fi_diag_load=FI_DELTA)
    eng.volume_cache = False                      # volumes are copied host->device every step
    for _ in range(args.warmup):
        q_e2e = nnal_b200.PW_NNAL.CNN_query(expr, model, None, padded, pool, None, 'entropy+fi')
    barrier()
    h0, d0 = eng.h2d_bytes, eng.d2h_bytes
    t0 = time.perf_counter()
    e2e_marks = [t0]
    for _ in range(args.steps):
        q_e2e = nnal_b200.PW_NNAL.CNN_query(expr, model, None, padded, pool, None, 'entropy+fi')
        e2e_marks.append(time.perf_counter())      # (the query returns host arrays: it has synchronised)
    eng.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_each = np.diff(np.array(e2e_marks)) * 1e3
    barrier()
    h2d = (eng.h2d_bytes - h0) / args.steps
    d2h = (eng.d2h_bytes - d0) / args.steps
    if world > 1:
        tms = torch.tensor([e2e_s], dtype=torch.float64, device='cuda')
        torch.distributed.all_reduce(tms, op=torch.distributed.ReduceOp.MAX)
        e2e_s = float(tms.item())
    e2e_value = pool_total * args.steps / e2e_s
    assert np.array_equal(q_e2e[0], q_res[0]) and np.array_equal(q_e2e[1], q_res[1]), 'resident and e2e legs disagree'
    eng.volume_cache = True

    # ---------------- stage evidence (extra keys) ----------------
    ent = run_entropy_round(args, eng, d_inds, n_local, lo, pool_total, st, k, barrier, world)
    fi = run_fi_extras(args, eng, model, padded, stats, pool, lo, hi, peaks, barrier, rank, world) if args.fi_B > 0 else None
    mc = run_mc_round(args, eng, model, lo, hi, d_inds, st, k) if args.mc_T > 0 else None
    sdp = run_sdp_round(args, eng, padded, pool, st, k) if args.sdp_B > 0 and world == 1 else None
    c4 = run_config4(eng, padded, stats, peaks, slices=args.config4_slices) if args.config4_slices > 0 and world == 1 else None
    up = run_upload(eng, padded) if world == 1 else None

    strong = run_strong_scaling(args, eng, model, rank, world, barrier) if args.strong_pool > 0 else None

    if rank != 0:
        return
    # ---------------- roofline of the dominant kernel (classes that share a kernel are pooled) ----------------
    kernels = {}
    for name, v in classes.items():
        if v['type'] == 0:
            kern = 'conv_wt_kernel' if v['tc'] == 2 else ('conv_tc_kernel' if v['tc'] else 'conv_simt_kernel')
        elif v['type'] == 2:
            kern = 'head_kernel' if name == layer_names[-1] else ('fc_tc_kernel' if v['tc'] else 'fc_simt_kernel')
        elif v['type'] == 1:
            continue
        else:
            kern = name
        kk = kernels.setdefault(kern, {'ms': 0., 'launches': 0, 'macs_per_sample': 0, 'classes': [], 'tc': v['tc']})
        kk['ms'] += v['ms']
        kk['launches'] += v['launches']
        kk['macs_per_sample'] += v['macs_per_sample'] if v['launches'] else 0
        kk['classes'].append(name)
    traffic = load_traffic()
    top = max((kk for kk in kernels if kk not in ('fi_greedy', 'fi_setup')), key=lambda kk: kernels[kk]['ms'])
    tinfo = kernels[top]
    per_launch_ms = tinfo['ms'] / max(1, tinfo['launches'])
    tr = [traffic.get(c) for c in tinfo['classes']]
    tr_bytes = None if any(t is None for t in tr) else sum(t['dram_bytes_per_sample'] for t in tr) * n_local * args.steps / max(1, tinfo['launches'])
    if tinfo['macs_per_sample'] > 0:
        flops_total = 2.0 * tinfo['macs_per_sample'] * n_local * args.steps          # over all launches of the timed region
        achieved = flops_total / (tinfo['ms'] * 1e-3) / 1e12
        peak = peaks['bf16_sustained']
        roofline = {'kernel': top, 'layers': tinfo['classes'], 'bound': 'tensor', 'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s',
                    'frac': achieved / peak, 'traffic': tr_bytes,
                    'launches': tinfo['launches'], 'ms_per_launch': per_launch_ms,
                    'share_of_step': tinfo['ms'] / dev_ms,
                    'executed': None if not tinfo['tc'] else {'achieved': 3 * achieved, 'frac': 3 * achieved / peak,
                                                             'what': 'tensor FLOPs issued by the split-precision scheme: hi.hi + hi.lo + lo.hi per product'},
                    'note': 'algorithmic FLOPs (2*MACs of %s) of all launches / their summed device time (CUDA events on the '
                            "library's stream); peak = %s sustained bf16" % ('+'.join(tinfo['classes']), peaks['source'])}
    else:
        bytes_per = {'gather': 15008.0, 'score': 12.0, 'topk': 4.0}.get(top, 0.0)
        achieved = bytes_per * n_local * args.steps / (tinfo['ms'] * 1e-3) / 1e9
        roofline = {'kernel': top, 'bound': 'hbm', 'achieved': achieved, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
                    'frac': achieved / peaks['hbm_gbs'], 'traffic': tr_bytes, 'share_of_step': tinfo['ms'] / dev_ms,
                    'note': 'peak = %s copy bandwidth' % peaks['source']}
    stage_ms = {kk: round(v['ms'] / args.steps, 4) for kk, v in classes.items()}
    stage_ms.update({'round:' + n_: round(float(v) / args.steps, 4) for n_, v in zip(stage_names, stage_acc)})
    kernel_ms = {kk: round(v['ms'] / args.steps, 4) for kk, v in kernels.items()}

    # ---------------- CPU baseline (bounded sample, rank 0, N=1 only) ----------------
    cpu = None
    if world == 1 and not args.no_cpu:
        fi_Bs = max(K_QUERY, int(round(args.fi_B * args.cpu_sample / float(args.pool))))
        dt, n, threads, det = cpu_reference_round(args.cpu_sample, fi_Bs)
        cpu = {'value': n / dt, 'unit': UNIT, 'cores': threads, 'kind': 'port', 'sample': _cpu_desc(n, fi_Bs, args.pool),
               'entropy_half_s': det['entropy_half_s'], 'fi_half_s': det['fi_half_s']}

    cfg = workload_config(args, world)
    if world > 1:
        cfg['greedy_step_exchange'] = fimod.last_exchange
    if strong:
        cfg['config3_check'] = {kk: strong[kk] for kk in ('pool', 'subjects', 'hash_entropy', 'hash_fi', 'primal_vs_dual_rel')}
    line = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': dev_ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
            'vs_baseline': None, 'dtype': 'f16x3 (fp16 hi/lo split operands, 3 tcgen05 MMAs per product, fp32 accumulate) + f32/f64 scoring and FI',
            'data': 'synthetic',
            'config': cfg,
            'clocks': clocks, 'gpu_launches': int(launches),
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                    'ms_per_step': 1e3 * e2e_s / args.steps, 'ms_per_step_min_median_max': [float(e2e_each.min()), float(np.median(e2e_each)), float(e2e_each.max())],
                    'ms_each': [round(float(x), 1) for x in e2e_each[:64]],
                    'api': 'nnal_b200.PW_NNAL.CNN_query(expr, model, sess, padded_imgs, pool_inds, tr_inds, "entropy+fi")'},
            'roofline': roofline, 'cpu_baseline': cpu, 'stage_ms_per_step': stage_ms, 'kernel_ms_per_step': kernel_ms,
            'entropy_round': ent, 'mc_round': mc, 'fi_sdp_round': sdp, 'config4': c4, 'volume_upload': up, 'fi_round': fi,
            'strong_scaling': strong}
    print(json.dumps(line))


def run_entropy_round(args, eng, d_inds, n_local, lo, pool_total, st, k, barrier, world):
    """The entropy query alone (round-1 headline; kept as a stage): pool pass without factors + top-k."""
    import torch
    from nnal_b200 import _lib as L
    from nnal_b200 import dist
    stream = torch.cuda.ExternalStream(eng.stream)

    def step():
        eng.pool_begin(n_local, 0)
        eng.pool_eval_device(0, d_inds.data_ptr(), n_local, 0, PATCH, st)
        eng.pool_score(L.SCORE_BINARY)
        return dist.topk_global(eng, k, lo, pool_total)[0]
    step()
    barrier()
    reps = max(2, min(args.steps, 5))
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(reps):
        step()
    ev1.record(stream)
    ev1.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device='cuda')
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        ms = float(t.item())
    return {'ms_per_round': ms, 'samples_per_s': pool_total / (ms * 1e-3)}


def run_mc_round(args, eng, model, lo, hi, d_inds, st, k):
    """One MC-entropy round (PW_NNAL.py:67-87) on the same pool: T dropout passes.  The conv trunk runs once per chunk,
    only the FC tail T times; the reference runs T complete batch_eval passes."""
    import torch
    from nnal_b200 import _lib as L
    n_local = hi - lo
    T = args.mc_T
    stream = torch.cuda.ExternalStream(eng.stream)
    eng.set_dropout_seed(5)

    def mc_step():
        eng.pool_mc_config(T, 0.5, model.dropout_layers, pos0=lo)
        try:
            eng.pool_begin(n_local, 0)
            eng.pool_eval_device(0, d_inds.data_ptr(), n_local, 0, PATCH, st)
        finally:
            eng.pool_mc_config(0, 1., [])
        eng.pool_score(L.SCORE_MC_BINARY)
        return eng.pool_topk(k)
    mc_step()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 2
    ev0.record(stream)
    for _ in range(reps):
        mc_step()
    ev1.record(stream)
    ev1.synchronize()
    ms = ev0.elapsed_time(ev1) / reps
    return {'method': 'MC-entropy', 'T': T, 'keep_prob': 0.5, 'ms_per_round': ms,
            'stochastic_passes_per_s': n_local * T / (ms * 1e-3),
            'note': 'conv trunk once per chunk + T FC-tail passes with Philox dropout fused into the FC epilogue / head'}


def run_sdp_round(args, eng, padded, pool, st, k):
    """The reference's literal FI selection (PW_NNAL.py:117-163) for B pre-filtered candidates: shrunk class-score
    gradients (one batched backward pass instead of 2B sess.run(tf.gradients) calls), A-matrices, SDP query distribution
    (first-order solver on the device, certified gap), sampling.  Host wall time per stage (the stages synchronise)."""
    from nnal_b200 import NNAL_tools
    B = min(args.sdp_B, len(pool))
    cand = pool[:B]
    res = None
    for rep in range(2):                       # first repetition warms the workspaces up
        eng.profile(True)
        t0 = time.perf_counter()
        post, g = eng.fi_shrunk_voxels(0, cand, PATCH, st, shape=padded[0].shape)
        t1 = time.perf_counter()
        fwd_ms, _ = eng.profile_read(120)
        bwd_ms, _ = eng.profile_read(121)
        eng.profile(False)
        t2 = time.perf_counter()
        r = eng.sdp_from_shrunk(g, post[1].astype(np.float64), 1e-5, tol=1e-4)       # A-matrices assembled on the device
        t3 = time.perf_counter()
        Q = NNAL_tools.sample_query_dstr(r['q'].copy(), k, replacement=True)
        t4 = time.perf_counter()
        res = {'B': int(B), 'k': int(k), 'tau': int(g.shape[2]), 'diag_load': 1e-5,
               'stage_ms': {'shrunk_gradients(gather+forward+backward)': 1e3 * (t1 - t0), 'sdp_solver(incl. A-matrices on the device)': 1e3 * (t3 - t2), 'sampling(host)': 1e3 * (t4 - t3)},
               'ms_per_round': 1e3 * (t4 - t0),
               'shrunk_device_ms': {'forward(all activations kept)': fwd_ms, 'backward(data gradients + layer sums)': bwd_ms},
               'backprops_per_s': 2.0 * B / (t1 - t0),
               'sdp': {'iterations': int(r['iterations']), 'objective': float(r['objective']), 'gap': float(r['gap']),
                       'us_per_iteration': 1e6 * (t3 - t2) / max(1, int(r['iterations'])),
                       'support': int((r['q'] > 1e-8).sum())},
               'n_selected': int(len(Q))}
    if not args.no_cpu and res is not None:
        # the same selection through the float64 oracle on a bounded sample of the candidates (reported baseline: the
        # reference itself runs two TF sess.run(tf.gradients) calls per candidate, which cannot be installed here)
        import oracle as O
        ns = 48
        x = O.normalize_batch_eval(O.get_patches(padded, cand[:ns], PATCH), st).astype(np.float32)
        layers = O.pw1_layers(2)
        w = O.he_init_weights(layers, (25, 25, 3), 4)
        t0 = time.perf_counter()
        po, go = O.shrunk_class_gradients(layers, w, x)
        t1 = time.perf_counter()
        Ao = O.gen_A_matrices(go[0], go[1], po[1], 1e-5)
        qo, to, phio, gapo, ito = O.sdp_solve(Ao, 1e-4)
        t2 = time.perf_counter()
        res['cpu_baseline'] = {'kind': 'port', 'cores': 1, 'sample': '%d candidates (NumPy float64 forward + one backward pass per '
                               'class + shrink + multiplicative SDP)' % ns,
                               'backprops_per_s': 2.0 * ns / (t1 - t0), 'sdp_ms': 1e3 * (t2 - t1), 'sdp_iterations': int(ito)}
    return res


def run_fi_extras(args, eng, model, padded, stats, pool, lo, hi, peaks, barrier, rank, world):
    """FI evidence on the same pool through the public API: the 'fi' query alone (what the reference's 'fi' branch costs a
    caller: pool pass + pre-filter + factors + greedy), and the Gram (primal) evaluation of its selection: per-GPU partial
    Grams on tensor cores, NCCL all-reduce, float64 (d+1)^2 solve -- primal objective against the greedy loop's dual one."""
    import torch
    import nnal_b200
    from nnal_b200 import fi as fimod
    expr = Expr()
    B = min(args.fi_B, len(pool))
    expr.pars = dict(k=K_QUERY, B=B, lambda_=0., patch_shape=PATCH, ntb=10000, stats=stats, fi_layers=2, fi_diag_load=FI_DELTA)
    nnal_b200.PW_NNAL.CNN_query(expr, model, None, padded, pool, None, 'fi')
    barrier()
    reps = max(1, min(args.steps, 3))
    t0 = time.perf_counter()
    for _ in range(reps):
        q, obj, red = fimod.query_single(expr, model, None, padded, pool, return_objective='reduced')
    eng.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / reps
    # Gram form of the last-layer objective for this selection (the report needs the factors of the round just run)
    expr.pars.update(fi_report=True, fi_layers=1)
    fimod.query_single(expr, model, None, padded, pool)             # warm-up of the Gram / solve workspaces
    eng.profile(True)
    t0 = time.perf_counter()
    q1, obj1, red1 = fimod.query_single(expr, model, None, padded, pool, return_objective='reduced')
    eng.synchronize()
    ms_rep = 1e3 * (time.perf_counter() - t0)
    gram_ms, _ = eng.profile_read(111)
    solve_ms, _ = eng.profile_read(113)
    eng.profile(False)
    rep = dict(fimod.last_report)
    d = eng.fi_info()['d']
    gram_flops = 2.0 * rep['n_candidates'] / world * (d + 1) ** 2
    out = {'B': int(B), 'k': K_QUERY, 'fi_layers': 2, 'delta': FI_DELTA,
           'fi_query_ms(host wall, incl. own pool pass)': ms, 'samples_per_s': len(pool) / (ms * 1e-3),
           'reduced_objective_final': float(red[-1]) if len(red) else None,
           'gram_report(fi_layers=1)': {
               'query_ms_with_report': ms_rep, 'pool_gram_ms': rep.get('gram_ms'), 'allreduce_ms': rep.get('allreduce_ms'),
               'allreduce_bytes': rep['gram_bytes'],
               'allreduce_bus_GBps': None if not rep.get('allreduce_ms') or world == 1 else
               2.0 * (world - 1) / world * rep['gram_bytes'] / (rep['allreduce_ms'] * 1e-3) / 1e9,
               'gram_gemm_ms(both Grams)': gram_ms, 'gram_tflops_algorithmic': gram_flops / max(rep.get('gram_ms') or 1e-9, 1e-9) / 1e9,
               'solve_ms(f64 Gauss-Jordan %dx%d)' % (d + 1, d + 1): solve_ms,
               'primal_last_layer': rep['primal_last_layer'], 'dual_last_layer': rep['dual_last_layer'],
               'dual_objective_of_greedy': rep['dual_objective'],
               'primal_vs_dual_rel': abs(rep['primal_last_layer'] / rep['dual_objective'] - 1.),
               'primal_reduced': rep['primal_reduced'], 'dual_reduced': rep['dual_reduced'], 'fi_ratio': rep['fi_ratio']}}
    return out


def run_upload(eng, padded):
    """Host->device time of the three volumes of the workload (170 MB) from pinned host memory (what the e2e leg uses, as
    the bench contract asks) and from PAGEABLE memory (what np.pad hands a caller of the reference): the library stages
    pageable arrays through its own pinned ring on 8 copy threads; `plain` is one cudaMemcpyAsync per modality."""
    out = {}
    nb = sum(a.nbytes for a in padded)
    pageable = [np.array(a, copy=True) for a in padded]
    cache = eng.volume_cache
    eng.volume_cache = False
    try:
        for name, arrs, plain in (('pinned', padded, 0), ('pageable_staged', pageable, 0), ('pageable_plain', pageable, 1)):
            eng.debug_option('plain_upload', plain)
            best = None
            for _ in range(4):
                eng.synchronize()
                t0 = time.perf_counter()
                eng.upload(0, arrs)
                eng.synchronize()
                dt = time.perf_counter() - t0
                best = dt if best is None or dt < best else best
            out[name] = {'ms': 1e3 * best, 'GBps': nb / best / 1e9}
    finally:
        eng.debug_option('plain_upload', 0)
        eng.volume_cache = cache
        eng.upload(0, padded)
    out['bytes'] = nb
    return out


def run_config4(eng, padded, stats, peaks, slices=180, reps=3):
    """Config 4 of BASELINE.json (memory-bound path): (i) gather the 25x25x3 patches of EVERY voxel of `slices` slices of
    the 256x256x180 volume, slice by slice as PW_analyze_results.full_slice_eval does (PW_analyze_results.py:689-715) --
    each slice's 65,536 patches (491 MB) go to a reused device buffer; (ii) pixel-wise entropy of a [c=2,256,256,180]
    float32 posterior tensor.  CUDA-event timing on the library's stream."""
    import torch
    from nnal_b200 import _lib as L
    st = np.array(stats, dtype=np.float64)
    X, Y, Z = VOL_SHAPE
    stream = torch.cuda.ExternalStream(eng.stream)
    per_slice = X * Y
    out = torch.empty((per_slice, 25, 25, 3), dtype=torch.float32, device='cuda')
    xy = torch.arange(per_slice, dtype=torch.int64, device='cuda') * Z
    idx = [xy + z for z in range(slices)]
    torch.cuda.synchronize()
    res = {}
    for name, norm in (('raw', L.NORM_NONE), ('normalised', L.NORM_BATCH_EVAL)):
        for z in range(min(3, slices)):
            eng.gather_device(0, idx[z].data_ptr(), per_slice, PATCH, st, norm, out.data_ptr())
        eng.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for z in range(slices):
            eng.gather_device(0, idx[z].data_ptr(), per_slice, PATCH, st, norm, out.data_ptr())
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        npatch = per_slice * slices
        gbs = npatch * 15008.0 / (ms * 1e-3) / 1e9
        res['gather_' + name] = {'patches': npatch, 'ms': ms, 'patches_per_s': npatch / (ms * 1e-3), 'algorithmic_GBps': gbs,
                                 'frac_of_hbm_peak': gbs / peaks['hbm_gbs'], 'bytes_per_patch': 15008,
                                 'hbm_write_GBps': npatch * 7500.0 / (ms * 1e-3) / 1e9,
                                 'note': 'algorithmic bytes count 7,500 B read + 7,500 B written + 8 B index per patch; overlapping '
                                         'patches are re-read from L2, so HBM itself sees about the write stream (hbm_write_GBps)'}
    n = X * Y * Z
    NSET = 4
    g = torch.Generator(device='cuda')
    g.manual_seed(5)
    posts, Hs = [], []
    for _ in range(NSET):
        logits = torch.randn((2, n), generator=g, device='cuda', dtype=torch.float32)
        posts.append(torch.softmax(logits, dim=0).contiguous())
        Hs.append(torch.empty(n, dtype=torch.float32, device='cuda'))
    torch.cuda.synchronize()
    for i in range(NSET):
        eng.entropy_device(posts[i].data_ptr(), 2, n, 1e-7, Hs[i].data_ptr())
    eng.synchronize()
    R = 8 * NSET
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    gate = torch.empty(1 << 28, dtype=torch.uint8, device='cuda')
    tot = 0.0
    for _ in range(reps):
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            gate.zero_()                                     # keeps the GPU busy while the launch train is queued
        e0.record(stream)
        for i in range(R):
            eng.entropy_device(posts[i % NSET].data_ptr(), 2, n, 1e-7, Hs[i % NSET].data_ptr())
        e1.record(stream)
        e1.synchronize()
        tot += e0.elapsed_time(e1) / R
    ms = tot / reps
    gbs = n * 12.0 / (ms * 1e-3) / 1e9
    p64 = posts[0].double()
    Href = -(p64 * torch.log(p64)).sum(0)
    err = float(((Hs[0].double() - Href).abs() / Href.abs().clamp_min(1e-12)).max())
    res['entropy_map'] = {'voxels': n, 'ms': ms, 'algorithmic_GBps': gbs, 'frac_of_hbm_peak': gbs / peaks['hbm_gbs'],
                          'bytes_per_voxel': 12, 'max_rel_err_vs_f64': err,
                          'l2': '%d rotating tensor sets of 141 MB (larger than L2), %d launches per timed train' % (NSET, R)}
    res['slices'] = slices
    del out, posts, Hs, gate
    torch.cuda.empty_cache()
    return res


def make_strong_workload(pool_total, S):
    """BASELINE config 3 / SURVEY.md 8d: S synthetic subjects (3 modalities 256x256x180 each, derived from the config-2
    volumes by a per-subject shift, gain and offset -- cheap to generate, distinct content and stats), pool_total/S distinct
    voxels per subject; train_stats (S, 2m) in the reader layout [i,2j] = mean, [i,2j+1] = std."""
    padded0, stats0, _ = make_workload(10)
    nvox = int(np.prod(VOL_SHAPE))
    per = pool_total // S
    allp, pools = [], []
    st = np.zeros((S, 2 * N_MOD))
    for s in range(S):
        gain, off = np.float32(1. + 0.03 * s), np.float32(2. * s)
        sub = []
        for j in range(N_MOD):
            core = np.roll(padded0[j][12:-12, 12:-12, :], 17 * s + 5 * j, axis=0) * gain + off
            buf = np.zeros_like(padded0[j])
            buf[12:-12, 12:-12, :] = core
            sub.append(buf)
            st[s, 2 * j], st[s, 2 * j + 1] = stats0[j][0] * gain + off, stats0[j][1] * gain
        allp.append(sub + [np.zeros((1, 1, 1), dtype=np.int8)])          # the mask is not read by the query path
        pools.append(np.random.RandomState(100 + s).choice(nvox, per, replace=False).astype(np.int64))
    return allp, pools, st


def run_strong_scaling(args, eng, model, rank, world, barrier):
    """BASELINE config 3 at ANY N: a fixed `--strong-pool`-patch pool of S = 8 subjects through the public multi-volume API
    (PW_NNAL.query_multimg, 'entropy+fi': one pool pass), FI over the last two FC layers WITHOUT pre-filter (B = n: every
    pool sample is a greedy candidate), sharded over the ranks.  Reports host wall time per round (max over ranks), a hash
    of the selected (subject, position) lists -- identical at N = 1/2/4/8 -- and the Gram evidence: per-GPU partial Grams of
    all candidates on tensor cores, NCCL all-reduce on the library's stream, the primal objective through the reduced Gram
    of the selection against its dual (kernel) value."""
    import torch
    import nnal_b200
    from nnal_b200 import fi as fimod
    S = 8
    n = args.strong_pool // S * S
    allp, pools, st = make_strong_workload(n, S)
    expr = Expr()
    expr.pars = dict(k=K_QUERY, B=n, lambda_=0., patch_shape=PATCH, ntb=10000, SDP_solver='CVXOPT', fi_layers=2)
    expr.train_stats, expr.nclass = st, 2
    eng.volume_cache = True
    Qe, Qf = nnal_b200.PW_NNAL.query_multimg(expr, model, None, allp, pools, None, 'entropy+fi')      # uploads + warm-up
    barrier()
    reps = 2
    t0 = time.perf_counter()
    for _ in range(reps):
        Qe, Qf, obj, red = fimod.query_multimg(expr, model, None, allp, pools, return_objective='reduced', also_entropy=True)
    eng.synchronize()
    ms = 1e3 * (time.perf_counter() - t0) / reps
    # the Gram form: last-layer FI of the SAME selection (fi_layers = 1 makes the greedy's dual objective the comparable one)
    expr.pars.update(fi_layers=1, fi_report=True)
    fimod.query_multimg(expr, model, None, allp, pools)
    barrier()
    t0 = time.perf_counter()
    Q1, obj1, red1 = fimod.query_multimg(expr, model, None, allp, pools, return_objective='reduced')
    eng.synchronize()
    ms1 = 1e3 * (time.perf_counter() - t0)
    rep = dict(fimod.last_report)
    vals = [ms, ms1, rep.get('gram_ms') or 0., rep.get('allreduce_ms') or 0.]
    if world > 1:
        t = torch.tensor(vals, dtype=torch.float64, device='cuda')
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
        vals = t.cpu().numpy().tolist()
    d = eng.fi_info()['d']
    rel = abs(rep['primal_last_layer'] / rep['dual_objective'] - 1.)
    assert rel < 1e-3, 'primal (Gram) and dual objectives disagree: %g' % rel
    return {'pool': int(n), 'subjects': S, 'k': K_QUERY, 'B': int(n), 'fi_layers': 2, 'delta': 1e-3, 'n_gpus': world,
            'scaling': 'strong (fixed pool)', 'ms_per_round(entropy+fi, host wall, max over ranks)': vals[0],
            'samples_per_s': n / (vals[0] * 1e-3),
            'hash_entropy': digest(*Qe), 'hash_fi': digest(*Qf), 'hash_fi_last_layer': digest(*Q1),
            'fi_reduced_objective_final': float(red[-1]),
            'gram': {'candidates_per_rank': rep['n_candidates'] // world, 'pool_gram_ms': vals[2], 'allreduce_ms': vals[3],
                     'allreduce_bytes': rep['gram_bytes'],
                     'allreduce_bus_GBps': None if world == 1 or not vals[3] else
                     2.0 * (world - 1) / world * rep['gram_bytes'] / (vals[3] * 1e-3) / 1e9,
                     'gram_tflops_algorithmic_per_gpu': 2.0 * (rep['n_candidates'] / world) * (d + 1) ** 2 / max(vals[2], 1e-9) / 1e9,
                     'query_ms_with_report(fi_layers=1)': vals[1]},
            'primal_last_layer': rep['primal_last_layer'], 'dual_objective_of_greedy': rep['dual_objective'],
            'dual_last_layer': rep['dual_last_layer'], 'primal_vs_dual_rel': rel, 'fi_ratio': rep['fi_ratio']}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--pool', type=int, default=100000, help='pool samples per GPU')
    ap.add_argument('--cpu-sample', type=int, default=5000)
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--fi-B', type=int, default=10000, help='FI pre-filter size of the query round')
    ap.add_argument('--sdp-B', type=int, default=10000, help='candidates of the extra literal-FI (shrunk gradients + SDP) round at 1 GPU (0: skip)')
    ap.add_argument('--no-p2p', action='store_true', help='greedy step messages through NCCL all-gather instead of the peer-memory exchange')
    ap.add_argument('--mc-T', type=int, default=10, help='MC-dropout passes of the extra MC-entropy round (0: skip)')
    ap.add_argument('--config4-slices', type=int, default=180, help='slices of the config-4 full-volume gather at 1 GPU (0: skip)')
    ap.add_argument('--strong-pool', type=int, default=1000000, help='fixed pool of the config-3 strong-scaling leg (0: skip)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the last timed step\'s outputs as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error('--steps must be at least 1 and --warmup at least 0')
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as td
        torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
        td.init_process_group('nccl')
    try:
        run_ours(args, rank, world)
    finally:
        if world > 1:
            import torch.distributed as td
            td.destroy_process_group()


if __name__ == '__main__':
    main()
