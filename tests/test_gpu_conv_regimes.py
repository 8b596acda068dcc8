"""Tensor-core convolutions against float64 past one sample group per CTA (``pytest -m gpu``; the plan-table test runs
without a GPU).

``conv_tc_kernel<Cfg>`` (csrc/conv_tc.cu) and ``conv_wt_kernel<Cfg>`` (csrc/conv_wt.cu) are persistent: they launch
min(groups, SMs) CTAs and CTA b walks the sample groups b, b + grid, ...  State carries over from one group to the next:
the input-buffer ring (NBUF buffers), the streamed weight ring (3 stages, for plans whose weights are not resident), the
NACC accumulators and the epilogue warpgroup that drains each tile group, the reversed tile-group order of odd samples
(NG = 2), the pooled raster cleared after each sample, the staging buffers of the fused gather, and the two row bands
of conv_wt.cu's single input raster.  Every tile plan is run here

1. on a grid capped at 2 and 3 CTAs (debug option ``conv_grid``) so that every CTA runs at least max(16, 2 P) groups, P
   being the number of groups after which all of its ring states repeat, against NumPy float64, and bit for bit
   against the same samples on the default grid (one group per CTA): the MMA sequence of an output does not depend on
   the CTA or iteration that computes it;
2. on the full grid at production size (16,384 samples forward, 2,048 backward), at SMs x G - 1, SMs x G and
   SMs x G + 1 samples and at one sample, against float64 torch on the device.

Sample s is scaled by 2^-(i mod 8), i = (s // G) // grid its iteration on its CTA, so a stale input buffer, weight stage
or pooled maximum of an earlier (larger) sample dominates the result instead of hiding in it, and every sample is held
to 3e-5 of ITS OWN max |ref|.  The plan constants come from the ``typedef Cfg<...>`` lines of the sources, and every
case asserts the regime it is there for."""
import math
import os
import re
from types import SimpleNamespace

import numpy as np
import pytest

import oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'nn-active-learning_b200', 'csrc')
SM_COUNT = 148                     # B200
TOL = 3e-5                         # per sample, relative to the sample's max |ref| (the conv bar of test_gpu_parity)
CAP_GROUPS = 73                    # groups of the capped-grid runs: 37 + 36 on 2 CTAs, 25 + 24 + 24 on 3 (P <= 12)
CAPS = (2, 3)
PROD_FWD, PROD_BWD = 16384, 2048   # samples per forward chunk / per chunk of the shrunk-gradient pass


# ------------------------------------------------------------------ plan table from the sources
def _src(name):
    return open(os.path.join(CSRC, name)).read()


def _args(s):
    return [a.strip() for a in s.split(',')]


def ctc_plans():
    """conv_tc.cu: name -> the Cfg constants (the arithmetic of struct Cfg)."""
    plans = {}
    for m in re.finditer(r'typedef Cfg<([^>]*)> (\w+);', _src('conv_tc.cu')):
        a = _args(m.group(1))
        H, W, CIN, COUT, KS, G, KPS, NBUF, TG = map(int, a[:9])
        opt = lambda i, d: a[i] if len(a) > i else d
        POOL, GATHER, RAW = opt(10, 'false') == 'true', opt(14, 'false') == 'true', opt(16, 'false') == 'true'
        KW = int(opt(12, '0')) or KS
        NACC = int(opt(15, '2'))
        HP, WP, Q = H + KS - 1, W + KW - 1, -(-CIN // 8)
        NK = (KS * KW * Q + 1) // 2
        NSTAGE_W = -(-NK // KPS)
        T = ((G - 1) * HP * WP + (H - 1) * WP + (W - 1)) // 128 + 1
        plans[m.group(2)] = SimpleNamespace(kernel='tc', H=H, W=W, CIN=CIN, COUT=COUT, KS=KS, G=G, NBUF=NBUF, T=T, TG=TG,
                                            NG=-(-T // TG), NACC=NACC, NSTAGE_W=NSTAGE_W, WRES=NSTAGE_W <= 3, POOL=POOL,
                                            GATHER=GATHER, RAW=RAW)
    return plans


def cwt_plans():
    """conv_wt.cu: 'wt:' + name -> the Cfg constants."""
    plans = {}
    for m in re.finditer(r'typedef Cfg<([^>]*)> (\w+);', _src('conv_wt.cu')):
        a = _args(m.group(1))
        H, W, CIN, COUT, KS, TAPS, G, RL = map(int, a[:8])
        WP, HP = W + KS - 1, H + KS - 1
        tile_out = 248 if TAPS == 2 else 256
        T = ((G - 1) * HP * WP + (H - 1) * WP + (W - 1)) // tile_out + 1
        plans['wt:' + m.group(2)] = SimpleNamespace(kernel='wt', H=H, W=W, CIN=CIN, COUT=COUT, KS=KS, G=G, T=T,
                                                    SPLIT=RL > 0, NBUF=1 if RL > 0 else 2, POOL=a[8] == 'true')
    return plans


def macro_list(name):
    m = re.search(r'#define %s\(X\)(.*)' % name, _src('conv_tc.cu'))
    return re.findall(r'X\((\w+)\)', m.group(1))


def period(p):
    """Groups after which every ring state of a CTA repeats."""
    lcm = lambda *v: math.lcm(*v)
    if p.kernel == 'wt':
        return lcm(2 * p.NBUF, 4 // math.gcd(p.T, 4), 2)              # input ring; 2 accumulators, T tiles per group
    P = lcm(2 * p.NBUF, 2 * p.NACC // math.gcd(p.NG, 2 * p.NACC), 2)   # input ring; accumulator + parity; reversal
    if not p.WRES:
        P = lcm(P, 6 // math.gcd(p.NG * p.NSTAGE_W, 6))              # 3-stage weight ring, NG * NSTAGE_W stages a group
    return P


# what the sources held when these tests were written (the weights column: 0 = resident, else streamed stages)
EXPECTED = {
    'CfgConv1': (1, 2, 6, 2, 2, 0), 'CfgConv1X': (1, 2, 5, 2, 2, 0), 'CfgConv1XG': (1, 2, 5, 3, 4, 0),
    'CfgConv3': (2, 2, 4, 1, 2, 0), 'CfgS1Conv3': (2, 2, 4, 1, 2, 0),
    'CfgConv4': (1, 2, 2, 1, 2, 9), 'CfgConv4Pool': (1, 2, 2, 1, 2, 9), 'CfgS1Conv4': (1, 2, 2, 1, 2, 9),
    'CfgS1Conv4Pool': (1, 2, 2, 1, 2, 9),
    'CfgS1Conv1': (1, 2, 7, 3, 2, 0), 'CfgS1Conv2': (1, 1, 7, 3, 2, 5), 'CfgConv2': (1, 2, 6, 2, 2, 5),
    'CfgBwd2': (1, 1, 6, 2, 2, 10), 'CfgS1Bwd2': (1, 1, 7, 3, 2, 10),
    'CfgBwd3': (1, 2, 2, 1, 2, 0), 'CfgS1Bwd3': (1, 2, 2, 1, 2, 0),
    'CfgBwd4': (1, 2, 2, 1, 2, 18), 'CfgS1Bwd4': (1, 2, 2, 1, 2, 18),
}
EXPECTED_WT = {'wt:CfgConv1': (2, False, 3), 'wt:CfgConv2': (1, True, 3), 'wt:CfgConv2Pool': (1, True, 3),
               'wt:CfgConv3': (2, False, 2)}               # (NBUF, SPLIT, T)

# plan -> how the tests reach it: (kind, H, Cin, Cout, ks, debug_conv mode) of the FORWARD layer
CASES = {
    'CfgConv1': ('fwd', 25, 3, 24, 5, 1), 'CfgConv2': ('fwd', 25, 24, 32, 5, 1), 'CfgConv3': ('fwd', 13, 32, 48, 3, 1),
    'CfgConv4': ('fwd', 13, 48, 96, 3, 1), 'CfgS1Conv1': ('fwd', 28, 1, 24, 5, 1), 'CfgS1Conv2': ('fwd', 28, 24, 32, 5, 1),
    'CfgS1Conv3': ('fwd', 14, 32, 48, 3, 1), 'CfgS1Conv4': ('fwd', 14, 48, 96, 3, 1),
    'CfgConv4Pool': ('pool', 13, 48, 96, 3, 4), 'CfgS1Conv4Pool': ('pool', 14, 48, 96, 3, 4),
    'CfgConv1X': ('fwd', 25, 3, 24, 5, 5),
    'CfgBwd2': ('bwd', 25, 24, 32, 5, None), 'CfgBwd3': ('bwd', 13, 32, 48, 3, None), 'CfgBwd4': ('bwd', 13, 48, 96, 3, None),
    'CfgS1Bwd2': ('bwd', 28, 24, 32, 5, None), 'CfgS1Bwd3': ('bwd', 14, 32, 48, 3, None),
    'CfgS1Bwd4': ('bwd', 14, 48, 96, 3, None),
    'wt:CfgConv1': ('fwd', 25, 3, 24, 5, 2), 'wt:CfgConv2': ('fwd', 25, 24, 32, 5, 2),
    'wt:CfgConv2Pool': ('pool', 25, 24, 32, 5, 3), 'wt:CfgConv3': ('fwd', 13, 32, 48, 3, 2),
}


def all_plans():
    p = ctc_plans()
    p.update(cwt_plans())
    return p


def groups_per_cta(ngroups, grid):
    return [-(-(ngroups - b) // grid) for b in range(grid)]


def capped_n(p):
    """Samples of the capped-grid runs: CAP_GROUPS groups, the last one half empty for G = 2."""
    return CAP_GROUPS * p.G - (p.G - 1)


def prod_sizes(p, kind):
    G = p.G
    return [PROD_BWD if kind == 'bwd' else PROD_FWD, SM_COUNT * G - 1, SM_COUNT * G, SM_COUNT * G + 1, 1]


def capped_regime(p, grid):
    """(groups per CTA, whether the regime is the one the capped case is there for)"""
    n = capped_n(p)
    ng = -(-n // p.G)
    per = groups_per_cta(ng, grid)
    ok = (min(per) >= max(16, 2 * period(p)) and per[-1] < per[0] and ng == CAP_GROUPS
          and (p.G == 1 or n % p.G == 1))
    return per, ok


def test_plan_table_and_regimes():
    """Every configuration the library launches has a row here with the constants of its Cfg line, and every GPU case
    below still gives the regime it states (a later edit of a Cfg line or of a case size cannot silently shrink the
    coverage)."""
    ctc, cwt = ctc_plans(), cwt_plans()
    names = macro_list('NNAL_CTC_FWD') + macro_list('NNAL_CTC_POOL') + macro_list('NNAL_CTC_BWD') + ['CfgConv1X', 'CfgConv1XG']
    assert len(names) == 18 and set(names) == set(ctc), set(names) ^ set(ctc)
    assert set(cwt) == set(EXPECTED_WT)
    for name in names:
        p = ctc[name]
        got = (p.G, p.NBUF, p.T, p.NG, p.NACC, 0 if p.WRES else p.NSTAGE_W)
        assert got == EXPECTED[name], '%s: (G, NBUF, T, NG, NACC, streamed stages) = %s' % (name, got)
        assert p.RAW == name.startswith(('CfgBwd', 'CfgS1Bwd')) and p.POOL == name.endswith('Pool')
    assert period(ctc['CfgConv1XG']) == 8
    for name, want in EXPECTED_WT.items():
        assert (cwt[name].NBUF, cwt[name].SPLIT, cwt[name].T) == want, name
    plans = all_plans()
    assert set(CASES) | {'CfgConv1XG'} == set(plans)
    for name, (kind, H, Cin, Cout, ks, mode) in CASES.items():
        p = plans[name]
        # the case's forward layer is the plan's shape (data gradients swap the channel counts)
        assert (p.H, p.KS) == (H, ks) and ((p.CIN, p.COUT) == (Cout, Cin) if kind == 'bwd' else
                                           p.COUT == Cout and p.CIN >= Cin), name
        assert kind == 'pool' if p.POOL else kind != 'pool'
        for grid in CAPS:
            per, ok = capped_regime(p, grid)
            assert ok, '%s on %d CTAs: groups per CTA %s, P = %d' % (name, grid, per, period(p))
        sizes = prod_sizes(p, kind)
        big = -(-sizes[0] // p.G)
        assert max(groups_per_cta(big, SM_COUNT)) >= (14 if kind == 'bwd' else 55), name
        assert [-(-n // p.G) for n in sizes[1:4]] == ([SM_COUNT - 1, SM_COUNT, SM_COUNT + 1] if p.G == 1 else
                                                      [SM_COUNT, SM_COUNT, SM_COUNT + 1]), name
    per, ok = capped_regime(plans['CfgConv1XG'], 3)
    assert ok and min(per) >= 2 * 8


# ------------------------------------------------------------------ GPU helpers
def scale_of(n, G, grid):
    """2^-(i mod 8) of every sample, i = the iteration of its group on its CTA."""
    s = np.arange(n)
    return np.ldexp(1.0, -(((s // G) // grid) % 8)).astype(np.float32)


def layer_params(Cin, Cout, ks, seed):
    rs = np.random.RandomState(seed)
    W = (rs.randn(ks, ks, Cin, Cout) * np.sqrt(2. / (ks * ks * Cin))).astype(np.float32)
    b = (rs.randn(Cout) * .1).astype(np.float32)
    return W, b


def make_input(kind, n, H, C, signed, scale, seed):
    """conv1: signed inputs; later layers: post-ReLU inputs with exact zeros; dz: signed, about half exact zeros."""
    import torch
    g = torch.Generator(device='cuda').manual_seed(seed)
    x = torch.randn(n, H, H, C, device='cuda', generator=g)
    if kind == 'bwd':
        x *= torch.rand(n, H, H, C, device='cuda', generator=g) < .5
    elif not signed:
        x.clamp_(min=0)
    x *= torch.from_numpy(scale).cuda()[:, None, None, None]
    return x.cpu().numpy()


def np_ref(kind, x, W, b):
    x64, W64 = x.astype(np.float64), W.astype(np.float64)
    if kind == 'bwd':
        # fi_oracle._backward: d_in[y, x, ci] = sum_{dy, dx, co} dz[y - dy + ph, x - dx + pw, co] W[dy, dx, ci, co]
        kh, kw = W.shape[:2]
        dzp = np.pad(x64, ((0, 0), (kh // 2, kh // 2), (kw // 2, kw // 2), (0, 0)), 'constant')
        win = np.lib.stride_tricks.sliding_window_view(dzp, (kh, kw), axis=(1, 2))
        return np.tensordot(win, W64[::-1, ::-1, :, :], axes=([4, 5, 3], [0, 1, 3]))
    r = np.maximum(O.conv2d_same(x64, W64, b.astype(np.float64)), 0)
    return O.max_pool_same(r) if kind == 'pool' else r


def torch_ref(kind, x, W, b):
    """float64 on the device: F.conv2d / conv_transpose2d (+ ReLU, + 2x2/s2 SAME max-pool = ceil-mode pooling)."""
    import torch
    import torch.nn.functional as F
    xt = torch.from_numpy(x).cuda().double().permute(0, 3, 1, 2)
    Wt = torch.from_numpy(W).cuda().double().permute(3, 2, 0, 1)          # [Cout][Cin][kh][kw]
    pad = W.shape[0] // 2
    if kind == 'bwd':
        r = F.conv_transpose2d(xt, Wt, padding=pad)
    else:
        r = F.conv2d(xt, Wt, torch.from_numpy(b).cuda().double(), padding=pad).clamp_min_(0)
        if kind == 'pool':
            r = F.max_pool2d(r, 2, 2, ceil_mode=True)
    return r.permute(0, 2, 3, 1).contiguous()


def per_sample_errors(got, ref):
    """(max |got - ref| per sample, max |ref| per sample) as float64 NumPy arrays; ref NumPy or a device tensor."""
    import torch
    if isinstance(ref, np.ndarray):
        e = np.abs(got.astype(np.float64) - ref).reshape(len(ref), -1).max(1)
        return e, np.abs(ref).reshape(len(ref), -1).max(1)
    g = torch.from_numpy(got).cuda().double()
    e = (g - ref).abs_().reshape(len(ref), -1).amax(1)
    return e.cpu().numpy(), ref.abs().reshape(len(ref), -1).amax(1).cpu().numpy()


def assert_per_sample(got, ref, what, G=1, grid=None, floor=None):
    """Every sample within TOL of its own max |ref| (plus ``floor`` when given); returns the worst relative error."""
    assert got.shape == tuple(ref.shape), (what, got.shape, tuple(ref.shape))
    e, s = per_sample_errors(got, ref)
    bound = TOL * s + (0 if floor is None else floor)
    rel = e / np.where(s > 0, s, 1)
    bad = np.flatnonzero(e > bound)
    if len(bad):
        i = bad[np.argmax(rel[bad])]
        where = '' if grid is None else ' (CTA %d, iteration %d)' % ((i // G) % grid, (i // G) // grid)
        pytest.fail('%s: %d samples off, worst sample %d%s: %.3g of its max %.3g' % (what, len(bad), i, where, e[i], s[i]))
    return float(rel.max())


def report(name, groups, worst):
    print('\nREGIME %s: %d groups per CTA max, worst per-sample error %.3g' % (name, groups, worst))


@pytest.fixture(scope='module')
def eng():
    import nnal_b200
    e = nnal_b200.get_engine()
    yield e
    e.debug_option('conv_grid', 0)
    for o in ('bw_no_ws', 'bw_no_tc8', 'wt_flags'):
        e.debug_option(o, 0)


def run(eng, kind, mode, x, W, b, grid=0):
    eng.debug_option('conv_grid', grid)
    try:
        return eng.debug_conv_bwd(x, W, 1) if kind == 'bwd' else eng.debug_conv(x, W, b, mode)
    finally:
        eng.debug_option('conv_grid', 0)


def cuda_core_variants(eng, x, W):
    for ws in (0, 1):
        for tc8 in (0, 1):
            eng.debug_option('bw_no_ws', ws)
            eng.debug_option('bw_no_tc8', tc8)
            try:
                yield 'fp32 CUDA cores bw_no_ws=%d bw_no_tc8=%d' % (ws, tc8), eng.debug_conv_bwd(x, W, 0)
            finally:
                eng.debug_option('bw_no_ws', 0)
                eng.debug_option('bw_no_tc8', 0)


def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


# ------------------------------------------------------------------ 1. capped grid: every ring state cycles, vs NumPy
@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(CASES))
def test_capped_grid_vs_f64(eng, name):
    """conv_grid = 2 and 3: >= 16 groups (>= 2 P) on every CTA, fewer on the last; NumPy float64 per sample at 3e-5 of
    the sample's own max, and bit-identical to the same samples on the default grid (one group per CTA).  Data
    gradients also on the fp32 CUDA-core kernel in all bw_no_ws / bw_no_tc8 variants."""
    assert _sm_count() == SM_COUNT
    p = all_plans()[name]
    kind, H, Cin, Cout, ks, mode = CASES[name]
    W, b = layer_params(Cin, Cout, ks, sum(map(ord, name)))
    n = capped_n(p)
    assert n <= SM_COUNT * p.G
    worst, most = 0., 0
    for grid in CAPS:
        per, ok = capped_regime(p, grid)
        assert ok, (per, period(p))
        most = max(most, max(per))
        C = Cout if kind == 'bwd' else Cin
        x = make_input(kind, n, H, C, Cin <= 3, scale_of(n, p.G, grid), 10 * grid + len(name))
        ref = np_ref(kind, x, W, b)
        got = run(eng, kind, mode, x, W, b, grid)
        worst = max(worst, assert_per_sample(got, ref, '%s on %d CTAs' % (name, grid), p.G, grid))
        plain = run(eng, kind, mode, x, W, b)
        diff = np.flatnonzero((got != plain).reshape(n, -1).any(1))
        assert not len(diff), '%s: %d CTAs differ from one group per CTA in samples %s' % (name, grid, diff[:10])
        if kind == 'bwd' and grid == CAPS[0]:
            for what, g in cuda_core_variants(eng, x, W):
                assert_per_sample(g, ref, '%s %s' % (name, what))
    report(name + ' capped', most, worst)


# ------------------------------------------------------------------ 2. full grid, production size, vs float64 torch
@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(CASES))
def test_full_grid_vs_f64(eng, name):
    """Production chunk (16,384 forward, 2,048 backward), SMs x G - 1, SMs x G, SMs x G + 1 samples and one sample on the
    default grid, against float64 torch on the device, every sample at 3e-5 of its own max.  Data gradients at production
    size also on the fp32 CUDA-core kernel."""
    assert _sm_count() == SM_COUNT
    p = all_plans()[name]
    kind, H, Cin, Cout, ks, mode = CASES[name]
    W, b = layer_params(Cin, Cout, ks, 7 + sum(map(ord, name)))
    worst, most = 0., 0
    for i, n in enumerate(prod_sizes(p, kind)):
        ng = -(-n // p.G)
        grid = min(ng, SM_COUNT)
        most = max(most, max(groups_per_cta(ng, grid)))
        x = make_input(kind, n, H, Cout if kind == 'bwd' else Cin, Cin <= 3, scale_of(n, p.G, grid), 100 + n)
        ref = torch_ref(kind, x, W, b)
        got = run(eng, kind, mode, x, W, b)
        worst = max(worst, assert_per_sample(got, ref, '%s n=%d' % (name, n), p.G, grid))
        if kind == 'bwd' and i == 0:
            for what, g in cuda_core_variants(eng, x, W):
                assert_per_sample(g, ref, '%s n=%d %s' % (name, n, what))
        del ref
    report(name + ' full grid', most, worst)


# ------------------------------------------------------------------ 3. data gradient of samples spanning 2^24
SPAN_BITS = 24


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(n for n in CASES if CASES[n][0] == 'bwd'))
def test_bwd_gradient_span(eng, name):
    """One call whose samples span 2^24 in magnitude (sample s scaled by 2^-k, k = 0 .. 24).

    The kernel multiplies the whole call's dz by one power of two 2^e that lifts max |dz| to [2^13, 2^14) and splits each
    scaled entry x into fp16 terms hi = fp16(x), lo = fp16(x - hi).  The residual x - hi - lo is at most 2^-22 |x| while lo
    is a normal fp16 number, and at most 2^-25 (half the subnormal spacing 2^-24) once it is not: an ABSOLUTE floor that
    does not shrink with the sample.  Carried through the products with the weights and scaled back by 2^-e, that floor
    adds at most 2^-25 2^-e sum_{taps, co} |W[., ., ci, co]| to an output.  So each sample must satisfy

        max |d_in - ref| <= 3e-5 max |ref| + 2^(-25 - e) max_ci sum_{dy, dx, co} |W[dy, dx, ci, co]|,

    and a sample whose scaled entries reach 2^2 (k <= 12) sees a floor below 1e-6 of its own scale: it must meet the
    plain 3e-5 bar.  The gradient of a confidently classified candidate is the tiny sample here: relative to its own
    size it carries an error of up to ~2^-14 when its dz is 2^-24 of the chunk's largest."""
    kind, H, Cin, Cout, ks, _ = CASES[name]
    W, _b = layer_params(Cin, Cout, ks, 11 + sum(map(ord, name)))
    n = 2 * SPAN_BITS + 1
    k = np.arange(n) * SPAN_BITS // (n - 1)
    x = make_input('bwd', n, H, Cout, True, np.ldexp(1.0, -k).astype(np.float32), 5)
    ref = np_ref('bwd', x, W, None)
    got = eng.debug_conv_bwd(x, W, 1)
    _, ex = np.frexp(np.abs(x).max())
    e = 14 - int(ex)
    floor = np.ldexp(np.abs(W.astype(np.float64)).sum(axis=(0, 1, 3)).max(), -25 - e)
    assert_per_sample(got, ref, '%s spanning 2^%d' % (name, SPAN_BITS), floor=floor)
    above = k <= 12
    worst = assert_per_sample(got[above], ref[above], '%s samples within 2^12 of the largest' % name)
    err, sc = per_sample_errors(got, ref)
    print('\nSPAN %s: samples within 2^12 %.3g, sample at 2^-%d %.3g of its max' % (name, worst, SPAN_BITS,
                                                                                  err[-1] / sc[-1]))


# ------------------------------------------------------------------ 4. conv1 gathering its own input (CfgConv1XG)
VOL = (64, 48, 8)                  # unpadded X, Y, Z: patches are 25 x 25 x 1, so each lies in one z slice
PS = (25, 25, 1)


@pytest.fixture(scope='module')
def gather_setup(eng):
    """PW1 with conv1 on the device and a 3-modality volume whose z slice z is scaled by 2^-z (mean 0, so the
    normalisation (x - 0) / sigma keeps the scale): a sample's magnitude is chosen by the slice of its voxel."""
    import nnal_b200
    from tests.util import pad_imgs
    rs = np.random.RandomState(3)
    imgs = [(rs.randn(*VOL) * 30 * np.ldexp(1.0, -np.arange(VOL[2]))[None, None, :]).astype(np.float32) for _ in range(3)]
    padded = pad_imgs(imgs, PS)
    stats = np.array([[0., 30. + j] for j in range(3)])
    layers = O.pw1_layers(2)
    w = O.he_init_weights(layers, (25, 25, 3), 4, bias_scale=.1)
    model = nnal_b200.NN.create_PW1(2)
    model.set_weights(w)
    eng.set_model(model)
    eng.upload(7, padded)
    return padded, stats, w['conv1'][0], w['conv1'][1].ravel()


def gather_inds(n, grid, seed):
    """Voxel ids of n samples: sample s in slice (s // grid) mod 8 at random x, y (consecutive ids far apart); each of the
    eight corners of the unpadded volume takes the first free sample of its slice, where there is one."""
    X, Y, Z = VOL
    rs = np.random.RandomState(seed)
    z = (np.arange(n) // grid) % Z
    x, y = rs.randint(0, X, n), rs.randint(0, Y, n)
    used = set()
    for cx in (0, X - 1):
        for cy in (0, Y - 1):
            for cz in (0, Z - 1):
                free = [s for s in np.flatnonzero(z == cz) if s not in used]
                if free:
                    used.add(free[0])
                    x[free[0]], y[free[0]] = cx, cy
    return np.ravel_multi_index((x, y, z), VOL).astype(np.int64)


def gather_ref(padded, stats, inds, W, b, on_device=False):
    p = O.normalize_batch_eval(O.get_patches(padded, inds, PS), stats)
    return p, (torch_ref('fwd', p, W, b) if on_device else np_ref('fwd', p, W, b))


@pytest.mark.gpu
def test_conv1_gather_capped_grid(eng, gather_setup):
    """CfgConv1XG (NG = 3, NACC = 4: P = 8) on 2 and 3 CTAs, 16+ samples each, the eight volume corners included: float64
    get_patches -> normalize_batch_eval -> conv at 3e-5 per sample; bit-identical to the default grid; and with the float64
    normalisation (wt_flags = 8) bit-identical to the stand-alone x-im2col'd conv1 on the float64-normalised patches."""
    padded, stats, W, b = gather_setup
    p = all_plans()['CfgConv1XG']
    worst, most = 0., 0
    for grid in CAPS:
        per, ok = capped_regime(p, grid)
        assert ok, per
        most = max(most, max(per))
        inds = gather_inds(CAP_GROUPS, grid, grid)
        X, Y, Z = VOL
        corners = np.ravel_multi_index(np.meshgrid([0, X - 1], [0, Y - 1], [0, Z - 1], indexing='ij'), VOL).ravel()
        assert np.isin(corners, inds).all()
        patches, ref = gather_ref(padded, stats, inds, W, b)
        eng.debug_option('conv_grid', grid)
        try:
            got = eng.debug_conv1_gather(7, inds, stats)
            eng.debug_option('wt_flags', 8)
            exact = eng.debug_conv1_gather(7, inds, stats)
        finally:
            eng.debug_option('wt_flags', 0)
            eng.debug_option('conv_grid', 0)
        worst = max(worst, assert_per_sample(got, ref, 'fused gather on %d CTAs' % grid, 1, grid))
        assert np.array_equal(got, eng.debug_conv1_gather(7, inds, stats)), 'grid cap %d changed the result' % grid
        x16 = eng.debug_conv(patches.astype(np.float32), W, b, 5)
        diff = np.flatnonzero((exact != x16).reshape(len(inds), -1).any(1))
        assert not len(diff), 'float64-normalised fused gather on %d CTAs != x-im2col conv1 in samples %s' % (grid, diff)
    report('CfgConv1XG capped', most, worst)


@pytest.mark.gpu
def test_conv1_gather_full_grid(eng, gather_setup):
    """CfgConv1XG on the full grid: a production chunk of 16,384 voxels, 147, 148 and 149 voxels and one, against float64
    torch on the float64-normalised patches, 3e-5 per sample."""
    padded, stats, W, b = gather_setup
    worst, most = 0., 0
    for n in prod_sizes(all_plans()['CfgConv1XG'], 'fwd'):
        grid = min(n, SM_COUNT)
        most = max(most, max(groups_per_cta(n, grid)))
        inds = gather_inds(n, grid, n)
        _, ref = gather_ref(padded, stats, inds, W, b, on_device=True)
        worst = max(worst, assert_per_sample(eng.debug_conv1_gather(7, inds, stats), ref, 'fused gather n=%d' % n, 1, grid))
        del ref
    report('CfgConv1XG full grid', most, worst)
