"""Greedy block-form FI with a class cap on the device (``fi_classes``; csrc/fi_block.cu kept classes) against the float64
kept-class oracle (tests/fi_block_cls_oracle.py): host factors in kept form, in-place candidates through NNAL.CNN_query on
wide heads, bit-identity with the uncapped greedy when every class is kept, and the argument checks."""
from collections import OrderedDict

import numpy as np
import pytest

import oracle as O
from tests import fi_block_cls_oracle as FC
from tests.test_gpu_mc_multi import conv_net, fc_only_net, IN_SHAPE

pytestmark = pytest.mark.gpu

LOSS_RTOL = 1e-3          # a device pick may differ from the float64 greedy's only at a near-tie of the criterion


class Expr(object):
    def __init__(self, **pars):
        self.pars = pars


@pytest.fixture(scope='module')
def nb():
    import nnal_b200
    return nnal_b200


def _factors(c, n, d, seed):
    """Peaked Dirichlet posteriors [c,n] with one-hot columns and exact zeros, float32 features [n,d]."""
    rs = np.random.RandomState(seed)
    P = rs.dirichlet(np.ones(c) * 0.2, n).T
    for i in range(0, n, 17):
        P[:, i] = 0.
        P[i % c, i] = 1.
    for i in range(5, n, 11):
        if i % 17 == 0:
            continue
        P[np.argmax(P[:, i]), i] = 0.
        P[:, i] /= P[:, i].sum()
    return P.astype(np.float32), rs.randn(n, d).astype(np.float32)


def _check_trajectory(cls, p, U64, c, delta, sel, red, red_rtol=1e-4):
    """``sel`` is a greedy trajectory of the kept-class criterion (every pick within LOSS_RTOL of the best loss), every
    reduced objective matches the float64 value of its prefix, and the last matches the float64 greedy's.  U64 [d,n]."""
    rep = FC.greedy_fi_block_cls_replay(cls, p, U64, c, delta, sel)
    assert np.all(rep[:, 0] <= rep[:, 1] * (1 + LOSS_RTOL)), 'a pick is not a greedy choice'
    assert np.all(np.abs(red / rep[:, 2] - 1) < red_rtol), np.abs(red / rep[:, 2] - 1).max()
    if np.all(rep[:, 0] <= rep[:, 1]):
        red_o = rep[-1, 2]
    else:
        red_o = FC.greedy_fi_block_cls(cls, p, U64, c, delta, len(sel))[2][-1]
    assert abs(red[-1] / red_o - 1) < 1e-3


@pytest.mark.parametrize('c', [3, 10, 32, 48, 100, 1000])
@pytest.mark.parametrize('r', [2, 5, 10, 32])
def test_given_factors(nb, c, r):
    n, d, k, delta = 300, 64, 20, 1e-3
    post, U = _factors(c, n, d, 7 * c + r)
    cls, p = FC.top_classes(post, r)
    q = cls.shape[1]
    eng = nb.get_engine()
    eng.fi_block_set_factors_cls(cls, p, U, c)
    sel, obj, red = eng.fi_block_greedy(k, delta)
    assert len(sel) == k and len(np.unique(sel)) == k
    _check_trajectory(cls, p, U.T.astype(np.float64), c, delta, sel, red)
    s = np.arange(1, k + 1)
    assert np.all(np.abs(obj - ((c * (d + 1) - s * (q - 1)) / delta + red)) <= 1e-12 * np.abs(obj))
    sel2, obj2, red2 = eng.fi_block_greedy(k, delta)
    assert np.array_equal(sel, sel2) and np.array_equal(red, red2) and np.array_equal(obj, obj2)


def _model(nb, layers, w, in_shape):
    m = nb.NN.CNN(in_shape, OrderedDict(layers), feature_layer=len(layers) - 2)
    m.set_weights(w)
    return m


def _query_check(nb, model, x, r, B, k):
    """NNAL.CNN_query(..., 'fi') with fi_classes = r: a greedy trajectory of the kept-class oracle on the device's own
    candidates, float32 posteriors and features; the device's kept classes are the oracle's; in-place candidates and
    the same kept classes handed over from the host give bit-identical results."""
    n = len(x)
    expr = Expr(k=k, B=B, lambda_=0., batch_size=128, fi_mode='block-greedy', fi_classes=r, fi_diag_load=1e-4)
    expr.pool_images = x
    q = nb.NNAL.CNN_query(model, expr, np.arange(n), 'fi', None)
    assert len(q) == min(k, B, n) and len(np.unique(q)) == len(q)
    q2, obj, red = nb.fi.query_whole_block(model, expr, np.arange(n), None, return_objective='reduced')
    assert np.array_equal(q, q2)
    eng = nb.get_engine()
    cand = eng.pool_topk(B) if B < n else np.arange(n)
    post = eng.pool_posteriors()[:, cand]
    F = eng.pool_feature_rows(cand)
    cls, p = eng.pool_top_classes(cand, r)
    cls_o, p_o = FC.top_classes(post, r)
    assert np.array_equal(cls, cls_o) and np.array_equal(p, p_o)
    pos = {int(v): i for i, v in enumerate(cand)}
    sel = np.array([pos[int(v)] for v in q])
    _check_trajectory(cls_o, p_o, F.T.astype(np.float64), eng.n_class, 1e-4, sel, red, red_rtol=1e-3)
    eng.fi_block_set_factors_cls(cls, p, F, eng.n_class)
    sel_h, obj_h, red_h = eng.fi_block_greedy(k, 1e-4)
    assert np.array_equal(sel_h, sel) and np.array_equal(obj_h, obj) and np.array_equal(red_h, red)


@pytest.mark.parametrize('c', [100, 257, 1000])
def test_query_wide_head(nb, c):
    layers = conv_net(c)
    w = O.he_init_weights(layers, IN_SHAPE, 5 + c, bias_scale=0.3)
    w[layers[-1][0]] = (w[layers[-1][0]][0] * np.float32(3.), w[layers[-1][0]][1])
    x = np.random.RandomState(6 + c).randn(400, *IN_SHAPE).astype(np.float32)
    _query_check(nb, _model(nb, layers, w, IN_SHAPE), x, 10, 100, 10)


def test_query_21841_classes(nb):
    """ImageNet-21k width, every candidate (no pre-filter), 10 classes kept."""
    c = 21841
    layers = fc_only_net(c)
    w = O.he_init_weights(layers, IN_SHAPE, 21, bias_scale=0.3)
    w[layers[-1][0]] = (w[layers[-1][0]][0] * np.float32(3.), w[layers[-1][0]][1])
    x = np.random.RandomState(22).randn(300, *IN_SHAPE).astype(np.float32)
    _query_check(nb, _model(nb, layers, w, IN_SHAPE), x, 10, 300, 15)


def test_query_config1_shape_1000_classes(nb):
    """PW1 layer dict on 28x28x1 with a 1,000-class head, 2,000 images, B = 100, k = 10."""
    layers = O.pw1_layers(1000)
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    x = np.random.RandomState(0).rand(2000, 28, 28, 1).astype(np.float32)
    _query_check(nb, _model(nb, layers, w, (28, 28, 1)), x, 10, 100, 10)


def _small(nb, c, seed):
    from tests.test_gpu_parity import SMALL
    layers = [(nm, s) for nm, s in SMALL[:-1]] + [('fc3', [c, 'fc'])]
    w = O.he_init_weights(layers, (9, 7, 2), seed, bias_scale=0.1)
    return _model(nb, layers, w, (9, 7, 2))


@pytest.mark.parametrize('c', [3, 10, 32])
def test_cap_at_or_above_c_is_uncapped(nb, c):
    """fi_classes >= c keeps every class in order: the selection and objectives of the unset key, bit for bit."""
    model = _small(nb, c, 50 + c)
    x = np.random.RandomState(51).rand(400, 9, 7, 2).astype(np.float32)
    base = dict(k=20, B=150, lambda_=0., batch_size=128, fi_mode='block-greedy')
    expr = Expr(**base)
    expr.pool_images = x
    want = nb.fi.query_whole_block(model, expr, np.arange(400), None, return_objective='reduced')
    for r in sorted({c, 32}):
        expr = Expr(fi_classes=r, **base)
        expr.pool_images = x
        got = nb.fi.query_whole_block(model, expr, np.arange(400), None, return_objective='reduced')
        for a, b in zip(got, want):
            assert np.array_equal(a, b)


def test_cap_lifts_k_limit(nb):
    """c = 32, k = 200: the dense form refuses k (c-1) = 6,200; ten kept classes need k (10-1) = 1,800."""
    c, n, d, k, delta = 32, 600, 32, 200, 1e-3
    post, U = _factors(c, n, d, 9)
    eng = nb.get_engine()
    eng.fi_block_set_factors(post, U)
    with pytest.raises(nb._lib.NnalError, match='error 4'):
        eng.fi_block_greedy(k, delta)
    cls, p = FC.top_classes(post, 10)
    eng.fi_block_set_factors_cls(cls, p, U, c)
    sel, obj, red = eng.fi_block_greedy(k, delta)
    assert len(np.unique(sel)) == k and np.all(np.isfinite(red))
    _check_trajectory(cls, p, U.T.astype(np.float64), c, delta, sel[:40], red[:40])


def test_errors(nb):
    e = nb.Engine(0)
    post, U = _factors(100, 500, 8, 1)
    cls, p = FC.top_classes(post, 10)

    def usable():
        e.fi_block_set_factors_cls(cls[:50], p[:50], U[:50], 100)
        assert len(e.fi_block_greedy(5, 1e-3)[0]) == 5

    try:
        usable()
        for r in (1, 33):                                     # class cap out of range
            with pytest.raises(ValueError):
                e.fi_block_set_factors_cls(np.tile(np.arange(r), (5, 1)), np.ones((5, r)), U[:5], 100)
            usable()
        bad = cls.copy()
        bad[3, [2, 3]] = bad[3, [3, 2]]                       # ids not ascending
        with pytest.raises(ValueError):
            e.fi_block_set_factors_cls(bad, p, U, 100)
        usable()
        bad = cls.copy()
        bad[7, -1] = 100                                      # id outside 0..c-1
        with pytest.raises(ValueError):
            e.fi_block_set_factors_cls(bad, p, U, 100)
        usable()
        e.fi_block_set_factors_cls(cls, p, U, 100)
        with pytest.raises(nb._lib.NnalError, match='error 4'):
            e.fi_block_greedy(456, 1e-3)                      # k (10-1) = 4,104 > 4,096
        usable()
        layers = conv_net(100)
        w = O.he_init_weights(layers, IN_SHAPE, 3, bias_scale=0.3)
        e.set_model(_model(nb, layers, w, IN_SHAPE))
        e.pool_begin(60, 1)
        e.pool_eval_images(np.random.RandomState(4).randn(60, *IN_SHAPE).astype(np.float32), 0)
        for r in (0, 1, 33):
            with pytest.raises(ValueError):
                e.fi_block_set_candidates_cls(None, r)
            with pytest.raises(ValueError):
                e.pool_top_classes(np.arange(5), r)
        with pytest.raises(nb._lib.NnalError, match='error 4'):
            e.fi_block_set_candidates(None)                   # no cap: c > 32 is still refused
        e.fi_block_set_candidates_cls(None, 10)
        assert len(e.fi_block_greedy(5, 1e-3)[0]) == 5
    finally:
        e.close()
    model = _small(nb, 5, 60)
    expr = Expr(k=5, B=50, lambda_=0., batch_size=64, fi_mode='block-greedy', fi_layers=2, fi_classes=3)
    expr.pool_images = np.random.RandomState(61).rand(80, 9, 7, 2).astype(np.float32)
    with pytest.raises(ValueError):
        nb.NNAL.CNN_query(model, expr, np.arange(80), 'fi', None)
    expr.pars.pop('fi_layers')
    assert len(nb.NNAL.CNN_query(model, expr, np.arange(80), 'fi', None)) == 5
