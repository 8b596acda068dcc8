"""Greedy multi-class FI selection in block form on the device (csrc/fi_block.cu, NNAL.CNN_query fi_mode='block-greedy')
against the float64 oracle (tests/fi_block_oracle.py: greedy_fi_block, greedy_fi_block_replay)."""
from collections import OrderedDict

import numpy as np
import pytest

import oracle as O
from tests import fi_block_oracle as FB
from tests.util import assert_topk_equivalent

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
    """Dirichlet posteriors [c,n] with one-hot columns and exact zeros, float32 features [n,d]."""
    rs = np.random.RandomState(seed)
    P = rs.dirichlet(np.ones(c) * 0.5, n).T
    for i in range(0, n, 17):
        P[:, i] = 0.
        P[i % c, i] = 1.
    for i in range(5, n, 11):
        P[rs.randint(c), i] = 0.
        P[:, i] /= P[:, i].sum()
    U = rs.randn(n, d).astype(np.float32)
    return P.astype(np.float32), U


def _check_trajectory(post64, U64, delta, sel, red, red_rtol=1e-4):
    """``sel`` is a greedy trajectory (every pick within LOSS_RTOL of the best loss), every reported reduced objective
    matches the float64 value of its prefix, and the final one matches the float64 greedy's.  post64 [c,n], U64 [d,n]."""
    rep = FB.greedy_fi_block_replay(post64, U64, delta, sel)
    assert np.all(rep[:, 0] <= rep[:, 1] * (1 + LOSS_RTOL)), 'a pick is not a greedy choice'
    assert np.all(np.abs(red / rep[:, 2] - 1) < red_rtol), np.abs(red / rep[:, 2] - 1).max()
    if np.all(rep[:, 0] <= rep[:, 1]):
        red_o = rep[-1, 2]                    # every pick is the float64 greedy's own
    else:
        red_o = FB.greedy_fi_block(post64, U64, delta, len(sel))[2][-1]
    assert abs(red[-1] / red_o - 1) < 1e-3


GRID = [(n, d, k) for (n, d, k) in [(300, 64, 40), (1000, 256, 25), (37, 20, 37), (500, 30, 170)]]


@pytest.mark.parametrize('c', [2, 3, 5, 10, 17])
@pytest.mark.parametrize('n,d,k', GRID)
def test_given_factors(nb, c, n, d, k):
    if k * (c - 1) > 4096:
        pytest.skip('k (c-1) > 4096')
    delta = 1e-3
    post, U = _factors(c, n, d, 100 * c + n)
    eng = nb.get_engine()
    eng.fi_block_set_factors(post, U)
    sel, obj, red = eng.fi_block_greedy(k, delta)
    assert len(sel) == min(k, n) and len(np.unique(sel)) == len(sel)
    _check_trajectory(post.astype(np.float64), U.T.astype(np.float64), delta, sel, red)
    s = np.arange(1, len(sel) + 1)
    D = c * (d + 1)
    assert np.all(np.abs(obj - ((D - s * (c - 1)) / delta + red)) <= 1e-12 * np.abs(obj))
    sel2, obj2, red2 = eng.fi_block_greedy(k, delta)
    assert np.array_equal(sel, sel2) and np.array_equal(red, red2) and np.array_equal(obj, obj2)


def test_binary_matches_fi_path(nb):
    """c = 2: the block greedy and the binary factored greedy (nnal_fi_greedy, one layer) answer the same question."""
    n, d, k, delta = 600, 48, 30, 1e-4
    post, U = _factors(2, n, d, 7)
    p64 = post.astype(np.float64)
    p1 = p64[1] / (p64[0] + p64[1])
    eng = nb.get_engine()
    eng.fi_block_set_factors(post, U)
    sel_b, _, red_b = eng.fi_block_greedy(k, delta)
    eng.fi_set_factors(p1, U)
    sel_1, _, red_1 = eng.fi_greedy(k, delta)
    assert np.all(np.abs(red_b / red_1 - 1) < 1e-5)
    U64 = U.T.astype(np.float64)
    for sel in (sel_b, sel_1):
        rep = FB.greedy_fi_block_replay(p64, U64, delta, sel)
        assert np.all(rep[:, 0] <= rep[:, 1] * (1 + LOSS_RTOL))


def _small(nb, c, seed):
    from tests.test_gpu_parity import SMALL
    layers = [(nm, s) for nm, s in SMALL[:-1]] + [('fc3', [c, 'fc'])]
    w = O.he_init_weights(layers, (9, 7, 2), seed, bias_scale=0.1)
    model = nb.NN.CNN((9, 7, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)
    return layers, w, model


def test_in_place_equals_host_factors(nb):
    """Candidates indexed in the pool pass give the same selection and bit-identical objectives as the same posteriors and
    features handed over from the host."""
    from nnal_b200.NNAL import _posteriors_on_device
    layers, w, model = _small(nb, 5, 21)
    x = np.random.RandomState(22).rand(400, 9, 7, 2).astype(np.float32)
    expr = Expr(k=20, B=100, lambda_=0., batch_size=128)
    expr.pool_images = x
    eng, _, _ = _posteriors_on_device(model, expr, np.arange(400), None, keep=1)
    cand = np.random.RandomState(23).choice(400, 150, replace=False).astype(np.int64)
    eng.fi_block_set_candidates(cand)
    sel, obj, red = eng.fi_block_greedy(20, 1e-5)
    post = eng.pool_posteriors()[:, cand]
    F = eng.pool_feature_rows(cand)
    eng.fi_block_set_factors(post, F)
    sel2, obj2, red2 = eng.fi_block_greedy(20, 1e-5)
    assert np.array_equal(sel, sel2) and np.array_equal(red, red2) and np.array_equal(obj, obj2)


def _api_check(nb, expr, model, n, post64, feat64, B, k):
    """(1) the device's candidates are a valid entropy top-B; (2) on those candidates the device's selection is a greedy
    trajectory of the float64 criterion and its final objective matches the float64 greedy's."""
    q = nb.NNAL.CNN_query(model, expr, np.arange(n), 'fi', None)
    assert len(q) == min(k, B, n) and len(np.unique(q)) == len(q)
    eng = nb.get_engine()
    pp = np.where(post64 == 0, 1e-8, post64)
    score = np.sum(pp * np.log(pp), axis=0)
    if B < n:
        cand = eng.pool_topk(B)
        assert_topk_equivalent(cand, score, B, 1e-3 * np.abs(score).max())
    else:
        cand = np.arange(n)
    pos = {int(v): i for i, v in enumerate(cand)}
    sel = np.array([pos[int(v)] for v in q])
    _, _, red = nb.fi.query_whole_block(model, expr, np.arange(n), None, return_objective='reduced')
    _check_trajectory(post64[:, cand], feat64[:, cand], float(expr.pars.get('fi_diag_load', 1e-5)), sel, red, red_rtol=1e-3)


@pytest.mark.parametrize('c,B', [(3, 100), (5, 100), (5, 1000)])
def test_api_small_net(nb, c, B):
    layers, w, model = _small(nb, c, 30 + c)
    x = np.random.RandomState(31).rand(400, 9, 7, 2).astype(np.float32)
    expr = Expr(k=20, B=B, lambda_=0., batch_size=128, fi_mode='block-greedy')
    expr.pool_images = x
    r = O.forward(layers, w, x, feature_layer=len(layers) - 2)
    _api_check(nb, expr, model, 400, r['posteriors'], r['feature_layer'], B, 20)


def test_api_config1_shape(nb):
    """PW1 layer dict on 28x28x1, c = 10, 2,000 images, B = 100, k = 10."""
    from tests.test_gpu_scale import _torch64
    layers = O.pw1_layers(10)
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    x = np.random.RandomState(0).rand(2000, 28, 28, 1).astype(np.float32)
    model = nb.NN.CNN((28, 28, 1), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)
    r = _torch64(layers, w, len(layers) - 2)(x)
    expr = Expr(k=10, B=100, lambda_=0., batch_size=500, fi_mode='block-greedy')
    expr.pool_images = x
    _api_check(nb, expr, model, 2000, r['posteriors'], r['feature_layer'], 100, 10)


def test_errors(nb):
    e = nb.Engine(0)
    try:
        with pytest.raises(nb._lib.NnalError):
            e.fi_block_greedy(5, 1e-3)                       # no candidates yet
        post, U = _factors(3, 3000, 8, 1)
        e.fi_block_set_factors(post, U)
        with pytest.raises(nb._lib.NnalError):
            e.fi_block_greedy(2049, 1e-3)                    # k (c-1) = 4098
        post33, U33 = _factors(33, 10, 4, 2)
        with pytest.raises(nb._lib.NnalError):
            e.fi_block_set_factors(post33, U33)
        with pytest.raises(ValueError):
            e.fi_block_set_factors(post[:, :10], U[:9])
        _, _, model = _small(nb, 3, 40)
        e.set_model(model)
        e.pool_begin(50, 0)
        e.pool_eval_images(np.random.RandomState(3).rand(50, 9, 7, 2).astype(np.float32), 0)
        with pytest.raises(nb._lib.NnalError):
            e.fi_block_set_candidates(None)                  # the pool pass kept no features
    finally:
        e.close()
