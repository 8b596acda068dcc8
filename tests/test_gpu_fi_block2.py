"""Greedy multi-class FI selection over the last two FC layers in block form on the device (csrc/fi_block.cu, n_layers = 2;
NNAL.CNN_query fi_mode='block-greedy', fi_layers=2) against the float64 oracle (tests/fi_block2_oracle.py)."""
from collections import OrderedDict

import numpy as np
import pytest

import oracle as O
from tests import fi_block2_oracle as FB2
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


def _factors2(c, n, d, dp, seed):
    """Dirichlet posteriors [c,n] with one-hot columns and exact zeros; ReLU-like float32 features U [n,d] (with zeros),
    previous activations A [n,dp], last-layer weights W [c,d]."""
    rs = np.random.RandomState(seed)
    P = rs.dirichlet(np.ones(c) * 0.5, n).T
    for i in range(0, n, 13):
        P[:, i] = 0.
        P[i % c, i] = 1.
    for i in range(5, n, 11):
        P[rs.randint(c), i] = 0.
        P[:, i] /= P[:, i].sum()
    U = np.maximum(rs.randn(n, d) - 0.2, 0).astype(np.float32)
    A = np.maximum(rs.randn(n, dp), 0).astype(np.float32)
    W = (rs.randn(c, d) / np.sqrt(d)).astype(np.float32)
    return P.astype(np.float32), U, A, W


def _check_trajectory(post, U, A, W, delta, sel, red, red_rtol=1e-4):
    """Every pick within LOSS_RTOL of the best float64 loss; every reported reduced objective within ``red_rtol`` of the
    float64 replay.  post [c,n], U [n,d], A [n,dp], W [c,d] (the float32 factors the device saw)."""
    f64 = lambda a: np.asarray(a, dtype=np.float64)
    K = FB2.two_layer_block_kernel(f64(post), f64(U).T, f64(A).T, f64(W))
    rep = FB2.greedy_block_kernel_replay(K, post.shape[0] - 1, delta, sel)
    assert np.all(rep[:, 0] <= rep[:, 1] * (1 + LOSS_RTOL)), 'a pick is not a greedy choice'
    err = np.abs(red / rep[:, 2] - 1)
    assert np.all(err < red_rtol), err.max()


# (c, n, d, d_prev, k): d != d_prev, d not a multiple of 32
CASES = [(c, 200, 45, 70, 20) for c in (2, 3, 5, 10)] + [(17, 160, 45, 70, 16), (32, 100, 45, 70, 10)] + \
        [(c, 120, 70, 33, 12) for c in (3, 10, 32)]


@pytest.mark.parametrize('c,n,d,dp,k', CASES)
def test_given_factors(nb, c, n, d, dp, k):
    delta = 1e-3
    post, U, A, W = _factors2(c, n, d, dp, 100 * c + n + d)
    eng = nb.get_engine()
    eng.fi_block_set_factors(post, U, A, W)
    sel, obj, red = eng.fi_block_greedy(k, delta)
    assert len(sel) == min(k, n) and len(np.unique(sel)) == len(sel)
    _check_trajectory(post, U, A, W, delta, sel, red)
    s = np.arange(1, len(sel) + 1)
    D = FB2.two_layer_dim(c, d, dp)
    assert np.all(np.abs(obj - ((D - s * (c - 1)) / delta + red)) <= 1e-12 * np.abs(obj))
    sel2, obj2, red2 = eng.fi_block_greedy(k, delta)
    assert np.array_equal(sel, sel2) and np.array_equal(red, red2) and np.array_equal(obj, obj2)


def test_binary_matches_fi_path(nb):
    """c = 2: the two-layer block greedy and the binary factored greedy (nnal_fi_greedy, two layers) answer the same question."""
    n, d, dp, k, delta = 600, 45, 70, 30, 1e-4
    post, U, A, W = _factors2(2, n, d, dp, 7)
    p64 = post.astype(np.float64)
    p1 = p64[1] / (p64[0] + p64[1])
    eng = nb.get_engine()
    eng.fi_block_set_factors(post, U, A, W)
    sel_b, _, red_b = eng.fi_block_greedy(k, delta)
    eng.fi_set_factors(p1, U, A, W)
    sel_1, _, red_1 = eng.fi_greedy(k, delta)
    assert np.all(np.abs(red_b / red_1 - 1) < 1e-5)
    for sel in (sel_b, sel_1):
        K = FB2.two_layer_block_kernel(p64, U.T.astype(np.float64), A.T.astype(np.float64), W.astype(np.float64))
        rep = FB2.greedy_block_kernel_replay(K, 1, delta, sel)
        assert np.all(rep[:, 0] <= rep[:, 1] * (1 + LOSS_RTOL))


def _small(nb, c, seed):
    from tests.test_gpu_parity import SMALL
    layers = [(nm, s) for nm, s in SMALL[:-1]] + [('fc3', [c, 'fc'])]
    w = O.he_init_weights(layers, (9, 7, 2), seed, bias_scale=0.1)
    model = nb.NN.CNN((9, 7, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)
    return layers, w, model


def test_in_place_equals_host_factors(nb):
    """Candidates indexed in the pool pass give the same selection and bit-identical objectives as the same posteriors,
    features, previous activations and weights handed over from the host."""
    from nnal_b200.NNAL import _posteriors_on_device
    layers, w, model = _small(nb, 5, 21)
    x = np.random.RandomState(22).rand(400, 9, 7, 2).astype(np.float32)
    expr = Expr(k=20, B=100, lambda_=0., batch_size=128)
    expr.pool_images = x
    eng, _, _ = _posteriors_on_device(model, expr, np.arange(400), None, keep=2)
    cand = np.random.RandomState(23).choice(400, 150, replace=False).astype(np.int64)
    eng.fi_block_set_candidates(cand, 2)
    sel, obj, red = eng.fi_block_greedy(20, 1e-5)
    post = eng.pool_posteriors()[:, cand]
    F = eng.pool_feature_rows(cand)
    Ap = eng.pool_prev_rows(cand)
    assert Ap.shape == (150, 40)
    eng.fi_block_set_factors(post, F, Ap, w['fc3'][0])
    sel2, obj2, red2 = eng.fi_block_greedy(20, 1e-5)
    assert np.array_equal(sel, sel2) and np.array_equal(red, red2) and np.array_equal(obj, obj2)
    _check_trajectory(post, F, Ap, w['fc3'][0], 1e-5, sel, red, red_rtol=1e-4)


def _api_check(nb, expr, model, n, post64, feat64, prev64, W, B, k):
    """(1) the device's candidates are a valid entropy top-B; (2) on those candidates the device's selection is a greedy
    trajectory of the float64 criterion on the float64 forward's factors, and its objectives match to 1e-3."""
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
    _check_trajectory(post64[:, cand], feat64[:, cand].T, prev64[:, cand].T, W, float(expr.pars.get('fi_diag_load', 1e-5)),
                      sel, red, red_rtol=1e-3)


@pytest.mark.parametrize('c,B', [(3, 100), (5, 100), (5, 1000)])
def test_api_small_net(nb, c, B):
    layers, w, model = _small(nb, c, 30 + c)
    x = np.random.RandomState(31).rand(400, 9, 7, 2).astype(np.float32)
    expr = Expr(k=20, B=B, lambda_=0., batch_size=128, fi_mode='block-greedy', fi_layers=2)
    expr.pool_images = x
    fl = len(layers) - 2
    r = O.forward(layers, w, x, feature_layer=fl, keep_acts=True)
    _api_check(nb, expr, model, 400, r['posteriors'], r['feature_layer'], r['acts'][fl]['in'], w['fc3'][0], B, 20)


def test_api_config1_shape(nb):
    """PW1 layer dict on 28x28x1, c = 10, 2,000 images, B = 100, k = 10, fi_layers = 2 (d = d_prev = 4096)."""
    from tests.test_gpu_scale import _torch64
    layers = O.pw1_layers(10)
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    x = np.random.RandomState(0).rand(2000, 28, 28, 1).astype(np.float32)
    fl = len(layers) - 2
    model = nb.NN.CNN((28, 28, 1), OrderedDict(layers), feature_layer=fl)
    model.set_weights(w)
    r = _torch64(layers, w, fl)(x)
    prev = _torch64(layers, w, fl - 1)(x)['feature_layer']
    expr = Expr(k=10, B=100, lambda_=0., batch_size=500, fi_mode='block-greedy', fi_layers=2)
    expr.pool_images = x
    _api_check(nb, expr, model, 2000, r['posteriors'], r['feature_layer'], prev, w['fc3'][0], 100, 10)


def test_errors(nb):
    e = nb.Engine(0)
    try:
        post, U, A, W = _factors2(3, 3000, 8, 6, 1)
        e.fi_block_set_factors(post, U, A, W)
        with pytest.raises(nb._lib.NnalError):
            e.fi_block_greedy(2049, 1e-3)                    # k (c-1) = 4098
        with pytest.raises(ValueError):
            e.fi_block_set_factors(post, U, A, None)         # both or neither
        with pytest.raises(ValueError):
            e.fi_block_set_factors(post, U, A[:10], W)       # A_prev rows
        with pytest.raises(ValueError):
            e.fi_block_set_factors(post, U, A, W[:, :5])     # w_last must be [c, d]
        # c = 2, 1.5 M candidates, k = 4096: the winners' columns would take 4096 * 1.5e6 * 5 * 8 B = 246 GB
        p2, U2, A2, W2 = _factors2(2, 1500000, 4, 4, 2)
        e.fi_block_set_factors(p2, U2, A2, W2)
        with pytest.raises(nb._lib.NnalError, match='GB'):
            e.fi_block_greedy(4096, 1e-3)
        del p2, U2, A2, W2
        _, _, model = _small(nb, 3, 40)
        e.set_model(model)
        e.pool_begin(50, 1)
        e.pool_eval_images(np.random.RandomState(3).rand(50, 9, 7, 2).astype(np.float32), 0)
        with pytest.raises(nb._lib.NnalError):
            e.fi_block_set_candidates(None, 2)               # the pool pass kept the feature layer only
        with pytest.raises(nb._lib.NnalError):
            e.pool_prev_rows(np.arange(5))
        e.fi_block_set_candidates(None, 1)                   # one layer still works from the same pass
        with pytest.raises(ValueError):
            e.fi_block_set_candidates(None, 3)               # NNAL_ERR_INVALID
    finally:
        e.close()
    layers, w, model = _small(nb, 3, 41)
    expr = Expr(k=5, B=50, lambda_=0., batch_size=64, fi_mode='block-greedy', fi_layers=3)
    expr.pool_images = np.random.RandomState(4).rand(60, 9, 7, 2).astype(np.float32)
    with pytest.raises(ValueError):
        nb.NNAL.CNN_query(model, expr, np.arange(60), 'fi', None)
