"""Multi-class MC-dropout and committee scorers on the device (NNAL.CNN_query 'MC-entropy', 'BALD', 'ensemble', 'QBC-JS';
score kinds 12 / 13; nnal_pool_mc_read_classes) against the float64 reference of tests/mc_multi_oracle.py."""
from collections import OrderedDict

import numpy as np
import pytest

import oracle as O
from tests import mc_multi_oracle as MM

pytestmark = pytest.mark.gpu

POST_TOL = 1e-4
ENT_TOL = 1e-3
SCORE_TOL = 1e-3


class Expr(object):
    def __init__(self, **pars):
        self.pars = pars


@pytest.fixture(scope='module')
def nb():
    import nnal_b200
    return nnal_b200


IN_SHAPE = (6, 6, 2)


def conv_net(c):
    """conv1 (Cin = 2) runs on CUDA cores; fc1 (72) and fc2 (136) on tensor cores."""
    return [('conv1', [8, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [72, 'fc']), ('fc2', [136, 'fc']),
            ('fc3', [c, 'fc'])]


def fc_only_net(c):
    """No trunk: the fp32 input is split into tensor-core planes once per chunk before the T tail passes."""
    return [('fc1', [64, 'fc']), ('fc2', [136, 'fc']), ('fc3', [c, 'fc'])]


def _model(nb, layers, w, sites, keep, in_shape=IN_SHAPE):
    m = nb.NN.CNN(in_shape, OrderedDict(layers), feature_layer=len(layers) - 2, dropout=[sites, keep])
    m.set_weights(w)
    return m


def _case(layers, n, seed, in_shape=IN_SHAPE):
    w = O.he_init_weights(layers, in_shape, seed, bias_scale=0.3)
    x = np.random.RandomState(seed + 1).randn(n, *in_shape).astype(np.float32)
    return w, x


def _mc_pass(eng, x, T, keep, sites, pos0=0):
    eng.pool_mc_config(T, keep, sites, pos0=pos0)
    try:
        eng.pool_begin(len(x))
        eng.pool_eval_images(x, 0)
    finally:
        eng.pool_mc_config(0, 1., [])


@pytest.mark.parametrize('net', ['conv', 'fc_only'])
@pytest.mark.parametrize('c', [3, 10, 32])
def test_class_means_match_oracle(nb, c, net):
    layers = conv_net(c) if net == 'conv' else fc_only_net(c)
    sites = [len(layers) - 3, len(layers) - 2, len(layers) - 1]
    w, x = _case(layers, 700, 10 + c)
    keep, T, seed = 0.7, 4, 0xabc0123 + c
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, w, sites, keep), None)
    tc = [eng.layer_info(i)[2] for i in range(len(layers))]
    assert tc == ([0, 0, 1, 1, 0] if net == 'conv' else [1, 1, 0])
    eng.set_dropout_seed(seed, first_pass=5)
    _mc_pass(eng, x, T, keep, sites)
    av_post, av_ent = eng.pool_mc_class_means()
    passes = MM.mc_passes(layers, w, x, np.arange(len(x)), T, keep, sites, seed, 5)
    want_post, want_ent = MM.class_running_means(passes)
    assert av_post.shape == (c, len(x))
    assert np.abs(av_post - want_post).max() < POST_TOL
    assert np.abs(av_ent - want_ent).max() < ENT_TOL
    assert np.abs(passes[-1] - MM.mc_passes(layers, w, x, np.arange(len(x)), 1, 1., sites, seed, 0)[0]).max() > 1e-2
    for kind in (12, 13):
        eng.pool_score(kind)
        assert np.abs(eng.pool_scores() - MM.scores(want_post, want_ent, kind)).max() < SCORE_TOL


def _pw1_trunk(layers, w, x):
    """Float64 input of fc1 of the PW1 layer dict: the torch float64 forward up to max2, read through an identity FC
    layer (exact: the pooled ReLU outputs are non-negative)."""
    from tests.test_gpu_scale import _torch64
    d = 7 * 7 * 96
    trunk = layers[:6] + [('id', [d, 'fc'])]
    wt = {k: w[k] for k, spec in layers[:6] if spec[1] == 'conv'}
    wt['id'] = (np.eye(d, dtype=np.float32), np.zeros((d, 1), dtype=np.float32))
    return _torch64(trunk, wt, 6)(x)['feature_layer']


def test_config1_shape(nb):
    """PW1 layer dict on 28x28x1, c = 10, 2,000 images, T = 10, dropout on fc1, fc2 and the logits: class means of 256
    samples spread over the pool against float64."""
    layers = O.pw1_layers(10)
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    x = np.random.RandomState(0).rand(2000, 28, 28, 1).astype(np.float32)
    sites, keep, T, seed = [6, 7, 8], 0.5, 10, 77
    model = nb.NN.CNN((28, 28, 1), OrderedDict(layers), feature_layer=len(layers) - 2, dropout=[sites, keep])
    model.set_weights(w)
    eng = nb.get_engine()
    eng.set_dropout_seed(seed)
    expr = Expr(k=10, MC_iters=T)
    expr.pool_images = x
    q = nb.NNAL.CNN_query(model, expr, np.arange(2000), 'BALD', None)
    assert len(q) == 10 and len(np.unique(q)) == 10
    av_post, av_ent = eng.pool_mc_class_means()
    sub = np.random.RandomState(1).choice(2000, 256, replace=False)
    sub = np.union1d(sub, q)
    passes = MM.mc_passes(layers, w, None, sub, T, keep, sites, seed, 0, h=_pw1_trunk(layers, w, x[sub]))
    want_post, want_ent = MM.class_running_means(passes)
    assert np.abs(av_post[:, sub] - want_post).max() < POST_TOL
    assert np.abs(av_ent[sub] - want_ent).max() < ENT_TOL
    # every pick is at least as good as the subset's 10th best up to the tolerance
    s = MM.scores(want_post, want_ent, 13)
    pos = {int(v): i for i, v in enumerate(sub)}
    assert np.all(s[[pos[int(v)] for v in q]] <= np.sort(s)[9] + SCORE_TOL)


def _check_selection(q, scores, k, tol):
    kth = np.sort(scores)[k - 1]
    assert len(q) == k and len(np.unique(q)) == k
    assert np.all(scores[q] <= kth + tol)
    assert np.all(np.isin(np.where(scores < kth - tol)[0], q))


@pytest.mark.parametrize('method', ['MC-entropy', 'BALD', 'ensemble', 'QBC-JS'])
@pytest.mark.parametrize('c', [2, 10])
def test_query_selections(nb, method, c, tmp_path):
    layers = conv_net(c)
    sites, keep, T, k, seed = [2, 3, 4], 0.6, 6, 25, 4242
    w, x = _case(layers, 600, 60 + c)
    model = _model(nb, layers, w, sites, keep)
    expr = Expr(k=k, MC_iters=T)
    expr.pool_images = x
    eng = nb.get_engine()
    eng.set_dropout_seed(seed, first_pass=2)
    if method in ('MC-entropy', 'BALD'):
        q = nb.NNAL.CNN_query(model, expr, np.arange(len(x)), method, None)
        _, want_post, want_ent, scores = MM.query_mc_whole(layers, w, x, k, T, keep, sites, seed, method, first_pass=2)
    else:
        members = [O.he_init_weights(layers, IN_SHAPE, 90 + 7 * i + c, bias_scale=0.3) for i in range(3)]
        holder = nb.NN.CNN(IN_SHAPE, OrderedDict(layers), feature_layer=len(layers) - 2)
        expr.pretrained_paths = []
        for i, m in enumerate(members):
            holder.set_weights(m)
            expr.pretrained_paths.append(str(tmp_path / ('member%d.npz' % i)))
            holder.save_weights(expr.pretrained_paths[-1])
        expr.model_holder = holder
        q = nb.NNAL.CNN_query(None, expr, np.arange(len(x)), method, None)
        _, want_post, want_ent, scores = MM.query_committee_whole(layers, members, x, k, method)
    av_post, av_ent = eng.pool_mc_class_means()
    assert np.abs(av_post - want_post).max() < POST_TOL and np.abs(av_ent - want_ent).max() < ENT_TOL
    _check_selection(q, scores, k, SCORE_TOL)


def test_masks_independent_of_chunking_and_sharding(nb):
    """Bit-equal class means whether the pool is evaluated whole, in chunks of 100, or as two shards with their pos0."""
    layers = conv_net(10)
    sites, keep, T, seed = [2, 3, 4], 0.7, 3, 7
    w, x = _case(layers, 333, 90)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, w, sites, keep), None)

    def run(lo, hi):
        eng.set_dropout_seed(seed)
        _mc_pass(eng, x[lo:hi], T, keep, sites, pos0=lo)
        return eng.pool_mc_class_means()
    whole = run(0, len(x))
    eng.debug_option('chunk', 100)
    try:
        chunked = run(0, len(x))
    finally:
        eng.debug_option('chunk', 0)
    assert np.array_equal(whole[0], chunked[0]) and np.array_equal(whole[1], chunked[1])
    a, b = run(0, 150), run(150, len(x))
    assert np.array_equal(np.concatenate([a[0], b[0]], axis=1), whole[0])
    assert np.array_equal(np.concatenate([a[1], b[1]]), whole[1])


def test_binary_kinds_agree(nb):
    """c = 2: kinds 12 / 13 select what kinds 10 / 11 select, from the same binary running means."""
    layers = conv_net(2)
    sites, keep, T, seed, k = [2, 3, 4], 0.6, 5, 99, 40
    w, x = _case(layers, 900, 5)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, w, sites, keep), None)
    eng.set_dropout_seed(seed)
    _mc_pass(eng, x, T, keep, sites)
    sel = {}
    for kind in (10, 11, 12, 13):
        eng.pool_score(kind)
        sel[kind] = (eng.pool_topk(k), eng.pool_scores())
    assert np.array_equal(sel[10][0], sel[12][0])
    assert np.array_equal(sel[11][0], sel[13][0]) and np.array_equal(sel[11][1], sel[13][1])
    av1, ent = eng.pool_mc_means()
    av_post, av_ent = eng.pool_mc_class_means()
    assert np.array_equal(av_post[1], av1) and np.array_equal(av_post[0], 1 - av1) and np.array_equal(av_ent, ent)


def test_errors(nb):
    e = nb.Engine(0)
    try:
        layers = conv_net(3)
        w, x = _case(layers, 50, 3)
        e.set_model(_model(nb, layers, w, [2, 3, 4], 0.5))
        e.pool_begin(len(x))
        e.pool_eval_images(x, 0)
        for kind in (12, 13):
            with pytest.raises(nb._lib.NnalError, match='error 3'):        # NNAL_ERR_STATE: no MC or committee pass
                e.pool_score(kind)
        _mc_pass(e, x, 2, 0.5, [2, 3, 4])
        e.pool_score(12)
        for kind in (10, 11):
            with pytest.raises(ValueError):                                # the binary kinds need c = 2
                e.pool_score(kind)
        with pytest.raises(ValueError):
            e.pool_mc_means()                                              # binary contract
        e.set_tensor_cores(False)
        try:
            with pytest.raises(nb._lib.NnalError, match='error 4'):        # FC tail off the tensor cores
                e.pool_mc_config(2, 0.5, [2, 3, 4])
        finally:
            e.set_tensor_cores(True)
        narrow = [('conv1', [8, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [60, 'fc']), ('fc2', [3, 'fc'])]
        wn, _ = _case(narrow, 1, 4)
        e.set_model(_model(nb, narrow, wn, [2, 3], 0.5))
        assert e.layer_info(2)[2] == 0
        with pytest.raises(nb._lib.NnalError, match='error 4'):
            e.pool_mc_config(2, 0.5, [2, 3])
        wide = conv_net(33)
        ww, _ = _case(wide, 1, 5)
        e.set_model(_model(nb, wide, ww, [2, 3, 4], 0.5))
        with pytest.raises(nb._lib.NnalError, match='error 4'):
            e.pool_mc_config(2, 0.5, [2, 3, 4])
        e.pool_begin(10)
        with pytest.raises(nb._lib.NnalError, match='error 4'):
            e.pool_ensemble_accumulate(0)
    finally:
        e.close()
