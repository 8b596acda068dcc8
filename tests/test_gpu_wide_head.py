"""Classifier heads with 64 or more classes (the wide head: FC GEMM for the logits, then wide_softmax_kernel) through every
whole-image query, against the float64 references oracle.forward and tests/mc_multi_oracle.py (both generic in c)."""
from collections import OrderedDict

import numpy as np
import pytest

import oracle as O
from tests import mc_multi_oracle as MM
from tests.test_gpu_mc_multi import Expr, conv_net, fc_only_net, IN_SHAPE
from tests.util import assert_topk_equivalent

pytestmark = pytest.mark.gpu

POST_TOL = 1e-4
SUM_TOL = 1e-5
ENT_TOL = 1e-3
SCORE_TOL = 1e-3


@pytest.fixture(scope='module')
def nb():
    import nnal_b200
    return nnal_b200


def _net(kind, c):
    return conv_net(c) if kind == 'conv' else fc_only_net(c)


def _case(layers, n, seed, in_shape=IN_SHAPE, scale=1.0):
    w = O.he_init_weights(layers, in_shape, seed, bias_scale=0.3)
    name = layers[-1][0]
    w[name] = (w[name][0] * np.float32(scale), w[name][1])
    x = np.random.RandomState(seed + 1).randn(n, *in_shape).astype(np.float32)
    return w, x


def _model(nb, layers, w, sites=None, keep=0.5, in_shape=IN_SHAPE):
    kw = {} if sites is None else dict(dropout=[sites, keep])
    m = nb.NN.CNN(in_shape, OrderedDict(layers), feature_layer=len(layers) - 2, **kw)
    m.set_weights(w)
    return m


def _posteriors(eng, x, pieces=None):
    eng.pool_begin(len(x))
    for lo, hi in (pieces or [(0, len(x))]):
        eng.pool_eval_images(x[lo:hi], lo)
    return eng.pool_posteriors()


@pytest.mark.parametrize('tc', [1, 0])
@pytest.mark.parametrize('net', ['conv', 'fc_only'])
@pytest.mark.parametrize('c', [64, 100, 101, 257, 1000])
def test_posteriors_match_float64(nb, c, net, tc):
    layers = _net(net, c)
    w, x = _case(layers, 500, 3 + c, scale=3.0)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, w), None)
    eng.set_tensor_cores(tc)
    try:
        assert eng.layer_info(len(layers) - 1)[2] == tc
        got = _posteriors(eng, x).astype(np.float64)
    finally:
        eng.set_tensor_cores(1)
    want = O.forward(layers, w, x)['posteriors']
    assert got.shape == (c, len(x))
    assert np.abs(got - want).max() < POST_TOL
    assert np.abs(got.sum(axis=0) - 1).max() < SUM_TOL


def test_no_class_limit(nb):
    """ImageNet-21k width: 21,841 classes, nothing in the softmax is sized by c."""
    c = 21841
    layers = fc_only_net(c)
    w, x = _case(layers, 300, 21, scale=3.0)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, w), None)
    assert eng.layer_info(len(layers) - 1)[2] == 1
    got = _posteriors(eng, x).astype(np.float64)
    want = O.forward(layers, w, x)['posteriors']
    assert np.abs(got - want).max() < POST_TOL
    assert np.abs(got.sum(axis=0) - 1).max() < SUM_TOL


def test_chunks_and_offsets_bit_equal(nb):
    """20,000 images (two 16,384-sample forward chunks) in one call, and in pieces at offsets that are not multiples of 32
    with lengths n mod 32 != 0: bit-equal posteriors."""
    c = 1000
    layers = conv_net(c)
    w, x = _case(layers, 20000, 8, scale=3.0)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, w), None)
    whole = _posteriors(eng, x)
    pieces = _posteriors(eng, x, [(0, 7), (7, 16391), (16391, 16400), (16400, 20000)])
    assert np.array_equal(whole, pieces)
    sub = np.random.RandomState(0).choice(len(x), 300, replace=False)
    assert np.abs(whole[:, sub] - O.forward(layers, w, x[sub])['posteriors']).max() < POST_TOL


def test_config1_shape(nb):
    """PW1 layer dict on 28x28x1 with fc3 = 1000, 2,000 images, conv trunk on the tensor cores: posteriors against float64,
    'entropy' and 'fi' (last-layer FI trace) selections."""
    from tests.test_gpu_scale import _torch64
    layers = O.pw1_layers(1000)
    w = O.he_init_weights(layers, (28, 28, 1), 1)
    x = np.random.RandomState(0).rand(2000, 28, 28, 1).astype(np.float32)
    model = _model(nb, layers, w, in_shape=(28, 28, 1))
    r = _torch64(layers, w, len(layers) - 2)(x)
    post, feat = r['posteriors'], r['feature_layer']
    expr = Expr(k=10, B=100, lambda_=0., batch_size=500)
    expr.pool_images = x
    q = nb.NNAL.CNN_query(model, expr, np.arange(2000), 'entropy', None)
    eng = nb.get_engine()
    got = eng.pool_posteriors().astype(np.float64)
    assert np.abs(got - post).max() < POST_TOL
    for i, (name, spec) in enumerate(layers):
        if spec[1] in ('conv', 'fc'):
            assert eng.layer_info(i)[2] != 0, '%s runs on CUDA cores' % name
    H = O.compute_entropy(post.copy())
    assert_topk_equivalent(q, -H, 10, 1e-3 * np.abs(H).max())
    q = nb.NNAL.CNN_query(model, expr, np.arange(2000), 'fi', None)
    tr = O.fi_trace_score(post, feat)
    assert_topk_equivalent(q, -tr, 10, 1e-3 * np.abs(tr).max())


@pytest.mark.parametrize('method', ['entropy', 'fi', 'rep-entropy', 'MC-entropy', 'BALD', 'ensemble', 'QBC-JS'])
@pytest.mark.parametrize('c', [100, 1000])
def test_query_selections(nb, c, method, tmp_path):
    layers = conv_net(c)
    sites, keep, T, k, B, seed = [2, 3, 4], 0.6, 5, 20, 80, 515
    w, x = _case(layers, 600, 40 + c, scale=3.0)
    model = _model(nb, layers, w, sites, keep)
    expr = Expr(k=k, B=B, lambda_=0., batch_size=128, MC_iters=T)
    expr.pool_images = x
    eng = nb.get_engine()
    pool = np.arange(len(x))
    if method == 'entropy':
        q = nb.NNAL.CNN_query(model, expr, pool, method, None)
        H = O.compute_entropy(O.forward(layers, w, x)['posteriors'])
        assert_topk_equivalent(q, -H, k, 1e-4)
    elif method == 'fi':
        q = nb.NNAL.CNN_query(model, expr, pool, method, None)
        r = O.forward(layers, w, x, feature_layer=len(layers) - 2)
        tr = O.fi_trace_score(r['posteriors'], r['feature_layer'])
        assert_topk_equivalent(q, -tr, k, 1e-4 * np.abs(tr).max())
    elif method == 'rep-entropy':
        q = nb.NNAL.CNN_query(model, expr, pool, method, None)
        qo, det = O.query_rep_entropy_whole(layers, w, x, k, B)
        assert len(q) == k and len(np.unique(q)) == k and np.all(np.isin(q, det['sel']))
        pos = {int(v): i for i, v in enumerate(det['sel'])}
        rep = O.facility_location_replay(det['sims'], [pos[int(v)] for v in q])
        assert np.all(rep[:, 0] >= rep[:, 1] - 1e-4 * np.abs(rep[:, 1])), 'picked a column clearly worse than the best'
    elif method in ('MC-entropy', 'BALD'):
        eng.set_dropout_seed(seed, first_pass=2)
        q = nb.NNAL.CNN_query(model, expr, pool, method, None)
        _, want_post, want_ent, scores = MM.query_mc_whole(layers, w, x, k, T, keep, sites, seed, method, first_pass=2)
        av_post, av_ent = eng.pool_mc_class_means()
        assert np.abs(av_post - want_post).max() < POST_TOL and np.abs(av_ent - want_ent).max() < ENT_TOL
        assert_topk_equivalent(q, scores, k, SCORE_TOL)
    else:
        members = [_case(layers, 1, 90 + 7 * i + c, scale=3.0)[0] for i in range(3)]
        holder = nb.NN.CNN(IN_SHAPE, OrderedDict(layers), feature_layer=len(layers) - 2)
        expr.pretrained_paths = []
        for i, m in enumerate(members):
            holder.set_weights(m)
            expr.pretrained_paths.append(str(tmp_path / ('member%d.npz' % i)))
            holder.save_weights(expr.pretrained_paths[-1])
        expr.model_holder = holder
        q = nb.NNAL.CNN_query(None, expr, pool, method, None)
        _, want_post, want_ent, scores = MM.query_committee_whole(layers, members, x, k, method)
        av_post, av_ent = eng.pool_mc_class_means()
        assert np.abs(av_post - want_post).max() < POST_TOL and np.abs(av_ent - want_ent).max() < ENT_TOL
        assert_topk_equivalent(q, scores, k, SCORE_TOL)


def _mc_pass(eng, x, T, keep, sites, pos0=0, offset_pieces=None):
    eng.pool_mc_config(T, keep, sites, pos0=pos0)
    try:
        eng.pool_begin(len(x))
        for lo, hi in (offset_pieces or [(0, len(x))]):
            eng.pool_eval_images(x[lo:hi], lo)
    finally:
        eng.pool_mc_config(0, 1., [])
    return eng.pool_mc_class_means()


@pytest.mark.parametrize('logits_site', [True, False])
@pytest.mark.parametrize('c', [64, 257, 1000])
def test_mc_class_means(nb, c, logits_site):
    layers = conv_net(c)
    sites = [2, 3, 4] if logits_site else [2, 3]
    keep, T, seed = 0.7, 4, 0x5eed + c
    w, x = _case(layers, 700, 70 + c, scale=3.0)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, w, sites, keep), None)
    assert eng.layer_info(len(layers) - 1)[2] == 1

    def run(lo, hi, pieces=None):
        eng.set_dropout_seed(seed, first_pass=3)
        return _mc_pass(eng, x[lo:hi], T, keep, sites, pos0=lo, offset_pieces=pieces)
    av_post, av_ent = run(0, len(x))
    passes = MM.mc_passes(layers, w, x, np.arange(len(x)), T, keep, sites, seed, 3)
    want_post, want_ent = MM.class_running_means(passes)
    assert av_post.shape == (c, len(x))
    assert np.abs(av_post - want_post).max() < POST_TOL
    assert np.abs(av_ent - want_ent).max() < ENT_TOL
    again = run(0, len(x), [(0, 333), (333, len(x))])
    assert np.array_equal(again[0], av_post) and np.array_equal(again[1], av_ent)
    a, b = run(0, 350), run(350, len(x))
    assert np.array_equal(np.concatenate([a[0], b[0]], axis=1), av_post)
    assert np.array_equal(np.concatenate([a[1], b[1]]), av_ent)


SDP_NET = [('conv1', [8, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('conv2', [12, 'conv', [5, 3]]),
           ('fc1', [72, 'fc']), ('fc2', [64, 'fc'])]


@pytest.mark.parametrize('c', [101, 104])
def test_sdp_path(nb, c):
    """fi_mode = 'sdp': one backward pass per class through the wide head.  c = 101: the last layer's dz.W on the FP32
    path (K = c not a multiple of 8); c = 104: on the tensor cores."""
    from tests.test_gpu_sdp import _assert_shrunk_close, OBJ_RTOL
    layers = SDP_NET + [('fc3', [c, 'fc'])]
    in_shape = (11, 8, 3)
    rs = np.random.RandomState(c)
    x = rs.rand(300, *in_shape).astype(np.float32)
    w = O.he_init_weights(layers, in_shape, 6, bias_scale=0.1)
    model = _model(nb, layers, w, in_shape=in_shape)
    k, B = 10, 40
    expr = Expr(k=k, B=B, lambda_=0., batch_size=128, fi_mode='sdp')
    expr.pool_images = x
    np.random.seed(9)
    u = np.random.sample(k)
    np.random.seed(9)
    q, soln, sel = nb.fi.query_whole_sdp(model, expr, np.arange(300), None, return_solution=True)
    assert soln['status'] == 'optimal'
    r = O.forward(layers, w, x)
    sel_o = O.uncertainty_filtering(r['posteriors'].copy(), B)
    assert set(sel.tolist()) == set(sel_o.tolist())
    eng = nb.get_engine()
    assert eng.layer_info(len(layers) - 1)[2] == 1
    post, g = eng.fi_shrunk_images(x[sel])
    po, go = O.shrunk_class_gradients(layers, w, x[sel])
    assert g.shape == (c, B, eng.fi_shrunk_tau())
    assert np.abs(post - po).max() < POST_TOL
    _assert_shrunk_close(g, go)
    A = O.gen_A_matrices_multiclass(po.copy(), go)
    qo, to, phio, gapo, ito = O.sdp_solve(A, 1e-4)
    assert abs(soln['primal objective'] / phio - 1) < OBJ_RTOL
    q_dev = np.array(soln['x'][:B])
    phi_c, gap_c = O.sdp_certificate(A, q_dev)
    assert abs(phi_c / phio - 1) < OBJ_RTOL
    assert np.array_equal(q, sel[O.sample_query_dstr(q_dev.copy(), k, u)])


def test_errors(nb):
    e = nb.Engine(0)
    try:
        for c in (33, 48, 63):
            layers = conv_net(c)
            w, x = _case(layers, 40, c)
            e.set_model(_model(nb, layers, w, [2, 3, 4], 0.5))
            e.pool_begin(len(x))
            with pytest.raises(nb._lib.NnalError, match='error 4'):
                e.pool_eval_images(x, 0)
            with pytest.raises(nb._lib.NnalError, match='error 4'):
                e.pool_mc_config(2, 0.5, [2, 3, 4])
    finally:
        e.close()
    # block-form greedy FI stops at 32 classes: the library's error after a successful pool pass, engine still usable
    layers = conv_net(100)
    w, x = _case(layers, 300, 100, scale=3.0)
    model = _model(nb, layers, w)
    expr = Expr(k=10, B=50, lambda_=0., batch_size=128, fi_mode='block-greedy')
    expr.pool_images = x
    with pytest.raises(nb._lib.NnalError, match='error 4'):
        nb.NNAL.CNN_query(model, expr, np.arange(len(x)), 'fi', None)
    q = nb.NNAL.CNN_query(model, expr, np.arange(len(x)), 'entropy', None)
    H = O.compute_entropy(O.forward(layers, w, x)['posteriors'])
    assert_topk_equivalent(q, -H, 10, 1e-4)
