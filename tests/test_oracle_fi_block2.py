"""Float64 reference of the multi-class block-form greedy FI selection over the last two FC layers
(tests/fi_block2_oracle.py): the block kernel against explicit per-class gradients, the incremental greedy against the
definitional greedy, the c = 2 reduction to the binary two-layer path, and NNAL.CNN_query(..., 'fi') with
fi_mode='block-greedy', fi_layers=2 over 1, 2 and 3 gloo ranks on the NumPy fake engine."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from tests import fi_block2_oracle as FB2
from tests.fi_block_oracle import multinomial_factor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _tiny(c, seed, n):
    """conv -> pool -> fc1 (12) -> fc2 (8, feature layer) -> fc3 (c); returns layers, weights, images, forward pass."""
    layers = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [12, 'fc']), ('fc2', [8, 'fc']),
              ('fc3', [c, 'fc'])]
    w = O.he_init_weights(layers, (5, 5, 2), seed, bias_scale=0.1)
    x = np.random.RandomState(seed + 1).rand(n, 5, 5, 2).astype(np.float32)
    r = O.forward(layers, w, x, feature_layer=3, keep_acts=True)
    return layers, w, x, r


def _class_gradients(layers, w, x, c):
    """[n][D, c]: column y = flattened gradient of log p_y over (W2, b2, W3, b3) (oracle.explicit_class_gradients)."""
    out = []
    for i in range(x.shape[0]):
        cols = [np.concatenate([g.ravel() for g in O.explicit_class_gradients(layers, w, x[i:i + 1], y, ['fc2', 'fc3'])])
                for y in range(c)]
        out.append(np.stack(cols, axis=1))
    return out


@pytest.mark.parametrize('c', [3, 5])
def test_kernel_matches_explicit_gradients(c):
    """K_ij = G_i^T G_j with G_i = [g_0 .. g_{c-1}] L_i: sum_y (e_y - pi) L[y, :] = L since 1^T L = 0, so G_i G_i^T =
    sum_y pi_y g_y g_y^T."""
    layers, w, x, r = _tiny(c, 3 + c, 9)
    post, U, A = r['posteriors'], r['feature_layer'], r['acts'][3]['in']
    Gs = [g @ multinomial_factor(post[:, i]) for i, g in enumerate(_class_gradients(layers, w, x, c))]
    assert Gs[0].shape[0] == FB2.two_layer_dim(c, 8, 12)
    Gall = np.concatenate(Gs, axis=1)
    K = FB2.two_layer_block_kernel(post, U, A, w['fc3'][0])
    assert np.abs(K - Gall.T @ Gall).max() < 1e-12 * np.abs(K).max()
    assert np.any(U == 0), 'the case must exercise the ReLU mask'


@pytest.mark.parametrize('c', [3, 5])
def test_greedy_matches_definition(c):
    layers, w, x, r = _tiny(c, 20 + c, 14)
    post, U, A = r['posteriors'], r['feature_layer'], r['acts'][3]['in']
    k, delta = 6, 1e-3
    Abar = []
    for i, g in enumerate(_class_gradients(layers, w, x, c)):
        p = post[:, i] / post[:, i].sum()
        Abar.append((g * p[None, :]) @ g.T)                     # sum_y pi_y g_y g_y^T
    S, f, red = FB2.greedy_fi_block2(post, U, A, w['fc3'][0], delta, k)
    S2, f2 = O.greedy_fi_direct(Abar, delta, k)
    assert np.array_equal(S, S2)
    assert np.allclose(f, f2, rtol=1e-9, atol=0)
    K = FB2.two_layer_block_kernel(post, U, A, w['fc3'][0])
    rep = FB2.greedy_block_kernel_replay(K, c - 1, delta, S)
    assert np.allclose(rep[:, 0], rep[:, 1], rtol=1e-12) and np.allclose(rep[:, 2], red, rtol=1e-12)


def test_binary_reduction():
    """c = 2: the two-layer block kernel is the binary two-layer kernel, and the greedy is the rank-one greedy."""
    n, d, dp, k, delta = 40, 7, 11, 9, 1e-4
    rs = np.random.RandomState(5)
    post = rs.dirichlet(np.ones(2), n).T
    post[:, 3] = [0., 1.]
    U = np.maximum(rs.randn(d, n), 0)
    A = np.maximum(rs.randn(dp, n), 0)
    W = rs.randn(2, d)
    p1 = post[1] / post.sum(0)
    Kt = O.last_layers_kernel(p1, U, A, W)
    K = FB2.two_layer_block_kernel(post, U, A, W)
    assert np.abs(K - Kt).max() < 1e-13 * np.abs(Kt).max()
    D = FB2.two_layer_dim(2, d, dp)
    assert D == O.last_layers_dim(2, d, dp)
    S, f, red = FB2.greedy_fi_block2(post, U, A, W, delta, k)
    S1, f1, red1 = O.greedy_fi_rank1(Kt, D, delta, k, return_reduced=True)
    assert np.array_equal(S, S1)
    assert np.allclose(red, red1, rtol=1e-10) and np.allclose(f, f1, rtol=1e-12)


def _launch(world, out, port):
    os.makedirs(out, exist_ok=True)
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR='127.0.0.1',
                   MASTER_PORT=str(port), OMP_NUM_THREADS='1')
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, 'tests', '_fi_block2_dist_worker.py'), out], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        o = p.communicate(timeout=600)[0].decode()
        assert p.returncode == 0, o[-3000:]
    return [np.load(os.path.join(out, 'rank%d.npz' % r)) for r in range(world)]


def test_block2_greedy_query_over_ranks(tmp_path):
    """Identical positions on every rank and world size, equal to the float64 oracle on the same candidates."""
    runs = [_launch(w, str(tmp_path / ('w%d' % w)), 29641 + w) for w in (1, 2, 3)]
    one = runs[0][0]
    for multi in runs:
        for r in multi:
            for key in ('q_pre', 'q_all'):
                assert np.array_equal(r[key], one[key]), key
            assert np.allclose(r['red_pre'], one['red_pre'], rtol=1e-12, atol=0)
    sys.path.insert(0, ROOT)
    from tests._fi_block2_dist_worker import make_case, K, B, DELTA
    layers, w, x = make_case()
    fl = len(layers) - 2
    r = O.forward(layers, w, x, feature_layer=fl, keep_acts=True)
    post, feat, prev = r['posteriors'], r['feature_layer'], r['acts'][fl]['in']
    q = np.where(post == 0, 1e-8, post)
    sel = O.stable_topk(np.sum(q * np.log(q), axis=0), B)        # SCORE_NEG_ENTROPY, eps 1e-8
    f32 = lambda a: a.astype(np.float32).astype(np.float64)     # the engine hands float32 factors over
    W3 = f32(w[layers[-1][0]][0])
    S, _, red = FB2.greedy_fi_block2(f32(post[:, sel]), f32(feat[:, sel]), f32(prev[:, sel]), W3, DELTA, K)
    assert np.array_equal(one['q_pre'], sel[S])
    assert np.allclose(one['red_pre'], red, rtol=1e-9)
    S, _, _ = FB2.greedy_fi_block2(f32(post), f32(feat), f32(prev), W3, DELTA, K)
    assert np.array_equal(one['q_all'], S)


def test_fi_layers_validated():
    """fi_layers other than 1 or 2 is refused before any device work."""
    from collections import OrderedDict
    import nnal_b200

    class Expr(object):
        pass

    from tests._fi_block2_dist_worker import make_case
    layers, w, x = make_case()
    model = nnal_b200.NN.CNN((5, 5, 2), OrderedDict(layers), feature_layer=len(layers) - 2)
    model.set_weights(w)
    expr = Expr()
    expr.pars = dict(k=3, B=10, fi_mode='block-greedy', fi_layers=3)
    expr.pool_images = x
    with pytest.raises(ValueError):
        nnal_b200.fi.query_whole_block(model, expr, np.arange(len(x)), None)
