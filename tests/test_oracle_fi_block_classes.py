"""Float64 reference of the class-capped block greedy FI (tests/fi_block_cls_oracle.py, ``fi_classes``): the truncation rule,
the compact greedy against the dense oracle on truncated posteriors, the query's argument checks, and
NNAL.CNN_query(..., 'fi') with fi_mode='block-greedy', fi_classes over 1, 2 and 3 gloo ranks on the NumPy fake engine."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from tests import fi_block_cls_oracle as FC
from tests import fi_block_oracle as FB

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_truncation_ties_and_zeros():
    post = np.array([[.2, 0., .5, 0.],
                     [.3, .6, 0., 0.],
                     [.2, 0., .5, 1.],
                     [.3, .4, 0., 0.]], dtype=np.float32)          # [c=4, n=4]
    cls, p = FC.top_classes(post, 3)
    # column 0: .3 at classes 1 and 3 first, then the tie of .2 goes to class 0;  column 1: two nonzeros, then the lowest
    # zero class;  column 2: ties at .5, then zeros from the lowest class;  column 3: one-hot, zeros from class 0
    assert cls.tolist() == [[0, 1, 3], [0, 1, 3], [0, 1, 2], [0, 1, 2]]
    assert np.array_equal(p, np.take_along_axis(post.T, cls, axis=1))
    t = FC.truncate_posteriors(post, 3)
    assert np.allclose(t[:, 0], [.25, .375, 0., .375]) and np.allclose(t.sum(axis=0), 1.)
    assert np.array_equal(t[:, 3], [0., 0., 1., 0.])
    assert t[2, 1] == 0. and t[0, 1] == 0.                     # a kept exact zero stays zero


def test_truncation_keeps_everything_at_r_ge_c():
    rs = np.random.RandomState(0)
    post = rs.dirichlet(np.ones(6), 20).T.astype(np.float32)
    for r in (6, 7, 32):
        cls, p = FC.top_classes(post, r)
        assert np.array_equal(cls, np.tile(np.arange(6), (20, 1))) and np.array_equal(p, post.T)
        p64 = post.astype(np.float64)
        assert np.allclose(FC.truncate_posteriors(post, r), p64 / p64.sum(axis=0), rtol=1e-15, atol=0)


def _case(c, n, d, seed):
    rs = np.random.RandomState(seed)
    P = rs.dirichlet(np.ones(c) * 0.3, n).T
    P[:, ::13] = 0.
    P[seed % c, ::13] = 1.
    return P.astype(np.float32), rs.randn(d, n)


@pytest.mark.parametrize('c', [3, 10, 33, 64])
@pytest.mark.parametrize('r', [2, 5, 10, 32])
def test_compact_greedy_equals_dense_on_truncated(c, r):
    """The kept-class greedy is greedy_fi_block on the truncated posteriors: same picks, same objective; the dense
    form's reduced objective carries (c - q)/delta per step for the c - q zero columns of every factor."""
    n, d, k, delta = 60, 12, 8, 1e-3
    post, U = _case(c, n, d, c + r)
    cls, p = FC.top_classes(post, r)
    q = cls.shape[1]
    S, f, red = FC.greedy_fi_block_cls(cls, p, U, c, delta, k)
    Sd, fd, redd = FB.greedy_fi_block(FC.truncate_posteriors(post, r), U, delta, k)
    s = np.arange(1, k + 1)
    assert np.array_equal(S, Sd)
    assert np.allclose(red + s * (c - q) / delta, redd, rtol=1e-10, atol=0)
    assert np.allclose(f, fd, rtol=1e-12, atol=0)
    rep = FC.greedy_fi_block_cls_replay(cls, p, U, c, delta, S)
    assert np.array_equal(rep[:, 0], rep[:, 1]) and np.allclose(rep[:, 2], red, rtol=1e-14, atol=0)


def test_uncapped_equals_dense():
    c, n, d, k, delta = 7, 50, 9, 10, 1e-4
    post, U = _case(c, n, d, 5)
    S, f, red = FC.greedy_fi_block_cls(*FC.top_classes(post, 32), U, c, delta, k)
    Sd, fd, redd = FB.greedy_fi_block(post, U, delta, k)
    assert np.array_equal(S, Sd) and np.allclose(red, redd, rtol=1e-11, atol=0) and np.allclose(f, fd, rtol=1e-13, atol=0)


def test_wide_compact_greedy_runs():
    """c = 21,841: the compact greedy never forms a c x (c-1) factor."""
    c, n, d, k = 21841, 40, 6, 5
    rs = np.random.RandomState(3)
    post = rs.gamma(0.05, size=(c, n)).astype(np.float32)
    post /= post.sum(axis=0)
    cls, p = FC.top_classes(post, 10)
    S, f, red = FC.greedy_fi_block_cls(cls, p, rs.randn(d, n), c, 1e-3, k)
    assert len(np.unique(S)) == k and np.all(np.isfinite(red))


class Expr(object):
    def __init__(self, **pars):
        self.pars = pars


@pytest.mark.parametrize('pars', [dict(fi_classes=1), dict(fi_classes=33), dict(fi_classes=10.0), dict(fi_classes='10'),
                                  dict(fi_classes=True), dict(fi_classes=10, fi_layers=2)])
def test_fi_classes_validated(pars):
    """Bad fi_classes values, and fi_classes with two layers, are refused before any device work."""
    import nnal_b200
    expr = Expr(k=3, B=10, fi_mode='block-greedy', **pars)
    with pytest.raises(ValueError):
        nnal_b200.fi.query_whole_block(None, expr, np.arange(10), None)


def _launch(world, out, port):
    os.makedirs(out, exist_ok=True)
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR='127.0.0.1',
                   MASTER_PORT=str(port), OMP_NUM_THREADS='1')
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, 'tests', '_fi_block_cls_dist_worker.py'), out],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        o = p.communicate(timeout=600)[0].decode()
        assert p.returncode == 0, o[-3000:]
    return [np.load(os.path.join(out, 'rank%d.npz' % r)) for r in range(world)]


def test_block_greedy_classes_query_over_ranks(tmp_path):
    """Identical positions on every rank and world size (the ranks exchange kept classes only), equal to the float64 oracle
    on the same candidates."""
    runs = [_launch(w, str(tmp_path / ('w%d' % w)), 29671 + w) for w in (1, 2, 3)]
    one = runs[0][0]
    for multi in runs:
        for r in multi:
            for key in ('q_pre', 'q_all'):
                assert np.array_equal(r[key], one[key]), key
            assert np.allclose(r['red_pre'], one['red_pre'], rtol=1e-12, atol=0)
    sys.path.insert(0, ROOT)
    from tests._fi_block_cls_dist_worker import make_case, K, B, DELTA, C, R
    layers, w, x = make_case()
    res = O.forward(layers, w, x, feature_layer=len(layers) - 2)
    post, feat = res['posteriors'], res['feature_layer']
    q = np.where(post == 0, 1e-8, post)
    sel = O.stable_topk(np.sum(q * np.log(q), axis=0), B)        # SCORE_NEG_ENTROPY, eps 1e-8
    f32 = lambda a: a.astype(np.float32).astype(np.float64)     # the engine hands float32 posteriors and features over
    cls, p = FC.top_classes(post[:, sel].astype(np.float32), R)
    S, _, red = FC.greedy_fi_block_cls(cls, p, f32(feat[:, sel]), C, DELTA, K)
    assert np.array_equal(one['q_pre'], sel[S])
    assert np.allclose(one['red_pre'], red, rtol=1e-9)
    cls, p = FC.top_classes(post.astype(np.float32), R)
    S, _, _ = FC.greedy_fi_block_cls(cls, p, f32(feat), C, DELTA, K)
    assert np.array_equal(one['q_all'], S)
