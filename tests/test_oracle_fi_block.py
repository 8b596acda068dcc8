"""Float64 reference of the multi-class block-form greedy FI selection (tests/fi_block_oracle.py): the closed-form factor of
diag(pi) - pi pi^T, the incremental greedy against the brute-force references, the c = 2 reduction to the binary path, and
NNAL.CNN_query(..., 'fi') with fi_mode='block-greedy' over 1, 2 and 3 gloo ranks on the NumPy fake engine."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from tests import fi_block_oracle as FB

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _posteriors(c, n, seed):
    """Dirichlet columns with one one-hot column and one column with exact zeros."""
    rs = np.random.RandomState(seed)
    P = rs.dirichlet(np.ones(c) * 0.7, n).T
    P[:, 0] = 0.
    P[c - 1, 0] = 1.
    if c > 2:
        P[1, 1] = 0.
        P[:, 1] /= P[:, 1].sum()
    return P


@pytest.mark.parametrize('c', [2, 3, 10, 32])
def test_multinomial_factor(c):
    rs = np.random.RandomState(c)
    cols = [rs.dirichlet(np.ones(c)), np.eye(c)[0], np.eye(c)[c - 1], np.eye(c)[c // 2]]
    z = rs.dirichlet(np.ones(c))
    z[::2] = 0.
    cols.append(z / z.sum())
    for p in cols:
        L = FB.multinomial_factor(p)
        assert L.shape == (c, c - 1)
        q = np.asarray(p, dtype=np.float64) / np.sum(p)
        assert np.abs(L @ L.T - (np.diag(q) - np.outer(q, q))).max() < 1e-14


def _direct_fi(post, U):
    Ut = np.vstack([U, np.ones(U.shape[1])])
    out = []
    for i in range(post.shape[1]):
        p = post[:, i] / post[:, i].sum()
        out.append(np.kron(np.diag(p) - np.outer(p, p), np.outer(Ut[:, i], Ut[:, i])))
    return out


@pytest.mark.parametrize('c', [2, 3, 5])
def test_greedy_block_matches_bruteforce(c):
    n, d, k, delta = 13, 5, 6, 1e-3
    post = _posteriors(c, n, 20 + c)
    U = np.random.RandomState(30 + c).randn(d, n)
    S, f, red = FB.greedy_fi_block(post, U, delta, k)
    D = c * (d + 1)
    S2, f2 = O.greedy_fi_dual_bruteforce(FB.last_layer_block_kernel(post, U), c - 1, D, delta, k)
    S3, f3 = O.greedy_fi_direct(_direct_fi(post, U), delta, k)
    assert np.array_equal(S, S2) and np.array_equal(S, S3)
    assert np.allclose(f, f2, rtol=1e-10, atol=0) and np.allclose(f, f3, rtol=1e-10, atol=0)
    s = np.arange(1, k + 1)
    assert np.allclose(f, (D - s * (c - 1)) / delta + red, rtol=1e-12, atol=0)
    rep = FB.greedy_fi_block_replay(post, U, delta, S)
    assert np.allclose(rep[:, 0], rep[:, 1], rtol=1e-12) and np.allclose(rep[:, 2], red, rtol=1e-12)


def test_block_kernel_binary_reduction():
    n, d, k, delta = 40, 7, 9, 1e-4
    post = _posteriors(2, n, 3)
    U = np.random.RandomState(4).randn(d, n)
    p1 = post[1] / post.sum(0)
    Kt = O.last_layers_kernel(p1, U)
    assert np.abs(FB.last_layer_block_kernel(post, U) - Kt).max() < 1e-13 * np.abs(Kt).max()
    S, f, red = FB.greedy_fi_block(post, U, delta, k)
    S1, f1, red1 = O.greedy_fi_rank1(Kt, 2 * (d + 1), delta, k, return_reduced=True)
    assert np.array_equal(S, S1)
    assert np.allclose(red, red1, rtol=1e-10) and np.allclose(f, f1, rtol=1e-12)


def _launch(world, out, port):
    os.makedirs(out, exist_ok=True)
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR='127.0.0.1',
                   MASTER_PORT=str(port), OMP_NUM_THREADS='1')
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, 'tests', '_fi_block_dist_worker.py'), out], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        o = p.communicate(timeout=600)[0].decode()
        assert p.returncode == 0, o[-3000:]
    return [np.load(os.path.join(out, 'rank%d.npz' % r)) for r in range(world)]


def test_block_greedy_query_over_ranks(tmp_path):
    """Identical positions on every rank and world size, equal to the float64 oracle on the same candidates."""
    runs = [_launch(w, str(tmp_path / ('w%d' % w)), 29631 + w) for w in (1, 2, 3)]
    one = runs[0][0]
    for multi in runs:
        for r in multi:
            for key in ('q_pre', 'q_all'):
                assert np.array_equal(r[key], one[key]), key
            assert np.allclose(r['red_pre'], one['red_pre'], rtol=1e-12, atol=0)
    sys.path.insert(0, ROOT)
    from tests._fi_block_dist_worker import make_case, K, B, DELTA
    layers, w, x = make_case()
    r = O.forward(layers, w, x, feature_layer=len(layers) - 2)
    post, feat = r['posteriors'], r['feature_layer']
    q = np.where(post == 0, 1e-8, post)
    sel = O.stable_topk(np.sum(q * np.log(q), axis=0), B)        # SCORE_NEG_ENTROPY, eps 1e-8
    f32 = lambda a: a.astype(np.float32).astype(np.float64)     # the engine hands float32 posteriors and features over
    S, _, red = FB.greedy_fi_block(f32(post[:, sel]), f32(feat[:, sel]), DELTA, K)
    assert np.array_equal(one['q_pre'], sel[S])
    assert np.allclose(one['red_pre'], red, rtol=1e-9)
    S, _, _ = FB.greedy_fi_block(f32(post), f32(feat), DELTA, K)
    assert np.array_equal(one['q_all'], S)
