"""Float64 reference of the multi-class MC-dropout and committee scorers (tests/mc_multi_oracle.py): the scores against
their formulas on hand-made posteriors, the c = 2 reduction to the binary scorers of oracle/mc_oracle.py, and
NNAL.CNN_query(..., 'MC-entropy' | 'BALD' | 'ensemble' | 'QBC-JS') over 1, 2 and 3 gloo ranks on the NumPy fake engine."""
import os
import subprocess
import sys

import numpy as np

import oracle as O
from oracle import mc_oracle as M
from tests import mc_multi_oracle as MM

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_scores_match_formulas():
    """Two passes over four samples of c = 3, written out by hand: a one-hot pass (zeros bumped by 1e-6), a uniform
    sample, and samples whose passes disagree."""
    P0 = np.array([[1., 1 / 3, .5, .2], [0., 1 / 3, .5, .3], [0., 1 / 3, 0., .5]])
    P1 = np.array([[0., 1 / 3, 0., .2], [1., 1 / 3, .5, .3], [0., 1 / 3, .5, .5]])
    av_post, av_ent = MM.class_running_means([P0, P1])
    assert np.array_equal(av_post, (P0 + P1) / 2)
    b = 1e-6 * np.log(1e-6)
    h1 = -(1. * np.log(1.) + 2 * b)                    # a one-hot pass: the two zero classes are bumped
    h_half = -(2 * .5 * np.log(.5) + b)
    h_mix = -(.2 * np.log(.2) + .3 * np.log(.3) + .5 * np.log(.5))
    assert np.allclose(av_ent, [h1, np.log(3), h_half, h_mix], rtol=1e-14, atol=0)
    H = np.array([-(2 * .5 * np.log(.5) + b), np.log(3), -(.5 * np.log(.5) + 2 * .25 * np.log(.25)), h_mix])
    assert np.allclose(MM.scores(av_post, av_ent, 12), -H, rtol=1e-14, atol=0)
    assert np.allclose(MM.scores(av_post, av_ent, 13), -(H - av_ent), rtol=1e-13, atol=1e-15)
    # the uniform sample has the largest predictive entropy; the disagreeing one-hot passes the largest BALD score
    assert O.stable_topk(MM.scores(av_post, av_ent, 12), 1)[0] == 1
    assert O.stable_topk(MM.scores(av_post, av_ent, 13), 1)[0] == 0
    # a pass with equal scores breaks the tie at the lowest position
    av_tie = np.tile(np.array([[.2], [.3], [.5]]), (1, 5))
    assert np.array_equal(O.stable_topk(MM.scores(av_tie, np.zeros(5), 12), 3), [0, 1, 2])


def test_binary_reduction():
    """c = 2: kind 13 is the binary BALD score (negated) and kind 12 ranks like |mean p - 1/2|, within 1e-12, from the
    binary running means and from the two-class ones alike."""
    rs = np.random.RandomState(5)
    passes = [rs.rand(400) for _ in range(6)]
    passes[0][:5] = 0.
    passes[1][5:9] = 1.
    av_p, av_e = M.mc_running_means(passes)
    s12 = MM.scores_from_binary(av_p, av_e, 12)
    s13 = MM.scores_from_binary(av_p, av_e, 13)
    assert np.abs(s13 + M.bald_scores(av_p, av_e)).max() < 1e-12
    assert np.abs(s12 + M.binary_entropy_bumped(av_p)).max() < 1e-12
    for k in (1, 17, 100):
        assert np.array_equal(O.stable_topk(s12, k), O.stable_topk(M.mc_entropy_scores(av_p), k))
        assert np.array_equal(O.stable_topk(s13, k), O.stable_topk(-M.bald_scores(av_p, av_e), k))
    two = [np.stack([1 - p, p]) for p in passes]
    av_post, av_ent = MM.class_running_means(two)
    assert np.abs(av_post[1] - av_p).max() < 1e-12 and np.abs(av_ent - av_e).max() < 1e-12
    assert np.abs(MM.scores(av_post, av_ent, 12) - s12).max() < 1e-12
    assert np.abs(MM.scores(av_post, av_ent, 13) - s13).max() < 1e-12


def test_tail_pass_is_forward_dropout():
    """The reference's single-trunk tail pass is mc_oracle.forward_dropout, bit for bit."""
    sys.path.insert(0, ROOT)
    from tests._mc_multi_dist_worker import make_case, DROPOUT_LAYERS, KEEP, SEED
    layers, w, _, x = make_case(5)
    pos = 100 + np.arange(len(x))
    got = MM.mc_passes(layers, w, x, pos, 3, KEEP, DROPOUT_LAYERS, SEED, 7, post_dtype=np.float64)
    for t in range(3):
        assert np.array_equal(got[t], M.forward_dropout(layers, w, x, pos, KEEP, DROPOUT_LAYERS, SEED, 7 + t)[1])


def _launch(world, out, port):
    os.makedirs(out, exist_ok=True)
    procs = []
    for r in range(world):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE=str(world), LOCAL_RANK=str(r), MASTER_ADDR='127.0.0.1',
                   MASTER_PORT=str(port), OMP_NUM_THREADS='1')
        procs.append(subprocess.Popen([sys.executable, os.path.join(ROOT, 'tests', '_mc_multi_dist_worker.py'), out], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT))
    for p in procs:
        o = p.communicate(timeout=600)[0].decode()
        assert p.returncode == 0, o[-3000:]
    return [np.load(os.path.join(out, 'rank%d.npz' % r)) for r in range(world)]


def test_query_over_ranks(tmp_path):
    """Identical positions on every rank and world size, equal to the float64 reference's selection over the whole pool."""
    runs = [_launch(w, str(tmp_path / ('w%d' % w)), 29671 + w) for w in (1, 2, 3)]
    one = runs[0][0]
    for multi in runs:
        for r in multi:
            for key in one.files:
                assert np.array_equal(r[key], one[key]), key
    sys.path.insert(0, ROOT)
    from tests._mc_multi_dist_worker import make_case, CLASSES, METHODS, K, T, KEEP, SEED, FIRST_PASS, DROPOUT_LAYERS
    for c in CLASSES:
        layers, w, members, x = make_case(c)
        for method in METHODS:
            if method in ('MC-entropy', 'BALD'):
                q = MM.query_mc_whole(layers, w, x, K, T, KEEP, DROPOUT_LAYERS, SEED, method, FIRST_PASS)[0]
            else:
                q = MM.query_committee_whole(layers, members, x, K, method)[0]
            assert len(q) == K
            assert np.array_equal(one['c%d_%s' % (c, method)], q), (c, method)
