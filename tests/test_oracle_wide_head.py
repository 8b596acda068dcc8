"""The float64 references behind the wide-head GPU tests (oracle.forward's softmax, the MC running means of
tests/mc_multi_oracle.py) at 1,000 and 21,841 classes with logits up to 80 in magnitude, against torch float64
log_softmax."""
import numpy as np
import pytest
import torch

import oracle as O
from tests import mc_multi_oracle as MM


def _fc_head(c, d, n, seed):
    """One FC layer on a [n,1,1,d] input whose logits span about +-80."""
    rs = np.random.RandomState(seed)
    x = rs.randn(n, 1, 1, d).astype(np.float32)
    W = rs.randn(c, d).astype(np.float32)
    b = rs.randn(c, 1).astype(np.float32)
    z = W.astype(np.float64) @ x.reshape(n, d).T.astype(np.float64) + b.astype(np.float64)
    s = np.float32(80.0 / np.abs(z).max())
    return [('fc1', [c, 'fc'])], {'fc1': (W * s, b * s)}, x


def _torch_post(layers, w, x):
    W, b = w[layers[0][0]]
    z = torch.from_numpy(W.astype(np.float64)) @ torch.from_numpy(x.reshape(len(x), -1).T.astype(np.float64))
    z = z + torch.from_numpy(b.astype(np.float64))
    return z, torch.log_softmax(z, dim=0)


@pytest.mark.parametrize('c', [1000, 21841])
def test_softmax_matches_torch_log_softmax(c):
    layers, w, x = _fc_head(c, 24, 64, c)
    z, logp = _torch_post(layers, w, x)
    assert 60 < float(z.abs().max()) <= 80.0001
    post = O.forward(layers, w, x)['posteriors']
    assert post.shape == (c, len(x))
    want = logp.exp().numpy()
    assert np.abs(post - want).max() < 1e-15
    assert np.abs(post.sum(axis=0) - 1).max() < 1e-12
    # the entropy the scores use, from the log-probabilities directly
    H = -(logp.exp() * logp).sum(dim=0).numpy()
    assert np.allclose(O.compute_entropy(post.copy()), H, rtol=0, atol=1e-12)


@pytest.mark.parametrize('c', [1000, 21841])
def test_class_running_means_match_torch(c):
    layers, w, x = _fc_head(c, 24, 48, c + 1)
    passes = []
    for t in range(3):
        ws = {'fc1': (w['fc1'][0] * np.float32(1 + 0.1 * t), w['fc1'][1])}
        passes.append(O.forward(layers, ws, x)['posteriors'].astype(np.float32).astype(np.float64))
    av_post, av_ent = MM.class_running_means(passes)
    P = torch.from_numpy(np.stack(passes))                                    # [T, c, n]
    want_post = P.mean(dim=0)
    Pb = torch.where(P == 0, P + 1e-6, P)
    want_ent = (-(Pb * Pb.log()).sum(dim=1)).mean(dim=0)
    assert np.abs(av_post - want_post.numpy()).max() < 1e-15
    assert np.abs(av_ent - want_ent.numpy()).max() < 1e-12
    for kind in (12, 13):
        m = torch.where(want_post == 0, want_post + 1e-6, want_post)
        h = -(m * m.log()).sum(dim=0)
        want = -h if kind == 12 else -(h - want_ent)
        assert np.abs(MM.scores(av_post, av_ent, kind) - want.numpy()).max() < 1e-12
