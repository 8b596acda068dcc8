"""CPU tests of tests/tf_same_ref.py, the float64 forward with TF SAME padding written out, and of the oracles against it.

The worked window cases below are TF's SAME rule applied by hand: out = ceil(n/s), pad_total = (out-1)*s + s - n,
pad_before = pad_total // 2, the rest after.  Padded pool cells are -inf and never win."""
import numpy as np
import pytest
import torch

import oracle as O
from oracle.torch_fp32 import TorchForward
from tests import tf_same_ref as R
from tests.test_gpu_forward_shapes import FORWARD_NETS, SHRUNK_NETS, pw1_with_pools
from tests.test_gpu_parity import SMALL
from tests.test_gpu_rep import NET as REP_NET
from tests.test_gpu_sdp import SMALL2
from tests.test_oracle import SMALL as ORACLE_SMALL
from tests.test_reference_dispatch_golden import LAYERS as DISPATCH_LAYERS

# (n, s) -> input indices of each pooled output, written out by hand
WORKED_WINDOWS = [
    (7, 3, [[0, 1], [2, 3, 4], [5, 6]]),          # pad_total 2: one row before, one after
    (5, 4, [[0, 1, 2], [3, 4]]),                  # pad_total 3: one before, two after
    (2, 5, [[0, 1]]),                             # window larger than the input: pad_total 3, one before
    (8, 3, [[0, 1, 2], [3, 4, 5], [6, 7]]),       # pad_total 1: after only
    (7, 2, [[0, 1], [2, 3], [4, 5], [6]]),        # s = 2: never anything before
    (9, 3, [[0, 1, 2], [3, 4, 5], [6, 7, 8]]),    # no padding
    (11, 5, [[0, 1, 2], [3, 4, 5, 6, 7], [8, 9, 10]]),
]


@pytest.mark.parametrize('n,s,windows', WORKED_WINDOWS)
def test_pool_windows_worked(n, s, windows):
    assert R.pool_windows(n, s) == windows
    assert O.pool_same_pads(n, s) == R.same_pads(n, s, s)


@pytest.mark.parametrize('n,s,windows', WORKED_WINDOWS)
def test_max_pool_1d_worked(n, s, windows):
    """All-negative input: a zero-padded or misaligned pool would show up in the maxima."""
    x = -1 - np.random.RandomState(n * 10 + s).rand(2, n, 1, 3)
    want = np.stack([x[:, w, :, :].max(axis=1) for w in windows], axis=1)
    got = R.max_pool(torch.tensor(x).permute(0, 3, 1, 2), s).permute(0, 2, 3, 1).numpy()
    assert np.array_equal(got, want)
    assert np.array_equal(O.max_pool_same(x, s), want)
    # the same pool along the other axis
    xt = x.transpose(0, 2, 1, 3)
    assert np.array_equal(O.max_pool_same(xt, s), want.transpose(0, 2, 1, 3))


def test_max_pool_2d_non_square_worked():
    """H = 7, W = 5, s = 3: rows {0,1} {2,3,4} {5,6}; columns {0,1,2} {3,4}."""
    rows, cols = [[0, 1], [2, 3, 4], [5, 6]], [[0, 1, 2], [3, 4]]
    x = -np.random.RandomState(3).rand(2, 7, 5, 4)
    want = np.empty((2, 3, 2, 4))
    for i, r in enumerate(rows):
        for j, c in enumerate(cols):
            want[:, i, j, :] = x[:, r][:, :, c].max(axis=(1, 2))
    got = R.max_pool(torch.tensor(x).permute(0, 3, 1, 2), 3).permute(0, 2, 3, 1).numpy()
    assert np.array_equal(got, want)
    out, am = O.max_pool_same(x, 3, return_argmax=True)
    assert np.array_equal(out, want)
    # argmax indexes the 3x3 window of the padded input: one padded row before rows {0,1}, none before columns
    for n in range(2):
        for k in range(4):
            a = am[n, 0, 0, k]
            assert x[n, a // 3 - 1, a % 3, k] == want[n, 0, 0, k]


def test_conv_pads():
    assert R.same_pads(9, 5, 1) == (2, 2)
    assert R.same_pads(9, 1, 1) == (0, 0)
    assert R.same_pads(4, 7, 1) == (3, 3)


def _close(a, b, tol):
    return np.abs(a - b).max() <= tol * max(1., np.abs(b).max())


SUITE_NETS = [(SMALL, (9, 7, 2)), (SMALL2, (11, 8, 3)), (REP_NET, (9, 9, 2)), (ORACLE_SMALL, (9, 7, 2)),
              (DISPATCH_LAYERS, (5, 5, 2)), (O.pw1_layers(2), (25, 25, 3)), (O.pw1_layers(5), (25, 25, 3))]


@pytest.mark.parametrize('idx', range(len(SUITE_NETS)))
def test_reference_equals_oracle_on_2x2_nets(idx):
    """Every 2x2-pool net of the suite, and PW1: the explicit-padding reference == oracle.forward to 1e-12."""
    layers, in_shape = SUITE_NETS[idx]
    w = O.he_init_weights(layers, in_shape, 10 + idx, bias_scale=0.1)
    x = np.random.RandomState(idx).randn(6 if in_shape[0] > 20 else 40, *in_shape).astype(np.float32)
    ref = R.forward(layers, w, x)
    ora = O.forward(layers, w, x, feature_layer=len(layers) - 2, keep_acts=True)
    assert _close(ref['logits'], ora['output'], 1e-12)
    assert _close(ref['posteriors'], ora['posteriors'], 1e-12)
    assert _close(ref['feature'], ora['feature_layer'], 1e-12)
    assert _close(ref['prev'], ora['acts'][len(layers) - 2]['in'], 1e-12)


ALL_NETS = [(name, layers, in_shape) for name, layers, in_shape in FORWARD_NETS] + \
           [('pw1_max1_3', pw1_with_pools(3, 2), (25, 25, 3)), ('pw1_max2_4', pw1_with_pools(2, 4), (25, 25, 3))]


@pytest.mark.parametrize('name,layers,in_shape', ALL_NETS, ids=[a[0] for a in ALL_NETS])
def test_oracles_equal_reference_on_forward_grid(name, layers, in_shape):
    """oracle.forward and the float64 torch oracle follow TF's SAME alignment for every pool size."""
    w = O.he_init_weights(layers, in_shape, 5, bias_scale=0.1)
    x = np.random.RandomState(2).randn(4 if in_shape[0] > 20 else 30, *in_shape).astype(np.float32)
    ref = R.forward(layers, w, x)
    ora = O.forward(layers, w, x, feature_layer=len(layers) - 2)
    assert _close(ora['posteriors'], ref['posteriors'], 1e-12)
    assert _close(ora['feature_layer'], ref['feature'], 1e-12)
    tf = TorchForward(layers, w, feature_layer=len(layers) - 2, dtype=torch.float64)(x)
    assert _close(tf['posteriors'], ref['posteriors'], 1e-12)
    assert _close(tf['feature_layer'], ref['feature'], 1e-12)


def test_misaligned_pool_differs():
    """The grid can tell the alignments apart: pooling from row 0 instead of TF's windows moves the posteriors."""
    name, layers, in_shape = [n for n in FORWARD_NETS if n[0] == 'pool_s4_c8_13x10'][0]
    w = O.he_init_weights(layers, in_shape, 5, bias_scale=0.1)
    x = np.random.RandomState(2).randn(30, *in_shape).astype(np.float32)
    ref = R.forward(layers, w, x)['posteriors']
    orig = R.same_pads
    try:
        R.same_pads = lambda n, k, s: (0, -(-n // s) * s - n) if k == s and s > 1 else orig(n, k, s)
        wrong = R.forward(layers, w, x)['posteriors']
    finally:
        R.same_pads = orig
    assert np.abs(wrong - ref).max() > 1e-2


@pytest.mark.parametrize('name,layers,in_shape', SHRUNK_NETS, ids=[a[0] for a in SHRUNK_NETS])
def test_oracle_gradients_vs_autograd_through_wide_pools(name, layers, in_shape):
    """fi_oracle's backward routes the pool gradient to TF's window (first maximum of the padded window): explicit
    gradients of log p_y == torch autograd through the explicit-padding reference."""
    w = O.he_init_weights(layers, in_shape, 6, bias_scale=0.1)
    x = np.random.RandomState(1).randn(1, *in_shape)
    c = layers[-1][1][0]
    names = [n for n, s in layers if s[1] != 'pool']
    for y in range(c):
        params = R.torch_params(w, requires_grad=True)
        logits, _, _ = R.forward_t(layers, params, torch.tensor(x))
        lp = torch.log_softmax(logits, 0)[y, 0]
        tg = torch.autograd.grad(lp, [t for n in names for t in params[n]])
        og = O.explicit_class_gradients(layers, w, x, y)
        assert len(og) == len(tg)
        for a, b in zip(og, tg):
            assert np.allclose(a, b.numpy().reshape(a.shape), rtol=1e-9, atol=1e-12)
