"""GPU tests of the generic-network forward (``pytest -m gpu``) across the layer shapes NN.CNN accepts, against the
explicit-padding float64 reference of tests/tf_same_ref.py (TF SAME semantics written out, no code shared with the
oracle package).

Every net runs through Engine.set_model -> pool_begin(n, keep=2) -> pool_eval_images with the tensor cores off and on.
The grid is chosen by code path: max-pools of window 2..5 on inputs of every residue H mod s (TF puts pad_total // 2
padded cells BEFORE the first window, so for s >= 3 the windows do not start at row 0), with channel counts that send
the pool through pool_split_kernel (C % 8 == 0) and pool_split_scalar_kernel; the CUDA-core conv's <8,1> and <8,4>
templates; tensor-core FC widths of 8 mod 16 (the per-element tail of the gemm_tc.cu epilogue) with format changes
both ways; the fused head for 2..32 classes with both of its feature loops; and a ragged last chunk."""
from collections import OrderedDict

import numpy as np
import pytest

import oracle as O
from oracle import mc_oracle as M
from tests import tf_same_ref as R

pytestmark = pytest.mark.gpu

POST_TOL = 1e-4      # north_star: posteriors within 1e-4 absolute
FEAT_RTOL = 2e-4     # feature rows: relative to their largest magnitude


def pool_net(s, C, c=3, fc=72):
    return [('conv1', [C, 'conv', [3, 3]]), ('max1', [[s, s], 'pool']), ('fc1', [fc, 'fc']), ('fc2', [c, 'fc'])]


def pw1_with_pools(s1, s2, nclass=2):
    layers = O.pw1_layers(nclass)
    layers[2] = ('max1', [[s1, s1], 'pool'])
    layers[5] = ('max2', [[s2, s2], 'pool'])
    return layers


# pool window s, trunk channels C, input H x W.  C = 8 / 16: pool_split_kernel; C = 6: pool_split_scalar_kernel (with
# the tensor cores on; fc1 then takes Ho*Wo*C >= 64, a multiple of 8).  Together they cover every H mod s and W mod s.
_POOLS = [(2, 8, 9, 6), (3, 8, 7, 8), (3, 8, 9, 10), (4, 8, 13, 10), (4, 8, 11, 12), (5, 8, 11, 14), (5, 16, 13, 10),
          (5, 16, 12, 9),
          (2, 6, 7, 8), (3, 6, 10, 11), (3, 6, 12, 7), (4, 6, 13, 11), (4, 6, 10, 16), (5, 6, 14, 17), (5, 6, 11, 18),
          (5, 6, 15, 20)]
POOL_NETS = [('pool_s%d_c%d_%dx%d' % (s, C, H, W), pool_net(s, C, c=2 + (i % 2)), (H, W, 2))
             for i, (s, C, H, W) in enumerate(_POOLS)]

# 8x7 -> 3x3 (3x3 pool, one padded column before) -> 5x5 pool on a 3x3 input (window larger than the input, one
# padded row and column before); the first pool feeds a CUDA-core conv, so it runs on fp32 activations
BIG_WINDOW = [('conv1', [8, 'conv', [3, 3]]), ('max1', [[3, 3], 'pool']), ('conv2', [64, 'conv', [3, 3]]),
              ('max2', [[5, 5], 'pool']), ('fc1', [72, 'fc']), ('fc2', [3, 'fc'])]

CONV_NETS = [
    # Cin = 1, 7x7 / 3x5 / 5x1 / 1x1 filters, Cout 5 (<8,1>), 12 and 24 (<8,4>), split output into a tensor-core FC
    ('conv_a', [('conv1', [5, 'conv', [7, 7]]), ('conv2', [12, 'conv', [3, 5]]), ('max1', [[2, 2], 'pool']),
                ('conv3', [6, 'conv', [5, 1]]), ('conv4', [24, 'conv', [1, 1]]), ('max2', [[3, 3], 'pool']),
                ('fc1', [64, 'fc']), ('fc2', [3, 'fc'])], (9, 11, 1)),
    ('conv_b', [('conv1', [5, 'conv', [1, 1]]), ('conv2', [6, 'conv', [5, 1]]), ('fc1', [72, 'fc']), ('fc2', [2, 'fc'])],
     (8, 6, 1)),
    ('conv_c', [('conv1', [12, 'conv', [3, 5]]), ('fc1', [136, 'fc']), ('fc2', [2, 'fc'])], (6, 5, 3)),
]

FC_NETS = [
    # K = 200 into N = 72 (split output), 136 (fp32 output) -> 56 and 264 on the CUDA cores (K = 136, 56) -> 328 on the
    # tensor cores again (K = 264): tensor-core -> CUDA-core -> tensor-core format changes
    ('fc_widths', [('conv1', [8, 'conv', [3, 3]]), ('fc1', [72, 'fc']), ('fc2', [136, 'fc']), ('fc3', [56, 'fc']),
                   ('fc4', [264, 'fc']), ('fc5', [328, 'fc']), ('fc6', [3, 'fc'])], (5, 5, 2)),
    # FC straight on the input (K = 72), all on the tensor cores; 264 and 136 write split planes through the tail
    ('fc_only', [('fc1', [64, 'fc']), ('fc2', [264, 'fc']), ('fc3', [136, 'fc']), ('fc4', [72, 'fc']),
                 ('fc5', [2, 'fc'])], (6, 12, 1)),
]
# layer_info(i)[2] with the tensor cores on: which layers the grid means to send through the tensor-core GEMM
EXPECT_TC = {'fc_widths': [0, 1, 1, 0, 0, 1, 0], 'fc_only': [1, 1, 1, 1, 0], 'conv_a': [0, 0, 0, 0, 0, 0, 1, 0],
             'conv_b': [0, 0, 1, 0],
             'conv_c': [0, 1, 0], 'big_window': [0, 0, 0, 0, 1, 0]}

# head_kernel<2>, <16>, <32>; d = 13 takes the scalar feature loop, d = 72 the float4 loop
HEAD_NETS = [('head_c%d_d%d' % (c, d), [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [d, 'fc']),
                                        ('fc2', [c, 'fc'])], (4, 4, 2))
             for c in (2, 3, 16, 17, 32) for d in (13, 72)]

FORWARD_NETS = POOL_NETS + [('big_window', BIG_WINDOW, (8, 7, 3))] + CONV_NETS + FC_NETS + HEAD_NETS

SHRUNK_NETS = [('shrunk_s3_c8', pool_net(3, 8, c=3), (7, 8, 2)),        # vec4 pool gradient, pad before in W
               ('shrunk_s5_c6', pool_net(5, 6, c=2), (14, 17, 2)),       # scalar pool gradient, pad before in W
               ('shrunk_s4_c8', pool_net(4, 8, c=2), (13, 10, 2)),       # pad before in H and W
               ('shrunk_big_window', BIG_WINDOW, (8, 7, 3))]


@pytest.fixture(scope='module')
def nb():
    import nnal_b200
    return nnal_b200


def _model(nb, layers, in_shape, w, dropout=None):
    m = nb.NN.CNN(in_shape, OrderedDict(layers), feature_layer=len(layers) - 2, dropout=dropout)
    m.set_weights(w)
    return m


def _centered(layers, in_shape, seed, x):
    """He-normal weights with the last bias shifted so that the binary posteriors of ``x`` straddle 0.5."""
    w = O.he_init_weights(layers, in_shape, seed, bias_scale=0.05)
    z = R.forward(layers, w, x)['logits']
    W, b = w[layers[-1][0]]
    med = np.median(z, axis=1)
    w[layers[-1][0]] = (W, b - (med - med.mean()).astype(np.float32).reshape(b.shape))
    return w


def _pool_pass(nb, layers, in_shape, w, x, tc, chunk=0):
    """posteriors [c, n], feature rows [n, d] and per-layer tensor-core use of one pool pass over host images."""
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, in_shape, w), None)
    eng.set_tensor_cores(tc)
    try:
        if chunk:
            eng.debug_option('chunk', chunk)
        n = x.shape[0]
        eng.pool_begin(n, keep=2)
        eng.pool_eval_images(x, 0)
        post = eng.pool_posteriors()
        feat = eng.pool_feature_rows(np.arange(n))
        uses = [eng.layer_info(i)[2] for i in range(len(layers))]
    finally:
        eng.debug_option('chunk', 0)
        eng.set_tensor_cores(1)
    return post, feat, uses


def _check(post, feat, ref):
    err = np.abs(post - ref['posteriors']).max()
    assert err < POST_TOL, 'posteriors off by %g' % err
    f = ref['feature'].T
    ferr = np.abs(feat - f).max()
    assert ferr <= FEAT_RTOL * np.abs(f).max(), 'feature rows off by %g (max %g)' % (ferr, np.abs(f).max())


@pytest.mark.parametrize('tc', [0, 1])
@pytest.mark.parametrize('name,layers,in_shape', FORWARD_NETS, ids=[a[0] for a in FORWARD_NETS])
def test_forward_grid(nb, name, layers, in_shape, tc):
    rs = np.random.RandomState(len(name) + 7 * in_shape[0])
    x = rs.randn(300, *in_shape).astype(np.float32)
    w = O.he_init_weights(layers, in_shape, 3 + in_shape[1], bias_scale=0.1)
    post, feat, uses = _pool_pass(nb, layers, in_shape, w, x, tc)
    if not tc:
        assert not any(uses)
    elif name.startswith('pool_'):
        assert uses[2] == 1, 'fc1 should run on the tensor cores (pool on split planes): %s' % uses
    elif name in EXPECT_TC:
        assert uses == EXPECT_TC[name]
    _check(post, feat, R.forward(layers, w, x))


@pytest.mark.parametrize('tc', [0, 1])
@pytest.mark.parametrize('s1,s2', [(3, 2), (2, 4)])
def test_pw1_with_wide_pools(nb, s1, s2, tc):
    """PW1 with max1 = 3x3 (25 -> 9, one padded row/column before) or max2 = 4x4 (13 -> 4, one before): the tensor-core
    conv output goes through the unfused split-plane pool."""
    layers = pw1_with_pools(s1, s2)
    rs = np.random.RandomState(10 * s1 + s2)
    x = rs.randn(96, 25, 25, 3).astype(np.float32)
    w = _centered(layers, (25, 25, 3), s1 + s2, x)
    ref = R.forward(layers, w, x)
    post, feat, uses = _pool_pass(nb, layers, (25, 25, 3), w, x, tc)
    if tc:
        assert uses[1] >= 1 and (uses[4] >= 1 or s1 != 2)       # conv2 (and conv4 at 13x13) on the tensor cores
    _check(post, feat, ref)


@pytest.mark.parametrize('name', ['pool_s3_c6_10x11', 'pool_s5_c8_11x14', 'fc_widths'])
def test_forward_ragged_chunks(nb, name):
    """777 samples in chunks of 200: the last chunk holds 177."""
    _, layers, in_shape = [n for n in FORWARD_NETS if n[0] == name][0]
    x = np.random.RandomState(5).randn(777, *in_shape).astype(np.float32)
    w = O.he_init_weights(layers, in_shape, 8, bias_scale=0.1)
    ref = R.forward(layers, w, x)
    post, feat, _ = _pool_pass(nb, layers, in_shape, w, x, 1, chunk=200)
    _check(post, feat, ref)
    post1, feat1, _ = _pool_pass(nb, layers, in_shape, w, x, 1)
    assert np.array_equal(post, post1) and np.array_equal(feat, feat1)


@pytest.mark.parametrize('N', [72, 136, 264, 328])
@pytest.mark.parametrize('K', [64, 72, 200])
@pytest.mark.parametrize('M', [1, 127, 129, 1000])
def test_fc_tail_widths_vs_f64(nb, M, N, K):
    """Isolated FC layer at widths of 8 mod 16 (the per-element tail of the tensor-core epilogue; 264 and 328 span
    two N tiles) and K not a multiple of 64, tensor cores and CUDA cores, against float64."""
    rs = np.random.RandomState(M + 3 * N + 7 * K)
    A = np.maximum(rs.randn(M, K), 0).astype(np.float32) * 3
    W = (rs.randn(N, K) * np.sqrt(2. / K)).astype(np.float32)
    b = (rs.randn(N) * .1).astype(np.float32)
    eng = nb.get_engine()
    for relu in (0, 1):
        ref = A.astype(np.float64) @ W.astype(np.float64).T + b
        if relu:
            ref = np.maximum(ref, 0)
        scale = np.abs(ref).max()
        for tc in (1, 0):
            got = eng.debug_fc(A, W, b, relu, tc)
            err = np.abs(got - ref).max()
            assert err < 2e-5 * scale, 'tc=%d relu=%d: off by %g of %g' % (tc, relu, err, scale)


MC_NET = [('conv1', [8, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [72, 'fc']), ('fc2', [136, 'fc']),
          ('fc3', [2, 'fc'])]


@pytest.mark.parametrize('keep', [0.5, 0.8])
def test_mc_dropout_tail_widths(nb, keep):
    """MC-dropout on a generic net whose dropped FC layers are 72 and 136 wide: every mask of the tensor-core epilogue's
    tail branch must match the Philox masks of the oracle (a wrong bit is an O(1) posterior error)."""
    in_shape, sites, seed, T = (6, 6, 2), [2, 3], 0x5eed1234abcd, 2
    x = np.random.RandomState(13).randn(257, *in_shape).astype(np.float32)
    w = _centered(MC_NET, in_shape, 14, x)
    eng = nb.get_engine()
    eng.set_model(_model(nb, MC_NET, in_shape, w, dropout=[sites, keep]), None)
    assert [eng.layer_info(i)[2] for i in range(len(MC_NET))] == [0, 0, 1, 1, 0]
    eng.set_dropout_seed(seed, first_pass=4)
    first = eng.pool_mc_config(T, keep, sites)
    try:
        eng.pool_begin(len(x))
        eng.pool_eval_images(x, 0)
    finally:
        eng.pool_mc_config(0, 1., [])
    av_post, _ = eng.pool_mc_means()
    last = eng.pool_posteriors()
    pos = np.arange(len(x))
    want = [M.forward_dropout(MC_NET, w, x, pos, keep, sites, seed, first + t)[1] for t in range(T)]
    assert np.abs(last - want[-1]).max() < POST_TOL
    assert np.abs(av_post - np.mean([p[1] for p in want], axis=0)).max() < POST_TOL
    det = R.forward(MC_NET, w, x)['posteriors']
    assert np.abs(want[-1] - det).max() > 1e-2                      # the masks matter


@pytest.mark.parametrize('tc', [1, 0])
@pytest.mark.parametrize('name,layers,in_shape', SHRUNK_NETS, ids=[a[0] for a in SHRUNK_NETS])
def test_shrunk_gradients_through_wide_pools(nb, name, layers, in_shape, tc):
    """Shrunk class-score gradients back through max-pools of window 3..5: the device routes each gradient to TF's
    window maximum, as the float64 oracle does."""
    from tests.test_gpu_sdp import _assert_shrunk_close
    rs = np.random.RandomState(len(name))
    x = rs.randn(120, *in_shape).astype(np.float32)
    w = O.he_init_weights(layers, in_shape, 21, bias_scale=0.1)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, in_shape, w), None)
    eng.set_tensor_cores(tc)
    try:
        post, g = eng.fi_shrunk_images(x)
    finally:
        eng.set_tensor_cores(1)
    po, go = O.shrunk_class_gradients(layers, w, x)
    assert np.abs(post - po).max() < POST_TOL
    _assert_shrunk_close(g[:, :, :-1], go[:, :, :-1])
    # The last layer's entry is (sum_j dz_j) (sum_k a_k + 1) / (d c + c) with sum_j dz_j = 1 - sum_j p_j: zero in exact
    # arithmetic, the float32 softmax's rounding on the device.  These nets have small gradients elsewhere, so it is
    # held to its own bound, 1e-6 >= |1 - sum_j p_j| for c <= 3 float32 posteriors, instead of to 1e-3 of the largest.
    a = O.forward(layers, w, x, keep_acts=True)['acts'][-1]['in']
    d, c = a.shape[0], go.shape[0]
    assert np.all(np.abs(g[:, :, -1]) <= 1e-6 * (np.abs(a).sum(axis=0) + 1) / (d * c + c))


def test_more_than_32_classes_is_an_error(nb):
    layers = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [16, 'fc']), ('fc2', [33, 'fc'])]
    w = O.he_init_weights(layers, (4, 4, 2), 1)
    x = np.random.RandomState(1).randn(5, 4, 4, 2).astype(np.float32)
    eng = nb.get_engine()
    with pytest.raises(nb._lib.NnalError):
        eng.set_model(_model(nb, layers, (4, 4, 2), w), None)
        eng.pool_begin(5)
        eng.pool_eval_images(x, 0)


@pytest.mark.parametrize('tc', [0, 1])
def test_conv_tile_beyond_shared_memory_is_an_error(nb, tc):
    """40x40x32 input, 3x3 filter: the padded input tile of the CUDA-core conv is 42*42*32*4 bytes > 200 KB."""
    layers = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [8, 'fc']), ('fc2', [2, 'fc'])]
    w = O.he_init_weights(layers, (40, 40, 32), 2)
    x = np.random.RandomState(2).randn(2, 40, 40, 32).astype(np.float32)
    eng = nb.get_engine()
    eng.set_model(_model(nb, layers, (40, 40, 32), w), None)
    eng.set_tensor_cores(tc)
    try:
        eng.pool_begin(2)
        with pytest.raises(nb._lib.NnalError, match='shared memory'):
            eng.pool_eval_images(x, 0)
    finally:
        eng.set_tensor_cores(1)
