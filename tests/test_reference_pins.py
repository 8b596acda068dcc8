"""Pins of the oracle against the UNMODIFIED reference (the original nn-active-learning sources) -- NumPy helpers, the
query dispatch over a fake TF session / fake cvxopt, the SDP programme.  oracle/check_against_reference.py runs them
against a reference tree and stores what the reference computed in tests/golden/.

The suite is self-contained: the oracle must reproduce every stored reference output (here, and in test_oracle.py,
test_oracle_sdp.py and test_reference_dispatch_golden.py).  With a reference tree at $NNAL_REFERENCE,
test_pins_hold_and_goldens_are_current also re-executes every pin against it and requires the goldens it would write to
equal the committed ones.  Only that test covers the pins whose reference outputs were never stored: NN.LLFC_grads /
NN.LLFC_hess, NNAL_tools.FC_gradnorms_batch, the 'random' queries (drop-in host code against the reference's under the
same np.random state) and the single-volume CNN_query 'MC-entropy' == 'entropy' identity.  Without the reference tree
those pins are not checked against the reference; the oracle's LLFC and FC-gradient-norm functions are still checked
against autograd and their defining identities in test_oracle.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

import oracle as O
from tests.test_reference_dispatch_golden import LAYERS, LAYERS_W, M, PS, _case

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('NNAL_REFERENCE')


def test_unpadded_masked_gather_reproduces_stored_reference(golden):
    """patch_utils.get_patches on UNPADDED volumes with a label mask (gather*_labels): the inputs are regenerated from the
    generator's RandomState(10) stream, checked against the stored padded volumes and indices, then gathered."""
    rs = np.random.RandomState(10)
    cases = [((9, 8, 5), (3, 3, 1), 2, np.float32), ((11, 10, 7), (5, 3, 3), 3, np.float64),
             ((30, 29, 6), (25, 25, 1), 3, np.float32), ((6, 6, 6), (1, 1, 1), 1, np.int16)]
    for ci, (shape, ps, m, dt) in enumerate(cases):
        rads = [(p - 1) // 2 for p in ps]
        imgs = [(rs.randn(*shape) * 50 + 100).astype(dt) for _ in range(m)]
        mask = (rs.rand(*shape) > .5).astype(np.int32)
        inds = rs.choice(int(np.prod(shape)), 17, replace=False)
        inds[:4] = [0, np.prod(shape) - 1, shape[2] - 1, shape[1] * shape[2]]
        padded = np.stack([np.pad(im, tuple((r, r) for r in rads), 'constant') for im in imgs])
        assert np.array_equal(padded, golden['gather%d_imgs' % ci]) and np.array_equal(inds, golden['gather%d_inds' % ci])
        out, labels = O.get_patches(imgs, inds, ps, False, mask)
        assert np.array_equal(out, golden['gather%d_out' % ci]), ci
        assert np.array_equal(labels, golden['gather%d_labels' % ci]), ci


def test_oracle_reproduces_stored_reference_outputs(golden):
    """Stored reference outputs the other CPU tests do not replay: PW_NNAL.stoch_approx_IF (LiSSA through the last FC
    layer, seeded draws) and the single-volume 'fi' branch of PW_NNAL.CNN_query with lambda_ > 0."""
    w = O.he_init_weights(LAYERS_W, (9, 7, 2), 6, bias_scale=0.1)
    r = O.forward(LAYERS_W, w, golden['w_pool'], feature_layer=len(LAYERS_W) - 2)
    V, labels = O.stoch_approx_IF(r['posteriors'][:, 40:47], r['feature_layer'][:, 40:47], r['posteriors'][:, :12],
                                  r['feature_layer'][:, :12], list(golden['if_draws']), 20.)
    assert np.array_equal(labels, golden['if_labels'])
    assert V.shape == golden['if_V'].shape
    assert np.allclose(V, golden['if_V'], rtol=1e-10, atol=1e-12 * np.abs(V).max())
    w, allp, pools, st, stats0 = _case(golden)
    q, _ = O.query_fi_sdp_single(LAYERS, w, allp[0][:M], np.array(pools[0]), PS, 16, stats0, 9, 30, golden['q_fi_u'],
                                 diag_load=1e-5, lambda_=0.2)
    assert np.array_equal(q, golden['q_fi_sdp_single_lambda'])


@pytest.mark.skipif(not REF or not os.path.isdir(REF), reason='no reference tree at $NNAL_REFERENCE')
def test_pins_hold_and_goldens_are_current(tmp_path, golden):
    env = dict(os.environ, NNAL_GOLD_OUT=str(tmp_path), OMP_NUM_THREADS='2')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'oracle', 'check_against_reference.py')], env=env,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900)
    out = r.stdout.decode()
    assert r.returncode == 0, out[-3000:]
    for needle in ('get_patches: oracle == reference', "PW_NNAL.CNN_query 'fi'", "query_multimg 'MC-entropy' / 'BALD'",
                   "NNAL.CNN_query 'entropy' / 'rep-entropy' / 'fi'", 'SDP_query_distribution / inequality_cvx_matrix',
                   'LLFC_grads / LLFC_hess'):
        assert needle in out, needle
    fresh = np.load(os.path.join(str(tmp_path), 'reference_numpy_helpers.npz'))
    assert sorted(fresh.files) == sorted(golden.files)
    for k in fresh.files:
        assert np.array_equal(fresh[k], golden[k]), k
