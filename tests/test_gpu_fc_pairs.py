"""GPU tests of the tensor-core FC GEMM's CTA pairs (``pytest -m gpu``).

A pair of CTAs computes a 256-row tile: the leader CTA owns rows 0..127 and its peer rows 128..255, and rows past M
are zero-filled by TMA and never stored.  A row's output must therefore not depend on where it lands in a pair.
debug_fc on A and on A with s extra rows put in front (s = 1, 128, 255 move every row across the leader / peer
boundary) must return bit-equal outputs for A's rows.  The base M leave the last pair full (512), half full (384),
holding a single row (257), and a lone leader with no peer rows at all (50); N = 328 and K = 200 add the epilogue's
per-element column tail and a K tail."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def eng():
    import nnal_b200
    return nnal_b200.get_engine()


@pytest.mark.parametrize('M', [512, 384, 257, 50])
@pytest.mark.parametrize('N,K', [(256, 128), (328, 200)])
def test_fc_row_independent_of_pair_position(eng, M, N, K):
    rs = np.random.RandomState(M + N + K)
    A = np.maximum(rs.randn(M, K), 0).astype(np.float32) * 3
    W = (rs.randn(N, K) * np.sqrt(2. / K)).astype(np.float32)
    b = (rs.randn(N) * .1).astype(np.float32)
    ref = eng.debug_fc(A, W, b, 1, 1)
    assert np.all(np.isfinite(ref)) and np.abs(ref).max() > 0
    for s in (1, 128, 255):
        front = np.maximum(rs.randn(s, K), 0).astype(np.float32) * 3
        got = eng.debug_fc(np.concatenate([front, A]), W, b, 1, 1)
        assert np.array_equal(got[s:], ref), 'shift %d: max difference %g' % (s, np.abs(got[s:] - ref).max())
