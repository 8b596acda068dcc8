"""GPU tests of the tensor-core GEMM (``fc_tc_pair_kernel``, csrc/gemm_tc.cu) and its callers in the regimes where
state carries over from one pair tile or one chunk to the next (``pytest -m gpu``).

The kernel runs persistent CTA pairs: at most 74 on a B200, each walking the pair tiles t = pair, pair + npairs, ...
in column bands of NBAND column blocks.  The shared-memory ring phase, the accumulator parity (the two TMEM
accumulators alternate once per chunk of CHUNK_KB k-blocks) and the accumulator-empty barrier all carry over from a
pair's tile to its next one.  Its callers cut their work into chunks: the FI Gram into chunks of 65,536 candidates,
added into H with ``accum``; the cosine-similarity passes into chunks of 32,768 pool rows and 2,048 labelled columns.
Every check here runs past those boundaries and compares with a float64 product that does not use this library
(NumPy, or torch float64 on the device for the large products).  Each shape asserts the regime it is there for from
the tile arithmetic, so that a later edit cannot silently shrink it."""
from collections import OrderedDict
from types import SimpleNamespace

import numpy as np
import pytest

import oracle as O

pytestmark = pytest.mark.gpu

# csrc/gemm_tc.cu: rows per CTA, rows per pair tile, columns per tile, k-block, band width in column blocks, k-blocks
# per accumulator chunk
BM, PAIR_M, BN, BK, NBAND, CHUNK_KB = 128, 256, 256, 64, 8, 8
MAX_PAIRS = 74                     # 148 SMs in clusters of 2: the most pairs cudaOccupancyMaxActiveClusters can report
PAIR_COUNTS = range(32, MAX_PAIRS + 1)   # pair counts a B200 grid of this kernel can have
GRAM_CH = 65536                    # csrc/fi.cu gram_core: candidates per Gram GEMM
ROW_CHUNK, CB = 32768, 2048        # csrc/sims.cu: pool rows per similarity GEMM, labelled columns per nnal_cross_sims GEMM


def cdiv(a, b):
    return -(-a // b)


def regime(M, N, K):
    """Tile arithmetic of fc_tc_pair_kernel for out[M][N] = A[M][K] . B[N][K]^T."""
    mblocks, nblocks, num_kb = cdiv(M, PAIR_M), cdiv(N, BN), cdiv(K, BK)
    return SimpleNamespace(mblocks=mblocks, nblocks=nblocks, ntiles=mblocks * nblocks, num_kb=num_kb,
                           chunks=cdiv(num_kb, CHUNK_KB), k_tail=K % BK,
                           bands=[min(NBAND, nblocks - b) for b in range(0, nblocks, NBAND)],
                           last_rows=M - (mblocks - 1) * PAIR_M, last_cols=N - (nblocks - 1) * BN)


def tile_index(m_blk, n_blk, mblocks, nblocks):
    """Index t of the pair tile (m_blk, n_blk) in the kernel's band order (the inverse of its tile_blocks)."""
    b = n_blk // NBAND
    wb = min(NBAND, nblocks - b * NBAND)
    return b * mblocks * NBAND + m_blk * wb + n_blk - b * NBAND


def worst_tile(err):
    """'pair tile t (row block, column block): max error' of the pair tile holding the largest entry of err [M, N]
    (a torch tensor)."""
    M, N = err.shape
    mb, nb_ = cdiv(M, PAIR_M), cdiv(N, BN)
    pad = err.new_zeros(mb * PAIR_M, nb_ * BN)
    pad[:M, :N] = err
    per = pad.reshape(mb, PAIR_M, nb_, BN).amax(dim=(1, 3))
    m, n = divmod(int(per.argmax()), nb_)
    return 'pair tile %d (row block %d, column block %d): %.3g' % (tile_index(m, n, mb, nb_), m, n, float(per[m, n]))


def rotate_blocks(X, blocks, size, axis=0):
    """X with its whole blocks of ``size`` along ``axis`` rotated by ``blocks`` blocks; a partial last block stays where
    it is, so every row (column) keeps its position inside its tile."""
    X = np.asarray(X)
    full = X.shape[axis] // size * size
    head, tail = np.split(X, [full], axis=axis)
    return np.concatenate([np.roll(head, blocks * size, axis=axis), tail], axis=axis)


def _device():
    import torch
    return 'cuda' if torch.cuda.is_available() else 'cpu'


def f64(a):
    import torch
    return torch.as_tensor(np.asarray(a)).to(_device(), torch.float64)


@pytest.fixture(scope='module')
def nb():
    import nnal_b200
    return nnal_b200


@pytest.fixture(scope='module')
def eng(nb):
    return nb.get_engine()


# ------------------------------------------------------------------ 1. FC GEMM, many tiles per pair, against float64
def fc_operands(M, N, K, seed):
    """Post-ReLU-like activations and He-scaled weights (the operands of test_gpu_parity.test_fc_tcgen05_vs_f64)."""
    rng = np.random.default_rng(seed)
    A = rng.standard_normal((M, K), dtype=np.float32)
    np.maximum(A, 0, out=A)
    A *= 3
    W = rng.standard_normal((N, K), dtype=np.float32) * np.float32(np.sqrt(2. / K))
    b = rng.standard_normal(N, dtype=np.float32) * np.float32(.1)
    return A, W, b


FC_CASES = [
    # bands 8 + 2; the last column block holds 8 columns (the epilogue's per-element tail); K tail of 8; 17 k-blocks =
    # 3 chunks, so consecutive tiles of one pair start on alternate accumulators; the last pair holds 32 leader rows
    # and no peer rows
    ((20000, 2312, 1032), lambda r: (r.bands == [8, 2] and r.last_cols == 8 and r.k_tail == 8 and r.chunks == 3
                                     and r.last_rows == 32)),
    # PW1 fc1 on one pool chunk: 1,024 tiles, 10 chunks (the last one of 2 k-blocks)
    ((16384, 4096, 4704), lambda r: r.ntiles == 1024 and r.chunks == 10 and r.num_kb % CHUNK_KB == 2),
    # PW1 fc2: exactly 8 chunks
    ((16384, 4096, 4096), lambda r: r.ntiles == 1024 and r.num_kb == 8 * CHUNK_KB),
    # 50 x 18 tiles in bands 8 + 8 + 2: one k-block per tile (the accumulator switches every tile), exactly one full
    # chunk, and a chunk of 8 plus a chunk of 1
    ((12800, 4608, 64), lambda r: r.bands == [8, 8, 2] and r.num_kb == 1),
    ((12800, 4608, 512), lambda r: r.bands == [8, 8, 2] and r.num_kb == CHUNK_KB),
    ((12800, 4608, 520), lambda r: r.bands == [8, 8, 2] and r.num_kb == CHUNK_KB + 1),
]


@pytest.mark.parametrize('shape,check', FC_CASES, ids=['%dx%dx%d' % s for s, _ in FC_CASES])
def test_fc_many_tiles_per_pair_vs_f64(eng, shape, check):
    """debug_fc at >= 10 pair tiles on every pair, ReLU off and on, tensor cores and CUDA cores, within 2e-5 of max|ref|
    of the float64 product."""
    import torch
    M, N, K = shape
    r = regime(M, N, K)
    assert r.ntiles >= 10 * MAX_PAIRS and check(r), r
    A, W, b = fc_operands(M, N, K, M + N + K)
    ref0 = f64(A) @ f64(W).T + f64(b)
    for relu in (0, 1):
        ref = ref0.clamp_min(0) if relu else ref0
        scale = float(ref.abs().max())
        for tc in (1, 0):
            err = (torch.from_numpy(eng.debug_fc(A, W, b, relu, tc)).to(ref.device, torch.float64) - ref).abs_()
            e = float(err.max())
            assert e < 2e-5 * scale, 'tc=%d relu=%d: off by %.3g of %.3g, worst %s' % (tc, relu, e, scale, worst_tile(err))


# ------------------------------------------------------------------ 2. tile placement must not change a single bit
PLACEMENT_CASES = [(20000, 2312, 1032), (12800, 4608, 64)]


@pytest.mark.parametrize('shape', PLACEMENT_CASES, ids=['%dx%dx%d' % s for s in PLACEMENT_CASES])
def test_fc_tile_placement_bit_exact(eng, shape):
    """Every output element gets the same MMA sequence whatever pair tile computes it (DESIGN §3).  Rotating A's whole
    row blocks by 1 and 3 pair tiles moves each tile's index t by wb or 3 wb inside its band; rotating W and b by one
    column block moves t by 1 and carries column blocks across band boundaries.  Either changes which pair, which
    wave, which accumulator and which band computes every tile while each row and column keeps its position inside
    the tile: the un-rotated output must be bit-equal to the plain call, and so must a repeated plain call."""
    import torch
    M, N, K = shape
    r = regime(M, N, K)
    # an odd number of chunks per tile: a pair's consecutive tiles start on alternate accumulators
    assert r.ntiles >= 10 * MAX_PAIRS and r.chunks % 2 == 1 and len(r.bands) > 1, r
    A, W, b = fc_operands(M, N, K, 3 * M + N)
    base = eng.debug_fc(A, W, b, 0, 1)

    def check(got, what):
        diff = got != base
        if diff.any():
            err = torch.from_numpy(np.abs(got.astype(np.float64) - base))
            pytest.fail('%s: %d elements differ, worst %s' % (what, int(diff.sum()), worst_tile(err)))

    check(eng.debug_fc(A, W, b, 0, 1), 'repeated call')
    for rb in (1, 3):
        # no grid of this kernel on a B200 maps a tile moved by rb * wb back onto its own pair
        assert all((rb * wb) % P for wb in r.bands for P in PAIR_COUNTS)
        got = eng.debug_fc(rotate_blocks(A, rb, PAIR_M), W, b, 0, 1)
        check(rotate_blocks(got, -rb, PAIR_M), 'A rotated by %d pair tiles' % rb)
    got = eng.debug_fc(A, rotate_blocks(W, 1, BN), rotate_blocks(b, 1, BN), 0, 1)
    check(rotate_blocks(got, -1, BN, axis=1), 'W and b rotated by one column block')


# ------------------------------------------------------------------ 3. FI Gram across candidate chunks
def gram_factors(n, d, seed):
    """The one-layer factors of test_gpu_fi._factors (u = 2 relu(N(0, 1)), p1 uniform with 1e-9, 1 - 1e-9 and 0.5
    first), drawn with NumPy's PCG64 generator, which is several times faster at these sizes."""
    rng = np.random.default_rng(seed)
    U = rng.standard_normal((n, d), dtype=np.float32)
    np.maximum(U, 0, out=U)
    U *= 2
    p1 = rng.random(n)
    p1[:3] = [1e-9, 1 - 1e-9, 0.5]
    return p1, U


def f64_gram(U, wq, rows=None):
    """Ut^T diag(wq) Ut, Ut = [U 1] (rows ``rows`` of U), float64 on the device."""
    import torch
    Ut = f64(U if rows is None else U[rows])
    Ut = torch.cat([Ut, Ut.new_ones(Ut.shape[0], 1)], dim=1)
    return (Ut * f64(wq)[:, None]).T @ Ut


def assert_gram(H, ref, what):
    import torch
    err = (torch.from_numpy(H).to(ref.device, torch.float64) - ref).abs_()
    scale = float(ref.abs().max())
    assert float(err.max()) < 1e-5 * scale, '%s: off by %.3g of %.3g, worst %s' % (what, float(err.max()), scale,
                                                                                 worst_tile(err))


@pytest.fixture(scope='module')
def factors_70k():
    return gram_factors(70000, 2311, 70)


GRAM_CASES = [
    # Dg = 2312: 10 x 10 tiles, bands 8 + 2, an 8-column tail; the second chunk of 4,464 candidates has a K tail of 48
    (70000, 2311, lambda r: r.ntiles == 100 and r.bands == [8, 2] and r.last_cols == 8 and r.k_tail == 48),
    # the bench's Gram, Dg = 4097: 289 tiles, bands 8 + 8 + 1, a 1-column tail and a last row block of one row
    (66000, 4096, lambda r: r.ntiles == 289 and r.bands == [8, 8, 1] and r.last_cols == 1 and r.last_rows == 1),
]


@pytest.mark.parametrize('n,d,check', GRAM_CASES, ids=['n%d-d%d' % (n, d) for n, d, _ in GRAM_CASES])
def test_gram_across_candidate_chunks(eng, factors_70k, n, d, check):
    """fi_gram over two candidate chunks: the second one is added into H with ``accum`` by the float4 epilogue and by
    its per-element column tail.  q = None and a Dirichlet q, within 1e-5 of max|H| of float64 Ut^T diag(wq) Ut."""
    r = regime(d + 1, d + 1, n - GRAM_CH)          # the tiles of the second (accumulating) chunk
    assert cdiv(n, GRAM_CH) == 2 and r.last_cols % 16 != 0 and check(r), r
    p1, U = factors_70k if (n, d) == (70000, 2311) else gram_factors(n, d, n + d)
    eng.fi_set_factors(p1, U)
    w = p1 * (1 - p1)
    for q in (None, np.random.RandomState(n).dirichlet(np.ones(n))):
        H = eng.fi_gram(q)
        assert H.shape == (d + 1, d + 1)
        assert_gram(H, f64_gram(U, (np.full(n, 1. / n) if q is None else q) * w), 'q=%s' % ('None' if q is None else 'dirichlet'))


def test_gram_subset_across_candidate_chunks_and_solve(eng, factors_70k):
    """fi_gram_subset over 66,000 shuffled candidates of the 70,000 (two chunks, so the second one reads its factor
    rows through the ``rows[i]`` indirection), then fi_gram_solve on that Gram against NumPy, as
    test_gpu_fi.test_fi_gram_subset_and_solve does at d <= 320."""
    import torch
    from nnal_b200 import dist
    p1, U = factors_70k
    n, d = U.shape
    rs = np.random.RandomState(9)
    S = rs.permutation(n)[:66000]
    assert cdiv(len(S), GRAM_CH) == 2 and regime(d + 1, d + 1, len(S) - GRAM_CH).k_tail
    q = rs.dirichlet(np.ones(len(S)))
    w = p1 * (1 - p1)
    eng.fi_set_factors(p1, U)
    Hp = eng.fi_gram(None)                                       # pool-wide Gram: the second operand of the FI ratio
    ptr, rows, ld = eng.fi_gram_device()
    G2 = dist.device_view(ptr, (rows * ld,), '<f4').clone()
    torch.cuda.synchronize()
    Hs = eng.fi_gram_subset(S, q, read=True)
    assert_gram(Hs, f64_gram(U, q * w[S], rows=S), 'subset')
    for delta in (1e-2, 1e-3):
        tr, ratio = eng.fi_gram_solve(delta, 2.0, G2.data_ptr())
        Minv = np.linalg.inv(delta * np.eye(d + 1) + 2. * Hs.astype(np.float64))
        assert abs(tr / np.trace(Minv) - 1) < 1e-9                # same float32 Gram in, float64 arithmetic
        want = np.sum(Minv * (delta * np.eye(d + 1) + 2. * Hp.astype(np.float64)))
        assert abs(ratio / want - 1) < 1e-8


# ------------------------------------------------------------------ 4. similarity GEMMs past ROW_CHUNK and CB
SIM_NET = [('conv1', [8, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [200, 'fc']), ('fc2', [2, 'fc'])]
SIM_IN = (8, 8, 2)
N_POOL = 70000                     # row chunks of 32,768 + 32,768 + 4,464
ZERO_ROWS = [40000, 68000]         # zero feature rows in the second and third row chunk


@pytest.fixture(scope='module')
def sim_pool(nb, eng):
    """Pool pass of N_POOL whole images keeping the feature layer fc1 (d = 200: a K tail); the images at ZERO_ROWS
    are zero, and with conv1 bias 0 and fc1 bias <= 0 their feature rows are exactly zero.  Returns the device's
    features [d, n]: the similarity passes are checked on them, apart from the forward."""
    assert N_POOL > 2 * ROW_CHUNK and N_POOL % ROW_CHUNK and [z // ROW_CHUNK for z in ZERO_ROWS] == [1, 2]
    rs = np.random.RandomState(31)
    x = rs.rand(N_POOL, *SIM_IN).astype(np.float32)
    x[ZERO_ROWS] = 0
    w = O.he_init_weights(SIM_NET, SIM_IN, 32, bias_scale=0.1)
    w['conv1'] = (w['conv1'][0], np.zeros_like(w['conv1'][1]))
    w['fc1'] = (w['fc1'][0], -np.abs(w['fc1'][1]))
    model = nb.NN.CNN(SIM_IN, OrderedDict(SIM_NET), feature_layer=2)
    model.set_weights(w)
    eng.set_model(model)
    eng.pool_begin(N_POOL, 1)
    eng.pool_eval_images(x, 0)
    F = eng.pool_features()
    assert F.shape == (200, N_POOL) and F.shape[0] % BK
    assert np.flatnonzero(~F.any(axis=0)).tolist() == ZERO_ROWS
    return F


def _live():
    return np.setdiff1d(np.arange(N_POOL), ZERO_ROWS)


def test_rep_greedy_past_row_chunks(eng, sim_pool):
    """rep_set on 301 columns (ldB = 304: the second N block ends in a per-element column tail) taken from all three
    row chunks and excluded as rows, then rep_greedy(25): every pick within 1e-4 of the best available facility-location
    score on float64 cosine sims of the remaining non-zero rows, and the reported values equal to the replayed scores
    to 1e-4."""
    F = sim_pool
    live = _live()
    rs = np.random.RandomState(5)
    pos = np.concatenate([rs.choice(live[(live >= a) & (live < b)], m, replace=False)
                          for a, b, m in [(0, ROW_CHUNK, 100), (ROW_CHUNK, 2 * ROW_CHUNK, 100), (2 * ROW_CHUNK, N_POOL, 101)]])
    B = len(pos)
    r = regime(N_POOL - 2 * ROW_CHUNK, B, F.shape[0])
    assert B == 301 and cdiv(B, 8) * 8 == 304 and r.nblocks == 2 and r.last_cols % 16, r
    cols = eng.pool_feature_rows(pos)
    assert np.array_equal(cols, F[:, pos].T)
    eng.rep_set(cols, pos, 25)
    sel, val = eng.rep_greedy(25)
    assert len(np.unique(sel)) == 25
    rows = np.setdiff1d(live, pos)
    sims = O.cosine_sims(F[:, rows].astype(np.float64), cols.T.astype(np.float64))
    rep = O.facility_location_replay(sims, sel)
    assert np.all(rep[:, 0] >= rep[:, 1] - 1e-4 * np.abs(rep[:, 1])), 'picked a column clearly worse than the best'
    assert np.allclose(val, rep[:, 0], rtol=1e-4, atol=0), np.abs(val / rep[:, 0] - 1).max()


def test_cross_sims_and_kcenter_past_chunks(eng, sim_pool):
    """cross_sims with 4,500 labelled rows (column chunks 2,048 + 2,048 + 404) over three row chunks against
    O.get_cross_sims within 2e-6 on every non-zero row; zero rows read +inf (never selected).  Then the k-center
    greedy from those similarities: picks valid under O.kcenter_replay (1e-5), never a zero row."""
    F = sim_pool
    live = _live()
    rs = np.random.RandomState(6)
    T = F[:, rs.choice(live, 4500, replace=False)]
    assert cdiv(T.shape[1], CB) == 3 and T.shape[1] % CB == 404
    sims = eng.cross_sims(np.ascontiguousarray(T.T))
    T64 = T.astype(np.float64)
    ref = np.concatenate([O.get_cross_sims(F[:, blk].astype(np.float64), T64) for blk in np.array_split(live, 16)])
    err = np.abs(sims[live] - ref)
    i = int(np.argmax(err))
    assert err[i] < 2e-6, 'row %d (row chunk %d): off by %.3g' % (live[i], live[i] // ROW_CHUNK, err[i])
    assert np.all(sims[ZERO_ROWS] == np.inf)
    eng.cs_begin(2, None, None, 20)
    sel, val = eng.cs_greedy(20)
    assert len(np.unique(sel)) == 20 and not np.isin(sel, ZERO_ROWS).any()
    compact = np.full(N_POOL, -1)
    compact[live] = np.arange(len(live))
    rep = O.kcenter_replay(F[:, live].astype(np.float64), ref, compact[sel])
    assert np.all(rep[:, 0] <= rep[:, 1] + 1e-5), 'picked a sample clearly more similar than the least similar one'
    assert np.allclose(val, rep[:, 0], rtol=0, atol=1e-5)
