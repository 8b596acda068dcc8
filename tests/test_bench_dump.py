"""bench.py --dump-outputs: the last timed step's outputs land in DIR as float32 / float64 .npy files that agree with each
other (the entropy answer is the top-k of the dumped posteriors, the FI answer lies inside the pre-filter), are identical
for two runs with the same arguments, and stay within the byte budget when the pool posteriors have to be sampled."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.util import assert_topk_equivalent

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
K = 100


def _run(out, *args):
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--dump-outputs', out] + list(args)
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=900, env=dict(os.environ, OMP_NUM_THREADS='4'))
    assert r.returncode == 0, r.stdout.decode()[-3000:]
    got = {f[:-4]: np.load(os.path.join(out, f)) for f in sorted(os.listdir(out))}
    for v in got.values():
        assert v.dtype in (np.float32, np.float64)
    return got


def test_dump_outputs_reference_arm(tmp_path):
    """Reference arm, 1000-sample pool, FI pre-filter B = 200: the dump is the step's own answer."""
    args = ['--impl', 'reference', '--steps', '1', '--warmup', '0', '--cpu-sample', '1000', '--pool', '1000', '--fi-B', '200']
    a = _run(str(tmp_path / 'a'), *args)
    assert sorted(a) == ['entropy_query', 'fi_query', 'pool_positions', 'pool_posteriors_class1']
    assert np.array_equal(a['pool_positions'], np.arange(1000))
    p1 = a['pool_posteriors_class1']
    assert p1.shape == (1000,) and ((p1 >= 0) & (p1 <= 1)).all()
    order = np.argsort(np.abs(p1 - .5), kind='stable')
    assert np.array_equal(a['entropy_query'], order[:K])
    fi = a['fi_query'].astype(np.int64)
    assert len(fi) == K and len(np.unique(fi)) == K and np.isin(fi, order[:200]).all()
    b = _run(str(tmp_path / 'b'), *args)
    assert sorted(b) == sorted(a)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize('shape,dtype,lo', [((2, 9000000), np.float32, 0), ((5000000,), np.float64, 123)])
def test_dump_outputs_samples_large_pool(tmp_path, shape, dtype, lo):
    """Pool posteriors larger than the budget: a fixed seeded sample of columns, as many as fit next to the other arrays."""
    import bench
    n = shape[-1]
    post = np.arange(n, dtype=dtype)                       # column j holds j (and -j): a sampled column shows where it came from
    if len(shape) == 2:
        post = np.stack([post, -post])
    small = {'entropy_query': np.arange(K), 'fi_objective': np.linspace(0, 1, K)}
    for rep in ('a', 'b'):
        out = str(tmp_path / rep)
        bench.dump_outputs(out, small, post, 'pool_posteriors', lo)
        files = {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}
        assert sum(os.path.getsize(os.path.join(out, f)) for f in os.listdir(out)) <= 64e6
        pos = files['pool_positions']
        m = len(pos)
        per_col = 8 + np.dtype(dtype).itemsize * (shape[0] if len(shape) > 1 else 1)
        assert 64e6 - per_col - 1e4 < sum(a.nbytes for a in files.values()) and m < n           # the budget is used
        assert pos.dtype == np.float64 and (np.diff(pos) > 0).all() and pos[0] >= lo and pos[-1] < lo + n
        cols = pos.astype(np.int64) - lo
        assert files['pool_posteriors'].dtype == dtype and files['pool_posteriors'].shape == shape[:-1] + (m,)
        assert np.array_equal(files['pool_posteriors'], post[..., cols])
        assert np.array_equal(files['entropy_query'], np.arange(K, dtype=np.float64))
        if rep == 'a':
            first = files
    for k in first:
        assert np.array_equal(first[k], files[k]), k


@pytest.mark.gpu
def test_dump_outputs_device_arm(tmp_path):
    """Device arm (the timed path of the headline), 20,000-sample pool, FI pre-filter B = 2,000, extras off."""
    a = _run(str(tmp_path / 'a'), '--gpus', '1', '--steps', '2', '--warmup', '1', '--pool', '20000', '--fi-B', '2000',
             '--no-cpu', '--sdp-B', '0', '--mc-T', '0', '--config4-slices', '0', '--strong-pool', '0')
    assert sorted(a) == ['entropy_query', 'fi_objective', 'fi_query', 'fi_reduced_objective', 'pool_positions',
                         'pool_posteriors']
    assert np.array_equal(a['pool_positions'], np.arange(20000))
    post = a['pool_posteriors']
    assert post.dtype == np.float32 and post.shape == (2, 20000)
    assert np.allclose(post.sum(0), 1, atol=1e-5)
    score = np.abs(post[1].astype(np.float64) - .5)
    assert_topk_equivalent(a['entropy_query'].astype(np.int64), score, K, 1e-6)
    fi = a['fi_query'].astype(np.int64)
    assert len(fi) == K and len(np.unique(fi)) == K
    assert (score[fi] <= np.sort(score)[1999] + 1e-6).all()                   # inside the pre-filter
    assert a['fi_objective'].shape == a['fi_reduced_objective'].shape == (K,)
    assert np.isfinite(a['fi_objective']).all() and np.isfinite(a['fi_reduced_objective']).all()
