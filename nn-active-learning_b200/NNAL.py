"""Drop-in for ``NNAL.CNN_query`` (whole-image active learning, NNAL.py:188-525)."""
import numpy as np

from . import _lib as L
from . import dist
from .engine import get_engine


def _pool_images(expr, pool_inds):
    """The reference loads pool images from disk with NN.load_winds (NN.py:1479-1527, broken
    upstream: cv2 import is commented out).  The drop-in reads them from ``expr.pool_images``
    (float array ``[N,H,W,C]``, already mean-subtracted) or ``expr.load_pool(inds)``."""
    if hasattr(expr, 'load_pool'):
        return np.asarray(expr.load_pool(pool_inds), dtype=np.float32)
    return np.asarray(expr.pool_images[np.asarray(pool_inds)], dtype=np.float32)


def _posteriors_on_device(model, expr, pool_inds, session, keep=0):
    eng = get_engine()
    eng.set_model(model, session)
    pool_inds = np.asarray(pool_inds)
    n = len(pool_inds)
    rank, world = dist.rank_world()
    b = dist.shard_bounds(n, world)
    lo, hi = int(b[rank]), int(b[rank + 1])
    eng.pool_begin(hi - lo, keep)
    eng.pool_eval_images(_pool_images(expr, pool_inds[lo:hi]), 0)
    return eng, lo, hi


def CNN_query(model, expr, pool_inds, method_name, session, col=True, extra_feed_dict={}):
    """NNAL.CNN_query (NNAL.py:188-525): returns positions into ``pool_inds``.

    ``entropy``: posteriors ``[c,n]`` -> compute_entropy (zeros -> 1e-7) -> argsort(-H)[:k]
    (NNAL.py:298-310).  ``fi``: see ``nnal_b200.fi.query_whole``; ``expr.pars['fi_mode'] = 'sdp'`` runs the reference's
    own multiclass A-matrix + SDP + sampling pipeline (``nnal_b200.fi.query_whole_sdp``); ``'block-greedy'`` runs the greedy
    last-layer FI selection for any number of classes (``nnal_b200.fi.query_whole_block``)."""
    k = expr.pars['k']
    if method_name == 'random':
        return np.random.permutation(len(pool_inds))[:k]
    if len(extra_feed_dict) > 0:
        raise NotImplementedError('extra_feed_dict is not part of the replaced path')
    if method_name == 'entropy':
        eng, lo, hi = _posteriors_on_device(model, expr, pool_inds, session)
        eng.pool_score(L.SCORE_NEG_ENTROPY, 10e-8)
        q, _ = dist.topk_global(eng, k, lo, len(pool_inds))
        return q
    if method_name == 'fi':
        from . import fi
        if expr.pars.get('fi_mode', 'greedy') == 'sdp':
            return fi.query_whole_sdp(model, expr, pool_inds, session)
        if expr.pars.get('fi_mode', 'greedy') == 'block-greedy':
            return fi.query_whole_block(model, expr, pool_inds, session)
        return fi.query_whole(model, expr, pool_inds, session)
    if method_name == 'rep-entropy':
        from . import rep
        return rep.query_rep_entropy_whole(model, expr, pool_inds, session)
    raise NotImplementedError('query method %r is not part of the replaced path' % method_name)
