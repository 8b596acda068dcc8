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


def _posteriors_on_device(model, expr, pool_inds, session, keep=0, mc=None):
    """Pool pass over this rank's block [lo, hi) of the pool.  ``mc = (T, keep_prob)`` runs T MC-dropout passes of the
    FC tail; the masks are keyed by global pool position (pos0 = lo), so they do not depend on the sharding."""
    eng = get_engine()
    eng.set_model(model, session)
    pool_inds = np.asarray(pool_inds)
    n = len(pool_inds)
    rank, world = dist.rank_world()
    b = dist.shard_bounds(n, world)
    lo, hi = int(b[rank]), int(b[rank + 1])
    if mc is not None:
        eng.pool_mc_config(mc[0], mc[1], model.dropout_layers, pos0=lo)
    try:
        eng.pool_begin(hi - lo, keep)
        eng.pool_eval_images(_pool_images(expr, pool_inds[lo:hi]), 0)
    finally:
        if mc is not None:
            eng.pool_mc_config(0, 1., [])
    return eng, lo, hi


def CNN_query(model, expr, pool_inds, method_name, session, col=True, extra_feed_dict={}):
    """NNAL.CNN_query (NNAL.py:188-525): returns positions into ``pool_inds``.

    ``entropy``: posteriors ``[c,n]`` -> compute_entropy (zeros -> 1e-7) -> argsort(-H)[:k]
    (NNAL.py:298-310).  ``fi``: see ``nnal_b200.fi.query_whole``; ``expr.pars['fi_mode'] = 'sdp'`` runs the reference's
    own multiclass A-matrix + SDP + sampling pipeline (``nnal_b200.fi.query_whole_sdp``); ``'block-greedy'`` runs the greedy
    FI selection for any number of classes (``nnal_b200.fi.query_whole_block``) over the last FC layer, or over the last two
    with ``expr.pars['fi_layers'] = 2``.

    Class counts: every method runs for 2 <= c <= 32 (fused head kernel) and for c >= 64 (wide head: FC GEMM for the
    logits, then a streaming softmax; chosen from the model's class count); 33 <= c <= 63 raises NnalError
    (NNAL_ERR_UNSUPPORTED).  ``fi_mode = 'block-greedy'`` runs for c <= 32, and for any c with ``expr.pars['fi_classes'] = r``
    (2 <= r <= 32, last FC layer only): each candidate keeps its min(r, c) most probable classes, renormalised.

    Bayesian and committee scorers, for those class counts (the binary definitions of PW_NNAL.py:67-87, 247-282 and
    :453-545 extended to c classes; ties go to the lowest position):
    ``MC-entropy`` / ``BALD``: ``expr.pars['MC_iters']`` MC-dropout passes at ``model.dropout_rate`` on
    ``model.dropout_layers`` (FC layers; the conv trunk runs once), float64 running means of every class posterior and of
    the per-pass entropies; k largest predictive entropies H(mean p), resp. k largest H(mean p) - mean H(p).
    ``ensemble`` / ``QBC-JS``: the same two scores over a committee, the weights of ``expr.pretrained_paths`` loaded into
    ``expr.model_holder`` one after the other (``perform_assign_ops``), each evaluated deterministically."""
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
    if method_name in ('MC-entropy', 'BALD'):
        eng, lo, hi = _posteriors_on_device(model, expr, pool_inds, session,
                                            mc=(int(expr.pars['MC_iters']), float(model.dropout_rate)))
        eng.pool_score(L.SCORE_MC_NEG_ENTROPY if method_name == 'MC-entropy' else L.SCORE_MC_NEG_BALD)
        q, _ = dist.topk_global(eng, k, lo, len(pool_inds))
        return q
    if method_name in ('ensemble', 'QBC-JS'):
        eng = None
        try:
            for i, path in enumerate(expr.pretrained_paths):
                expr.model_holder.perform_assign_ops(path, session)
                eng, lo, hi = _posteriors_on_device(expr.model_holder, expr, pool_inds, session)
                eng.pool_ensemble_accumulate(i)
        finally:
            if eng is not None:
                eng.pool_ensemble_end()
        eng.pool_score(L.SCORE_MC_NEG_ENTROPY if method_name == 'ensemble' else L.SCORE_MC_NEG_BALD)
        q, _ = dist.topk_global(eng, k, lo, len(pool_inds))
        return q
    if method_name == 'rep-entropy':
        from . import rep
        return rep.query_rep_entropy_whole(model, expr, pool_inds, session)
    raise NotImplementedError('query method %r is not part of the replaced path' % method_name)
