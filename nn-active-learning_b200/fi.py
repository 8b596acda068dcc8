"""Fisher-information (FI) queries: the ``'fi'`` branches of ``PW_NNAL.CNN_query``
(PW_NNAL.py:89-163), ``PW_NNAL.query_multimg`` (:547-627) and ``NNAL.CNN_query`` (NNAL.py:312-464).

The reference builds one tau x tau conditional FI per pre-filtered sample from 2B single-sample
``sess.run(tf.gradients)`` calls, solves an SDP for a query distribution and SAMPLES k indices from it
with the unseeded global RNG.  The drop-in keeps the reference's pipeline shape -- uncertainty
pre-filter to B (:108-115, 549-551), conditional FIs of the B candidates, selection of k -- but

* keeps the FI of the last ``fi_layers`` (default 2) fully-connected layers in factored form
  (NN.LLFC_grads NN.py:905-955, NNAL_tools.FC_gradnorms_batch NNAL_tools.py:725-775), and
* replaces SDP + sampling by the deterministic greedy minimisation of the SAME objective
  ``tr((sum_i q_i A_i)^-1)`` (NNAL_tools.py:589-602) at ``q = uniform(S)`` (DESIGN.md, FI section).

``expr.pars['fi_mode'] = 'sdp'`` runs the reference's own pipeline instead (``query_single_sdp``, ``query_multimg_sdp``,
``query_whole_sdp``): conditional FIs in the reference's shrunk coordinates from one batched backward pass on the device
(csrc/shrunk.cu), the SDP query distribution by a certified first-order device solver (csrc/sdp.cu), and
``NNAL_tools.sample_query_dstr`` with NumPy's global generator (<= k unique positions, as upstream); optional keys
``sdp_tol`` (default 1e-4) and ``fi_diag_load``.

``expr.pars`` keys read: ``k``, ``B`` (reference keys) and the optional ``fi_layers`` (1 or 2) and
``fi_diag_load`` (the reference's ``diag_load``: 1e-5 single-volume PW_NNAL.py:738-745, 1e-3 multi-volume
:573-578)."""
import contextlib

import numpy as np

from . import _lib as L
from . import dist, patch_utils
from .engine import get_engine


def greedy_select(eng, k, delta, gids=None):
    """Greedy FI selection over the engine's current candidate set.

    Single process: one device-side loop (``nnal_fi_greedy``).  Several ranks: every step all-gathers one
    fixed-size message per rank (its local best: loss, id, factor rows, K_SS row) and every rank applies the
    same global winner.  ``gids``: global candidate ids of
    this rank's candidates (ascending), used for the result and for tie-breaking (lowest id).
    Returns (selected global ids in selection order, objective after each step, its kernel-dependent part
    ``tr((delta I + K_SS/s)^-1)`` -- the full objective is ``(D - s)/delta`` plus that)."""
    n_local = eng.fi_info()['n']
    if gids is None:
        gids = np.arange(n_local, dtype=np.int64)
    if not dist.is_dist():
        sel, obj, red = eng.fi_greedy(k, delta)
        return gids[sel], obj, red
    import torch
    import torch.distributed as td
    rank, world = dist.rank_world()
    n_total = int(dist.allreduce_sum_(torch.tensor([n_local], dtype=torch.int64, device=dist._device())).item())
    k = min(int(k), n_total)
    if k == 0:
        return np.zeros(0, dtype=np.int64), np.zeros(0), np.zeros(0)
    D = eng.fi_info()['D']
    eng.fi_begin(k, delta)
    eng.fi_set_gids(gids)
    # Device-resident loop: per step every rank packs its local best (loss, id, factor rows, K_SS row) into a
    # fixed-size message, the messages are all-gathered on the engine's stream and every rank applies the
    # global winner -- the host only enqueues.
    nbytes = eng.fi_msg_bytes()
    dev = eng.message_device
    send = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
    global last_exchange
    p2p = _p2p_ready(eng, world, rank, nbytes)
    last_exchange = 'nvlink peer memory (csrc/p2p.cu)' if p2p else 'all_gather_into_tensor'
    recv = None if p2p else torch.zeros(world * nbytes, dtype=torch.uint8, device=dev)
    ctx = torch.cuda.stream(torch.cuda.ExternalStream(eng.stream)) if dev == 'cuda' else contextlib.nullcontext()
    with ctx:
        for t in range(k):
            eng.fi_step_pack(t, send.data_ptr())
            if p2p:
                # one kernel: peer stores of the message into every rank's buffer over NVLink + flag wait (csrc/p2p.cu)
                gathered = eng.p2p_allgather(send.data_ptr(), nbytes, eng._p2p_seq)
                eng._p2p_seq += 1
            else:
                td.all_gather_into_tensor(recv, send)
                gathered = recv.data_ptr()
            eng.fi_step_apply_gathered(t, gathered, world, rank)
        if p2p:
            eng.synchronize()          # `send` is read by the last exchange kernel
    sel, red = eng.fi_result(k)
    s = np.arange(1, k + 1, dtype=np.float64)
    return sel, (D - s) / delta + red, red


last_exchange = None        # how the last multi-rank greedy_select moved its step messages
p2p_enabled = True          # peer-memory exchange of the greedy step messages where CUDA IPC works; False: NCCL all-gather


def _p2p_ready(eng, world, rank, nbytes):
    """Sets up (once per message size) the peer-memory exchange of csrc/p2p.cu: every rank allocates its receive buffer, the
    64-byte CUDA IPC handles are all-gathered and opened.  Collective; returns False on every rank if any rank cannot (gloo /
    fake engine, IPC refused by the container) -- the loop then uses ``all_gather_into_tensor``."""
    import torch
    import torch.distributed as td
    if not p2p_enabled or getattr(eng, 'message_device', 'cpu') != 'cuda' or not hasattr(eng, 'p2p_alloc') or \
            td.get_backend() != 'nccl' or world > 16:
        return False
    if getattr(eng, '_p2p_key', None) == (world, rank, nbytes):
        return True
    if getattr(eng, '_p2p_key', None) == 'failed':
        return False
    def agreed(ok):
        flag = torch.tensor([1 if ok else 0], dtype=torch.int32, device='cuda')
        td.all_reduce(flag, op=td.ReduceOp.MIN)
        return int(flag.item()) == 1
    if getattr(eng, '_p2p_key', None) is not None:
        eng.synchronize()              # a buffer of another message size is replaced: nobody may still be using it
        td.barrier()
    ok, h = True, None
    try:
        h = eng.p2p_alloc(world, rank, nbytes)
    except Exception:
        ok = False
    if agreed(ok):
        mine = torch.frombuffer(bytearray(h), dtype=torch.uint8).cuda()
        allh = torch.empty(world * 64, dtype=torch.uint8, device='cuda')
        td.all_gather_into_tensor(allh, mine)
        try:
            eng.p2p_open(allh.cpu().numpy().tobytes())
        except Exception:
            ok = False
        ok = agreed(ok)
    else:
        ok = False
    if not ok:
        eng._p2p_key = 'failed'
        return False
    eng._p2p_key = (world, rank, nbytes)
    if not hasattr(eng, '_p2p_seq'):
        eng._p2p_seq = 0
    return True


last_report = None          # dict left by the last FI query run with expr.pars['fi_report'] = True (see gram_report)


def gram_allreduce(eng):
    """Sums the per-GPU Gram partials left on the device by ``fi_gram`` / ``fi_gram_subset`` over all ranks: NCCL
    all-reduce of the (d+1) x ld float32 matrix on the engine's stream (SURVEY.md 8e collective 2).  In place; returns the
    bytes reduced (0 in a single process).  gloo / fake engine (CPU tests): the host copy is reduced instead."""
    if not dist.is_dist():
        return 0
    if getattr(eng, 'message_device', 'cpu') != 'cuda':
        return eng.fi_gram_allreduce_host()
    ptr, rows, ld = eng.fi_gram_device()
    return dist.allreduce_device_f32_(eng, ptr, rows * ld)


def gram_report(eng, sel_gids, gids, delta, cand_rows=None, pool_gram=True):
    """Primal (Gram) form of the FI objective for the selection ``sel_gids`` (global candidate ids) on the engine's
    current candidate set (``gids``: global ids of the local candidates, ascending).

    Every rank builds its partial of the weighted penultimate-feature Gram ``H = sum_i q_i w_i [u_i;1][u_i;1]^T`` on
    tensor cores -- (a) over ALL its candidates at ``q = 1/n`` (the pool's last-layer Fisher information) and (b) over
    its members of the selection at ``q = uniform(S)`` -- the partials are summed with an NCCL all-reduce, and the
    reference's objective ``tr((sum_i q_i A_i)^-1)`` (NNAL_tools.py:589-602) restricted to the last layer,
    ``tr((delta I + 2 H_S)^-1) + (d+1)/delta``, is evaluated on the device, together with the Fisher-information ratio
    ``tr((delta I + 2 H_S)^-1 (delta I + 2 H_pool))``.  ``dual_last_layer`` is the same objective through the k x k
    kernel of the selected samples (float64, host): the two must agree, on every rank."""
    import torch
    rank, world = dist.rank_world()
    gids = np.asarray(gids, dtype=np.int64)
    sel_gids = np.asarray(sel_gids, dtype=np.int64)
    k = len(sel_gids)
    n_local = len(gids)
    d = eng.fi_info()['d']
    n_total = n_local
    if dist.is_dist():
        n_total = int(dist.allreduce_sum_(torch.tensor([n_local], dtype=torch.int64, device=dist._device())).item())
    rep = {'k': int(k), 'n_candidates': int(n_total), 'delta': float(delta), 'gram_bytes': 0}
    cuda = getattr(eng, 'message_device', 'cpu') == 'cuda'
    G2 = None
    if pool_gram and n_total > 0:
        ev = None
        if cuda:
            stream = torch.cuda.ExternalStream(eng.stream)
            ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
            ev[0].record(stream)
        eng.fi_gram(np.full(n_local, 1. / n_total), read=False)
        if ev:
            ev[1].record(stream)
        rep['gram_bytes'] = gram_allreduce(eng)
        if ev:
            ev[2].record(stream)
            ev[2].synchronize()
            rep['gram_ms'], rep['allreduce_ms'] = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
        if cuda:
            ptr, rows, ld = eng.fi_gram_device()
            with dist.engine_stream(eng):
                G2 = dist.device_view(ptr, (rows * ld,), '<f4').clone()
        else:
            G2 = eng.fi_gram_read().copy()
    # members of the selection owned by this rank (gids is ascending)
    pos = np.searchsorted(gids, sel_gids)
    pos = np.minimum(pos, max(n_local - 1, 0))
    mine = (gids[pos] == sel_gids) if n_local else np.zeros(k, dtype=bool)
    loc = pos[mine]
    eng.fi_gram_subset(loc, np.full(len(loc), 1. / max(k, 1)))
    gram_allreduce(eng)
    tr, ratio = eng.fi_gram_solve(delta, 2.0, None if G2 is None else (G2.data_ptr() if cuda else G2))
    rep['primal_last_layer'] = tr + (d + 1) / delta
    rep['primal_reduced'] = tr - (d + 1 - min(k, d + 1)) / delta
    rep['fi_ratio'] = ratio
    # dual form of the same last-layer objective from the selected samples' rows (k x k, float64 on the host)
    rows_local = loc if cand_rows is None else np.asarray(cand_rows)[loc]
    F = eng.pool_feature_rows(rows_local).astype(np.float64) if len(loc) else np.zeros((0, d))
    p1 = eng.pool_posteriors()[1].astype(np.float64)[rows_local] if len(loc) else np.zeros(0)
    blk = np.zeros((k, d + 2))
    blk[np.nonzero(mine)[0], :d] = F
    blk[np.nonzero(mine)[0], d] = 1.
    blk[np.nonzero(mine)[0], d + 1] = p1
    if dist.is_dist():
        t = torch.from_numpy(blk).to(dist._device())
        dist.allreduce_sum_(t)
        blk = t.cpu().numpy()
    Ut, p = blk[:, :d + 1], blk[:, d + 1]
    sw = np.sqrt(p * (1. - p))
    K1 = 2. * (Ut @ Ut.T) * np.outer(sw, sw) / max(k, 1)
    lam = np.linalg.eigvalsh(K1) if k else np.zeros(0)
    red = float(np.sum(1. / (delta + np.maximum(lam, 0.))))
    rep['dual_reduced'] = red
    rep['dual_last_layer'] = (2 * (d + 1) - k) / delta + red
    return rep


def _maybe_report(expr, eng, chosen, gids, delta, obj, cand_rows=None):
    """``expr.pars['fi_report'] = True``: leave the Gram-form (primal) evaluation of the selection in ``fi.last_report``."""
    global last_report
    if not expr.pars.get('fi_report', False):
        return
    last_report = gram_report(eng, chosen, gids, delta, cand_rows)
    last_report['dual_objective'] = float(obj[-1]) if len(obj) else None


def _pars(expr, default_delta):
    nl = int(expr.pars.get('fi_layers', 2))
    delta = float(expr.pars.get('fi_diag_load', default_delta))
    return nl, delta


def _one_pass(eng, n_local, nl):
    """Keep the FC factors of the WHOLE local pool in one pass (and index the B candidates in place) when they fit the
    factor budget -- a fraction of the device memory, ``Engine.factor_budget`` -- instead of re-running gather + forward
    over the candidates (what the reference does, PW_NNAL.py:117-131).  Same factors either way: the forward pass does not
    depend on which samples share a chunk."""
    per = 4 * (eng.feat_dim + (eng.prev_dim if nl == 2 else 0))
    return n_local * per <= eng.factor_budget_bytes()


def _ret(q, obj, red, q_ent, return_objective, also_entropy):
    out = (q, obj, red) if return_objective == 'reduced' else ((q, obj) if return_objective else q)
    if also_entropy:
        return (q_ent,) + (out if isinstance(out, tuple) else (out,))
    return out


def query_single(expr, model, sess, padded_imgs, pool_inds, return_objective=False, also_entropy=False):
    """``PW_NNAL.CNN_query(..., 'fi')``: positions into ``pool_inds`` (greedy selection order).
    ``also_entropy``: the same pool pass also answers the ``'entropy'`` query (k smallest |p - 0.5|, PW_NNAL.py:51-65);
    returns ``(q_entropy, q_fi[, ...])`` -- the combined round of ``method_name = 'entropy+fi'``."""
    from .PW_NNAL import _score_pool_single, _stats_list
    k, B = int(expr.pars['k']), int(expr.pars['B'])
    nl, delta = _pars(expr, 1e-5)
    pool_inds = np.asarray(pool_inds)
    n = len(pool_inds)
    eng = get_engine()
    eng.set_model(model, sess)
    rank, world = dist.rank_world()
    b = dist.shard_bounds(n, world)
    one_pass = B >= n or _one_pass(eng, int(b[rank + 1] - b[rank]), nl)
    eng, lo, hi = _score_pool_single(expr, model, sess, padded_imgs, pool_inds, keep=nl if one_pass else 0)
    q_ent = None
    cand_rows = None
    if B < n or also_entropy:
        eng.pool_score(L.SCORE_BINARY)
    if B < n:
        sel_inds, _ = dist.topk_global(eng, max(B, k) if also_entropy else B, lo, n)
        if also_entropy:
            q_ent, sel_inds = sel_inds[:k], sel_inds[:B]          # both lists are prefixes of one ascending ranking
        own = (sel_inds >= lo) & (sel_inds < hi)
        mine = sel_inds[own]
        if one_pass:
            cand_rows = mine - lo                                 # candidates = rows of the pool pass, indexed in place
            eng.fi_set_candidates(cand_rows, nl)
        else:
            # second pass over this rank's candidates, keeping the factors of the last FC layers
            eng.pool_begin(len(mine), nl)
            if len(mine):
                imgs = list(padded_imgs)
                eng.pool_eval(0, pool_inds[mine], 0, expr.pars['patch_shape'], _stats_list(expr.pars['stats'], len(imgs)),
                              L.NORM_BATCH_EVAL, shape=imgs[0].shape)
            eng.fi_set_candidates(None, nl)
    else:
        if also_entropy:
            q_ent, _ = dist.topk_global(eng, k, lo, n)
        sel_inds = np.arange(n, dtype=np.int64)
        own = (sel_inds >= lo) & (sel_inds < hi)
        eng.fi_set_candidates(None, nl)
    gids = np.nonzero(own)[0].astype(np.int64)
    chosen, obj, red = greedy_select(eng, min(k, len(sel_inds)), delta, gids)
    _maybe_report(expr, eng, chosen, gids, delta, obj, cand_rows)
    return _ret(sel_inds[chosen], obj, red, q_ent, return_objective, also_entropy)


def query_multimg(expr, model, sess, all_padded_imgs, pool_inds, return_objective=False, also_entropy=False):
    """``PW_NNAL.query_multimg(..., 'fi')``: list of S arrays of local positions into ``pool_inds[s]``.
    Candidate order = the reference's: subject-major, uncertainty order inside a subject
    (``A += gen_A_matrices(...)`` per subject, PW_NNAL.py:566-578); without a pre-filter (``B >= n``) the candidates are
    the pool in its own (subject-major) order."""
    from .PW_NNAL import _pool_pass_multimg
    k, B = int(expr.pars['k']), int(expr.pars['B'])
    nl, delta = _pars(expr, 1e-3)
    eng = get_engine()
    eng.set_model(model, sess)
    s = len(pool_inds)
    m = len(all_padded_imgs[0]) - 1
    sizes = [len(pool_inds[i]) for i in range(s)]
    n = int(np.sum(sizes))
    rank, world = dist.rank_world()
    b = dist.shard_bounds(n, world)
    one_pass = B >= n or _one_pass(eng, int(b[rank + 1] - b[rank]), nl)
    eng, lo, hi, sizes, n = _pool_pass_multimg(expr, model, sess, all_padded_imgs, pool_inds, keep=nl if one_pass else 0)
    cum = np.append(-1, np.cumsum(sizes) - 1)
    q_ent = None
    cand_rows = None
    if B < n or also_entropy:
        eng.pool_score(L.SCORE_BINARY)
    if also_entropy:
        q_ent = patch_utils.global2local_inds(dist.topk_global(eng, k, lo, n)[0], sizes)
    if B < n:
        sorted_inds, _ = dist.topk_global(eng, B, lo, n)
        set_of = cum.searchsorted(sorted_inds) - 1
        order = np.argsort(set_of, kind='stable')
        G = sorted_inds[order]                       # global positions, subject-major candidate order
        G_set = set_of[order]
        own = (G >= lo) & (G < hi)
        if one_pass:
            cand_rows = G[own] - lo
            eng.fi_set_candidates(cand_rows, nl)
        else:
            eng.pool_begin(int(own.sum()), nl)
            off = 0
            for i in range(s):
                sel = own & (G_set == i)
                ni = int(sel.sum())
                if ni == 0:
                    continue
                local = G[sel] - (cum[i] + 1)
                imgs = list(all_padded_imgs[i][:-1])
                eng.upload(i, imgs)
                stats = np.array([[expr.train_stats[i, 2 * j], expr.train_stats[i, 2 * j + 1]] for j in range(m)],
                                 dtype=np.float64)
                eng.pool_eval(i, np.asarray(pool_inds[i])[local], off, expr.pars['patch_shape'], stats, L.NORM_BATCH_EVAL,
                              shape=imgs[0].shape)
                off += ni
            eng.fi_set_candidates(None, nl)
    else:
        G = np.arange(n, dtype=np.int64)
        own = (G >= lo) & (G < hi)
        eng.fi_set_candidates(None, nl)
    gids = np.nonzero(own)[0].astype(np.int64)
    chosen, obj, red = greedy_select(eng, min(k, len(G)), delta, gids)
    _maybe_report(expr, eng, chosen, gids, delta, obj, cand_rows)
    Q = patch_utils.global2local_inds(G[chosen], sizes)
    return _ret(Q, obj, red, q_ent, return_objective, also_entropy)


def _gather_shrunk(post, g):
    """All-gather of per-rank shrunk-gradient slices (candidates are block-partitioned over the ranks in candidate
    order): ``post`` [c,m_r], ``g`` [c,m_r,tau] -> [c,B], [c,B,tau] on every rank.  No-op in a single process."""
    if not dist.is_dist():
        return post, g
    c, tau = g.shape[0], g.shape[2]
    P = dist.allgather_concat(np.ascontiguousarray(post.T, dtype=np.float32).ravel()).reshape(-1, c).T
    G = dist.allgather_concat(np.ascontiguousarray(np.transpose(g, (1, 0, 2)), dtype=np.float64).ravel())
    return np.ascontiguousarray(P), np.ascontiguousarray(np.transpose(G.reshape(-1, c, tau), (1, 0, 2)))


def _my_slice(n):
    rank, world = dist.rank_world()
    b = dist.shard_bounds(n, world)
    return int(b[rank]), int(b[rank + 1])


def _sdp_sample(A, expr, return_solution, shrunk=None, ref_F=None):
    """SDP query distribution + the reference's sampler (PW_NNAL.py:154-163).  The draw uses NumPy's global
    generator like the reference; with several ranks, rank 0's draw is broadcast.  ``shrunk = (g, p1, diag_load)``:
    binary A-matrices assembled on the device instead of ``A``.  ``ref_F`` [d, B]: the zero-mean refined feature matrix of
    the ``lambda_ > 0`` programme (PW_NNAL.py:139-155)."""
    from . import NNAL_tools
    k = int(expr.pars['k'])
    tol = float(expr.pars.get('sdp_tol', 1e-4))
    lambda_ = expr.pars.get('lambda_', 0)
    if shrunk is not None and not (lambda_ > 0):
        soln = NNAL_tools.SDP_query_distribution_from_shrunk(shrunk[0], shrunk[1], shrunk[2], k, tol=tol)
        nA = shrunk[0].shape[1]
    else:
        if shrunk is not None:                       # regularised programme: the solver takes explicit A-matrices
            from .PW_NNAL import _A_from_shrunk
            A = _A_from_shrunk(shrunk[0], shrunk[1], shrunk[2], as_list=False)
        soln = NNAL_tools.SDP_query_distribution(A, lambda_ if ref_F is not None else 0, ref_F, k, tol=tol)
        nA = len(A)
    q_opt = np.array(soln['x'][:nA])
    Q_inds = NNAL_tools.sample_query_dstr(q_opt.copy(), k, replacement=True)
    if dist.is_dist():
        buf = np.full(k + 1, -1, dtype=np.int64)
        buf[0] = len(Q_inds)
        buf[1:1 + len(Q_inds)] = Q_inds
        buf = dist.broadcast_array(buf, 0)
        Q_inds = buf[1:1 + int(buf[0])]
    return (Q_inds, soln) if return_solution else (Q_inds, None)


def query_single_sdp(expr, model, sess, padded_imgs, pool_inds, return_solution=False):
    """``PW_NNAL.CNN_query(..., 'fi')`` as the reference runs it (PW_NNAL.py:89-163): posteriors -> the B most
    uncertain samples (:107-115) -> conditional FIs in shrunk coordinates (gen_A_matrices, diag_load 1e-5) -> SDP
    query distribution -> ``sample_query_dstr`` (<= k unique positions, sorted).  Positions into ``pool_inds``.
    The candidates' patches are gathered on the device; with several ranks each one back-propagates its block of the B
    candidates, the shrunk gradients (B x 2 x tau numbers) are all-gathered and every rank solves the same SDP."""
    from .PW_NNAL import _score_pool_single, _stats_list
    B = int(expr.pars['B'])
    pool_inds = np.asarray(pool_inds)
    n = len(pool_inds)
    eng, lo, hi = _score_pool_single(expr, model, sess, padded_imgs, pool_inds, keep=0)
    if B < n:
        eng.pool_score(L.SCORE_BINARY)
        sel_inds, _ = dist.topk_global(eng, B, lo, n)
    else:
        sel_inds = np.arange(n, dtype=np.int64)
    imgs = list(padded_imgs)
    a, e = _my_slice(len(sel_inds))              # the backward pass is sharded over the ranks, the tiny SDP is replicated
    post, g = eng.fi_shrunk_voxels(0, pool_inds[sel_inds[a:e]], expr.pars['patch_shape'],
                                   _stats_list(expr.pars['stats'], len(imgs)), L.NORM_BATCH_EVAL, shape=imgs[0].shape)
    post, g = _gather_shrunk(post, g)
    ref_F = None
    if expr.pars.get('lambda_', 0) > 0:
        # PW_NNAL.py:139-151: feature_layer of the B candidates (batch_eval), refined to full row rank, rows made zero-mean.
        # (B candidates through one more forward pass on every rank: the matrix is B/2 x B at most.)
        from .PW_NNAL import refine_feature_matrix
        eng.pool_begin(len(sel_inds), 1)
        eng.pool_eval(0, pool_inds[sel_inds], 0, expr.pars['patch_shape'], _stats_list(expr.pars['stats'], len(imgs)),
                      L.NORM_BATCH_EVAL, shape=imgs[0].shape)
        F = eng.pool_features().astype(np.float64)
        ref_F = refine_feature_matrix(F, B)
        ref_F -= np.mean(ref_F, axis=1, keepdims=True)
    Q_inds, soln = _sdp_sample(None, expr, return_solution,
                               shrunk=(g, post[1].astype(np.float64), float(expr.pars.get('fi_diag_load', 1e-5))), ref_F=ref_F)
    q = sel_inds[Q_inds]
    return (q, soln, sel_inds) if return_solution else q


def query_multimg_sdp(expr, model, sess, all_padded_imgs, pool_inds, return_solution=False):
    """``PW_NNAL.query_multimg(..., 'fi')`` as the reference runs it (PW_NNAL.py:547-627): B most uncertain samples of
    the concatenated pool, per-subject A-matrices with diag_load 1e-3 (:566-578) in subject-major order, SDP,
    sampling, ``global2local_inds`` of the sampled candidates' pool positions."""
    from .PW_NNAL import _bin_filter_core
    B = int(expr.pars['B'])
    eng = get_engine()
    sorted_inds, _, lo, hi, sizes = _bin_filter_core(expr, model, sess, all_padded_imgs, pool_inds, B)
    s = len(pool_inds)
    m = len(all_padded_imgs[0]) - 1
    cum = np.append(-1, np.cumsum(sizes) - 1)
    set_of = cum.searchsorted(sorted_inds) - 1
    order = np.argsort(set_of, kind='stable')
    G = sorted_inds[order]                       # global positions, subject-major candidate order
    G_set = set_of[order]
    delta = float(expr.pars.get('fi_diag_load', 1e-3))
    a, e = _my_slice(len(G))                     # this rank's block of the candidate list
    mine = np.zeros(len(G), dtype=bool)
    mine[a:e] = True
    posts, gs = [], []
    for i in range(s):
        sel = mine & (G_set == i)
        if not sel.any():
            continue
        local = G[sel] - (cum[i] + 1)
        imgs = list(all_padded_imgs[i][:-1])
        eng.upload(i, imgs)
        stats = np.array([[expr.train_stats[i, 2 * j], expr.train_stats[i, 2 * j + 1]] for j in range(m)],
                         dtype=np.float64)
        # the gradient patches come from get_patches_multimg upstream (PW_NNAL.py:553-559): EVERY channel of modality
        # block ch/d3 is normalised (patch_utils.py:1203-1207), unlike batch_eval's channels 0..m-1 of the posterior pass
        post, g = eng.fi_shrunk_voxels(i, np.asarray(pool_inds[i])[local], expr.pars['patch_shape'], stats,
                                       L.NORM_MULTIMG, shape=imgs[0].shape)
        posts.append(post)
        gs.append(g)
    tau = eng.fi_shrunk_tau()
    post = np.concatenate(posts, axis=1) if posts else np.zeros((2, 0), dtype=np.float32)
    g = np.concatenate(gs, axis=1) if gs else np.zeros((2, 0, tau))
    post, g = _gather_shrunk(post, g)
    Q_inds, soln = _sdp_sample(None, expr, return_solution, shrunk=(g, post[1].astype(np.float64), delta))
    Q = patch_utils.global2local_inds(G[Q_inds], sizes)
    return (Q, soln, G) if return_solution else Q


def _A_multiclass_from_shrunk(sel_posteriors, g, diag_load=1e-5, max_classes=10):
    """Multiclass conditional FIs in shrunk coordinates as NNAL.CNN_query builds them inline (NNAL.py:354-414), from the
    device's shrunk gradients ``g`` [c,B,tau].  Per candidate: posteriors below 1e-6 are zeroed IN PLACE in the caller's
    array (:361-362) and the survivors renormalised (:364-365); with ten or more survivors only the ten most probable are
    kept and renormalised once more (:379-400); every kept class j adds ``g_j g_j^T / p_j`` AND one ``diag_load * I``
    (:404-409 -- the load is inside the class loop upstream, so it scales with the number of kept classes)."""
    tau = g.shape[2]
    load = np.eye(tau) * diag_load
    out = []
    for i in range(sel_posteriors.shape[1]):
        col = sel_posteriors[:, i]                   # a view: the zeroing below is visible to the caller, as upstream
        col[col < 1e-6] = 0.
        keep = np.flatnonzero(col > 0.)
        w = col[keep] / np.sum(col[keep])
        if len(keep) >= max_classes:
            top = np.argsort(-w, kind='stable')[:max_classes]
            keep, w = keep[top], w[top]
            w = w / np.sum(w)
        Ai = np.zeros((tau, tau))
        for j, cls in enumerate(keep):
            Ai += np.outer(g[cls, i], g[cls, i]) / w[j] + load
        out.append(Ai)
    return out


def query_whole_sdp(model, expr, pool_inds, session, return_solution=False):
    """``NNAL.CNN_query(..., 'fi')`` as the reference runs it (NNAL.py:312-464) with ``lambda_ = 0``: posteriors ->
    ``uncertainty_filtering`` to B (:326-333) -> per-sample multiclass A-matrices in shrunk coordinates (:354-414; the
    per-class ``session.run(model.grad_posts[y])`` calls are one batched backward pass per class on the device) -> SDP
    query distribution (:456-459) -> ``sample_query_dstr`` (:462-464).  Positions into ``pool_inds``."""
    from .NNAL import _pool_images, _posteriors_on_device
    B = int(expr.pars['B'])
    pool_inds = np.asarray(pool_inds)
    n = len(pool_inds)
    eng, lo, hi = _posteriors_on_device(model, expr, pool_inds, session, keep=0)
    if B < n:
        eng.pool_score(L.SCORE_NEG_ENTROPY, 1e-8)
        sel_inds, _ = dist.topk_global(eng, B, lo, n)
    else:
        sel_inds = np.arange(n, dtype=np.int64)
    a, e = _my_slice(len(sel_inds))
    post, g = eng.fi_shrunk_images(_pool_images(expr, pool_inds[sel_inds[a:e]]))
    post, g = _gather_shrunk(post, g)
    A = _A_multiclass_from_shrunk(post.astype(np.float64), g)
    ref_F = None
    if expr.pars.get('lambda_', 0) > 0:
        # NNAL.py:414-447: features of the B candidates (model.extract_features), the int(B/2) rows with the most positive
        # entries, tail dropped until full row rank (warning below 10 rows) and cond <= 1e6 (a single row left switches the
        # regulariser off, :440-442), rows made zero-mean
        import warnings
        eng.pool_begin(len(sel_inds), 1)
        eng.pool_eval_images(_pool_images(expr, pool_inds[sel_inds]), 0)
        F = eng.pool_features().astype(np.float64)
        order = np.argsort(-np.sum(F > 0, axis=1))[:int(B / 2)]
        while np.linalg.matrix_rank(F[order, :]) < len(order):
            order = order[:-1]
            if len(order) < 10:
                warnings.warn("Few features (%d) are selected" % len(order))
        off = False
        while np.linalg.cond(F[order, :]) > 1e6:
            order = order[:-1]
            if len(order) == 1:
                off = True
                break
        if not off:
            ref_F = F[order, :] - np.mean(F[order, :], axis=1, keepdims=True)
    Q_inds, soln = _sdp_sample(A, expr, return_solution, ref_F=ref_F)
    q = sel_inds[Q_inds]
    return (q, soln, sel_inds) if return_solution else q


def query_whole(model, expr, pool_inds, session):
    """``NNAL.CNN_query(..., 'fi')`` (NNAL.py:312-464).  Binary models: uncertainty pre-filter to B
    (entropy, NNAL_tools.uncertainty_filtering) + last-layer factored greedy.  c > 2: the k pool
    samples with the largest last-layer FI trace ``(1-|pi|^2)(|u|^2+1)``, the closed form the
    reference itself uses in its self-contained FI scorer (NNAL.py:121-139)."""
    from .NNAL import _posteriors_on_device
    k, B = int(expr.pars['k']), int(expr.pars['B'])
    nl, delta = _pars(expr, 1e-5)
    pool_inds = np.asarray(pool_inds)
    n = len(pool_inds)
    eng, lo, hi = _posteriors_on_device(model, expr, pool_inds, session, keep=1)
    if eng.n_class != 2:
        eng.pool_score(L.SCORE_NEG_FI_TRACE)
        q, _ = dist.topk_global(eng, k, lo, n)
        return q
    if B < n:
        eng.pool_score(L.SCORE_NEG_ENTROPY, 1e-8)
        sel_inds, _ = dist.topk_global(eng, B, lo, n)
    else:
        sel_inds = np.arange(n, dtype=np.int64)
    own = (sel_inds >= lo) & (sel_inds < hi)
    eng.fi_set_candidates(sel_inds[own] - lo, 1)
    gids = np.nonzero(own)[0].astype(np.int64)
    chosen, _, _ = greedy_select(eng, min(k, len(sel_inds)), delta, gids)
    return sel_inds[chosen]


def query_whole_block(model, expr, pool_inds, session, return_objective=False):
    """``NNAL.CNN_query(..., 'fi')`` with ``expr.pars['fi_mode'] = 'block-greedy'``: greedy minimisation of the FI
    objective ``tr((sum_{i in S} F_i/|S| + delta I)^-1)`` for 2 <= c <= 32 classes (k (c-1) <= 4096; with more classes the
    library raises NNAL_ERR_UNSUPPORTED after the pool pass, before it allocates the block system, unless ``fi_classes`` is
    set) in the block form of csrc/fi_block.cu.  ``expr.pars['fi_layers']`` (default 1) picks the parameters: 1 = the last FC
    layer, ``F_i = (diag pi_i - pi_i pi_i^T) (x) [u_i;1][u_i;1]^T`` (NN.LLFC_hess, NN.py:891-901); 2 = the last two FC
    layers, as the binary path's default, adding the score ``(M_i W3^T (e_y - pi_i)) (x) [a_i;1]`` of the previous FC
    layer (M_i = diag 1[u_i > 0], a_i its input).  Entropy pre-filter to B exactly as ``query_whole``, then the greedy
    over ``min(k, B)`` steps.  Keys read: ``k``, ``B``, ``fi_diag_load`` (default 1e-5), ``fi_layers`` (1 or 2; anything
    else raises ValueError), ``fi_classes`` (optional, one layer only: an integer 2 <= r <= 32; every candidate keeps its
    min(r, c) most probable classes, ties to the lower class, renormalised in float64, as the reference's multi-class
    A-matrices keep at most ten (NNAL.py:379-400); the greedy then runs for any c with k (min(r, c) - 1) <= 4096, and with
    r >= c it is the uncapped greedy bit for bit).  Returns positions into ``pool_inds`` in selection order (and, with
    ``return_objective``, the objective and its kernel-dependent part per step).

    Several ranks: every rank reads its own candidates' posteriors and feature rows (and, for two layers, the previous FC
    output), the B candidates are all-gathered and put in pre-filter order on every rank, and every rank runs the same
    deterministic greedy on them.  With ``fi_classes`` each rank selects its own candidates' kept classes on the device and
    the ranks exchange ids and posteriors of the kept classes only."""
    from .NNAL import _posteriors_on_device
    k, B = int(expr.pars['k']), int(expr.pars['B'])
    delta = float(expr.pars.get('fi_diag_load', 1e-5))
    nl = expr.pars.get('fi_layers', 1)
    if nl not in (1, 2):
        raise ValueError("fi_layers must be 1 or 2 for fi_mode='block-greedy', got %r" % (nl,))
    nl = int(nl)
    cap = expr.pars.get('fi_classes')
    if cap is not None:
        if isinstance(cap, (bool, np.bool_)) or not isinstance(cap, (int, np.integer)) or not 2 <= cap <= 32:
            raise ValueError('fi_classes must be an integer from 2 to 32, got %r' % (cap,))
        if nl == 2:
            raise ValueError('fi_classes covers the last FC layer only (fi_layers = 1)')
        cap = int(cap)
    pool_inds = np.asarray(pool_inds)
    n = len(pool_inds)
    eng, lo, hi = _posteriors_on_device(model, expr, pool_inds, session, keep=nl)
    if B < n:
        eng.pool_score(L.SCORE_NEG_ENTROPY, 1e-8)
        sel_inds, _ = dist.topk_global(eng, B, lo, n)
    else:
        sel_inds = np.arange(n, dtype=np.int64)
    if not dist.is_dist():
        if cap is not None:
            eng.fi_block_set_candidates_cls(sel_inds - lo, cap)
        elif nl == 1:
            eng.fi_block_set_candidates(sel_inds - lo)
        else:
            eng.fi_block_set_candidates(sel_inds - lo, nl)
    else:
        own = (sel_inds >= lo) & (sel_inds < hi)
        rows = sel_inds[own] - lo
        c = eng.n_class
        F = eng.pool_feature_rows(rows)
        d = F.shape[1]
        gpos = dist.allgather_concat(sel_inds[own].astype(np.int64))
        Fg = dist.allgather_concat(np.ascontiguousarray(F, dtype=np.float32).ravel()).reshape(-1, d)
        order = np.argsort(gpos, kind='stable')
        perm = order[np.searchsorted(gpos[order], sel_inds)]          # gathered row of every candidate, pre-filter order
        if cap is not None:
            cls, p = eng.pool_top_classes(rows, cap)
            Cg = dist.allgather_concat(cls.ravel()).reshape(-1, cls.shape[1])
            Pg = dist.allgather_concat(p.ravel()).reshape(-1, cls.shape[1])
            eng.fi_block_set_factors_cls(Cg[perm], Pg[perm], Fg[perm], c)
        else:
            post = eng.pool_posteriors()[:, rows] if len(rows) else np.zeros((c, 0), dtype=np.float32)
            P = dist.allgather_concat(np.ascontiguousarray(post.T, dtype=np.float32).ravel()).reshape(-1, c)
            if nl == 1:
                eng.fi_block_set_factors(P[perm].T, Fg[perm])
            else:
                A = eng.pool_prev_rows(rows)
                Ag = dist.allgather_concat(np.ascontiguousarray(A, dtype=np.float32).ravel()).reshape(-1, A.shape[1])
                layers = list(model.layer_dict.items()) if isinstance(model.layer_dict, dict) else list(model.layer_dict)
                W3 = np.asarray(model.get_weights(session)[layers[-1][0]][0], dtype=np.float32)     # [c, d]
                eng.fi_block_set_factors(P[perm].T, Fg[perm], Ag[perm], W3)
    chosen, obj, red = eng.fi_block_greedy(min(k, len(sel_inds)), delta)
    q = sel_inds[chosen]
    if return_objective == 'reduced':
        return q, obj, red
    return (q, obj) if return_objective else q
