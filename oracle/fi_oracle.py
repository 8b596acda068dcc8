"""Float64 restatement of the reference's Fisher-information (FI) scoring (TEST ORACLE).

Restates NN.get_gradients (NN.py:621-645), NNAL_tools.shrink_gradient
(NNAL_tools.py:778-831), PW_NNAL.gen_A_matrices (PW_NNAL.py:738-816), the
multiclass twin (NNAL.py:354-414), NN.LLFC_grads / LLFC_hess (NN.py:874-955),
NNAL_tools.FC_gradnorms_batch (NNAL_tools.py:725-775), the closed-form trace
score (NNAL.py:121-139), the SDP objective tr((sum_i q_i A_i)^-1)
(NNAL_tools.py:576-659) and the seeded sampler (NNAL_tools.py:844-896).

The reference has NO greedy FI selection (its ``fi`` query is an SDP followed by
unseeded random sampling); the deterministic greedy restatement adopted by this
build (SURVEY.md §8a, DESIGN.md §FI) is defined here:

    f(S) = tr( ( (1/|S|) sum_{i in S} Abar_i + delta I )^-1 ),   Abar_i = A_i - delta I
    greedy: S <- S + argmin_{j not in S} f(S + j)      (lowest position on ties)

which is exactly the SDP objective of NNAL_tools.py:589-602 evaluated at
q = uniform(S).
"""
import numpy as np
from .nnal_oracle import forward, stable_topk, batch_eval, get_patches, normalize_batch_eval, pool_same_pads

__all__ = [
    'class_score_factors', 'explicit_class_gradients', 'shrink_gradient',
    'shrunk_class_gradients', 'gen_A_matrices', 'gen_A_matrices_multiclass',
    'LLFC_grads', 'LLFC_hess', 'stoch_approx_IF', 'sdp_solve_reg', 'sdp_solve_reg_slsqp', 'refine_feature_matrix', 'FC_gradnorms_batch', 'fi_trace_score',
    'mnist_fi_score', 'sdp_objective', 'fi_objective_direct', 'greedy_fi_direct',
    'fi_objective_dual', 'greedy_fi_dual_bruteforce', 'greedy_fi_rank1',
    'last_layers_kernel', 'last_layers_dim', 'weighted_gram', 'fi_objective_from_gram',
    'sample_query_dstr', 'append_zero', 'last_layers_factors', 'greedy_fi_replay', 'query_fi_single',
    'query_fi_multimg', 'sdp_certificate', 'sdp_solve', 'sdp_solve_slsqp', 'query_fi_sdp_single',
    'query_fi_sdp_multimg', 'query_fi_sdp_whole',
]


# --------------------------------------------------------------------------
# backward pass: d log p_y / d theta  (NN.py:621-645 builds tf.gradients(log
# posteriors[j,0], gpars); semantics of tf.gradients through relu/max_pool/conv2d)
# --------------------------------------------------------------------------
def _backward(layers, weights, acts, dlogits):
    """Back-propagate ``dlogits`` [c,N] through the stored activations.  Returns a
    list (per layer, same order as ``layers``) of dicts holding ``dz`` (gradient at
    the layer's pre-activation) for conv/fc layers."""
    n_layers = len(layers)
    N = dlogits.shape[1]
    out = [None] * n_layers
    d = dlogits
    flat = True
    for i in range(n_layers - 1, -1, -1):
        name, spec = layers[i]
        rec = acts[i]
        last = (i == n_layers - 1)
        if spec[1] == 'fc':
            W = weights[name][0].astype(np.float64)
            dz = d if last else d * (rec['z'] > 0)
            out[i] = {'dz': dz}
            d = W.T @ dz
            flat = True
        else:
            nhwc = rec['out_nhwc']
            if flat and d.ndim == 2:
                # undo flatten_tf: flat [C*W*H, N] -> [C,W,H,N] -> transpose -> [N,H,W,C]
                _, H, Wd, C = nhwc.shape
                d = np.transpose(d.reshape(C, Wd, H, N))
                flat = False
            if spec[1] == 'pool':
                s = spec[0][0]
                x = rec['in']
                _, H, Wd, C = x.shape
                Ho, Wo = nhwc.shape[1], nhwc.shape[2]
                am = rec['argmax']                       # [N,Ho,Wo,C] index in s*s window of the padded input
                dxp = np.zeros((N, Ho, Wo, C, s * s))
                np.put_along_axis(dxp, am[..., None], d[..., None], axis=-1)
                dxp = dxp.reshape(N, Ho, Wo, C, s, s).transpose(0, 1, 4, 2, 5, 3)
                dxp = dxp.reshape(N, Ho * s, Wo * s, C)
                pt, pl = pool_same_pads(H, s)[0], pool_same_pads(Wd, s)[0]
                d = dxp[:, pt:pt + H, pl:pl + Wd, :]
            elif spec[1] == 'conv':
                W = weights[name][0].astype(np.float64)
                kh, kw, cin, cout = W.shape
                ph, pw = kh // 2, kw // 2
                dz = d * (rec['z'] > 0)
                out[i] = {'dz': dz}
                # dx[y',x',ci] = sum_{dy,dx,co} dz[y'-dy+ph, x'-dx+pw, co] W[dy,dx,ci,co]
                dzp = np.pad(dz, ((0, 0), (ph, ph), (pw, pw), (0, 0)), 'constant')
                win = np.lib.stride_tricks.sliding_window_view(dzp, (kh, kw), axis=(1, 2))
                Wf = W[::-1, ::-1, :, :]                 # flipped taps
                d = np.tensordot(win, Wf, axes=([4, 5, 3], [0, 1, 3]))
    return out


def class_score_factors(layers, weights, x, feature_layer=None):
    """Forward + one backward per class.  Returns (fwd, back) with ``back[y][i]['dz']``
    the gradient of log p_y at layer i's pre-activation for every sample in the batch
    (tf.gradients(log posteriors[y, n]) semantics; the reference only ever feeds one
    sample, NN.py:639-645 uses column 0)."""
    fwd = forward(layers, weights, x, feature_layer, keep_acts=True)
    post = fwd['posteriors']
    c, N = post.shape
    back = []
    for y in range(c):
        e = np.zeros((c, N))
        e[y, :] = 1.
        back.append(_backward(layers, weights, fwd['acts'], e - post))
    return fwd, back


def explicit_class_gradients(layers, weights, x1, y, grad_layers=None):
    """Explicit gradient list [gW_1, gb_1, gW_2, gb_2, ...] of log p_y for ONE
    sample ``x1`` [1,H,W,C] in TF variable shapes and creation order (W then b per
    layer), as ``sess.run(model.grad_posts[str(y)])`` returns (PW_NNAL.py:795-804).
    Small models only (materialises every parameter gradient)."""
    fwd, back = class_score_factors(layers, weights, x1)
    names = [n for n, s in layers if s[1] in ('conv', 'fc')]
    if grad_layers:
        names = list(grad_layers)
    grads = []
    for name in names:
        i = [n for n, _ in layers].index(name)
        spec = layers[i][1]
        rec = fwd['acts'][i]
        dz = back[y][i]['dz']
        if spec[1] == 'fc':
            a = rec['in'][:, 0]
            grads += [np.outer(dz[:, 0], a), dz[:, 0].reshape(-1, 1)]
        else:
            W = weights[name][0]
            kh, kw, cin, cout = W.shape
            ph, pw = kh // 2, kw // 2
            xin = np.pad(rec['in'], ((0, 0), (ph, ph), (pw, pw), (0, 0)), 'constant')
            win = np.lib.stride_tricks.sliding_window_view(xin, (kh, kw), axis=(1, 2))
            # win [1,H,W,C,kh,kw]; gW[kh,kw,ci,co] = sum_pos win[pos,ci,kh,kw] dz[pos,co]
            gW = np.tensordot(win[0], dz[0], axes=([0, 1], [0, 1]))      # [C,kh,kw,co]
            grads += [np.transpose(gW, (1, 2, 0, 3)), dz[0].sum(axis=(0, 1))]
    return grads


def shrink_gradient(grad, method='sum'):
    """NNAL_tools.shrink_gradient(grad,'sum') (NNAL_tools.py:784-796): per layer
    (sum gW + sum gb) / (size W + len b)."""
    if method != 'sum':
        raise ValueError('oracle restates only the "sum" mode used by the query code')
    layer_num = int(len(grad) / 2)
    shrunk = np.zeros(layer_num)
    for t in range(layer_num):
        grW, grb = grad[2 * t], grad[2 * t + 1]
        shrunk[t] = (np.sum(grW) + np.sum(grb)) / (np.prod(grW.shape) + len(grb))
    return np.ravel(shrunk)


def shrunk_class_gradients(layers, weights, x, grad_layers=None, feature_layer=None):
    """Closed form of shrink_gradient(...,'sum') on the factored gradients, for a
    whole batch: returns (post [c,N], g [c,N,tau]).  FC layer: gW = dz a^T ->
    sum gW = (sum dz)(sum a); conv layer: sum gW = sum_pos (sum_co dz)(box-sum over
    the kh x kw window of sum_ci x_padded) (SURVEY §8a row 9)."""
    fwd, back = class_score_factors(layers, weights, x, feature_layer)
    names = [n for n, s in layers if s[1] in ('conv', 'fc')]
    if grad_layers:
        names = list(grad_layers)
    c, N = fwd['posteriors'].shape
    g = np.zeros((c, N, len(names)))
    lnames = [n for n, _ in layers]
    for y in range(c):
        for t, name in enumerate(names):
            i = lnames.index(name)
            spec = layers[i][1]
            rec = fwd['acts'][i]
            dz = back[y][i]['dz']
            W, b = weights[name]
            size = np.prod(W.shape) + len(b)
            if spec[1] == 'fc':
                sdz = dz.sum(axis=0)
                g[y, :, t] = (sdz * rec['in'].sum(axis=0) + sdz) / size
            else:
                kh, kw = W.shape[0], W.shape[1]
                ph, pw = kh // 2, kw // 2
                D = dz.sum(axis=-1)                                   # [N,H,W]
                xs = np.pad(rec['in'].sum(axis=-1), ((0, 0), (ph, ph), (pw, pw)), 'constant')
                box = np.lib.stride_tricks.sliding_window_view(xs, (kh, kw), axis=(1, 2)).sum(axis=(-1, -2))
                g[y, :, t] = ((D * box).sum(axis=(1, 2)) + D.sum(axis=(1, 2))) / size
    return fwd['posteriors'], g


# --------------------------------------------------------------------------
# conditional FI matrices in shrunk coordinates
# --------------------------------------------------------------------------
def gen_A_matrices(g0, g1, sel_posts, diag_load=1e-5):
    """PW_NNAL.gen_A_matrices (PW_NNAL.py:738-816), binary case.  ``g0``/``g1``
    [B,tau] are the shrunk gradients of log p_0 / log p_1, ``sel_posts`` P(class 1).
    p<1e-6 -> p=0 and only g0 is used; p>1-1e-6 -> p=1 and only g1 (:770-793);
    A_i = (1-p) g0 g0^T + p g1 g1^T + diag_load I (:810-814)."""
    A = []
    tau = g0.shape[1]
    for i in range(len(sel_posts)):
        p = sel_posts[i]
        if p < 1e-6:
            p = 0.
            a0, a1 = g0[i], np.zeros(tau)
        elif p > 1 - 1e-6:
            p = 1.
            a0, a1 = np.zeros(tau), g1[i]
        else:
            a0, a1 = g0[i], g1[i]
        Ai = (1. - p) * np.outer(a0, a0) + p * np.outer(a1, a1)
        A += [Ai + np.eye(tau) * diag_load]
    return A


def gen_A_matrices_multiclass(sel_posteriors, g):
    """Multiclass twin inside NNAL.CNN_query (NNAL.py:354-414), restated as
    written: zero posteriors < 1e-6 IN PLACE (:361-362), renormalise the rest,
    keep all if fewer than 10 non-zero classes else the 10 largest renormalised
    (:379-400), A_i = sum_j [ g_j g_j^T / ptilde_j + 1e-5 I ] -- the diagonal load
    is added once PER CLASS (:404-409).  ``g`` is [c,B,tau]."""
    c, B = sel_posteriors.shape
    tau = g.shape[2]
    A = []
    for i in range(B):
        xp = sel_posteriors[:, i]
        xp[xp < 1e-6] = 0.
        nz = np.where(xp > 0.)[0]
        nzp = xp[nz] / np.sum(xp[nz])
        if len(nz) < 10:
            sel_classes, new_posts = nz, nzp
        else:
            sel = stable_topk(-nzp, 10)
            sel_classes = nz[sel]
            new_posts = nzp[sel]
            new_posts = new_posts / np.sum(new_posts)
        Ai = np.zeros((tau, tau))
        for j in range(len(sel_classes)):
            sg = g[sel_classes[j], i]
            Ai += np.outer(sg, sg) / new_posts[j] + np.eye(tau) * 1e-5
        A += [Ai]
    return A


# --------------------------------------------------------------------------
# last-layer factored scores (NN.py:874-955, NNAL_tools.py:725-775, NNAL.py:121-139)
# --------------------------------------------------------------------------
def LLFC_grads(pies, U, labels=None):
    """NN.LLFC_grads (NN.py:905-955): [(e_y - pi) (x) u ; (e_y - pi)] as a
    ((d+1)c, n) matrix; label = argmax posterior if none given (:928-931)."""
    c, n = pies.shape
    d = U.shape[0]
    flag = labels is None
    if flag:
        labels = np.argmax(pies, axis=0)
    hot = np.zeros((c, n))
    for j in range(c):
        hot[j, labels == j] = 1
    rep_U = np.tile(U, (c, 1))
    dJ_dW = np.repeat(hot, d, axis=0) * rep_U - np.repeat(pies, d, axis=0) * rep_U
    dJ_db = hot - pies
    G = np.concatenate((dJ_dW, dJ_db), axis=0)
    return (G, labels) if flag else G


def LLFC_hess(pi, u):
    """NN.LLFC_hess (NN.py:874-903) for one sample: ``pi`` [c,1], ``u`` [d,1];
    A(pi) = diag(pi) (repeat(pi) - I)^T = -(diag pi - pi pi^T); Hessian =
    [[kron(A,uu^T), kron(A,u)],[kron(A,u^T), A]]."""
    d = u.shape[0]
    c = pi.shape[0]
    repM = np.repeat(pi, c, axis=1) - np.eye(c)
    A = np.diag(pi[:, 0]) @ repM.T
    H = np.zeros(((d + 1) * c, (d + 1) * c))
    H[:c * d, :c * d] = np.kron(A, np.outer(u, u))
    H[:c * d, c * d:] = np.kron(A, u)
    H[c * d:, :c * d] = np.kron(A, u.T)
    H[c * d:, c * d:] = A
    return H


def stoch_approx_IF(pool_post, pool_U, tr_post, tr_U, draws, scale=50.):
    """PW_NNAL.stoch_approx_IF (PW_NNAL.py:851-881): stochastic (LiSSA-style) approximation of the influence of the
    pool samples through the last FC layer.  ``grads`` = LLFC_grads of the pool at its predicted (weak) labels (:861-866);
    ``V_0 = grads``; per iteration one random training sample r_t (``draws[t]``; upstream ``np.random.randint(ntr)``,
    :873), ``H = -LLFC_hess`` of it (:874-876), ``V_{t+1} = grads + V_t - H V_t / scale`` (:879).  ``pool_post`` [c,n],
    ``pool_U`` [d,n] = model.posteriors / model.feature_layer of the pool; ``tr_post`` [c,ntr], ``tr_U`` [d,ntr] those of the
    training patches.  Returns (V [(d+1)c, n], weak labels [n]); dense, as written upstream."""
    grads, weak = LLFC_grads(pool_post, pool_U)
    V = grads
    for r in draws:
        H = -LLFC_hess(tr_post[:, r:r + 1], tr_U[:, r:r + 1])
        V = grads + V - H @ V / scale
    return V, weak


def FC_gradnorms_batch(J, fc_inputs, fc_weights):
    """NNAL_tools.FC_gradnorms_batch (NNAL_tools.py:725-775): squared gradient
    norms of the class-0 posterior J0 w.r.t. each FC layer's parameters,
    ||dz||^2 (||a||^2 + 1), back-propagated with ReLU masks (:757-767).
    ``fc_inputs[i]`` is the input activation [d_i,N] of FC layer i and
    ``fc_weights[i]`` its W; ``J`` [2,N] posteriors."""
    L = len(fc_inputs)
    N = J.shape[1]
    norms = np.zeros((L, N))
    W = None
    dz = None
    a = None
    for i in reversed(range(L)):
        if i == L - 1:
            dJ0_da = np.array([J[0, :] * J[1, :], -J[0, :] * J[1, :]])
            fp_z = 1
        else:
            dJ0_da = W.T @ dz
            fp_z = np.array(a > 0, dtype=int)
        a = fc_inputs[i]
        dz = fp_z * dJ0_da
        norms[i, :] = np.sum(dz ** 2, axis=0) * (np.sum(a ** 2, axis=0) + 1.)
        W = fc_weights[i]
    return norms


def fi_trace_score(post, U):
    """Trace of the per-sample last-layer FI, tr((diag pi - pi pi^T) (x) [u;1][u;1]^T)
    = (1 - ||pi||^2)(||u||^2 + 1) (closed form behind NNAL.py:124-139)."""
    return (1. - np.sum(post ** 2, axis=0)) * (np.sum(U ** 2, axis=0) + 1.)


def mnist_fi_score(pool_images, pool_posteriors):
    """The score as written in NNAL.querying_iterations_MNIST (NNAL.py:124-139):
    ``pool_images`` [d,n], ``pool_posteriors`` [n,c];
    (||x||^2/max||x||^2 + 1)(1 - ||p||^2)."""
    norms = np.sum(pool_images ** 2, axis=0)
    norms = norms / norms.max()
    return (norms + 1) * (1 - np.sum(pool_posteriors ** 2, axis=1))


# --------------------------------------------------------------------------
# FI objective and greedy selection
# --------------------------------------------------------------------------
def sdp_objective(A, q):
    """tr((sum_i q_i A_i)^-1): the quantity sum_j t_j the SDP of
    NNAL_tools.py:589-602 / 612-659 minimises at its optimum for a given q."""
    Iq = sum(q[i] * A[i] for i in range(len(A)))
    return np.trace(np.linalg.inv(Iq))


def sdp_certificate(A, q):
    """(phi, gap) for a feasible q: phi = tr(M^-1), M = sum_i q_i A_i, and the duality
    certificate gap = max_i tr(M^-1 A_i M^-1) / phi - 1.  phi is convex in q with
    d phi / d q_i = -tr(M^-1 A_i M^-1) and sum_i q_i tr(M^-1 A_i M^-1) = phi, so
    phi* >= phi - (max_i d_i - phi): the SDP optimum of NNAL_tools.py:612-659 lies within
    ``gap`` (relative) of phi."""
    A = np.asarray(A, dtype=np.float64)
    q = np.asarray(q, dtype=np.float64)
    M = np.tensordot(q, A, axes=(0, 0))
    Mi = np.linalg.inv(M)
    P = Mi @ Mi
    d = np.tensordot(A, P, axes=([1, 2], [0, 1]))
    phi = np.trace(Mi)
    return phi, d.max() / phi - 1.


def sdp_solve(A, tol=1e-4, max_iter=200000, gamma=0.5):
    """Float64 restatement of the query-distribution problem the reference gives cvxopt
    (NNAL_tools.SDP_query_distribution NNAL_tools.py:612-659 with lambda_ = 0: minimise
    sum_j t_j s.t. [[sum q_i A_i, e_j],[e_j^T, t_j]] >= 0, q >= 0, sum q = 1  <=>
    minimise tr((sum_i q_i A_i)^-1) over the simplex), solved by the multiplicative
    algorithm q_i <- q_i (d_i / phi)^gamma until the certificate of ``sdp_certificate``
    drops below ``tol``.  Returns (q, t = diag(M^-1), phi, gap, iterations)."""
    A = np.asarray(A, dtype=np.float64)
    n, tau, _ = A.shape
    Af = A.reshape(n, -1)
    q = np.ones(n) / n
    it = 0
    while True:
        Mi = np.linalg.inv((q @ Af).reshape(tau, tau))
        d = Af @ (Mi @ Mi).ravel()
        phi = np.trace(Mi)
        gap = d.max() / phi - 1.
        if gap <= tol or it >= max_iter:
            return q, np.diag(Mi).copy(), phi, gap, it
        q = q * (d / phi) ** gamma
        q /= q.sum()
        it += 1


def sdp_solve_reg(A, lambda_, X_pool, tol=1e-4, max_iter=20000):
    """The regularised query-distribution problem of NNAL_tools.SDP_query_distribution with ``lambda_ > 0``
    (NNAL_tools.py:625-644): objective ``sum_j t_j - lambda sum_i q_i |x_i|^2`` (``c`` vector :630-632) under the extra
    equalities ``X_pool q = 0`` next to ``sum q = 1`` (:635-644), ``X_pool`` [d, n] = the zero-mean refined feature matrix.
    With t_j = (M^-1)_jj:  minimise  Phi(q) = tr(M(q)^-1) - lambda c^T q,  c_i = |x_i|^2, over {q >= 0, 1^T q = 1, X q = 0}.

    Solved by a multiplicative (natural-gradient) method that keeps EVERY iterate feasible: with d_i = <M^-2, A_i>,
    h = d + lambda c, the multipliers mu of X q = 0 are the weighted regression of h on the features,
    (X diag(q) X^T) mu = X (q.h); then g = h - X^T mu, nu = q.g, and  q_i <- q_i (1 + theta (g_i / nu - 1))  preserves
    1^T q = 1 and X q = 0 for every theta, is a descent direction (dPhi = -theta Var_q(g) / nu) and has the KKT points as
    fixed points.  theta: largest step in (0, 1] that keeps q > 0, halved until Phi decreases (Armijo).  By convexity
    Phi(q) - Phi* <= max_i g_i - nu for any mu: the loop stops when that, relative to |Phi| (or tr M^-1), is below ``tol``.
    Returns (q, t = diag(M^-1), Phi, gap, iterations)."""
    A = np.asarray(A, dtype=np.float64)
    X = np.asarray(X_pool, dtype=np.float64)
    n, tau, _ = A.shape
    Af = A.reshape(n, -1)
    c = np.sum(X ** 2, axis=0)
    q = np.ones(n) / n

    def value(qq):
        Mi = np.linalg.inv((qq @ Af).reshape(tau, tau))
        return np.trace(Mi) - lambda_ * (c @ qq), Mi
    Phi, Mi = value(q)
    it = 0
    while True:
        h = Af @ (Mi @ Mi).ravel() + lambda_ * c
        W = (X * q) @ X.T
        W += np.eye(len(W)) * (1e-14 * np.trace(W) / max(len(W), 1))
        mu = np.linalg.solve(W, X @ (q * h))
        g = h - X.T @ mu
        nu = q @ g
        scale = max(abs(Phi), np.trace(Mi))
        gap = (g.max() - nu) / scale
        if gap <= tol or it >= max_iter:
            return q, np.diag(Mi).copy(), Phi, gap, it
        r = g / nu - 1.
        neg = r < 0
        theta = min(1., 0.99 * np.min(-1. / r[neg])) if neg.any() else 1.
        slope = (q @ (g * g) - nu * nu) / nu                     # = Var_q(g) / nu >= 0
        while True:
            qn = q * (1. + theta * r)
            Pn, Mn = value(qn)
            if Pn <= Phi - 1e-4 * theta * slope or theta < 1e-12:
                break
            theta *= .5
        q, Phi, Mi = qn, Pn, Mn
        it += 1


def sdp_solve_reg_slsqp(A, lambda_, X_pool):
    """Independent check of ``sdp_solve_reg`` for SMALL n: the same convex programme handed to scipy's SLSQP."""
    from scipy.optimize import minimize
    A = np.asarray(A, dtype=np.float64)
    X = np.asarray(X_pool, dtype=np.float64)
    n, tau, _ = A.shape
    Af = A.reshape(n, -1)
    c = np.sum(X ** 2, axis=0)

    def f(q):
        Mi = np.linalg.inv((q @ Af).reshape(tau, tau))
        return np.trace(Mi) - lambda_ * (c @ q), -(Af @ (Mi @ Mi).ravel()) - lambda_ * c
    scale = abs(f(np.ones(n) / n)[0])
    E = np.concatenate([X, np.ones((1, n))], axis=0)
    b = np.zeros(len(E))
    b[-1] = 1.
    res = minimize(lambda q: tuple(v / scale for v in f(q)), np.ones(n) / n, jac=True, method='SLSQP', bounds=[(0., 1.)] * n,
                   constraints=[{'type': 'eq', 'fun': lambda q: E @ q - b, 'jac': lambda q: E}],
                   options={'maxiter': 3000, 'ftol': 1e-15})
    return res.x, f(res.x)[0]


def sdp_solve_slsqp(A, q0=None):
    """Independent check of ``sdp_solve`` for SMALL n: the same convex programme handed to
    scipy's SLSQP (equality sum q = 1, bounds q >= 0, analytic gradient).  Returns (q, phi)."""
    from scipy.optimize import minimize
    A = np.asarray(A, dtype=np.float64)
    n, tau, _ = A.shape
    Af = A.reshape(n, -1)

    def f(q):
        Mi = np.linalg.inv((q @ Af).reshape(tau, tau))
        return np.trace(Mi), -(Af @ (Mi @ Mi).ravel())
    scale = f(np.ones(n) / n)[0]
    res = minimize(lambda q: tuple(v / scale for v in f(q)), np.ones(n) / n if q0 is None else q0, jac=True,
                   method='SLSQP', bounds=[(0., 1.)] * n,
                   constraints=[{'type': 'eq', 'fun': lambda q: q.sum() - 1., 'jac': lambda q: np.ones(n)}],
                   options={'maxiter': 2000, 'ftol': 1e-14})
    q = np.clip(res.x, 0., None)
    q /= q.sum()
    return q, f(q)[0]


def refine_feature_matrix(F, B):
    """PW_NNAL.refine_feature_matrix (PW_NNAL.py:819-849): the int(B/2) feature rows with the most positive entries
    (:826-828), the last one dropped while the matrix is rank deficient (:830-834) and while its condition number exceeds
    1e6 (:837-842, stopping at a single row)."""
    nnz_feats = np.sum(F > 0, axis=1)
    feat_inds = np.argsort(-nnz_feats)[:int(B / 2)]
    ref_F = F[feat_inds, :]
    while np.linalg.matrix_rank(ref_F) < len(feat_inds):
        feat_inds = feat_inds[:-1]
        ref_F = F[feat_inds, :]
    while np.linalg.cond(ref_F) > 1e6:
        feat_inds = feat_inds[:-1]
        ref_F = F[feat_inds, :]
        if len(feat_inds) == 1:
            break
    return ref_F


def query_fi_sdp_single(layers, weights, padded_imgs, pool_inds, patch_shape, ntb, stats, k, B, u,
                        diag_load=1e-5, tol=1e-4, lambda_=0.):
    """PW_NNAL.CNN_query 'fi' as the reference runs it (PW_NNAL.py:89-163) with lambda_ = 0:
    posteriors -> the B most uncertain (:107-115) -> re-gather + normalise (:122-131) ->
    gen_A_matrices in shrunk coordinates (:133-137) -> SDP query distribution (:154-157) ->
    sample_query_dstr with the k uniform draws ``u`` (:160-163).  Returns (positions into
    ``pool_inds``, details)."""
    pool_inds = np.asarray(pool_inds)
    posts = batch_eval(layers, weights, padded_imgs, pool_inds, patch_shape, ntb, stats, 'posteriors')[0]
    if B < len(pool_inds):
        sel = stable_topk(np.abs(posts - .5), B)
    else:
        sel = np.arange(len(pool_inds))
    x = normalize_batch_eval(get_patches(padded_imgs, pool_inds[sel], patch_shape), stats).astype(np.float32)
    post, g = shrunk_class_gradients(layers, weights, x)
    A = gen_A_matrices(g[0], g[1], posts[sel], diag_load)
    ref_F = None
    if lambda_ > 0:
        # PW_NNAL.py:139-155: features of the candidates, refined, rows made zero-mean, regularised programme
        F = batch_eval(layers, weights, padded_imgs, pool_inds[sel], patch_shape, ntb, stats, 'feature_layer')[0]
        ref_F = refine_feature_matrix(F, len(sel) if B >= len(pool_inds) else B)
        ref_F = ref_F - np.repeat(np.expand_dims(np.mean(ref_F, axis=1), axis=1), F.shape[1], axis=1)
        q, t, phi, gap, it = sdp_solve_reg(A, lambda_, ref_F, tol)
    else:
        q, t, phi, gap, it = sdp_solve(A, tol)
    Q = sample_query_dstr(q.copy(), k, u)
    return sel[Q], {'sel': sel, 'A': A, 'q': q, 't': t, 'phi': phi, 'gap': gap, 'g': g, 'post': post, 'x': x, 'ref_F': ref_F}


def query_fi_sdp_multimg(layers, weights, all_padded_imgs, pool_inds, patch_shape, ntb, train_stats, k, B, u,
                         diag_load=1e-3, tol=1e-4):
    """PW_NNAL.query_multimg 'fi' as the reference runs it (PW_NNAL.py:547-627, 'CVXOPT' branch, lambda_ = 0, without
    the live pdb.set_trace() of :612): B most uncertain samples of the concatenated pool (:549-551) -> per-subject
    patches normalised by get_patches_multimg (:554-558) -> A-matrices subject by subject with diag_load 1e-3 and the
    filter's posteriors (:566-578) -> SDP (:601-606) -> sample_query_dstr with the k uniform draws ``u`` (:614-615) ->
    global2local_inds over the per-subject candidate counts (:617-622).  Returns (list of per-subject local positions
    into ``pool_inds[s]``, details)."""
    from .nnal_oracle import bin_uncertainty_filter_multimg, global2local_inds, get_patches_multimg
    s = len(pool_inds)
    sel_inds, sel_posts = bin_uncertainty_filter_multimg(layers, weights, all_padded_imgs, pool_inds, patch_shape, ntb,
                                                         train_stats, B)
    img_inds = [np.array(pool_inds[i])[sel_inds[i]] for i in range(s)]
    patches, _ = get_patches_multimg(all_padded_imgs, img_inds, patch_shape, train_stats)
    A = []
    for i in range(s):
        if len(img_inds[i]) == 0:
            continue
        post, g = shrunk_class_gradients(layers, weights, np.asarray(patches[i]).astype(np.float32))
        A += gen_A_matrices(g[0], g[1], sel_posts[i], diag_load)
    q, t, phi, gap, it = sdp_solve(A, tol)
    draws = sample_query_dstr(q.copy(), k, u)
    sizes = [len(sel_inds[i]) for i in range(s)]
    local = global2local_inds(draws, sizes)
    Q = [np.array(sel_inds[i])[local[i]] for i in range(s)]
    return Q, {'A': A, 'q': q, 'phi': phi, 'gap': gap, 'sel_inds': sel_inds}


def query_fi_sdp_whole(layers, weights, pool_x, k, B, u, tol=1e-4):
    """NNAL.CNN_query 'fi' as the reference runs it (NNAL.py:312-464) with lambda_ = 0 on an in-memory pool ``pool_x``
    [n,H,W,C]: posteriors -> uncertainty_filtering to B (:326-333) -> multiclass A-matrices in shrunk coordinates
    (:354-414) -> SDP query distribution (:456-459) -> sample_query_dstr with the k uniform draws ``u`` (:462-464).
    Returns (positions into the pool, details)."""
    from .nnal_oracle import uncertainty_filtering
    r = forward(layers, weights, pool_x)
    posteriors = r['posteriors']
    if B < posteriors.shape[1]:
        sel = uncertainty_filtering(posteriors, B)
        sel_post = posteriors[:, sel]
    else:
        sel = np.arange(posteriors.shape[1])
        sel_post = posteriors
    post, g = shrunk_class_gradients(layers, weights, pool_x[sel])
    A = gen_A_matrices_multiclass(sel_post, g)
    q, t, phi, gap, it = sdp_solve(A, tol)
    Q = sample_query_dstr(q.copy(), k, u)
    return sel[Q], {'sel': sel, 'A': A, 'q': q, 'phi': phi, 'gap': gap}


def fi_objective_direct(Abar, S, delta):
    """f(S) = tr(((1/|S|) sum_{i in S} Abar_i + delta I)^-1) (definition)."""
    tau = Abar[0].shape[0]
    M = sum(Abar[i] for i in S) / float(len(S)) + delta * np.eye(tau)
    return np.trace(np.linalg.inv(M))


def greedy_fi_direct(Abar, delta, k):
    """Definitional greedy: brute-force evaluation of f(S+j) for every candidate
    at every step.  Returns (indices in selection order, f(S_t) per step)."""
    n = len(Abar)
    S, objs = [], []
    for _ in range(min(k, n)):
        best, bj = None, -1
        for j in range(n):
            if j in S:
                continue
            v = fi_objective_direct(Abar, S + [j], delta)
            if best is None or v < best:
                best, bj = v, j
        S.append(bj)
        objs.append(best)
    return np.array(S), np.array(objs)


def fi_objective_dual(Kss, s, D, delta):
    """f(S) through the kernel (dual / Gram) form.  With Abar_i = Gt_i Gt_i^T
    (Gt_i the D x r_i scaled score factor) and Kss = Gt_S^T Gt_S (r x r):
        f(S) = (D - r)/delta + tr((delta I_r + Kss/s)^-1)
    (the non-zero spectra of Gt Gt^T and Gt^T Gt coincide)."""
    r = Kss.shape[0]
    return (D - r) / delta + np.trace(np.linalg.inv(delta * np.eye(r) + Kss / float(s)))


def greedy_fi_dual_bruteforce(K, rank, D, delta, k):
    """Brute-force greedy on a block kernel ``K`` [(n*rank),(n*rank)] (sample i owns
    rows i*rank..(i+1)*rank-1).  Used for c>2 (rank = c) in config 1."""
    n = K.shape[0] // rank
    S, objs = [], []
    for _ in range(min(k, n)):
        best, bj = None, -1
        for j in range(n):
            if j in S:
                continue
            T = S + [j]
            rows = np.concatenate([np.arange(i * rank, (i + 1) * rank) for i in T])
            v = fi_objective_dual(K[np.ix_(rows, rows)], len(T), D, delta)
            if best is None or v < best:
                best, bj = v, j
        S.append(bj)
        objs.append(best)
    return np.array(S), np.array(objs)


def greedy_fi_rank1(Kt, D, delta, k, return_reduced=False):
    """Incremental greedy for rank-one conditional FIs Abar_i = gt_i gt_i^T with
    scaled kernel Kt_ij = <gt_i, gt_j> (this is the algorithm the CUDA path runs;
    DESIGN.md §FI).  At step t (|S| = t), alpha = (t+1) delta, C = (alpha I +
    Kt_SS)^-1, and for candidate j with k_j = Kt[j,S]:
        r_j = Kt_jj - k_j^T C k_j,   e_j = ||C k_j||^2,
        loss_j = (1 + e_j)/(alpha + r_j)
        f(S+j) = (t+1) [ (D - t)/alpha - 1/alpha + tr(C) ... ]  (see below)
    argmin_j loss_j = argmin_j f(S+j).  Objective after the pick:
        f(S') = (D - s')/delta + tr((delta I + Kt_S'S'/s')^-1),  s' = t+1.
    Returns (indices, f per step[, reduced objective per step]) where the reduced
    objective is the kernel-dependent term tr((delta I + Kt_SS/s)^-1)."""
    n = Kt.shape[0]
    diag = np.diag(Kt).copy()
    S, objs, red = [], [], []
    avail = np.ones(n, dtype=bool)
    for t in range(min(k, n)):
        alpha = (t + 1) * delta
        if t == 0:
            r = diag.copy()
            e = np.zeros(n)
        else:
            Kss = Kt[np.ix_(S, S)]
            C = np.linalg.inv(alpha * np.eye(t) + Kss)
            kjs = Kt[:, S]                       # [n,t]
            Y = kjs @ C
            r = diag - np.sum(Y * kjs, axis=1)
            e = np.sum(Y * Y, axis=1)
        loss = (1. + e) / (alpha + r)
        loss[~avail] = np.inf
        j = int(np.argmin(loss))                 # first minimum = lowest position
        S.append(j)
        avail[j] = False
        s = t + 1
        Kss = Kt[np.ix_(S, S)]
        rv = np.trace(np.linalg.inv(delta * np.eye(s) + Kss / float(s)))
        red.append(rv)
        objs.append((D - s) / delta + rv)
    if return_reduced:
        return np.array(S), np.array(objs), np.array(red)
    return np.array(S), np.array(objs)


def last_layers_dim(c, d, d_prev=None):
    """Parameter count D of the last FC layer ((d+1)c, NN.py:891-901) plus, if
    ``d_prev`` is given, the previous FC layer (d (d_prev+1))."""
    D = (d + 1) * c
    if d_prev is not None:
        D += d * (d_prev + 1)
    return D


def last_layers_kernel(p1, U, A_prev=None, W_last=None):
    """Scaled score kernel Kt_ij = sqrt(w_i w_j) <gbar_i, gbar_j> for the BINARY
    model (c=2), w_i = p_i (1-p_i).  Last layer: gbar_i = v (x) [u_i;1], v=(1,-1)
    (F_i = (diag pi - pi pi^T) (x) ut ut^T = w_i (v v^T) (x) ut ut^T, NN.py:891-901),
    so <gbar_i,gbar_j> = 2 (u_i.u_j + 1).  With ``A_prev``/``W_last`` the previous FC
    layer's factor is added (FC_gradnorms_batch back-propagation,
    NNAL_tools.py:757-767): delta2_i = (W_last^T v) * 1[u_i>0], gradient
    delta2_i (x) [a_i;1], inner product (delta2_i.delta2_j)(a_i.a_j + 1)."""
    w = p1 * (1. - p1)
    K = 2. * (U.T @ U + 1.)
    if A_prev is not None:
        v = np.array([1., -1.])
        beta = (W_last.T @ v)                       # [d]
        Mk = (U > 0) * beta[:, None]                # [d,n] masked back-prop signal
        K = K + (Mk.T @ Mk) * (A_prev.T @ A_prev + 1.)
    sw = np.sqrt(w)
    return K * sw[:, None] * sw[None, :]


def weighted_gram(U, wq):
    """Weighted penultimate-feature Gram  H = Ut diag(wq) Ut^T, Ut = [U;1]
    ((d+1) x (d+1)); for c=2 the pool FI sum_i q_i F_i equals (v v^T) (x) H with
    wq_i = q_i p_i (1-p_i) (SURVEY §8a row 11)."""
    Ut = np.concatenate([U, np.ones((1, U.shape[1]))], axis=0)
    return (Ut * wq[None, :]) @ Ut.T


def fi_objective_from_gram(H, c, delta):
    """tr((delta I + (v v^T) (x) H)^-1) for c=2 through the (d+1)^2 Gram only:
    (D - (d+1))/delta + tr((delta I + 2H)^-1)   (||v||^2 = 2)."""
    assert c == 2
    d1 = H.shape[0]
    D = c * d1
    return (D - d1) / delta + np.trace(np.linalg.inv(delta * np.eye(d1) + 2. * H))


# --------------------------------------------------------------------------
# sampling from a query distribution (NNAL_tools.py:844-896, :833-842)
# --------------------------------------------------------------------------
def sample_query_dstr(q_dstr, k, u):
    """NNAL_tools.sample_query_dstr with replacement=True (NNAL_tools.py:844-872)
    with the k uniform draws ``u`` supplied by the caller (the reference draws
    them from the global unseeded np.random): clamp negatives IN PLACE, inverse
    CDF, np.unique, clip index n -> n-1."""
    q_dstr[q_dstr < 0] = 0.
    Q = np.unique(q_dstr.cumsum().searchsorted(np.asarray(u)[:k]))
    Q[Q == len(q_dstr)] = len(q_dstr) - 1
    return Q


def append_zero(A):
    """NNAL_tools.append_zero (NNAL_tools.py:833-842)."""
    d = A.shape[0]
    A = np.insert(A, d, 0, axis=1)
    return np.insert(A, d, 0, axis=0)


# --------------------------------------------------------------------------
# the adopted FI query (DESIGN.md, FI section): reference pipeline shape
# (pre-filter to B, conditional FIs of the B candidates, pick k) with the
# factored last-layer FI and the deterministic greedy selection
# --------------------------------------------------------------------------
def last_layers_factors(layers, weights, x):
    """Factors of the last two FC layers for a batch ``x`` [N,H,W,C]: P(class 1) [N],
    U [d,N] (input of the last FC = model.feature_layer for PW1, NN.py:1346),
    A_prev [d_prev,N] (input of the FC before it) and W_last [c,d]."""
    fwd = forward(layers, weights, x, keep_acts=True)
    acts = fwd['acts']
    return (fwd['posteriors'][1], acts[-1]['in'], acts[-2]['in'],
            weights[layers[-1][0]][0].astype(np.float64))


def greedy_fi_replay(Kt, D, delta, S):
    """Replays a given selection sequence ``S`` through the greedy criterion of
    ``greedy_fi_rank1``: for every step returns (loss of S[t], best available loss,
    objective after taking S[t]).  Used to accept selections that differ from the
    oracle's only at ties within tolerance."""
    n = Kt.shape[0]
    diag = np.diag(Kt).copy()
    avail = np.ones(n, dtype=bool)
    out = []
    for t in range(len(S)):
        alpha = (t + 1) * delta
        prev = list(S[:t])
        if t == 0:
            r, e, trC = diag.copy(), np.zeros(n), 0.
        else:
            C = np.linalg.inv(alpha * np.eye(t) + Kt[np.ix_(prev, prev)])
            kjs = Kt[:, prev]
            Y = kjs @ C
            r = diag - np.sum(Y * kjs, axis=1)
            e = np.sum(Y * Y, axis=1)
            trC = np.trace(C)
        loss = (1. + e) / (alpha + r)
        loss[~avail] = np.inf
        j = int(S[t])
        assert avail[j], 'selection repeats a candidate'
        s = t + 1
        obj = (D - s) / delta + s * (trC + loss[j])
        out.append((loss[j], loss.min(), obj))
        avail[j] = False
    return np.array(out)


def _fi_select(p1, U, A_prev, W_last, k, n_layers, delta):
    two = n_layers == 2
    Kt = last_layers_kernel(p1, U, A_prev if two else None, W_last if two else None)
    D = last_layers_dim(2, U.shape[0], A_prev.shape[0] if two else None)
    S, obj = greedy_fi_rank1(Kt, D, delta, k)
    return S, obj, Kt, D


def query_fi_single(layers, weights, padded_imgs, pool_inds, patch_shape, ntb, stats, k, B,
                    n_layers=2, delta=1e-5):
    """PW_NNAL.CNN_query 'fi' (PW_NNAL.py:89-163) with the adopted selection:
    posteriors -> uncertainty pre-filter to B (:108-115) -> re-gather + normalise the B
    patches (:122-130) -> factored FIs -> greedy k.  Returns (positions into
    ``pool_inds`` in selection order, objective per step, details)."""
    pool_inds = np.asarray(pool_inds)
    posts = batch_eval(layers, weights, padded_imgs, pool_inds, patch_shape, ntb, stats, 'posteriors')[0]
    if B < len(pool_inds):
        sel = stable_topk(np.abs(posts - .5), B)
    else:
        sel = np.arange(len(pool_inds))
    x = normalize_batch_eval(get_patches(padded_imgs, pool_inds[sel], patch_shape), stats).astype(np.float32)
    p1, U, A_prev, W_last = last_layers_factors(layers, weights, x)
    S, obj, Kt, D = _fi_select(p1, U, A_prev, W_last, k, n_layers, delta)
    return sel[S], obj, {'sel': sel, 'Kt': Kt, 'D': D, 'p1': p1, 'U': U, 'A_prev': A_prev, 'W_last': W_last,
                         'posts': posts, 'S': S}


def query_fi_multimg(layers, weights, all_padded_imgs, pool_inds, patch_shape, ntb, train_stats, k, B,
                     n_layers=2, delta=1e-3):
    """PW_NNAL.query_multimg 'fi' (PW_NNAL.py:547-627) with the adopted selection;
    candidate order subject-major as the reference's ``A +=`` loop (:566-578).
    Returns (list of per-subject local positions, objective per step, details)."""
    from .nnal_oracle import bin_uncertainty_filter_multimg, global2local_inds
    s = len(pool_inds)
    m = len(all_padded_imgs[0]) - 1
    sel_inds, sel_posts = bin_uncertainty_filter_multimg(layers, weights, all_padded_imgs, pool_inds,
                                                         patch_shape, ntb, train_stats, B)
    P, Us, As = [], [], []
    W_last = None
    for i in range(s):
        if len(sel_inds[i]) == 0:
            continue
        stats = [[train_stats[i, 2 * j], train_stats[i, 2 * j + 1]] for j in range(m)]
        vox = np.asarray(pool_inds[i])[sel_inds[i]]
        x = normalize_batch_eval(get_patches(all_padded_imgs[i][:m], vox, patch_shape), stats).astype(np.float32)
        p1, U, A_prev, W_last = last_layers_factors(layers, weights, x)
        P.append(p1); Us.append(U); As.append(A_prev)
    p1, U, A_prev = np.concatenate(P), np.concatenate(Us, axis=1), np.concatenate(As, axis=1)
    S, obj, Kt, D = _fi_select(p1, U, A_prev, W_last, k, n_layers, delta)
    sizes = [len(sel_inds[i]) for i in range(s)]
    local = global2local_inds(S, sizes)
    Q = [np.array(sel_inds[i])[local[i]] for i in range(s)]
    return Q, obj, {'Kt': Kt, 'D': D, 'S': S, 'sel_inds': sel_inds}
