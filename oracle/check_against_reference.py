"""Pin the oracle against the reference's own pure-NumPy functions and write the
golden vectors in tests/golden/.

The reference (the original nn-active-learning sources, read-only, at $NNAL_REFERENCE) is
imported IN PLACE under ``sys.modules`` stubs for its missing third-party imports
(SURVEY.md §4); only its NumPy-only helpers are executed, unchanged.  This script is the
generator of every file in tests/golden/; the tests need only those files.

    NNAL_REFERENCE=<tree> python oracle/check_against_reference.py     # check + (re)write goldens
"""
import os
import sys
import warnings
from unittest.mock import MagicMock

import numpy as np

REF = os.environ.get('NNAL_REFERENCE')
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
GOLD = os.environ.get('NNAL_GOLD_OUT', os.path.join(ROOT, 'tests', 'golden'))   # NNAL_GOLD_OUT: check only, write elsewhere


def import_reference():
    if not REF or not os.path.isdir(REF):
        sys.exit('set NNAL_REFERENCE to the directory of the original nn-active-learning sources')
    for m in ['tensorflow', 'tensorflow.examples', 'tensorflow.examples.tutorials',
              'tensorflow.examples.tutorials.mnist', 'tensorflow.python',
              'tensorflow.python.ops', 'tensorflow.python.framework', 'nrrd', 'cvxopt',
              'cvxpy', 'h5py', 'cv2', 'alexnet', 'skimage', 'skimage.measure',
              'skimage.segmentation', 'skimage.util', 'nibabel', 'imageio', 'matplotlib',
              'matplotlib.pyplot', 'pydensecrf', 'pydensecrf.utils', 'pydensecrf.densecrf']:
        sys.modules.setdefault(m, MagicMock())
    sys.path.insert(0, REF)
    import patch_utils, NNAL_tools, PW_NNAL, PW_NN   # noqa: E401
    return patch_utils, NNAL_tools, PW_NNAL, PW_NN


def main():
    sys.path.insert(0, ROOT)
    import oracle as O
    ref_pu, ref_tools, ref_pw, ref_pwnn = import_reference()
    os.makedirs(GOLD, exist_ok=True)
    gold = {}

    # ---- gather: bit-exact vs patch_utils.get_patches (padded / unpadded / mask / d3>1)
    rs = np.random.RandomState(10)
    cases = [((9, 8, 5), (3, 3, 1), 2, np.float32), ((11, 10, 7), (5, 3, 3), 3, np.float64),
             ((30, 29, 6), (25, 25, 1), 3, np.float32), ((6, 6, 6), (1, 1, 1), 1, np.int16)]
    for ci, (shape, ps, m, dt) in enumerate(cases):
        rads = [(p - 1) // 2 for p in ps]
        imgs = [(rs.randn(*shape) * 50 + 100).astype(dt) for _ in range(m)]
        padded = [np.pad(im, tuple((r, r) for r in rads), 'constant') for im in imgs]
        mask = (rs.rand(*shape) > .5).astype(np.int32)
        inds = rs.choice(int(np.prod(shape)), 17, replace=False)
        inds[:4] = [0, np.prod(shape) - 1, shape[2] - 1, shape[1] * shape[2]]   # corners
        r1 = ref_pu.get_patches(padded, inds, ps)
        o1 = O.get_patches(padded, inds, ps)
        assert r1.dtype == o1.dtype == np.float64 and np.array_equal(r1, o1), ci
        r2, l2 = ref_pu.get_patches(imgs, inds, ps, False, mask)
        o2, ol2 = O.get_patches(imgs, inds, ps, False, mask)
        assert np.array_equal(r2, o2) and np.array_equal(l2, ol2) and np.array_equal(r1, r2)
        gold['gather%d_imgs' % ci] = np.stack(padded)
        gold['gather%d_inds' % ci] = inds
        gold['gather%d_pshape' % ci] = np.array(ps)
        gold['gather%d_out' % ci] = r1
        gold['gather%d_labels' % ci] = l2
    print('get_patches: oracle == reference (bit-exact) on %d cases' % len(cases))

    # ---- multi-image gather + normalise
    S, m, ps = 3, 2, (5, 5, 1)
    shape = (12, 11, 4)
    allp, img_inds = [], []
    for s in range(S):
        imgs = [(rs.randn(*shape) * 30 + 100).astype(np.float32) for _ in range(m)]
        padded = [np.pad(im, ((2, 2), (2, 2), (0, 0)), 'constant') for im in imgs]
        allp.append(padded + [(rs.rand(*shape) > .7).astype(np.int8)])
        img_inds.append(list(rs.choice(int(np.prod(shape)), [6, 0, 9][s], replace=False)))
    stats = np.abs(rs.randn(S, 2 * m)) * 20 + 50
    rp, rl = ref_pu.get_patches_multimg(allp, img_inds, ps, stats)
    op, ol = O.get_patches_multimg(allp, img_inds, ps, stats)
    for s in range(S):
        assert np.array_equal(np.asarray(rp[s]), np.asarray(op[s]))
        assert np.array_equal(np.asarray(rl[s]), np.asarray(ol[s]))
    gold['multi_imgs'] = np.stack([np.stack(a[:m]) for a in allp])
    gold['multi_masks'] = np.stack([a[m] for a in allp])
    for s in range(S):
        gold['multi_inds%d' % s] = np.array(img_inds[s], dtype=np.int64)
        gold['multi_out%d' % s] = np.asarray(rp[s], dtype=np.float64)
        gold['multi_labels%d' % s] = np.asarray(rl[s])
    gold['multi_stats'] = stats
    print('get_patches_multimg: oracle == reference (bit-exact)')

    # ---- global2local_inds (known answer from SURVEY §4 + random)
    ka = ref_pu.global2local_inds([0, 3, 4, 9, 2], [3, 2, 5])
    assert [list(a) for a in ka] == [[0, 2], [0, 1], [4]]
    gi = rs.permutation(40)[:23]
    sizes = [7, 0, 13, 20]
    rr = ref_pu.global2local_inds(gi, sizes)
    oo = O.global2local_inds(gi, sizes)
    assert all(np.array_equal(a, b) for a, b in zip(rr, oo))
    gold['g2l_inds'] = gi
    gold['g2l_sizes'] = np.array(sizes)
    for i, a in enumerate(rr):
        gold['g2l_out%d' % i] = a
    print('global2local_inds: oracle == reference')

    # ---- entropy / uncertainty filtering (incl. in-place zero bump)
    P = rs.dirichlet(np.ones(4), size=50).T
    P[:, 3] = [1, 0, 0, 0]
    P[:, 7] = [.5, .5, 0, 0]
    Pa, Pb = P.copy(), P.copy()
    re_, oe = ref_tools.compute_entropy(Pa), O.compute_entropy(Pb)
    assert np.array_equal(re_, oe) and np.array_equal(Pa, Pb) and Pa[1, 3] == 10e-8
    ka = ref_tools.compute_entropy(np.array([[.5, 1, .2], [.5, 0, .8]]))
    assert np.allclose(ka, [0.693147181, 1.61180957e-06, 0.500402424], rtol=1e-8)
    gold['entropy_P'] = P
    gold['entropy_H'] = re_
    Pa, Pb = P.copy(), P.copy()
    ru, ou = ref_tools.uncertainty_filtering(Pa, 9), O.uncertainty_filtering(Pb, 9)
    assert np.array_equal(ru, ou) and np.array_equal(Pa, Pb) and Pa[1, 3] == 1e-8
    gold['unc_sel'] = ru
    posts = rs.rand(200)
    rb, ob = ref_pw.binary_uncertainty_filter(posts, 20), O.binary_uncertainty_filter(posts, 20)
    assert np.array_equal(rb, ob)
    gold['bin_posts'] = posts
    gold['bin_sel'] = rb
    print('compute_entropy / uncertainty_filtering / binary_uncertainty_filter: oracle == reference')

    # ---- shrink_gradient on explicit gradients of a small net; closed form agrees
    ka = ref_tools.shrink_gradient([np.ones((2, 3)), 2 * np.ones(2),
                                    np.arange(4).reshape(2, 2), np.zeros(2)], 'sum')
    assert np.allclose(ka, [1.25, 1.0])
    layers = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']),
              ('conv2', [6, 'conv', [3, 3]]), ('max2', [[2, 2], 'pool']),
              ('fc1', [16, 'fc']), ('fc2', [12, 'fc']), ('fc3', [3, 'fc'])]
    w = O.he_init_weights(layers, (7, 7, 2), 11, bias_scale=0.1)
    x = rs.randn(3, 7, 7, 2)
    post, g = O.shrunk_class_gradients(layers, w, x)
    for n in range(3):
        for y in range(3):
            grads = O.explicit_class_gradients(layers, w, x[n:n + 1], y)
            rsg = ref_tools.shrink_gradient(grads, 'sum')
            assert np.allclose(rsg, O.shrink_gradient(grads, 'sum'), rtol=0, atol=0)
            assert np.allclose(rsg, g[y, n], rtol=1e-9, atol=1e-15), (rsg, g[y, n])
    gold['shrink_x'] = x
    gold['shrink_g'] = g
    gold['shrink_post'] = post
    print('shrink_gradient: reference(explicit grads) == oracle closed form')

    # ---- sample_query_dstr with injected uniforms; append_zero
    q = rs.dirichlet(np.ones(30))
    q[3] = -1e-3
    u = rs.rand(8)
    state = np.random.get_state()
    np.random.seed(123)
    u123 = np.random.sample(8)
    np.random.seed(123)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        rq = ref_tools.sample_query_dstr(q.copy(), 8, replacement=True)
    np.random.set_state(state)
    oq = O.sample_query_dstr(q.copy(), 8, u123)
    assert np.array_equal(rq, oq)
    gold['sample_q'] = q
    gold['sample_u'] = u123
    gold['sample_out'] = rq
    A = rs.randn(3, 3)
    assert np.array_equal(ref_tools.append_zero(A), O.append_zero(A))
    print('sample_query_dstr / append_zero: oracle == reference')

    # ---- similarity helpers and the greedy loops of the representativeness queries
    F1 = np.maximum(rs.randn(16, 40), 0)
    F2 = np.maximum(rs.randn(16, 23), 0)
    r_self, r_cross = ref_pw.get_self_sims(F1), ref_pw.get_cross_sims(F1, F2)
    assert np.allclose(r_self, O.get_self_sims(F1), rtol=1e-13) and np.allclose(r_cross, O.get_cross_sims(F1, F2), rtol=1e-13)
    gold['sims_F1'], gold['sims_F2'], gold['sims_self'], gold['sims_cross'] = F1, F2, r_self, r_cross
    # the literal greedy facility-location loop of NNAL.py:506-521 / PW_NNAL.py:329-343 (copied control flow, run on
    # the reference's arithmetic: np.sum(np.max(sims[:, cand_Q], axis=1)) / np.argmax / np.delete)
    sims = O.cosine_sims(F1[:, :25], F1[:, 25:])
    B, k = sims.shape[1], 6
    Q_inds, nQ = [], np.arange(B)
    for i in range(k):
        rep = np.zeros(B - i)
        for j in range(B - i):
            rep[j] = np.sum(np.max(sims[:, Q_inds + [nQ[j]]], axis=1))
        Q_inds += [nQ[np.argmax(rep)]]
        nQ = np.delete(nQ, np.argmax(rep))
    assert np.array_equal(Q_inds, O.greedy_facility_location(sims, k)[0])
    gold['fl_sims'], gold['fl_Q'] = sims, np.array(Q_inds)
    # the k-center loop of PW_NNAL.py:437-448
    Fu = F1
    norms_u = np.sqrt(np.sum(Fu ** 2, axis=0))
    s0 = r_cross.copy()
    sims1, Qk = s0.copy(), []
    for t in range(5):
        q_ind = np.argmin(sims1)
        Qk += [q_ind]
        s_ind = np.dot(Fu[:, q_ind].T, Fu) / (norms_u * norms_u[q_ind])
        sims1 = np.maximum(sims1, s_ind)
        sims1[q_ind] = np.inf
    assert np.array_equal(Qk, O.kcenter_greedy(Fu, s0, 5)[0])
    gold['kc_Q'] = np.array(Qk)
    print('get_self_sims / get_cross_sims / facility-location / k-center loops: oracle == reference')

    # ---- the SDP the reference hands to cvxopt (NNAL_tools.SDP_query_distribution :612-659 with lambda_ = 0, constraint
    # matrices from inequality_cvx_matrix :661-720), captured from the UNMODIFIED reference functions: cvxopt itself is
    # absent, so `matrix` is replaced by a shape-preserving float64 array type (what cvxopt.matrix makes of a NumPy array)
    # and `solvers.sdp` by a recorder.  The oracle's solution must be feasible for exactly these constraints and its
    # objective c^T x must equal tr((sum q_i A_i)^-1): this pins the PROGRAMME (not cvxopt's arithmetic).
    class FakeMatrix(np.ndarray):
        def __new__(cls, a):
            arr = np.array(a, dtype=np.float64)
            if arr.ndim == 0:
                arr = arr.reshape(1, 1)
            elif arr.ndim == 1:
                arr = arr.reshape(-1, 1)              # cvxopt makes a column of a 1-D array
            return arr.view(cls)

        def trans(self):
            return FakeMatrix(np.asarray(self).T)

    captured = {}

    class FakeSolvers(object):
        options = {}

        @staticmethod
        def sdp(c, Gs=None, hs=None, A=None, b=None):
            captured.update(c=np.asarray(c), Gs=[np.asarray(g) for g in Gs], hs=[np.asarray(h) for h in hs],
                            A=np.asarray(A), b=np.asarray(b))
            return {'status': 'captured', 'x': np.zeros(len(c))}

    ref_tools.matrix, ref_tools.solvers = FakeMatrix, FakeSolvers
    n_s, tau_s = 12, 3
    sg = rs.randn(2, n_s, tau_s) * 0.05
    sp = rs.rand(n_s)
    A_s = O.gen_A_matrices(sg[0], sg[1], sp, 1e-3)
    ref_tools.SDP_query_distribution(A_s, 0., None, 5)
    c_vec, Gs, hs, A_eq, b_eq = captured['c'], captured['Gs'], captured['hs'], captured['A'], captured['b']
    assert c_vec.shape == (n_s + tau_s, 1) and len(Gs) == tau_s + 1 and A_eq.shape == (1, n_s + tau_s)
    qs, ts, phis, gaps, its = O.sdp_solve(A_s, 1e-8)
    xs = np.concatenate([qs, ts])
    assert abs((A_eq @ xs).item() - b_eq.item()) < 1e-12                      # sum q = 1
    assert abs((c_vec[:, 0] @ xs).item() - phis) < 1e-9 * phis                # objective = sum_j t_j = tr(M^-1)
    M_s = np.tensordot(qs, np.array(A_s), axes=(0, 0))
    for j in range(tau_s + 1):
        m = int(round(np.sqrt(Gs[j].shape[0])))
        slack = (hs[j] - (Gs[j] @ xs).reshape(m, m)).astype(np.float64)     # cvxopt: G x + s = h, s >= 0 (PSD)
        slack = (slack + slack.T) / 2
        assert np.linalg.eigvalsh(slack).min() > -1e-9 * np.abs(slack).max(), j
        if j < tau_s:                                                       # [[sum q_i A_i, e_j], [e_j^T, t_j]]
            e = np.zeros((tau_s, 1)); e[j] = 1
            blk = np.block([[M_s, e], [e.T, np.array([[ts[j]]])]])
            assert np.allclose(slack, blk, rtol=1e-12, atol=1e-15), j
        else:                                                               # positivity block: diag(q)
            assert np.allclose(slack, np.diag(qs), rtol=1e-12, atol=1e-15)
    gold['sdp_A'] = np.array(A_s)
    gold['sdp_c'] = c_vec
    for j in range(tau_s + 1):
        gold['sdp_G%d' % j] = Gs[j]
        gold['sdp_h%d' % j] = hs[j]
    gold['sdp_Aeq'], gold['sdp_beq'] = A_eq, b_eq
    gold['sdp_q'], gold['sdp_t'], gold['sdp_phi'] = qs, ts, np.array(phis)
    # the same with lambda_ > 0 (:625-644): c = [-lambda |x_i|^2 ; 1], equalities [X_pool, 0; 1^T, 0] x = [0; 1].  The oracle's
    # feasible multiplicative solver must satisfy exactly these constraints, with c^T x = tr(M^-1) - lambda sum q_i |x_i|^2.
    lam_s = 0.3
    X_s = np.maximum(rs.randn(4, n_s), 0)
    X_s = X_s - X_s.mean(axis=1, keepdims=True)
    ref_tools.SDP_query_distribution(A_s, lam_s, X_s, 5)
    c_r, A_r, b_r = captured['c'], captured['A'], captured['b']
    assert A_r.shape == (5, n_s + tau_s) and b_r.shape[0] == 5
    qr, tr_, Phir, gapr, itr = O.sdp_solve_reg(A_s, lam_s, X_s, 1e-9)
    xr = np.concatenate([qr, tr_])
    assert np.abs(A_r @ xr - b_r[:, 0]).max() < 1e-12                          # X q = 0 and sum q = 1
    assert abs((c_r[:, 0] @ xr).item() - Phir) < 1e-9 * abs(Phir)             # objective = sum t_j - lambda sum q_i |x_i|^2
    assert qr.min() >= 0
    q_sl, Phi_sl = O.sdp_solve_reg_slsqp(A_s, lam_s, X_s)
    assert abs(Phir / Phi_sl - 1) < 1e-6
    gold['sdpr_X'], gold['sdpr_lambda'] = X_s, np.array(lam_s)
    gold['sdpr_c'], gold['sdpr_Aeq'], gold['sdpr_beq'] = c_r, A_r, b_r
    gold['sdpr_q'], gold['sdpr_Phi'] = qr, np.array(Phir)
    print('SDP_query_distribution / inequality_cvx_matrix: the reference\'s programme (captured c, G, h, A, b) == '
          'min tr((sum q_i A_i)^-1) over the simplex; oracle solution feasible, objective equal')

    # ---- PW_NNAL.gen_A_matrices (:738-816), UNMODIFIED, driven by a fake session whose run() returns the explicit
    # tf.gradients-shaped lists [gW_1, gb_1, ...] of the float64 restatement: pins the per-sample loop, the two clamped
    # branches, shrink_gradient and the diagonal load against the oracle's closed form on the factored gradients.
    layers_b = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('conv2', [6, 'conv', [3, 3]]),
                ('fc1', [10, 'fc']), ('fc2', [2, 'fc'])]
    w_b = O.he_init_weights(layers_b, (7, 7, 2), 13, bias_scale=0.1)
    xb = rs.randn(6, 7, 7, 2)
    tau_b = 4

    class FakeModel(object):
        x, keep_prob = 'x', 'keep_prob'
        grad_posts = {'0': [(0, t) for t in range(2 * tau_b)], '1': [(1, t) for t in range(2 * tau_b)]}

    class FakeSess(object):
        def run(self, fetches, feed_dict=None):
            y = fetches[0][0]
            return O.explicit_class_gradients(layers_b, w_b, feed_dict['x'], y)

    class FakeExpr(object):
        pars = {'patch_shape': (7, 7, 1)}
        nclass = 2
    post_b, g_b = O.shrunk_class_gradients(layers_b, w_b, xb)
    sel_posts_b = post_b[1].copy()
    sel_posts_b[0], sel_posts_b[1] = 1e-7, 1 - 1e-7                          # the clamped branches (:770-793)
    A_ref = ref_pw.gen_A_matrices(FakeExpr(), FakeModel(), FakeSess(), xb, sel_posts_b, 1e-5)
    A_ora = O.gen_A_matrices(g_b[0], g_b[1], sel_posts_b, 1e-5)
    assert len(A_ref) == 6 and A_ref[0].shape == (tau_b, tau_b)
    for a, b in zip(A_ref, A_ora):
        assert np.allclose(a, b, rtol=1e-9, atol=1e-18)
    gold['genA_x'], gold['genA_posts'], gold['genA_out'] = xb, sel_posts_b, np.array(A_ref)
    print('gen_A_matrices: reference (fake session with explicit gradients) == oracle closed form')

    # ---- the query dispatch itself, UNMODIFIED, over a fake TF session: PW_NN.batch_eval (:357-539; batching, gather,
    # normalisation, sess.run, P(class 1) slice), PW_NNAL.CNN_query 'entropy' (:51-65), bin_uncertainty_filter_multimg
    # (:684-736) and query_multimg 'entropy' (:226-230).  sess.run(model.posteriors / feature_layer) is answered by the
    # float64 restatement of the TF graph on the float32-cast feed (TF casts the float64 patches to the placeholder's
    # float32), so everything AROUND the graph is the reference's own code.
    from collections import OrderedDict   # noqa: F401
    ps_q, m_q, S_q = (5, 5, 1), 2, 3
    shape_q = (12, 11, 4)
    layers_q = [('conv1', [4, 'conv', [3, 3]]), ('max1', [[2, 2], 'pool']), ('fc1', [16, 'fc']), ('fc2', [12, 'fc']),
                ('fc3', [2, 'fc'])]
    w_q = O.he_init_weights(layers_q, (5, 5, m_q), 7, bias_scale=0.1)
    fl_q = len(layers_q) - 2

    class FakeDim(object):
        def __init__(self, v):
            self.value = v

    class FakeTensor(object):
        def __init__(self, name, shape):
            self.name, self.shape = name, [FakeDim(d) for d in shape]

    class QModel(object):
        x, keep_prob = 'x', 'keep_prob'
        posteriors = FakeTensor('posteriors', (2, None))
        feature_layer = FakeTensor('feature_layer', (12, None))

    class QSess(object):
        def run(self, var, feed_dict=None):
            r = O.forward(layers_q, w_q, np.asarray(feed_dict['x']).astype(np.float32), feature_layer=fl_q)
            return r[var.name]

    allp_q, pools_q, st_q = [], [], np.zeros((S_q, 2 * m_q))
    for s_ in range(S_q):
        imgs = [np.clip(rs.randn(*shape_q) * 30 + 100, 0, None).astype(np.float32) for _ in range(m_q)]
        allp_q.append([np.pad(im, ((2, 2), (2, 2), (0, 0)), 'constant') for im in imgs] +
                      [(rs.rand(*shape_q) > .5).astype(np.int8)])
        pools_q.append(list(rs.choice(int(np.prod(shape_q)), [70, 0, 95][s_], replace=False)))
        for j in range(m_q):
            st_q[s_, 2 * j], st_q[s_, 2 * j + 1] = imgs[j].mean(), imgs[j].std()
    stats0 = [[st_q[0, 2 * j], st_q[0, 2 * j + 1]] for j in range(m_q)]
    pool0 = np.array(pools_q[0])

    class QExpr(object):
        pars = dict(k=9, B=30, lambda_=0., patch_shape=ps_q, ntb=16, stats=stats0, img_paths=[None] * m_q)
        train_stats = st_q
        nclass = 2
    # batch_eval: posteriors and feature_layer, batch size not dividing n
    rp, rf = ref_pwnn.batch_eval(QModel(), QSess(), allp_q[0][:m_q], pool0, ps_q, 16, stats0, ['posteriors', 'feature_layer'])
    op_, of_ = O.batch_eval(layers_q, w_q, allp_q[0][:m_q], pool0, ps_q, 16, stats0, ['posteriors', 'feature_layer'])
    assert np.array_equal(rp, op_) and np.array_equal(rf, of_)
    # single-volume entropy query
    rq = ref_pw.CNN_query(QExpr(), QModel(), QSess(), allp_q[0][:m_q], pool0, None, 'entropy')
    oq, _ = O.query_entropy_single(layers_q, w_q, allp_q[0][:m_q], pool0, ps_q, 16, stats0, 9)
    assert np.array_equal(rq, oq)
    # multi-volume filter and entropy query (one subject with an empty pool)
    rsel, rposts = ref_pw.bin_uncertainty_filter_multimg(QExpr(), QModel(), QSess(), allp_q, pools_q, 25)
    osel, oposts = O.bin_uncertainty_filter_multimg(layers_q, w_q, allp_q, pools_q, ps_q, 16, st_q, 25)
    for a, b in zip(rsel, osel):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    for a, b in zip(rposts, oposts):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    rQ = ref_pw.query_multimg(QExpr(), QModel(), QSess(), allp_q, pools_q, None, 'entropy')
    oQ = O.query_entropy_multimg(layers_q, w_q, allp_q, pools_q, ps_q, 16, st_q, 9)
    for a, b in zip(rQ, oQ):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    # ---- the whole single-volume 'fi' branch of PW_NNAL.CNN_query (:89-163), UNMODIFIED: posteriors -> B most uncertain
    # -> get_patches + normalise -> gen_A_matrices (sess.run(model.grad_posts[y]) answered with the restatement's explicit
    # gradient lists) -> refine_feature_matrix -> NNAL_tools.SDP_query_distribution (solvers.sdp answered by the oracle's
    # solver on the A-matrices recovered from the constraint matrix it is handed) -> sample_query_dstr (np.random seeded).
    tau_q = 4

    class FiModel(QModel):
        grad_posts = {'0': [(0, t) for t in range(2 * tau_q)], '1': [(1, t) for t in range(2 * tau_q)]}

    class FiSess(QSess):
        def run(self, var, feed_dict=None):
            if isinstance(var, list):
                return O.explicit_class_gradients(layers_q, w_q, np.asarray(feed_dict['x']).astype(np.float32), var[0][0])
            return QSess.run(self, var, feed_dict)

    class OracleSolvers(object):
        options = {}
        last = {}

        @staticmethod
        def sdp(c, Gs=None, hs=None, A=None, b=None):
            G0 = np.asarray(Gs[0])
            nvar = G0.shape[1]
            d1 = int(round(np.sqrt(G0.shape[0])))
            nq = nvar - (d1 - 1)
            A_rec = [(-G0[:, i]).reshape(d1, d1).T[:d1 - 1, :d1 - 1] for i in range(nq)]
            Aeq = np.asarray(A)
            if Aeq.shape[0] > 1:                       # lambda_ > 0: recover X_pool and lambda from the equalities and c
                X = Aeq[:-1, :nq]
                cn = np.sum(X ** 2, axis=0)
                lam = float(np.median(-np.asarray(c)[:nq, 0][cn > 0] / cn[cn > 0]))
                q, t, phi, gap, it = O.sdp_solve_reg(A_rec, lam, X, 1e-4)
                OracleSolvers.last = {'A': np.array(A_rec), 'q': q, 'phi': phi, 'X': X, 'lambda': lam}
            else:
                q, t, phi, gap, it = O.sdp_solve(A_rec, 1e-4)
                OracleSolvers.last = {'A': np.array(A_rec), 'q': q, 'phi': phi}
            return {'status': 'optimal', 'x': np.concatenate([q, t])}

    ref_tools.solvers = OracleSolvers
    np.random.seed(77)
    u77 = np.random.sample(9)
    np.random.seed(77)
    import contextlib
    import io
    with contextlib.redirect_stdout(io.StringIO()):        # the branch prints the condition number / solver status
        rq_fi = ref_pw.CNN_query(QExpr(), FiModel(), FiSess(), allp_q[0][:m_q], pool0, None, 'fi')
    oq_fi, det = O.query_fi_sdp_single(layers_q, w_q, allp_q[0][:m_q], pool0, ps_q, 16, stats0, 9, 30, u77, diag_load=1e-5)
    A_o = np.array(det['A'])                                # explicit vs closed-form shrink: round-off only
    assert np.allclose(OracleSolvers.last['A'], A_o, rtol=1e-9, atol=1e-12 * np.abs(A_o).max())
    assert np.array_equal(np.asarray(rq_fi), oq_fi), (rq_fi, oq_fi)
    gold['q_fi_sdp_single'] = np.asarray(rq_fi)
    gold['q_fi_u'] = u77
    # the same branch with lambda_ > 0: feature_layer of the candidates -> refine_feature_matrix -> zero-mean rows -> the
    # regularised programme (:139-155)
    class LExpr(QExpr):
        pars = dict(QExpr.pars, lambda_=0.2)
    np.random.seed(77)
    with contextlib.redirect_stdout(io.StringIO()):
        rq_fil = ref_pw.CNN_query(LExpr(), FiModel(), FiSess(), allp_q[0][:m_q], pool0, None, 'fi')
    oq_fil, detl = O.query_fi_sdp_single(layers_q, w_q, allp_q[0][:m_q], pool0, ps_q, 16, stats0, 9, 30, u77, diag_load=1e-5,
                                         lambda_=0.2)
    assert abs(OracleSolvers.last['lambda'] - 0.2) < 1e-12
    assert np.array_equal(OracleSolvers.last['X'], detl['ref_F'])             # same refined, centred feature rows
    assert np.array_equal(np.asarray(rq_fil), oq_fil), (rq_fil, oq_fil)
    gold['q_fi_sdp_single_lambda'] = np.asarray(rq_fil)
    # the multi-volume twin (:547-627, 'CVXOPT' branch) -- its live pdb.set_trace() (:612) is made a no-op
    class MExpr(QExpr):
        pars = dict(QExpr.pars, k=11, B=40, SDP_solver='CVXOPT')
    ref_pw.pdb.set_trace = lambda *a, **k: None
    np.random.seed(78)
    u78 = np.random.sample(11)
    np.random.seed(78)
    with contextlib.redirect_stdout(io.StringIO()):
        rQ_fi = ref_pw.query_multimg(MExpr(), FiModel(), FiSess(), allp_q, pools_q, None, 'fi')
    oQ_fi, _ = O.query_fi_sdp_multimg(layers_q, w_q, allp_q, pools_q, ps_q, 16, st_q, 11, 40, u78)
    assert len(rQ_fi) == S_q
    for a, b in zip(rQ_fi, oQ_fi):
        assert np.array_equal(np.asarray(a), np.asarray(b)), (rQ_fi, oQ_fi)
    for s_ in range(S_q):
        gold['q_fi_sdp_multi%d' % s_] = np.asarray(rQ_fi[s_], dtype=np.int64)
    gold['q_fi_u_multi'] = u78
    # the same branch with d3 = 3 (patch 5x5x3, m = 2 -> 6 channels): the posterior pass normalises channels 0..m-1 only
    # (PW_NN.batch_eval, PW_NN.py:503-506) while the gradient patches come from get_patches_multimg, which normalises whole
    # modality blocks ch/d3 (patch_utils.py:1203-1207) -- the two differ as soon as d3 > 1
    ps_3 = (5, 5, 3)
    w_3 = O.he_init_weights(layers_q, (5, 5, m_q * 3), 8, bias_scale=0.1)
    # (channels m..m*d3-1 reach the posterior pass unnormalised, ~100: shrink conv1 so that the posteriors do not saturate
    # into exact ties, which np.argsort's unstable sort and the oracle's stable one would break differently)
    w_3['conv1'] = (w_3['conv1'][0] * np.float32(0.01), w_3['conv1'][1])
    allp_3 = [[np.pad(im, ((0, 0), (0, 0), (1, 1)), 'constant') for im in sub[:m_q]] + [sub[m_q]] for sub in allp_q]

    class Q3Sess(object):
        def run(self, var, feed_dict=None):
            x = np.asarray(feed_dict['x']).astype(np.float32)
            if isinstance(var, list):
                return O.explicit_class_gradients(layers_q, w_3, x, var[0][0])
            return O.forward(layers_q, w_3, x, feature_layer=fl_q)[var.name]

    class M3Expr(QExpr):
        pars = dict(QExpr.pars, k=11, B=40, SDP_solver='CVXOPT', patch_shape=ps_3)
    np.random.seed(79)
    u79 = np.random.sample(11)
    np.random.seed(79)
    with contextlib.redirect_stdout(io.StringIO()):
        rQ_3 = ref_pw.query_multimg(M3Expr(), FiModel(), Q3Sess(), allp_3, pools_q, None, 'fi')
    oQ_3, _ = O.query_fi_sdp_multimg(layers_q, w_3, allp_3, pools_q, ps_3, 16, st_q, 11, 40, u79)
    for a, b in zip(rQ_3, oQ_3):
        assert np.array_equal(np.asarray(a), np.asarray(b)), (rQ_3, oQ_3)
    for s_ in range(S_q):
        gold['q_fi_sdp_multi_d3_%d' % s_] = np.asarray(rQ_3[s_], dtype=np.int64)
    gold['q_fi_u_d3'] = u79
    print("PW_NNAL.query_multimg 'fi' with d3 = 3 (block-wise normalisation of the gradient patches): oracle == reference")
    # representativeness queries of query_multimg: 'rep-entropy' (:284-351) and 'core-set' (:353-451)
    class RExpr(QExpr):
        pars = dict(QExpr.pars, k=11, B=30)
        labeled_stats = st_q
        labeled_paths = train_paths = ['same']
    # (upstream, these two branches call batch_eval on every subject and raise IndexError on an empty per-subject pool,
    # PW_NN.py:447-449: subject 1 gets a pool here)
    pools_r = [pools_q[0], list(rs.choice(int(np.prod(shape_q)), 20, replace=False)), pools_q[2]]
    rQ_rep = ref_pw.query_multimg(RExpr(), QModel(), QSess(), allp_q, pools_r, None, 'rep-entropy')
    oQ_rep, _ = O.query_rep_entropy_multimg(layers_q, w_q, allp_q, pools_r, ps_q, 16, st_q, 11, 30)
    for a, b in zip(rQ_rep, oQ_rep):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    labeled_q = [list(rs.choice(int(np.prod(shape_q)), 9, replace=False)) for _ in range(S_q)]
    rQ_cs = ref_pw.query_multimg(RExpr(), QModel(), QSess(), allp_q, pools_r, labeled_q, 'core-set')
    oQ_cs, _ = O.query_core_set_multimg(layers_q, w_q, allp_q, pools_r, labeled_q, ps_q, 16, st_q, st_q, 11)
    for a, b in zip(rQ_cs, oQ_cs):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    for s_ in range(S_q):
        gold['q_rep%d' % s_] = np.asarray(rQ_rep[s_], dtype=np.int64)
        gold['q_cs%d' % s_] = np.asarray(rQ_cs[s_], dtype=np.int64)
        gold['q_labeled%d' % s_] = np.array(labeled_q[s_], dtype=np.int64)
        gold['q_pool_r%d' % s_] = np.array(pools_r[s_], dtype=np.int64)
    print("PW_NNAL.query_multimg 'fi' / 'rep-entropy' / 'core-set', unmodified over fake session / solver: oracle == reference")
    # MC-dropout queries of query_multimg: 'MC-entropy' (:232-244) and 'BALD' (:247-282), unmodified.  The fake session
    # plays tf.nn.dropout with the oracle's counter-based masks: it counts the samples it is fed (subjects and batches
    # arrive in pool order) to know their global pool positions and the pass they belong to.
    from oracle import mc_oracle as Mc
    n_tot = sum(len(p_) for p_ in pools_q)
    drop_layers, keep_q, seed_q, first_q = [2, 3, 4], 0.6, 77, 3

    class McModel(QModel):
        dropout_rate = keep_q

    class McSess(object):
        def __init__(self):
            self.seen = 0

        def run(self, var, feed_dict=None):
            xb_ = np.asarray(feed_dict['x']).astype(np.float32)
            kp = feed_dict['keep_prob']
            assert var.name == 'posteriors' and kp == keep_q
            pass_id, off = divmod(self.seen, n_tot)
            self.seen += xb_.shape[0]
            pos = off + np.arange(xb_.shape[0])
            return Mc.forward_dropout(layers_q, w_q, xb_, pos, kp, drop_layers, seed_q, first_q + pass_id)[1]

    class McExpr(QExpr):
        pars = dict(QExpr.pars, k=11, B=40, MC_iters=4)
    for meth, key in (('MC-entropy', 'q_mc'), ('BALD', 'q_bald')):
        rQ_mc = ref_pw.query_multimg(McExpr(), McModel(), McSess(), allp_q, pools_q, None, meth)
        oQ_mc = Mc.query_mc_multimg(layers_q, w_q, allp_q, pools_q, ps_q, st_q, 11, 4, keep_q, drop_layers, seed_q, meth,
                                    first_pass=first_q)[0]
        for s_ in range(S_q):
            assert np.array_equal(np.asarray(rQ_mc[s_]), np.asarray(oQ_mc[s_])), (meth, rQ_mc, oQ_mc)
            gold['%s%d' % (key, s_)] = np.asarray(rQ_mc[s_], dtype=np.int64)
    print("PW_NNAL.query_multimg 'MC-entropy' / 'BALD', unmodified over a fake session with the oracle's dropout masks: "
          "oracle == reference")
    # 'random' (:32-35, :198-205): the drop-in's host code against the reference's, same generator state
    import nnal_b200
    np.random.seed(91)
    rq_rand = ref_pw.CNN_query(QExpr(), None, None, allp_q[0][:m_q], pool0, None, 'random')
    rQ_rand = ref_pw.query_multimg(QExpr(), None, None, allp_q, pools_q, None, 'random')
    np.random.seed(91)
    pq_rand = nnal_b200.PW_NNAL.CNN_query(QExpr(), None, None, allp_q[0][:m_q], pool0, None, 'random')
    pQ_rand = nnal_b200.PW_NNAL.query_multimg(QExpr(), None, None, allp_q, pools_q, None, 'random')
    assert np.array_equal(rq_rand, pq_rand) and all(np.array_equal(a, b) for a, b in zip(rQ_rand, pQ_rand))
    print("'random' queries: drop-in host code == reference (same np.random state)")
    # single-volume CNN_query 'MC-entropy' (:67-87) AS WRITTEN hands x_feed_dict to batch_eval in the `mask` slot: every
    # pass runs with keep_prob = 1 and the query equals 'entropy'.  (The drop-in applies dropout, as query_multimg does.)
    class NoDropSess(QSess):
        def run(self, var, feed_dict=None):
            assert feed_dict['keep_prob'] == 1.
            return QSess.run(self, var, feed_dict)

    class Mc1Expr(QExpr):
        pars = dict(QExpr.pars, MC_iters=3)
    rq_mc1 = ref_pw.CNN_query(Mc1Expr(), McModel(), NoDropSess(), allp_q[0][:m_q], pool0, None, 'MC-entropy')
    assert np.array_equal(np.asarray(rq_mc1), np.asarray(rq))
    print("PW_NNAL.CNN_query 'MC-entropy' (single volume) as written == 'entropy': x_feed_dict lands in batch_eval's mask slot")
    # committee queries of query_multimg, no-label branch: 'ensemble' (:453-490) and 'QBC-JS' (:492-545), unmodified.
    # expr.model_holder.perform_assign_ops(path, sess) switches the weight set the fake session evaluates.
    wsets = [O.he_init_weights(layers_q, (5, 5, m_q), 20 + i, bias_scale=0.1) for i in range(3)]

    class Holder(QModel):
        current = [0]

        def perform_assign_ops(self, path, sess):
            Holder.current[0] = path

    class CSess(object):
        def run(self, var, feed_dict=None):
            assert feed_dict['keep_prob'] == 1.
            r = O.forward(layers_q, wsets[Holder.current[0]], np.asarray(feed_dict['x']).astype(np.float32), feature_layer=fl_q)
            return r[var.name]

    class CExpr(QExpr):
        pars = dict(QExpr.pars, k=11, B=40)
        model_holder = Holder()
        pretrained_paths = [0, 1, 2]
    for meth, key in (('ensemble', 'q_ens'), ('QBC-JS', 'q_qbc')):
        rQ_c = ref_pw.query_multimg(CExpr(), None, CSess(), allp_q, pools_q, [[], [], []], meth)
        oQ_c = Mc.query_committee_multimg(layers_q, wsets, allp_q, pools_q, ps_q, 16, st_q, 11, meth)[0]
        for s_ in range(S_q):
            assert np.array_equal(np.asarray(rQ_c[s_]), np.asarray(oQ_c[s_])), (meth, rQ_c, oQ_c)
            gold['%s%d' % (key, s_)] = np.asarray(rQ_c[s_], dtype=np.int64)
    print("PW_NNAL.query_multimg 'ensemble' / 'QBC-JS' (no-label branch), unmodified over a fake session: oracle == reference")
    ref_tools.solvers = FakeSolvers
    print("PW_NNAL.CNN_query 'fi' (gen_A_matrices + SDP_query_distribution + sample_query_dstr), unmodified over fake "
          "session / solver: oracle.query_fi_sdp_single == reference")

    gold['q_imgs'] = np.stack([np.stack(a[:m_q]) for a in allp_q])
    gold['q_stats'] = st_q
    for s_ in range(S_q):
        gold['q_pool%d' % s_] = np.array(pools_q[s_], dtype=np.int64)
        gold['q_multi%d' % s_] = np.asarray(rQ[s_], dtype=np.int64)
        gold['q_filt%d' % s_] = np.asarray(rsel[s_], dtype=np.int64)
    gold['q_single'] = np.asarray(rq)
    gold['q_posts0'] = rp
    print('PW_NN.batch_eval / PW_NNAL.CNN_query / bin_uncertainty_filter_multimg / query_multimg (entropy), unmodified '
          'over a fake session: oracle == reference')

    # ---- NNAL_tools.FC_gradnorms_batch (:725-775), UNMODIFIED over a fake session: squared gradient norms of P(class 0)
    # w.r.t. every FC layer, back-propagated with ReLU masks (SURVEY row a11: "last two layers' scores")
    fwd_fc = O.forward(layers_q, w_q, rs.randn(13, 5, 5, m_q).astype(np.float32), keep_acts=True)
    fc_names = [n_ for n_, sp_ in layers_q if sp_[1] == 'fc']
    idx_of = {n_: i_ for i_, (n_, _) in enumerate(layers_q)}

    class EvalW(object):
        def __init__(self, W):
            self.W = W

        def eval(self):
            return self.W.astype(np.float64)

    class GModel(object):
        x, keep_prob, posteriors = 'x', 'keep_prob', 'posteriors'
        FC_inputs = [(n_, ('in', n_)) for n_ in fc_names]
        var_dict = {n_: [EvalW(w_q[n_][0]), None] for n_ in fc_names}

    class GSess(object):
        def run(self, var, feed_dict=None):
            if var == 'posteriors':
                return fwd_fc['posteriors']
            return fwd_fc['acts'][idx_of[var[1]]]['in']
    rn = ref_tools.FC_gradnorms_batch(GModel(), np.zeros((13, 1)), GSess())
    on = O.FC_gradnorms_batch(fwd_fc['posteriors'], [fwd_fc['acts'][idx_of[n_]]['in'] for n_ in fc_names],
                              [w_q[n_][0].astype(np.float64) for n_ in fc_names])
    assert rn.shape == on.shape == (3, 13) and np.array_equal(rn, on)
    print('FC_gradnorms_batch: oracle == reference (fake session)')

    # ---- whole-image dispatch NNAL.CNN_query (:188-525) 'entropy' and 'fi', UNMODIFIED: only the image-file loader
    # NN.load_winds (cv2, commented out upstream) is replaced by an in-memory pool; NNAL_tools.idxBatch_posteriors and
    # NN.gen_batch_inds (random batches) are the reference's own.
    import NNAL as ref_nnal
    layers_w = [('conv1', [6, 'conv', [3, 3]]), ('conv2', [5, 'conv', [5, 5]]), ('max1', [[2, 2], 'pool']),
                ('conv3', [8, 'conv', [3, 3]]), ('max2', [[2, 2], 'pool']),
                ('fc1', [40, 'fc']), ('fc2', [24, 'fc']), ('fc3', [3, 'fc'])]
    w_w = O.he_init_weights(layers_w, (9, 7, 2), 6, bias_scale=0.1)
    pool_w = rs.rand(90, 9, 7, 2).astype(np.float32)
    tau_w = 6

    class WOut(object):
        def get_shape(self):
            return [FakeDim(3), FakeDim(None)]

    class WModel(object):
        x = 'x'
        posteriors = FakeTensor('posteriors', (3, None))
        output = WOut()
        grad_posts = {str(y): [(y, t) for t in range(2 * tau_w)] for y in range(3)}

        def extract_features(self, inds, expr, session):
            return O.forward(layers_w, w_w, pool_w[np.asarray(inds)], feature_layer=len(layers_w) - 2)['feature_layer']

    class WSess(object):
        def run(self, var, feed_dict=None):
            xw = np.asarray(feed_dict['x']).astype(np.float32)
            if isinstance(var, dict):
                return {key: O.explicit_class_gradients(layers_w, w_w, xw, int(key)) for key in var}
            return O.forward(layers_w, w_w, xw)['posteriors']

    class WExpr(object):
        pars = dict(k=7, B=20, lambda_=0, batch_size=32, target_shape=None, mean=None)
        imgs_path_file = None
    ref_nnal.NN.load_winds = lambda inds, path_file, target_shape, mean: (pool_w[np.asarray(inds)], None)
    ref_tools.NN.load_winds = ref_nnal.NN.load_winds
    np.random.seed(5)
    rq_w = ref_nnal.CNN_query(WModel(), WExpr(), np.arange(90), 'entropy', WSess())
    oq_w = O.query_entropy_whole(layers_w, w_w, pool_w, 7)[0]
    assert np.array_equal(np.asarray(rq_w), np.asarray(oq_w))
    ref_tools.solvers = OracleSolvers
    np.random.seed(6)
    with contextlib.redirect_stdout(io.StringIO()):
        # draws of the sampler: the reference consumes np.random for its batches first, so replay the same sequence
        rq_wfi = ref_nnal.CNN_query(WModel(), WExpr(), np.arange(90), 'fi', WSess())
    np.random.seed(6)
    np.random.permutation(90)                      # NN.gen_batch_inds inside idxBatch_posteriors (n >= batch_size)
    u_w = np.random.sample(7)
    oq_wfi, _ = O.query_fi_sdp_whole(layers_w, w_w, pool_w, 7, 20, u_w)
    assert np.array_equal(np.asarray(rq_wfi), oq_wfi), (rq_wfi, oq_wfi)
    ref_tools.solvers = FakeSolvers
    np.random.seed(7)
    with contextlib.redirect_stdout(io.StringIO()):
        rq_wrep = ref_nnal.CNN_query(WModel(), WExpr(), np.arange(90), 'rep-entropy', WSess())
    oq_wrep, _ = O.query_rep_entropy_whole(layers_w, w_w, pool_w, 7, 20)
    assert np.array_equal(np.asarray(rq_wrep), np.asarray(oq_wrep)), (rq_wrep, oq_wrep)
    gold['w_rep'] = np.asarray(rq_wrep)
    gold['w_pool'], gold['w_entropy'], gold['w_fi_sdp'], gold['w_fi_u'] = pool_w, np.asarray(rq_w), np.asarray(rq_wfi), u_w
    print("NNAL.CNN_query 'entropy' / 'rep-entropy' / 'fi' (multiclass A-matrices + SDP + sampling), unmodified over fake session / solver / "
          "in-memory pool: oracle == reference")

    # ---- NN.LLFC_grads (:905-955) and NN.LLFC_hess (:874-903), UNMODIFIED over a fake session: last-layer score
    # factors [(e_y - pi) (x) u ; (e_y - pi)] and the Hessian kron(A(pi), [u;1][u;1]^T) (SURVEY row a11)
    import NN as ref_nn
    r3 = O.forward(layers_w, w_w, pool_w[:9], feature_layer=len(layers_w) - 2)

    class LModel(object):
        posteriors, feature_layer, prediction = 'posteriors', 'feature_layer', 'prediction'

    class LSess(object):
        def __init__(self, cols):
            self.cols = cols

        def run(self, var, feed_dict=None):
            if var == 'prediction':
                return np.argmax(r3['posteriors'][:, self.cols], axis=0)
            return r3[var][:, self.cols]
    allc = np.arange(9)
    rg, rlab = ref_nn.LLFC_grads(LModel(), LSess(allc), None)
    og = O.LLFC_grads(r3['posteriors'], r3['feature_layer'])
    og = og[0] if isinstance(og, tuple) else og
    assert np.array_equal(rg, og) and np.array_equal(rlab, np.argmax(r3['posteriors'], axis=0))
    lab = rs.randint(0, 3, 9)
    assert np.array_equal(ref_nn.LLFC_grads(LModel(), LSess(allc), None, lab), O.LLFC_grads(r3['posteriors'], r3['feature_layer'], lab))
    rH = ref_nn.LLFC_hess(LModel(), LSess(np.array([4])), None)
    oH = O.LLFC_hess(r3['posteriors'][:, 4:5], r3['feature_layer'][:, 4:5])
    assert rH.shape == oH.shape and np.allclose(rH, oH, rtol=1e-13, atol=0)
    print('LLFC_grads / LLFC_hess: oracle == reference (fake session)')

    # ---- PW_NNAL.stoch_approx_IF (:851-881), UNMODIFIED over a fake session that answers posteriors / feature_layer /
    # prediction for whatever patches it is fed: LiSSA recursion V <- grads + V - H V / scale through the last FC layer
    r_all = O.forward(layers_w, w_w, pool_w, feature_layer=len(layers_w) - 2)

    class IfModel(object):
        x, keep_prob = 'x', 'keep_prob'
        posteriors, feature_layer, prediction = 'posteriors', 'feature_layer', 'prediction'

    class IfSess(object):
        def run(self, var, feed_dict=None):
            r = O.forward(layers_w, w_w, np.asarray(feed_dict['x']).astype(np.float32), feature_layer=len(layers_w) - 2)
            return np.argmax(r['posteriors'], axis=0) if var == 'prediction' else r[var]
    tr_x, pl_x = pool_w[:12], pool_w[40:47]
    np.random.seed(31)
    draws_if = [np.random.randint(12) for _ in range(25)]
    np.random.seed(31)
    rV, rlab_if = ref_pw.stoch_approx_IF(IfModel(), IfSess(), tr_x, pl_x, 25, 20)
    oV, olab_if = O.stoch_approx_IF(r_all['posteriors'][:, 40:47], r_all['feature_layer'][:, 40:47], r_all['posteriors'][:, :12],
                                    r_all['feature_layer'][:, :12], draws_if, 20.)
    assert np.array_equal(rlab_if, olab_if) and rV.shape == oV.shape
    assert np.allclose(rV, oV, rtol=1e-10, atol=1e-12 * np.abs(oV).max())
    gold['if_V'], gold['if_labels'], gold['if_draws'] = rV, np.asarray(rlab_if), np.array(draws_if)
    print('PW_NNAL.stoch_approx_IF: oracle == reference (fake session, seeded np.random)')

    np.savez_compressed(os.path.join(GOLD, 'reference_numpy_helpers.npz'), **gold)
    print('wrote', os.path.join(GOLD, 'reference_numpy_helpers.npz'))


if __name__ == '__main__':
    main()
