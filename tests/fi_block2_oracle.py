"""Float64 reference of the multi-class block-form greedy FI selection over the last TWO FC layers that csrc/fi_block.cu runs
with n_layers = 2 (``NNAL.CNN_query(..., 'fi')`` with ``fi_mode='block-greedy'``, ``fi_layers=2``): the block kernel, and the
incremental greedy and its replay on any block kernel.  Test infrastructure: the product never imports it."""
import numpy as np

from tests.fi_block_oracle import multinomial_factor


def _factors(post):
    post = np.asarray(post, dtype=np.float64)
    c, n = post.shape
    return np.stack([multinomial_factor(post[:, i]) for i in range(n)]) if n else np.zeros((0, c, c - 1))


def two_layer_dim(c, d, d_prev):
    """Parameter count of the last FC layer (c(d+1)) and the one before it (d(d_prev+1))."""
    return c * (d + 1) + d * (d_prev + 1)


def two_layer_block_kernel(post, U, A_prev, W_last):
    """Block kernel of the FI over the last two FC layers: sample i owns r = c-1 rows and
        K_ij = L_i^T (s_ij I + s'_ij W3 diag(m_i o m_j) W3^T) L_j,   s = u.u + 1,  s' = a.a + 1,  m = 1[u > 0],
    L_i = multinomial_factor(post[:, i]).  ``post`` [c,n], ``U`` [d,n] feature layer, ``A_prev`` [d_p,n] input of the
    feature layer's FC, ``W_last`` [c,d] last FC weights.  Computed as the Gram of the factors: the second term is
    H_i^T H_j s'_ij with H_i = M_i W3^T L_i.  (n r) x (n r); for c = 2 it equals ``last_layers_kernel(p1, U, A_prev, W_last)``."""
    Ls = _factors(post)
    n, c, r = Ls.shape
    U = np.asarray(U, dtype=np.float64)
    A = np.asarray(A_prev, dtype=np.float64)
    W = np.asarray(W_last, dtype=np.float64)
    S = U.T @ U + 1.
    Sp = A.T @ A + 1.
    K = np.einsum('ixy,jxz->iyjz', Ls, Ls) * S[:, None, :, None]
    H = np.einsum('xk,ixy->iky', W, Ls) * (U.T > 0)[:, :, None]
    K += np.einsum('iky,jkz->iyjz', H, H) * Sp[:, None, :, None]
    return K.reshape(n * r, n * r)


def _losses(K, r, S, delta):
    """Greedy criterion of every candidate at |S| = t on the block kernel ``K``: loss_j = tr(Sigma_j^-1 (I + E_j)), tr C."""
    n = K.shape[0] // r
    Kb = K.reshape(n, r, n, r)
    Kd = np.einsum('iyiz->iyz', Kb)
    t = len(S)
    alpha = (t + 1) * delta
    I = np.eye(r)
    if t == 0:
        Sig = alpha * I + Kd
        E = np.zeros_like(Kd)
        trC = 0.
    else:
        rows = np.concatenate([np.arange(a * r, (a + 1) * r) for a in S])
        m = len(rows)
        C = np.linalg.inv(alpha * np.eye(m) + K[np.ix_(rows, rows)])
        kall = K[rows, :]                                    # [m, n r]: k_j = kall[:, j-block]
        Y = (C @ kall).reshape(m, n, r)
        kall = kall.reshape(m, n, r)
        G = np.einsum('pjy,pjz->jyz', kall, Y, optimize=True)
        E = np.einsum('pjy,pjz->jyz', Y, Y, optimize=True)
        Sig = alpha * I + Kd - G
        trC = np.trace(C)
    loss = np.trace(np.linalg.solve(Sig, I + E), axis1=1, axis2=2)
    return loss, trC


def greedy_block_kernel(K, r, D, delta, k):
    """Incremental greedy on a block kernel (sample i owns rows i r .. (i+1) r - 1), the step csrc/fi_block.cu runs: at
    |S| = t, alpha = (t+1) delta, C = (alpha I + K_SS)^-1, Y_j = C k_j, Sigma_j = alpha I + K_jj - k_j^T Y_j,
    loss_j = tr(Sigma_j^-1 (I + Y_j^T Y_j)), first minimum.  Returns (indices in selection order, objective
    f = (D - s r)/delta + red per step, reduced objective red = s (tr C + loss) per step)."""
    n = K.shape[0] // r
    avail = np.ones(n, dtype=bool)
    S, objs, red = [], [], []
    for t in range(min(k, n)):
        loss, trC = _losses(K, r, S, delta)
        loss[~avail] = np.inf
        j = int(np.argmin(loss))
        S.append(j)
        avail[j] = False
        s = t + 1
        red.append(s * (trC + loss[j]))
        objs.append((D - s * r) / delta + red[-1])
    return np.array(S, dtype=np.int64), np.array(objs), np.array(red)


def greedy_block_kernel_replay(K, r, delta, S):
    """Replays a selection ``S`` through the criterion of ``greedy_block_kernel``: per step (loss of S[t], best available
    loss, reduced objective after taking S[t])."""
    n = K.shape[0] // r
    avail = np.ones(n, dtype=bool)
    out = []
    for t in range(len(S)):
        loss, trC = _losses(K, r, list(S[:t]), delta)
        loss[~avail] = np.inf
        j = int(S[t])
        assert avail[j], 'selection repeats a candidate'
        out.append((loss[j], loss.min(), (t + 1) * (trC + loss[j])))
        avail[j] = False
    return np.array(out)


def greedy_fi_block2(post, U, A_prev, W_last, delta, k):
    """``greedy_block_kernel`` on ``two_layer_block_kernel``; shapes as there."""
    post = np.asarray(post)
    c = post.shape[0]
    K = two_layer_block_kernel(post, U, A_prev, W_last)
    return greedy_block_kernel(K, c - 1, two_layer_dim(c, np.shape(U)[0], np.shape(A_prev)[0]), delta, k)
