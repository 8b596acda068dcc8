"""Float64 reference of the multi-class block-form greedy FI selection that csrc/fi_block.cu runs
(``NNAL.CNN_query(..., 'fi')`` with ``fi_mode='block-greedy'``): the closed-form factor of diag(pi) - pi pi^T, the block
kernel, the incremental greedy and its replay.  Test infrastructure: the product never imports it."""
import numpy as np


def multinomial_factor(pi):
    """Closed-form c x (c-1) factor L with L L^T = diag(pi) - pi pi^T (NN.LLFC_hess, NN.py:891-901) of the posteriors
    ``pi`` renormalised in float64.  With a_j = sum_{k>=j} pi_k and b_j = sum_{k>j} pi_k (tail sums):
    L[j,j] = sqrt(pi_j b_j / a_j), L[i,j] = -pi_i sqrt(pi_j / (a_j b_j)) for i > j; column j is zero when pi_j = 0 or
    b_j = 0 (no pivots, exact for one-hot posteriors)."""
    p = np.asarray(pi, dtype=np.float64).ravel()
    p = p / p.sum()
    c = len(p)
    tail = np.zeros(c + 1)
    for j in range(c - 1, -1, -1):
        tail[j] = tail[j + 1] + p[j]
    L = np.zeros((c, c - 1))
    for j in range(c - 1):
        a, b = tail[j], tail[j + 1]
        if p[j] > 0 and b > 0:
            L[j, j] = np.sqrt(p[j] * b / a)
            L[j + 1:, j] = -p[j + 1:] * np.sqrt(p[j] / (a * b))
    return L


def _block_factors(post, U):
    post = np.asarray(post, dtype=np.float64)
    U = np.asarray(U, dtype=np.float64)
    Ls = np.stack([multinomial_factor(post[:, i]) for i in range(post.shape[1])]) if post.shape[1] else \
        np.zeros((0, post.shape[0], post.shape[0] - 1))
    Sfull = U.T @ U + 1.
    return Ls, Sfull


def last_layer_block_kernel(post, U):
    """Block kernel of the last-layer FI for c classes: sample i owns r = c-1 rows, K_ij = (L_i^T L_j)(u_i.u_j + 1) with
    L_i = multinomial_factor(post[:, i]); ``post`` [c,n], ``U`` [d,n].  (n r) x (n r); for c = 2 it equals
    ``last_layers_kernel(p1, U)``."""
    Ls, Sfull = _block_factors(post, U)
    n, c, r = Ls.shape
    K = np.einsum('ixy,jxz->iyjz', Ls, Ls) * Sfull[:, None, :, None]
    return K.reshape(n * r, n * r)


def _block_losses(Ls, Sfull, Kd, S, delta):
    """Greedy criterion of every candidate at |S| = t: loss_j = tr(Sigma_j^-1 (I + E_j)) and tr C (DESIGN.md, FI section)."""
    n, c, r = Ls.shape
    t = len(S)
    alpha = (t + 1) * delta
    I = np.eye(r)
    if t == 0:
        Sig = alpha * I + Kd
        E = np.zeros_like(Kd)
        trC = 0.
    else:
        S = np.asarray(S)
        Lsel = Ls[S]
        m = t * r
        Kss = (np.einsum('axy,bxz->aybz', Lsel, Lsel) * Sfull[np.ix_(S, S)][:, None, :, None]).reshape(m, m)
        C = np.linalg.inv(alpha * np.eye(m) + Kss)
        Z = np.einsum('pay,axy->pxa', C.reshape(m, t, r), Lsel)                  # Z = C Lblk^T  as [rho, x, a]
        sj = Sfull[S, :]                                                         # [t, n]
        W = (Z.reshape(m * c, t) @ sj).reshape(m, c, n)                          # sum_a s_{w_a j} Z[:, a-block]
        Y = np.einsum('pxj,jxy->jpy', W, Ls, optimize=True)                      # Y_j = C k_j
        kj = (np.einsum('axz,jxy->jazy', Lsel, Ls, optimize=True) * sj.T[:, :, None, None]).reshape(n, m, r)
        G = np.einsum('jpy,jpz->jyz', kj, Y, optimize=True)
        E = np.einsum('jpy,jpz->jyz', Y, Y, optimize=True)
        Sig = alpha * I + Kd - G
        trC = np.trace(C)
    loss = np.trace(np.linalg.solve(Sig, I + E), axis1=1, axis2=2)
    return loss, trC


def greedy_fi_block(post, U, delta, k):
    """Incremental greedy on the block kernel (the algorithm csrc/fi_block.cu runs).  At |S| = t, alpha = (t+1) delta,
    C = (alpha I + K_SS)^-1, k_j = [K_ij]_{i in S}, Y_j = C k_j, Sigma_j = alpha I + K_jj - k_j^T Y_j, E_j = Y_j^T Y_j,
    loss_j = tr(Sigma_j^-1 (I + E_j)); the first minimum is taken.  Returns (indices in selection order, objective
    f = (D - s r)/delta + red per step, reduced objective red = tr((delta I + K_SS/s)^-1) = s (tr C + loss) per step),
    D = c(d+1).  ``post`` [c,n], ``U`` [d,n]."""
    Ls, Sfull = _block_factors(post, U)
    n, c, r = Ls.shape
    D = c * (np.asarray(U).shape[0] + 1)
    Kd = np.einsum('ixy,ixz->iyz', Ls, Ls) * np.diag(Sfull)[:, None, None]
    avail = np.ones(n, dtype=bool)
    S, objs, red = [], [], []
    for t in range(min(k, n)):
        loss, trC = _block_losses(Ls, Sfull, Kd, S, delta)
        loss[~avail] = np.inf
        j = int(np.argmin(loss))
        S.append(j)
        avail[j] = False
        s = t + 1
        red.append(s * (trC + loss[j]))
        objs.append((D - s * r) / delta + red[-1])
    return np.array(S, dtype=np.int64), np.array(objs), np.array(red)


def greedy_fi_block_replay(post, U, delta, S):
    """Replays a selection sequence ``S`` through the criterion of ``greedy_fi_block``: per step (loss of S[t], best
    available loss, reduced objective after taking S[t]).  Used to accept selections that differ only at ties."""
    Ls, Sfull = _block_factors(post, U)
    n, c, r = Ls.shape
    Kd = np.einsum('ixy,ixz->iyz', Ls, Ls) * np.diag(Sfull)[:, None, None]
    avail = np.ones(n, dtype=bool)
    out = []
    for t in range(len(S)):
        loss, trC = _block_losses(Ls, Sfull, Kd, list(S[:t]), delta)
        loss[~avail] = np.inf
        j = int(S[t])
        assert avail[j], 'selection repeats a candidate'
        out.append((loss[j], loss.min(), (t + 1) * (trC + loss[j])))
        avail[j] = False
    return np.array(out)
