"""Float64 reference of the block-form greedy FI with a class cap (``fi_classes``, csrc/fi_block.cu kept classes): each
candidate keeps its r-hat = min(r, c) most probable classes, and the greedy runs in kept-class coordinates, so nothing is
sized by c beyond one scattered factor per winner (usable at c = 1,000 and 21,841).  Test infrastructure: the product
never imports it."""
import numpy as np

from tests.fi_block_oracle import multinomial_factor


def top_classes(post, r):
    """Kept classes of every column of ``post`` [c,n] (float32): the min(r, c) largest values, ties to the lower class index,
    in ascending class order.  Returns (ids [n,q] int64, float32 posteriors [n,q])."""
    post = np.asarray(post, dtype=np.float32)
    q = min(int(r), post.shape[0])
    order = np.argsort(-post, axis=0, kind='stable')[:q]          # stable: equal values keep ascending class order
    cls = np.sort(order.T, axis=1)
    return cls.astype(np.int64), np.take_along_axis(post.T, cls, axis=1)


def renormalise(p):
    """Kept posteriors [n,q] over their float64 sum taken in ascending class order (zero rows stay zero)."""
    p = np.asarray(p, dtype=np.float64)
    s = np.cumsum(p, axis=1)[:, -1:]
    return np.where(s > 0, p / np.where(s > 0, s, 1.), 0.)


def truncate_posteriors(post, r):
    """The truncated posteriors as a dense [c,n] float64 array: kept classes renormalised, every other class zero."""
    post = np.asarray(post, dtype=np.float32)
    cls, p = top_classes(post, r)
    out = np.zeros(post.shape)
    np.put_along_axis(out.T, cls, renormalise(p), axis=1)
    return out


def _run(cls, p, U, c, delta, k=None, S=None):
    """Greedy (S None) or replay of S in kept-class coordinates: K_ij = s_ij sum over shared classes of L_i^T L_j."""
    cls = np.asarray(cls, dtype=np.int64)
    U = np.asarray(U, dtype=np.float64)
    n, q = cls.shape
    r = q - 1
    Ls = np.stack([multinomial_factor(pi) for pi in renormalise(p)]) if n else np.zeros((0, q, r))
    Kd = np.einsum('ixy,ixz->iyz', Ls, Ls) * ((U * U).sum(axis=0) + 1.)[:, None, None]
    I = np.eye(r)
    avail = np.ones(n, dtype=bool)
    cols, sel, objs, red, rep = [], [], [], [], []
    D = c * (U.shape[0] + 1)
    steps = min(k, n) if S is None else len(S)
    for t in range(steps):
        alpha = (t + 1) * delta
        if t == 0:
            Sig, E, trC = alpha * I + Kd, np.zeros_like(Kd), 0.
        else:
            kj = np.stack(cols, axis=1).reshape(n, t * r, r)                 # [j, (a,y), z] = K_{w_a j}[y,z]
            Kss = kj[sel].transpose(1, 0, 2).reshape(t * r, t * r)
            C = np.linalg.inv(alpha * np.eye(t * r) + Kss)
            Y = np.einsum('pq,jqz->jpz', C, kj)
            Sig = alpha * I + Kd - np.einsum('jpy,jpz->jyz', kj, Y)
            E = np.einsum('jpy,jpz->jyz', Y, Y)
            trC = np.trace(C)
        loss = np.trace(np.linalg.solve(Sig, I + E), axis1=1, axis2=2)
        loss[~avail] = np.inf
        if S is None:
            j = int(np.argmin(loss))
        else:
            j = int(S[t])
            assert avail[j], 'selection repeats a candidate'
            rep.append((loss[j], loss.min(), (t + 1) * (trC + loss[j])))
        sel.append(j)
        avail[j] = False
        red.append((t + 1) * (trC + loss[j]))
        objs.append((D - (t + 1) * r) / delta + red[-1])
        La = np.zeros((c, r))                                                # winner's factor scattered over all classes
        La[cls[j]] = Ls[j]
        sa = U[:, j] @ U + 1.
        cols.append(np.einsum('jxy,jxz->jyz', La[cls], Ls) * sa[:, None, None])
    if S is not None:
        return np.array(rep)
    return np.array(sel, dtype=np.int64), np.array(objs), np.array(red)


def greedy_fi_block_cls(cls, p, U, c, delta, k):
    """Greedy selection over candidates given by kept classes ``cls`` [n,q], their posteriors ``p`` [n,q] and features
    ``U`` [d,n], for a c-class model.  Returns (indices in selection order, objective f = (D - s (q-1))/delta + red,
    reduced objective red per step), D = c(d+1): ``greedy_fi_block`` of the truncated posteriors."""
    return _run(cls, p, U, c, delta, k=k)


def greedy_fi_block_cls_replay(cls, p, U, c, delta, S):
    """Per step of the sequence ``S``: (loss of S[t], best available loss, reduced objective after taking S[t])."""
    return _run(cls, p, U, c, delta, S=S)
