"""Float64 reference of the multi-class MC-dropout and committee scorers of NNAL.CNN_query ('MC-entropy', 'BALD',
'ensemble', 'QBC-JS') for 2 <= c <= 32 classes.  TEST INFRASTRUCTURE ONLY.

The binary definitions (PW_NNAL.py:67-87, 247-282; oracle/mc_oracle.py) extended to c classes:
  * av_post [c,n]: running mean over passes (committee members) of the posteriors, av = (x + t av) / (t + 1)
  * av_ent [n]: running mean of the per-pass entropies -sum_j p_j log p_j, zero probabilities bumped by 1e-6
  * kind 12 (MC-entropy / ensemble): -H(av_post);  kind 13 (BALD / QBC-JS): -(H(av_post) - av_ent);  k smallest
    (= k largest H, resp. mutual information), ties to the lowest position
At c = 2 the device keeps the binary statistics (mean P(class 1)) and scores with P(class 0) = 1 - P(class 1);
``scores_from_binary`` restates that form.

The posteriors of every pass go through float32 (``post_dtype``) before the float64 recurrences, as the device's head
writes float32 posteriors."""
import numpy as np

import oracle as O
from oracle import mc_oracle as M


def class_entropy_bumped(P):
    """-sum_j p_j log p_j over axis 0 of [c,n], zeros bumped by 1e-6 (the binary BALD's bump, PW_NNAL.py:258-264)."""
    P = np.array(P, dtype=np.float64)
    P[P == 0] += 1e-6
    return -np.sum(P * np.log(P), axis=0)


def class_running_means(pass_posts):
    """``pass_posts``: T arrays [c,n].  Returns (av_post [c,n], av_ent [n]) with the reference's recurrence."""
    av_post, av_ent = 0, 0
    for t, P in enumerate(pass_posts):
        P = np.asarray(P, dtype=np.float64)
        av_post = (P + t * av_post) / (t + 1)
        av_ent = (class_entropy_bumped(P) + t * av_ent) / (t + 1)
    return av_post, av_ent


def scores(av_post, av_ent, kind):
    """Device score of kind 12 (-H(av_post)) or 13 (-(H(av_post) - av_ent)) from the c-class running means."""
    h = class_entropy_bumped(av_post)
    return -h if kind == 12 else -(h - av_ent)


def scores_from_binary(av_p1, av_ent, kind):
    """Kinds 12 / 13 at c = 2 from the binary running means (mean P(class 1), binary entropy), as the device computes them."""
    h = M.binary_entropy_bumped(av_p1)
    return -h if kind == 12 else -(h - av_ent)


def fc_input(layers, weights, x, dropout_layers):
    """Input [d,N] of the first dropped-out FC layer (the deterministic conv trunk's flattened output)."""
    return O.forward(layers, weights, x, keep_acts=True)['acts'][min(dropout_layers)]['in']


def tail_pass(layers, weights, h, positions, keep_prob, dropout_layers, seed, pass_id):
    """One stochastic pass of the FC tail from ``h`` = fc_input(...): the arithmetic of mc_oracle.forward_dropout with the
    trunk evaluated once.  Returns the posteriors [c,N]."""
    for i in range(min(dropout_layers), len(layers)):
        name, _ = layers[i]
        W, b = weights[name]
        z = W.astype(np.float64) @ h + b.astype(np.float64).reshape(-1, 1)
        h = z if i == len(layers) - 1 else np.maximum(z, 0)
        if i in dropout_layers:
            keep = M.dropout_keep_mask(seed, pass_id, i, positions, h.shape[0], keep_prob)
            h = np.where(keep, h / keep_prob, 0.)
    e = np.exp(h - h.max(axis=0, keepdims=True))
    return e / e.sum(axis=0, keepdims=True)


def mc_passes(layers, weights, x, positions, T, keep_prob, dropout_layers, seed, first_pass=0, h=None,
              post_dtype=np.float32):
    """T stochastic passes [c,N] with the engine's pass ids first_pass + t and masks keyed by ``positions``."""
    if h is None:
        h = fc_input(layers, weights, x, dropout_layers)
    return [tail_pass(layers, weights, h, positions, keep_prob, dropout_layers, seed, first_pass + t)
            .astype(post_dtype).astype(np.float64) for t in range(T)]


def _select(av_post, av_ent, method, k):
    kind = 12 if method in ('MC-entropy', 'ensemble') else 13
    s = scores_from_binary(av_post[1], av_ent, kind) if av_post.shape[0] == 2 else scores(av_post, av_ent, kind)
    return O.stable_topk(s, k), s


def binary_ent(pass_posts):
    """The binary per-pass entropy running mean the device keeps at c = 2 (of P(class 1) alone)."""
    return M.mc_running_means([P[1] for P in pass_posts])[1]


def query_mc_whole(layers, weights, x, k, T, keep_prob, dropout_layers, seed, method, first_pass=0, post_dtype=np.float32):
    """NNAL.CNN_query 'MC-entropy' / 'BALD' over the whole pool ``x`` [N,H,W,C].
    Returns (positions, av_post [c,N], av_ent [N], scores)."""
    passes = mc_passes(layers, weights, x, np.arange(len(x)), T, keep_prob, dropout_layers, seed, first_pass,
                       post_dtype=post_dtype)
    av_post, av_ent = class_running_means(passes)
    if av_post.shape[0] == 2:
        av_ent = binary_ent(passes)
    q, s = _select(av_post, av_ent, method, k)
    return q, av_post, av_ent, s


def query_committee_whole(layers, weight_sets, x, k, method, post_dtype=np.float32):
    """NNAL.CNN_query 'ensemble' / 'QBC-JS': every weight set evaluated deterministically.
    Returns (positions, av_post [c,N], av_ent [N], scores)."""
    passes = [O.forward(layers, w, x)['posteriors'].astype(post_dtype).astype(np.float64) for w in weight_sets]
    av_post, av_ent = class_running_means(passes)
    if av_post.shape[0] == 2:
        av_ent = binary_ent(passes)
    q, s = _select(av_post, av_ent, method, k)
    return q, av_post, av_ent, s
