"""Float64 NumPy restatement of the reference query-scoring path (TEST ORACLE).

Every function cites the reference file:line (relative to the upstream
jsourati/nn-active-learning tree) whose behaviour it restates.  Nothing here is
used by the product path; see ``oracle/__init__.py``.
"""
import numpy as np

__all__ = [
    'pw1_layers', 'he_init_weights', 'layer_shapes',
    'get_patches', 'get_patches_multimg', 'global2local_inds',
    'normalize_batch_eval', 'conv2d_same', 'pool_same_pads', 'max_pool_same', 'flatten_tf',
    'forward', 'batch_eval', 'compute_entropy', 'uncertainty_filtering',
    'binary_uncertainty_filter', 'stable_topk', 'bin_uncertainty_filter_multimg',
    'pixelwise_entropy', 'query_entropy_single', 'query_entropy_multimg',
    'query_entropy_whole',
]


# --------------------------------------------------------------------------
# model description (NN.py:1319-1359 create_PW1; NN.py:56-345 CNN builder)
# --------------------------------------------------------------------------
def pw1_layers(nclass=2):
    """Layer list of the patch-wise CNN ``create_PW1`` (NN.py:1328-1336), kept as
    an ordered list of (name, spec) with the reference's spec format
    ``[out,'conv',[kh,kw]]`` / ``[[ph,pw],'pool']`` / ``[out,'fc']``."""
    return [('conv1', [24, 'conv', [5, 5]]),
            ('conv2', [32, 'conv', [5, 5]]),
            ('max1', [[2, 2], 'pool']),
            ('conv3', [48, 'conv', [3, 3]]),
            ('conv4', [96, 'conv', [3, 3]]),
            ('max2', [[2, 2], 'pool']),
            ('fc1', [4096, 'fc']),
            ('fc2', [4096, 'fc']),
            ('fc3', [nclass, 'fc'])]


def layer_shapes(layers, in_shape):
    """Per-layer output shapes.  conv: SAME stride 1 (NN.py:258-290); pool: SAME,
    window=stride (NN.py:1473-1477) -> ceil(n/s); fc: column vector of length out
    (NN.py:303-327).  Returns list of tuples: (H,W,C) before flattening, (D,) after."""
    H, W, C = in_shape
    cur = (H, W, C)
    out = []
    for name, spec in layers:
        if spec[1] == 'conv':
            cur = (cur[0], cur[1], spec[0])
        elif spec[1] == 'pool':
            s = spec[0][0]
            cur = (-(-cur[0] // s), -(-cur[1] // s), cur[2])
        elif spec[1] == 'fc':
            cur = (spec[0],)
        else:
            raise ValueError("Layer's type should be either 'fc', 'conv' or 'pool'.")
        out.append(cur)
    return out


def he_init_weights(layers, in_shape, seed, bias_scale=0.0):
    """Synthetic weights in the TF layouts of NN.py:270-283 (conv
    ``[kh,kw,cin,cout]`` + ``[cout]``) and NN.py:311-320 (fc ``[out,in]`` +
    ``[out,1]``) with the He-normal init of NN.py:1430-1464 (std=sqrt(2/fan_in),
    zero bias; ``bias_scale`` > 0 adds N(0,bias_scale^2) biases so tests exercise
    the bias path).  Values are float32-representable."""
    rs = np.random.RandomState(seed)
    shapes = layer_shapes(layers, in_shape)
    weights = {}
    cur = tuple(in_shape)
    for (name, spec), shp in zip(layers, shapes):
        if spec[1] == 'conv':
            kh, kw = spec[2]
            cin, cout = cur[2], spec[0]
            std = np.sqrt(2.0 / (kh * kw * cin))
            W = (rs.randn(kh, kw, cin, cout) * std).astype(np.float32)
            b = (rs.randn(cout) * bias_scale).astype(np.float32)
            weights[name] = (W, b)
        elif spec[1] == 'fc':
            fin = int(np.prod(cur))
            std = np.sqrt(2.0 / fin)
            W = (rs.randn(spec[0], fin) * std).astype(np.float32)
            b = (rs.randn(spec[0], 1) * bias_scale).astype(np.float32)
            weights[name] = (W, b)
        cur = shp
    return weights


# --------------------------------------------------------------------------
# patch gather (patch_utils.py:1087-1212, :829-866)
# --------------------------------------------------------------------------
def get_patches(imgs, inds, patch_shape, padded=True, mask=None):
    """patch_utils.get_patches (patch_utils.py:1087-1173), vectorised.

    Output float64 ``(b, d1, d2, m*d3)``; channel ``j*d3+dz`` holds modality j,
    depth offset dz; indices are raveled C-order voxel ids of the UNPADDED volume
    (:1144); zero padding when ``padded`` is False (:1118-1132)."""
    d1, d2, d3 = patch_shape
    m = len(imgs)
    rads = [int((patch_shape[i] - 1) / 2.) for i in range(3)]
    if not padded:
        pimgs = [np.pad(img, ((rads[0],) * 2, (rads[1],) * 2, (rads[2],) * 2),
                        'constant') for img in imgs]
        orig_shape = imgs[0].shape
    else:
        pimgs = list(imgs)
        ps = imgs[0].shape
        orig_shape = (ps[0] - 2 * rads[0], ps[1] - 2 * rads[1], ps[2] - 2 * rads[2])
    inds = np.asarray(inds)
    multinds = np.unravel_index(inds, orig_shape)
    b = len(inds)
    patches = np.zeros((b, d1, d2, m * d3))
    # slice [c-r : c+r+1] with c = multind + r  ->  offsets 0..2r from multind (:1148-1165)
    ox = np.arange(2 * rads[0] + 1)
    oy = np.arange(2 * rads[1] + 1)
    oz = np.arange(2 * rads[2] + 1)
    if (len(ox), len(oy), len(oz)) != (d1, d2, d3):
        # even patch sizes make the reference's slice assignment fail as well
        raise ValueError('could not broadcast patch of shape %s into %s'
                         % ((len(ox), len(oy), len(oz)), (d1, d2, d3)))
    X = multinds[0][:, None, None, None] + ox[None, :, None, None]
    Y = multinds[1][:, None, None, None] + oy[None, None, :, None]
    Z = multinds[2][:, None, None, None] + oz[None, None, None, :]
    for j in range(m):
        patches[:, :, :, j * d3:(j + 1) * d3] = pimgs[j][X, Y, Z]
    if mask is not None:
        return patches, mask[multinds]
    return patches


def get_patches_multimg(all_padded_imgs, img_inds, patch_shape, stats):
    """patch_utils.get_patches_multimg (patch_utils.py:1175-1212): per subject,
    gather with the subject's (unpadded) mask as last list element, then
    normalise modality block k with stats[j,2k], stats[j,2k+1] (:1203-1207)."""
    m = len(all_padded_imgs[0]) - 1
    s = len(img_inds)
    d3 = patch_shape[2]
    b_patches = [[] for _ in range(s)]
    b_labels = [[] for _ in range(s)]
    for j in range(s):
        if len(img_inds[j]) > 0:
            patches, labels = get_patches(all_padded_imgs[j][:m], img_inds[j],
                                          patch_shape, True, all_padded_imgs[j][m])
            for k in range(m):
                mu = stats[j, k * 2]
                sigma = stats[j, k * 2 + 1]
                patches[:, :, :, k * d3:(k + 1) * d3] = (
                    patches[:, :, :, k * d3:(k + 1) * d3] - mu) / sigma
            b_patches[j] = patches
            b_labels[j] = labels
    return b_patches, b_labels


def global2local_inds(batch_inds, set_sizes):
    """patch_utils.global2local_inds (patch_utils.py:829-866): order-preserving
    split of global positions into per-set local positions."""
    cumvols = np.append(-1, np.cumsum(set_sizes) - 1)
    set_inds = cumvols.searchsorted(batch_inds) - 1
    return [np.array(batch_inds)[set_inds == i] - cumvols[i] - 1
            for i in range(len(set_sizes))]


def normalize_batch_eval(batch_tensors, stats):
    """The normalisation of PW_NN.batch_eval (PW_NN.py:503-506): channels
    0..m-1 only (correct only for d3==1 -- restated as written), float64."""
    for j in range(len(stats)):
        batch_tensors[:, :, :, j] = (batch_tensors[:, :, :, j] - stats[j][0]) / stats[j][1]
    return batch_tensors


# --------------------------------------------------------------------------
# forward pass with TF-1.x semantics (NN.py:184-188, 258-340, 1473-1477)
# --------------------------------------------------------------------------
def conv2d_same(x, W, b):
    """tf.nn.conv2d(x, W, [1,1,1,1], 'SAME') + b (NN.py:285-289): NHWC
    cross-correlation, filter [kh,kw,cin,cout], symmetric zero pad k//2."""
    kh, kw, cin, cout = W.shape
    ph, pw = kh // 2, kw // 2
    xp = np.pad(x, ((0, 0), (ph, ph), (pw, pw), (0, 0)), 'constant')
    win = np.lib.stride_tricks.sliding_window_view(xp, (kh, kw), axis=(1, 2))
    # win: [N,H,W,C,kh,kw]
    out = np.tensordot(win, W, axes=([4, 5, 3], [0, 1, 2]))
    return out + b.reshape(1, 1, 1, cout)


def pool_same_pads(n, s):
    """TF SAME padding of a window-s, stride-s pool along an axis of length n:
    out = ceil(n/s), pad_total = out*s - n, (pad_before, pad_after) =
    (pad_total // 2, pad_total - pad_total // 2)."""
    tot = -(-n // s) * s - n
    return tot // 2, tot - tot // 2


def max_pool_same(x, s=2, return_argmax=False):
    """tf.nn.max_pool(ksize=s, strides=s, 'SAME') (NN.py:1473-1477): output
    ceil(n/s); the pad_total = out*s - n padded cells are split with the
    smaller half BEFORE the first row/column (``pool_same_pads``; nothing before
    for s = 2) and never win.  ``return_argmax`` indexes the s*s window of the
    PADDED input."""
    N, H, W, C = x.shape
    Ho, Wo = -(-H // s), -(-W // s)
    pt, pl = pool_same_pads(H, s)[0], pool_same_pads(W, s)[0]
    xp = np.full((N, Ho * s, Wo * s, C), -np.inf, dtype=x.dtype)
    xp[:, pt:pt + H, pl:pl + W, :] = x
    xr = xp.reshape(N, Ho, s, Wo, s, C).transpose(0, 1, 3, 5, 2, 4).reshape(N, Ho, Wo, C, s * s)
    out = xr.max(axis=-1)
    if return_argmax:
        return out, xr.argmax(axis=-1)   # first max in (row-major) window order
    return out


def flatten_tf(x):
    """reshape(transpose(x), [C*W*H, -1]) (NN.py:296-301, 337-340): tf.transpose
    with no perm reverses axes [N,H,W,C]->[C,W,H,N]; flat row = c*(W*H)+w*H+h."""
    N = x.shape[0]
    return np.transpose(x).reshape(-1, N)


def forward(layers, weights, x, feature_layer=None, keep_acts=False, dtype=np.float64):
    """Forward graph of NN.CNN (NN.py:56-345) at keep_prob=1 (dropout identity,
    PW_NN.py:514-515).  ``x`` is [N,H,W,C].  Returns dict with ``output`` [c,N]
    (logits, no activation on the last layer NN.py:231-241), ``posteriors`` [c,N]
    (softmax over classes, NN.py:184-188), ``feature_layer`` [d,N] (output of layer
    index ``feature_layer``, NN.py:173-176), and with ``keep_acts`` the per-layer
    inputs/outputs needed by the gradient oracle."""
    h = np.asarray(x, dtype=dtype)
    n_layers = len(layers)
    feat = None
    acts = []
    flat = False
    for i, (name, spec) in enumerate(layers):
        last = (i == n_layers - 1)
        nxt = layers[i + 1][1][1] if not last else None
        rec = {'name': name, 'type': spec[1], 'in': h}
        if spec[1] == 'conv':
            W, b = weights[name]
            z = conv2d_same(h, W.astype(dtype), b.astype(dtype))
            h = np.maximum(z, 0)
            rec['z'] = z
            rec['out_nhwc'] = h
            if nxt == 'fc':
                h = flatten_tf(h)
                flat = True
        elif spec[1] == 'pool':
            if keep_acts:
                h, am = max_pool_same(h, spec[0][0], return_argmax=True)
                rec['argmax'] = am
            else:
                h = max_pool_same(h, spec[0][0])
            rec['out_nhwc'] = h
            if nxt == 'fc':
                h = flatten_tf(h)
                flat = True
        elif spec[1] == 'fc':
            W, b = weights[name]
            if not flat:          # fc directly on the input (not used by PW1)
                h = flatten_tf(h)
                flat = True
                rec['in'] = h
            z = W.astype(dtype) @ h + b.astype(dtype).reshape(-1, 1)
            rec['z'] = z
            h = z if last else np.maximum(z, 0)
        else:
            raise ValueError("Layer's type should be either 'fc', 'conv' or 'pool'.")
        rec['out'] = h
        if keep_acts:
            acts.append(rec)
        if feature_layer is not None and i == feature_layer:
            feat = h
    logits = h
    zmax = logits.max(axis=0, keepdims=True)
    e = np.exp(logits - zmax)
    post = e / e.sum(axis=0, keepdims=True)
    res = {'output': logits, 'posteriors': post, 'feature_layer': feat}
    if keep_acts:
        res['acts'] = acts
    return res


def batch_eval(layers, weights, img_dat, inds, patch_shape, batch_size, stats,
               varnames, feature_layer=None, fwd=None):
    """PW_NN.batch_eval (PW_NN.py:357-539) for ``posteriors`` / ``feature_layer``
    / ``prediction``: contiguous batches of ``batch_size`` (:447-451), gather
    (:498-501), float64 normalisation of channels 0..m-1 (:503-506), feed cast to
    float32 (placeholder dtype, NN.py:1339-1345), forward; ``posteriors`` keeps
    P(class 1) only (:526-529).  ``fwd`` may replace the forward (e.g. a float32
    torch implementation for CPU-baseline timing)."""
    if not isinstance(varnames, list):
        varnames = [varnames]
    if feature_layer is None:
        feature_layer = len(layers) - 2
    inds = np.asarray(inds)
    n = len(inds)
    batch_ends = np.arange(0, n, batch_size)
    if len(batch_ends) == 0 or batch_ends[-1] != n:
        batch_ends = np.append(batch_ends, n)
    vals_list = []
    for var in varnames:
        vals = None
        for i in range(1, len(batch_ends)):
            sl = slice(batch_ends[i - 1], batch_ends[i])
            bt = get_patches(img_dat, inds[sl], patch_shape)
            bt = normalize_batch_eval(bt, stats)
            xin = bt.astype(np.float32)          # TF feed cast
            r = (fwd or (lambda xx: forward(layers, weights, xx, feature_layer)))(xin)
            if var == 'posteriors':
                if vals is None:
                    vals = np.zeros(n)
                vals[sl] = r['posteriors'][1, :]
            elif var == 'feature_layer':
                if vals is None:
                    vals = np.zeros((r['feature_layer'].shape[0], n))
                vals[:, sl] = r['feature_layer']
            elif var == 'prediction':
                if vals is None:
                    vals = np.zeros(n)
                vals[sl] = np.argmax(r['posteriors'], axis=0)
            else:
                raise ValueError('oracle batch_eval: unsupported variable %s' % var)
        if vals is None:
            vals = np.zeros(n)
        vals_list += [vals]
    return vals_list


# --------------------------------------------------------------------------
# scoring (NNAL_tools.py:22-36, 71-85; PW_NNAL.py:64, 671-736)
# --------------------------------------------------------------------------
def compute_entropy(PMFs):
    """NNAL_tools.compute_entropy (NNAL_tools.py:71-85): zeros bumped by 10e-8
    IN PLACE, then -sum p log p over axis 0 of [c,n]."""
    PMFs[PMFs == 0] += 10e-8
    return -np.sum(PMFs * np.log(PMFs), axis=0)


def stable_topk(scores, k):
    """argsort(scores)[:k] with the tie-break this build defines (SURVEY H7):
    lowest position first (stable sort).  The reference uses NumPy's default
    unstable sort, so ties are unordered there."""
    return np.argsort(scores, kind='stable')[:k]


def uncertainty_filtering(posteriors, B):
    """NNAL_tools.uncertainty_filtering (NNAL_tools.py:22-36): zeros bumped by
    1e-8 IN PLACE, entropy over axis 0, B largest."""
    posteriors[posteriors == 0] += 1e-8
    entropies = -np.sum(posteriors * np.log(posteriors), axis=0)
    return stable_topk(-entropies, B)


def binary_uncertainty_filter(posts, B):
    """PW_NNAL.binary_uncertainty_filter (PW_NNAL.py:671-681)."""
    return stable_topk(np.abs(np.array(posts) - 0.5), B)


def pixelwise_entropy(post):
    """-sum_c p log p over axis 0 of a [c,h,w,z] posterior tensor
    (eval_utils.py:153-154,173-175 shape; zero guard as compute_entropy)."""
    p = np.array(post, dtype=np.float64)
    return compute_entropy(p.reshape(p.shape[0], -1)).reshape(p.shape[1:])


def bin_uncertainty_filter_multimg(layers, weights, all_padded_imgs, pool_inds,
                                   patch_shape, ntb, train_stats, B):
    """PW_NNAL.bin_uncertainty_filter_multimg (PW_NNAL.py:684-736)."""
    s = len(pool_inds)
    img_ind_sizes = [len(pool_inds[i]) for i in range(s)]
    m = len(all_padded_imgs[0]) - 1
    H = [[] for _ in range(s)]
    for i in range(s):
        if len(pool_inds[i]) == 0:
            continue
        stats = [[train_stats[i, 2 * j], train_stats[i, 2 * j + 1]] for j in range(m)]
        H[i] = list(batch_eval(layers, weights, all_padded_imgs[i][:-1], pool_inds[i],
                               patch_shape, ntb, stats, 'posteriors')[0])
    tH = np.abs(np.concatenate(H) - 0.5)
    sorted_inds = stable_topk(tH, B)
    sel_inds = global2local_inds(sorted_inds, img_ind_sizes)
    sel_posts = [np.array(H[i])[sel_inds[i]] for i in range(s)]
    return sel_inds, sel_posts


def query_entropy_single(layers, weights, padded_imgs, pool_inds, patch_shape, ntb,
                         stats, k):
    """PW_NNAL.CNN_query 'entropy' branch (PW_NNAL.py:51-65)."""
    posts = batch_eval(layers, weights, padded_imgs, pool_inds, patch_shape, ntb,
                       stats, 'posteriors')[0]
    return stable_topk(np.abs(posts - .5), k), posts


def query_entropy_multimg(layers, weights, all_padded_imgs, pool_inds, patch_shape,
                          ntb, train_stats, k):
    """PW_NNAL.query_multimg 'entropy' branch (PW_NNAL.py:226-230)."""
    return bin_uncertainty_filter_multimg(layers, weights, all_padded_imgs, pool_inds,
                                          patch_shape, ntb, train_stats, k)[0]


def query_entropy_whole(layers, weights, pool_x, k, feature_layer=None):
    """NNAL.CNN_query 'entropy' branch (NNAL.py:298-310) on an in-memory pool
    [n,H,W,C] (the reference loads images with NN.load_winds, which is broken
    upstream -- SURVEY §2 row 6): posteriors [c,n] -> compute_entropy ->
    argsort(-H)[:k]."""
    post = forward(layers, weights, pool_x.astype(np.float32), feature_layer)['posteriors']
    H = compute_entropy(post)
    return stable_topk(-H, k), H, post
