"""Independent float64 reference of the NN.CNN forward pass with TensorFlow's SAME padding written out.

It shares no code with ``oracle.nnal_oracle.forward``: every conv and every max-pool is padded explicitly with
``F.pad`` (zeros for conv, -inf for pool) by the amounts TF's documented SAME rule gives ("Notes on padding" in the
``tf.nn`` API docs), then run with no implicit padding:

    out         = ceil(n / stride)
    pad_total   = max((out - 1) * stride + window - n, 0)
    pad_before  = pad_total // 2,   pad_after = pad_total - pad_before

For the reference's layers (conv: odd window, stride 1; pool: window == stride, NN.py:1473-1477) this puts
(k-1)/2 zeros on both sides of a conv input, and for a pool with s >= 3 it can put padding BEFORE the first
row/column (H = 7, s = 3: windows {0,1}, {2,3,4}, {5,6}).
"""
import numpy as np
import torch
import torch.nn.functional as F


def same_pads(n, window, stride):
    """(pad_before, pad_after) of TF SAME padding along an axis of length ``n``."""
    out = -(-n // stride)
    total = max((out - 1) * stride + window - n, 0)
    return total // 2, total - total // 2


def pool_windows(n, s):
    """Input indices covered by each output of a window-``s``, stride-``s`` SAME pool along an axis of length ``n``."""
    before, _ = same_pads(n, s, s)
    return [[i for i in range(j * s - before, j * s - before + s) if 0 <= i < n] for j in range(-(-n // s))]


def max_pool(h, s):
    """SAME max-pool of an NCHW float64 tensor, window = stride = ``s``."""
    (t, b), (l, r) = same_pads(h.shape[2], s, s), same_pads(h.shape[3], s, s)
    return F.max_pool2d(F.pad(h, (l, r, t, b), value=-float('inf')), s, s)


def conv(h, W, b):
    """SAME conv, stride 1, of an NCHW tensor with a TF-layout filter ``W`` [kh, kw, cin, cout] and bias ``b``."""
    kh, kw = W.shape[0], W.shape[1]
    (t, bo), (l, r) = same_pads(h.shape[2], kh, 1), same_pads(h.shape[3], kw, 1)
    return F.conv2d(F.pad(h, (l, r, t, bo)), W.permute(3, 2, 0, 1), b.reshape(-1))


def flatten(h):
    """NN.py:296-301 flattening of an NCHW tensor: reshape(transpose(NHWC)) -> [C*W*H, N], row = c*(W*H) + w*H + h."""
    return h.permute(1, 3, 2, 0).reshape(-1, h.shape[0])


def forward_t(layers, params, x, feature_layer=None):
    """Torch forward on float64 tensors.  ``params``: name -> (W, b) in the TF layouts of ``he_init_weights``;
    ``x`` [N, H, W, C].  Returns (logits [c, N], feature [d, N], prev [d', N]): ``prev`` is the input of the feature
    layer (flattened)."""
    n_layers = len(layers)
    fl = n_layers - 2 if feature_layer is None else feature_layer
    h = x.permute(0, 3, 1, 2)
    feat = prev = None
    for i, (name, spec) in enumerate(layers):
        if spec[1] == 'fc' and h.dim() == 4:
            h = flatten(h)
        if i == fl:
            prev = flatten(h) if h.dim() == 4 else h
        if spec[1] == 'conv':
            h = torch.relu(conv(h, *params[name]))
        elif spec[1] == 'pool':
            if spec[0][0] != spec[0][1]:
                raise ValueError('square pools only')
            h = max_pool(h, spec[0][0])
        elif spec[1] == 'fc':
            W, b = params[name]
            h = W @ h + b.reshape(-1, 1)
            if i != n_layers - 1:
                h = torch.relu(h)
        else:
            raise ValueError("Layer's type should be either 'fc', 'conv' or 'pool'.")
        if i == fl:
            feat = flatten(h) if h.dim() == 4 else h
    return h, feat, prev


def torch_params(weights, requires_grad=False):
    return {k: tuple(torch.tensor(np.asarray(a, np.float64), requires_grad=requires_grad) for a in v)
            for k, v in weights.items()}


@torch.no_grad()
def forward(layers, weights, x, feature_layer=None):
    """NumPy in, NumPy out: dict with ``posteriors`` [c, N] (softmax over classes), ``logits`` [c, N], ``feature``
    (output of layer ``feature_layer``, default the one before the last) and ``prev`` (its input), float64."""
    logits, feat, prev = forward_t(layers, torch_params(weights), torch.tensor(np.asarray(x, np.float64)), feature_layer)
    return {'posteriors': torch.softmax(logits, dim=0).numpy(), 'logits': logits.numpy(),
            'feature': None if feat is None else feat.numpy(), 'prev': None if prev is None else prev.numpy()}
