"""Float32 torch-CPU restatement of the forward pass (TEST ORACLE / CPU BASELINE ONLY).

Same TF semantics as ``oracle.nnal_oracle.forward`` (conv SAME stride 1 + bias + ReLU, max-pool
SAME with TF's split of the padding (``pool_same_pads``), flatten row = c*(W*H)+w*H+h, column-batch FC, softmax over classes; NN.py:184-188,
258-340, 1473-1477) but in float32 on all host cores, which is the closest stand-in for the
reference's TensorFlow-CPU execution that can run here (TensorFlow 1.x is not installable;
BASELINE.md §4).  Used by bench.py's ``cpu_baseline`` / ``--impl reference`` legs and by tests as
a fast second opinion."""
import numpy as np
import torch
import torch.nn.functional as F

from .nnal_oracle import pool_same_pads


class TorchForward(object):
    def __init__(self, layers, weights, feature_layer=None, threads=None, dtype=torch.float32):
        """``dtype=torch.float64`` gives a fast float64 oracle for full-size pools (same arithmetic as
        ``oracle.nnal_oracle.forward``, BLAS summation order)."""
        if threads:
            torch.set_num_threads(threads)
        self.layers = list(layers)
        self.feature_layer = feature_layer
        self.dtype = dtype
        self.params = {}
        for name, spec in self.layers:
            if spec[1] == 'conv':
                W, b = weights[name]
                self.params[name] = (torch.from_numpy(np.ascontiguousarray(np.transpose(W, (3, 2, 0, 1)))).to(dtype),
                                     torch.from_numpy(np.ravel(b).copy()).to(dtype))
            elif spec[1] == 'fc':
                W, b = weights[name]
                self.params[name] = (torch.from_numpy(np.ascontiguousarray(W)).to(dtype),
                                     torch.from_numpy(np.ravel(b).copy()).to(dtype))

    @torch.no_grad()
    def __call__(self, x):
        h = torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(self.dtype).permute(0, 3, 1, 2)
        flat = False
        feat = None
        n_layers = len(self.layers)
        for i, (name, spec) in enumerate(self.layers):
            if spec[1] == 'conv':
                W, b = self.params[name]
                h = F.relu(F.conv2d(h, W, b, padding=(W.shape[2] // 2, W.shape[3] // 2)))
            elif spec[1] == 'pool':
                s = spec[0][0]
                (pt, pb), (pl, pr) = pool_same_pads(h.shape[2], s), pool_same_pads(h.shape[3], s)
                if pt or pl:
                    h = F.max_pool2d(F.pad(h, (pl, pr, pt, pb), value=-float('inf')), s, s)
                else:                 # padding after only (always for s = 2): ceil mode is the same window set
                    h = F.max_pool2d(h, s, s, ceil_mode=True)
            else:
                if not flat:
                    h = h.permute(1, 3, 2, 0).reshape(-1, h.shape[0])     # [C,W,H,N] -> [C*W*H, N]
                    flat = True
                W, b = self.params[name]
                h = W @ h + b[:, None]
                if i != n_layers - 1:
                    h = F.relu(h)
            if self.feature_layer is not None and i == self.feature_layer:
                feat = h
        post = torch.softmax(h, dim=0)
        return {'output': h.numpy(), 'posteriors': post.numpy(),
                'feature_layer': None if feat is None else feat.numpy()}
