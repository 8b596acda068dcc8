"""Thin object wrapper over the C-ABI context: owns one ``nnal_ctx`` per process/GPU,
uploads models and volumes, and exposes the pool pass to the reference-named shims."""
import ctypes as C
import os

import numpy as np

from . import _lib as L


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p)


class Engine(object):
    def __init__(self, device=None):
        lib = L.load()
        if device is None:
            device = int(os.environ.get('LOCAL_RANK', '0'))
        h = C.c_void_p()
        rc = lib.nnal_ctx_create(int(device), C.byref(h))
        if rc == L.ERR_NO_DEVICE:
            raise L.NnalError('no usable sm_100 (B200) CUDA device %d: nnal_b200 has no CPU fallback' % device)
        if rc != 0:
            raise L.NnalError('nnal_ctx_create failed with code %d' % rc)
        self.lib = lib
        self.h = h
        self.device = device
        self._model_key = None
        self._model_ref = None
        self._model_token = None
        self._vol_keys = {}
        self._m = {}
        self.volume_cache = True
        self.h2d_bytes = 0
        self.d2h_bytes = 0

    # ------------------------------------------------------------------
    def _chk(self, rc):
        if rc != 0:
            msg = self.lib.nnal_last_error(self.h)
            msg = msg.decode() if msg else ''
            if rc == L.ERR_INVALID:
                raise ValueError(msg or 'invalid argument')
            if rc == L.ERR_OVERFLOW:
                raise L.NnalOverflowError(msg)
            raise L.NnalError('libnnal_b200 error %d: %s' % (rc, msg))

    def close(self):
        if self.h:
            self.lib.nnal_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    factor_budget = 0.35       # fraction of the device memory the FC factors of a whole pool pass may occupy (fi._one_pass)

    def factor_budget_bytes(self):
        free, total = C.c_uint64(), C.c_uint64()
        self._chk(self.lib.nnal_device_memory(self.h, C.byref(free), C.byref(total)))
        return int(self.factor_budget * total.value)

    def synchronize(self):
        self._chk(self.lib.nnal_synchronize(self.h))

    @property
    def stream(self):
        return self.lib.nnal_stream(self.h)

    @property
    def launches(self):
        return int(self.lib.nnal_launch_count(self.h))

    def profile(self, enable):
        self._chk(self.lib.nnal_profile(self.h, 1 if enable else 0))

    def profile_read(self, cls):
        t, c = C.c_double(), C.c_longlong()
        self._chk(self.lib.nnal_profile_read(self.h, int(cls), C.byref(t), C.byref(c)))
        return t.value, c.value

    def layer_info(self, layer):
        ty, macs, tc = C.c_int(), C.c_longlong(), C.c_int()
        self._chk(self.lib.nnal_model_layer_info(self.h, int(layer), C.byref(ty), C.byref(macs), C.byref(tc)))
        return ty.value, macs.value, tc.value

    def pool_eval_device(self, subject, d_inds_ptr, n, offset, patch_shape, stats, norm_mode=L.NORM_BATCH_EVAL):
        """Pool pass over indices already resident in device memory (int64 device pointer)."""
        d1, d2, d3 = [int(p) for p in patch_shape]
        st = None if stats is None else np.ascontiguousarray(stats, dtype=np.float64)
        self._chk(self.lib.nnal_pool_eval_device_inds(self.h, int(subject), C.c_void_p(int(d_inds_ptr)), int(n),
                                                      int(offset), d1, d2, d3,
                                                      None if st is None else _ptr(st), int(norm_mode)))

    def debug_option(self, name, value):
        """Test-only kernel-selection switch (``nnal_debug_option``)."""
        self._chk(self.lib.nnal_debug_option(self.h, str(name).encode(), int(value)))

    def _load_scores_for_test(self, scores):
        s = np.ascontiguousarray(scores, dtype=np.float64).ravel()
        self._chk(self.lib.nnal_debug_set_pool_scores(self.h, _ptr(s) if s.size else None, s.size))
        self._pool_n = s.size

    def debug_fc(self, A, W, b, relu, use_tc):
        A = np.ascontiguousarray(A, dtype=np.float32)
        W = np.ascontiguousarray(W, dtype=np.float32)
        b = np.ascontiguousarray(b, dtype=np.float32).ravel()
        M, K = A.shape
        N = W.shape[0]
        out = np.empty((M, N), dtype=np.float32)
        self._chk(self.lib.nnal_debug_fc(self.h, _ptr(A), _ptr(W), _ptr(b), M, N, K, int(relu), int(use_tc), _ptr(out)))
        return out

    def debug_conv(self, x, W, b, use_tc):
        x = np.ascontiguousarray(x, dtype=np.float32)
        W = np.ascontiguousarray(W, dtype=np.float32)
        b = np.ascontiguousarray(b, dtype=np.float32).ravel()
        n, H, Wd, Cin = x.shape
        ks, _, _, Cout = W.shape
        # use_tc: 0 CUDA cores, 1 tcgen05 (positions on M), 2 weight-stationary tcgen05, 3 = 2 + fused 2x2 max-pool, 4 = 1 + fused pool, 5 = conv1 on the x-im2col'd input
        out = np.empty((n, (H + 1) // 2, (Wd + 1) // 2, Cout) if int(use_tc) in (3, 4) else (n, H, Wd, Cout), dtype=np.float32)
        self._chk(self.lib.nnal_debug_conv(self.h, _ptr(x), _ptr(W), _ptr(b), n, H, Wd, Cin, Cout, ks, int(use_tc),
                                           _ptr(out)))
        return out

    def debug_conv_bwd(self, dz, W, use_tc):
        """Data gradient [n, H, Wd, Cin] of one conv layer from dz [n, H, Wd, Cout] and its filter [ks, ks, Cin, Cout]:
        use_tc 1 the tensor-core kernel of the shrunk-gradient pass, 0 the fp32 CUDA-core kernel."""
        dz = np.ascontiguousarray(dz, dtype=np.float32)
        W = np.ascontiguousarray(W, dtype=np.float32)
        n, H, Wd, Cout = dz.shape
        ks, _, Cin, _ = W.shape
        out = np.empty((n, H, Wd, Cin), dtype=np.float32)
        self._chk(self.lib.nnal_debug_conv_bwd(self.h, _ptr(dz), _ptr(W), n, H, Wd, Cin, Cout, ks, int(use_tc), _ptr(out)))
        return out

    def debug_conv1_gather(self, subject, inds, stats, norm_mode=L.NORM_BATCH_EVAL):
        """Output [n, 25, 25, 24] of the model's conv1 gathering its own 25 x 25 x 1 patches at ``inds`` from the volume
        uploaded as ``subject``."""
        inds = np.ascontiguousarray(inds, dtype=np.int64).ravel()
        st = None if stats is None else np.ascontiguousarray(stats, dtype=np.float64)
        out = np.empty((inds.size, 25, 25, 24), dtype=np.float32)
        self._chk(self.lib.nnal_debug_conv1_gather(self.h, int(subject), _ptr(inds), inds.size,
                                                   None if st is None else _ptr(st), int(norm_mode), _ptr(out)))
        return out

    def set_tensor_cores(self, enable):
        self._chk(self.lib.nnal_set_tensor_cores(self.h, 1 if enable else 0))

    # ------------------------------------------------------------------
    # model
    # ------------------------------------------------------------------
    def host_hash(self, a):
        """64-bit content hash of a C-contiguous host array (multi-threaded in the library)."""
        a = np.ascontiguousarray(a)
        out = C.c_uint64()
        self._chk(self.lib.nnal_host_hash(_ptr(a), a.nbytes, C.byref(out)))
        return out.value

    def set_model(self, model, sess=None):
        """Uploads ``model`` (an ``nnal_b200.NN.CNN``, or any object exposing ``layer_dict``,
        ``input_shape``, ``feature_layer_index`` and ``get_weights(sess)``) unless the same
        weights are already resident.

        The weights are read from the model on EVERY call (``var.eval()`` for a live reference model, NN.py:391-394)
        and re-uploaded when the content hash of any array, the layer list or the input shape changed: a model that
        the reference fine-tuned between two queries is picked up without any ``refresh()`` call."""
        # fast path for models that own PRIVATE copies of their weights and version them (nnal_b200.NN.CNN: set_weights is
        # the only way in and it copies): same object, same version -> nothing to do.  Everything else is re-read.
        token = model.weights_token() if hasattr(model, 'weights_token') else None
        if token is not None and self._model_ref is model and token == self._model_token:
            return
        weights = model.get_weights(sess)
        layers = list(model.layer_dict.items()) if isinstance(model.layer_dict, dict) else list(model.layer_dict)
        specs = (L.LayerSpec * len(layers))()
        for i, (name, spec) in enumerate(layers):
            if spec[1] == 'conv':
                specs[i] = L.LayerSpec(L.LAYER_CONV, int(spec[0]), int(spec[2][0]), int(spec[2][1]))
            elif spec[1] == 'pool':
                specs[i] = L.LayerSpec(L.LAYER_POOL, 0, int(spec[0][0]), int(spec[0][1]))
            elif spec[1] == 'fc':
                specs[i] = L.LayerSpec(L.LAYER_FC, int(spec[0]), 0, 0)
            else:
                raise ValueError("Layer's type should be either 'fc', 'conv' or 'pool'.")
        H, W, Cc = model.input_shape
        fl = model.feature_layer_index if model.feature_layer_index is not None else -1
        arrs = []
        for i, (name, spec) in enumerate(layers):
            if spec[1] == 'pool':
                continue
            Wt, b = weights[name]
            arrs.append((i, np.ascontiguousarray(Wt, dtype=np.float32), np.ascontiguousarray(np.ravel(b), dtype=np.float32)))
        key = (tuple((n, str(sp)) for n, sp in layers), (int(H), int(W), int(Cc)), int(fl),
               tuple((a.shape, self.host_hash(a), self.host_hash(b)) for _, a, b in arrs))
        self._model_ref, self._model_token = (model, token) if token is not None else (None, None)
        if key == self._model_key:
            return
        self._chk(self.lib.nnal_model_set(self.h, specs, len(layers), int(H), int(W), int(Cc), int(fl)))
        for i, Wt, b in arrs:
            self.h2d_bytes += Wt.nbytes + b.nbytes
            self._chk(self.lib.nnal_model_set_weights(self.h, i, _ptr(Wt), _ptr(b)))
        nc, fd, pd = C.c_int(), C.c_int(), C.c_int()
        self._chk(self.lib.nnal_model_info(self.h, C.byref(nc), C.byref(fd), C.byref(pd)))
        self.n_class, self.feat_dim, self.prev_dim = nc.value, fd.value, pd.value
        self._model_key = key

    # ------------------------------------------------------------------
    # volumes
    # ------------------------------------------------------------------
    @staticmethod
    def _as_device_dtype(a):
        a = np.asarray(a)
        if a.dtype == np.float32 or a.dtype == np.float64:
            return np.ascontiguousarray(a)
        if a.dtype in (np.int8, np.uint8, np.int16, np.uint16):
            return np.ascontiguousarray(a, dtype=np.float32)      # exact
        return np.ascontiguousarray(a, dtype=np.float64)          # exact up to 2^53

    def set_volume(self, subject, imgs, pads=(0, 0, 0), shared=False):
        """``imgs``: list of m arrays (X,Y,Z) of one subject (already padded unless ``pads``).  ``shared``: every rank
        passes this same volume in this same call (replicated single-volume pools): with NCCL each rank then copies 1/world
        of it over PCIe and the parts are all-gathered over NVLink."""
        arrs = [self._as_device_dtype(a) for a in imgs]
        if any(a.ndim != 3 or a.shape != arrs[0].shape for a in arrs):
            raise ValueError('all modalities must be 3-D arrays of one shape')
        if any(a.dtype != arrs[0].dtype for a in arrs):
            arrs = [np.ascontiguousarray(a, dtype=np.float64) for a in arrs]
        # Cache: the reference passes the same padded arrays on every query (PW_AL.py:848-853).  A subject is skipped
        # only if the FULL content of every modality is unchanged (64-bit hash over all bytes, nnal_host_hash): an
        # in-place edit anywhere in a volume triggers a re-upload.
        key = None
        if self.volume_cache:
            key = tuple((a.shape, a.dtype.str, self.host_hash(a)) for a in arrs) + (tuple(int(p) for p in pads),)
        hit = key is not None and self._vol_keys.get(subject) == key
        if shared:
            hit = self._all_ranks_agree(hit)          # the sharded upload is a collective: skip it only if EVERY rank can
        if hit:
            return
        X, Y, Z = arrs[0].shape
        dt = L.F64 if arrs[0].dtype == np.float64 else L.F32
        if shared and self._upload_sharded(subject, arrs, dt, pads):
            self._vol_keys[subject] = key
            return
        ptrs = (C.c_void_p * len(arrs))(*[a.ctypes.data for a in arrs])
        self.h2d_bytes += sum(a.nbytes for a in arrs)
        self._chk(self.lib.nnal_volume_set(self.h, int(subject), len(arrs), ptrs, dt, X, Y, Z,
                                           int(pads[0]), int(pads[1]), int(pads[2])))
        self._vol_keys[subject] = key

    @staticmethod
    def _all_ranks_agree(flag):
        from . import dist
        if not dist.is_dist():
            return flag
        import torch
        t = torch.tensor([1 if flag else 0], dtype=torch.int32, device=dist._device())
        dist._td().all_reduce(t, op=dist._td().ReduceOp.MIN)
        return bool(t.item())

    def _upload_sharded(self, subject, arrs, dt, pads):
        """Every rank holds the same host arrays: copy this rank's 1/world slice of each modality host->device and
        all-gather the slices over NVLink on the engine's stream.  Returns False when not applicable."""
        from . import dist
        if not dist.is_dist() or dist._td().get_backend() != 'nccl':
            return False
        import torch
        td = dist._td()
        rank, world = dist.rank_world()
        X, Y, Z = arrs[0].shape
        elems = X * Y * Z
        chunk = -(-elems // world)
        tdt = torch.float64 if arrs[0].dtype == np.float64 else torch.float32
        with dist.engine_stream(self):
            # modality j is gathered straight into its slot; the padding of the last chunk spills into the start of the
            # next slot and is overwritten by that modality's own gather (same stream: ordered); one spare chunk at the end
            stage = torch.empty(len(arrs) * elems + chunk, dtype=tdt, device='cuda')
            send = torch.zeros(chunk, dtype=tdt, device='cuda')
            for j, a in enumerate(arrs):
                flat = a.reshape(-1)
                a0, a1 = min(rank * chunk, elems), min((rank + 1) * chunk, elems)
                if a1 > a0:
                    send[:a1 - a0].copy_(torch.from_numpy(flat[a0:a1]), non_blocking=True)
                    self.h2d_bytes += (a1 - a0) * a.itemsize
                td.all_gather_into_tensor(stage[j * elems:j * elems + world * chunk], send)
            self._chk(self.lib.nnal_volume_set_device(self.h, int(subject), len(arrs), C.c_void_p(stage.data_ptr()), dt, X, Y, Z,
                                                      int(pads[0]), int(pads[1]), int(pads[2])))
            torch.cuda.current_stream().synchronize()       # `stage` / `send` are released after the re-layout kernel ran
        return True

    def invalidate_volumes(self):
        self._vol_keys = {}

    # ------------------------------------------------------------------
    # gather
    # ------------------------------------------------------------------
    @staticmethod
    def _check_inds(inds, padded_shape, patch_shape, pads):
        inds = np.ascontiguousarray(inds, dtype=np.int64).ravel()
        orig = tuple(int(padded_shape[i] + 2 * pads[i] - (patch_shape[i] - 1)) for i in range(3))
        nvox = int(np.prod(orig))
        if inds.size and (inds.min() < 0 or inds.max() >= nvox):
            # np.unravel_index raises ValueError (patch_utils.py:1144)
            raise ValueError('index %d is out of bounds for array with size %d'
                             % (int(inds.max() if inds.max() >= nvox else inds.min()), nvox))
        return inds, orig

    def gather(self, subject, inds, patch_shape, stats=None, norm_mode=L.NORM_NONE, shape=None, pads=(0, 0, 0)):
        inds, _ = self._check_inds(inds, shape, patch_shape, pads)
        d1, d2, d3 = [int(p) for p in patch_shape]
        m = self._m[subject]
        out = np.empty((inds.size, d1, d2, m * d3), dtype=np.float64)
        st = None if stats is None else np.ascontiguousarray(stats, dtype=np.float64)
        self.h2d_bytes += inds.nbytes
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_gather(self.h, int(subject), _ptr(inds), inds.size, d1, d2, d3,
                                       None if st is None else _ptr(st), int(norm_mode), _ptr(out)))
        return out

    def upload(self, subject, imgs, pads=(0, 0, 0), shared=False):
        self.set_volume(subject, imgs, pads, shared)
        self._m[subject] = len(imgs)

    def gather_device(self, subject, d_inds_ptr, n, patch_shape, stats, norm_mode, d_out_ptr):
        """float32 patches of ``n`` voxels (int64 DEVICE indices) into a DEVICE buffer [n,d1,d2,m*d3]."""
        d1, d2, d3 = [int(p) for p in patch_shape]
        st = None if stats is None else np.ascontiguousarray(stats, dtype=np.float64)
        self._chk(self.lib.nnal_gather_device_f32(self.h, int(subject), C.c_void_p(int(d_inds_ptr)), int(n), d1, d2, d3,
                                                  None if st is None else _ptr(st), int(norm_mode), C.c_void_p(int(d_out_ptr))))

    def entropy_device(self, d_post_ptr, c, n, eps, d_out_ptr):
        """float32 entropy map [n] from float32 posteriors [c,n], both in device memory."""
        self._chk(self.lib.nnal_entropy_device_f32(self.h, C.c_void_p(int(d_post_ptr)), int(c), int(n), float(eps),
                                                   C.c_void_p(int(d_out_ptr))))

    # ------------------------------------------------------------------
    # pool pass
    # ------------------------------------------------------------------
    def pool_begin(self, n, keep=0):
        self._chk(self.lib.nnal_pool_begin(self.h, int(n), int(keep)))
        self._pool_n = int(n)

    def pool_eval(self, subject, inds, offset, patch_shape, stats, norm_mode=L.NORM_BATCH_EVAL, shape=None):
        inds, _ = self._check_inds(inds, shape, patch_shape, (0, 0, 0))
        d1, d2, d3 = [int(p) for p in patch_shape]
        st = None if stats is None else np.ascontiguousarray(stats, dtype=np.float64)
        self.h2d_bytes += inds.nbytes
        self._chk(self.lib.nnal_pool_eval(self.h, int(subject), _ptr(inds), inds.size, int(offset), d1, d2, d3,
                                          None if st is None else _ptr(st), int(norm_mode)))

    def pool_eval_images(self, x, offset):
        x = np.ascontiguousarray(x, dtype=np.float32)
        self.h2d_bytes += x.nbytes
        self._chk(self.lib.nnal_pool_eval_images(self.h, _ptr(x), x.shape[0], int(offset)))

    def pool_posteriors(self):
        out = np.empty((self.n_class, self._pool_n), dtype=np.float32)
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_pool_posteriors(self.h, _ptr(out)))
        return out

    def pool_features(self, start=0, n=None):
        n = self._pool_n - start if n is None else n
        out = np.empty((self.feat_dim, n), dtype=np.float32)
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_pool_features(self.h, int(start), int(n), _ptr(out)))
        return out

    # ------------------------------------------------------------------
    # MC-dropout
    # ------------------------------------------------------------------
    dropout_seed = 0          # masks are a pure function of (seed, pass counter, layer, pool position, unit)
    dropout_pass = 0          # advances by T with every stochastic pool pass, like TF's stateful generator would

    def set_dropout_seed(self, seed, first_pass=0):
        self.dropout_seed = int(seed) & 0xffffffffffffffff
        self.dropout_pass = int(first_pass)

    def pool_mc_config(self, T, keep_prob, layers, pos0=0):
        """MC mode for the following pool_begin / pool_eval calls (T = 0: off).  Returns the id of the first pass."""
        lay = np.ascontiguousarray(layers, dtype=np.int32)
        first = self.dropout_pass
        self._chk(self.lib.nnal_pool_mc_config(self.h, int(T), float(keep_prob), self.dropout_seed, first & 0xffffffff,
                                               int(pos0), _ptr(lay) if lay.size else None, int(lay.size)))
        if T > 0:
            self.dropout_pass += int(T)
        return first

    def pool_ensemble_accumulate(self, t):
        """Fold committee member t's deterministic pool pass into the running means (t = 0 opens)."""
        self._chk(self.lib.nnal_pool_ensemble_accumulate(self.h, int(t)))

    def pool_ensemble_end(self):
        self._chk(self.lib.nnal_pool_ensemble_end(self.h))

    def pool_mc_means(self):
        av_post = np.empty(self._pool_n, dtype=np.float64)
        av_ent = np.empty(self._pool_n, dtype=np.float64)
        self.d2h_bytes += av_post.nbytes + av_ent.nbytes
        self._chk(self.lib.nnal_pool_mc_read(self.h, _ptr(av_post), _ptr(av_ent)))
        return av_post, av_ent

    def pool_mc_class_means(self):
        """Running means of every class after an MC-dropout or committee pass: (av_post [c,n], av_ent [n]), float64."""
        av_post = np.empty((self.n_class, self._pool_n), dtype=np.float64)
        av_ent = np.empty(self._pool_n, dtype=np.float64)
        self.d2h_bytes += av_post.nbytes + av_ent.nbytes
        self._chk(self.lib.nnal_pool_mc_read_classes(self.h, _ptr(av_post), _ptr(av_ent)))
        return av_post, av_ent

    def pool_score(self, kind, eps=0.0):
        self._chk(self.lib.nnal_pool_score(self.h, int(kind), float(eps)))

    def pool_scores(self):
        out = np.empty(self._pool_n, dtype=np.float64)
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_pool_scores_read(self.h, _ptr(out)))
        return out

    def pool_topk(self, k, with_scores=False):
        k = int(min(max(k, 0), self._pool_n))
        idx = np.empty(k, dtype=np.int64)
        sc = np.empty(k, dtype=np.float64)
        self.d2h_bytes += idx.nbytes + (sc.nbytes if with_scores else 0)
        self._chk(self.lib.nnal_pool_topk(self.h, k, _ptr(idx), _ptr(sc) if with_scores else None))
        return (idx, sc) if with_scores else idx

    def pool_topk_device(self, k, k_pad, pos_offset, d_pairs_ptr):
        """k best (score, pos_offset + position) pairs of the current pool scores into DEVICE memory (16 B each)."""
        self._chk(self.lib.nnal_pool_topk_device(self.h, int(k), int(k_pad), int(pos_offset), C.c_void_p(int(d_pairs_ptr))))

    def topk_merge_pairs(self, d_pairs_ptr, n_pairs, k):
        """Global k smallest of ``n_pairs`` gathered pairs -> (positions, scores) on the host; padding slots dropped."""
        k = int(k)
        pos = np.empty(k, dtype=np.int64)
        sc = np.empty(k, dtype=np.float64)
        self.d2h_bytes += pos.nbytes + sc.nbytes
        self._chk(self.lib.nnal_topk_merge_pairs(self.h, C.c_void_p(int(d_pairs_ptr)), int(n_pairs), k, _ptr(pos), _ptr(sc)))
        valid = pos != np.iinfo(np.int64).max
        return pos[valid], sc[valid]

    # ------------------------------------------------------------------
    # Fisher information
    # ------------------------------------------------------------------
    def fi_set_candidates(self, cand=None, n_layers=2):
        """Candidates = pool positions ``cand`` (None: every pool sample) of the current pool pass."""
        if cand is None:
            self._chk(self.lib.nnal_fi_set_candidates(self.h, None, 0, int(n_layers)))
        else:
            cand = np.ascontiguousarray(cand, dtype=np.int64).ravel()
            self.h2d_bytes += cand.nbytes
            self._chk(self.lib.nnal_fi_set_candidates(self.h, _ptr(cand), cand.size, int(n_layers)))

    def fi_set_factors(self, p1, U, A_prev=None, w_last=None):
        """Candidates from host factors: ``p1`` [n], ``U`` [n,d], ``A_prev`` [n,d_prev], ``w_last`` [2,d]."""
        p1 = np.ascontiguousarray(p1, dtype=np.float64).ravel()
        U = np.ascontiguousarray(U, dtype=np.float32)
        n, d = U.shape
        if p1.size != n:
            raise ValueError('p1 and U disagree on the number of candidates')
        if A_prev is not None:
            A_prev = np.ascontiguousarray(A_prev, dtype=np.float32)
            w_last = np.ascontiguousarray(w_last, dtype=np.float32)
            if A_prev.shape[0] != n or w_last.shape != (2, d):
                raise ValueError('A_prev must be [n,d_prev] and w_last [2,d]')
        self.h2d_bytes += p1.nbytes + U.nbytes + (A_prev.nbytes + w_last.nbytes if A_prev is not None else 0)
        self._chk(self.lib.nnal_fi_set_factors(self.h, n, d, 0 if A_prev is None else A_prev.shape[1], _ptr(p1), _ptr(U),
                                               None if A_prev is None else _ptr(A_prev),
                                               None if A_prev is None else _ptr(w_last)))

    def fi_info(self):
        n, nl, d, dp, D = C.c_int64(), C.c_int(), C.c_int(), C.c_int(), C.c_double()
        self._chk(self.lib.nnal_fi_info(self.h, C.byref(n), C.byref(nl), C.byref(d), C.byref(dp), C.byref(D)))
        return {'n': n.value, 'n_layers': nl.value, 'd': d.value, 'd_prev': dp.value, 'D': D.value}

    def fi_gram(self, q=None, read=True):
        """Weighted Gram ``sum_i q_i p_i(1-p_i) [u_i;1][u_i;1]^T`` ((d+1)x(d+1) float32)."""
        info = self.fi_info()
        if q is not None:
            q = np.ascontiguousarray(q, dtype=np.float64).ravel()
            if q.size != info['n']:
                raise ValueError('q must have one weight per candidate')
            self.h2d_bytes += q.nbytes
        out = np.empty((info['d'] + 1, info['d'] + 1), dtype=np.float32) if read else None
        if read:
            self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_fi_gram(self.h, None if q is None else _ptr(q), None if out is None else _ptr(out)))
        return out

    def fi_gram_subset(self, cand, q_sub, read=False):
        """Gram over the candidate subset ``cand`` (indices into the candidate list) with weights ``q_sub``; stays on
        the device unless ``read``."""
        cand = np.ascontiguousarray(cand, dtype=np.int64).ravel()
        q_sub = np.ascontiguousarray(q_sub, dtype=np.float64).ravel()
        if cand.size != q_sub.size:
            raise ValueError('one weight per subset candidate expected')
        d = self.fi_info()['d']
        out = np.empty((d + 1, d + 1), dtype=np.float32) if read else None
        self.h2d_bytes += cand.nbytes + q_sub.nbytes
        if read:
            self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_fi_gram_subset(self.h, _ptr(cand) if cand.size else None, cand.size,
                                               _ptr(q_sub) if cand.size else None, None if out is None else _ptr(out)))
        return out

    def fi_gram_solve(self, delta, scale=2.0, d_G2_ptr=None):
        """(tr((delta I + scale H)^-1), tr((delta I + scale H)^-1 (delta I + scale G2)) or None) for the Gram H on the
        device, float64 blocked Gauss-Jordan."""
        tr, ra = C.c_double(), C.c_double()
        self._chk(self.lib.nnal_fi_gram_solve(self.h, float(delta), float(scale),
                                              None if d_G2_ptr is None else C.c_void_p(int(d_G2_ptr)), C.byref(tr), C.byref(ra)))
        self.d2h_bytes += 16
        return tr.value, (ra.value if d_G2_ptr is not None else None)

    def fi_gram_device(self):
        """(device pointer, rows, row stride) of the Gram left on the device by ``fi_gram``."""
        rows, ld = C.c_int64(), C.c_int64()
        p = self.lib.nnal_fi_gram_ptr(self.h, C.byref(rows), C.byref(ld))
        return p, rows.value, ld.value

    def fi_gram_read(self):
        info = self.fi_info()
        out = np.empty((info['d'] + 1, info['d'] + 1), dtype=np.float32)
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_fi_gram_read(self.h, _ptr(out)))
        return out

    def fi_greedy(self, k, delta):
        """Returns (candidate indices in selection order, objective per step, reduced objective)."""
        k = int(min(k, self.fi_info()['n']))
        sel = np.empty(k, dtype=np.int64)
        obj = np.empty(k, dtype=np.float64)
        red = np.empty(k, dtype=np.float64)
        self.d2h_bytes += sel.nbytes + obj.nbytes
        self._chk(self.lib.nnal_fi_greedy(self.h, k, float(delta), _ptr(sel), _ptr(obj), _ptr(red)))
        return sel, obj, red

    def fi_block_set_candidates(self, cand=None, n_layers=1):
        """Multi-class block-form FI over the last ``n_layers`` (1 or 2) FC layers: candidates = pool positions ``cand``
        (None: every pool sample) of the current pool pass, which must have kept the feature layer (and, for two layers,
        the previous FC output: ``keep >= 2``)."""
        if cand is None:
            self._chk(self.lib.nnal_fi_block_set_candidates_nl(self.h, None, 0, int(n_layers)))
            self._fi_block_n = self._pool_n
        else:
            cand = np.ascontiguousarray(cand, dtype=np.int64).ravel()
            self.h2d_bytes += cand.nbytes
            self._chk(self.lib.nnal_fi_block_set_candidates_nl(self.h, _ptr(cand) if cand.size else None, cand.size,
                                                               int(n_layers)))
            self._fi_block_n = cand.size

    def fi_block_set_factors(self, post, U, A_prev=None, w_last=None):
        """Multi-class block-form FI candidates from host factors: ``post`` [c,n] posteriors, ``U`` [n,d] features; for
        the last two FC layers also ``A_prev`` [n,d_prev] (input of the feature layer's FC) and ``w_last`` [c,d] (last FC
        weights), both or neither."""
        post = np.ascontiguousarray(post, dtype=np.float32)
        U = np.ascontiguousarray(U, dtype=np.float32)
        if post.ndim != 2 or U.ndim != 2 or post.shape[1] != U.shape[0]:
            raise ValueError('post must be [c,n] and U [n,d] for the same n')
        c, n = post.shape
        d = U.shape[1]
        if (A_prev is None) != (w_last is None):
            raise ValueError('two-layer FI needs both A_prev and w_last')
        if A_prev is not None:
            A_prev = np.ascontiguousarray(A_prev, dtype=np.float32)
            w_last = np.ascontiguousarray(w_last, dtype=np.float32)
            if A_prev.ndim != 2 or A_prev.shape[0] != n or A_prev.shape[1] < 1 or w_last.shape != (c, d):
                raise ValueError('A_prev must be [n,d_prev] and w_last [c,d]')
            self.h2d_bytes += A_prev.nbytes + w_last.nbytes
        self.h2d_bytes += post.nbytes + U.nbytes
        self._chk(self.lib.nnal_fi_block_set_factors_nl(self.h, n, c, d, 0 if A_prev is None else A_prev.shape[1], _ptr(post),
                                                        _ptr(U), None if A_prev is None else _ptr(A_prev),
                                                        None if A_prev is None else _ptr(w_last)))
        self._fi_block_n = n

    def fi_block_set_candidates_cls(self, cand, r):
        """One-layer block-form FI candidates from the current pool pass (as ``fi_block_set_candidates``), each keeping its
        ``min(r, c)`` most probable classes, 2 <= r <= 32, renormalised (include/nnal_b200.h); any class count."""
        if cand is None:
            self._chk(self.lib.nnal_fi_block_set_candidates_cls(self.h, None, 0, int(r)))
            self._fi_block_n = self._pool_n
        else:
            cand = np.ascontiguousarray(cand, dtype=np.int64).ravel()
            self.h2d_bytes += cand.nbytes
            self._chk(self.lib.nnal_fi_block_set_candidates_cls(self.h, _ptr(cand) if cand.size else None, cand.size, int(r)))
            self._fi_block_n = cand.size

    def fi_block_set_factors_cls(self, cls, p, U, c):
        """One-layer block-form FI candidates from host factors in kept-class form: ``cls`` [n,r] class ids (strictly
        ascending per row, < ``c``), ``p`` [n,r] their posteriors, ``U`` [n,d] features."""
        cls = np.ascontiguousarray(cls, dtype=np.int32)
        p = np.ascontiguousarray(p, dtype=np.float32)
        U = np.ascontiguousarray(U, dtype=np.float32)
        if cls.ndim != 2 or p.shape != cls.shape or U.ndim != 2 or U.shape[0] != cls.shape[0]:
            raise ValueError('cls and p must be [n,r] and U [n,d] for the same n')
        n, r = cls.shape
        self.h2d_bytes += cls.nbytes + p.nbytes + U.nbytes
        self._chk(self.lib.nnal_fi_block_set_factors_cls(self.h, n, int(c), r, U.shape[1], _ptr(cls), _ptr(p), _ptr(U)))
        self._fi_block_n = n

    def pool_top_classes(self, rows, r):
        """The ``min(r, c)`` most probable classes of pool rows ``rows`` of the current pool pass (ties: lower class), as
        the class-capped block FI keeps them: (ids [n,q] int32 ascending, posteriors [n,q] float32)."""
        rows = np.ascontiguousarray(rows, dtype=np.int64).ravel()
        q = min(int(r), self.n_class)
        cls = np.empty((rows.size, q), dtype=np.int32)
        p = np.empty((rows.size, q), dtype=np.float32)
        self.h2d_bytes += rows.nbytes
        self.d2h_bytes += cls.nbytes + p.nbytes
        self._chk(self.lib.nnal_pool_top_classes(self.h, _ptr(rows) if rows.size else None, rows.size, int(r), _ptr(cls),
                                                 _ptr(p)))
        return cls, p

    def fi_block_greedy(self, k, delta):
        """Block-form greedy FI selection.  Returns (candidate indices in selection order, objective per step, reduced
        objective ``tr((delta I + K_SS/s)^-1)`` per step)."""
        k = int(k)
        n = getattr(self, '_fi_block_n', None)
        if n is not None:
            k = min(k, n)
        sel = np.empty(max(k, 1), dtype=np.int64)
        obj = np.empty(max(k, 1), dtype=np.float64)
        red = np.empty(max(k, 1), dtype=np.float64)
        self.d2h_bytes += 16 * k
        self._chk(self.lib.nnal_fi_block_greedy(self.h, k, float(delta), _ptr(sel), _ptr(obj), _ptr(red)))
        return sel[:k], obj[:k], red[:k]

    # ------------------------------------------------------------------
    # the reference's shrunk FI coordinates + SDP query distribution
    # ------------------------------------------------------------------
    def fi_shrunk_tau(self):
        tau = C.c_int()
        self._chk(self.lib.nnal_fi_shrunk_tau(self.h, C.byref(tau)))
        return tau.value

    def fi_shrunk_images(self, x):
        """Shrunk class-score gradients of host samples ``x`` [n,H,W,C]: (posteriors [c,n] float32, g [c,n,tau] float64)."""
        x = np.ascontiguousarray(x, dtype=np.float32)
        n = x.shape[0]
        post = np.empty((self.n_class, n), dtype=np.float32)
        g = np.empty((self.n_class, n, self.fi_shrunk_tau()), dtype=np.float64)
        self.h2d_bytes += x.nbytes
        self.d2h_bytes += post.nbytes + g.nbytes
        self._chk(self.lib.nnal_fi_shrunk_images(self.h, _ptr(x), n, _ptr(post), _ptr(g)))
        return post, g

    def fi_shrunk_voxels(self, subject, inds, patch_shape, stats, norm_mode=L.NORM_BATCH_EVAL, shape=None):
        """Same, for voxels of an uploaded subject (gathered and normalised on the device)."""
        inds, _ = self._check_inds(inds, shape, patch_shape, (0, 0, 0))
        d1, d2, d3 = [int(p) for p in patch_shape]
        st = None if stats is None else np.ascontiguousarray(stats, dtype=np.float64)
        post = np.empty((self.n_class, inds.size), dtype=np.float32)
        g = np.empty((self.n_class, inds.size, self.fi_shrunk_tau()), dtype=np.float64)
        self.h2d_bytes += inds.nbytes
        self.d2h_bytes += post.nbytes + g.nbytes
        self._chk(self.lib.nnal_fi_shrunk_voxels(self.h, int(subject), _ptr(inds), inds.size, d1, d2, d3,
                                                 None if st is None else _ptr(st), int(norm_mode), _ptr(post), _ptr(g)))
        return post, g

    def sdp_query_distribution(self, A, tol=1e-4, max_iter=200000, gamma=1.0):
        """min tr((sum_i q_i A_i)^-1) over the simplex; ``A`` [n,tau,tau] float64.  ``gamma``: exponent of the
        multiplicative update; above 0.5 it is used until the objective increases once, then 0.5 (monotone).
        Returns dict(q, t, objective, gap, iterations)."""
        A = np.ascontiguousarray(A, dtype=np.float64)
        if A.ndim != 3 or A.shape[1] != A.shape[2]:
            raise ValueError('A must be [n, tau, tau]')
        n, tau = A.shape[0], A.shape[1]
        q = np.empty(n, dtype=np.float64)
        t = np.empty(tau, dtype=np.float64)
        obj, gap, it = C.c_double(), C.c_double(), C.c_int64()
        self.h2d_bytes += A.nbytes
        self.d2h_bytes += q.nbytes
        self._chk(self.lib.nnal_sdp_query_distribution(self.h, _ptr(A), n, tau, float(tol), int(max_iter), float(gamma),
                                                       _ptr(q), _ptr(t), C.byref(obj), C.byref(gap), C.byref(it)))
        return {'q': q, 't': t, 'objective': obj.value, 'gap': gap.value, 'iterations': it.value}

    def sdp_query_distribution_reg(self, A, lambda_, X, tol=1e-4, max_iter=20000):
        """The feature-regularised programme (``lambda_ > 0``, NNAL_tools.py:625-644): min tr((sum q_i A_i)^-1) - lambda sum
        q_i |x_i|^2 over {q >= 0, sum q = 1, X q = 0}; ``A`` [n,tau,tau], ``X`` [d,n] float64."""
        A = np.ascontiguousarray(A, dtype=np.float64)
        X = np.ascontiguousarray(X, dtype=np.float64)
        if A.ndim != 3 or A.shape[1] != A.shape[2] or X.ndim != 2 or X.shape[1] != A.shape[0]:
            raise ValueError('A must be [n, tau, tau] and X [d, n]')
        n, tau = A.shape[0], A.shape[1]
        q = np.empty(n, dtype=np.float64)
        t = np.empty(tau, dtype=np.float64)
        obj, gap, it = C.c_double(), C.c_double(), C.c_int64()
        self.h2d_bytes += A.nbytes + X.nbytes
        self.d2h_bytes += q.nbytes
        self._chk(self.lib.nnal_sdp_query_distribution_reg(self.h, _ptr(A), n, tau, float(lambda_), _ptr(X), X.shape[0], float(tol),
                                                           int(max_iter), _ptr(q), _ptr(t), C.byref(obj), C.byref(gap), C.byref(it)))
        return {'q': q, 't': t, 'objective': obj.value, 'gap': gap.value, 'iterations': it.value}

    def sdp_from_shrunk(self, g, p1, diag_load, tol=1e-4, max_iter=200000, gamma=1.0):
        """``sdp_query_distribution`` on the binary A-matrices of ``gen_A_matrices``, assembled on the device from the
        shrunk gradients ``g`` [2,n,tau] and ``p1`` [n] = P(class 1)."""
        g = np.ascontiguousarray(g, dtype=np.float64)
        p1 = np.ascontiguousarray(p1, dtype=np.float64).ravel()
        if g.ndim != 3 or g.shape[0] != 2 or g.shape[1] != p1.size:
            raise ValueError('g must be [2, n, tau] and p1 [n]')
        n, tau = g.shape[1], g.shape[2]
        q = np.empty(n, dtype=np.float64)
        t = np.empty(tau, dtype=np.float64)
        obj, gap, it = C.c_double(), C.c_double(), C.c_int64()
        self.h2d_bytes += g.nbytes + p1.nbytes
        self.d2h_bytes += q.nbytes
        self._chk(self.lib.nnal_sdp_from_shrunk(self.h, _ptr(g), _ptr(p1), n, tau, float(diag_load), float(tol), int(max_iter),
                                                float(gamma), _ptr(q), _ptr(t), C.byref(obj), C.byref(gap), C.byref(it)))
        return {'q': q, 't': t, 'objective': obj.value, 'gap': gap.value, 'iterations': it.value}

    def if_lissa(self, pool_post, pool_U, labels, tr_post, tr_U, scale):
        """Last-layer influence recursion (``nnal_if_lissa``): ``pool_post`` [c,n], ``pool_U`` [n,d], ``labels`` [n],
        ``tr_post`` [T,c], ``tr_U`` [T,d] in iteration order -> V [(d+1)c, n] float64."""
        pool_post = np.ascontiguousarray(pool_post, dtype=np.float32)
        pool_U = np.ascontiguousarray(pool_U, dtype=np.float32)
        labels = np.ascontiguousarray(labels, dtype=np.int64).ravel()
        tr_post = np.ascontiguousarray(tr_post, dtype=np.float32)
        tr_U = np.ascontiguousarray(tr_U, dtype=np.float32)
        c, n = pool_post.shape
        d = pool_U.shape[1]
        T = tr_post.shape[0]
        if pool_U.shape[0] != n or labels.size != n or tr_U.shape != (T, d) or (T and tr_post.shape[1] != c):
            raise ValueError('inconsistent factor shapes')
        V = np.empty(((d + 1) * c, n), dtype=np.float64)
        self.h2d_bytes += pool_post.nbytes + pool_U.nbytes + labels.nbytes + tr_post.nbytes + tr_U.nbytes
        self.d2h_bytes += V.nbytes
        self._chk(self.lib.nnal_if_lissa(self.h, n, c, d, _ptr(pool_post), _ptr(pool_U), _ptr(labels), T,
                                         _ptr(tr_post) if T else None, _ptr(tr_U) if T else None, float(scale), _ptr(V)))
        return V

    def fi_begin(self, k, delta):
        self._chk(self.lib.nnal_fi_begin(self.h, int(k), float(delta)))

    def fi_step_local_best(self, step):
        loss, cand, trc = C.c_double(), C.c_int64(), C.c_double()
        self._chk(self.lib.nnal_fi_step_local_best(self.h, int(step), C.byref(loss), C.byref(cand), C.byref(trc)))
        return loss.value, cand.value, trc.value

    def fi_winner_factors(self, step, cand):
        """Message of the step's winner (local candidate ``cand``): factors + its K_SS row."""
        out = np.empty(self.fi_factor_len(step), dtype=np.float32)
        nf = C.c_int64()
        self._chk(self.lib.nnal_fi_winner_factors(self.h, int(step), int(cand), _ptr(out), C.byref(nf)))
        self.d2h_bytes += out.nbytes
        return out

    def fi_factor_len(self, step):
        nf = C.c_int64()
        self._chk(self.lib.nnal_fi_winner_factors(self.h, int(step), 0, None, C.byref(nf)))
        return nf.value

    # device-resident multi-rank step (messages live in device memory; the caller all-gathers them)
    def fi_set_gids(self, gids):
        gids = np.ascontiguousarray(gids, dtype=np.int64).ravel()
        self.h2d_bytes += gids.nbytes
        self._chk(self.lib.nnal_fi_set_gids(self.h, _ptr(gids) if gids.size else None, gids.size))

    def fi_msg_bytes(self):
        b = C.c_int64()
        self._chk(self.lib.nnal_fi_msg_bytes(self.h, C.byref(b)))
        return b.value

    def fi_step_pack(self, step, d_msg_ptr):
        self._chk(self.lib.nnal_fi_step_pack(self.h, int(step), C.c_void_p(int(d_msg_ptr))))

    def fi_step_apply_gathered(self, step, d_msgs_ptr, world, rank):
        self._chk(self.lib.nnal_fi_step_apply_gathered(self.h, int(step), C.c_void_p(int(d_msgs_ptr)), int(world), int(rank)))

    # peer-memory exchange of the greedy step messages (csrc/p2p.cu)
    def p2p_alloc(self, world, rank, slot_bytes):
        h = (C.c_ubyte * 64)()
        self._chk(self.lib.nnal_p2p_alloc(self.h, int(world), int(rank), int(slot_bytes), C.cast(h, C.c_void_p)))
        return bytes(h)

    def p2p_open(self, handles):
        buf = (C.c_ubyte * len(handles)).from_buffer_copy(handles)
        self._chk(self.lib.nnal_p2p_open(self.h, C.cast(buf, C.c_void_p)))

    def p2p_base(self):
        out = C.c_void_p()
        self._chk(self.lib.nnal_p2p_base(self.h, C.byref(out)))
        return out.value

    def p2p_open_local(self, bases):
        arr = (C.c_void_p * len(bases))(*[int(b) for b in bases])
        self._chk(self.lib.nnal_p2p_open_local(self.h, C.cast(arr, C.c_void_p)))

    def p2p_allgather(self, d_send_ptr, nbytes, seq):
        out = C.c_void_p()
        self._chk(self.lib.nnal_p2p_allgather(self.h, C.c_void_p(int(d_send_ptr)), int(nbytes), int(seq), C.byref(out)))
        return out.value

    def fi_result(self, k):
        sel = np.empty(int(k), dtype=np.int64)
        red = np.empty(int(k), dtype=np.float64)
        self.d2h_bytes += sel.nbytes + red.nbytes
        self._chk(self.lib.nnal_fi_result(self.h, int(k), _ptr(sel), _ptr(red)))
        return sel, red

    message_device = 'cuda'

    def fi_step_apply(self, step, factors, owner_is_local, cand_local):
        factors = np.ascontiguousarray(factors, dtype=np.float32)
        self.h2d_bytes += factors.nbytes
        self._chk(self.lib.nnal_fi_step_apply(self.h, int(step), _ptr(factors), factors.size, 1 if owner_is_local else 0,
                                              int(cand_local)))

    # ------------------------------------------------------------------
    # representativeness queries (rep-entropy, core-set)
    # ------------------------------------------------------------------
    def pool_feature_rows(self, pos):
        """Feature-layer rows of pool positions ``pos`` as ``[len(pos), d]`` float32."""
        pos = np.ascontiguousarray(pos, dtype=np.int64).ravel()
        out = np.empty((pos.size, self.feat_dim), dtype=np.float32)
        self.h2d_bytes += pos.nbytes
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_pool_feature_rows(self.h, _ptr(pos) if pos.size else None, pos.size,
                                                  _ptr(out) if pos.size else None))
        return out

    def pool_prev_rows(self, pos):
        """Rows of the previous FC layer's output (input of the feature layer's FC) at pool positions ``pos`` as
        ``[len(pos), prev_dim]`` float32; the pool pass must have kept it (``keep >= 2``)."""
        pos = np.ascontiguousarray(pos, dtype=np.int64).ravel()
        out = np.empty((pos.size, self.prev_dim), dtype=np.float32)
        self.h2d_bytes += pos.nbytes
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_pool_prev_rows(self.h, _ptr(pos) if pos.size else None, pos.size,
                                               _ptr(out) if pos.size else None))
        return out

    def rep_set(self, cols, excl_pos, k):
        cols = np.ascontiguousarray(cols, dtype=np.float32)
        excl = np.ascontiguousarray(excl_pos, dtype=np.int64).ravel()
        self.h2d_bytes += cols.nbytes + excl.nbytes
        self._rep_B = cols.shape[0]
        self._chk(self.lib.nnal_rep_set(self.h, _ptr(cols) if cols.size else None, cols.shape[0],
                                        _ptr(excl) if excl.size else None, excl.size, int(k)))

    def rep_step_scores(self, d_scores_ptr):
        self._chk(self.lib.nnal_rep_step_scores(self.h, C.c_void_p(int(d_scores_ptr))))

    def rep_step_pick(self, step, d_scores_ptr):
        self._chk(self.lib.nnal_rep_step_pick(self.h, int(step), C.c_void_p(int(d_scores_ptr))))

    def rep_greedy(self, k):
        k = int(min(k, self._rep_B))
        sel = np.empty(k, dtype=np.int64)
        val = np.empty(k, dtype=np.float64)
        self.d2h_bytes += sel.nbytes + val.nbytes
        self._chk(self.lib.nnal_rep_greedy(self.h, k, _ptr(sel), _ptr(val)))
        return sel, val

    def sel_result(self, k):
        sel = np.empty(int(k), dtype=np.int64)
        val = np.empty(int(k), dtype=np.float64)
        self.d2h_bytes += sel.nbytes + val.nbytes
        self._chk(self.lib.nnal_sel_result(self.h, int(k), _ptr(sel), _ptr(val)))
        return sel, val

    def cross_sims(self, F2):
        """max_j cos(pool row i, F2[j]) for every sample of the current pool pass (float64 [n])."""
        F2 = np.ascontiguousarray(F2, dtype=np.float32)
        out = np.empty(self._pool_n, dtype=np.float64)
        self.h2d_bytes += F2.nbytes
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_cross_sims(self.h, _ptr(F2), F2.shape[0], _ptr(out)))
        return out

    def cs_begin(self, init, sims0, gids, k):
        s0 = None if sims0 is None else np.ascontiguousarray(sims0, dtype=np.float64)
        g = None if gids is None else np.ascontiguousarray(gids, dtype=np.int64)
        self._chk(self.lib.nnal_cs_begin(self.h, int(init), None if s0 is None else _ptr(s0),
                                         None if g is None or g.size == 0 else _ptr(g), int(k)))

    def cs_msg_bytes(self):
        b = C.c_int64()
        self._chk(self.lib.nnal_cs_msg_bytes(self.h, C.byref(b)))
        return b.value

    def cs_step_pack(self, step, d_msg_ptr):
        self._chk(self.lib.nnal_cs_step_pack(self.h, int(step), C.c_void_p(int(d_msg_ptr))))

    def cs_step_apply_gathered(self, step, d_msgs_ptr, world, rank):
        self._chk(self.lib.nnal_cs_step_apply_gathered(self.h, int(step), C.c_void_p(int(d_msgs_ptr)), int(world), int(rank)))

    def cs_greedy(self, k):
        k = int(min(k, self._pool_n))
        sel = np.empty(k, dtype=np.int64)
        val = np.empty(k, dtype=np.float64)
        self.d2h_bytes += sel.nbytes + val.nbytes
        self._chk(self.lib.nnal_cs_greedy(self.h, k, _ptr(sel), _ptr(val)))
        return sel, val

    # ------------------------------------------------------------------
    # stand-alone helpers
    # ------------------------------------------------------------------
    def entropy(self, P, kind=L.SCORE_ENTROPY, eps=10e-8):
        P = np.ascontiguousarray(P, dtype=np.float64)
        c, n = P.shape
        out = np.empty(n, dtype=np.float64)
        self.h2d_bytes += P.nbytes
        self.d2h_bytes += out.nbytes
        self._chk(self.lib.nnal_entropy(self.h, _ptr(P), c, n, int(kind), float(eps), _ptr(out)))
        return out

    def topk(self, scores, k):
        s = np.ascontiguousarray(scores, dtype=np.float64).ravel()
        k = int(min(max(k, 0), s.size))
        idx = np.empty(k, dtype=np.int64)
        self.h2d_bytes += s.nbytes
        self.d2h_bytes += idx.nbytes
        self._chk(self.lib.nnal_topk(self.h, _ptr(s), s.size, k, _ptr(idx)))
        return idx


_engine = None


def get_engine():
    """Process-wide engine on the GPU named by LOCAL_RANK (one process per GPU)."""
    global _engine
    if _engine is None:
        _engine = Engine()
    return _engine


def reset_engine():
    global _engine
    if _engine is not None:
        _engine.close()
    _engine = None
