"""ctypes binding of libnnal_b200.so (the C ABI declared in include/nnal_b200.h)."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libnnal_b200.so')

c_i64p = C.POINTER(C.c_int64)
c_f32p = C.POINTER(C.c_float)
c_f64p = C.POINTER(C.c_double)
c_vp = C.c_void_p


class LayerSpec(C.Structure):
    _fields_ = [('type', C.c_int32), ('out', C.c_int32), ('kh', C.c_int32), ('kw', C.c_int32)]


# name -> (restype, argtypes); every symbol include/nnal_b200.h declares
SIGNATURES = {
    'nnal_version': (C.c_int, []),
    'nnal_ctx_create': (C.c_int, [C.c_int, C.POINTER(c_vp)]),
    'nnal_ctx_destroy': (C.c_int, [c_vp]),
    'nnal_last_error': (C.c_char_p, [c_vp]),
    'nnal_launch_count': (C.c_longlong, [c_vp]),
    'nnal_set_tensor_cores': (C.c_int, [c_vp, C.c_int]),
    'nnal_synchronize': (C.c_int, [c_vp]),
    'nnal_stream': (c_vp, [c_vp]),
    'nnal_device_memory': (C.c_int, [c_vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    'nnal_host_hash': (C.c_int, [c_vp, C.c_uint64, C.POINTER(C.c_uint64)]),
    'nnal_profile': (C.c_int, [c_vp, C.c_int]),
    'nnal_profile_read': (C.c_int, [c_vp, C.c_int, c_f64p, C.POINTER(C.c_longlong)]),
    'nnal_model_layer_info': (C.c_int, [c_vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_longlong),
                                        C.POINTER(C.c_int)]),
    'nnal_model_set': (C.c_int, [c_vp, C.POINTER(LayerSpec), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    'nnal_model_set_weights': (C.c_int, [c_vp, C.c_int, c_vp, c_vp]),
    'nnal_model_info': (C.c_int, [c_vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    'nnal_volume_set': (C.c_int, [c_vp, C.c_int, C.c_int, C.POINTER(c_vp), C.c_int, C.c_int64, C.c_int64,
                                  C.c_int64, C.c_int64, C.c_int64, C.c_int64]),
    'nnal_volume_set_device': (C.c_int, [c_vp, C.c_int, C.c_int, c_vp, C.c_int, C.c_int64, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_int64, C.c_int64]),
    'nnal_volume_clear': (C.c_int, [c_vp]),
    'nnal_gather': (C.c_int, [c_vp, C.c_int, c_vp, C.c_int64, C.c_int, C.c_int, C.c_int, c_vp, C.c_int, c_vp]),
    'nnal_gather_device_f32': (C.c_int, [c_vp, C.c_int, c_vp, C.c_int64, C.c_int, C.c_int, C.c_int, c_vp, C.c_int, c_vp]),
    'nnal_entropy_device_f32': (C.c_int, [c_vp, c_vp, C.c_int, C.c_int64, C.c_double, c_vp]),
    'nnal_pool_begin': (C.c_int, [c_vp, C.c_int64, C.c_int]),
    'nnal_pool_eval': (C.c_int, [c_vp, C.c_int, c_vp, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int, c_vp, C.c_int]),
    'nnal_pool_eval_images': (C.c_int, [c_vp, c_vp, C.c_int64, C.c_int64]),
    'nnal_pool_eval_device_inds': (C.c_int, [c_vp, C.c_int, c_vp, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_int,
                                             c_vp, C.c_int]),
    'nnal_pool_posteriors': (C.c_int, [c_vp, c_vp]),
    'nnal_pool_features': (C.c_int, [c_vp, C.c_int64, C.c_int64, c_vp]),
    'nnal_pool_score': (C.c_int, [c_vp, C.c_int, C.c_double]),
    'nnal_pool_mc_config': (C.c_int, [c_vp, C.c_int, C.c_double, C.c_ulonglong, C.c_uint, C.c_longlong, c_vp, C.c_int]),
    'nnal_pool_mc_read': (C.c_int, [c_vp, c_vp, c_vp]),
    'nnal_pool_ensemble_accumulate': (C.c_int, [c_vp, C.c_int]),
    'nnal_pool_ensemble_end': (C.c_int, [c_vp]),
    'nnal_pool_scores_read': (C.c_int, [c_vp, c_vp]),
    'nnal_pool_topk': (C.c_int, [c_vp, C.c_int64, c_vp, c_vp]),
    'nnal_pool_topk_device': (C.c_int, [c_vp, C.c_int64, C.c_int64, C.c_int64, c_vp]),
    'nnal_topk_merge_pairs': (C.c_int, [c_vp, c_vp, C.c_int64, C.c_int64, c_vp, c_vp]),
    'nnal_entropy': (C.c_int, [c_vp, c_vp, C.c_int, C.c_int64, C.c_int, C.c_double, c_vp]),
    'nnal_topk': (C.c_int, [c_vp, c_vp, C.c_int64, C.c_int64, c_vp]),
    'nnal_debug_option': (C.c_int, [c_vp, C.c_char_p, C.c_long]),
    'nnal_debug_set_pool_scores': (C.c_int, [c_vp, c_vp, C.c_int64]),
    'nnal_debug_fc': (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, c_vp]),
    'nnal_debug_conv': (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                  C.c_int, c_vp]),
    'nnal_rep_set': (C.c_int, [c_vp, c_vp, C.c_int64, c_vp, C.c_int64, C.c_int64]),
    'nnal_rep_step_scores': (C.c_int, [c_vp, c_vp]),
    'nnal_rep_step_pick': (C.c_int, [c_vp, C.c_int64, c_vp]),
    'nnal_rep_greedy': (C.c_int, [c_vp, C.c_int64, c_vp, c_vp]),
    'nnal_sel_result': (C.c_int, [c_vp, C.c_int64, c_vp, c_vp]),
    'nnal_cross_sims': (C.c_int, [c_vp, c_vp, C.c_int64, c_vp]),
    'nnal_cs_begin': (C.c_int, [c_vp, C.c_int, c_vp, c_vp, C.c_int64]),
    'nnal_cs_msg_bytes': (C.c_int, [c_vp, c_i64p]),
    'nnal_cs_step_pack': (C.c_int, [c_vp, C.c_int64, c_vp]),
    'nnal_cs_step_apply_gathered': (C.c_int, [c_vp, C.c_int64, c_vp, C.c_int, C.c_int]),
    'nnal_cs_greedy': (C.c_int, [c_vp, C.c_int64, c_vp, c_vp]),
    'nnal_pool_feature_rows': (C.c_int, [c_vp, c_vp, C.c_int64, c_vp]),
    'nnal_fi_set_candidates': (C.c_int, [c_vp, c_vp, C.c_int64, C.c_int]),
    'nnal_fi_set_factors': (C.c_int, [c_vp, C.c_int64, C.c_int, C.c_int, c_vp, c_vp, c_vp, c_vp]),
    'nnal_fi_info': (C.c_int, [c_vp, c_i64p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), c_f64p]),
    'nnal_fi_gram': (C.c_int, [c_vp, c_vp, c_vp]),
    'nnal_fi_gram_subset': (C.c_int, [c_vp, c_vp, C.c_int64, c_vp, c_vp]),
    'nnal_fi_gram_solve': (C.c_int, [c_vp, C.c_double, C.c_double, c_vp, c_f64p, c_f64p]),
    'nnal_fi_gram_ptr': (c_vp, [c_vp, c_i64p, c_i64p]),
    'nnal_fi_gram_read': (C.c_int, [c_vp, c_vp]),
    'nnal_fi_greedy': (C.c_int, [c_vp, C.c_int64, C.c_double, c_vp, c_vp, c_vp]),
    'nnal_fi_begin': (C.c_int, [c_vp, C.c_int64, C.c_double]),
    'nnal_fi_step_local_best': (C.c_int, [c_vp, C.c_int64, c_f64p, c_i64p, c_f64p]),
    'nnal_fi_winner_factors': (C.c_int, [c_vp, C.c_int64, C.c_int64, c_vp, c_i64p]),
    'nnal_fi_set_gids': (C.c_int, [c_vp, c_vp, C.c_int64]),
    'nnal_fi_msg_bytes': (C.c_int, [c_vp, c_i64p]),
    'nnal_fi_step_pack': (C.c_int, [c_vp, C.c_int64, c_vp]),
    'nnal_fi_step_apply_gathered': (C.c_int, [c_vp, C.c_int64, c_vp, C.c_int, C.c_int]),
    'nnal_fi_result': (C.c_int, [c_vp, C.c_int64, c_vp, c_vp]),
    'nnal_fi_block_set_candidates': (C.c_int, [c_vp, c_vp, C.c_int64]),
    'nnal_fi_block_set_factors': (C.c_int, [c_vp, C.c_int64, C.c_int, C.c_int, c_vp, c_vp]),
    'nnal_fi_block_greedy': (C.c_int, [c_vp, C.c_int64, C.c_double, c_vp, c_vp, c_vp]),
    'nnal_p2p_alloc':(C.c_int, [c_vp, C.c_int, C.c_int, C.c_int64, c_vp]),
    'nnal_p2p_open': (C.c_int, [c_vp, c_vp]),
    'nnal_p2p_allgather': (C.c_int, [c_vp, c_vp, C.c_int64, C.c_uint64, c_vp]),
    'nnal_p2p_base': (C.c_int, [c_vp, c_vp]),
    'nnal_p2p_open_local': (C.c_int, [c_vp, c_vp]),
    'nnal_fi_step_apply': (C.c_int, [c_vp, C.c_int64, c_vp, C.c_int64, C.c_int, C.c_int64]),
    'nnal_fi_shrunk_tau': (C.c_int, [c_vp, C.POINTER(C.c_int)]),
    'nnal_fi_shrunk_images': (C.c_int, [c_vp, c_vp, C.c_int64, c_vp, c_vp]),
    'nnal_fi_shrunk_voxels': (C.c_int, [c_vp, C.c_int, c_vp, C.c_int64, C.c_int, C.c_int, C.c_int, c_vp, C.c_int, c_vp,
                                        c_vp]),
    'nnal_if_lissa': (C.c_int, [c_vp, C.c_int64, C.c_int, C.c_int, c_vp, c_vp, c_vp, C.c_int64, c_vp, c_vp, C.c_double, c_vp]),
    'nnal_sdp_query_distribution': (C.c_int, [c_vp, c_vp, C.c_int64, C.c_int, C.c_double, C.c_int64, C.c_double, c_vp,
                                              c_vp, c_f64p, c_f64p, c_i64p]),
    'nnal_sdp_query_distribution_reg': (C.c_int, [c_vp, c_vp, C.c_int64, C.c_int, C.c_double, c_vp, C.c_int, C.c_double, C.c_int64,
                                                  c_vp, c_vp, c_f64p, c_f64p, c_i64p]),
    'nnal_sdp_from_shrunk': (C.c_int, [c_vp, c_vp, c_vp, C.c_int64, C.c_int, C.c_double, C.c_double, C.c_int64, C.c_double,
                                       c_vp, c_vp, c_f64p, c_f64p, c_i64p]),
}

NNAL_OK, ERR_INVALID, ERR_CUDA, ERR_STATE, ERR_UNSUPPORTED, ERR_NO_DEVICE, ERR_OVERFLOW = 0, 1, 2, 3, 4, 5, 6
LAYER_CONV, LAYER_POOL, LAYER_FC = 0, 1, 2
F32, F64 = 0, 1
NORM_NONE, NORM_BATCH_EVAL, NORM_MULTIMG = 0, 1, 2
SCORE_BINARY, SCORE_NEG_ENTROPY, SCORE_ENTROPY, SCORE_NEG_FI_TRACE = 0, 1, 2, 3
SCORE_MC_BINARY, SCORE_NEG_BALD = 10, 11

_lib = None


class NnalError(RuntimeError):
    pass


class NnalOverflowError(NnalError, OverflowError):
    """An input, weight or activation left the fp16 operand range of the tensor-core path (NNAL_ERR_OVERFLOW)."""


def load():
    """Loads the shared library; raises (never falls back) when it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NnalError('libnnal_b200.so not found at %s: build it with `python -c "import __graft_entry__ as g; '
                        'g.build()"` (nvcc, sm_100a). There is no CPU fallback.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
