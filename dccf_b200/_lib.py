"""ctypes binding of the C-ABI library (include/dccf_b200.h -> dccf_b200/libdccf_b200.so).

PyTorch is used only for device memory and streams: every entry point takes raw device pointers
(`tensor.data_ptr()`) and the current CUDA stream.  There is NO CPU fallback: if the library is
missing, fails to load, or a call returns an error, a `DccfError` is raised.
"""
import ctypes
import os

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, 'libdccf_b200.so')
ABI_VERSION = 40
DIM = 64


class DccfError(RuntimeError):
    pass


class Dims(ctypes.Structure):
    _fields_ = [('n_users', ctypes.c_int32), ('n_items', ctypes.c_int32), ('dim', ctypes.c_int32),
                ('feat_dim', ctypes.c_int32), ('n_samples', ctypes.c_int32), ('n_attr', ctypes.c_int32),
                ('user_base', ctypes.c_int32), ('_pad', ctypes.c_int32)]


class Expo(ctypes.Structure):
    _fields_ = [('mode', ctypes.c_int32), ('_pad', ctypes.c_int32), ('dense', ctypes.c_void_p),
                ('mf_user', ctypes.c_void_p), ('mf_item', ctypes.c_void_p), ('mf_user_bias', ctypes.c_void_p),
                ('mf_item_bias', ctypes.c_void_p), ('propensity', ctypes.c_void_p),
                ('mf_global_bias', ctypes.c_float), ('mf_min_propensity', ctypes.c_float)]


class Rng(ctypes.Structure):
    _fields_ = [('noise_mode', ctypes.c_int32), ('mask_mode', ctypes.c_int32), ('noise', ctypes.c_void_p),
                ('mask', ctypes.c_void_p), ('noise_std', ctypes.c_float), ('p_drop', ctypes.c_float),
                ('seed', ctypes.c_uint64), ('offset', ctypes.c_uint64), ('offset_dev', ctypes.c_void_p)]


class Adam(ctypes.Structure):
    _fields_ = [('lr', ctypes.c_double), ('beta1', ctypes.c_double), ('beta2', ctypes.c_double),
                ('eps', ctypes.c_double), ('l2', ctypes.c_double), ('weight_decay', ctypes.c_double),
                ('clip', ctypes.c_double), ('step', ctypes.c_int32), ('rule', ctypes.c_int32),
                ('step_dev', ctypes.c_void_p)]


class AdamTable(ctypes.Structure):
    _fields_ = [('table', ctypes.c_void_p), ('m', ctypes.c_void_p), ('v', ctypes.c_void_p), ('n_rows', ctypes.c_int64),
                ('rec_keys', ctypes.c_void_p), ('rec_grads', ctypes.c_void_p), ('n_seg', ctypes.c_int32),
                ('_pad', ctypes.c_int32), ('seg_len', ctypes.c_int64), ('key_seg_stride', ctypes.c_int64),
                ('grad_seg_stride', ctypes.c_int64), ('head', ctypes.c_void_p), ('next', ctypes.c_void_p),
                ('rec_row', ctypes.c_void_p), ('csr_off', ctypes.c_void_p), ('csr', ctypes.c_void_p),
                ('csr_pool', ctypes.c_void_p)]


class DpChannel(ctypes.Structure):
    _fields_ = [('peer_bases', ctypes.c_uint64 * 8), ('flag_off', ctypes.c_int64), ('epoch_dev', ctypes.c_void_p),
                ('seg_floats', ctypes.c_int64)]


class DpSync(ctypes.Structure):
    _fields_ = [('world', ctypes.c_int32), ('rank', ctypes.c_int32), ('n_wait', ctypes.c_int32), ('n_done', ctypes.c_int32),
                ('wait', DpChannel * 3), ('done', DpChannel * 3), ('loss_parts', ctypes.c_void_p),
                ('loss_stride', ctypes.c_int64), ('n_loss', ctypes.c_int32), ('flags', ctypes.c_int32),
                ('loss_out', ctypes.c_void_p)]


class LinkExtra(ctypes.Structure):
    _fields_ = [('epoch_ptrs_dev', ctypes.c_void_p), ('cursor_dev', ctypes.c_void_p), ('X_out', ctypes.c_void_p),
                ('sample_item_out', ctypes.c_void_p), ('Y_out', ctypes.c_void_p), ('stage_counter', ctypes.c_void_p),
                ('pf_user', ctypes.c_void_p * 3), ('pf_item', ctypes.c_void_p * 3), ('pf_feat', ctypes.c_void_p),
                ('pf_dense', ctypes.c_void_p * 4), ('pf_dense_bytes', ctypes.c_int64 * 4),
                ('sync', ctypes.POINTER(DpSync)), ('rec_row_user', ctypes.c_void_p), ('rec_row_item', ctypes.c_void_p)]


class BatchRef(ctypes.Structure):
    _fields_ = [('epoch_ptrs_dev', ctypes.c_void_p), ('cursor_dev', ctypes.c_void_p)]


class AdamTensor(ctypes.Structure):
    _fields_ = [('p', ctypes.c_void_p), ('m', ctypes.c_void_p), ('v', ctypes.c_void_p), ('n', ctypes.c_int64),
                ('g_parts', ctypes.c_void_p), ('n_parts', ctypes.c_int32), ('_pad', ctypes.c_int32),
                ('part_stride', ctypes.c_int64)]


_P = ctypes.c_void_p
_SIGNATURES = {
    # name: (restype, argtypes)   — one entry per symbol declared in include/dccf_b200.h
    'dccf_last_error': (ctypes.c_char_p, []),
    'dccf_abi_version': (ctypes.c_int, []),
    'dccf_noise_fill': (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_uint64,
                                       ctypes.c_uint64, ctypes.c_int64, _P]),
    'dccf_dropout_mask_fill': (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int32, ctypes.c_float, ctypes.c_uint64,
                                              ctypes.c_uint64, ctypes.c_int64, _P]),
    'dccf_score_fwd': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, _P, _P, ctypes.POINTER(Expo), _P, _P,
                                      ctypes.c_int64, ctypes.POINTER(Rng), _P, _P, _P, _P, _P, _P, _P]),
    'dccf_tc_operand_floats': (ctypes.c_int64, [ctypes.c_int32]),
    'dccf_tc_prepare': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'dccf_score_fwd_tc': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, _P, ctypes.POINTER(Expo), _P, _P,
                                         ctypes.c_int64, ctypes.POINTER(Rng), _P, _P, _P, _P, _P]),
    'dccf_score_gather': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, ctypes.POINTER(Expo), _P, _P, ctypes.c_int64,
                                         _P, _P, _P]),
    'dccf_bwd_splits': (ctypes.c_int32, [ctypes.c_int64]),
    'dccf_bpr_bwd': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, _P, _P, _P, _P, ctypes.c_int64,
                                    ctypes.POINTER(Rng), ctypes.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'dccf_train_w_image_floats': (ctypes.c_int64, [ctypes.c_int32]),
    'dccf_train_fwd_ksplits': (ctypes.c_int32, [ctypes.c_int64, ctypes.c_int32]),
    'dccf_train_bwd_splits': (ctypes.c_int32, [ctypes.c_int64, ctypes.c_int32]),
    'dccf_train_fwd_tc': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, _P, _P, ctypes.POINTER(Expo), _P, _P,
                                         ctypes.c_int64, ctypes.POINTER(Rng), _P, _P, _P, _P, _P, _P, _P, _P]),
    'dccf_train_bwd_tc': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, _P, _P, _P, _P, ctypes.c_int64,
                                         ctypes.POINTER(Rng), ctypes.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                         _P, _P]),
    'dccf_train_fused_smem_bytes': (ctypes.c_int64, [ctypes.c_int32, ctypes.c_int32, ctypes.c_int32]),
    'dccf_train_fwd_bwd_tc': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, _P, _P, _P, ctypes.POINTER(Expo), _P, _P, _P,
                                             ctypes.c_int64, ctypes.c_int64, ctypes.POINTER(Rng), ctypes.c_int32, _P, _P, _P,
                                             ctypes.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P,
                                             ctypes.POINTER(BatchRef), ctypes.c_int32, _P, _P]),
    'dccf_adam_sweep': (ctypes.c_int, [_P, _P, _P, ctypes.c_int64, _P, _P, ctypes.c_int64, _P, _P,
                                       ctypes.POINTER(Adam), _P]),
    'dccf_adam_sweep_seg': (ctypes.c_int, [_P, _P, _P, ctypes.c_int64, _P, _P, ctypes.c_int32, ctypes.c_int64,
                                           ctypes.c_int64, ctypes.c_int64, _P, _P, ctypes.POINTER(Adam), _P]),
    'dccf_sum_parts': (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, _P, _P]),
    'dccf_adam_dense': (ctypes.c_int, [_P, _P, _P, ctypes.c_int64, _P, ctypes.c_int32, ctypes.c_int64,
                                       ctypes.POINTER(Adam), _P]),
    'dccf_adam_step': (ctypes.c_int, [ctypes.POINTER(AdamTable), ctypes.c_int32, ctypes.POINTER(AdamTensor),
                                      ctypes.c_int32, ctypes.POINTER(Adam), _P]),
    'dccf_adam_blocks': (ctypes.c_int32, [ctypes.c_int32, _P, _P, ctypes.c_int32, _P, ctypes.c_int32, _P, _P]),
    'dccf_adam_link_ids': (ctypes.c_int, [ctypes.POINTER(Dims), _P, _P, ctypes.c_int64, ctypes.c_int32, ctypes.c_int64,
                                          ctypes.c_int32, _P, _P, _P, _P, ctypes.POINTER(Expo), _P, _P, _P, _P,
                                          ctypes.POINTER(LinkExtra), _P]),
    'dccf_adam_untouched': (ctypes.c_int, [ctypes.POINTER(AdamTable), ctypes.c_int32, ctypes.POINTER(Adam), ctypes.c_int32,
                                           _P]),
    'dccf_adam_csr_build': (ctypes.c_int, [ctypes.POINTER(AdamTable), ctypes.c_int32, _P]),
    'dccf_adam_touched': (ctypes.c_int, [ctypes.POINTER(AdamTable), ctypes.c_int32, ctypes.POINTER(AdamTensor),
                                         ctypes.c_int32, ctypes.POINTER(Adam), ctypes.c_int32, _P, ctypes.c_int32,
                                         ctypes.c_int32, _P, _P, _P, _P, ctypes.POINTER(DpSync), _P]),
    'dccf_train_prep_w_image': (ctypes.c_int, [_P, ctypes.c_int32, _P, _P]),
    'dccf_debug_timeline_train': (ctypes.c_int, [_P]),
    'dccf_debug_timeline_adam': (ctypes.c_int, [_P]),
    'dccf_debug_timeline_dp': (ctypes.c_int, [_P]),
    'dccf_stage_batch': (ctypes.c_int, [_P, _P, ctypes.c_int64, ctypes.c_int32, _P, _P, _P, _P]),
    'dccf_state_advance': (ctypes.c_int, [_P, _P, ctypes.c_uint64, _P]),
    'dccf_dp_push': (ctypes.c_int, [_P, ctypes.c_int64, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, _P, _P, _P]),
    'dccf_dp_push_fold': (ctypes.c_int, [_P, ctypes.c_int64, _P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, _P, _P,
                                         _P, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64,
                                         _P, ctypes.c_int32, ctypes.c_int64, ctypes.c_int64, ctypes.c_int64, _P]),
    'dccf_dp_wait': (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int32, ctypes.c_int64, _P, _P]),
    'dccf_dp_flag_floats': (ctypes.c_int64, []),
    'dccf_dp_done': (ctypes.c_int, [_P, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64, _P, _P]),
    'dccf_full_scores_splits': (ctypes.c_int32, [ctypes.c_int32, ctypes.c_int32]),
    'dccf_full_scores_ws_floats': (ctypes.c_int64, [ctypes.c_int32]),
    'dccf_full_scores': (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, _P, _P, _P, _P, _P, ctypes.c_float, _P,
                                        ctypes.c_int32, _P, _P, _P, _P, _P, _P, _P, _P]),
    'dccf_mf_step_ctas': (ctypes.c_int32, [ctypes.c_int64]),
    'dccf_mf_step': (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, _P, _P, _P, _P, _P, _P, ctypes.c_float, _P, _P,
                                    ctypes.c_int64, ctypes.c_int32, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    'dccf_mf_bias_grad': (ctypes.c_int, [ctypes.POINTER(AdamTable), ctypes.POINTER(AdamTable), _P, _P, _P, _P,
                                         ctypes.c_int32, ctypes.c_float, _P, _P]),
    'dccf_mf_scores': (ctypes.c_int, [ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(Expo), _P, _P, ctypes.c_int64, _P,
                                      _P, _P]),
    'dccf_sample_negatives': (ctypes.c_int, [_P, _P, _P, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32, ctypes.c_int64,
                                             ctypes.c_int64, _P, _P, _P, _P, _P]),
    'dccf_confounder_draw': (ctypes.c_int, [_P, _P, _P, ctypes.c_int64, ctypes.c_int64, _P]),
    'dccf_confounder_draw_dev': (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int64, _P, _P]),
    'dccf_rank_eval': (ctypes.c_int, [_P, _P, _P, _P, _P, ctypes.c_int64, ctypes.c_int32, _P, _P, _P, _P]),
    'dccf_rank_eval_ws_bytes': (ctypes.c_int64, [ctypes.c_int64]),
    'dccf_rank_eval_multi': (ctypes.c_int, [_P, _P, _P, _P, _P, ctypes.c_int64, ctypes.POINTER(ctypes.c_int32),
                                            ctypes.c_int32, _P, _P, _P, _P, _P, _P]),
    'dccf_topk_metrics': (ctypes.c_int, [_P, ctypes.c_int64, ctypes.c_int32, _P, _P, ctypes.POINTER(ctypes.c_int32),
                                         ctypes.c_int32, _P, _P, _P, _P, _P]),
}

_LIB = None


def exported_symbols():
    return sorted(_SIGNATURES)


def load(path=None):
    """dlopen the library and bind every declared symbol.  Raises DccfError when impossible."""
    global _LIB
    if _LIB is not None and path is None:
        return _LIB
    path = path or LIB_PATH
    if not os.path.exists(path):
        raise DccfError('%s not found: build it with `python -m dccf_b200.build` (the DCCF B200 path has no '
                        'CPU fallback)' % path)
    try:
        lib = ctypes.CDLL(path)
    except OSError as e:
        raise DccfError('cannot load %s: %s' % (path, e))
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            raise DccfError('%s does not export %s' % (path, name))
        fn.restype = res
        fn.argtypes = args
    if lib.dccf_abi_version() != ABI_VERSION:
        raise DccfError('ABI mismatch: library %d, binding %d — rebuild with `python -m dccf_b200.build --force`'
                        % (lib.dccf_abi_version(), ABI_VERSION))
    _LIB = lib
    return lib


def check(rc, what):
    if rc != 0:
        msg = load().dccf_last_error()
        raise DccfError('%s failed (%d): %s' % (what, rc, msg.decode() if msg else ''))


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise DccfError('expected a CUDA tensor, got device %s — the DCCF B200 kernels have no CPU path' % t.device)
    if not t.is_contiguous():
        raise DccfError('expected a contiguous tensor')
    return ctypes.c_void_p(t.data_ptr())


def stream_ptr():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
