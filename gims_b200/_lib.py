"""ctypes binding of libgims_b200.so (the C ABI of include/gims_b200.h).

The product path has no fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os

from .build import LIB_PATH

MAX_LAYERS = 64
MAX_KENC = 8
MAX_KPTS = 16384
MAX_BATCH = 4
STATUS_EDGE_OVERFLOW = 1
STATUS_SINKHORN_TIMEOUT = 2
STATUS_ERROR_MASK = 0xff
STATUS_SINKHORN_FAST = 0x100
STATUS_SINKHORN_EXACT = 0x200
GEMM_SIMT, GEMM_TC, GEMM_TC_F16, GEMM_BF16 = 0, 1, 2, 3
GEMM_MODES = {'simt': GEMM_SIMT, 'tf32': GEMM_TC, 'tc': GEMM_TC, 'f16': GEMM_TC_F16, 'bf16': GEMM_BF16}
STATUS_FP16_RANGE = 4
STATUS_KEYPOINT_OVERFLOW = 8
PROF = {'gemm': 1, 'attention': 2, 'sinkhorn': 3, 'score': 4, 'cosine': 5, 'sage_gather': 6}


class GimsError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [
        ('descriptor_dim', C.c_int),
        ('num_layers', C.c_int),
        ('layer_is_cross', C.c_int * MAX_LAYERS),
        ('kenc_num', C.c_int),
        ('kenc_dims', C.c_int * (MAX_KENC + 1)),
        ('sinkhorn_iterations', C.c_int),
        ('match_threshold', C.c_float),
    ]


class PairInputs(C.Structure):
    _fields_ = [
        ('kpts', C.c_void_p * 2),
        ('desc', C.c_void_p * 2),
        ('scores', C.c_void_p * 2),
        ('n', C.c_int * 2),
        ('desc_channel_major', C.c_int),
        ('img_w', C.c_float * 2),
        ('img_h', C.c_float * 2),
        ('radius', C.c_double),
        ('k_rank', C.c_longlong * 2),
        ('min_size', C.c_int),
        ('edge_cap', C.c_int),
        ('gemm_mode', C.c_int),
    ]


class PairOutputs(C.Structure):
    _fields_ = [
        ('n_kept_dev', C.c_void_p),
        ('kept_idx', C.c_void_p * 2),
        ('csr_indptr', C.c_void_p * 2),
        ('csr_indices', C.c_void_p * 2),
        ('n_edges_dev', C.c_void_p),
        ('n_comp_dev', C.c_void_p),
        ('thr_dev', C.c_void_p),
        ('kpts', C.c_void_p * 2),
        ('feat', C.c_void_p * 2),
        ('scores', C.c_void_p * 2),
        ('mdesc', C.c_void_p),
        ('matches', C.c_void_p * 2),
        ('mscores', C.c_void_p * 2),
        ('indices', C.c_void_p * 2),
        ('u', C.c_void_p),
        ('v', C.c_void_p),
        ('couplings', C.c_void_p),
        ('desc_gnn', C.c_void_p),
        ('desc_in', C.c_void_p),
        ('status_dev', C.c_void_p),
    ]


class NamedTensor(C.Structure):
    """gims_named_tensor (include/gims_b200.h)."""
    _fields_ = [('name', C.c_char_p), ('data', C.c_void_p), ('numel', C.c_int64)]


# name -> (restype, argtypes); every symbol include/gims_b200.h declares
SIGNATURES = {
    'gims_version': (C.c_int, []),
    'gims_last_error': (C.c_char_p, []),
    'gims_launch_count': (C.c_longlong, []),
    'gims_profile_begin': (C.c_int, [C.c_int, C.c_int]),
    'gims_profile_end': (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int)]),
    'gims_model_create': (C.c_int, [C.POINTER(Config), C.c_void_p, C.POINTER(C.c_int64), C.c_int,
                                    C.POINTER(C.c_void_p)]),
    'gims_model_destroy': (None, [C.c_void_p]),
    'gims_packed_blob_count': (C.c_int, [C.POINTER(Config)]),
    'gims_pack_weights_floats': (C.c_size_t, [C.POINTER(Config)]),
    'gims_pack_weights': (C.c_int, [C.POINTER(Config), C.POINTER(NamedTensor), C.c_int, C.c_void_p, C.c_size_t,
                                    C.POINTER(C.c_int64), C.c_int]),
    'gims_agc_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'gims_agc_build': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_longlong,
                                 C.c_int, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p, C.c_void_p]),
    'gims_sage_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    'gims_kenc_forward': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_float, C.c_float, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    'gims_attn_scratch_floats': (C.c_size_t, [C.c_int]),
    'gims_attn_layer_forward': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    'gims_final_scores': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p]),
    'gims_set_gemm_mode': (C.c_int, [C.c_int]),
    'gims_get_gemm_mode': (C.c_int, []),
    'gims_linear': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                              C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'gims_debug_attention_trace': (C.c_int, [C.c_void_p]),
    'gims_debug_gemm_trace': (C.c_int, [C.c_void_p]),
    'gims_debug_sinkhorn_trace': (C.c_int, [C.c_void_p]),
    'gims_split_tf32': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    'gims_sinkhorn_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'gims_couplings_ld': (C.c_int, [C.c_int]),
    'gims_sinkhorn_match': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_float, C.c_void_p,
                                      C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'gims_sinkhorn_max_columns': (C.c_int, []),
    'gims_extract_patches': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                       C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    'gims_debug_bicubic_table': (C.c_int, [C.c_void_p]),
    'gims_pyramid_layout': (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.c_void_p, C.c_void_p, C.c_void_p]),
    'gims_pyramid_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    'gims_gaussian_pyramid': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.c_void_p]),
    'gims_debug_gaussian_kernel': (C.c_int, [C.c_double, C.c_void_p, C.POINTER(C.c_int)]),
    'gims_sift_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int, C.c_int, C.c_int]),
    'gims_sift_detect': (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_size_t,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    'gims_gt_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'gims_gt_matches': (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_float, C.c_int, C.c_void_p,
                                  C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    'gims_match_counts': (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    'gims_homography_workspace_bytes': (C.c_size_t, [C.c_int, C.c_int]),
    'gims_find_homographies': (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_int, C.c_double,
                                         C.c_ulonglong, C.c_void_p, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    'gims_pair_workspace_bytes': (C.c_size_t, [C.c_void_p, C.c_int, C.c_int, C.c_int]),
    'gims_forward_pair': (C.c_int, [C.c_void_p, C.POINTER(PairInputs), C.POINTER(PairOutputs), C.c_void_p,
                                    C.c_size_t, C.c_void_p]),
    'gims_batch_workspace_bytes': (C.c_size_t, [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_int]),
    'gims_forward_pairs': (C.c_int, [C.c_void_p, C.c_int, C.POINTER(PairInputs), C.POINTER(PairOutputs), C.c_void_p,
                                     C.c_size_t, C.c_void_p]),
}

_LIB = None


def lib():
    """Load libgims_b200.so (once).  Raises GimsError if it has not been built."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = os.environ.get('GIMS_B200_LIB', LIB_PATH)
    if not os.path.exists(path):
        raise GimsError('libgims_b200.so not found at %s — run `python -m gims_b200.build` '
                        '(there is no CPU/PyTorch fallback for this path)' % path)
    handle = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)     # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    mode = os.environ.get('GIMS_GEMM_MODE')
    if mode:
        handle.gims_set_gemm_mode(GEMM_MODES[mode.lower()])
    _LIB = handle
    return _LIB


def check(rc, what):
    if rc != 0:
        msg = lib().gims_last_error()
        raise GimsError('%s failed (%d): %s' % (what, rc, msg.decode() if msg else ''))


def ptr(t):
    """Device/host pointer of a contiguous torch tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), 'tensor passed to the C ABI must be contiguous'
    return C.c_void_p(t.data_ptr())
