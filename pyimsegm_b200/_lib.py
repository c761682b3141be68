"""
ctypes binding of ``libimsegm_b200.so`` (the C-ABI declared in ``include/imsegm_b200.h``).

There is NO fallback: if the shared library is missing or a CUDA device is absent the calls raise.
torch is used only for device memory (tensors as containers) and streams.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libimsegm_b200.so')

_lib = None

ISB_OK, ISB_ERR_ARG, ISB_ERR_CUDA, ISB_ERR_CAPACITY, ISB_ERR_UNSUPPORTED = 0, -1, -2, -3, -4
DTYPE_CODES = {'uint8': 0, 'uint16': 1, 'float32': 2, 'float64': 3}

_vp, _i, _d, _sz, _ll = C.c_void_p, C.c_int, C.c_double, C.c_size_t, C.c_longlong



class SlicBand(C.Structure):
    """isb_slic_band_t of include/imsegm_b200.h"""
    _fields_ = [('slab_rows', C.c_int32), ('width', C.c_int32), ('image_rows', C.c_int32), ('y_off', C.c_int32),
                ('own_lo', C.c_int32), ('own_hi', C.c_int32), ('halo', C.c_int32),
                ('n_seeds', C.c_int32), ('step_y', C.c_int32), ('step_x', C.c_int32), ('slic_zero', C.c_int32),
                ('step', C.c_double), ('lab_slab', C.c_void_p), ('plane_stride', C.c_size_t), ('seeds_yx', C.c_void_p),
                ('labels_slab', C.c_void_p), ('ws', C.c_void_p), ('ws_bytes', C.c_size_t)]


_bp = C.POINTER(SlicBand)

#: every symbol declared in include/imsegm_b200.h: name -> (restype, argtypes)
SIGNATURES = {
    'isb_last_error': (C.c_char_p, []),
    'isb_abi_version': (_i, []),
    'isb_launch_count': (_ll, []),
    'isb_note_graph_replay': (_i, [_ll]),
    'isb_profile_enable': (_i, [_i]),
    'isb_profile_stage_count': (_i, []),
    'isb_profile_stage_name': (C.c_char_p, [_i]),
    'isb_profile_collect': (_i, [C.POINTER(_d), C.POINTER(_ll)]),
    'isb_slic_prepare': (_i, [_vp, _i, _i, _i, _i, C.POINTER(_d), _i, _d, _i, _vp, _vp, _vp]),
    'isb_image_minmax': (_i, [_vp, _i, _ll, _vp, _vp]),
    'isb_slic_band_begin': (_i, [_bp, _vp]),
    'isb_slic_band_assign': (_i, [_bp, _vp]),
    'isb_slic_band_update': (_i, [_bp, _vp, _vp]),
    'isb_slic_band_import': (_i, [_bp, _vp, _vp, _vp]),
    'isb_slic_band_finalize': (_i, [_bp, _vp, _vp]),
    'isb_segment_stats_accumulate': (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _vp, _vp]),
    'isb_segment_stats_deviation': (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    'isb_segment_stats_finish': (_i, [_i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    'isb_slic_kmeans_workspace_bytes': (_sz, [_i, _i, _i, _i, _i]),
    'isb_slic_kmeans': (_i, [_vp, _i, _i, _vp, _i, _i, _i, _d, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'isb_slic3d_prepare': (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _i, _d, _vp, _vp, _vp]),
    'isb_slic3d_kmeans_workspace_bytes': (_sz, [_i, _i, _i, _i]),
    'isb_slic3d_kmeans': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _i, _d, C.POINTER(_d), _i, _vp, _vp, _sz, _vp]),
    'isb_connectivity3d_workspace_bytes': (_sz, [_i, _i, _i, _i]),
    'isb_enforce_connectivity3d': (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'isb_connectivity_workspace_bytes': (_sz, [_i, _i]),
    'isb_enforce_connectivity': (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'isb_segment_stats_workspace_bytes': (_sz, [_i]),
    'isb_segment_stats_2d': (_i, [_vp, _i, _vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'isb_adjacency_workspace_bytes': (_sz, [_i, _i]),
    'isb_adjacency_edges': (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _vp, _sz, _vp]),
    'isb_adjacency_edges_3d': (_i, [_vp, _i, _i, _i, _i, _vp, _i, _vp, _vp, _sz, _vp]),
    'isb_centroids_3d': (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    'isb_gc_energies_workspace_bytes': (_sz, [_i, _i, _i]),
    'isb_gc_energies': (_i, [_vp, _i, _vp, _i, _vp, _i, _vp, _vp, _i, _i, _d, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    'isb_alpha_expansion_workspace_bytes': (_sz, [_i, _i, _i]),
    'isb_alpha_expansion': (_i, [_i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _sz, _vp]),
    'isb_gmm_workspace_bytes': (_sz, [_i, _i, _i, _i]),
    'isb_gmm_params_len': (_i, [_i, _i]),
    'isb_gmm_fit_predict': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _d, _d, _i, C.c_ulonglong, _vp, _vp, _vp, _vp, _sz, _vp]),
    'isb_gmm_model_len': (_i, [_i, _i]),
    'isb_gmm_predict_workspace_bytes': (_sz, [_i, _i, _i]),
    'isb_gmm_predict': (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp, _sz, _vp]),
    'isb_lm_workspace_bytes':(_sz, [_i, _i, _i, _i]),
    'isb_lm_acc_doubles': (_sz, [_i, _i]),
    'isb_lm_texture_accumulate': (_i, [_vp, _i, _vp, _i, _i, _i, _i, _i, _vp, _i, C.POINTER(_d), _vp, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'isb_lm_texture_finish': (_i, [_i, _i, _i, _vp, _vp, _vp, _i, _i, _vp]),
    'isb_lm_texture': (_i, [_vp, _i, _vp, _i, _i, _i, _vp, _i, C.POINTER(_d), _vp, _i, _i, _i, _i, _vp, _i, _i, _vp, _sz, _vp]),
    'isb_umma_selftest': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    'isb_umma_rate': (_i, [_i, _i, _i, _i, _vp, _vp]),
    'isb_fp64_latency': (_i, [_i, _vp, _vp]),
    'isb_fill_i32': (_i, [_vp, _ll, _i, _vp]),
    'isb_combine': (_i, [_vp, _vp, _ll, _i, _vp]),
    'isb_gray_stats_workspace_bytes': (_sz, [_i]),
    'isb_gray_stats': (_i, [_vp, _i, _vp, _ll, _i, _i, _vp, _i, _i, _vp, _sz, _vp]),
    'isb_label_hist_2d': (_i, [_vp, _vp, _i, _i, _i, _vp, _vp]),
    'isb_ray_features_2d': (_i, [_vp, _i, _i, _vp, _i, _vp, _vp, _i, _i, _vp, _vp]),
    'isb_filter_response_2d': (_i, [_vp, _i, _i, _i, _vp, _i, _i, _i, _vp, _vp]),
    'isb_gaussian_filter_2d': (_i, [_vp, _i, _i, _i, _vp, _i, _vp, _vp, _vp]),
    'isb_disc_label_hist': (_i, [_vp, _vp, _i, _i, _vp, _i, _vp, _i, _vp, _i, _i, _i, _vp, _vp, _vp]),
    'isb_region_label_hist': (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    'isb_gather': (_i, [_vp, _ll, _vp, _vp, _i, _vp, _vp, _vp]),
    'isb_segment_median_workspace_bytes': (_sz, [_ll, _i]),
    'isb_segment_median': (_i, [_vp, _i, _vp, _ll, _i, _i, _vp, _vp, _sz, _vp]),
    'isb_binary_opening_disk': (_i, [_vp, _i, _i, _i, _vp, _vp, _vp]),
}


class NativeLibraryError(RuntimeError):
    pass


def lib():
    """load the CUDA extension; raises (never falls back) when it has not been built"""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise NativeLibraryError(
                'pyimsegm_b200: %s is missing -- build it with `python -m pyimsegm_b200.build` '
                '(there is no CPU fallback)' % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError here = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status):
    if status != ISB_OK:
        msg = lib().isb_last_error().decode(errors='replace')
        if status == ISB_ERR_ARG:
            raise ValueError('imsegm_b200: ' + msg)
        if status == ISB_ERR_UNSUPPORTED:
            raise NotImplementedError('imsegm_b200: ' + msg)
        raise RuntimeError('imsegm_b200 (status %d): %s' % (status, msg))


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise NativeLibraryError('pyimsegm_b200 needs a CUDA device (B200 / sm_100a); there is no CPU fallback')
    return torch


def ptr(t):
    """device pointer of a torch tensor (or None)"""
    return None if t is None else C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
