"""ctypes binding of libmeshdiff_b200.so (the C ABI declared in include/meshdiff_b200.h).

There is deliberately no fallback: if the library is missing or a call fails, an exception is raised.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libmeshdiff_b200.so")

_lib = None


class NativeError(RuntimeError):
    pass


class UNetConfigC(ctypes.Structure):
    _fields_ = [
        ("image_size", ctypes.c_int),
        ("nf", ctypes.c_int),
        ("n_levels", ctypes.c_int),
        ("ch_mult", ctypes.c_int * 8),
        ("num_res_blocks", ctypes.c_int),
        ("level0_blocks", ctypes.c_int),
        ("n_attn", ctypes.c_int),
        ("attn_resolutions", ctypes.c_int * 4),
        ("num_channels", ctypes.c_int),
        ("stem_ksize", ctypes.c_int),
        ("use_pos_bias", ctypes.c_int),
        ("max_batch", ctypes.c_int),
        ("precision", ctypes.c_int),
        ("training", ctypes.c_int),
    ]


class SamplerCondC(ctypes.Structure):
    """mdb_sampler_cond (include/meshdiff_b200.h)."""
    _fields_ = [
        ("partial", ctypes.c_void_p), ("partial_bstride", ctypes.c_longlong),
        ("partial_mask", ctypes.c_void_p), ("mask_bstride", ctypes.c_longlong),
        ("channel", ctypes.c_int), ("mean_coef", ctypes.c_float), ("std", ctypes.c_float),
        ("noise", ctypes.c_void_p),
    ]


# name -> (restype, argtypes); the symbol list is checked against the header by tests/test_abi.py
_vp, _i, _ll, _f, _u64, _d = ctypes.c_void_p, ctypes.c_int, ctypes.c_longlong, ctypes.c_float, ctypes.c_ulonglong, ctypes.c_double
SIGNATURES = {
    "mdb_last_error": (ctypes.c_char_p, []),
    "mdb_version": (_i, []),
    "mdb_unet_create": (_i, [ctypes.POINTER(UNetConfigC), ctypes.POINTER(_vp)]),
    "mdb_unet_create_dry": (_i, [ctypes.POINTER(UNetConfigC), ctypes.POINTER(_vp)]),
    "mdb_unet_destroy": (None, [_vp]),
    "mdb_unet_num_params": (_i, [_vp]),
    "mdb_unet_param_info": (_i, [_vp, _i, ctypes.POINTER(ctypes.c_char_p), ctypes.POINTER(_ll), ctypes.POINTER(_i), ctypes.POINTER(_ll)]),
    "mdb_unet_set_param": (_i, [_vp, ctypes.c_char_p, _vp, _ll, _i, _vp]),
    "mdb_unet_get_param": (_i, [_vp, ctypes.c_char_p, _vp, _ll, _i, _vp]),
    "mdb_unet_commit": (_i, [_vp, _vp]),
    "mdb_unet_set_params": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "mdb_unet_forward": (_i, [_vp, _vp, _vp, _vp, _i, _vp]),
    "mdb_unet_info": (_i, [_vp, ctypes.POINTER(_d), ctypes.POINTER(_ll), ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    "mdb_unet_profile": (_i, [_vp, _vp, _vp, _vp, _i, _vp, ctypes.c_char_p, _i, ctypes.POINTER(_f), _i, ctypes.POINTER(_i)]),
    "mdb_unet_set_dropout": (_i, [_vp, _f, _u64]),
    "mdb_unet_backward": (_i, [_vp, _vp, _vp, _ll, _i, _i, _vp]),
    "mdb_unet_grad_offset": (_i, [_vp, ctypes.c_char_p, ctypes.POINTER(_ll)]),
    "mdb_unet_grad_ready": (_i, [_vp, ctypes.c_char_p, ctypes.POINTER(_i)]),
    "mdb_unet_backward_marked": (_i, [_vp, _vp, _vp, _ll, _i, _i, ctypes.POINTER(_i), ctypes.POINTER(_vp), _i, _vp]),
    "mdb_unet_debug_stats": (_i, [_vp, _vp, _ll, ctypes.POINTER(_ll)]),
    "mdb_unet_train_info": (_i, [_vp, ctypes.POINTER(_d), ctypes.POINTER(_i), ctypes.POINTER(_ll)]),
    "mdb_unet_profile_backward": (_i, [_vp, _vp, _vp, _i, _vp, ctypes.c_char_p, _i, ctypes.POINTER(_f), _i, ctypes.POINTER(_i)]),
    "mdb_fingerprint": (_i, [_vp, _vp, _i, _vp, _vp]),
    "mdb_sampler_update": (_i, [_vp, _vp, _vp, _vp, _vp, _f, _f, _ll, _i, _i, _u64, _u64, ctypes.POINTER(SamplerCondC), _vp]),
    "mdb_sampler_run": (_i, [_vp, _vp, _vp, _vp, ctypes.POINTER(_f), ctypes.POINTER(_f), ctypes.POINTER(_f), _i, _i, _u64, _vp, _vp,
                             _i, ctypes.POINTER(SamplerCondC), ctypes.POINTER(_f), ctypes.POINTER(_f), _i, _vp]),
    "mdb_ddpm_loss": (_i, [_vp, _vp, _vp, _d, _vp, _vp, _vp, _i, _i, _ll, _vp]),
    "mdb_ddpm_perturb": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _ll, _vp]),
    "mdb_chunk_elems": (_i, []),
    "mdb_grad_clip_coef": (_i, [_vp, _vp, _vp, _i, _f, _vp, _vp, _vp, _vp]),
    "mdb_adam_ema_step": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _f, _f, _f, _f, _f, _i, _vp, _f, _vp]),
    "mdb_ema_update": (_i, [_vp, _vp, _vp, _vp, _i, _f, _vp]),
    "mdb_allreduce_grads": (_i, [_vp, _vp, _ll, _i, _vp]),
    "mdb_conv3d": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _vp]),
    "mdb_groupnorm_act": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _i, _i, _vp]),
    "mdb_conv3d_backward": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _i, _ll, _ll, _i, _i, _i, _vp, _vp]),
    "mdb_groupnorm_act_backward": (_i, [_vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _ll, _i, _f, _u64,
                                        _i, _i, _vp]),
    "mdb_conv3d_dgrad_gn_backward": (_i, [_vp, _vp, _i, _i, _i, _i, _vp, _i, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                          _i, _f, _u64, _i, _vp]),
    "mdb_colsum": (_i, [_vp, _ll, _i, _i, _ll, _vp, _ll, _vp, _i, _vp, _ll, _i, _vp]),
    "mdb_downsum2x": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "mdb_batch_sum": (_i, [_vp, _vp, _i, _ll, _i, _i, _vp]),
    "mdb_zero_stuff2x": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "mdb_softmax_bwd_rows": (_i, [_vp, _vp, _ll, _i, _i, _vp]),
    "mdb_transpose_vc": (_i, [_vp, _ll, _i, _vp, _i, _i, _i, _i, _vp]),
    "mdb_im2col": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "mdb_marching_tets_prepare": (_i, [_vp, _i, _i, _i, ctypes.POINTER(_vp)]),
    "mdb_marching_tets_destroy": (None, [_vp]),
    "mdb_marching_tets_info": (_i, [_vp, ctypes.POINTER(_i), ctypes.POINTER(_i)]),
    "mdb_marching_tets_uvs": (_i, [_vp, _vp, _vp]),
    "mdb_marching_tets_count": (_i, [_vp, _vp, _i, ctypes.POINTER(_i), _vp]),
    "mdb_mesh_auto_normals": (_i, [_vp, _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "mdb_mesh_compute_tangents": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "mdb_marching_tets_extract": (_i, [_vp, _vp, _ll, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "mdb_marching_tets_vertex_ids": (_i, [_vp, _i, _vp, _vp]),
    "mdb_marching_tets_backward": (_i, [_vp, _vp, _ll, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
}


def lib():
    """Loads the shared library (building it in-tree first if the sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise NativeError("libmeshdiff_b200.so is missing and could not be built; there is no fallback path")
    L = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(code):
    if code != 0:
        raise NativeError(lib().mdb_last_error().decode())


def ptr(t):
    """Raw device/host pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


def current_stream():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
