"""ctypes binding of liboflib_b200.so (include/oflib_b200.h). No fallback: if the CUDA library is missing or a call
fails, an exception is raised -- the product path never routes through CPU code."""
import ctypes as C
import os

from . import build as _build

# enums of include/oflib_b200.h
U8, I16, U16, F32, F64, I32, I64 = 0, 1, 2, 3, 4, 5, 6
ARITH_NATIVE, ARITH_RINT = 0, 1
RULE_STRICT, RULE_GT_HALF, RULE_GE_HALF = 0, 1, 2
OP_ADD, OP_SUB, OP_MUL, OP_DIV, OP_POW = 0, 1, 2, 3, 4
PAD_CONSTANT, PAD_EDGE, PAD_SYMMETRIC = 0, 1, 2
PAD_MODES = {'constant': PAD_CONSTANT, 'edge': PAD_EDGE, 'symmetric': PAD_SYMMETRIC}
FIT_LMS, FIT_RANSAC, FIT_LMEDS = 0, 1, 2
FIT_METHODS = {'lms': FIT_LMS, 'ransac': FIT_RANSAC, 'lmeds': FIT_LMEDS}


class OflibCudaError(RuntimeError):
    """A call into liboflib_b200.so failed (bad argument, CUDA error, unsupported configuration)."""


_vp, _i, _f, _d, _sz = C.c_void_p, C.c_int, C.c_float, C.c_double, C.c_size_t

_SIGNATURES = {
    'ofk_last_error': (C.c_char_p, []),
    'ofk_version': (_i, []),
    'ofk_warp_t': (_i, [_vp, _i, _i, _i, _vp, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    'ofk_warp_t_ex': (_i, [_vp, _i, _i, _i, _vp, _f, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i,
                           _vp]),
    'ofk_combine3': (_i, [_vp, _vp, _vp, _vp, _i, _f, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'ofk_valid_geom_t': (_i, [_vp, _f, _vp, _vp, _i, _i, _i, _vp]),
    'ofk_from_matrix': (_i, [_vp, _i, _f, _vp, _i, _i, _i, _vp]),
    'ofk_addsub': (_i, [_i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'ofk_scale': (_i, [_i, _vp, _d, _d, _i, _vp, _sz, _vp]),
    'ofk_scale_array': (_i, [_i, _vp, _vp, _i, _vp, _sz, _vp]),
    'ofk_nonzero_flags': (_i, [_vp, _vp, _f, _vp, _i, _i, _i, _vp]),
    'ofk_check_finite': (_i, [_vp, _sz, _vp, _vp]),
    'ofk_pad': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    'ofk_mask_and': (_i, [_vp, _vp, _vp, _sz, _vp]),
    'ofk_crop': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _vp]),
    'ofk_extent': (_i, [_vp, _vp, _f, _f, _vp, _i, _i, _i, _vp]),
    'ofk_resize_flow': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _d, _d, _vp]),
    'ofk_greater': (_i, [_vp, _f, _vp, _sz, _vp]),
    'ofk_decode_kitti': (_i, [_vp, _vp, _vp, _sz, _vp]),
    'ofk_decode_sintel_mask': (_i, [_vp, _vp, _sz, _vp]),
    'ofk_vis_magnitude': (_i, [_vp, _f, _vp, _vp, _sz, _vp]),
    'ofk_kth_smallest_workspace': (_sz, [_i]),
    'ofk_kth_smallest': (_i, [_vp, _sz, _vp, _i, _vp, _vp, _sz, _vp]),
    'ofk_visualise': (_i, [_vp, _vp, _f, _i, _i, _i, _f, _vp, _i, _i, _vp]),
    'ofk_visualise_batch_workspace': (_sz, [_i, _i, _i]),
    'ofk_visualise_batch': (_i, [_vp, _vp, _f, _i, _i, _i, _f, _vp, _i, _i, _i, _vp, _sz, _vp]),
    'ofk_track_bilinear': (_i, [_vp, _vp, _sz, _i, _i, _vp, _vp, _vp]),
    'ofk_track': (_i, [_vp, _vp, _i, _i, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'ofk_fit_matrix_workspace': (_sz, [_i, _i, _i, _i, _i, _i]),
    'ofk_fit_matrix': (_i, [_vp, _vp, _i, _i, _i, _i, _f, _i, _vp, _vp, _vp, _i, _i, _i, _vp, _sz, _vp]),
    'ofk_accumulate_workspace': (_sz, [_i, _i]),
    'ofk_accumulate': (_i, [_vp, _vp, _i, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'ofk_accumulate_fold_workspace': (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    'ofk_accumulate_fold': (_i, [_vp, _vp, _i, _i, _f, _i, _i, _i, _i, _i, _vp, _vp, _vp, _sz, _vp]),
    'ofk_consistency': (_i, [_vp, _vp, _vp, _vp, _i, _f, _f, _vp, _vp, _i, _i, _i, _vp]),
    'ofk_evaluate_workspace': (_sz, [_i, _i, _i]),
    'ofk_evaluate': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _sz, _vp]),
    'ofk_points_inside_area':(_i, [_vp, _sz, _i, _i, _vp, _vp]),
    'ofk_forward_s_workspace': (_sz, [_i, _i, _i]),
    'ofk_forward_s': (_i, [_vp, _i, _vp, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    'ofk_cast': (_i, [_vp, _i, _vp, _i, _sz, _vp]),
    'ofk_forward_s_set_flip_tol': (_i, [C.c_double]),
    'ofk_forward_s_set_disable': (_i, [C.c_int]),
    'ofk_forward_s_ex': (_i, [_vp, _i, _vp, _f, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    'ofk_combine12_workspace': (_sz, [_i, _i, _i, _i, _i]),
    'ofk_combine12': (_i, [_i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _sz, _vp]),
    'ofk_combine2_t': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'ofk_mesh_sample': (_i, [_vp, _f, _i, _vp, _i, _vp, _vp, _f, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'ofh_warp_t': (_i, [_vp, _i, _i, _i, _vp, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i]),
    'ofh_combine3': (_i, [_vp, _vp, _vp, _vp, _i, _f, _vp, _vp, _vp, _i, _i, _i, _i]),
    'ofh_apply_combine3': (_i, [_vp, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _f, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i]),
    'ofh_visualise': (_i, [_vp, _vp, _f, _i, _i, _i, _f, _vp, _i, _i, _i, _i]),
    'ofh_evaluate': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i]),
    'ofh_release': (_i, []),
    'ofk_rt_device_count': (_i, [C.POINTER(_i)]),
    'ofk_rt_set_device': (_i, [_i]),
    'ofk_rt_get_device': (_i, [C.POINTER(_i)]),
    'ofk_rt_device_info': (_i, [_i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_sz), C.POINTER(_sz)]),
    'ofk_rt_malloc': (_i, [C.POINTER(_vp), _sz, _vp]),
    'ofk_rt_free': (_i, [_vp, _vp]),
    'ofk_rt_host_alloc': (_i, [C.POINTER(_vp), _sz]),
    'ofk_rt_host_free': (_i, [_vp]),
    'ofk_rt_host_register': (_i, [_vp, _sz]),
    'ofk_rt_host_unregister': (_i, [_vp]),
    'ofk_rt_memcpy_h2d': (_i, [_vp, _vp, _sz, _vp]),
    'ofk_rt_memcpy_d2h': (_i, [_vp, _vp, _sz, _vp]),
    'ofk_rt_memcpy_d2d': (_i, [_vp, _vp, _sz, _vp]),
    'ofk_rt_memset': (_i, [_vp, _i, _sz, _vp]),
    'ofk_rt_stream_create': (_i, [C.POINTER(_vp)]),
    'ofk_rt_stream_destroy': (_i, [_vp]),
    'ofk_rt_stream_sync': (_i, [_vp]),
    'ofk_rt_device_sync': (_i, []),
    'ofk_rt_event_create': (_i, [C.POINTER(_vp)]),
    'ofk_rt_event_destroy': (_i, [_vp]),
    'ofk_rt_event_record': (_i, [_vp, _vp]),
    'ofk_rt_stream_wait_event': (_i, [_vp, _vp]),
    'ofk_rt_event_sync': (_i, [_vp]),
    'ofk_rt_event_elapsed_ms': (_i, [_vp, _vp, C.POINTER(_f)]),
    'ofk_rt_launch_count': (C.c_ulonglong, []),
    'ofk_rt_path_count': (C.c_ulonglong, [C.c_int]),
}

_NO_CHECK = {'ofk_last_error', 'ofk_version', 'ofk_forward_s_workspace', 'ofk_combine12_workspace', 'ofk_kth_smallest_workspace',
             'ofk_visualise_batch_workspace', 'ofk_fit_matrix_workspace', 'ofk_accumulate_workspace',
             'ofk_accumulate_fold_workspace', 'ofk_evaluate_workspace', 'ofk_rt_launch_count', 'ofk_rt_path_count'}

_lib = None


def symbols():
    """Names of every entry point the header declares (used by the symbol-export test)."""
    return sorted(_SIGNATURES)


def library_path():
    """The in-tree library; OFK_LIB_PATH names another build of it (A/B measurements of two builds inside one job)."""
    return os.environ.get('OFK_LIB_PATH') or _build.lib_path()


def load():
    """Load the shared library (once). Raises ImportError with build instructions if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = library_path()
    if not os.path.exists(path):
        raise ImportError(
            "oflibnumpy_b200: the CUDA library {} is missing. Build it with `python -m oflibnumpy_b200.build` "
            "(needs nvcc); there is no CPU fallback.".format(path))
    lib = C.CDLL(path)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here means header and library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().ofk_last_error().decode('utf-8', 'replace')


def call(name, *args):
    """Call an entry point and raise OflibCudaError on a non-zero return code."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if name in _NO_CHECK:
        return rc
    if rc != 0:
        raise OflibCudaError("{} failed (code {}): {}".format(name, rc, last_error()))
    return rc
