"""ctypes binding of the C-ABI library `lib/libsis_b200.so` (declared in include/sis_b200.h).

The library is the product's only compute path: there is no CPU or PyTorch fallback.  If the shared object is
missing, `load()` raises and every op fails loudly.
"""
import ctypes
import os
from ctypes import (POINTER, Structure, c_char_p, c_double, c_float, c_int, c_int64, c_uint8, c_uint32, c_uint64, c_void_p)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libsis_b200.so')

SIS_F32, SIS_F16, SIS_F64 = 0, 1, 2
PRECISION_FP32, PRECISION_BF16X3 = 0, 1


class LabelJob(Structure):
    """`sis_label_job` (include/sis_b200.h)."""
    _fields_ = [
        ('activation_idx', c_int),
        ('d_centroids', c_void_p), ('k', c_int),
        ('d_cluster_class_bits', c_void_p), ('n_class', c_int), ('image_size', c_int),
        ('d_ids_u8', c_void_p), ('d_ids_i64', c_void_p), ('d_masks', c_void_p), ('d_margin', c_void_p), ('d_hist', c_void_p),
    ]


class KmeansFit(Structure):
    """`sis_kmeans_fit` (include/sis_b200.h)."""
    _fields_ = [
        ('d_points', c_void_p), ('n', c_int64), ('channels', c_int),
        ('k', c_int), ('d_centers', c_void_p), ('d_counts', c_void_p),
        ('d_state', c_void_p),
    ]


class ForwardArgs(Structure):
    """`sis_forward_args` (include/sis_b200.h)."""
    _fields_ = [
        ('batch', c_int),
        ('n_styles', c_int),
        ('d_styles', c_void_p * 2),
        ('input_is_latent', c_int),
        ('styles_are_wplus', c_int),
        ('inject_index', c_int),
        ('truncation', c_float),
        ('d_truncation_latent', c_void_p),
        ('truncation_latent_rows', c_int),
        ('d_noise', POINTER(c_void_p)),
        ('noise_batch_stride', POINTER(c_int64)),
        ('d_image', c_void_p),
        ('d_latent_out', c_void_p),
        ('d_activations', POINTER(c_void_p)),
        ('precision', c_int),
        ('n_label_jobs', c_int),
        ('label_jobs', POINTER(LabelJob)),
    ]


_SIGNATURES = {
    'sis_last_error': (c_char_p, []),
    'sis_version': (c_int, []),
    'sis_launch_count': (c_uint64, []),
    'sis_watchdog_code': (c_uint32, []),
    'sis_watchdog_clear': (None, []),
    'sis_profile_enable': (c_int, [c_int]),
    'sis_profile_collect': (c_int, [POINTER(ctypes.c_double), POINTER(c_uint64), c_int]),
    'sis_fused_bias_act': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int64, c_int64, c_int64, c_int, c_int,
                                   c_float, c_float, c_void_p]),
    'sis_upfirdn2d_out_size': (c_int, [c_int] * 6),
    'sis_upfirdn2d': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int64] + [c_int] * 13 + [c_void_p]),
    'sis_generator_create': (c_int, [c_int, c_int, c_int, c_int, POINTER(c_void_p)]),
    'sis_generator_create_swagan': (c_int, [c_int, c_int, c_int, c_int, POINTER(c_void_p)]),
    'sis_generator_destroy': (c_int, [c_void_p]),
    'sis_generator_set_param': (c_int, [c_void_p, c_char_p, c_void_p, c_int64]),
    'sis_generator_prepare': (c_int, [c_void_p, c_void_p]),
    'sis_generator_n_latent': (c_int, [c_void_p]),
    'sis_generator_num_layers': (c_int, [c_void_p]),
    'sis_generator_activation_shape': (c_int, [c_void_p, c_int, POINTER(c_int), POINTER(c_int)]),
    'sis_generator_style': (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    'sis_generator_forward': (c_int, [c_void_p, POINTER(ForwardArgs), c_void_p]),
    'sis_generator_check': (c_int, [c_void_p, c_void_p]),
    'sis_modulated_conv2d': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_int,
                                     c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    'sis_to_rgb': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p,
                           c_void_p, c_void_p]),
    'sis_wavelet_to_rgb': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                   c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    'sis_equal_linear': (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int, c_float, c_int, c_void_p, c_void_p]),
    'sis_pixel_norm': (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p]),
    'sis_noise_injection': (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'sis_label_assign': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_int,
                                 c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    'sis_class_masks_from_ids': (c_int, [c_void_p, c_int64, c_void_p, c_int, c_int, c_void_p, c_void_p]),
    'sis_nearest_resize_u8': (c_int, [c_void_p, c_int64, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    'sis_or_u8': (c_int, [c_void_p, c_void_p, c_int64, c_void_p]),
    'sis_make_image_u8': (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    'sis_contour_stage_workspace_bytes': (c_int, [c_int, c_int, c_int, c_int, c_int, POINTER(c_int64)]),
    'sis_contour_stage': (c_int, [POINTER(c_void_p), POINTER(c_void_p), c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_double,
                                  c_char_p, POINTER(c_int), c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_void_p]),
    'sis_png_write_pairs': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, POINTER(c_char_p), c_int, c_int, c_int]),
    'sis_pixel_ensemble_create': (c_int, [POINTER(c_void_p), c_int, c_int, c_int]),
    'sis_pixel_ensemble_destroy': (None, [c_void_p]),
    'sis_pixel_ensemble_set_param': (c_int, [c_void_p, c_int, c_char_p, c_void_p, c_int64]),
    'sis_pixel_ensemble_prepare': (c_int, [c_void_p, c_void_p]),
    'sis_pixel_ensemble_label': (c_int, [c_void_p, c_int, POINTER(c_void_p), POINTER(c_int), POINTER(c_int), c_int, c_int, c_void_p, c_void_p,
                                         c_void_p, c_void_p, c_void_p]),
    'sis_pixel_ensemble_check': (c_int, [c_void_p, c_void_p]),
    'sis_pixel_train_create': (c_int, [POINTER(c_void_p), c_int, c_int, c_int, c_int]),
    'sis_pixel_train_destroy': (None, [c_void_p]),
    'sis_pixel_train_set_param': (c_int, [c_void_p, c_int, c_char_p, c_void_p, c_int64]),
    'sis_pixel_train_set_data': (c_int, [c_void_p, c_int, POINTER(c_void_p), POINTER(c_int), POINTER(c_int), c_int, c_int, c_void_p]),
    'sis_pixel_train_prepare': (c_int, [c_void_p, POINTER(c_uint64), c_int, c_void_p]),
    'sis_pixel_train_steps': (c_int, [c_void_p, c_int, c_void_p]),
    'sis_pixel_train_status': (c_int, [c_void_p, POINTER(ctypes.c_int32), POINTER(c_int64), c_void_p]),
    'sis_pixel_train_read_param': (c_int, [c_void_p, c_int, c_char_p, c_void_p, c_int64, c_void_p]),
    'sis_pixel_train_read_losses': (c_int, [c_void_p, c_int, c_void_p, c_int64, c_void_p]),
    'sis_kmeans_state_bytes': (c_int, []),
    'sis_kmeans_init_state': (c_int, [c_void_p, c_uint64, c_int, c_int64, c_int, c_float, c_void_p]),
    'sis_kmeans_steps': (c_int, [POINTER(KmeansFit), c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load():
    """Load libsis_b200.so (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` or '
            f'`make -C synthesis_in_style_b200/csrc`. There is no CPU / PyTorch fallback for this path.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(status: int):
    if status != 0:
        msg = load().sis_last_error()
        wd = int(load().sis_watchdog_code())
        tail = f'; tcgen05 watchdog fired earlier: code 0x{wd:x}' if wd else ''
        raise RuntimeError(f'libsis_b200: {msg.decode() if msg else "unknown error"} (status {status}){tail}')


PROFILE_CATEGORIES = ('mapping', 'conv_tc', 'blur_split', 'torgb', 'conv_simt', 'label', 'blur_simt', 'other', 'conv_tc_narrow')


def profile_enable(on: bool):
    check(load().sis_profile_enable(int(on)))


def profile_collect():
    """{category: (total ms, launches)} since the last collect."""
    n = len(PROFILE_CATEGORIES)
    ms = (ctypes.c_double * n)()
    cnt = (c_uint64 * n)()
    check(load().sis_profile_collect(ms, cnt, n))
    return {PROFILE_CATEGORIES[i]: (float(ms[i]), int(cnt[i])) for i in range(n)}


def launch_count() -> int:
    return int(load().sis_launch_count())


def current_stream_ptr(device=None):
    import torch
    return c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return c_void_p(t.data_ptr()) if t is not None else c_void_p(0)


def require_cuda(t, name: str):
    import torch
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        # same failure mode as the reference's CHECK_CUDA (fused_bias_act.cpp:13, upfirdn2d.cpp:15)
        raise RuntimeError(f'{name} must be a CUDA tensor')
