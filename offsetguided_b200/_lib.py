"""ctypes binding of libogdecoder.so (include/og_decoder.h).

This is the stub a maintainer of the reference would add to call the library from
``decoder/`` (INTEGRATION.md).  There is no fallback: if the library is missing or a
call fails, a Python exception is raised.
"""
import ctypes
import os

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG_DIR, 'libogdecoder.so')

OG_LIMB_COLS = 13
OG_POSE_COLS = 6
OG_MAX_TOPK = 128
OG_MAX_IN_FLIGHT = 16
OG_DTYPE_F32 = 0
OG_DTYPE_BF16 = 1
OG_DTYPE_F16 = 2

c_int32_p = ctypes.POINTER(ctypes.c_int32)
c_float_p = ctypes.POINTER(ctypes.c_float)


class OgConfig(ctypes.Structure):
    _fields_ = [
        ('n_keypoints', ctypes.c_int32),
        ('n_limbs', ctypes.c_int32),
        ('limb_from', c_int32_p),
        ('limb_to', c_int32_p),
        ('topk', ctypes.c_int32),
        ('thre_hmp', ctypes.c_float),
        ('min_len', ctypes.c_float),
        ('resize_factor', ctypes.c_float),
        ('dist_max', ctypes.c_float),
        ('use_scale', ctypes.c_int32),
        ('person_thre', ctypes.c_double),
        ('sort_dim', ctypes.c_int32),
        ('device', ctypes.c_int32),
        ('max_images', ctypes.c_int32),
    ]


class OgResult(ctypes.Structure):
    _fields_ = [
        ('poses', c_float_p),
        ('offsets', c_int32_p),
        ('counts', c_int32_p),
        ('n_images', ctypes.c_int32),
        ('total_rows', ctypes.c_int32),
        ('n_keypoints', ctypes.c_int32),
        ('buffer_id', ctypes.c_int32),
        ('coco_keypoints', c_float_p),
        ('coco_scores', ctypes.POINTER(ctypes.c_double)),
        ('coco_images', c_int32_p),
    ]


class OgError(RuntimeError):
    pass


_vp = ctypes.c_void_p
_i = ctypes.c_int
_i64_p = ctypes.POINTER(ctypes.c_int64)
# name -> (restype, argtypes); every symbol include/og_decoder.h declares
SIGNATURES = {
    'og_last_error': (ctypes.c_char_p, []),
    'og_status_string': (ctypes.c_char_p, [_i]),
    'og_abi_version': (_i, []),
    'og_create': (_i, [ctypes.POINTER(OgConfig), ctypes.POINTER(_vp)]),
    'og_destroy': (_i, [_vp]),
    'og_hmp_nms_f32': (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    'og_topk_channel_f32': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    'og_nms_topk_f32': (_i, [_vp, _vp, _i, _i, _i, ctypes.c_float, _vp, _vp, _vp, _vp]),
    'og_limb_score_f32': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    'og_limb_score_ex_f32': (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    'og_group_f32': (_i, [_vp, _vp, _i, _vp, ctypes.c_int32, _vp, _vp, _vp, _vp]),
    'og_scored_offset_f32': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp]),
    'og_flip_fuse_f32': (_i, [_vp, _vp, _vp, c_int32_p, c_int32_p, c_int32_p, _i, _i, _i, _i, _vp, _vp, _vp]),
    'og_flip_average_f32': (_i, [_vp, c_int32_p, _i, _i, _i, _i, _i, _vp, _vp]),
    'og_flip_cat_offsets_f32': (_i, [_vp, c_int32_p, c_int32_p, _i, _i, _i, _i, _i, _vp, _vp]),
    'og_resize_f32': (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp]),
    'og_decode_maps': (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    'og_decode_maps_ex': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _vp]),
    'og_decode_features_host': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i,
                                     c_int32_p, c_int32_p, c_int32_p, _i, _vp]),
    'og_decode_features_dev': (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i,
                                    c_int32_p, c_int32_p, c_int32_p, _i, _vp]),
    'og_decode_features_dev_ex': (_i, [_vp, _vp, _vp, _i, ctypes.c_int64, ctypes.c_int64, _i, _i, _i, _i, _i,
                                       _i, _i, c_int32_p, c_int32_p, c_int32_p, _i, _vp]),
    'og_decode_features_dev_strided': (_i, [_vp, _vp, _vp, _i, _i64_p, _i64_p, _i, _i, _i, _i, _i, _i, _i,
                                            c_int32_p, c_int32_p, c_int32_p, _i, _vp]),
    'og_fetch_poses': (_i, [_vp, ctypes.POINTER(c_float_p), ctypes.POINTER(c_int32_p),
                            ctypes.POINTER(c_int32_p), ctypes.POINTER(ctypes.c_int32)]),
    'og_decode_features_heads_dev': (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i,
                                          _i, _i, c_int32_p, c_int32_p, c_int32_p, _i, _vp]),
    'og_plan_features': (_i, [_vp, _vp, _vp, _i, ctypes.c_int64, ctypes.c_int64, _i, _i, _i, _i, _i,
                              _i, _i, c_int32_p, c_int32_p, c_int32_p, _i, ctypes.POINTER(ctypes.c_int32)]),
    'og_plan_features_strided': (_i, [_vp, _vp, _vp, _i, _i64_p, _i64_p, _i, _i, _i, _i, _i, _i, _i,
                                      c_int32_p, c_int32_p, c_int32_p, _i, ctypes.POINTER(ctypes.c_int32)]),
    'og_plan_launch': (_i, [_vp, ctypes.c_int32, _vp]),
    'og_fetch_result': (_i, [_vp, ctypes.POINTER(OgResult)]),
    'og_set_frames': (_i, [_vp, ctypes.POINTER(ctypes.c_double), _i]),
    'og_pending': (_i, [_vp]),
    'og_copy_intermediates': (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    'og_launch_count': (ctypes.c_int64, [_vp]),
    'og_set_fused': (_i, [_vp, _i]),
    'og_set_graph': (_i, [_vp, _i]),
    'og_graph_replay_count': (ctypes.c_int64, [_vp]),
    'og_graph_build_count': (ctypes.c_int64, [_vp]),
    'og_debug_k3_profile': (_i, [ctypes.POINTER(ctypes.c_uint64), _i]),
    'og_fused_redo_count': (ctypes.c_int64, [_vp]),
    'og_k3_redo_count': (ctypes.c_int64, [_vp]),
    'og_set_zero_copy': (_i, [_vp, _i]),
    'og_zero_copy_count': (ctypes.c_int64, [_vp]),
    'og_enable_stage_timing': (_i, [_vp, _i]),
    'og_last_stage_times_ms': (_i, [_vp, c_float_p]),
}

_lib = None


def load():
    """Load the shared library (once).  Raises OgError when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise OgError(
            f'{LIB_PATH} is missing: build it with `python -m offsetguided_b200.build` '
            '(or __graft_entry__.build()).  There is no CPU fallback.')
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.og_abi_version() != 2:
        raise OgError(f'ABI version mismatch: library reports {lib.og_abi_version()}')
    _lib = lib
    return lib


def check(status):
    if status != 0:
        lib = load()
        raise OgError('%s: %s' % (lib.og_status_string(status).decode(),
                                  lib.og_last_error().decode()))


def int64_array(values):
    values = [int(v) for v in values]
    return (ctypes.c_int64 * max(len(values), 1))(*values)


def int32_array(values):
    values = [int(v) for v in values]
    return (ctypes.c_int32 * max(len(values), 1))(*values)
