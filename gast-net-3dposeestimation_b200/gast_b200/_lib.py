"""ctypes binding of csrc/libgast_b200.so (C ABI: include/gast_b200.h).

There is no fallback: if the shared library is missing or fails to load, importing the
engine raises with the build command.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get('GAST_B200_LIB') or os.path.join(os.path.dirname(_HERE), 'csrc', 'libgast_b200.so')
# (GAST_B200_LIB: alternative build of the same library, used only for A/B experiments)

GAST_MAX_STAGES = 8
KIND_MODEL, KIND_BLOCK, KIND_LOCAL, KIND_MGLOBAL, KIND_SEMCH, KIND_GLOBAL_HEAD = range(6)

# every symbol include/gast_b200.h declares
SYMBOLS = ['gast_create', 'gast_destroy', 'gast_bind', 'gast_prepare', 'gast_out_frames',
           'gast_receptive_field', 'gast_workspace_bytes', 'gast_forward', 'gast_forward_mpjpe',
           'gast_last_launch_count', 'gast_last_tc_launch_count', 'gast_set_timing',
           'gast_get_timings', 'gast_set_gemm_core', 'gast_debug_gemm', 'gast_bind_grads',
           'gast_train_workspace_bytes', 'gast_forward_train', 'gast_backward', 'gast_set_dropout_state', 'gast_tta_prepare', 'gast_tta_merge',
           'gast_stream_state_bytes', 'gast_stream_workspace_bytes', 'gast_stream_push',
           'gast_stream_delay', 'gast_stream_delayed_state_bytes', 'gast_stream_delayed_workspace_bytes',
           'gast_stream_push_delayed',
           'gast_chunk_gather', 'gast_keypoints_convert', 'gast_normalize_screen', 'gast_camera_to_world',
           'gast_mpjpe_workspace_bytes', 'gast_mpjpe', 'gast_p_mpjpe', 'gast_adam_chunk', 'gast_adam_step',
           'gast_last_error', 'gast_version']


class GastCfg(C.Structure):
    _fields_ = [
        ('kind', C.c_int32), ('num_joints', C.c_int32), ('in_features', C.c_int32),
        ('channels', C.c_int32), ('channels_out', C.c_int32), ('num_stages', C.c_int32),
        ('filter_widths', C.c_int32 * GAST_MAX_STAGES),
        ('causal', C.c_int32), ('dense', C.c_int32), ('strided', C.c_int32),
        ('heads', C.c_int32), ('semch_shared_e', C.c_int32), ('semch_bias', C.c_int32),
        ('sym_nnz', C.c_int32), ('con_nnz', C.c_int32),
        ('sym_rows', C.POINTER(C.c_int32)), ('sym_cols', C.POINTER(C.c_int32)),
        ('con_rows', C.POINTER(C.c_int32)), ('con_cols', C.POINTER(C.c_int32)),
        ('device', C.c_int32),
    ]


_lib = None


def load():
    """Load the library once; raise loudly when it is absent (no CPU / torch fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            'gast_b200: %s not found. Build it with `python __graft_entry__.py build` '
            '(or gast-net-3dposeestimation_b200/csrc/build.sh). There is no fallback path.' % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.gast_create.argtypes = [C.POINTER(vp), C.POINTER(GastCfg)]
    lib.gast_create.restype = C.c_int
    lib.gast_destroy.argtypes = [vp]
    lib.gast_destroy.restype = None
    lib.gast_bind.argtypes = [vp, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(vp), C.POINTER(C.c_int64)]
    lib.gast_bind.restype = C.c_int
    lib.gast_prepare.argtypes = [vp, vp]
    lib.gast_prepare.restype = C.c_int
    lib.gast_out_frames.argtypes = [vp, C.c_int32, C.c_int32]
    lib.gast_out_frames.restype = C.c_int32
    lib.gast_receptive_field.argtypes = [vp]
    lib.gast_receptive_field.restype = C.c_int32
    lib.gast_workspace_bytes.argtypes = [vp, C.c_int32, C.c_int32, C.c_int32]
    lib.gast_workspace_bytes.restype = C.c_size_t
    lib.gast_forward.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, C.c_size_t, vp]
    lib.gast_forward.restype = C.c_int
    lib.gast_forward_mpjpe.argtypes = [vp, vp, vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp, C.c_size_t, vp]
    lib.gast_forward_mpjpe.restype = C.c_int
    lib.gast_last_launch_count.argtypes = [vp]
    lib.gast_last_launch_count.restype = C.c_int32
    lib.gast_last_tc_launch_count.argtypes = [vp]
    lib.gast_last_tc_launch_count.restype = C.c_int32
    lib.gast_set_timing.argtypes = [vp, C.c_int32]
    lib.gast_set_timing.restype = C.c_int
    lib.gast_get_timings.argtypes = [vp, C.c_int32, C.POINTER(C.c_float), C.POINTER(C.c_int32)]
    lib.gast_get_timings.restype = C.c_int32
    lib.gast_set_gemm_core.argtypes = [vp, C.c_int32]
    lib.gast_set_gemm_core.restype = C.c_int
    lib.gast_debug_gemm.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                    C.POINTER(C.c_float), vp]
    lib.gast_debug_gemm.restype = C.c_int
    lib.gast_bind_grads.argtypes = [vp, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(vp), C.POINTER(C.c_int64)]
    lib.gast_bind_grads.restype = C.c_int
    lib.gast_train_workspace_bytes.argtypes = [vp, C.c_int32, C.c_int32, C.c_float]
    lib.gast_train_workspace_bytes.restype = C.c_size_t
    lib.gast_forward_train.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_float, C.c_uint64, vp, C.c_size_t, vp]
    lib.gast_forward_train.restype = C.c_int
    lib.gast_backward.argtypes = [vp, vp, vp, C.c_size_t, vp]
    lib.gast_backward.restype = C.c_int
    lib.gast_set_dropout_state.argtypes = [vp, vp]
    lib.gast_set_dropout_state.restype = C.c_int
    lib.gast_stream_state_bytes.argtypes = [vp, C.c_int32]
    lib.gast_stream_state_bytes.restype = C.c_size_t
    lib.gast_stream_workspace_bytes.argtypes = [vp, C.c_int32]
    lib.gast_stream_workspace_bytes.restype = C.c_size_t
    lib.gast_stream_push.argtypes = [vp, vp, C.c_int64, vp, vp, C.c_int32, vp, vp, C.c_size_t, vp]
    lib.gast_stream_push.restype = C.c_int
    ip = C.POINTER(C.c_int32)
    lib.gast_stream_delay.argtypes = [vp]
    lib.gast_stream_delay.restype = C.c_int32
    lib.gast_stream_delayed_state_bytes.argtypes = [vp, C.c_int32, C.c_int32]
    lib.gast_stream_delayed_state_bytes.restype = C.c_size_t
    lib.gast_stream_delayed_workspace_bytes.argtypes = [vp, C.c_int32, C.c_int32]
    lib.gast_stream_delayed_workspace_bytes.restype = C.c_size_t
    lib.gast_stream_push_delayed.argtypes = [vp, vp, C.c_size_t, C.c_int64, vp, vp, C.c_int32, vp, vp, C.c_int32,
                                             ip, ip, ip, ip, vp, C.c_size_t, vp]
    lib.gast_stream_push_delayed.restype = C.c_int
    lib.gast_tta_prepare.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, ip, ip, vp]
    lib.gast_tta_prepare.restype = C.c_int
    lib.gast_tta_merge.argtypes = [vp, vp, C.c_int32, C.c_int32, C.c_int32, ip, ip, vp]
    lib.gast_tta_merge.restype = C.c_int
    fp = C.POINTER(C.c_float)
    lib.gast_chunk_gather.argtypes = [vp, vp, vp, vp, C.c_int32, vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                      C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, ip, ip, C.c_int32, ip, ip,
                                      vp, vp, vp, vp]
    lib.gast_chunk_gather.restype = C.c_int
    lib.gast_keypoints_convert.argtypes = [vp, vp, vp, C.c_int32, C.c_int32, C.c_int32, vp]
    lib.gast_keypoints_convert.restype = C.c_int
    lib.gast_normalize_screen.argtypes = [vp, vp, C.c_int64, C.c_float, C.c_float, C.c_int32, vp]
    lib.gast_normalize_screen.restype = C.c_int
    lib.gast_camera_to_world.argtypes = [vp, vp, C.c_int64, fp, fp, vp]
    lib.gast_camera_to_world.restype = C.c_int
    lib.gast_mpjpe_workspace_bytes.argtypes = []
    lib.gast_mpjpe_workspace_bytes.restype = C.c_size_t
    lib.gast_mpjpe.argtypes = [vp, vp, C.c_int64, C.c_int32, vp, vp, C.c_float, vp, vp]
    lib.gast_mpjpe.restype = C.c_int
    lib.gast_p_mpjpe.argtypes = [vp, vp, C.c_int32, C.c_int32, vp, vp]
    lib.gast_p_mpjpe.restype = C.c_int
    lib.gast_adam_chunk.argtypes = []
    lib.gast_adam_chunk.restype = C.c_int32
    lib.gast_adam_step.argtypes = [vp, C.c_int32, vp, vp, vp, C.c_double, C.c_double, C.c_double, C.c_double,
                                   C.c_double, C.c_int64, vp]
    lib.gast_adam_step.restype = C.c_int
    lib.gast_last_error.argtypes = []
    lib.gast_last_error.restype = C.c_char_p
    lib.gast_version.argtypes = []
    lib.gast_version.restype = C.c_char_p
    _lib = lib
    return lib


def last_error():
    return load().gast_last_error().decode('utf-8', 'replace')
