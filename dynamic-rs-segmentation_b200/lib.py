"""ctypes binding of libdrs.so (include/drs.h).

The library is the product: there is no Python or CPU fallback.  ``load()`` raises if the shared
object has not been built (``python dynamic-rs-segmentation_b200/csrc/build.py`` or
``__graft_entry__.build()``), and every compute call raises ``DrsError`` with the library's message
when it fails (e.g. no sm_100 device).
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DRS_LIB", os.path.join(_HERE, "libdrs.so"))    # DRS_LIB: an alternative build (experiments)

NET_TYPES = {
    "dilated_icpr_original": 0,        # isprs:761
    "dilated_grsl": 1,                 # isprs:962
    "dilated_icpr_rate6_densely": 2,   # isprs:914
    "dilated_grsl_rate8": 3,           # isprs:996 (contest / coffee key)
    "dilated8_grsl": 3,                # isprs CLI key (isprs:1672-1673)
    "dilated_icpr_rate6": 4,           # isprs:886
    "dilated_icpr_rate6_small": 5,     # isprs:791
    "dilated_icpr_rate6_nodilation": 6,  # isprs:852
    "dilated_icpr_rate1": 7,           # coffee:788
    "dilated_icpr_vary_rate": 8,       # coffee:816
    "dilated_icpr_old": 9,             # contest:574
    "dilated_grsl_old": 1,             # contest:606 == dilated_grsl
    "dilated_icpr_rate6_avgpool": 10,  # isprs:819 (dispatched by the coffee script, coffee:1215)
    "dilated_icpr_rate6_SE": 11,       # isprs:1036
    "dilated_icpr_rate6_squeeze": 12,  # isprs:1064
}
PREC = {"fp32": 0, "f16": 1, "bf16": 2}
SCENE_F64, SCENE_F32 = 0, 1
GRID = {"isprs": 0, "contest": 1, "coffee": 2}


class DrsError(RuntimeError):
    pass


class Config(C.Structure):
    _fields_ = [("net_type", C.c_int32), ("channels", C.c_int32), ("num_classes", C.c_int32),
                ("precision", C.c_int32), ("weight_decay", C.c_float), ("lr_initial", C.c_float),
                ("decay_steps", C.c_int32), ("decay_rate", C.c_float), ("momentum", C.c_float),
                ("bn_decay", C.c_float), ("bn_eps", C.c_float), ("bn_unbiased_ema", C.c_int32),
                ("device", C.c_int32), ("isprs_scopes", C.c_int32)]


class MtState(C.Structure):
    """np.random.get_state() as include/drs.h:drs_mt_state."""
    _fields_ = [("key", C.c_uint32 * 624), ("pos", C.c_int32), ("has_gauss", C.c_int32), ("gauss", C.c_double)]


ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p)

_P = C.c_void_p
_SIGNATURES = {
    "drs_create": (C.c_int, [C.POINTER(_P), C.POINTER(Config)]),
    "drs_destroy": (C.c_int, [_P]),
    "drs_last_error": (C.c_char_p, []),
    "drs_version": (C.c_int, []),
    "drs_set_stream": (C.c_int, [_P, _P]),
    "drs_synchronize": (C.c_int, [_P]),
    "drs_num_variables": (C.c_int, [_P]),
    "drs_variable_name": (C.c_int, [_P, C.c_int, C.c_char_p, C.c_int, C.POINTER(C.c_int64)]),
    "drs_set_variable": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "drs_get_variable": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "drs_get_gradient": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "drs_save": (C.c_int, [_P, C.c_char_p]),
    "drs_load": (C.c_int, [_P, C.c_char_p]),
    "drs_npz_write": (C.c_int, [C.c_char_p, C.c_int32, C.POINTER(C.c_char_p), C.POINTER(_P), C.POINTER(C.c_int32), C.POINTER(C.c_int64)]),
    "drs_npz_entry": (C.c_int, [C.c_char_p, C.c_int32, C.c_char_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int64),
                                C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "drs_npz_read": (C.c_int, [C.c_char_p, C.c_char_p, _P, C.c_int64]),
    "drs_forward_host": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P]),
    "drs_forward_dev": (C.c_int, [_P, _P, C.c_int32, C.c_int32, _P, _P]),
    "drs_train_step_host": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.POINTER(C.c_float), _P, _P]),
    "drs_train_step_dev": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.POINTER(C.c_float), _P, _P]),
    "drs_train_step_async": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, C.POINTER(C.c_int64)]),
    "drs_train_result": (C.c_int, [_P, C.c_int64, C.POINTER(C.c_float), _P]),
    "drs_gather_plan_dev": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, C.c_int64, _P, _P, _P]),
    "drs_reserve_workspace": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32]),
    "drs_train_prepare": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, _P, _P]),
    "drs_set_ignore_label": (C.c_int, [_P, C.c_int32]),
    "drs_set_allreduce": (C.c_int, [_P, ALLREDUCE_FN, _P, C.c_int32, C.c_int32]),
    "drs_comm_unique_id": (C.c_int, [_P]),
    "drs_comm_init": (C.c_int, [_P, _P, C.c_int32, C.c_int32, C.c_int32]),
    "drs_comm_destroy": (C.c_int, [_P]),
    "drs_scene_gather_labels": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, _P]),
    "drs_scene_upload": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "drs_scene_upload_rows": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int32, C.c_int32]),
    "drs_scene_free": (C.c_int, [_P, C.c_int32]),
    "drs_set_gather_fp16": (C.c_int, [_P, C.c_int32]),
    "drs_set_normalization": (C.c_int, [_P, _P, _P]),
    "drs_gather_dev": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "drs_gather_rot_dev": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P, _P]),
    "drs_planner_create": (C.c_int, [C.POINTER(_P)]),
    "drs_planner_destroy": (C.c_int, [_P]),
    "drs_mt_normal": (C.c_int, [_P, C.POINTER(MtState), C.c_double, C.c_double, _P, C.c_int64, C.c_int32]),
    "drs_mt_randint": (C.c_int, [C.POINTER(MtState), C.c_uint32, _P, C.c_int64]),
    "drs_plan_isprs_batch": (C.c_int, [_P, C.POINTER(MtState), _P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P,
                                       _P, _P, _P, _P, _P, _P, _P, C.c_int64, C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int32]),
    "drs_grid_positions": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, C.c_int64,
                                     C.POINTER(C.c_int64)]),
    "drs_accumulate_argmax": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "drs_scene_infer": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "drs_confusion_dev": (C.c_int, [_P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _P]),
    "drs_scene_infer_host": (C.c_int, [_P, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                       C.c_int32, _P, _P]),
    "drs_scene_infer_multiscale": (C.c_int, [_P, C.c_int32, C.c_int32, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P]),
    "drs_debug_np_softmax": (C.c_int, [_P, C.c_int64, C.c_int32, _P]),
    "drs_debug_np_expf": (C.c_int, [_P, C.c_int64, _P]),
    "drs_debug_multiscale_softmax_add": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P, _P]),
    "drs_scene_confusion": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, _P]),
    "drs_launch_count": (C.c_int64, [_P]),
    "drs_set_profiling": (C.c_int, [_P, C.c_int32]),
    "drs_profile_read": (C.c_int, [_P, C.POINTER(C.c_float), C.POINTER(C.c_int64), C.POINTER(C.c_double)]),
    "drs_last_conv_ms": (C.c_int, [_P, C.POINTER(C.c_float)]),
    "drs_debug_activation": (C.c_int, [_P, C.c_char_p, _P, C.c_int64]),
    "drs_debug_conv": (C.c_int, [_P, _P, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_int32, C.c_int32, _P]),
    "drs_bench_conv": (C.c_int, [_P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                 C.c_int32, C.POINTER(C.c_float), _P]),
    "drs_debug_dgrad": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
    "drs_debug_layer": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "drs_debug_conv_schedule": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P, _P, C.c_int32, C.POINTER(C.c_int32)]),
    "drs_debug_wgrad": (C.c_int, [_P, _P, _P, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _P]),
}
EXPORTS = sorted(_SIGNATURES)

_lib = None


def load():
    """dlopen libdrs.so and declare the prototypes.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise DrsError("libdrs.so not built (%s missing): run `python dynamic-rs-segmentation_b200/csrc/build.py`; "
                       "there is no CPU fallback" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        if "DRS_LIB" in os.environ and not hasattr(lib, name):
            continue                 # A/B runs against an older build (tools/ab_lib.py)
        fn = getattr(lib, name)      # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc):
    if rc != 0:
        raise DrsError(load().drs_last_error().decode("utf-8", "replace"))


def ptr(a):
    """Raw address of a NumPy array / torch tensor / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    return a.ctypes.data
