"""ctypes binding of include/catfish_b200.h (the C-ABI shared library).

The product path has no CPU fallback: if ``libcatfish_b200.so`` is missing it is
built with nvcc (``catfish_b200.build``); if that fails, or a compute entry is
called without a CUDA device, the call raises.
"""

import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcatfish_b200.so")

CF_OK = 0
CF_ERR_BAD_ARG = -1
CF_ERR_CUDA = -2
CF_ERR_NO_DEVICE = -3
CF_ERR_EMPTY_READ = -4
CF_ERR_CAPACITY = -5
CF_ERR_ALLOC = -6

NET_RESNET_RNN, NET_RNN, NET_RESNET = 0, 1, 2
ENGINE_AUTO, ENGINE_TCGEN05, ENGINE_SIMT = 0, 1, 2
ENGINE_NAMES = {ENGINE_AUTO: "auto", ENGINE_TCGEN05: "tcgen05", ENGINE_SIMT: "simt"}

c_i64_p = ctypes.POINTER(ctypes.c_int64)
c_void = ctypes.c_void_p


class ModelDesc(ctypes.Structure):
    _fields_ = [("network_type", ctypes.c_int32), ("window", ctypes.c_int32),
                ("layer_size", ctypes.c_int32), ("n_layers", ctypes.c_int32),
                ("layer_size_res", ctypes.c_int32), ("n_layers_res", ctypes.c_int32),
                ("bn_epsilon", ctypes.c_float), ("engine", ctypes.c_int32)]


# name -> (restype, argtypes); every symbol include/catfish_b200.h declares
SIGNATURES = {
    "cf_abi_version": (ctypes.c_int, []),
    "cf_last_error": (ctypes.c_char_p, []),
    "cf_device_count": (ctypes.c_int, []),
    "cf_model_create": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.POINTER(c_void), c_i64_p,
                                       ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(c_void)]),
    "cf_model_destroy": (None, [c_void]),
    "cf_model_num_tensors": (ctypes.c_int, [ctypes.POINTER(ModelDesc)]),
    "cf_model_engine": (ctypes.c_int, [c_void]),
    "cf_model_operand_format": (ctypes.c_int, [c_void]),
    "cf_model_reserve": (ctypes.c_int, [c_void, ctypes.c_int64, ctypes.c_int32]),
    "cf_infer_windows": (ctypes.c_int, [c_void, c_void, ctypes.c_int64, c_void, c_void]),
    "cf_infer_reads": (ctypes.c_int, [c_void, c_void, c_i64_p, ctypes.c_int32, c_void, c_void, c_void,
                                      ctypes.c_int64, ctypes.c_double, ctypes.c_int32, ctypes.c_int32,
                                      ctypes.c_int32, c_void]),
    "cf_infer_reads_host": (ctypes.c_int, [c_void, c_void, c_i64_p, ctypes.c_int32, c_void, c_void, c_void,
                                           ctypes.c_int64, ctypes.c_double, ctypes.c_int32, ctypes.c_int32,
                                           ctypes.c_int32, c_i64_p, c_void]),
    "cf_exec_create": (ctypes.c_int, [c_void, ctypes.POINTER(c_void)]),
    "cf_exec_destroy": (None, [c_void]),
    "cf_exec_reserve": (ctypes.c_int, [c_void, ctypes.c_int64, ctypes.c_int32]),
    "cf_exec_infer_reads": (ctypes.c_int, [c_void, c_void, c_i64_p, ctypes.c_int32, c_void, c_void, c_void,
                                           ctypes.c_int64, ctypes.c_double, ctypes.c_int32, ctypes.c_int32,
                                           ctypes.c_int32, c_void]),
    "cf_max_intervals": (ctypes.c_int64, [ctypes.c_int64, ctypes.c_int32, ctypes.c_int32]),
    "cf_normalize_reads": (ctypes.c_int, [ctypes.c_int32, c_void, c_i64_p, ctypes.c_int32, c_void, c_void, c_void]),
    "cf_call_intervals": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int32, c_i64_p, ctypes.c_int32,
                                         c_void, c_void, ctypes.c_int64, ctypes.c_double, ctypes.c_int32,
                                         ctypes.c_int32, ctypes.c_int32, c_void]),
    "cf_class_from_threshold": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int64, ctypes.c_double, c_void, c_void]),
    "cf_correct_short": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int64, ctypes.c_int32, c_void, c_void]),
    "cf_hp_in_pred": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int64, ctypes.c_int32, ctypes.c_int32,
                                     ctypes.c_int64, c_void, ctypes.c_int64, c_void, c_void]),
    "cf_profile_enable": (ctypes.c_int, [c_void, ctypes.c_int32]),
    "cf_profile_num_classes": (ctypes.c_int, []),
    "cf_profile_class_name": (ctypes.c_char_p, [ctypes.c_int32]),
    "cf_profile_read": (ctypes.c_int, [c_void, ctypes.POINTER(ctypes.c_double), c_i64_p, ctypes.c_int32]),
    "cf_merge_chunks": (ctypes.c_int, [ctypes.c_int32, c_void, c_i64_p, c_i64_p, ctypes.c_int32, ctypes.c_int64, c_void, c_void,
                                       c_void, c_void, c_void]),
    "cf_split_raw": (ctypes.c_int, [ctypes.c_int32, c_void, c_i64_p, ctypes.c_int32, c_void, c_void, ctypes.c_int64, c_void,
                                    ctypes.c_int64, c_void, c_void]),
    "cf_validate_windows": (ctypes.c_int, [c_void, c_void, c_void, ctypes.c_int64, ctypes.c_int64, ctypes.c_double, c_i64_p,
                                           ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double), c_void]),
    "cf_validate_windows_sweep": (ctypes.c_int, [c_void, c_void, c_void, ctypes.c_int64, ctypes.c_int64, c_void, ctypes.c_int32,
                                                 c_i64_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double),
                                                 c_void]),
    "cf_sweep_thresholds": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int32, c_void, ctypes.c_int64, c_void, ctypes.c_int32,
                                           c_i64_p, c_void]),
    "cf_curve_create": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int32, c_void, ctypes.c_int64, c_void,
                                       ctypes.POINTER(c_void)]),
    "cf_curve_summary": (ctypes.c_int, [c_void, c_i64_p, c_i64_p, c_i64_p, c_i64_p, ctypes.POINTER(ctypes.c_double),
                                        ctypes.POINTER(ctypes.c_double)]),
    "cf_curve_read": (ctypes.c_int, [c_void, ctypes.c_int64, ctypes.c_int64, c_void, c_void]),
    "cf_curve_destroy": (None, [c_void]),
    "cf_vote_events": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int64, c_i64_p, ctypes.c_int64, ctypes.c_int64,
                                      ctypes.c_int64, c_void, c_i64_p, c_i64_p, c_i64_p, ctypes.POINTER(ctypes.c_int32),
                                      c_void]),
    "cf_selftest_f16e5": (ctypes.c_int, [ctypes.c_int32, c_void, ctypes.c_int32, ctypes.c_int32, c_void, ctypes.c_int32, c_void, c_void]),
    "cf_launch_count": (ctypes.c_int64, []),
    "cf_trainer_create": (ctypes.c_int, [ctypes.POINTER(ModelDesc), ctypes.POINTER(c_void), c_i64_p, ctypes.c_int32,
                                         ctypes.POINTER(c_void), ctypes.POINTER(c_void), ctypes.c_int32,
                                         ctypes.POINTER(c_void)]),
    "cf_trainer_destroy": (None, [c_void]),
    "cf_trainer_step": (ctypes.c_int, [c_void, c_void, c_void, ctypes.c_int64, ctypes.c_float, ctypes.c_float,
                                       ctypes.c_uint64, ctypes.c_int64, ctypes.POINTER(ctypes.c_double),
                                       ctypes.POINTER(ctypes.c_double), c_void]),
    "cf_trainer_gradients": (ctypes.c_int, [c_void, c_void, c_void, ctypes.c_int64, ctypes.c_float, ctypes.c_uint64,
                                            ctypes.c_int64, ctypes.POINTER(c_void), ctypes.POINTER(ctypes.c_double),
                                            c_void]),
    "cf_trainer_read": (ctypes.c_int, [c_void, ctypes.POINTER(c_void), ctypes.POINTER(c_void), ctypes.POINTER(c_void)]),
}

_lib = None


def load_library():
    """Load (building first if needed) the shared library; raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("CF_LIB_PATH", LIB_PATH)      # override: A/B-testing a differently built library
    if path == LIB_PATH and not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build()
    lib = ctypes.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so lacks a declared symbol
        fn.restype = restype
        fn.argtypes = argtypes
    if lib.cf_abi_version() != 1:
        raise RuntimeError("libcatfish_b200.so ABI version mismatch")
    _lib = lib
    return lib


class CatfishError(RuntimeError):
    pass


def last_error():
    return load_library().cf_last_error().decode("utf-8", "replace")


def check(status):
    """Map a cf_status to the exception type the reference would raise."""
    if status == CF_OK:
        return
    msg = last_error()
    if status == CF_ERR_BAD_ARG:
        raise ValueError(msg)
    if status == CF_ERR_EMPTY_READ:
        raise IndexError(msg)
    if status == CF_ERR_ALLOC:
        raise MemoryError(msg)
    raise CatfishError("catfish_b200 error %d: %s" % (status, msg))


def launch_count():
    return int(load_library().cf_launch_count())


def profile_enable(model_handle, on=True):
    check(load_library().cf_profile_enable(model_handle, 1 if on else 0))


def profile_read(model_handle):
    """{kernel_class: (milliseconds, launches)} accumulated since profile_enable."""
    lib = load_library()
    n = lib.cf_profile_num_classes()
    ms = (ctypes.c_double * n)()
    cnt = (ctypes.c_int64 * n)()
    check(lib.cf_profile_read(model_handle, ms, cnt, n))
    return {lib.cf_profile_class_name(i).decode(): (ms[i], int(cnt[i])) for i in range(n)}
