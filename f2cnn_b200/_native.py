"""ctypes binding of libf2cnn_b200.so (C ABI: include/f2cnn_b200.h).

The shared library is built in-tree by `make -C f2cnn_b200/csrc` (or
`__graft_entry__.build()`).  There is deliberately no fallback: if the library is missing
or no CUDA device is usable, importing / calling raises."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("F2CNN_B200_LIB") or os.path.join(_HERE, "libf2cnn_b200.so")  # env override: tuning builds

F2_OK = 0
F2_I16, F2_F32, F2_F64 = 0, 1, 2
F2_ROWS_ENVELOPE, F2_ROWS_HILBERT, F2_ROWS_LOWPASS = 0, 1, 2
F2_ERR_INVALID, F2_ERR_CUDA, F2_ERR_WORKSPACE, F2_ERR_UNSUPPORTED, F2_ERR_INDEX = 1, 2, 3, 4, 5
ABI_VERSION = 6
F2_PLAN_FLOAT64_SECTIONS = 1


class F2Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("libf2cnn_b200 error %d: %s" % (code, msg))
        self.code = code


class RunArgs(ctypes.Structure):
    """struct f2_run_args; struct_size is filled in by __init__ (the library rejects short structs)."""
    _fields_ = [
        ("struct_size", ctypes.c_uint32),
        ("wave", ctypes.c_void_p),
        ("wave_dtype", ctypes.c_int),
        ("lpf", ctypes.c_int),
        ("cutoff_hz", ctypes.c_double),
        ("gfb", ctypes.c_void_p),
        ("gfb_dtype", ctypes.c_int),
        ("env", ctypes.c_void_p),
        ("env_dtype", ctypes.c_int),
        ("env_t", ctypes.c_void_p),
        ("dec", ctypes.c_void_p),
        ("ev_fused_start", ctypes.c_void_p),
        ("ev_fused_stop", ctypes.c_void_p),
        ("windows", ctypes.c_void_p),
        ("win_offsets", ctypes.c_void_p),
        ("win_dots", ctypes.c_int),
    ]

    def __init__(self, *args, **kw):
        super().__init__(*args, **kw)
        self.struct_size = ctypes.sizeof(RunArgs)


class WinRun(ctypes.Structure):
    """struct f2_win_run: `count` windows, window i = frames first_frame+i .. +dots-1 -> row row0+i."""
    _fields_ = [("first_frame", ctypes.c_int64), ("row0", ctypes.c_int64), ("count", ctypes.c_int64)]


_lib = None

# name -> (restype, argtypes): every symbol include/f2cnn_b200.h declares
SIGNATURES = {
    "f2_last_error": (ctypes.c_char_p, []),
    "f2_abi_version": (ctypes.c_int, []),
    "f2_plan_create": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.c_int, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_void_p)]),
    "f2_bank_check": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.c_int, ctypes.POINTER(ctypes.c_double),
                                     ctypes.POINTER(ctypes.c_int)]),
    "f2_plan_create_ex": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.c_int, ctypes.c_int, ctypes.c_uint,
                                         ctypes.POINTER(ctypes.c_void_p)]),
    "f2_bank_check_groups": (ctypes.c_int, [ctypes.POINTER(ctypes.c_double), ctypes.c_int,
                                            ctypes.POINTER(ctypes.c_double)]),
    "f2_plan_float64_groups": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_ubyte), ctypes.c_int]),
    "f2_plan_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_plan_channels": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_plan_set_warmup": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "f2_plan_get_warmup": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int),
                                          ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]),
    "f2_batch_create": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64), ctypes.c_int, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_int64, ctypes.POINTER(ctypes.c_void_p)]),
    "f2_batch_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_batch_total_samples": (ctypes.c_int64, [ctypes.c_void_p]),
    "f2_batch_total_frames": (ctypes.c_int64, [ctypes.c_void_p]),
    "f2_batch_num_items": (ctypes.c_int64, [ctypes.c_void_p]),
    "f2_batch_frame_offsets": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(ctypes.c_int64)]),
    "f2_batch_workspace_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int]),
    "f2_batch_run": (ctypes.c_int, [ctypes.c_void_p, ctypes.POINTER(RunArgs), ctypes.c_void_p, ctypes.c_size_t,
                                    ctypes.c_void_p]),
    "f2_batch_run_cutoffs": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                            ctypes.POINTER(ctypes.c_double), ctypes.c_int, ctypes.c_void_p,
                                            ctypes.c_int64, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "f2_envelope_rows_workspace_bytes":(ctypes.c_size_t, [ctypes.c_int64, ctypes.c_int64]),
    "f2_envelope_rows": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64,
                                        ctypes.c_int64, ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_int,
                                        ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "f2_rows_op": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_int64,
                                  ctypes.c_int, ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_int,
                                  ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "f2_gather_windows_cn": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                            ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]),
    "f2_gather_windows": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64,
                                         ctypes.c_int, ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p]),
    "f2_gather_index": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64,
                                       ctypes.c_void_p, ctypes.c_void_p]),
    "f2_dense_frames": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int64,
                                       ctypes.c_int64, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                       ctypes.c_void_p]),
    "f2_label_fit": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                    ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]),
    "f2_label_accuracy": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p,
                                         ctypes.c_void_p]),
    "f2_window_runs": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.POINTER(ctypes.c_int), ctypes.c_void_p, ctypes.c_int64,
                                      ctypes.POINTER(ctypes.c_int64), ctypes.POINTER(ctypes.c_int64)]),
    "f2_place_windows": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_int64,
                                        ctypes.c_void_p, ctypes.c_int]),
    "f2_placer_create": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "f2_placer_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_placer_threads": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_placer_submit": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "f2_placer_wait": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_placer_trace": (ctypes.c_int64, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int]),
    "f2_host_alloc": (ctypes.c_int, [ctypes.c_size_t, ctypes.POINTER(ctypes.c_void_p)]),
    "f2_host_free": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t]),
    "f2_host_pin": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t]),
    "f2_host_unpin": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_cnn_create": (ctypes.c_int, [ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.POINTER(ctypes.c_void_p)]),
    "f2_cnn_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_cnn_workspace_bytes": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_int64]),
    "f2_cnn_forward": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int, ctypes.c_int64,
                                      ctypes.c_int64, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t,
                                      ctypes.c_void_p]),
    "f2_cnn_forward_segments": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int,
                                               ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                               ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p]),
    "f2_cnn_workspace_layout": (ctypes.c_int, [ctypes.c_int64, ctypes.POINTER(ctypes.c_int64),
                                               ctypes.POINTER(ctypes.c_size_t)]),
    "f2_umma_selftest": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]),
    "f2_upload_spans": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                       ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p]),
    "f2_event_create": (ctypes.c_int, [ctypes.POINTER(ctypes.c_void_p)]),
    "f2_event_destroy": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_event_record": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p]),
    "f2_event_synchronize": (ctypes.c_int, [ctypes.c_void_p]),
    "f2_event_elapsed_ms": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_void_p, ctypes.POINTER(ctypes.c_float)]),
    "f2_lowpass_coefficients": (ctypes.c_int, [ctypes.c_double, ctypes.POINTER(ctypes.c_double),
                                               ctypes.POINTER(ctypes.c_double)]),
}


def lib():
    """Load the shared library once; raise (never fall back) when it is not there."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s not found: build it with `make -C f2cnn_b200/csrc` (nvcc, sm_100a). "
                "f2cnn_b200 has no CPU or PyTorch fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)  # AttributeError if the header and the library drifted apart
            fn.restype = res
            fn.argtypes = args
        if L.f2_abi_version() != ABI_VERSION:
            raise ImportError("libf2cnn_b200.so ABI %d, binding expects %d" % (L.f2_abi_version(), ABI_VERSION))
        _lib = L
    return _lib


def check(code):
    if code != F2_OK:
        raise F2Error(code, lib().f2_last_error().decode("utf-8", "replace"))
