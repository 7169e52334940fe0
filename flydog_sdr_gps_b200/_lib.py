"""ctypes binding of the C ABI (include/acq_b200.h).  Fails loudly if the CUDA library is missing:
there is no CPU fallback anywhere in this package."""
import ctypes as C
import os

from . import _build

_lib = None


class AcqSat(C.Structure):
    _fields_ = [("prn", C.c_int32), ("t1", C.c_int32), ("t2", C.c_int32), ("type", C.c_int32)]


class AcqParams(C.Structure):
    _fields_ = [("struct_size", C.c_uint32),
                ("dop_lo", C.c_int32), ("dop_hi", C.c_int32), ("half_bin", C.c_int32), ("k_noncoh", C.c_int32),
                ("thr_l1", C.c_float), ("thr_e1b", C.c_float), ("wrap_mode", C.c_int32), ("sample_bits", C.c_int32),
                ("code_doppler", C.c_int32), ("reserved", C.c_int32 * 6)]


# every symbol include/acq_b200.h declares: (name, restype, argtypes)
_P = C.c_void_p
_SIGNATURES = [
    ("acq_last_error", C.c_char_p, []),
    ("acq_abi_version", C.c_int, []),
    ("acq_params_default", C.c_int, [C.POINTER(AcqParams)]),
    ("acq_create", C.c_int, [C.POINTER(_P), C.POINTER(AcqParams), C.POINTER(AcqSat), C.c_int, C.c_int]),
    ("acq_destroy", C.c_int, [_P]),
    ("acq_search", C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P]),
    ("acq_search_grid", C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P]),
    ("acq_search_device", C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, _P]),
    ("acq_search_aided", C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int, _P, _P]),
    ("acq_search_aided_device", C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P, C.c_int, _P, _P]),
    ("acq_submit", C.c_int, [_P, _P, C.c_int, _P, C.c_int, _P]),
    ("acq_poll", C.c_int, [_P]),
    ("acq_wait", C.c_int, [_P]),
    ("acq_refine", C.c_int, [_P, _P, C.c_int, _P]),
    ("acq_detected", C.c_int, [_P, _P]),
    ("acq_get_code_spectrum", C.c_int, [_P, C.c_int, _P]),
    ("acq_get_capture_spectrum", C.c_int, [_P, _P, C.c_int, _P, _P]),
    ("acq_n_sats", C.c_int, [_P]),
    ("acq_get_params", C.c_int, [_P, C.POINTER(AcqParams)]),
    ("acq_launch_count", C.c_int64, [_P]),
    ("acq_set_profiling", C.c_int, [_P, C.c_int]),
    ("acq_get_kernel_ms", C.c_int, [_P, C.POINTER(C.c_float), C.c_int]),
    ("acq_device_info", C.c_int, [_P, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    ("acq_plan_launch", C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int64, C.c_int, _P]),
    ("acq_microbench", C.c_int, [C.c_int, C.POINTER(C.c_double), C.c_int]),
]


class AcqLaunchPlan(C.Structure):
    _fields_ = [("kernel", C.c_int32), ("grid", C.c_int32), ("claims", C.c_int32), ("chunk_big", C.c_int32),
                ("chunk_mid", C.c_int32), ("n_big", C.c_uint32), ("n_mid", C.c_uint32), ("n_chunks", C.c_int64)]


def exported_symbols():
    return [s[0] for s in _SIGNATURES]


def lib_path():
    return _build.LIB


def _bind(path):
    if not os.path.exists(path):
        raise RuntimeError("%s is missing and could not be built; the engine has no CPU fallback" % os.path.basename(path))
    L = C.CDLL(path)
    for name, res, args in _SIGNATURES:
        fn = getattr(L, name)  # AttributeError if the library does not export the header's symbol
        fn.restype = res
        fn.argtypes = args
    return L


def load():
    """Load libacq_b200.so (building it first if sources are newer).  Raises if that is impossible."""
    global _lib
    if _lib is None:
        path = os.environ.get("ACQ_B200_LIB")  # experiment variant of the same CUDA library (A/B runs)
        if not path:
            path = _build.build() if _build.needs_build() else _build.LIB
        _lib = _bind(path)
    return _lib


_variants = {}


def load_variant(name):
    """An experiment variant of the library (tools/build_variants.py; A/B forms of the kernels live only there),
    loaded NEXT TO the product library -- used by the tests that assert bitwise equality between kernel forms."""
    if name not in _variants:
        _variants[name] = _bind(_build.build_variant(name))
    return _variants[name]
