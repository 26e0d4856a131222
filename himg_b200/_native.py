"""ctypes binding of include/himg_cuda.h (libhimgcu.so).  No fallback: if the library is missing
or no CUDA device is usable, calls raise."""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_lib", "libhimgcu.so")

OK, REJECT, ERR_ARG, ERR_CUDA, ERR_CAPACITY, ERR_UNSUPPORTED = range(6)
STRICT, LENIENT = 0, 1

_u8p = C.c_void_p  # raw addresses (host numpy or device torch pointers)

# name -> (restype, argtypes): every symbol include/himg_cuda.h declares
SIGNATURES = {
    "himgcu_abi_version": (C.c_int, []),
    "himgcu_device_count": (C.c_int, []),
    "himgcu_create": (C.c_int, [C.c_int, C.POINTER(C.c_void_p)]),
    "himgcu_destroy": (None, [C.c_void_p]),
    "himgcu_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "himgcu_reset_stream": (C.c_int, [C.c_void_p]),
    "himgcu_synchronize": (C.c_int, [C.c_void_p]),
    "himgcu_last_error": (C.c_char_p, [C.c_void_p]),
    "himgcu_fnv1a64": (C.c_uint64, [_u8p, C.c_size_t]),
    "himgcu_encode_bound": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "himgcu_encode": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p,
                                C.c_size_t, C.POINTER(C.c_size_t)]),
    "himgcu_decode_info": (C.c_int, [_u8p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "himgcu_decode": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_int, _u8p, C.c_size_t, C.POINTER(C.c_int),
                                C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "himgcu_encode_batch": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p,
                                      C.c_size_t, C.c_void_p]),
    "himgcu_encode_status": (C.c_int, [C.c_void_p]),
    "himgcu_decode_batch": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                      C.c_int, _u8p, C.c_void_p]),
    "himgcu_decode_region": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p,
                                       C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "himgcu_decode_batch_region": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_void_p, C.c_int, C.c_int, _u8p, C.c_void_p]),
    "himgcu_decode_batch_region_mixed": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                                   C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, _u8p, C.c_void_p]),
    "himgcu_encode_batch_mixed": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_int, C.c_int, _u8p, C.c_size_t, C.c_void_p]),
    "himgcu_decode_batch_mixed": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                                            C.c_int, C.c_int, C.c_void_p, _u8p, C.c_void_p]),
    "himgcu_decode_scaled": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_int, C.c_int, _u8p, C.c_size_t, C.POINTER(C.c_int),
                                       C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "himgcu_decode_batch_scaled": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                             C.c_int, C.c_int, _u8p, C.c_void_p]),
    "himgcu_decode_batch_mixed_scaled": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int,
                                                   C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, _u8p, C.c_void_p]),
    "himgcu_decode_region_scaled": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                              C.c_int, _u8p, C.c_size_t, C.POINTER(C.c_int), C.POINTER(C.c_int),
                                              C.POINTER(C.c_int)]),
    "himgcu_decode_batch_region_scaled": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                                    C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_int, _u8p, C.c_void_p]),
    "himgcu_decode_batch_region_mixed_scaled": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                                          C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int,
                                                          C.c_int, _u8p, C.c_void_p]),
    "himgcu_host_alloc": (C.c_void_p, [C.c_size_t]),
    "himgcu_host_free": (None, [C.c_void_p]),
    "himgcu_encode_batch_host": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p,
                                           C.c_size_t, C.c_void_p, C.c_void_p]),
    "himgcu_decode_batch_host": (C.c_int, [C.c_void_p, _u8p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int,
                                           C.c_int, _u8p, C.c_void_p]),
    "himgcu_stage_lowres": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p]),
    "himgcu_lres_size": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "himgcu_lres_stride": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "himgcu_stage_lres_encode": (C.c_int, [C.c_void_p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _u8p]),
    "himgcu_stage_forward": (C.c_int, [C.c_void_p, _u8p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_int, _u8p]),
    "himgcu_stage_huff_compress": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_int, C.c_int, C.c_int, _u8p,
                                             C.c_size_t, C.c_void_p]),
    "himgcu_stage_huff_uncompress": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.c_int, _u8p, C.c_size_t, C.c_void_p]),
    "himgcu_stage_lres_decode": (C.c_int, [C.c_void_p, _u8p, C.c_size_t, C.c_int, C.c_int, C.c_int, C.c_int,
                                           C.c_void_p, _u8p]),
    "himgcu_stage_inverse": (C.c_int, [C.c_void_p, _u8p, _u8p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       C.c_void_p, C.c_void_p, C.c_void_p, _u8p]),
    "himgcu_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "himgcu_profile_reset": (C.c_int, [C.c_void_p]),
    "himgcu_profile_count": (C.c_int, [C.c_void_p]),
    "himgcu_profile_get": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_char_p), C.POINTER(C.c_double),
                                     C.POINTER(C.c_int)]),
    "himgcu_launch_count": (C.c_uint64, [C.c_void_p]),
    "himgcu_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_longlong]),
}

_lib = None


def load():
    """Load libhimgcu.so and bind every declared symbol.  Raises if the library is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension must be built (python -m himg_b200.build); "
            "there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class HimgError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"himgcu error {code}: {msg}")
        self.code = code
