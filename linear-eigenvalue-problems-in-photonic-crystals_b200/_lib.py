"""ctypes binding of libpcb200.so (C ABI declared in include/pcb200.h).

The product loads ``csrc/libpcb200.so`` (built by ``build.py`` for sm_100a) and nothing else:
if the library is missing, or no CUDA device is visible, the first native call raises --
there is no CPU fallback.  ``use_library(path)`` exists so that ``tests/`` can point the
binding at the host-emulation build of the *same kernel sources* (tests/emu); the package
itself never calls it.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_LIB = os.path.join(_HERE, "csrc", "libpcb200.so")

_lib = None
_lib_path = None

c_void_pp = C.POINTER(C.c_void_p)
c_double_p = C.POINTER(C.c_double)
c_int64_p = C.POINTER(C.c_int64)

# name -> (restype, argtypes); every symbol of include/pcb200.h
SIGNATURES = {
    "pcb_last_error": (C.c_char_p, []),
    "pcb_backend": (C.c_char_p, []),
    "pcb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "pcb_supported_sizes": (C.c_int, [C.POINTER(C.c_int), C.c_int]),
    "pcb_ctx_create": (C.c_int, [C.c_int, C.c_int, c_void_pp]),
    "pcb_ctx_destroy": (None, [C.c_void_p]),
    "pcb_sync": (C.c_int, [C.c_void_p]),
    "pcb_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong)]),
    "pcb_ctx_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int]),
    "pcb_ctx_record": (C.c_int, [C.c_void_p, C.c_int]),
    "pcb_ctx_wait": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "pcb_mem_info": (C.c_int, [C.c_void_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "pcb_timer_start": (C.c_int, [C.c_void_p]),
    "pcb_timer_stop": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "pcb_malloc": (C.c_int, [C.c_void_p, C.c_size_t, c_void_pp]),
    "pcb_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pcb_host_alloc": (C.c_int, [C.c_size_t, c_void_pp]),
    "pcb_host_free": (C.c_int, [C.c_void_p]),
    "pcb_memcpy_h2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "pcb_memcpy_d2h": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "pcb_memcpy_d2d": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "pcb_memset_zero": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "pcb_block_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, c_void_pp]),
    "pcb_block_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, c_void_pp]),
    "pcb_fill_uniform": (C.c_int, [C.c_void_p, C.c_int, c_void_pp, C.c_ulonglong]),
    "pcb_diel_create": (C.c_int, [C.c_void_p, C.c_int, c_int64_p, C.c_longlong, c_int64_p, C.c_longlong,
                                  c_double_p, c_double_p, C.c_int, c_double_p, c_void_pp]),
    "pcb_diel_destroy": (None, [C.c_void_p]),
    "pcb_op_create": (C.c_int, [C.c_void_p, c_double_p, C.c_double, C.c_double, C.c_double, C.c_void_p, c_void_pp]),
    "pcb_op_update": (C.c_int, [C.c_void_p, c_double_p, C.c_double, C.c_double, C.c_double, C.c_void_p]),
    "pcb_op_destroy": (None, [C.c_void_p]),
    "pcb_apply": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp]),
    "pcb_apply_host": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong]),
    "pcb_apply_timed": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp, C.POINTER(C.c_float), C.POINTER(C.c_int)]),
    "pcb_residual": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp, c_void_pp, c_double_p, c_double_p]),
    "pcb_gram2": (C.c_int, [C.c_void_p, C.c_int, c_void_pp, c_void_pp, C.c_void_p, C.c_void_p]),
    "pcb_gram2_top": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp, C.c_void_p, C.c_void_p]),
    "pcb_update": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp, c_void_pp, c_void_pp, C.c_void_p]),
    "pcb_update_resid": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp, c_void_pp, c_void_pp, C.c_void_p, c_double_p, c_void_pp, c_double_p]),
    "pcb_update_resid_start": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp, c_void_pp, c_void_pp, C.c_void_p, c_double_p, c_void_pp]),
    "pcb_update_resid_wait": (C.c_int, [C.c_void_p, C.c_int, c_double_p]),
    "pcb_block_launch_info": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]),
    "pcb_coldots": (C.c_int, [C.c_void_p, C.c_int, c_void_pp, c_void_pp, C.c_void_p]),
    "pcb_axpby": (C.c_int, [C.c_void_p, C.c_int, c_void_pp, c_void_pp, C.c_double, C.c_double]),
    "pcb_geometry_mask": (C.c_int, [C.c_void_p, C.c_int, c_double_p, C.c_void_p, C.c_void_p]),
    "pcb_ctx_create_slab": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, c_void_pp]),
    "pcb_comm_unique_id": (C.c_int, [C.c_void_p]),
    "pcb_comm_init": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "pcb_comm_set_host_callbacks": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "pcb_comm_destroy": (C.c_int, [C.c_void_p]),
    "pcb_comm_share": (C.c_int, [C.c_void_p, C.c_void_p, c_void_pp]),
    "pcb_comm_unshare": (C.c_int, [C.c_void_p, c_void_pp]),
    "pcb_comm_barrier": (C.c_int, [C.c_void_p]),
    "pcb_apply_dist": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_void_pp, c_void_pp, C.POINTER(C.c_int), C.c_int, c_void_pp, c_void_pp]),
    "pcb_comm_allreduce_timed": (C.c_int, [C.c_void_p, C.c_longlong, C.c_int, C.POINTER(C.c_float)]),
    "pcb_slab_exchange": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), c_void_pp, c_void_pp]),
}

APPLY_FFT, APPLY_IFFT, APPLY_A, APPLY_H, APPLY_P, APPLY_M, APPLY_KA, APPLY_KAH, APPLY_KB = range(9)
DIEL_NONE, DIEL_CHIRAL, DIEL_TRIVIAL, DIEL_CROSSDOF = range(4)


class PcbError(RuntimeError):
    pass


def _bind(path):
    if not os.path.exists(path):
        raise PcbError(f"native library not found: {path} -- run `python build.py` in "
                       f"{_HERE} (nvcc, sm_100a); there is no CPU fallback")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError if the library does not export it
        fn.restype = res
        fn.argtypes = args
    return lib


def use_library(path):
    """Bind a specific build of the C ABI (tests only: the host-emulation library)."""
    global _lib, _lib_path
    _lib = _bind(path)
    _lib_path = path
    return _lib


def lib():
    global _lib, _lib_path
    if _lib is None:
        _lib = _bind(DEFAULT_LIB)
        _lib_path = DEFAULT_LIB
    return _lib


def lib_path():
    lib()
    return _lib_path


def backend():
    return lib().pcb_backend().decode()


def check(rc, what=""):
    if rc != 0:
        msg = lib().pcb_last_error().decode(errors="replace")
        raise PcbError(f"{what} failed (rc={rc}): {msg}")


def ptr_array(ptrs):
    arr = (C.c_void_p * len(ptrs))(*ptrs)
    return arr
