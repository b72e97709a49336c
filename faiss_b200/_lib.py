"""ctypes loader for libfaiss_b200.so.  Fails loudly: there is no Python / CPU fallback."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfaiss_b200.so")


class FaissError(RuntimeError):
    """Raised for a non-zero status from the C ABI (c_api/error_c.h:19-35 codes)."""

    def __init__(self, code, msg):
        super().__init__("faiss_b200 error %d: %s" % (code, msg))
        self.code = code


if not os.path.exists(LIB_PATH):
    raise ImportError(
        "faiss_b200: %s is missing. Build it with `python faiss_b200/build.py` (nvcc, sm_100a). "
        "There is no CPU fallback." % LIB_PATH
    )

lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)

lib.faiss_get_last_error.restype = ctypes.c_char_p
lib.faiss_b200_launch_count.restype = ctypes.c_longlong
lib.faiss_b200_kernel_timing.restype = None
lib.faiss_b200_kernel_timing.argtypes = [ctypes.c_int]
lib.faiss_b200_kernel_timing_collect.argtypes = [ctypes.c_char_p, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int)]
lib.faiss_b200_version.restype = ctypes.c_char_p
lib.faiss_Index_ntotal.restype = ctypes.c_int64
lib.faiss_Index_ntotal.argtypes = [ctypes.c_void_p]
lib.faiss_Index_d.argtypes = [ctypes.c_void_p]
lib.faiss_Index_is_trained.argtypes = [ctypes.c_void_p]
lib.faiss_Index_metric_type.argtypes = [ctypes.c_void_p]
lib.faiss_Index_verbose.argtypes = [ctypes.c_void_p]
lib.faiss_Index_set_verbose.argtypes = [ctypes.c_void_p, ctypes.c_int]
lib.faiss_Index_set_verbose.restype = None
lib.faiss_Index_free.argtypes = [ctypes.c_void_p]
lib.faiss_Index_free.restype = None
lib.faiss_StandardGpuResources_free.argtypes = [ctypes.c_void_p]
lib.faiss_StandardGpuResources_free.restype = None
lib.faiss_GpuIndexIVF_nprobe.restype = ctypes.c_size_t
lib.faiss_GpuIndexIVF_nprobe.argtypes = [ctypes.c_void_p]
lib.faiss_GpuIndexIVF_nlist.restype = ctypes.c_size_t
lib.faiss_GpuIndexIVF_nlist.argtypes = [ctypes.c_void_p]
lib.faiss_GpuIndexIVF_get_list_size.restype = ctypes.c_size_t
lib.faiss_GpuIndexIVF_get_list_size.argtypes = [ctypes.c_void_p, ctypes.c_size_t]


def check(code):
    if code != 0:
        raise FaissError(code, lib.faiss_get_last_error().decode(errors="replace"))
