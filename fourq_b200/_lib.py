"""ctypes binding of libfourq_b200.so (include/fourq_b200.h).  There is no CPU fallback: if the library is missing
or no CUDA device is visible, calls raise."""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libfourq_b200.so")

FQ_OK, FQ_ERR_NO_DEVICE, FQ_ERR_CUDA, FQ_ERR_ARG = 0, -1, -2, -3

# op codes of fq_dev_run (include/fourq_b200.h)
FPOP = {"mul": 0, "sqr": 1, "inv": 2, "add": 3, "sub": 4, "neg": 5, "invsqrt": 6}      # FQ_FP_* of the header
DEVOP = {"fp_mul": 32, "fp_sqr": 33, "fp_inv": 34, "fp_add": 35, "fp_sub": 36, "fp_neg": 37, "fp_invsqrt": 38,
         "fp2_mul": 0, "fp2_sqr": 1, "fp2_inv": 2, "fp2_add": 3, "fp2_sub": 4, "fp2_neg": 5, "fp2_conj": 6, "fp2_invsqrt": 7, "fp2_select": 8, "fp_select": 9,
         "decode": 16, "decode_spec": 29, "encode": 17, "dh": 18, "dh_affine": 19, "dh_base": 20, "mul_base": 21, "x25519": 22,
         "dh_endo": 23, "dh_endo_affine": 24, "dh_endo_base": 25, "mul_endo_base": 26, "dh_base_comb": 27, "mul_base_comb": 28, "on_curve": 30,
         "f25519_mul": 48, "f25519_sqr": 49, "f25519_inv": 50, "f25519_add": 51, "f25519_sub": 52}


class FourQError(RuntimeError):
    pass


_lib = None


def lib():
    """The loaded shared library; raises FourQError if it has not been built (python -m fourq_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise FourQError("%s not found: build it with `python -m fourq_b200.build` (needs nvcc). "
                         "fourq_b200 has no CPU implementation." % LIB_PATH)
    _lib = bind(ctypes.CDLL(LIB_PATH))
    return _lib


def bind(L):
    """Sets the argument and result types of every entry point of include/fourq_b200.h on a loaded library."""
    vp, sz, i = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
    sigs = {
        "fq_version": ([], i), "fq_device_count": ([], i), "fq_last_error": ([], ctypes.c_char_p),
        "fq_set_device_base": ([i], i), "fq_set_select_mode": ([i], i), "fq_get_select_mode": ([], i), "fq_trim": ([], i), "fq_last_kernel_ms": ([], ctypes.c_float),
        "fq_last_rows_per_device": ([ctypes.POINTER(sz), i], i),
        "fq_fp2_mul": ([vp, vp, vp, sz, i], i), "fq_fp2_add": ([vp, vp, vp, sz, i], i), "fq_fp2_sub": ([vp, vp, vp, sz, i], i),
        "fq_fp2_sqr": ([vp, vp, sz, i], i), "fq_fp2_inv": ([vp, vp, sz, i], i), "fq_fp2_neg": ([vp, vp, sz, i], i),
        "fq_fp2_conj": ([vp, vp, sz, i], i), "fq_fp2_invsqrt": ([vp, vp, sz, i], i),
        "fq_fp_select": ([vp, vp, vp, vp, sz, i], i), "fq_fp2_select": ([vp, vp, vp, vp, sz, i], i),
        "fq_fp_op": ([i, vp, vp, vp, sz, i], i),
        "fq_fp25519_op": ([i, vp, vp, vp, sz, i], i),
        "fq_decode": ([vp, vp, vp, sz, i], i), "fq_decode_spec": ([vp, vp, vp, sz, i], i), "fq_encode": ([vp, vp, sz, i], i), "fq_point_on_curve": ([vp, vp, sz, i], i),
        "fq_dh": ([vp, vp, vp, vp, sz, i], i), "fq_dh_affine": ([vp, vp, vp, vp, sz, i], i),
        "fq_dh_base": ([vp, vp, vp, sz, i], i), "fq_mul_base": ([vp, vp, sz, i], i),
        "fq_dh_endo": ([vp, vp, vp, vp, sz, i], i), "fq_dh_endo_affine": ([vp, vp, vp, vp, sz, i], i),
        "fq_dh_endo_base": ([vp, vp, vp, sz, i], i), "fq_mul_endo_base": ([vp, vp, sz, i], i),
        "fq_dh_base_comb": ([vp, vp, vp, sz, i], i), "fq_mul_base_comb": ([vp, vp, sz, i], i),
        "fq_x25519": ([vp, vp, vp, sz, i], i),
        "fq_base_create": ([vp, i, vp, ctypes.POINTER(vp)], i), "fq_base_destroy": ([vp], i),
        "fq_dh_fixed": ([vp, vp, vp, vp, sz, i], i), "fq_mul_fixed": ([vp, vp, vp, sz, i], i),
        "fq_base_dev_run": ([vp, i, i, vp, vp, vp, sz, i, ctypes.POINTER(ctypes.c_float)], i),
        "fq_host_alloc": ([ctypes.POINTER(vp), sz], i), "fq_host_free": ([vp], i),
        "fq_host_alloc_sliced": ([ctypes.POINTER(vp), sz, sz, i], i), "fq_device_numa_node": ([i], i),
        "fq_dev_alloc": ([i, ctypes.POINTER(vp), sz], i), "fq_dev_free": ([i, vp], i),
        "fq_dev_upload": ([i, vp, vp, sz], i), "fq_dev_download": ([i, vp, vp, sz], i),
        "fq_dev_run": ([i, i, vp, vp, vp, vp, sz, i, ctypes.POINTER(ctypes.c_float)], i),
        "fq_dev_run3": ([i, i, vp, vp, vp, vp, vp, sz, i, ctypes.POINTER(ctypes.c_float)], i),
        "fq_dev_flush_l2": ([i], i), "fq_dev_last_phase_ms": ([ctypes.POINTER(ctypes.c_float)], i),
        "fq_imad_peak": ([i, ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_double)], i),
    }
    for name, (argtypes, restype) in sigs.items():
        fn = getattr(L, name)
        fn.argtypes, fn.restype = argtypes, restype
    return L


EXPORTS = ["fq_version", "fq_device_count", "fq_last_error", "fq_set_device_base", "fq_set_select_mode", "fq_get_select_mode", "fq_trim", "fq_last_kernel_ms", "fq_last_rows_per_device", "fq_fp2_mul",
           "fq_fp2_sqr", "fq_fp2_inv", "fq_fp2_add", "fq_fp2_sub", "fq_fp2_neg", "fq_fp2_conj", "fq_fp2_invsqrt", "fq_fp_select", "fq_fp2_select", "fq_fp_op", "fq_fp25519_op", "fq_decode", "fq_decode_spec", "fq_encode", "fq_point_on_curve",
           "fq_dh", "fq_dh_affine", "fq_dh_base", "fq_mul_base", "fq_dh_endo", "fq_dh_endo_affine", "fq_dh_endo_base",
           "fq_mul_endo_base", "fq_dh_base_comb", "fq_mul_base_comb", "fq_base_create", "fq_base_destroy", "fq_dh_fixed", "fq_mul_fixed",
           "fq_base_dev_run", "fq_x25519", "fq_host_alloc", "fq_host_free", "fq_host_alloc_sliced", "fq_device_numa_node",
           "fq_dev_alloc", "fq_dev_free", "fq_dev_upload", "fq_dev_download", "fq_dev_run", "fq_dev_run3", "fq_dev_last_phase_ms", "fq_dev_flush_l2", "fq_imad_peak"]


def check(rc):
    if rc != FQ_OK:
        raise FourQError("fourq_b200 error %d: %s" % (rc, lib().fq_last_error().decode("utf-8", "replace")))


def rows(a, width, name="array"):
    """Validates a (N, width) uint8 C-contiguous array (the batched form of the reference's 32-byte strings)."""
    if not isinstance(a, np.ndarray) or a.dtype != np.uint8:
        raise TypeError("%s must be a numpy uint8 array of shape (N, %d)" % (name, width))
    if a.ndim != 2 or a.shape[1] != width:
        # the reference raises "Malformed point: length {} != 32" (curve4q.py:50-51) for single strings
        raise ValueError("%s must have shape (N, %d), got %r" % (name, width, a.shape))
    if not a.flags["C_CONTIGUOUS"]:
        a = np.ascontiguousarray(a)
    return a


def ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else None
