"""ctypes binding of libgpk.so (C ABI declared in include/gpk.h).

There is no CPU fallback: if the library is missing or no CUDA device is present the
product path raises. torch is used only as the device-memory allocator / stream owner.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libgpk.so")
_lib = None

c_double_p = ctypes.POINTER(ctypes.c_double)
c_int_p = ctypes.POINTER(ctypes.c_int)
i64 = ctypes.c_int64
vp = ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/gpk.h declares
SIGNATURES = {
    "gpk_version": (ctypes.c_int, []),
    "gpk_last_error": (ctypes.c_char_p, []),
    "gpk_npad": (i64, [i64]),
    "gpk_create": (ctypes.c_int, [i64, i64, vp, vp, ctypes.POINTER(vp)]),
    "gpk_destroy": (ctypes.c_int, [vp]),
    "gpk_set_stream": (ctypes.c_int, [vp, vp]),
    "gpk_set_data": (ctypes.c_int, [vp, vp, vp]),
    "gpk_kernel_matrix": (ctypes.c_int, [vp, i64, vp, i64, i64, c_double_p, ctypes.c_int, vp, i64, vp]),
    "gpk_factorize": (ctypes.c_int, [vp, c_double_p, ctypes.c_int]),
    "gpk_factorize_matrix": (ctypes.c_int, [vp, vp, i64, ctypes.c_int]),
    "gpk_nll_matrix": (ctypes.c_int, [vp, c_double_p]),
    "gpk_logdet": (ctypes.c_int, [vp, c_double_p]),
    "gpk_nll_grad": (ctypes.c_int, [vp, c_double_p, c_double_p, c_double_p, ctypes.c_int]),
    "gpk_grad_trace_partial": (ctypes.c_int, [vp, i64, i64, c_double_p]),
    "gpk_solve": (ctypes.c_int, [vp, vp, i64, vp]),
    "gpk_inverse": (ctypes.c_int, [vp, vp, i64]),
    "gpk_solve_residual": (ctypes.c_int, [vp, c_double_p]),
    "gpk_get_alpha": (ctypes.c_int, [vp, vp]),
    "gpk_import_state": (ctypes.c_int, [vp, c_double_p, vp, ctypes.c_int]),
    "gpk_predict": (ctypes.c_int, [vp, vp, i64, ctypes.c_double, vp, vp, ctypes.c_int]),
    "gpk_predict_cross": (ctypes.c_int, [vp, vp, i64, i64, vp, ctypes.c_double, vp, vp]),
    "gpk_predict_cov": (ctypes.c_int, [vp, vp, i64, vp, i64, vp, i64]),
    "gpk_predict_cov_cross": (ctypes.c_int, [vp, vp, i64, i64, vp, i64, i64, vp, i64, vp, i64]),
    "gpk_predict_grad": (ctypes.c_int, [vp, vp, i64, ctypes.c_double, vp, vp, vp, vp]),
    "gpk_propagate_ga": (ctypes.c_int, [vp, vp, vp, i64, ctypes.c_int, ctypes.c_double, vp, vp]),
    "gpk_propagate_ga_parts": (ctypes.c_int, [vp, vp, vp, i64, ctypes.c_int, vp, vp]),
    "gpk_propagate_exact": (ctypes.c_int, [vp, vp, vp, vp, vp, i64, ctypes.c_double, vp, vp]),
    "gpk_set_kernel": (ctypes.c_int, [vp, ctypes.c_int]),
    "gpk_kernel_matrix_periodic": (ctypes.c_int, [vp, i64, vp, i64, i64, c_double_p, ctypes.c_int, vp, i64, vp]),
    "gpk_set_route": (ctypes.c_int, [vp, ctypes.c_int, i64, ctypes.c_int, i64]),
    "gpk_get_route": (ctypes.c_int, [vp, c_int_p]),
    "gpk_set_batch_rows": (ctypes.c_int, [vp, i64]),
}

# measurement / test hooks (include/gpk_test.h): bound for tests/ and bench.py, never called by the product layer
TEST_SIGNATURES = {
    "gpk_test_potrf_inv": (ctypes.c_int, [vp, vp, i64, i64, vp, c_int_p, vp]),
    "gpk_test_oz_residues": (ctypes.c_int, [vp, i64, i64, i64, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp]),
    "gpk_test_oz_gemm": (ctypes.c_int, [vp, i64, ctypes.c_int, ctypes.c_int, vp, i64, ctypes.c_int, ctypes.c_int, vp, i64,
                                        i64, i64, i64, ctypes.c_double, ctypes.c_double, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_int, i64, ctypes.c_int, ctypes.POINTER(ctypes.c_float), vp]),
    "gpk_test_overlap": (ctypes.c_int, [ctypes.c_int]),
    "gpk_test_poison": (ctypes.c_int, [ctypes.c_int]),
    "gpk_test_position_lock": (ctypes.c_int, [ctypes.c_int]),
    "gpk_profile": (ctypes.c_int, [ctypes.c_int]),
    "gpk_profile_read": (ctypes.c_int, [c_double_p, ctypes.POINTER(i64), ctypes.POINTER(i64), c_double_p]),
    "gpk_microbench_i8": (ctypes.c_int, [i64, ctypes.c_double, c_double_p]),
}


class GpkError(RuntimeError):
    pass


def lib_path():
    return _LIB_PATH


def load():
    """Load libgpk.so and declare every prototype. Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise GpkError(
            "libgpk.so not found at %s: build it with `python scikit-gpuppy_b200/build_native.py` "
            "(there is no CPU fallback)" % _LIB_PATH)
    lib = ctypes.CDLL(_LIB_PATH)
    for name, (res, args) in list(SIGNATURES.items()) + list(TEST_SIGNATURES.items()):
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().gpk_last_error().decode("utf-8", "replace")


def check(rc, what=""):
    """0 -> ok; k>0 -> LinAlgError (not positive definite); <0 -> GpkError (-4: the INT8 workspace does not fit)."""
    if rc == 0:
        return
    if rc > 0:
        raise np.linalg.LinAlgError("%s: leading minor %d of K is not positive definite" % (what, rc))
    raise GpkError("%s failed (%d): %s" % (what, rc, last_error()))


def theta_ptr(theta):
    th = np.ascontiguousarray(np.asarray(theta, dtype=np.float64))
    return th, th.ctypes.data_as(c_double_p)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise GpkError("no CUDA device: the skgpuppy B200 path has no CPU fallback")
    return torch


def ptr(t):
    """Device pointer of a contiguous float64 CUDA tensor (or None)."""
    if t is None:
        return None
    assert t.is_cuda and t.dtype.is_floating_point and t.element_size() == 8 and t.is_contiguous()
    return ctypes.c_void_p(t.data_ptr())


def current_stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
