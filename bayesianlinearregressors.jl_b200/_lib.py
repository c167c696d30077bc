"""ctypes binding of libblr_cuda (include/blr_cuda.h).

This is the same symbol set the Julia glue `ccall`s (julia/src/libblr.jl); Python stands in for Julia because
there is no Julia toolchain in this image.  There is deliberately NO fallback: if the shared library is
missing, fails to load, or no sm_100 device is present, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
LIB_PATH = os.path.join(CSRC, "libblr_cuda.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "blr_cuda.h")

# error codes (include/blr_cuda.h)
E_INVALID, E_CUDA, E_NCCL, E_DIM, E_NODEVICE, E_NOMEM = -1, -2, -3, -4, -5, -6
COLVECS, ROWVECS = 0, 1
LAMBDA_DIAGONAL, LAMBDA_DENSE = 0, 1
NOISE_SCALAR, NOISE_VECTOR, NOISE_DENSE = 0, 1, 2

c_double_p = C.POINTER(C.c_double)
c_void_pp = C.POINTER(C.c_void_p)


class Prior(C.Structure):
    _fields_ = [("mw", c_double_p), ("lambda_kind", C.c_int), ("lambda_", c_double_p), ("ld", C.c_int64), ("D", C.c_int64)]


class Noise(C.Structure):
    _fields_ = [("kind", C.c_int), ("scalar", C.c_double), ("vec", C.c_void_p), ("dense", C.c_void_p), ("dense_ld", C.c_int64)]


class LogpdfGrads(C.Structure):
    """blr_logpdf_grads: NULL fields are not computed."""

    _fields_ = [("dmw", c_double_p), ("dlambda", c_double_p), ("dsigma2", c_double_p), ("dsigma2_dev", C.c_void_p),
                ("dy_dev", C.c_void_p), ("dX_dev", C.c_void_p), ("ld_dX", C.c_int64)]


# name -> (restype, argtypes); every symbol include/blr_cuda.h declares (checked by tests/test_abi.py)
SIGNATURES = {
    "blr_version": (C.c_int, []),
    "blr_ctx_create": (C.c_int, [c_void_pp, C.c_int]),
    "blr_ctx_destroy": (C.c_int, [C.c_void_p]),
    "blr_last_error": (C.c_char_p, [C.c_void_p]),
    "blr_ctx_sync": (C.c_int, [C.c_void_p]),
    "blr_ctx_stream": (C.c_int, [C.c_void_p, c_void_pp]),
    "blr_ctx_set_form": (C.c_int, [C.c_void_p, C.c_int]),
    "blr_ctx_get_form": (C.c_int, [C.c_void_p, C.POINTER(C.c_int)]),
    "blr_ctx_wait_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_stream_wait_ctx": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_launch_count": (C.c_int64, [C.c_void_p]),
    "blr_last_timings": (C.c_int, [C.c_void_p, c_double_p]),
    "blr_host_alloc": (C.c_int, [C.c_void_p, C.c_int64, c_void_pp]),
    "blr_host_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_nccl_unique_id": (C.c_int, [C.c_void_p]),
    "blr_comm_init_rank": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int]),
    "blr_comm_destroy": (C.c_int, [C.c_void_p]),
    "blr_x_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, c_void_pp]),
    "blr_x_wrap_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, c_void_pp]),
    "blr_x_alloc": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int, c_void_pp]),
    "blr_x_device_ptr": (C.c_int, [C.c_void_p, C.c_void_p, c_void_pp, C.POINTER(C.c_int64)]),
    "blr_x_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_vec_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, c_void_pp]),
    "blr_vec_wrap_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, c_void_pp]),
    "blr_vec_alloc": (C.c_int, [C.c_void_p, C.c_int64, c_void_pp]),
    "blr_vec_device_ptr": (C.c_int, [C.c_void_p, C.c_void_p, c_void_pp]),
    "blr_vec_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "blr_vec_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_x_synth": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64]),
    "blr_vec_synth_noise": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64]),
    "blr_vec_synth_targets": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64, C.c_void_p]),
    "blr_x_rff": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, c_void_pp]),
    "blr_x_features": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_double, c_void_pp]),
    "blr_x_features_vjp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_void_p,
                                     C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "blr_stats_create": (C.c_int, [C.c_void_p, C.c_int64, c_void_pp]),
    "blr_stats_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_stats_zero": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_stats_accumulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Noise)]),
    "blr_stats_accumulate_host": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_void_p, C.c_int,
         C.c_double, C.c_void_p, C.c_int64],
    ),
    "blr_stats_allreduce": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_stats_allreduce_all": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int]),
    "blr_comm_init_all": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "blr_stats_device_ptr": (C.c_int, [C.c_void_p, C.c_void_p, c_void_pp, C.POINTER(C.c_int64)]),
    "blr_stats_download": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "blr_stats_upload": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "blr_infer_from_stats": (
        C.c_int,
        [C.c_void_p, C.POINTER(Prior), C.c_void_p, c_double_p, C.c_void_p, C.c_void_p, C.c_void_p, c_void_pp],
    ),
    "blr_logpdf_multi": (C.c_int, [C.c_void_p, C.POINTER(Prior), C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.POINTER(Noise),
                                  C.c_void_p]),
    "blr_logpdf_grad": (C.c_int, [C.c_void_p, C.POINTER(Prior), C.c_void_p, C.c_void_p, C.POINTER(Noise), c_double_p,
                                  C.POINTER(LogpdfGrads)]),
    "blr_logpdf_multi_grad": (C.c_int, [C.c_void_p, C.POINTER(Prior), C.c_void_p, C.c_void_p, C.c_int64, C.c_int64,
                                        C.POINTER(Noise), c_double_p, c_double_p, C.POINTER(LogpdfGrads)]),
    "blr_infer": (
        C.c_int,
        [C.c_void_p, C.POINTER(Prior), C.c_void_p, C.c_void_p, C.POINTER(Noise), c_double_p, C.c_void_p, C.c_void_p,
         C.c_void_p, c_void_pp],
    ),
    "blr_post_create": (C.c_int, [C.c_void_p, C.POINTER(Prior), C.c_int64, c_void_pp]),
    "blr_post_free": (C.c_int, [C.c_void_p, C.c_void_p]),
    "blr_post_dim": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "blr_mean_var": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Noise), C.c_void_p, C.c_void_p]),
    "blr_mean_var_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Noise), C.c_void_p, C.c_void_p]),
    "blr_cov": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Noise), C.c_void_p]),
    "blr_rand_finite": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Noise), C.c_int64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p],
    ),
    "blr_rand_finite_dev": (
        C.c_int,
        [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(Noise), C.c_int64, C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p],
    ),
    "blr_rand_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_uint64, C.c_void_p]),
    "blr_apply_weights": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "blr_calibrate_dmma": (C.c_int, [C.c_void_p, c_double_p]),
    "blr_calibrate_dmma_cfg": (C.c_int, [C.c_void_p, C.c_int, C.c_int, c_double_p]),
    "blr_calibrate_gram_inner": (C.c_int, [C.c_void_p, c_double_p]),
    "blr_calibrate_mixed": (C.c_int, [C.c_void_p, c_double_p]),
    "blr_calibrate_dfma": (C.c_int, [C.c_void_p, c_double_p]),
    "blr_calibrate_hbm": (C.c_int, [C.c_void_p, c_double_p]),
}

_lib = None


def build(verbose: bool = False) -> str:
    """Compile libblr_cuda.so in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j", str(min(8, os.cpu_count() or 1))]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        sys.stderr.write(res.stdout[-4000:] + "\n" + res.stderr[-4000:] + "\n")
        raise RuntimeError("building libblr_cuda.so failed")
    if verbose:
        print(res.stdout[-2000:])
    return LIB_PATH


def load():
    """dlopen the library and attach prototypes.  Raises if the extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    # LIBBLR_CUDA=<path>: load another build of the SAME library (the strict-arrive sanitizer variant, `make strict`);
    # the same variable names the library in the Julia glue (julia/src/libblr.jl)
    path = os.environ.get("LIBBLR_CUDA") or LIB_PATH
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: the CUDA extension has not been built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`).  There is no CPU fallback."
        )
    lib = C.CDLL(path, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class BLRError(RuntimeError):
    """Argument / CUDA / NCCL failure reported by libblr_cuda (Julia side: ErrorException)."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"libblr_cuda error {code}: {msg}")
        self.code = code


class DimensionMismatch(BLRError):
    """length(y) != size(X, 2)  (src/bayesian_linear_regression.jl:74 throws an ErrorException)."""


class PosDefException(ArithmeticError):
    """LinearAlgebra.PosDefException(info): Cholesky hit a non-positive pivot of order `info`."""

    def __init__(self, info: int):
        super().__init__(f"matrix is not positive definite; Cholesky factorization failed (info={info})")
        self.info = info
