"""ctypes loader of the C-ABI library (csrc/libcv_b200.so, include/cv_b200.h).

There is no CPU fallback: if the shared library is missing this raises, and if
no CUDA device is present every compute entry point returns CV_ERR_CUDA, which
`check()` turns into an exception.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
# CV_B200_SO: development override (tools/ A/B runs of differently compiled builds); the product is the in-tree library
SO_PATH = os.environ.get("CV_B200_SO") or os.path.join(CSRC, "libcv_b200.so")

OK, ERR_EMPTY, ERR_NAN, ERR_ARG, ERR_ASSERT, ERR_CUDA, ERR_OOM, ERR_UNSUPPORTED = range(8)
_NAMES = {1: "EMPTY", 2: "NAN", 3: "ARG", 4: "ASSERT", 5: "CUDA", 6: "OOM", 7: "UNSUPPORTED"}


class CvError(RuntimeError):
    """Non-zero status from the C ABI. `.code` is the CV_ERR_* value; where the
    reference would panic (unwrap/assert/index) the code says which panic."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"CV_ERR_{_NAMES.get(code, code)}: {msg}")
        self.code = code


def build(force: bool = False, variant: int | None = None) -> str:
    """Compile csrc/ for sm_100a with nvcc (in-tree, so the .so travels to the GPU box)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".inl"))]
    srcs += [os.path.join(_HERE, "..", "include", f) for f in ("cv_b200.h", "cv_b200_debug.h")]
    stale = (not os.path.exists(SO_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(SO_PATH) for s in srcs)
    if force or stale:
        cmd = ["make", "-C", CSRC, "-s", "-B", "-j4"]
        if variant is not None:
            cmd.append(f"VARIANT={variant}")
        subprocess.check_call(cmd)
    return SO_PATH


_lib = None

_dp, _u32p, _i64p, _u64p, _u8p, _i32p = (
    C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.POINTER(C.c_int64),
    C.POINTER(C.c_uint64), C.POINTER(C.c_uint8), C.POINTER(C.c_int32),
)

# name -> (restype, argtypes); mirrors include/cv_b200.h (the drop-in boundary) one to one
SIGNATURES = {
    "cv_hmm_create": (C.c_int, [C.c_int, C.c_int, _u64p, _dp, _dp, _dp, C.c_int, C.POINTER(C.c_void_p)]),
    "cv_hmm_destroy": (None, [C.c_void_p]),
    "cv_hmm_nstates": (C.c_int, [C.c_void_p]),
    "cv_hmm_nobs": (C.c_int64, [C.c_void_p]),
    "cv_decode_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cv_decode_batch_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cv_decode_batch_dev_f32": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "cv_decode_batch_u16u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "cv_decode_batch_keep": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "cv_decode_batch_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "cv_decode_batch_dev_u8": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "cv_cp_solve": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64,
                              C.c_void_p, _dp, _u64p, _u64p]),
    "cv_cp_dist_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_int64, C.c_void_p, C.POINTER(C.c_void_p)]),
    "cv_cp_dist_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "cv_cp_dist_destroy": (None, [C.c_void_p]),
    "cv_cp_solve_dist": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_uint64,
                                   C.c_void_p, _dp, _u64p, _u64p]),
    "cv_cp_plan_cuts": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "cv_cfn_tables": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                C.c_void_p, _dp, _i64p, _dp]),
    "cv_mle": (C.c_int, [C.c_int, C.c_int, _u64p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                         C.c_void_p, C.c_int64, C.c_int, _dp]),
    "cv_baum_welch": (C.c_int, [C.c_int, C.c_int, _u64p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int64, C.c_int, C.c_double, C.c_int, _dp, C.POINTER(C.c_int), _i64p, _dp]),
    "cv_last_error": (C.c_char_p, []),
    "cv_launch_count": (C.c_uint64, []),
    "cv_set_timing": (None, [C.c_int]),
    "cv_last_kernel_ms": (C.c_double, [C.c_void_p]),
    "cv_last_backtrace_ms": (C.c_double, [C.c_void_p]),
    "cv_host_alloc": (C.c_void_p, [C.c_uint64]),
    "cv_host_free": (None, [C.c_void_p]),
}

# test / bench hooks, include/cv_b200_debug.h
DEBUG_SIGNATURES = {
    "cv_debug_cp_last_state": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "cv_debug_cp_last_ub": (C.c_int, [C.c_void_p, C.c_void_p, C.c_uint64, _u64p]),
    "cv_debug_ordered_sum": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, _dp]),
    "cv_debug_set_small_config": (None, [C.c_int]),
    "cv_debug_set_chunks": (None, [C.c_int]),
    "cv_debug_set_chain_max_batch": (None, [C.c_longlong]),
    "cv_debug_set_pipeline": (None, [C.c_int, C.c_int]),
    "cv_debug_probe_fp64": (C.c_int, [C.c_int, C.c_int, C.c_int, _dp, _dp]),
    "cv_debug_set_balanced_split": (None, [C.c_int]),
    "cv_debug_set_fwd_ldc": (None, [C.c_int]),
    "cv_debug_set_em_light": (None, [C.c_int]),
    "cv_debug_set_bt_split": (None, [C.c_int]),
    "cv_debug_set_uneven_chunks": (None, [C.c_int]),
    "cv_debug_set_prefilter": (None, [C.c_int]),
    "cv_debug_set_large_group_rb": (None, [C.c_longlong]),
    "cv_debug_set_cp_leaf_batch": (None, [C.c_int]),
}


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise ImportError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback."
            )
        L = C.CDLL(SO_PATH)
        for name, (res, args) in {**SIGNATURES, **DEBUG_SIGNATURES}.items():
            fn = getattr(L, name)  # AttributeError if the .so does not export a declared symbol
            fn.restype, fn.argtypes = res, args
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise CvError(rc, lib().cv_last_error().decode("utf-8", "replace"))
