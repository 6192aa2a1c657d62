"""ctypes binding of libpigp.so (the C ABI declared in include/pigp.h).

There is no CPU fallback: if the library is missing or no CUDA device is
present, calls fail loudly.
"""
import ctypes as C
import os

MAX_TERMS = 8
MAX_GROUPS = 4
TILE = 128
LAYOUT_FULL, LAYOUT_LOWER = 0, 1
IPC_HANDLE_BYTES = 64
ABI_VERSION = 3
MAX_BATCH = 65535
KERNEL_TYPES = {"se": 0, "mt52": 52, "mt72": 72, "mt92": 92}

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PIGP_LIB") or os.path.join(_HERE, "libpigp.so")  # PIGP_LIB: alternate build (kernel tuning only)


class Term(C.Structure):
    _fields_ = [("group", C.c_int32), ("order", C.c_int32 * 3), ("coef", C.c_double)]


class BlockDesc(C.Structure):
    _fields_ = [("n_terms", C.c_int32), ("shift_first", C.c_int32), ("shift_second", C.c_int32),
                ("reserved", C.c_int32), ("terms", Term * MAX_TERMS)]


class PlanDesc(C.Structure):
    _fields_ = [("dim", C.c_int32), ("product_form", C.c_int32), ("n_groups", C.c_int32), ("symmetric", C.c_int32),
                ("n_row_blocks", C.c_int32), ("n_col_blocks", C.c_int32),
                ("sec_row", C.POINTER(C.c_int64)), ("sec_col", C.POINTER(C.c_int64)),
                ("pts_row_host", C.POINTER(C.c_double)), ("pts_col_host", C.POINTER(C.c_double)),
                ("table", C.POINTER(BlockDesc)), ("lbox", C.c_double * 3),
                ("noise_lo_block", C.c_int32), ("noise_hi_block", C.c_int32), ("kernel_type", C.c_int32),
                ("reserved", C.c_int32)]


class PigpError(RuntimeError):
    pass


_lib = None

_SIGNATURES = {
    "pigp_abi_version": (C.c_int, []),
    "pigp_last_error": (C.c_char_p, []),
    "pigp_set_device": (C.c_int, [C.c_int]),
    "pigp_plan_create": (C.c_int, [C.POINTER(PlanDesc), C.POINTER(C.c_void_p)]),
    "pigp_plan_destroy": (None, [C.c_void_p]),
    "pigp_plan_rows": (C.c_int64, [C.c_void_p]),
    "pigp_plan_cols": (C.c_int64, [C.c_void_p]),
    "pigp_plan_theta_len": (C.c_int32, [C.c_void_p]),
    "pigp_plan_set_points_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "pigp_assemble": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pigp_assemble_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_int]),
    "pigp_assemble_diag": (C.c_int, [C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p]),
    "pigp_solver_create": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "pigp_solver_destroy": (None, [C.c_void_p]),
    "pigp_solver_create_dist": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "pigp_solver_dsolver": (C.c_void_p, [C.c_void_p]),
    "pigp_nll": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pigp_nll_grad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pigp_nll_grad_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p]),
    "pigp_nll_grad_batch": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p]),
    "pigp_nll_grad_batch_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "pigp_predict": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p,
                               C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "pigp_predict_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p,
                                    C.c_void_p, C.c_int, C.c_void_p]),
    "pigp_predict_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double,
                                          C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    "pigp_adam_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_double, C.c_double,
                                 C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "pigp_adam_batch_host": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_double, C.c_double,
                                       C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "pigp_potrf_lower": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pigp_potri_lower": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pigp_dgemm": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int64,
                             C.c_int, C.c_double, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "pigp_assemble_owned": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_int64,
                                      C.c_void_p]),
    "pigp_trace_grad": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                  C.c_void_p]),
    "pigp_dsolver_create": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "pigp_dsolver_destroy": (None, [C.c_void_p]),
    "pigp_dsolver_slab": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_int64)]),
    "pigp_dsolver_ipc_handle": (C.c_int, [C.c_void_p, C.c_void_p]),
    "pigp_ipc_open": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "pigp_ipc_close": (C.c_int, [C.c_void_p]),
    "pigp_dsolver_connect": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "pigp_dsolver_set_shared_device": (C.c_int, [C.c_void_p, C.c_int]),
    "pigp_device_uuid": (C.c_int, [C.c_void_p]),
    "pigp_dsolver_nll_grad": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p,
                                        C.c_void_p]),
    "pigp_dsolver_nll_grad_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p,
                                             C.c_void_p]),
    "pigp_dsolver_reset": (C.c_int, [C.c_void_p]),
    "pigp_launch_count": (C.c_int64, []),
    "pigp_set_side_stream": (C.c_int, [C.c_int]),
    "pigp_set_lookahead": (C.c_int, [C.c_int]),
    "pigp_debug_potf2_stamps": (C.c_int, [C.c_void_p]),
    "pigp_profile_start": (C.c_int, []),
    "pigp_profile_stop": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
}
PROF_CLASSES = ("assemble", "gemm", "potf2", "gradient", "misc")
EXPORTS = tuple(_SIGNATURES)


def lib():
    """The loaded library (raises PigpError when it has not been built)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise PigpError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                            "(there is no CPU fallback)")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.pigp_abi_version() != ABI_VERSION:
            raise PigpError("libpigp.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc):
    if rc != 0:
        msg = lib().pigp_last_error()
        raise PigpError(f"pigp error {rc}: {msg.decode() if msg else ''}")


def launch_count():
    return int(lib().pigp_launch_count())


def profile_start():
    check(lib().pigp_profile_start())


def profile_stop():
    """-> {class: dict(ms=, launches=, flops=)} for the launches since profile_start()."""
    n = len(PROF_CLASSES)
    ms, cnt, fl = (C.c_double * n)(), (C.c_int64 * n)(), (C.c_double * n)()
    check(lib().pigp_profile_stop(ms, cnt, fl))
    return {name: dict(ms=ms[i], launches=int(cnt[i]), flops=fl[i]) for i, name in enumerate(PROF_CLASSES)}
