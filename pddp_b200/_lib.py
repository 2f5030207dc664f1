"""ctypes binding of the C-ABI library (include/pddp_b200.h -> pddp_b200/lib/libpddp_b200.so).

There is no CPU fallback: if the library is missing or a call fails this module raises."""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PDDP_B200_LIB") or os.path.join(_HERE, "lib", "libpddp_b200.so")   # (override: A/B experiment builds)

F32, F64 = 0, 1
PROBLEM_MAJOR, BATCH_INNER = 0, 1
GEO_PENDULUM, GEO_CARTPOLE, GEO_DOUBLE_CARTPOLE, GEO_RENDEZVOUS = 0, 1, 2, 3
MAX_DA, MAX_NU = 8, 4
STATUS_NOT_PD, STATUS_NAN = 1, 2
BNN_INPUT_INFER, BNN_INPUT_RESAMPLE, BNN_INPUT_MEAN = 0, 1, 2

GEO_INFO = {  # geo -> (D, nu, angular, non-angular)
    GEO_PENDULUM: (2, 1, (0,), (1,)),
    GEO_CARTPOLE: (4, 1, (2,), (0, 1, 3)),
    GEO_DOUBLE_CARTPOLE: (6, 1, (2, 4), (0, 1, 3, 5)),
    GEO_RENDEZVOUS: (8, 4, (), tuple(range(8))),       # ref: examples/rendezvous (known dynamics and BNN)
}


class Shape(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("dtype", "layout", "geo", "enc", "B", "N", "nz", "nu")]


class Cost(C.Structure):
    _fields_ = [("Q", C.c_double * (MAX_DA * MAX_DA)), ("Q_term", C.c_double * (MAX_DA * MAX_DA)),
                ("R", C.c_double * (MAX_NU * MAX_NU)), ("x_goal", C.c_double * MAX_DA),
                ("u_goal", C.c_double * MAX_NU)]


class KnownDynamics(C.Structure):
    _fields_ = [("p", C.c_double * 8)]


class BNN(C.Structure):
    _fields_ = [("P", C.c_int32), ("H0", C.c_int32), ("H1", C.c_int32)] + [
        (n, C.c_void_p) for n in ("W0", "b0", "W1", "b1", "W2", "b2", "mask0", "mask1", "eps0",
                                  "X_mean", "X_std_inv", "dX_mean", "dX_std")] + [
        ("input_mode", C.c_int32), ("eps_in", C.c_void_p), ("eps_out", C.c_void_p), ("independent_noise", C.c_int32)]


_P = C.c_void_p
_SIGNATURES = {
    "pddp_version": (C.c_char_p, []),
    "pddp_last_error": (C.c_char_p, []),
    "pddp_linearize_known": (C.c_int, [C.POINTER(Shape), C.POINTER(KnownDynamics), C.POINTER(Cost)]
                             + [_P] * 17),
    "pddp_backward": (C.c_int, [C.POINTER(Shape)] + [_P] * 16),
    "pddp_rollout_known": (C.c_int, [C.POINTER(Shape), C.POINTER(KnownDynamics), C.POINTER(Cost)]
                           + [_P] * 5 + [C.c_int32] + [_P] * 10),
    "pddp_accept_update": (C.c_int, [C.POINTER(Shape)] + [_P] * 4 + [C.c_double, C.c_double]
                           + [_P] * 13),
    "pddp_cost_derivatives": (C.c_int, [C.POINTER(Shape), C.POINTER(Cost)] + [_P] * 11),
    "pddp_bnn_workspace_bytes": (C.c_int64, [C.POINTER(Shape), C.POINTER(BNN), C.c_int32]),
    "pddp_linearize_bnn": (C.c_int, [C.POINTER(Shape), C.POINTER(BNN), C.POINTER(Cost)] + [_P] * 16
                           + [_P, C.c_int64, _P]),
    "pddp_rollout_bnn": (C.c_int, [C.POINTER(Shape), C.POINTER(BNN), C.POINTER(Cost)] + [_P] * 5
                         + [C.c_int32] + [_P] * 10 + [_P, C.c_int64, _P]),
    "pddp_bnn_train_workspace_bytes": (C.c_int64, [_P]),
    "pddp_bnn_train": (C.c_int, [_P] * 12 + [_P, C.c_int64, _P]),
    "pddp_env_step_known": (C.c_int, [C.POINTER(Shape), C.POINTER(KnownDynamics)] + [_P] * 4),
    "pddp_profile_enable": (None, [C.c_int]),
    "pddp_profile_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "pddp_launch_count": (C.c_int64, []),
}
EXPORTS = tuple(_SIGNATURES)

_lib = None


def load():
    """Loads the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("pddp_b200: %s is missing -- build it with `python -c 'import "
                           "__graft_entry__ as g; g.build()'` (or make -C pddp_b200/csrc). "
                           "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), "pddp_b200: tensors passed to the C ABI must be contiguous"
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def check(code, what):
    if code != 0:
        msg = load().pddp_last_error().decode()
        raise RuntimeError("pddp_b200.%s failed (%d): %s" % (what, code, msg))


def dtype_code(dtype):
    if dtype == torch.float32:
        return F32
    if dtype == torch.float64:
        return F64
    raise TypeError("pddp_b200 supports float32 and float64, got %s" % dtype)


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError("pddp_b200: %s must live on a CUDA device (no CPU fallback)" % what)
