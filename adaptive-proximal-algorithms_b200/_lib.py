"""ctypes binding of libadaprox_cuda.so (include/adaprox.h).

The product path has no CPU fallback: if the shared library is missing or no
CUDA device is usable, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ADAPROX_LIB") or os.path.join(_HERE, "libadaprox_cuda.so")   # ADAPROX_LIB: A/B builds

c_id = C.c_int64
c_dp = C.POINTER(C.c_double)


class Prox(C.Structure):
    _fields_ = [("kind", C.c_int32), ("conjugate", C.c_int32), ("lam", C.c_double), ("lo", C.c_double),
                ("hi", C.c_double), ("lo_vec", c_id), ("hi_vec", c_id), ("shift", c_id)]


class Problem(C.Structure):
    _fields_ = [("f_kind", C.c_int32), ("f_ipar", C.c_int32), ("f_mat", c_id), ("f_vec", c_id), ("f_c", C.c_double),
                ("g", Prox), ("h", Prox), ("A_mat", c_id), ("n", C.c_int64), ("m_dual", C.c_int64)]


class Options(C.Structure):
    _fields_ = [("solver", C.c_int32), ("rule", C.c_int32), ("gamma", C.c_double), ("t", C.c_double),
                ("norm_A", C.c_double), ("delta", C.c_double), ("Theta", C.c_double), ("xi", C.c_double),
                ("nu", C.c_double), ("r", C.c_double), ("R", C.c_double), ("eta", C.c_double),
                ("shrink", C.c_double), ("sigma", C.c_double), ("muf", C.c_double), ("mug", C.c_double),
                ("theta", C.c_double), ("gamma_max", C.c_double), ("phi", C.c_double), ("tol", C.c_double),
                ("maxit", C.c_int64), ("want_objective", C.c_int32), ("counting_f", C.c_int32),
                ("counting_g", C.c_int32), ("counting_h", C.c_int32), ("counting_A", C.c_int32),
                ("max_records", C.c_int64)]


class Record(C.Structure):
    _fields_ = [("it", C.c_int64), ("gamma", C.c_double), ("sigma", C.c_double), ("norm_res", C.c_double),
                ("f_x", C.c_double), ("g_x", C.c_double), ("h_Ax", C.c_double), ("f_evals", C.c_int64),
                ("grad_f_evals", C.c_int64), ("prox_g_evals", C.c_int64), ("prox_h_evals", C.c_int64),
                ("A_evals", C.c_int64), ("At_evals", C.c_int64)]


class Result(C.Structure):
    _fields_ = [("iters", C.c_int64), ("flags", C.c_uint32), ("reserved", C.c_int32), ("f_evals", C.c_int64),
                ("grad_f_evals", C.c_int64), ("prox_g_evals", C.c_int64), ("prox_h_evals", C.c_int64),
                ("A_evals", C.c_int64), ("At_evals", C.c_int64), ("n_records", C.c_int64),
                ("final_gamma", C.c_double), ("final_sigma", C.c_double), ("final_norm_res", C.c_double),
                ("solve_ms", C.c_double), ("kernel_launches", C.c_int64),
                ("matrix_passes", C.c_int64), ("collective", C.c_int64)]


# enum values of include/adaprox.h
F_ZERO, F_LEAST_SQUARES, F_LOGISTIC, F_QUADRATIC, F_CUBIC, F_WORST_QUADRATIC, F_SIMPLE2D, F_QUADRATIC_GRAM = range(8)
P_ZERO, P_IND_ZERO, P_NORM_L1, P_NORM_L2, P_IND_BOX = range(5)
(S_ADAPTIVE_PRIMAL_DUAL, S_ADAPTIVE_PROXGRAD, S_LINESEARCH_PRIMAL_DUAL, S_BACKTRACKING_PROXGRAD,
 S_BACKTRACKING_NESTEROV, S_FIXED_NESTEROV, S_MALITSKY_POCK, S_AGRAAL) = range(8)
RULE_FIXED, RULE_MM, RULE_OUR, RULE_OUR_PLUS = range(4)
FLAG_CONVERGED, FLAG_STEP_TOO_SMALL, FLAG_NONFINITE, FLAG_LS_CAP, FLAG_COMM = 1, 2, 4, 8, 16

# every symbol include/adaprox.h declares: name -> (restype, argtypes)
_h = C.c_void_p
SYMBOLS = {
    "adaprox_version": (C.c_int, []),
    "adaprox_create": (C.c_int, [C.POINTER(_h), C.c_int]),
    "adaprox_destroy": (C.c_int, [_h]),
    "adaprox_last_error": (C.c_char_p, [_h]),
    "adaprox_device_info": (C.c_int, [_h, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "adaprox_matrix_upload_colmajor": (C.c_int, [_h, c_dp, C.c_int64, C.c_int64, C.c_int64, C.POINTER(c_id)]),
    "adaprox_matrix_upload_rowmajor": (C.c_int, [_h, c_dp, C.c_int64, C.c_int64, C.c_int64, C.POINTER(c_id)]),
    "adaprox_matrix_upload_csr": (C.c_int, [_h, C.c_int64, C.c_int64, C.c_int64, C.POINTER(C.c_int64),
                                            C.POINTER(C.c_int32), c_dp, C.POINTER(c_id)]),
    "adaprox_matrix_free": (C.c_int, [_h, c_id]),
    "adaprox_matrix_shape": (C.c_int, [_h, c_id, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "adaprox_vector_upload": (C.c_int, [_h, c_dp, C.c_int64, C.POINTER(c_id)]),
    "adaprox_vector_download": (C.c_int, [_h, c_id, c_dp, C.c_int64]),
    "adaprox_vector_free": (C.c_int, [_h, c_id]),
    "adaprox_generate_planted_lasso": (C.c_int, [_h, C.c_int64, C.c_int64, C.c_int64, C.c_int64, C.c_double, C.c_uint64,
                                                 C.c_double, C.c_double, C.c_int32, C.POINTER(c_id), C.POINTER(c_id),
                                                 c_dp, c_dp, c_dp]),
    "adaprox_mul": (C.c_int, [_h, c_id, c_dp, c_dp]),
    "adaprox_amul": (C.c_int, [_h, c_id, c_dp, c_dp]),
    "adaprox_eval_f": (C.c_int, [_h, C.POINTER(Problem), c_dp, c_dp, c_dp]),
    "adaprox_prox_eval": (C.c_int, [_h, C.POINTER(Prox), c_dp, C.c_int64, C.c_double, c_dp, c_dp]),
    "adaprox_stepsize": (C.c_int, [C.POINTER(Options), C.c_double, C.c_double, C.c_double, C.c_double, C.c_double,
                                   c_dp, c_dp, c_dp]),
    "adaprox_logistic_grad_hessian": (C.c_int, [_h, c_id, c_id, c_dp, c_dp, c_dp]),
    "adaprox_solve": (C.c_int, [_h, C.POINTER(Problem), C.POINTER(Options), c_dp, c_dp, c_dp, c_dp,
                                C.POINTER(Record), C.POINTER(Result)]),
    "adaprox_solve_lambda_path": (C.c_int, [_h, C.POINTER(Problem), C.POINTER(Options), C.c_int64, c_dp, c_dp, c_dp, c_dp,
                                            C.POINTER(C.c_int64), c_dp, c_dp, c_dp, c_dp, C.c_int64, C.POINTER(Result)]),
    "adaprox_solve_box_path": (C.c_int, [_h, C.POINTER(Problem), C.POINTER(Options), C.c_int64, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp,
                                         C.POINTER(C.c_int64), c_dp, c_dp, c_dp, c_dp, c_dp, C.c_int64, C.POINTER(Result)]),
    "adaprox_solve_pd_lambda_path": (C.c_int, [_h, C.POINTER(Problem), C.POINTER(Options), C.c_int64, c_dp, c_dp, c_dp, c_dp, c_dp,
                                               c_dp, C.POINTER(C.c_int64), c_dp, c_dp, c_dp, c_dp, C.c_int64, C.POINTER(Result)]),
    "adaprox_time_path_gemm":(C.c_int, [_h, c_id, C.c_int64, C.c_int, C.c_int, c_dp]),
    "adaprox_comm_unique_id": (C.c_int, [C.c_void_p]),
    "adaprox_comm_init": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p]),
    "adaprox_comm_info": (C.c_int, [_h, C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "adaprox_p2p_export": (C.c_int, [_h, C.c_int64, C.c_void_p]),
    "adaprox_p2p_attach": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p]),
    "adaprox_p2p_reset": (C.c_int, [_h]),
    "adaprox_matrix_set_shard": (C.c_int, [_h, c_id, C.c_int64, C.c_int64]),
    "adaprox_time_kernel": (C.c_int, [_h, c_id, C.c_int, C.c_int, c_dp]),
}

_lib = None


def load():
    """Load the shared library and type every symbol.  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)          # AttributeError if the header and the library disagree
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class AdaproxError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"adaprox status {code}: {msg}")
        self.code = code
