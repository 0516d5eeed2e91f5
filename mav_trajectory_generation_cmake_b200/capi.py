"""ctypes binding of libminsnap_b200.so (include/minsnap_b200.h).

The library is built in-tree by ``mav_trajectory_generation_cmake_b200.build`` and loaded
from ``lib/``.  There is no fallback: if the shared object is missing or the machine has no
CUDA device, loading / calling raises.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libminsnap_b200.so")

OK = 0
ERR_ARG, ERR_CUDA, ERR_UNSUPPORTED, ERR_NO_DEVICE, ERR_WORKSPACE = 1, 2, 3, 4, 5
STATUS_NONPOSITIVE_PIVOT, STATUS_BAD_TIME, STATUS_NONFINITE = 1, 2, 4

_vp, _i, _l, _d, _sz = C.c_void_p, C.c_int, C.c_long, C.c_double, C.c_size_t

# name -> (restype, argtypes); mirrors include/minsnap_b200.h one to one
SIGNATURES = {
    "minsnap_abi_version": (_i, []),
    "minsnap_error_string": (C.c_char_p, [_i]),
    "minsnap_last_cuda_error": (C.c_char_p, []),
    "minsnap_device_info": (_i, [_vp, _vp, _vp, _vp, _vp]),
    "minsnap_reorder": (_i, [_i, _i, _l, _vp, _vp, _vp, _vp]),
    "minsnap_estimate_segment_times": (_i, [_l, _i, _i, _vp, _d, _d, _d, _vp, _vp]),
    "minsnap_segment_matrices": (_i, [_l, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_solve_workspace_bytes": (_sz, [_i, _i]),
    "minsnap_solve": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "minsnap_coeffs_from_constraints": (_i, [_l, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "minsnap_cost": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "minsnap_solve_standard": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _d, _d, _d, _vp, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_sample_uniform": (_i, [_l, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp, _vp]),
    "minsnap_sample_at": (_i, [_l, _i, _i, _i, _vp, _vp, _i, _vp, _l, _i, _vp, _vp, _vp]),
    "minsnap_evaluate_range": (_i, [_l, _i, _i, _i, _vp, _vp, _d, _d, _d, _i, _i, _vp, _vp, _vp, _vp]),
    "minsnap_cost_sweep": (_i, [_l, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_extrema_max_roots": (_i, [_i, _i, _i]),
    "minsnap_extrema": (_i, [_l, _i, _i, _i, _vp, _vp, _i, _i, C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                             _vp]),
    "minsnap_extrema_host": (_i, [_l, _i, _i, _i, _vp, _vp, _i, _i, C.c_uint32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                                  _vp]),
    "minsnap_sample_uniform_host": (_i, [_l, _i, _i, _i, _vp, _vp, _i, _i, _vp, _vp]),
    "minsnap_cost_sweep_host": (_i, [_l, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_time_objective_host": (_i, [_l, _i, _i, _i, _i, _i, _vp, _vp, _vp, _d, _vp, _vp, _vp]),
    "minsnap_time_gradient_host": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _d, _d, _d, _vp, _vp]),
    "minsnap_collision_cost_host": (_i, [_l, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _i, _d, _d, _d, _d, _d, _vp,
                                         _vp, _vp]),
    "minsnap_time_objective": (_i, [_l, _i, _i, _i, _i, _i, _vp, _vp, _vp, _d, _vp, _vp, _vp, _vp]),
    "minsnap_time_gradient": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _d, _d, _d, _vp, _vp, _vp]),
    "minsnap_optimize_segment_times": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _i, _d, _i, _d, _d, _d, _vp, _vp]),
    "minsnap_soft_constraint_cost": (_i, [_l, _i, _i, _i, _vp, _vp, _i, _vp, _vp, _d, _d, _i, _vp, _vp, _vp, _vp]),
    "minsnap_time_objective_soft": (_i, [_l, _i, _i, _i, _i, _i, _vp, _vp, _vp, _d, _i, _vp, _vp, _d, _d, _i, _vp, _vp, _vp,
                                         _vp, _vp]),
    "minsnap_optimize_segment_times_soft": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _i, _d, _i, _d, _d, _d, _i, _vp, _vp, _d,
                                                 _d, _i, _vp, _vp, _vp]),
    "minsnap_collision_cost": (_i, [_l, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _i, _d, _d, _d, _d, _d, _vp, _vp,
                                    _vp, _vp]),
    "minsnap_collision_gradient": (_i, [_l, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _i, _d, _d, _d, _d, _d, _vp,
                                        _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_collision_gradient_host": (_i, [_l, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _d, _d, _vp, _vp, _i, _d, _d, _d, _d, _d,
                                             _vp, _i, _i, _vp, _vp, _vp, _vp]),
    "minsnap_derivative_gradient": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _sz, _vp]),
    "minsnap_derivative_gradient_host": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_free_objective": (_i, [_l, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _d, _d, _d, _vp, _vp, _vp, _d, _d, _vp, _vp,
                                    _i, _d, _d, _d, _d, _d, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_optimize_free_constraints": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _d, _d, _d, _vp, _vp, _vp, _d, _d,
                                               _vp, _vp, _i, _d, _d, _d, _d, _d, _i, _i, _d, _d, _d, _vp, _vp, _vp]),
    "minsnap_soft_constraint_gradient": (_i, [_l, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _vp, _d, _d, _i, _vp, _vp, _vp, _vp,
                                              _vp, _vp, _vp]),
    "minsnap_free_objective_soft": (_i, [_l, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _d, _d, _d, _vp, _vp, _vp, _d, _d, _vp,
                                         _vp, _i, _d, _d, _d, _d, _d, _i, _vp, _vp, _d, _d, _i, _d, _vp, _vp, _vp, _vp, _vp,
                                         _vp]),
    "minsnap_optimize_free_constraints_soft": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _i, _d, _d, _d, _vp, _vp, _vp, _d,
                                                    _d, _vp, _vp, _i, _d, _d, _d, _d, _d, _i, _vp, _vp, _d, _d, _i, _d, _i,
                                                    _i, _d, _d, _d, _vp, _vp, _vp, _vp]),
    "minsnap_host_alloc": (_i, [_vp, _sz]),
    "minsnap_host_free": (_i, [_vp]),
    "minsnap_reorder_host": (_i, [_i, _i, _l, _vp, _vp, _vp]),
    "minsnap_solve_host": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_solve_standard_host": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp, _d, _d, _d, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_sample_at_host": (_i, [_l, _i, _i, _i, _vp, _vp, _i, _vp, _l, _i, _vp, _vp]),
    "minsnap_evaluate_range_host": (_i, [_i, _i, _i, _vp, _vp, _d, _d, _d, _i, _i, _vp, _vp, _vp]),
    "minsnap_segment_matrices_host": (_i, [_l, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_estimate_segment_times_host": (_i, [_l, _i, _i, _vp, _d, _d, _d, _vp]),
    "minsnap_coeffs_from_constraints_host": (_i, [_l, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "minsnap_cost_host": (_i, [_l, _i, _i, _i, _i, _vp, _vp, _vp]),
    "minsnap_npy_write_f64": (_i, [C.c_char_p, _vp, _i, _vp]),
    "minsnap_npy_read_f64": (_i, [C.c_char_p, _vp, _sz, _vp, _vp]),
    "minsnap_sampled_table_rows": (_i, [_i, _vp, _d]),
    "minsnap_sampled_table_host": (_i, [_i, _i, _i, _vp, _vp, _d, _vp, _i, _vp, _vp]),
    "minsnap_table_write_text": (_i, [C.c_char_p, _vp, _i, _i]),
    "minsnap_random_positions_host": (_i, [_l, _i, _i, _vp, _vp, C.c_uint64, _vp]),
    "minsnap_fp64_peak": (_i, [_i, _vp]),
}


class MinsnapError(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        detail = ""
        try:
            detail = _lib.minsnap_last_cuda_error().decode()
        except Exception:
            pass
        msg = _lib.minsnap_error_string(code).decode() if _lib is not None else str(code)
        super().__init__("%s failed: %s (%d) %s" % (where, msg, code, detail))


_lib = None


def load():
    """Load libminsnap_b200.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libminsnap_b200.so is missing (%s). Build it with "
            "`python -m mav_trajectory_generation_cmake_b200.build`; there is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the library lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(code, where):
    if code != OK:
        raise MinsnapError(code, where)
