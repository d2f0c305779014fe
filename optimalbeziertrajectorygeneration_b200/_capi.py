"""ctypes binding of libbezgpu.so (include/bezgpu.h).

There is NO CPU fallback: importing this module without the built library, or
calling into it without a CUDA device, raises.  The library is built in-tree by
``__graft_entry__.build()`` / ``python -m optimalbeziertrajectorygeneration_b200._build``.
"""
import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libbezgpu.so")

c_double_p = ctypes.c_void_p      # raw device/host addresses (tensor.data_ptr())
c_plan_p = ctypes.c_void_p


class BezGpuError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise BezGpuError(
            "libbezgpu.so is not built (%s). Run `python -c 'import __graft_entry__ as g; g.build()'` "
            "-- there is no CPU fallback for the Bezier constraint path." % LIB_PATH)
    return ctypes.CDLL(LIB_PATH)


_lib = _load()

I, D, P, L64 = ctypes.c_int, ctypes.c_double, ctypes.c_void_p, ctypes.c_int64

class ReduceOpts(ctypes.Structure):
    """bez_reduce_opts of include/bezgpu.h."""
    _fields_ = [("itemmin", ctypes.c_void_p), ("min_pitch", ctypes.c_int64), ("peer_min", ctypes.c_void_p),
                ("npeers", ctypes.c_int), ("active_mask", ctypes.c_void_p), ("threshold", ctypes.c_double),
                ("list_count", ctypes.c_void_p), ("list_idx", ctypes.c_void_p), ("list_val", ctypes.c_void_p),
                ("list_cap", ctypes.c_int64)]


# name -> (restype, argtypes); must list every symbol include/bezgpu.h declares
SIGNATURES = {
    "bez_last_error": (ctypes.c_char_p, []),
    "bez_version": (I, []),
    "bez_plan_create": (I, [I, I, I, I, P, P, P, ctypes.POINTER(c_plan_p)]),
    "bez_plan_destroy": (I, [c_plan_p]),
    "bez_plan_info": (I, [c_plan_p, ctypes.POINTER(I), ctypes.POINTER(I), ctypes.POINTER(I),
                          ctypes.POINTER(I)]),
    "bez_assemble_cpts": (I, [c_plan_p, P, I, I, I, I, I, I, I, D,
                              P, P, P, P, P, P, P, P, P, P, P, P]),
    "bez_assemble_cpts_sets": (I, [c_plan_p, P, I, I, I, I, I, I, I, D,
                                   P, P, P, P, P, P, P, P, P, I, P, P, P]),
    "bez_pair_sepsq_elev": (I, [c_plan_p, P, I, I, L64, L64, D, P, P, P]),
    "bez_pair_sepsq_elev_p2p": (I, [c_plan_p, P, I, I, L64, L64, D, P, P, P, I, P]),
    "bez_speed_sq_elev": (I, [c_plan_p, P, P, I, I, I, I, D, D, P, P]),
    "bez_pair_sepsq_elev_ex": (I, [c_plan_p, P, I, I, L64, L64, D, P, ctypes.POINTER(ReduceOpts), P]),
    "bez_speed_sq_elev_ex": (I, [c_plan_p, P, P, I, I, I, I, D, D, P, ctypes.POINTER(ReduceOpts), P]),
    "bez_angrate_tables_create": (I, [I, I, I, P, P, P, P, ctypes.POINTER(c_plan_p)]),
    "bez_angrate_tables_destroy": (I, [c_plan_p]),
    "bez_angrate_sq": (I, [c_plan_p, P, P, I, I, I, I, I, D, D, P, P]),
    "bez_curve_elev": (I, [P, P, L64, I, I, P, P]),
    "bez_curve_diff": (I, [P, P, P, L64, L64, I, P, P]),
    "bez_curve_mul": (I, [P, P, P, L64, I, I, P, P]),
    "bez_curve_normsq": (I, [P, P, L64, I, I, P, P]),
    "bez_curve_eval": (I, [P, P, L64, I, I, D, D, P, P]),
    "bez_objective_euclidean": (I, [c_plan_p, P, I, I, I, P, P]),
    "bez_objective_accel": (I, [c_plan_p, P, P, I, I, I, P, P]),
    "bez_objective_grad": (I, [c_plan_p, P, I, D, I, I, I, P, P, P]),
    "bez_split": (I, [P, P, I, I, I, P, P, P]),
    "bez_extrema_scratch_doubles": (ctypes.c_size_t, [I, I, I]),
    "bez_extrema": (I, [P, I, I, D, I, I, P, P, P, P]),
    "bez_gjk": (I, [P, P, P, P, I, I, I, P, P, P, P, P]),
    "bez_mindist_scratch_doubles": (ctypes.c_size_t, [I, I, I, I]),
    "bez_mindist": (I, [P, P, I, I, I, I, I, D, I, ctypes.c_longlong, P, P, P, P]),
    "bez_mindist2poly_scratch_doubles": (ctypes.c_size_t, [I, I, I]),
    "bez_mindist2poly": (I, [P, P, P, I, I, I, I, D, I, ctypes.c_longlong, P, P, P, P]),
    "bez_collcheck_scratch_doubles": (ctypes.c_size_t, [I, I, I]),
    "bez_collcheck": (I, [P, P, I, I, I, I, I, D, P, P, P]),
    "bez_collcheck2poly_scratch_doubles": (ctypes.c_size_t, [I, I]),
    "bez_collcheck2poly": (I, [P, P, P, I, I, I, I, ctypes.c_longlong, P, P, P, P]),
    "bez_fd_quotient": (I, [P, P, I, L64, P, P]),
    "bez_fd_quotient_batched": (I, [P, P, L64, I, L64, P, P]),
    "bez_jac_sepsq_elev": (I, [c_plan_p, P, I, I, I, I, P, P, I, I, P, L64, P]),
    "bez_jac_speed_sq_elev": (I, [c_plan_p, P, I, I, I, I, D, D, P, P, I, I, P, L64, P]),
    "bez_jac_sepsq_elev_batched": (I, [c_plan_p, P, I, I, I, I, I, P, P, I, L64, I, P, L64, P]),
    "bez_jac_speed_sq_elev_batched": (I, [c_plan_p, P, P, I, I, I, I, I, D, P, P, I, I, P, L64, P]),
    "bez_jac_angrate_scratch_doubles": (ctypes.c_size_t, [I, I, I, I]),
    "bez_jac_angrate_sq": (I, [c_plan_p, P, P, I, I, I, I, I, I, I, P, P, I, D, I, P, P, L64, P]),
}

OPTIONAL = {}


def _bind(table, required):
    for name, (res, args) in table.items():
        try:
            fn = getattr(_lib, name)
        except AttributeError:
            if required:
                raise BezGpuError("libbezgpu.so does not export %s; rebuild it" % name)
            continue
        fn.restype = res
        fn.argtypes = args


_bind(SIGNATURES, True)


def last_error():
    return _lib.bez_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise BezGpuError("%s failed (code %d): %s" % (what, rc, last_error()))


def call(name, *args):
    """Invoke an entry point that returns a status code and raise on failure."""
    check(getattr(_lib, name)(*args), name)


lib = _lib
