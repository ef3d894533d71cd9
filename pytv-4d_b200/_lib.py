"""ctypes binding of libpytv_b200.so (C ABI declared in include/pytv_b200.h).

There is no CPU fallback: if the library has not been built, or no CUDA device is present, the first
compute call raises.  Build with `python -c "import __graft_entry__ as g; g.build()"` or `make -C
pytv-4d_b200/csrc`.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PYTVB_LIB_PATH") or os.path.join(_HERE, "csrc", "libpytv_b200.so")   # override: tuning builds

SCHEME_ID = {"upwind": 0, "downwind": 1, "central": 2, "hybrid": 3}
F32, F64 = 0, 1


class Problem(ctypes.Structure):
    """struct pytvb_problem (include/pytv_b200.h)."""
    _fields_ = [
        ("scheme", ctypes.c_int32),
        ("dtype", ctypes.c_int32),
        ("Nz", ctypes.c_int64),
        ("M", ctypes.c_int64),
        ("Ni", ctypes.c_int64),
        ("Nj", ctypes.c_int64),
        ("z_offset", ctypes.c_int64),
        ("Nz_global", ctypes.c_int64),
        ("reg_z_over_reg", ctypes.c_double),
        ("reg_time", ctypes.c_double),
        ("factor_reg_static", ctypes.c_double),
        ("mask_static", ctypes.c_void_p),
        ("time_scale", ctypes.c_void_p),
        ("time_scale_lo", ctypes.c_void_p),
        ("time_scale_hi", ctypes.c_void_p),
    ]


def make_problem(scheme, dtype_id, shape, reg_z_over_reg=1.0, reg_time=0.0, factor_reg_static=0.0, mask_static_ptr=None,
                 z_offset=0, Nz_global=None, time_scale_ptr=None):
    Nz, M, Ni, Nj = (int(s) for s in shape)
    rz = float(reg_z_over_reg)
    return Problem(SCHEME_ID[scheme] if isinstance(scheme, str) else int(scheme), int(dtype_id), Nz, M, Ni, Nj, int(z_offset),
                   int(Nz if Nz_global is None else Nz_global), rz, float(reg_time), float(factor_reg_static),
                   ctypes.c_void_p(mask_static_ptr) if mask_static_ptr else None,
                   ctypes.c_void_p(time_scale_ptr) if time_scale_ptr else None, None, None)


_VP = ctypes.c_void_p
_PB = ctypes.POINTER(Problem)
_PROTOTYPES = {
    "pytvb_version": (ctypes.c_int, []),
    "pytvb_build_id": (ctypes.c_char_p, []),
    "pytvb_last_error": (ctypes.c_char_p, []),
    "pytvb_launch_count": (ctypes.c_uint64, []),
    "pytvb_num_components": (ctypes.c_int, [_PB]),
    "pytvb_reduce_workspace_bytes": (ctypes.c_size_t, [_PB]),
    "pytvb_tv_workspace_bytes": (ctypes.c_size_t, [_PB]),
    "pytvb_D": (ctypes.c_int, [_PB, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_DT": (ctypes.c_int, [_PB, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_l21": (ctypes.c_int, [_PB, _VP, ctypes.c_int64, _VP, _VP, _VP, _VP]),
    "pytvb_apply_mask": (ctypes.c_int, [_PB, _VP, _VP, ctypes.c_int, _VP]),
    "pytvb_tv": (ctypes.c_int, [_PB, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_gd_update": (ctypes.c_int, [_PB, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP]),
    "pytvb_tv_value": (ctypes.c_int, [_PB, _VP, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_dual": (ctypes.c_int, [_PB, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_primal_rof": (ctypes.c_int, [_PB, _VP, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_primal_readme": (ctypes.c_int, [_PB, _VP, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_dual_p2p": (ctypes.c_int, [_PB, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_primal_p2p": (ctypes.c_int, [_PB, ctypes.c_int, _VP, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_primal_data": (ctypes.c_int, [_PB, ctypes.c_int, _VP, _VP, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP, _VP,
                                            _VP]),
    "pytvb_cp_dual_adj": (ctypes.c_int, [_PB, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_dual_adj_p2p": (ctypes.c_int, [_PB, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_primal_adj": (ctypes.c_int, [_PB, ctypes.c_int, _VP, _VP, _VP, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP,
                                           _VP]),
    "pytvb_cp_primal_adj_p2p": (ctypes.c_int, [_PB, ctypes.c_int, _VP, _VP, _VP, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP,
                                               _VP, _VP, _VP, _VP]),
    "pytvb_cp_dual_f16y": (ctypes.c_int, [_PB, _VP, _VP, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_cp_primal_rof_f16y": (ctypes.c_int, [_PB, _VP, _VP, _VP, _VP, ctypes.c_double, ctypes.c_double, ctypes.c_double, _VP, _VP, _VP, _VP, _VP]),
    "pytvb_tv_host": (ctypes.c_int, [_PB, _VP, _VP, _VP, ctypes.POINTER(ctypes.c_double)]),
    "pytvb_cp_create": (ctypes.c_int, [_PB, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.c_double, ctypes.POINTER(_VP)]),
    "pytvb_cp_reset_host": (ctypes.c_int, [_VP, _VP]),
    "pytvb_cp_step_host": (ctypes.c_int, [_VP, _VP, _VP, ctypes.POINTER(ctypes.c_double)]),
    "pytvb_cp_destroy": (ctypes.c_int, [_VP]),
}

_lib = None


def lib():
    """The loaded library; raises loudly when it is missing (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("pytv_b200: %s has not been built (run __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOTYPES.items():
            fn = getattr(handle, name)   # AttributeError if the ABI and the header drifted apart
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class PytvError(RuntimeError):
    pass


def check(rc):
    if rc != 0:
        raise PytvError("pytv_b200 call failed (%d): %s" % (rc, lib().pytvb_last_error().decode("utf-8", "replace")))
