"""ctypes binding of libo3d_b200.so (the C ABI declared in include/o3d_b200.h).

The product path has NO fallback: if the shared library is missing or a kernel reports an error, a
RuntimeError is raised.  Build with `python -c "import __graft_entry__ as g; g.build()"` (nvcc, sm_100a).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libo3d_b200.so")

_p = ctypes.c_void_p
_i = ctypes.c_int
_f = ctypes.c_float
_d = ctypes.c_double

# name -> argtypes (restype is int unless listed in _RESTYPE); mirrors include/o3d_b200.h
PROTOTYPES = {
    "o3d_version": [],
    "o3d_last_error": [],
    "o3d_opt_threads": [_i],
    "o3d_device_sms": [],
    "o3d_fps": [_p, _i, _i, _i, _p, _p],
    "o3d_gather": [_p, _p, _i, _i, _i, _i, _p, _p],
    "o3d_gather_grad": [_p, _p, _i, _i, _i, _i, _p, _p],
    "o3d_ball_query": [_p, _p, _i, _i, _i, _f, _i, _p, _p],
    "o3d_group": [_p, _p, _i, _i, _i, _i, _i, _p, _p],
    "o3d_group_grad": [_p, _p, _i, _i, _i, _i, _i, _p, _p],
    "o3d_three_nn": [_p, _p, _i, _i, _i, _p, _p, _p],
    "o3d_three_interpolate": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "o3d_three_interpolate_grad": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "o3d_ballquery_group": [_p, _p, _p, _i, _i, _i, _i, _f, _i, _i, _p, _p, _p],
    "o3d_ballquery_group_grad": [_p, _p, _i, _i, _i, _i, _i, _f, _i, _p, _p, _p, _p],
    "o3d_three_nn_interpolate": [_p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p],
    "o3d_three_nn_interpolate_grad": [_p, _p, _p, _i, _i, _i, _i, _p, _p],
    "o3d_group_rows": [_p, _p, _i, _i, _i, _i, _p, _p],
    "o3d_group_rows_grad": [_p, _p, _i, _i, _i, _i, _p, _p],
    "o3d_xcorr_boxaware_fwd": [_p, _p, _i, _i, _i, _i, _i, _p, _p],
    "o3d_xcorr_p2b_fwd": [_p, _p, _i, _i, _i, _i, _f, _p, _p, _p, _p],
    "o3d_xcorr_p2b_bwd": [_p, _p, _p, _p, _p, _p, _i, _i, _i, _i, _f, _p, _p, _p],
    "o3d_pw_fwd": [_p, _i, _p, _p, _i, _p, _i, _p, _i, _i, _i, _p, _i, _p, _p, _i, _p, _p, _p, _i, _p],
    "o3d_pw_dgrad": [_p, _i, _p, _i, _p, _p, _p, _p, _p, _i, _i, _p, _i, _i, _i, _i, _p, _i, _p, _i, _p, _p, _i, _p, _p,
                     _p],
    "o3d_pw_wgrad": [_p, _i, _p, _i, _p, _p, _p, _p, _p, _i, _i, _p, _i, _p, _p, _i, _i, _i, _i, _p, _i, _p],
    "o3d_bn_fwd_finalize": [_p, _p, _d, _p, _p, _p, _p, _p, _f, _f, _i, _i, _p, _p, _p, _p, _p],
    "o3d_bn_bwd_finalize": [_p, _p, _d, _p, _p, _p, _i, _i, _p, _p, _p, _p, _p, _p],
    "o3d_pool_finalize": [_p, _p, _p, _p, _p, _i, _i, _i, _i, _p, _i, _p, _p, _p],
    "o3d_pool_bwd_prep": [_p, _i, _p, _i, _p, _i, _i, _i, _i, _p, _p, _p, _p],
    "o3d_act_apply": [_p, _i, _p, _p, _i, _i, _i, _p, _i, _p],
    "o3d_dense_bwd_prep": [_p, _i, _p, _i, _p, _i, _i, _i, _i, _p, _i, _p, _p, _p],
    "o3d_pw_tc_wtile_bytes": [_i, _i],
    "o3d_debug_set": [_i, _i],
    "o3d_pw_tc_pretile": [_p, _i, _i, _i, _p, _p],
    "o3d_pw_fwd_tc": [_p, _i, _p, _p, _i, _p, _p, _i, _i, _i, _p, _i, _p, _p, _i, _p, _p, _p, _i, _p],
    "o3d_pw_dgrad_tc": [_p, _i, _p, _i, _p, _p, _p, _p, _p, _i, _i, _p, _i, _i, _i, _p, _i, _p, _i, _p, _p, _i, _p, _p,
                        _p],
    "o3d_pw_wgrad_tc2_workspace_floats": [],
    "o3d_pw_wgrad_tc2": [_p, _i, _p, _i, _p, _p, _p, _p, _p, _i, _i, _p, _i, _p, _p, _i, _i, _i, _i, _p, _i, _p,
                         ctypes.c_longlong, _p],
    "o3d_adam_step": [_p, _p, _p, _p, ctypes.c_longlong, _p, _f, _f, _f, _f, _p],
    "o3d_crop_box_frame": [_p, _p, _p, _p, _p, _p, _i, _i, _p, _p, _p],
    "o3d_resample": [_p, _p, _p, _p, _i, _i, _i, _p, _p, _p, _p, _p],
    "o3d_lift_stats": [_p, _i, _i, _p, _p, _p, _p, _p],
    "o3d_lift_scatter": [_p, _i, _i, _p, _p, _p, _i, _p, _p, _p, _p],
    "o3d_stack_workspace_bytes": [_p, _i],
    "o3d_stack_prepared_bytes": [_p],
    "o3d_stack_prepare": [_p, _p, _p],
    "o3d_stack_forward": [_p, _p, _p, _p, _i, _p],
    "o3d_stack_backward": [_p, _p, _p, _p, _p, _p, _p, _p],
    "o3d_sa_fused_prepared_bytes": [_p],
    "o3d_sa_fused_prepare": [_p, _p, _p],
    "o3d_sa_fused_forward": [_p, _p, _p, _p, _p, _i, _i, _i, _i, ctypes.c_float, _i, _i, _p, _i, _p, _p],
}
_RESTYPE = {"o3d_last_error": ctypes.c_char_p, "o3d_pw_tc_wtile_bytes": ctypes.c_longlong,
            "o3d_stack_workspace_bytes": ctypes.c_longlong, "o3d_stack_prepared_bytes": ctypes.c_longlong,
            "o3d_sa_fused_prepared_bytes": ctypes.c_longlong, "o3d_pw_wgrad_tc2_workspace_floats": ctypes.c_longlong}

MAX_LAYERS = 8
_I8, _F8, _P8 = ctypes.c_int * MAX_LAYERS, ctypes.c_float * MAX_LAYERS, ctypes.c_void_p * MAX_LAYERS


class LiftDesc(ctypes.Structure):
    """ctypes mirror of `o3d_lift_t` (include/o3d_b200.h, block 4)."""
    _fields_ = [("z", _p), ("ldz", _i), ("ridx", _p), ("ridx_mod", _i), ("rows_per_cloud", _i), ("pos_per_cloud", _i),
                ("grp", _i), ("s", _p), ("u", _p),
                ("d_z", _p), ("d_s", _p), ("d_u", _p)]


class StackDesc(ctypes.Structure):
    """ctypes mirror of `o3d_stack_t` (include/o3d_b200.h, block 4)."""
    _fields_ = [("n_layers", _i), ("P", _i), ("K0", _i), ("S", _i), ("training", _i), ("use_tc", _i),
                ("xyz_first", _i), ("c0", _i), ("dx_cols", _i),
                ("cin", _I8), ("cout", _I8), ("relu", _I8), ("has_bn", _I8),
                ("momentum", _F8), ("eps", _F8),
                ("weight", _P8), ("bias", _P8), ("gamma", _P8), ("beta", _P8),
                ("running_mean", _P8), ("running_var", _P8), ("num_batches_tracked", _P8),
                ("d_weight", _P8), ("d_bias", _P8), ("d_gamma", _P8), ("d_beta", _P8),
                ("lift", ctypes.POINTER(LiftDesc)), ("accumulate", _i), ("prepared", _p)]

_lib = None


def lib():
    """Load (once) and return the CDLL; raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"open3dsot_b200: native library not found at {LIB_PATH}. There is no CPU or PyTorch fallback; "
                "build it with `python -c \"import __graft_entry__ as g; g.build()\"` (needs nvcc).")
        L = ctypes.CDLL(LIB_PATH)
        for name, args in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the .so is stale -> rebuild
            fn.argtypes = args
            fn.restype = _RESTYPE.get(name, ctypes.c_int)
        _lib = L
    return _lib


def check(status, name):
    if status != 0:
        msg = lib().o3d_last_error()
        raise RuntimeError(f"{name} failed with status {status}: {msg.decode() if msg else ''}")
