"""ctypes binding of libphoenix_b200.so (the C ABI declared in include/phoenix_b200.h).

There is no CPU fallback: if the library has not been built, or no sm_100a device is present, the product path
raises.  Build with ``python -m phoenix_b200.build`` (nvcc, sm_100a).
"""
import ctypes
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libphoenix_b200.so")

PHX_OK = 0
METHOD_IDS = {"euler": 0, "midpoint": 1, "rk4": 2, "dopri5": 3}
PARAMS_ALL = 0x3F   # adjoint parameter mask: bit i = the i-th ODENet parameter in reference order
NORM_SEMINORM = 0x40   # OR-ed into an adjoint solve's mask: the dopri5 error norm leaves out the parameter block
PREC_FP32, PREC_TF32, PREC_3XTF32 = 0, 1, 3
ENGINE_RESIDENT, ENGINE_ROWS, ENGINE_STREAM = 0, 1, 2
ST_OK, ST_DT_UNDERFLOW, ST_NONFINITE, ST_MAX_STEPS, ST_RUNNING = 0, 1, 2, 3, 99

EXPORTS = [
    "phx_ctx_create", "phx_ctx_destroy", "phx_last_error", "phx_ctx_num_sms", "phx_resident_max_rows",
    "phx_ctx_set_profile", "phx_profile_slots", "phx_plan_describe",
    "phx_ctx_set_precision", "phx_ctx_get_precision", "phx_tc_min_rows", "phx_tc_plan_describe",
    "phx_packed_bytes", "phx_pack_weights", "phx_rhs_forward", "phx_rhs_vjp", "phx_rhs_workspace_bytes",
    "phx_solve_workspace_bytes", "phx_solve_workspace_init_bytes", "phx_solve_workspace_init", "phx_solve_forward",
    "phx_solve_adjoint", "phx_solve_forward_many", "phx_solve_adjoint_many",
    "phx_stream_workspace_bytes", "phx_stream_solve_forward", "phx_stream_solve_adjoint",
    "phx_rows_supported", "phx_rows_plan_describe", "phx_rows_workspace_bytes", "phx_solve_forward_rows",
    "phx_solve_adjoint_rows", "phx_unpack_grads", "phx_packed_grad_bytes", "phx_rows_grad_parts",
    "phx_unpack_grads_masked", "phx_solve", "phx_grid_workspace_bytes",
    "phx_prior_loss", "phx_prior_setup", "phx_tc_set_pair", "phx_tc_prof_dump", "phx_ctx_set_global_norm", "phx_peer_allreduce", "phx_peer_allreduce_nvls", "phx_mse_grad", "phx_hill_planes", "phx_hill_cache_set",
]


class PhxStatus(ctypes.Structure):
    _fields_ = [("code", ctypes.c_int32), ("n_accepted", ctypes.c_int32), ("n_rejected", ctypes.c_int32),
                ("n_rhs", ctypes.c_int32), ("n_logged", ctypes.c_int32), ("reserved", ctypes.c_int32),
                ("t_fail", ctypes.c_double), ("dt_fail", ctypes.c_double)]


class PhxSolveDesc(ctypes.Structure):
    """phx_solve_desc: one solve request of phx_solve (the 8-byte fields first, so there is no padding)."""
    _fields_ = ([(name, ctypes.c_void_p) for name in (
                    "packed", "t_host", "y0", "y_out", "y_saved", "grad_y", "adj_y0", "grads", "grid_dt", "grid_steps",
                    "grid_out_step", "grid_out_slope", "workspace")]
                + [("workspace_bytes", ctypes.c_size_t), ("status", ctypes.c_void_p), ("steplog", ctypes.c_void_p),
                   ("rtol", ctypes.c_double), ("atol", ctypes.c_double), ("max_num_steps", ctypes.c_int64),
                   ("first_step", ctypes.c_double), ("safety", ctypes.c_double), ("ifactor", ctypes.c_double),
                   ("dfactor", ctypes.c_double)]
                + [(name, ctypes.c_int32) for name in (
                    "engine", "adjoint", "G", "H", "B", "N", "T", "t_is_f32", "reversed", "method", "param_mask",
                    "steplog_cap")])


class PhoenixLibraryError(RuntimeError):
    pass


_lib = None
_lock = threading.Lock()
_ctx = {}


def _declare(lib):
    c_int, c_size_t, c_void_p, c_double, c_int64 = (ctypes.c_int, ctypes.c_size_t, ctypes.c_void_p, ctypes.c_double,
                                                   ctypes.c_int64)
    lib.phx_ctx_create.argtypes = [c_int, ctypes.POINTER(c_void_p)]
    lib.phx_ctx_create.restype = c_int
    lib.phx_ctx_destroy.argtypes = [c_void_p]
    lib.phx_ctx_destroy.restype = None
    lib.phx_last_error.argtypes = []
    lib.phx_last_error.restype = ctypes.c_char_p
    lib.phx_ctx_num_sms.argtypes = [c_void_p]
    lib.phx_ctx_num_sms.restype = c_int
    lib.phx_resident_max_rows.argtypes = [c_int]
    lib.phx_resident_max_rows.restype = c_int
    lib.phx_ctx_set_profile.argtypes = [c_void_p, c_void_p]
    lib.phx_ctx_set_profile.restype = c_int
    lib.phx_plan_describe.argtypes = [c_int] * 5 + [ctypes.POINTER(ctypes.c_int32)]
    lib.phx_plan_describe.restype = c_int
    lib.phx_profile_slots.argtypes = []
    lib.phx_profile_slots.restype = c_int
    lib.phx_ctx_set_precision.argtypes = [c_void_p, c_int]
    lib.phx_ctx_set_precision.restype = c_int
    lib.phx_ctx_get_precision.argtypes = [c_void_p]
    lib.phx_ctx_get_precision.restype = c_int
    lib.phx_tc_plan_describe.argtypes = [c_int, c_int, ctypes.POINTER(ctypes.c_int32)]
    lib.phx_tc_plan_describe.restype = c_int
    lib.phx_tc_min_rows.argtypes = []
    lib.phx_tc_min_rows.restype = c_int
    lib.phx_packed_bytes.argtypes = [c_int, c_int]
    lib.phx_packed_bytes.restype = c_size_t
    lib.phx_pack_weights.argtypes = [c_void_p, c_int, c_int] + [c_void_p] * 7 + [c_void_p]
    lib.phx_pack_weights.restype = c_int
    lib.phx_rhs_workspace_bytes.argtypes = [c_int, c_int, c_int]
    lib.phx_rhs_workspace_bytes.restype = c_size_t
    lib.phx_rhs_forward.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                    c_size_t, c_void_p]
    lib.phx_rhs_forward.restype = c_int
    lib.phx_rhs_vjp.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                c_void_p, c_int, c_void_p, c_size_t, c_void_p]
    lib.phx_rhs_vjp.restype = c_int
    lib.phx_solve_workspace_bytes.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_int]
    lib.phx_solve_workspace_bytes.restype = c_size_t
    lib.phx_solve_workspace_init_bytes.argtypes = []
    lib.phx_solve_workspace_init_bytes.restype = c_size_t
    lib.phx_solve_workspace_init.argtypes = [c_void_p, c_size_t, c_void_p]
    lib.phx_solve_workspace_init.restype = c_int
    fwd = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, ctypes.POINTER(c_double), c_int, c_int, c_int,
           c_int, c_double, c_double, c_int64, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p, c_int, c_void_p]
    adj = [c_void_p, c_int, c_int, c_int, c_void_p, ctypes.POINTER(c_double), c_int, c_int, c_int, c_double,
           c_double, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p, c_void_p,
           c_int, c_void_p]
    lib.phx_solve_forward.argtypes = fwd
    lib.phx_solve_forward.restype = c_int
    lib.phx_solve_adjoint.argtypes = adj
    lib.phx_solve_adjoint.restype = c_int
    lib.phx_solve_forward_many.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                           ctypes.POINTER(c_double), c_int, c_int, c_int, c_double, c_double, c_int64,
                                           c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]
    lib.phx_solve_forward_many.restype = c_int
    lib.phx_solve_adjoint_many.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_void_p, ctypes.POINTER(c_double), c_int,
                                           c_int, c_int, c_double, c_double, c_int64, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]
    lib.phx_solve_adjoint_many.restype = c_int
    lib.phx_stream_workspace_bytes.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_int]
    lib.phx_stream_workspace_bytes.restype = c_size_t
    lib.phx_stream_solve_forward.argtypes = fwd
    lib.phx_stream_solve_forward.restype = c_int
    lib.phx_stream_solve_adjoint.argtypes = adj
    lib.phx_stream_solve_adjoint.restype = c_int
    lib.phx_rows_supported.argtypes = [c_void_p, c_int, c_int, c_int]
    lib.phx_rows_supported.restype = c_int
    lib.phx_rows_plan_describe.argtypes = [c_int] * 4 + [ctypes.POINTER(ctypes.c_int32)]
    lib.phx_rows_plan_describe.restype = c_int
    lib.phx_rows_workspace_bytes.argtypes = [c_void_p, c_int, c_int, c_int, c_int, c_int]
    lib.phx_rows_workspace_bytes.restype = c_size_t
    # (ctx, G, H, N, packed, y0, t, T, t_is_f32, reversed, method, rtol, atol, max_steps, y_out, ws, ws_bytes, status,
    #  steplog, steplog_cap, stream)
    lib.phx_solve_forward_rows.argtypes = fwd
    lib.phx_solve_forward_rows.restype = c_int
    # (ctx, G, H, N, packed, t, T, t_is_f32, method, rtol, atol, max_steps, y_saved, grad_y, adj_y0, grads_packed_parts,
    #  ws, ws_bytes, status, steplog, steplog_cap, stream)
    lib.phx_solve_adjoint_rows.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, ctypes.POINTER(c_double), c_int, c_int,
                                           c_int, c_double, c_double, c_int64, c_void_p, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_size_t, c_void_p, c_void_p, c_int, c_void_p]
    lib.phx_solve_adjoint_rows.restype = c_int
    lib.phx_unpack_grads.argtypes = [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_void_p]
    lib.phx_rows_grad_parts.argtypes = [c_void_p, c_int, c_int, c_int]
    lib.phx_rows_grad_parts.restype = c_int
    lib.phx_unpack_grads.restype = c_int
    lib.phx_unpack_grads_masked.argtypes = [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_int, c_void_p]
    lib.phx_unpack_grads_masked.restype = c_int
    lib.phx_solve.argtypes = [c_void_p, ctypes.POINTER(PhxSolveDesc), c_void_p]
    lib.phx_solve.restype = c_int
    lib.phx_grid_workspace_bytes.argtypes = [c_int, c_int, c_int64]
    lib.phx_grid_workspace_bytes.restype = c_size_t
    lib.phx_prior_loss.argtypes = [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, ctypes.c_float, c_void_p,
                                   c_void_p, c_void_p, c_size_t, c_void_p]
    lib.phx_prior_loss.restype = c_int
    lib.phx_prior_setup.argtypes = [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.phx_prior_setup.restype = c_int
    lib.phx_ctx_set_global_norm.argtypes = [c_void_p, c_void_p, c_void_p, c_int]
    lib.phx_ctx_set_global_norm.restype = c_int
    lib.phx_peer_allreduce.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_size_t, ctypes.c_uint, ctypes.c_float,
                                       c_void_p]
    lib.phx_peer_allreduce.restype = c_int
    lib.phx_mse_grad.argtypes = [c_void_p, c_int, c_int, c_void_p, c_size_t, c_void_p, ctypes.c_float, c_void_p, c_size_t,
                                 c_void_p]
    lib.phx_mse_grad.restype = c_int
    lib.phx_hill_planes.argtypes = [c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]
    lib.phx_hill_planes.restype = c_int
    lib.phx_hill_cache_set.argtypes = [c_void_p, c_void_p, c_size_t, c_void_p, c_void_p]
    lib.phx_hill_cache_set.restype = c_int
    lib.phx_peer_allreduce_nvls.argtypes = [c_void_p, c_void_p, c_void_p, c_int, c_int, c_size_t, ctypes.c_uint,
                                            ctypes.c_float, c_void_p]
    lib.phx_peer_allreduce_nvls.restype = c_int
    lib.phx_packed_grad_bytes.argtypes = [c_int, c_int]
    lib.phx_packed_grad_bytes.restype = c_size_t


def load():
    """Load the shared library (once).  Raises PhoenixLibraryError if it is missing — never falls back."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise PhoenixLibraryError(
                    "phoenix_b200: %s not found. Build it with `python -m phoenix_b200.build` (needs nvcc, "
                    "sm_100a). There is no CPU fallback." % LIB_PATH)
            lib = ctypes.CDLL(LIB_PATH)
            _declare(lib)
            _lib = lib
    return _lib


def last_error():
    msg = load().phx_last_error()
    return msg.decode() if msg else ""


def check(rc, what):
    if rc != PHX_OK:
        msg = last_error()
        if rc == -3:
            raise NotImplementedError("phoenix_b200 %s: %s" % (what, msg))
        raise PhoenixLibraryError("phoenix_b200 %s failed (code %d): %s" % (what, rc, msg))


def ctx(device_index):
    """phx_ctx for a CUDA device index (cached for the life of the process)."""
    c = _ctx.get(device_index)
    if c is None:
        lib = load()
        out = ctypes.c_void_p()
        check(lib.phx_ctx_create(int(device_index), ctypes.byref(out)), "ctx_create")
        c = out
        _ctx[device_index] = c
    return c
