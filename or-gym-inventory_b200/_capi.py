"""ctypes binding of the C ABI declared in include/orgym_b200.h.

The shared library `liborgym_b200.so` is built in-tree by `__graft_entry__.build()`
(nvcc, sm_100a).  There is no CPU fallback: `lib()` raises if the library is
missing, and every compute call fails with ORGYM_E_CUDA when no GPU is present.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ORGYM_B200_LIB selects another build of the same library (kernel-tuning experiments: tools/build_variants.py)
LIB_PATH = os.environ.get("ORGYM_B200_LIB") or os.path.join(_HERE, "csrc", "liborgym_b200.so")

OK, E_INVALID, E_CUDA, E_UNSUPPORTED = 0, -1, -2, -3
AUTORESET_DISABLED, AUTORESET_NEXT_STEP, AUTORESET_SAME_STEP = 0, 1, 2
ERR_STEP_PAST_END, ERR_INT32_RANGE = 1, 2
DIST_POISSON, DIST_BINOMIAL, DIST_RANDINT, DIST_GEOMETRIC, DIST_USER = 1, 2, 3, 4, 5

c_i64p = C.POINTER(C.c_int64)
c_i32p = C.POINTER(C.c_int32)
c_f64p = C.POINTER(C.c_double)
c_f32p = C.POINTER(C.c_float)
c_u8p = C.POINTER(C.c_uint8)


class Dist(C.Structure):
    _fields_ = [("kind", C.c_int32), ("p0", C.c_double), ("p1", C.c_double), ("user_D", c_i64p),
                ("user_D_len", C.c_int32)]


class InvConfig(C.Structure):
    _fields_ = [("num_stages", C.c_int32), ("periods", C.c_int32), ("backlog", C.c_int32),
                ("wide_state", C.c_int32), ("init_inv", c_i64p), ("capacity", c_i64p), ("lead_time", c_i64p),
                ("unit_price", c_f64p), ("unit_cost", c_f64p), ("demand_cost", c_f64p), ("holding_cost", c_f64p),
                ("alpha", C.c_double), ("dist", Dist)]


class InvInfo(C.Structure):
    _fields_ = [("demand", C.c_void_p), ("sales", C.c_void_p), ("unfulfilled", C.c_void_p),
                ("profit", C.c_void_p), ("final_obs", C.c_void_p), ("info_ld", C.c_int64)]


MLP_MAX_LAYERS, MLP_MAX_WIDTH, MLP_TANH, MLP_RELU = 4, 256, 1, 2


class Mlp(C.Structure):
    """orgym_mlp_t: an actor network evaluated inside the fused rollout (device pointers to float32 weights)."""
    _fields_ = [("num_layers", C.c_int32), ("activation", C.c_int32), ("width", C.c_int32 * (MLP_MAX_LAYERS + 1)),
                ("weight", C.c_void_p * MLP_MAX_LAYERS), ("bias", C.c_void_p * MLP_MAX_LAYERS)]


class InvRolloutIn(C.Structure):
    _fields_ = [("policy", C.c_int32), ("param", C.c_double * 4), ("actions", C.c_void_p),
                ("act_stride_env", C.c_int64), ("act_stride_t", C.c_int64), ("demand", C.c_void_p),
                ("dem_stride_env", C.c_int64), ("dem_stride_t", C.c_int64), ("scratch", C.c_void_p),
                ("mlp", C.POINTER(Mlp))]


class InvRolloutOut(C.Structure):
    _fields_ = [("ep_return", C.c_void_p), ("stats", C.c_void_p), ("reward_traj", C.c_void_p),
                ("final_I", C.c_void_p), ("final_B", C.c_void_p), ("summary", C.c_void_p), ("stats32", C.c_void_p),
                ("action_traj", C.c_void_p)]


class NvConfig(C.Structure):
    _fields_ = [("lead_time", C.c_int32), ("step_limit", C.c_int32), ("max_inventory", C.c_double),
                ("max_order_quantity", C.c_double), ("p_max", C.c_double), ("h_max", C.c_double),
                ("k_max", C.c_double), ("mu_max", C.c_double)]


class NvInfo(C.Structure):
    _fields_ = [("demand", C.c_void_p), ("parts", C.c_void_p), ("final_obs", C.c_void_p), ("info_ld", C.c_int64)]


class NvRolloutIn(C.Structure):
    _fields_ = [("policy", C.c_int32), ("param", C.c_double * 4), ("actions", C.c_void_p),
                ("act_stride_env", C.c_int64), ("act_stride_t", C.c_int64), ("demand", C.c_void_p),
                ("dem_stride_env", C.c_int64), ("dem_stride_t", C.c_int64), ("fixed_params", C.c_void_p),
                ("mlp", C.POINTER(Mlp))]


class NvRolloutOut(C.Structure):
    _fields_ = [("ep_return", C.c_void_p), ("stats", C.c_void_p), ("reward_traj", C.c_void_p),
                ("action_traj", C.c_void_p), ("final_obs", C.c_void_p), ("summary", C.c_void_p)]


class NetConfig(C.Structure):
    _fields_ = [("num_periods", C.c_int32), ("backlog", C.c_int32), ("alpha", C.c_double),
                ("num_main", C.c_int32), ("node_I0", c_f64p), ("node_h", c_f64p), ("node_is_factory", c_u8p),
                ("node_is_retail", c_u8p), ("node_C", c_f64p), ("node_v", c_f64p), ("node_o", c_f64p),
                ("num_reorder", C.c_int32), ("re_supplier", c_i32p), ("re_purchaser", c_i32p), ("re_lead", c_i32p),
                ("re_p", c_f64p), ("re_g", c_f64p),
                ("num_retail", C.c_int32), ("rt_retailer", c_i32p), ("rt_p", c_f64p), ("rt_b", c_f64p),
                ("rt_dist", C.POINTER(Dist)),
                ("succ_ptr", c_i32p), ("succ_idx", c_i32p), ("pred_ptr", c_i32p), ("pred_idx", c_i32p)]


class NetInfo(C.Structure):
    _fields_ = [("demand", C.c_void_p), ("sales", C.c_void_p), ("profit", C.c_void_p),
                ("profit_total", C.c_void_p), ("final_obs", C.c_void_p), ("info_ld", C.c_int64)]


class NetRolloutIn(C.Structure):
    _fields_ = [("policy", C.c_int32), ("actions", C.c_void_p), ("act_stride_env", C.c_int64),
                ("act_stride_t", C.c_int64), ("demand", C.c_void_p), ("dem_stride_env", C.c_int64),
                ("dem_stride_t", C.c_int64), ("mlp", C.POINTER(Mlp)), ("action_high", C.c_void_p)]


class NetRolloutOut(C.Structure):
    _fields_ = [("ep_return", C.c_void_p), ("stats", C.c_void_p), ("reward_traj", C.c_void_p),
                ("final_X", C.c_void_p), ("final_Y", C.c_void_p), ("final_U", C.c_void_p), ("summary", C.c_void_p),
                ("action_traj", C.c_void_p)]


# every symbol include/orgym_b200.h declares: name -> (restype, argtypes)
_H = C.c_void_p
SYMBOLS = {
    "orgym_last_error": (C.c_char_p, []),
    "orgym_version": (C.c_int, []),
    "orgym_device_count": (C.c_int, []),
    "orgym_invmgmt_create": (C.c_int, [C.POINTER(InvConfig), C.c_int64, C.c_int, C.POINTER(_H)]),
    "orgym_invmgmt_destroy": (C.c_int, [_H]),
    "orgym_invmgmt_state_bytes": (C.c_int64, [_H]),
    "orgym_invmgmt_obs_dim": (C.c_int32, [_H]),
    "orgym_invmgmt_act_dim": (C.c_int32, [_H]),
    "orgym_invmgmt_reset": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p,
                                      C.c_void_p]),
    "orgym_invmgmt_step": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                     C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(InvInfo), C.c_void_p]),
    "orgym_invmgmt_export_state": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "orgym_invmgmt_rollout": (C.c_int, [_H, C.c_uint64, C.c_int64, C.c_uint32, C.POINTER(InvRolloutIn),
                                        C.POINTER(InvRolloutOut), C.c_void_p]),
    "orgym_newsvendor_create": (C.c_int, [C.POINTER(NvConfig), C.c_int64, C.c_int, C.POINTER(_H)]),
    "orgym_newsvendor_destroy": (C.c_int, [_H]),
    "orgym_newsvendor_state_bytes": (C.c_int64, [_H]),
    "orgym_newsvendor_obs_dim": (C.c_int32, [_H]),
    "orgym_newsvendor_reset": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "orgym_newsvendor_step": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.POINTER(NvInfo), C.c_void_p]),
    "orgym_newsvendor_export_params": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p]),
    "orgym_newsvendor_rollout": (C.c_int, [_H, C.c_uint64, C.c_int64, C.c_uint32, C.POINTER(NvRolloutIn),
                                           C.POINTER(NvRolloutOut), C.c_void_p]),
    "orgym_netinv_create": (C.c_int, [C.POINTER(NetConfig), C.c_int64, C.c_int, C.POINTER(_H)]),
    "orgym_netinv_destroy": (C.c_int, [_H]),
    "orgym_netinv_state_bytes": (C.c_int64, [_H]),
    "orgym_netinv_obs_dim": (C.c_int32, [_H]),
    "orgym_netinv_reset": (C.c_int, [_H, C.c_void_p, C.c_int, C.c_uint64, C.c_int64, C.c_void_p, C.c_void_p,
                                     C.c_void_p]),
    "orgym_netinv_step": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.POINTER(NetInfo), C.c_void_p]),
    "orgym_netinv_export_state": (C.c_int, [_H, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p]),
    "orgym_netinv_rollout": (C.c_int, [_H, C.c_void_p, C.c_uint64, C.c_int64, C.c_uint32, C.POINTER(NetRolloutIn),
                                       C.POINTER(NetRolloutOut), C.c_void_p]),
    "orgym_invmgmt_rollout_scratch_bytes": (C.c_int64, [_H]),
    "orgym_invmgmt_specialise": (C.c_int, [_H, C.POINTER(InvRolloutIn)]),
    "orgym_invmgmt_codegen": (C.c_int, [C.POINTER(InvConfig), C.POINTER(InvRolloutIn), C.c_int, C.c_char_p, C.c_int64,
                                        C.POINTER(C.c_int64)]),
    "orgym_invmgmt_is_specialised": (C.c_int, [_H]),
    "orgym_invmgmt_value_bounds": (C.c_int, [C.POINTER(InvConfig), C.POINTER(C.c_double), C.POINTER(C.c_double),
                                             C.POINTER(C.c_double)]),
    "orgym_netinv_codegen": (C.c_int, [C.POINTER(NetConfig), C.c_int, C.c_char_p, C.c_int64, C.POINTER(C.c_int64)]),
    "orgym_netinv_is_specialised": (C.c_int, [_H]),
    "orgym_report_scratch_bytes": (C.c_int64, [C.c_int64]),
    "orgym_evaluation_report": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int32, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "orgym_errors": (C.c_int, [_H, C.POINTER(C.c_uint32), C.c_int, C.c_void_p]),
    "orgym_sample_demand": (C.c_int, [C.POINTER(Dist), C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int,
                                      C.c_void_p, C.c_void_p]),
    "orgym_sample_poisson_mu": (C.c_int, [C.c_void_p, C.c_uint64, C.c_int64, C.c_int64, C.c_int32, C.c_int,
                                          C.c_void_p, C.c_void_p]),
}

_lib = None


class OrgymError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"orgym_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load liborgym_b200.so (once).  Raises if it has not been built -- there is no fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  or-gym-inventory_b200 has no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        missing = [name for name in SYMBOLS if not hasattr(L, name)]
        if missing:  # the header and the library disagree: refuse to run on a partial build
            raise ImportError(f"{LIB_PATH} does not export {missing}; rebuild it")
        for name, (res, args) in SYMBOLS.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(code):
    if code != 0:
        msg = lib().orgym_last_error()
        raise OrgymError(code, msg.decode() if msg else "?")
    return code


def make_dist(kind, p0=0.0, p1=0.0, user_D=None, keep=None):
    """Build an orgym_dist_t; `keep` collects the numpy buffers that must outlive the struct."""
    import numpy as np
    d = Dist()
    d.kind = int(kind)
    d.p0 = float(p0)
    d.p1 = float(p1)
    if user_D is not None:
        arr = np.ascontiguousarray(np.asarray(user_D, dtype=np.int64))
        if keep is not None:
            keep.append(arr)
        d.user_D = arr.ctypes.data_as(c_i64p)
        d.user_D_len = int(arr.size)
    else:
        d.user_D = None
        d.user_D_len = 0
    return d
