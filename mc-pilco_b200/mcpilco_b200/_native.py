"""ctypes binding of libmcpilco_b200.so (include/mcpilco_b200.h).  No torch types cross this boundary:
only raw device pointers, sizes and POD structs.  The library must have been built in-tree
(`python __graft_entry__.py` or `mcpilco_b200._build.build()`); a missing library is a hard error —
there is no CPU fallback on this path."""
import ctypes as C
import os

MAX_D, MAX_DS, MAX_DU, MAX_E, MAX_DP, MAX_POLY, MAX_DEG = 32, 16, 8, 16, 32, 3, 3
ABI_VERSION = 8
OZAKI_EXP_NONFINITE = 1 << 20  # row exponent of the INT8 contraction's digit planes for a row with a NaN / inf
_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmcpilco_b200.so")

f64p = C.POINTER(C.c_double)


class GpSpec(C.Structure):
    _fields_ = [("D", C.c_int32), ("has_se", C.c_int32), ("n_poly", C.c_int32), ("poly_deg", C.c_int32 * MAX_POLY),
                ("lambda_", C.c_double), ("mean0", C.c_double), ("sigma_n2", C.c_double), ("inv_ls", C.c_double * MAX_D),
                ("poly_w2", ((C.c_double * (MAX_D + 1)) * MAX_DEG) * MAX_POLY)]


class Gp(C.Structure):
    _fields_ = [("spec", GpSpec), ("N", C.c_int32), ("ld_kinv", C.c_int32), ("Xtr", C.c_void_p), ("alpha", C.c_void_p),
                ("Kinv", C.c_void_p), ("var_scale", C.c_double), ("kinv_planes", C.c_void_p), ("kinv_exp", C.c_void_p),
                ("ozaki_slices", C.c_int32), ("ld_linv", C.c_int32), ("Linv", C.c_void_p), ("kdiag_max", C.c_double)]


class Model(C.Structure):
    _fields_ = [("Ds", C.c_int32), ("Du", C.c_int32), ("E", C.c_int32), ("D", C.c_int32), ("kind", C.c_int32),
                ("use_trig", C.c_int32), ("n_na", C.c_int32), ("n_a", C.c_int32), ("na_idx", C.c_int32 * MAX_DS),
                ("a_idx", C.c_int32 * MAX_DS), ("vel_idx", C.c_int32 * MAX_E), ("pos_idx", C.c_int32 * MAX_E),
                ("particle_pred", C.c_int32), ("_pad", C.c_int32), ("T", C.c_double)]


class Policy(C.Structure):
    _fields_ = [("kind", C.c_int32), ("nb", C.c_int32), ("Dp", C.c_int32), ("Du", C.c_int32), ("Ds", C.c_int32),
                ("n_na", C.c_int32), ("n_a", C.c_int32), ("na_idx", C.c_int32 * MAX_DS), ("a_idx", C.c_int32 * MAX_DS),
                ("squash", C.c_int32), ("has_bias", C.c_int32), ("use_drop", C.c_int32), ("u_max", C.c_double * MAX_DU),
                ("inv_scale", C.c_double * MAX_DP), ("log_ls", C.c_void_p), ("centers", C.c_void_p), ("W", C.c_void_p),
                ("bias", C.c_void_p), ("target_traj", C.c_void_p)]


class Cost(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_idx", C.c_int32), ("idx", C.c_int32 * MAX_DS), ("target", C.c_double * MAX_DS),
                ("inv_ls", C.c_double * MAX_DS), ("target_traj", C.c_void_p)]


class Meas(C.Structure):
    _fields_ = [("enabled", C.c_int32), ("n_pos", C.c_int32), ("pos_idx", C.c_int32 * MAX_E), ("vel_idx", C.c_int32 * MAX_E),
                ("std_pos", C.c_double * MAX_E), ("b0", C.c_double), ("b1", C.c_double), ("a0", C.c_double), ("a1", C.c_double),
                ("T", C.c_double)]


class Noise(C.Structure):
    _fields_ = [("eps", C.c_void_p), ("masks", C.c_void_p), ("meas_eps", C.c_void_p), ("seed", C.c_uint64),
                ("particle_offset", C.c_uint64), ("p_dropout", C.c_double), ("seed_dev", C.c_void_p)]


class Rollout(C.Structure):
    _fields_ = [("M", C.c_int32), ("H", C.c_int32), ("need_grad", C.c_int32), ("M_global", C.c_int32), ("model", Model),
                ("policy", Policy), ("cost", Cost), ("meas", Meas), ("noise", Noise), ("gps", C.POINTER(Gp)),
                ("x0", C.c_void_p), ("states", C.c_void_p), ("inputs", C.c_void_p), ("jac", C.c_void_p),
                ("pol_in", C.c_void_p), ("costs", C.c_void_p), ("cost_out", C.c_void_p), ("cost_stats", C.c_void_p),
                ("workspace", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class RolloutGrad(C.Structure):
    _fields_ = [("grad_states", C.c_void_p), ("grad_inputs", C.c_void_p), ("grad_cost", C.c_double), ("g_log_ls", C.c_void_p),
                ("g_centers", C.c_void_p), ("g_W", C.c_void_p), ("g_bias", C.c_void_p), ("g_x0", C.c_void_p)]


# every symbol include/mcpilco_b200.h declares: (restype, argtypes)
SYMBOLS = {
    "mcpilco_abi_version": (C.c_int, []),
    "mcpilco_last_error": (C.c_char_p, []),
    "mcpilco_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "mcpilco_set_device": (C.c_int, [C.c_int]),
    "mcpilco_gp_covariance": (C.c_int, [C.POINTER(GpSpec), C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p]),
    "mcpilco_gp_diag_covariance": (C.c_int, [C.POINTER(GpSpec), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "mcpilco_gp_precompute_workspace_bytes": (C.c_size_t, [C.c_int]),
    "mcpilco_gp_precompute": (C.c_int, [C.POINTER(GpSpec), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mcpilco_gp_sod_workspace_bytes": (C.c_size_t, [C.c_int]),
    "mcpilco_gp_sod_select": (C.c_int, [C.POINTER(GpSpec), C.c_void_p, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                        C.c_void_p]),
    "mcpilco_gp_nlml_grad_size": (C.c_int, []),
    "mcpilco_gp_nlml_workspace_bytes": (C.c_size_t, [C.c_int]),
    "mcpilco_gp_nlml": (C.c_int, [C.POINTER(GpSpec), C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "mcpilco_gp_predict_workspace_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "mcpilco_gp_predict": (C.c_int, [C.POINTER(Gp), C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_size_t, C.c_void_p]),
    "mcpilco_rollout_workspace_bytes": (C.c_size_t, [C.c_int] * 8),
    "mcpilco_rollout_fwd": (C.c_int, [C.POINTER(Rollout), C.c_void_p]),
    "mcpilco_rollout_bwd": (C.c_int, [C.POINTER(Rollout), C.POINTER(RolloutGrad), C.c_void_p]),
    "mcpilco_policy_forward": (C.c_int, [C.POINTER(Policy), C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_uint64, C.c_uint64,
                                         C.c_void_p, C.c_void_p]),
    "mcpilco_policy_backward_workspace_bytes": (C.c_size_t, [C.c_int] * 4),
    "mcpilco_policy_backward": (C.c_int, [C.POINTER(Policy), C.c_int, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_uint64, C.c_uint64,
                                          C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t,
                                          C.c_void_p]),
    "mcpilco_init_particles": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "mcpilco_ozaki_available": (C.c_int, []),
    "mcpilco_ozaki_plane_bytes": (C.c_size_t, [C.c_int, C.c_int]),
    "mcpilco_ozaki_prepare": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "mcpilco_ozaki_scratch_bytes": (C.c_size_t, [C.c_int, C.c_int, C.c_int]),
    "mcpilco_ozaki_contract": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p,
                                         C.c_size_t, C.c_void_p]),
    "mcpilco_prof_enable": (C.c_int, [C.c_int]),
    "mcpilco_prof_read": (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.POINTER(C.c_double)]),
    "mcpilco_launch_count": (C.c_uint64, [C.c_int]),
    "mcpilco_struct_sizes": (C.c_int, [C.POINTER(C.c_size_t), C.c_int]),
}

_lib = None


class NativeError(RuntimeError):
    pass


def lib():
    """Load (once) and return the shared library with typed entry points."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeError("libmcpilco_b200.so is not built (%s): run `python __graft_entry__.py` / mcpilco_b200._build.build(); "
                          "this path has no CPU fallback" % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)  # AttributeError if the symbol is missing
        fn.restype, fn.argtypes = res, args
    if L.mcpilco_abi_version() != ABI_VERSION:
        raise NativeError("ABI mismatch: library %d, binding %d" % (L.mcpilco_abi_version(), ABI_VERSION))
    sizes = (C.c_size_t * 16)()
    k = L.mcpilco_struct_sizes(sizes, 16)
    mine = [C.sizeof(x) for x in (GpSpec, Gp, Model, Policy, Cost, Meas, Noise, Rollout, RolloutGrad)]
    if k != len(mine) or list(sizes[:k]) != mine:
        raise NativeError("struct layout mismatch: library %s, binding %s" % (list(sizes[:k]), mine))
    _lib = L
    return L


def check(rc):
    if rc != 0:
        raise NativeError("mcpilco_b200 native call failed (%d): %s" % (rc, lib().mcpilco_last_error().decode()))
