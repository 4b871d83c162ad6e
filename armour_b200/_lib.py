"""ctypes binding of armour_b200/libarmour_b200.so — the C ABI declared in include/armour_b200.h.

The shared library holds the CUDA kernels; there is no CPU fallback.  Importing this module only
loads the library (so symbol checks work on a box without a GPU); creating a context needs a GPU.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# ARMOUR_B200_LIB: developer override used by tools/exp_k1.py to compare differently tuned builds of the SAME CUDA library
LIB_PATH = os.environ.get("ARMOUR_B200_LIB") or os.path.join(_HERE, "libarmour_b200.so")
NF = 7

OK, ERR_ARG, ERR_CUDA, ERR_OBSTACLES, ERR_CAPACITY, ERR_STATE, ERR_NOMEM = 0, -1, -2, -3, -4, -5, -6


class ArmourError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"armour_b200 error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int), ("device", C.c_int), ("robot_model", C.c_int), ("num_time_steps", C.c_int),
        ("max_obstacles", C.c_int), ("max_problems", C.c_int), ("cap_link_monomials", C.c_int),
        ("cap_torque_monomials", C.c_int), ("cap_work_monomials", C.c_int), ("simplify_threshold", C.c_double),
        ("k_range", C.c_double * NF), ("mass_uncertainty", C.c_double), ("inertia_uncertainty", C.c_double),
    ]


dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int)
up = C.POINTER(C.c_ulonglong)


class ReachsetTables(C.Structure):
    _fields_ = [
        ("cap_link", C.c_int), ("cap_u", C.c_int), ("link_n", ip), ("link_center", dp), ("link_key", up),
        ("link_coeff", dp), ("u_n", ip), ("u_center", dp), ("u_key", up), ("u_coeff", dp), ("u_radius", dp),
        ("torque_radius", dp), ("link_gens", dp),
    ]


# name -> (restype, argtypes); every symbol include/armour_b200.h declares
SIGNATURES = {
    "armour_config_default": (C.c_int, [C.POINTER(Config)]),
    "armour_ctx_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "armour_ctx_destroy": (C.c_int, [C.c_void_p]),
    "armour_ctx_reserve": (C.c_int, [C.c_void_p, C.c_int, C.c_int]),
    "armour_ctx_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "armour_ctx_synchronize": (C.c_int, [C.c_void_p]),
    "armour_status_string": (C.c_char_p, [C.c_int]),
    "armour_last_error": (C.c_char_p, [C.c_void_p]),
    "armour_abi_version": (C.c_int, []),
    "armour_kernel_launches": (C.c_longlong, [C.c_void_p]),
    "armour_num_joints": (C.c_int, [C.c_void_p]),
    "armour_num_time_steps": (C.c_int, [C.c_void_p]),
    "armour_num_constraints": (C.c_int, [C.c_void_p, C.c_int]),
    "armour_reachsets_build": (C.c_int, [C.c_void_p, dp, dp, dp, dp, C.c_int]),
    "armour_get_torque_radius": (C.c_int, [C.c_void_p, dp]),
    "armour_get_link_independent_generators": (C.c_int, [C.c_void_p, dp]),
    "armour_get_bounds": (C.c_int, [C.c_void_p, dp, dp]),
    "armour_eval_g": (C.c_int, [C.c_void_p, dp, dp]),
    "armour_eval_jac_g": (C.c_int, [C.c_void_p, dp, dp]),
    "armour_eval_g_jac": (C.c_int, [C.c_void_p, dp, dp, dp]),
    "armour_get_link_sliced_center": (C.c_int, [C.c_void_p, dp]),
    "armour_verdict": (C.c_int, [C.c_void_p, dp, ip, ip]),
    "armour_cost": (C.c_int, [C.c_void_p, dp, dp, dp, dp]),
    "armour_batch_reachsets_build": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp, dp, C.c_int]),
    "armour_batch_eval": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp]),
    "armour_batch_eval_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "armour_batch_reachsets_build_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                                      C.c_void_p, C.c_int]),
    "armour_batch_verdict_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "armour_batch_get_torque_radius": (C.c_int, [C.c_void_p, C.c_int, dp]),
    "armour_batch_get_link_independent_generators": (C.c_int, [C.c_void_p, C.c_int, dp]),
    "armour_batch_get_bounds": (C.c_int, [C.c_void_p, C.c_int, dp, dp]),
    "armour_batch_get_build_status": (C.c_int, [C.c_void_p, C.c_int, ip]),
    "armour_batch_get_monomial_counts": (C.c_int, [C.c_void_p, C.c_int, ip, ip]),
    "armour_batch_get_candidate_counts": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "armour_chunk_intervals": (C.c_int, []),
    "armour_eval_image_layout": (C.c_int, [C.c_void_p, C.POINTER(C.c_longlong)]),
    "armour_batch_get_eval_images": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "armour_jacobian_nnz": (C.c_longlong, [C.c_void_p, C.c_int]),
    "armour_jacobian_structure": (C.c_int, [C.c_void_p, C.c_int, ip, ip]),
    "armour_eval_jac_g_structured": (C.c_int, [C.c_void_p, dp, dp]),
    "armour_batch_eval_structured": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp]),
    "armour_batch_eval_structured_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "armour_measure_fp64_peak": (C.c_int, [C.c_void_p, dp]),
    "armour_solver_options_default": (None, [C.c_void_p]),
    "armour_batch_solve_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p]),
    "armour_batch_solve": (C.c_int, [C.c_void_p, C.c_int, dp, C.c_void_p, dp, ip, ip, ip]),
    "armour_export_reachsets": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(ReachsetTables)]),
    "armour_import_reachsets": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.POINTER(ReachsetTables), dp, dp, dp, dp,
                                          C.c_int]),
}


class ControllerGains(C.Structure):
    """armour_controller_gains (include/armour_b200.h)."""
    _fields_ = [("Kr", dp), ("alpha", C.c_double), ("V_max", C.c_double), ("r_norm_threshold", C.c_double),
                ("apply_friction", C.c_int)]


_gp = C.POINTER(ControllerGains)
SIGNATURES.update({
    "armour_controller_create": (C.c_int, [C.c_char_p, C.c_double, C.c_int, C.POINTER(C.c_void_p)]),
    "armour_controller_create_error": (C.c_char_p, []),
    "armour_controller_destroy": (None, [C.c_void_p]),
    "armour_controller_num_joints": (C.c_int, [C.c_void_p]),
    "armour_controller_last_error": (C.c_char_p, [C.c_void_p]),
    "armour_controller_kernel_launches": (C.c_longlong, [C.c_void_p]),
    "armour_controller_set_stream": (C.c_int, [C.c_void_p, C.c_void_p]),
    "armour_controller_synchronize": (C.c_int, [C.c_void_p]),
    "armour_controller_get_interval_model": (C.c_int, [C.c_void_p, dp]),
    "armour_controller_rnea": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp, dp, C.c_int, C.c_int, dp, dp, dp]),
    "armour_controller_rnea_device": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_int] + [C.c_void_p] * 3),
    "armour_controller_update": (C.c_int, [C.c_void_p, C.c_int, _gp, dp, dp, dp, dp, dp, dp, dp, dp, ip]),
    "armour_controller_update_device": (C.c_int, [C.c_void_p, C.c_int, _gp] + [C.c_void_p] * 10),
})

SIGNATURES.update({
    "armour_armtd_ctx_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "armour_armtd_build": (C.c_int, [C.c_void_p, dp, dp, dp, dp, dp, C.c_int]),
    "armour_armtd_num_constraints": (C.c_int, [C.c_void_p]),
    "armour_armtd_eval": (C.c_int, [C.c_void_p, dp, dp, dp]),
    "armour_armtd_get_bounds": (C.c_int, [C.c_void_p, dp, dp]),
    "armour_armtd_verdict": (C.c_int, [C.c_void_p, dp, ip, ip]),
    "armour_armtd_cost": (C.c_int, [C.c_void_p, dp, dp, dp, dp]),
    "armour_armtd_get_link_sliced_center": (C.c_int, [C.c_void_p, dp]),
    "armour_armtd_get_link_independent_generators": (C.c_int, [C.c_void_p, dp]),
    "armour_armtd_batch_ctx_create": (C.c_int, [C.POINTER(Config), C.POINTER(C.c_void_p)]),
    "armour_armtd_batch_build": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp, dp, dp, C.c_int]),
    "armour_armtd_batch_build_device": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 5 + [C.c_int, C.c_void_p]),
    "armour_armtd_batch_eval": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp]),
    "armour_armtd_batch_eval_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "armour_armtd_batch_verdict_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "armour_armtd_batch_cost": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp, dp]),
    "armour_armtd_batch_get_link_independent_generators": (C.c_int, [C.c_void_p, C.c_int, dp]),
    "armour_armtd_batch_solve": (C.c_int, [C.c_void_p, C.c_int, dp, C.c_void_p, dp, ip, ip, ip]),
    "armour_armtd_batch_solve_device": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 6),
})


class SolverOptions(C.Structure):
    """armour_solver_options (include/armour_b200.h)."""
    _fields_ = [("max_iter", C.c_int), ("tol", C.c_double), ("torque_tol", C.c_double), ("collision_tol", C.c_double),
                ("qp_sweeps", C.c_int), ("qp_update_budget", C.c_int)]


class RolloutOptions(C.Structure):
    """armour_rollout_options (include/armour_b200.h)."""
    _fields_ = [("struct_size", C.c_int), ("max_replans", C.c_int), ("lookahead", C.c_double), ("goal_radius", C.c_double),
                ("audit_samples", C.c_int), ("solver", SolverOptions)]


class RolloutOut(C.Structure):
    """armour_rollout_out (include/armour_b200.h): output arrays, any may be NULL."""
    _fields_ = [("outcome", ip), ("replans", ip), ("infeasible", ip), ("final_state", dp), ("min_clearance", dp),
                ("log_state", dp), ("log_q_des", dp), ("log_k", dp), ("log_int", ip), ("log_clearance", dp)]


# outcome of a closed-loop episode (ARMOUR_ROLLOUT_*)
ROLLOUT_BUDGET, ROLLOUT_ARRIVED, ROLLOUT_COLLISION, ROLLOUT_LIMIT = 0, 1, 2, 3

SIGNATURES.update({
    "armour_rollout_options_default": (None, [C.POINTER(RolloutOptions)]),
    "armour_batch_rollout_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                              C.POINTER(RolloutOptions), C.POINTER(RolloutOut)]),
    "armour_batch_rollout": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp, C.c_int, C.POINTER(RolloutOptions),
                                       C.POINTER(RolloutOut)]),
    "armour_batch_clearance_device": (C.c_int, [C.c_void_p, C.c_int] + [C.c_void_p] * 3 + [C.c_int, C.c_void_p, C.c_void_p]),
    "armour_batch_clearance": (C.c_int, [C.c_void_p, C.c_int, dp, ip, dp, C.c_int, dp, ip]),
    "armour_armtd_batch_rollout_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                    C.POINTER(RolloutOptions), C.POINTER(RolloutOut)]),
    "armour_armtd_batch_rollout": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp, C.c_int, C.POINTER(RolloutOptions),
                                             C.POINTER(RolloutOut)]),
    "armour_armtd_offline_jrs": (C.c_int, [C.c_void_p, C.c_int, dp, dp, dp]),
    "armour_armtd_offline_jrs_device": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
})


_LIB = None


def load():
    """Load libarmour_b200.so; raises (loudly) if the CUDA extension has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; "
                "g.build()' or make -C armour_b200/csrc). armour_b200 has no CPU fallback.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _LIB = lib
    return _LIB
