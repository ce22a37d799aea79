"""ctypes binding of libcplb.so (the C ABI in include/cpl_batched.h).

The library is the product; this module only declares its prototypes.  It fails loudly when
the shared object is missing -- there is no Python/NumPy fallback for the evaluation path.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcplb.so")

OK, INVALID_ARGUMENT, OUT_OF_RANGE, RUNTIME_ERROR, CUDA_ERROR, NULL_POINTER = range(6)
ENV_NONE, ENV_GROUND, ENV_SUPERQUADRIC = 0, 1, 2
INSTANCE_MAJOR, COMPONENT_MAJOR = 0, 1
HOST_JAC_CONSTANTS_PRESENT = 1
DEVICE_INPUTS_READY = 2
JAC_PACKED = 4
JAC_COMPUTED = 8   # ... and without the slots that are copies +-x[col] (cplb_get_jacobian_slot_sources)
SLOT_CONSTANT, SLOT_COPY, SLOT_NEGATED_COPY, SLOT_COMPUTED = 0, 1, 2, 3
KERNEL_AUTO, KERNEL_PER_CONTACT, KERNEL_PER_INSTANCE = 0, 1, 2
KERNEL_WARP_TILE, KERNEL_CTA_TILE = 1, 2
BLOCK_COM, BLOCK_FORCE, BLOCK_POSITION, BLOCK_NORMAL = 0, 1, 2, 3

dp = C.POINTER(C.c_double)
ip = C.POINTER(C.c_int32)


# cplb_instance_params in member order: (name, fixed length, length per contact); doubles per instance = fixed + per_contact * nc
INSTANCE_PARAMS = (("mass", 1, 0), ("wrench", 6, 0), ("mu", 1, 0), ("force_threshold", 0, 1), ("ground_z", 1, 0), ("com_ref", 3, 0),
                   ("com_weight", 1, 0), ("pos_ref", 0, 3), ("force_ref", 0, 3), ("pos_weight", 0, 1), ("force_weight", 0, 1))


class InstanceParams(C.Structure):
    """cplb_instance_params: optional per-instance parameter arrays (NULL = the problem's shared value)."""
    _fields_ = [(name, C.c_void_p) for name, _, _ in INSTANCE_PARAMS]


class EvalArgs(C.Structure):
    _fields_ = [
        ("num_instances", C.c_int64),
        ("layout", C.c_int32),
        ("host_flags", C.c_int32),
        ("ld", C.c_int64),
        ("x", C.c_void_p),
        ("g", C.c_void_p),
        ("jac", C.c_void_p),
        ("cost", C.c_void_p),
        ("grad", C.c_void_p),
        ("per_instance", C.POINTER(InstanceParams)),
    ]


class SolverOptions(C.Structure):
    """cplb_solver_options"""
    _fields_ = [("tol", C.c_double), ("mu_init", C.c_double), ("bound_push", C.c_double), ("bound_frac", C.c_double),
                ("nlp_scaling_max_gradient", C.c_double), ("constr_viol_tol", C.c_double), ("polish_viol_tol", C.c_double),
                ("bound_relax_factor", C.c_double), ("max_iter", C.c_int32), ("max_backtracks", C.c_int32),
                ("tail_instances", C.c_int32)]


class SolveOutputs(C.Structure):
    """cplb_solve_outputs"""
    _fields_ = [("x", C.c_void_p), ("status", C.c_void_p), ("iterations", C.c_void_p), ("cost", C.c_void_p), ("constr_viol", C.c_void_p),
                ("dual_inf", C.c_void_p), ("lam", C.c_void_p), ("rounds", C.POINTER(C.c_int32)), ("evaluations", C.POINTER(C.c_int64)),
                ("instance_evaluations", C.POINTER(C.c_int64)),
                ("tail_instances", C.POINTER(C.c_int64))]


class DerivativeTestOptions(C.Structure):
    """cplb_derivative_test_options"""
    _fields_ = [("perturbation", C.c_double), ("tol", C.c_double)]


class DerivativeTestOutputs(C.Structure):
    """cplb_derivative_test_outputs (device pointers; None = not wanted)"""
    _fields_ = [("num_wrong", C.c_void_p), ("num_wrong_outside", C.c_void_p), ("max_rel_error", C.c_void_p), ("worst_row", C.c_void_p),
                ("worst_col", C.c_void_p), ("jac_fd", C.c_void_p), ("grad_fd", C.c_void_p)]


class JacobianProductsArgs(C.Structure):
    """cplb_jacobian_products_args (device pointers; None = NULL)"""
    _fields_ = [("num_instances", C.c_int64), ("x", C.c_void_p), ("per_instance", C.POINTER(InstanceParams)), ("lambda_", C.c_void_p),
                ("obj_factor", C.c_void_p), ("x_bar", C.c_void_p), ("v", C.c_void_p), ("g_dot", C.c_void_p), ("f_dot", C.c_void_p)]


# name -> (restype, argtypes); every symbol include/cpl_batched.h declares
PROTOTYPES = {
    "cplb_create": (C.c_int, [C.c_int32, C.POINTER(C.c_char_p), C.c_int, C.c_double, C.c_int32, C.POINTER(C.c_void_p)]),
    "cplb_create_sharded": (C.c_int, [C.c_int32, C.POINTER(C.c_char_p), C.c_int, C.c_double, C.c_int32, ip, C.POINTER(C.c_void_p)]),
    "cplb_get_num_shards": (C.c_int, [C.c_void_p, ip]),
    "cplb_get_shard": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, ip, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "cplb_eval_device_shard": (C.c_int, [C.c_void_p, C.c_int32, C.POINTER(EvalArgs), C.c_void_p]),
    "cplb_destroy": (None, [C.c_void_p]),
    "cplb_last_error": (C.c_char_p, []),
    "cplb_abi_version": (C.c_int32, []),
    "cplb_get_dims": (C.c_int, [C.c_void_p, ip, ip, ip]),
    "cplb_get_jacobian_structure": (C.c_int, [C.c_void_p, ip, ip]),
    "cplb_get_sorted_order": (C.c_int, [C.c_void_p, ip]),
    "cplb_get_block_column": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, ip]),
    "cplb_get_contact_row": (C.c_int, [C.c_void_p, C.c_char_p, ip]),
    "cplb_get_jacobian_constants": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint8), dp]),
    "cplb_fill_jacobian_constants": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, dp]),
    "cplb_get_packed_jacobian_map": (C.c_int, [C.c_void_p, ip, ip]),
    "cplb_unpack_jacobian": (C.c_int, [C.c_void_p, C.c_int64, dp, dp]),
    "cplb_get_jacobian_slot_sources": (C.c_int, [C.c_void_p, ip, ip, ip]),
    "cplb_expand_jacobian": (C.c_int, [C.c_void_p, C.c_int64, dp, dp, dp]),
    "cplb_get_variable_bounds": (C.c_int, [C.c_void_p, dp, dp]),
    "cplb_get_constraint_bounds": (C.c_int, [C.c_void_p, dp, dp]),
    "cplb_set_mass": (C.c_int, [C.c_void_p, C.c_double]),
    "cplb_get_mass": (C.c_int, [C.c_void_p, dp]),
    "cplb_set_reduction_order": (C.c_int, [C.c_void_p, C.c_int32]),
    "cplb_set_manipulation_wrench": (C.c_int, [C.c_void_p, dp]),
    "cplb_get_manipulation_wrench": (C.c_int, [C.c_void_p, dp]),
    "cplb_set_mu": (C.c_int, [C.c_void_p, C.c_double]),
    "cplb_get_mu": (C.c_int, [C.c_void_p, dp]),
    "cplb_set_ground_z": (C.c_int, [C.c_void_p, C.c_double]),
    "cplb_get_ground_z": (C.c_int, [C.c_void_p, dp]),
    "cplb_set_superquadric": (C.c_int, [C.c_void_p, dp, dp, dp]),
    "cplb_get_superquadric": (C.c_int, [C.c_void_p, dp, dp, dp]),
    "cplb_set_force_threshold": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "cplb_get_force_threshold": (C.c_int, [C.c_void_p, C.c_char_p, dp]),
    "cplb_set_bounds": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, dp, dp]),
    "cplb_get_bounds": (C.c_int, [C.c_void_p, C.c_int, C.c_char_p, dp, dp]),
    "cplb_set_pos_ref": (C.c_int, [C.c_void_p, C.c_char_p, dp]),
    "cplb_get_pos_ref": (C.c_int, [C.c_void_p, C.c_char_p, dp]),
    "cplb_set_force_ref": (C.c_int, [C.c_void_p, C.c_char_p, dp]),
    "cplb_get_force_ref": (C.c_int, [C.c_void_p, C.c_char_p, dp]),
    "cplb_set_com_ref": (C.c_int, [C.c_void_p, dp]),
    "cplb_get_com_ref": (C.c_int, [C.c_void_p, dp]),
    "cplb_set_com_weight": (C.c_int, [C.c_void_p, C.c_double]),
    "cplb_get_com_weight": (C.c_int, [C.c_void_p, dp]),
    "cplb_set_pos_weight": (C.c_int, [C.c_void_p, C.c_double]),
    "cplb_set_force_weight": (C.c_int, [C.c_void_p, C.c_double]),
    "cplb_set_contact_pos_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "cplb_get_contact_pos_weight": (C.c_int, [C.c_void_p, C.c_char_p, dp]),
    "cplb_set_contact_force_weight": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "cplb_get_contact_force_weight": (C.c_int, [C.c_void_p, C.c_char_p, dp]),
    "cplb_eval_device": (C.c_int, [C.c_void_p, C.POINTER(EvalArgs), C.c_void_p]),
    "cplb_eval_host": (C.c_int, [C.c_void_p, C.POINTER(EvalArgs)]),
    "cplb_eval_host_begin": (C.c_int, [C.c_void_p, C.POINTER(EvalArgs), C.POINTER(C.c_int32)]),
    "cplb_eval_host_wait": (C.c_int, [C.c_void_p, C.c_int32]),
    "cplb_solver_default_options": (None, [C.POINTER(SolverOptions)]),
    "cplb_solve_device": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(InstanceParams), C.POINTER(SolverOptions), C.POINTER(SolveOutputs), C.c_void_p]),
    "cplb_derivative_test_default_options": (None, [C.POINTER(DerivativeTestOptions)]),
    "cplb_derivative_test_device": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.POINTER(InstanceParams), C.POINTER(DerivativeTestOptions),
                                              C.POINTER(DerivativeTestOutputs), C.c_void_p]),
    "cplb_jacobian_products_device": (C.c_int, [C.c_void_p, C.POINTER(JacobianProductsArgs), C.c_void_p]),
    "cplb_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "cplb_host_free": (C.c_int, [C.c_void_p]),
    "cplb_set_component_major_kernel": (C.c_int, [C.c_void_p, C.c_int32]),
    "cplb_set_instance_major_kernel": (C.c_int, [C.c_void_p, C.c_int32]),
    "cplb_get_device": (C.c_int, [C.c_void_p, ip]),
    "cplb_get_launch_count": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64)]),
    "cplb_timing_begin": (C.c_int, [C.c_void_p]),
    "cplb_timing_end": (C.c_int, [C.c_void_p, dp, C.POINTER(C.c_int64)]),
}

_lib = None


def load():
    """dlopen libcplb.so.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C centroidalplanner_b200/csrc`. The evaluator has no CPU fallback."
            )
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib
