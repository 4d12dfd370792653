"""ctypes binding of libparopt_b200.so (the C ABI in include/paropt_b200.h).

The product has no CPU path: importing works anywhere (so that the CPU test
suite can check the exported symbols), but creating a Context without a CUDA
device raises.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PCU_LIB", os.path.join(HERE, "libparopt_b200.so"))

_lib = None

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class Weighting(C.Structure):
    _fields_ = [("nwcon", C.c_int), ("wstart", C.c_int), ("nw", C.c_int),
                ("wstride", C.c_int), ("coef0", C.c_double),
                ("coef_rest", C.c_double), ("wconst", C.c_double)]


class BlockWeighting(C.Structure):
    _fields_ = [("nblocks", C.c_int), ("wstart", C.c_int), ("nw", C.c_int),
                ("wstride", C.c_int), ("nb", C.c_int), ("coef", c_double_p),
                ("wconst", c_double_p)]


class SepQuadParams(C.Structure):
    _fields_ = [("ntotal", C.c_int64), ("ncon", C.c_int), ("nw", C.c_int),
                ("seed", C.c_uint64), ("lam_min", C.c_double),
                ("lam_max", C.c_double), ("b_lo", C.c_double), ("b_w", C.c_double),
                ("a_lo", C.c_double), ("a_w", C.c_double), ("beta_c", C.c_double),
                ("beta_n", C.c_double), ("beta_u", C.c_double),
                ("x0_lo", C.c_double * 2), ("x0_w", C.c_double * 2),
                ("lb", C.c_double * 2), ("ub", C.c_double * 2),
                ("householder", C.c_int)]


GET_VARS_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p)
EVAL_OBJ_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, c_double_p, c_double_p)
EVAL_GRAD_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                           C.POINTER(C.c_void_p))


QN_CORR_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, c_double_p, C.c_void_p,
                         C.c_void_p, C.c_void_p)
WRITE_OUT_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_void_p)
HVEC_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, c_double_p, C.c_void_p, C.c_void_p,
                      C.c_void_p)


HDIAG_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, c_double_p, C.c_void_p, C.c_void_p)


class Callbacks(C.Structure):
    _fields_ = [("user", C.c_void_p), ("get_vars_and_bounds", GET_VARS_CB),
                ("eval_obj_con", EVAL_OBJ_CB),
                ("eval_obj_con_gradient", EVAL_GRAD_CB),
                ("qn_update_correction", QN_CORR_CB),
                ("write_output", WRITE_OUT_CB),
                ("eval_hvec_product", HVEC_CB)]


HOST_GET_VARS_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, c_double_p, c_double_p,
                               c_double_p)
HOST_EVAL_OBJ_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, c_double_p, c_double_p,
                               c_double_p)
HOST_EVAL_GRAD_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, c_double_p, c_double_p,
                                C.POINTER(c_double_p))


HOST_WRITE_OUT_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, C.c_int, c_double_p)
HOST_HVEC_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, c_double_p, c_double_p, C.c_int,
                           c_double_p, c_double_p, c_double_p)


HOST_HDIAG_CB = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int, c_double_p, c_double_p, C.c_int,
                            c_double_p, c_double_p)


class HostCallbacks(C.Structure):
    _fields_ = [("user", C.c_void_p), ("get_vars_and_bounds", HOST_GET_VARS_CB),
                ("eval_obj_con", HOST_EVAL_OBJ_CB),
                ("eval_obj_con_gradient", HOST_EVAL_GRAD_CB),
                ("write_output", HOST_WRITE_OUT_CB),
                ("eval_hvec_product", HOST_HVEC_CB)]


VP = C.c_void_p

# name -> (restype, argtypes); every symbol include/paropt_b200.h declares
SIGNATURES = {
    "pcu_version": (C.c_char_p, []),
    "pcu_ctx_create": (VP, [C.c_int]),
    "pcu_ctx_destroy": (None, [VP]),
    "pcu_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "pcu_ctx_init_comm": (C.c_int, [VP, C.c_char_p, C.c_int, C.c_int]),
    "pcu_ctx_rank": (C.c_int, [VP]),
    "pcu_ctx_size": (C.c_int, [VP]),
    "pcu_ctx_sync": (C.c_int, [VP]),
    "pcu_ctx_stream": (VP, [VP]),
    "pcu_ctx_kernel_launches": (C.c_int64, [VP]),
    "pcu_ctx_set_param": (C.c_int, [VP, C.c_char_p, C.c_int]),
    "pcu_ctx_profile": (C.c_int, [VP, C.c_int]),
    "pcu_ctx_profile_count": (C.c_int, [VP]),
    "pcu_ctx_profile_get": (C.c_int, [VP, C.c_int, C.c_char_p, C.c_int, c_double_p,
                                      C.POINTER(C.c_int64)]),
    "pcu_ctx_timer_start": (C.c_int, [VP]),
    "pcu_ctx_timer_stop": (C.c_int, [VP, c_double_p]),
    "pcu_vec_create": (VP, [VP, C.c_int]),
    "pcu_vec_destroy": (None, [VP]),
    "pcu_vec_size": (C.c_int, [VP]),
    "pcu_vec_set": (C.c_int, [VP, C.c_double]),
    "pcu_vec_zero": (C.c_int, [VP]),
    "pcu_vec_copy": (C.c_int, [VP, VP]),
    "pcu_vec_norm": (C.c_int, [VP, c_double_p]),
    "pcu_vec_maxabs": (C.c_int, [VP, c_double_p]),
    "pcu_vec_l1norm": (C.c_int, [VP, c_double_p]),
    "pcu_vec_dot": (C.c_int, [VP, VP, c_double_p]),
    "pcu_vec_mdot": (C.c_int, [VP, C.POINTER(VP), C.c_int, c_double_p]),
    "pcu_blockmat_create": (VP, [VP, C.c_int, C.POINTER(Weighting)]),
    "pcu_blockmat_create_blocks": (VP, [VP, C.c_int, C.POINTER(BlockWeighting)]),
    "pcu_sparsemat_create": (VP, [VP, C.c_int, C.c_int, c_int_p, c_int_p, C.c_int]),
    "pcu_sparsemat_destroy": (None, [VP]),
    "pcu_sparsemat_set_data": (C.c_int, [VP, c_double_p]),
    "pcu_sparsemat_data_device_ptr": (c_double_p, [VP]),
    "pcu_sparsemat_factor": (C.c_int, [VP, VP, VP, VP]),
    "pcu_sparsemat_apply3": (C.c_int, [VP, VP, VP, VP]),
    "pcu_sparsemat_apply4": (C.c_int, [VP, VP, VP, VP, VP]),
    "pcu_sparsemat_mult_add": (C.c_int, [VP, C.c_double, VP, VP]),
    "pcu_sparsemat_mult_transpose_add": (C.c_int, [VP, C.c_double, VP, VP]),
    "pcu_sparsemat_info": (C.c_int, [VP, c_int_p, c_int_p, c_int_p, c_int_p]),
    "pcu_sparsemat_symbolic": (C.c_int, [VP] + [c_int_p] * 11),
    "pcu_blockmat_destroy": (None, [VP]),
    "pcu_blockmat_factor": (C.c_int, [VP, VP, VP, VP]),
    "pcu_blockmat_apply3": (C.c_int, [VP, VP, VP, VP]),
    "pcu_blockmat_apply4": (C.c_int, [VP, VP, VP, VP, VP]),
    "pcu_qn_create": (VP, [VP, C.c_int, C.c_char_p, C.c_int]),
    "pcu_qn_destroy": (None, [VP]),
    "pcu_qn_set_option": (C.c_int, [VP, C.c_char_p, C.c_char_p]),
    "pcu_qn_reset": (C.c_int, [VP]),
    "pcu_qn_max_size": (C.c_int, [VP]),
    "pcu_qn_update": (C.c_int, [VP, VP, VP, C.POINTER(C.c_int)]),
    "pcu_qn_mult": (C.c_int, [VP, VP, VP]),
    "pcu_qn_mult_add": (C.c_int, [VP, C.c_double, VP, VP]),
    "pcu_qn_compact": (C.c_int, [VP, c_double_p, c_double_p, c_double_p, C.POINTER(VP)]),
    "pcu_ip_set_quasi_newton": (C.c_int, [VP, VP]),
    "pcu_vec_scale": (C.c_int, [VP, C.c_double]),
    "pcu_vec_axpy": (C.c_int, [VP, C.c_double, VP]),
    "pcu_vec_device_ptr": (VP, [VP]),
    "pcu_vec_host_ptr": (VP, [VP]),
    "pcu_vec_is_managed": (C.c_int, [VP]),
    "pcu_ip_reset_design_and_bounds": (C.c_int, [VP]),
    "pcu_ip_set_penalty_gamma": (C.c_int, [VP, C.c_double]),
    "pcu_ip_set_penalty_gamma_array": (C.c_int, [VP, c_double_p]),
    "pcu_ip_get_penalty_gamma": (C.c_int, [VP, c_double_p]),
    "pcu_ip_reset_problem": (C.c_int, [VP, VP]),
    "pcu_ip_reset_quasi_newton": (C.c_int, [VP]),
    "pcu_ip_write_solution": (C.c_int, [VP, C.c_char_p]),
    "pcu_ip_read_solution": (C.c_int, [VP, C.c_char_p]),
    "pcu_vec_to_host": (C.c_int, [VP, VP, C.c_int]),
    "pcu_vec_from_host": (C.c_int, [VP, VP, C.c_int]),
    "pcu_problem_create": (VP, [VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                C.c_int, C.POINTER(Weighting), C.POINTER(Callbacks)]),
    "pcu_problem_create_host": (VP, [VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                     C.c_int, C.POINTER(Weighting),
                                     C.POINTER(HostCallbacks)]),
    "pcu_problem_transfer_bytes": (C.c_int, [VP, C.POINTER(C.c_int64),
                                             C.POINTER(C.c_int64)]),
    "pcu_problem_host_times": (C.c_int, [VP, c_double_p, c_double_p, c_double_p]),
    "pcu_problem_destroy": (None, [VP]),
    "pcu_problem_set_hessian_diag": (C.c_int, [VP, VP, HDIAG_CB]),
    "pcu_problem_set_hessian_diag_host": (C.c_int, [VP, VP, HOST_HDIAG_CB]),
    "pcu_ctx_allreduce_sum": (C.c_int, [VP, c_double_p, C.c_int]),
    "pcu_problem_create_sepquad_host": (VP, [VP, C.POINTER(SepQuadParams), C.c_int,
                                             C.POINTER(VP)]),
    "pcu_problem_sepquad_host_free": (None, [VP]),
    "pcu_problem_create_sepquad": (VP, [VP, C.POINTER(SepQuadParams)]),
    "pcu_problem_create_rosenbrock": (VP, [VP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "pcu_problem_sizes": (C.c_int, [VP, c_int_p, c_int_p, c_int_p]),
    "pcu_problem_callback_ms": (C.c_double, [VP]),
    "pcu_ip_create": (VP, [VP]),
    "pcu_ip_destroy": (None, [VP]),
    "pcu_ip_set_option_float": (C.c_int, [VP, C.c_char_p, C.c_double]),
    "pcu_ip_set_option_int": (C.c_int, [VP, C.c_char_p, C.c_int]),
    "pcu_ip_set_option_str": (C.c_int, [VP, C.c_char_p, C.c_char_p]),
    "pcu_ip_optimize": (C.c_int, [VP]),
    "pcu_ip_begin": (C.c_int, [VP]),
    "pcu_ip_iterate": (C.c_int, [VP, C.c_int, c_int_p]),
    "pcu_ip_get_point": (C.c_int, [VP] + [C.POINTER(VP)] * 6),
    "pcu_ip_get_dense": (C.c_int, [VP] + [c_double_p] * 6),
    "pcu_ip_barrier_param": (C.c_double, [VP]),
    "pcu_ip_complementarity": (C.c_int, [VP, c_double_p]),
    "pcu_ip_counters": (C.c_int, [VP, c_int_p, c_int_p, c_int_p]),
    "pcu_ip_status": (C.c_int, [VP]),
    "pcu_tr_create": (VP, [VP]),
    "pcu_tr_destroy": (None, [VP]),
    "pcu_tr_set_option_float": (C.c_int, [VP, C.c_char_p, C.c_double]),
    "pcu_tr_set_option_int": (C.c_int, [VP, C.c_char_p, C.c_int]),
    "pcu_tr_set_option_str": (C.c_int, [VP, C.c_char_p, C.c_char_p]),
    "pcu_tr_optimize": (C.c_int, [VP]),
    "pcu_tr_status": (C.c_int, [VP]),
    "pcu_tr_history_len": (C.c_int, [VP]),
    "pcu_tr_history_get": (C.c_int, [VP, C.c_int, c_double_p]),
    "pcu_tr_history_info": (C.c_char_p, [VP, C.c_int]),
    "pcu_tr_point": (VP, [VP]),
    "pcu_tr_interior_point": (VP, [VP]),
    "pcu_tr_penalty_gamma": (C.c_int, [VP, c_double_p]),
    "pcu_ip_history_len": (C.c_int, [VP]),
    "pcu_ip_history_get": (C.c_int, [VP, C.c_int, c_double_p, C.c_int]),
    "pcu_ip_history_info": (C.c_char_p, [VP, C.c_int]),
    "pcu_ip_iter_times": (C.c_int, [VP, C.c_int, c_double_p, c_double_p, c_double_p]),
    "pcu_ip_vars_vec": (VP, [VP, C.c_int, C.c_int]),
    "pcu_ip_vars_dense_get": (C.c_int, [VP, C.c_int, c_double_p]),
    "pcu_ip_vars_dense_set": (C.c_int, [VP, C.c_int, c_double_p]),
    "pcu_ip_state_vec": (VP, [VP, C.c_int]),
    "pcu_ip_set_obj_con": (C.c_int, [VP, C.c_double, c_double_p]),
    "pcu_ip_set_barrier": (C.c_int, [VP, C.c_double, C.c_double]),
    "pcu_ip_qn_update": (C.c_int, [VP, VP, VP, c_int_p]),
    "pcu_ip_qn_reset": (C.c_int, [VP]),
    "pcu_ip_qn_mult": (C.c_int, [VP, VP, VP]),
    "pcu_ip_qn_compact": (C.c_int, [VP, c_double_p, c_int_p, c_double_p, c_double_p]),
    "pcu_ip_kkt_res": (C.c_int, [VP, C.c_int, C.c_double, C.c_int]),
    "pcu_ip_res_norm": (C.c_int, [VP] + [c_double_p] * 4),
    "pcu_ip_comp": (C.c_int, [VP, c_double_p]),
    "pcu_ip_setup_kkt_diag": (C.c_int, [VP, C.c_int]),
    "pcu_ip_setup_kkt": (C.c_int, [VP, C.c_int]),
    "pcu_ip_kkt_step": (C.c_int, [VP, C.c_int, C.c_int, C.c_int]),
    "pcu_ip_add_kkt_res_step": (C.c_int, [VP, C.c_int, C.c_int]),
    "pcu_ip_kkt_solve": (C.c_int, [VP, C.c_int, C.c_int, C.c_int]),
    "pcu_ip_max_step": (C.c_int, [VP, C.c_double, C.c_int, c_double_p, c_double_p]),
    "pcu_ip_comp_step": (C.c_int, [VP, C.c_double, C.c_double, C.c_int, c_double_p]),
    "pcu_ip_merit_init_deriv": (C.c_int, [VP, C.c_double, c_double_p, c_double_p]),
    "pcu_ip_get_gram": (C.c_int, [VP, c_double_p, c_double_p, c_int_p]),
    "pcu_gram_wide_plan": (C.c_int, [C.c_int] + [c_int_p] * 5 + [C.POINTER(C.c_ubyte)] * 3),
}


def load():
    """Loads the shared library; fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "paropt_b200: %s is missing -- run `python -m paropt_b200.build` "
            "(there is no CPU fallback)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = lib
    return lib
