"""ctypes binding of libcuddh_b200.so (include/cuddh_b200.h). The library is the product: if it is missing
or fails to load this module raises — there is no CPU fallback."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libcuddh_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "cuddh_b200.h")

c_i64 = C.c_int64
c_vp = C.c_void_p
c_dp = C.c_void_p  # device or host pointers are passed as raw addresses

# cuddh_apply_{d,f}_fn: int (*)(void* ctx, const T* x, T* y, void* stream); non-zero aborts the solve
APPLY_D = C.CFUNCTYPE(C.c_int, c_vp, c_vp, c_vp, c_vp)
APPLY_F = C.CFUNCTYPE(C.c_int, c_vp, c_vp, c_vp, c_vp)
# cuddh_apply_batch_f_fn: int (*)(void* ctx, int k, const float* const* x, float* const* y, void* stream); x, y: host pointer arrays
APPLY_BATCH_F = C.CFUNCTYPE(C.c_int, c_vp, C.c_int, C.POINTER(c_vp), C.POINTER(c_vp), c_vp)


class SolverOut(C.Structure):
    _fields_ = [("success", C.c_int), ("num_iter", C.c_int), ("num_matvec", C.c_int), ("n_res", C.c_int)]


class GmresOptions(C.Structure):
    _fields_ = [("orth", C.c_int), ("comm", C.c_void_p), ("d_mask", C.c_void_p), ("time_orth", C.c_int), ("flexible", C.c_int)]


class GmresStats(C.Structure):
    _fields_ = [("orth_bytes", C.c_double), ("orth_ms", C.c_double), ("reorth", C.c_int), ("allreduces", C.c_int)]


class CuddhError(RuntimeError):
    pass


_lib = None


def _proto(lib):
    P = C.POINTER
    sig = {
        "cuddh_b200_version": (C.c_int, []),
        "cuddh_b200_last_error": (C.c_char_p, []),
        "cuddh_b200_launch_count": (c_i64, []),
        "cuddh_b200_quadrature": (C.c_int, [C.c_int, C.c_int, c_vp, c_vp]),
        "cuddh_b200_basis_create": (C.c_int, [C.c_int, P(c_vp)]),
        "cuddh_b200_basis_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_basis_eval": (C.c_int, [c_vp, C.c_int, c_vp, c_vp]),
        "cuddh_b200_basis_deriv": (C.c_int, [c_vp, C.c_int, c_vp, c_vp]),
        "cuddh_b200_basis_nodes": (C.c_int, [c_vp, c_vp, c_vp]),
        "cuddh_b200_mesh_uniform_rect": (C.c_int, [C.c_int, C.c_double, C.c_double, C.c_int, C.c_double, C.c_double, P(c_vp)]),
        "cuddh_b200_mesh_from_vertices": (C.c_int, [c_i64, c_vp, c_i64, c_vp, P(c_vp)]),
        "cuddh_b200_mesh_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_mesh_sizes": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_mesh_edges": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_mesh_boundary_edges": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_mesh_h": (C.c_int, [c_vp, P(C.c_double), P(C.c_double)]),
        "cuddh_b200_h1space_create": (C.c_int, [c_vp, C.c_int, P(c_vp)]),
        "cuddh_b200_h1space_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_h1space_size": (c_i64, [c_vp]),
        "cuddh_b200_h1space_global_indices": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_h1space_physical_coordinates": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_h1space_device_indices": (c_vp, [c_vp]),
        "cuddh_b200_h1space_device_coordinates": (c_vp, [c_vp]),
        "cuddh_b200_h1space_host_indices": (c_vp, [c_vp]),
        "cuddh_b200_h1space_host_coordinates": (c_vp, [c_vp]),
        "cuddh_b200_h1space_device_corners": (c_vp, [c_vp]),
        "cuddh_b200_element_metrics": (C.c_int, [c_vp, C.c_int, c_vp, C.c_int, c_dp, c_vp]),
        "cuddh_b200_linear_functional_assemble": (C.c_int, [c_vp, C.c_int, c_vp, c_dp, C.c_double, c_dp, c_vp]),
        "cuddh_b200_mesh_vertices": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_mesh_elements": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_facespace_indices_ptr": (c_vp, [c_vp, C.c_int, C.c_int]),
        "cuddh_b200_facespace_n_faces": (c_i64, [c_vp]),
        "cuddh_b200_face_linear_functional_assemble": (C.c_int, [c_vp, C.c_int, c_vp, c_dp, C.c_double, c_dp, c_vp]),
        "cuddh_b200_ensemble_create": (C.c_int, [c_vp, C.c_int, c_vp, P(c_vp)]),
        "cuddh_b200_ensemble_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_ensemble_info": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_ensemble_array": (c_vp, [c_vp, C.c_char_p, P(c_i64)]),
        "cuddh_b200_facespace_create": (C.c_int, [c_vp, c_i64, c_vp, P(c_vp)]),
        "cuddh_b200_facespace_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_facespace_size": (c_i64, [c_vp]),
        "cuddh_b200_facespace_subspace_indices": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_facespace_global_indices": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_facespace_restrict": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_facespace_prolong": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_facespace_orth": (C.c_int, [c_vp, c_dp, c_vp]),
        "cuddh_b200_stiffness_create": (C.c_int, [c_vp, C.c_int, C.c_int, P(c_vp)]),
        "cuddh_b200_mass_create": (C.c_int, [c_vp, c_dp, C.c_int, P(c_vp)]),
        "cuddh_b200_diag_inv_mass_create": (C.c_int, [c_vp, c_dp, P(c_vp)]),
        "cuddh_b200_facemass_create": (C.c_int, [c_vp, c_dp, C.c_int, P(c_vp)]),
        "cuddh_b200_diag_inv_facemass_create": (C.c_int, [c_vp, c_dp, P(c_vp)]),
        "cuddh_b200_helmholtz_create": (C.c_int, [C.c_double, c_dp, c_dp, c_vp, c_vp, P(c_vp)]),
        "cuddh_b200_operator_apply": (C.c_int, [c_vp, C.c_double, C.c_int, c_dp, c_dp, c_vp]),
        "cuddh_b200_facemass_apply_h1": (C.c_int, [c_vp, C.c_double, c_dp, c_dp, c_vp]),
        "cuddh_b200_operator_time_phases": (C.c_int, [c_vp, c_dp, c_dp, C.c_int, P(C.c_float), P(C.c_float), c_vp]),
        "cuddh_b200_operator_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_operator_bytes": (c_i64, [c_vp]),
        "cuddh_b200_operator_kernel_kind": (C.c_int, [c_vp]),
        "cuddh_b200_operator_bytes_moved": (c_i64, [c_vp]),
        "cuddh_b200_operator_is_affine": (C.c_int, [c_vp]),
        "cuddh_b200_h1space_check_plan": (C.c_int, [c_vp, C.c_int, P(c_i64)]),
        "cuddh_b200_axpby_d": (C.c_int, [c_i64, C.c_double, c_dp, C.c_double, c_dp, c_vp]),
        "cuddh_b200_axpby_f": (C.c_int, [c_i64, C.c_float, c_dp, C.c_float, c_dp, c_vp]),
        "cuddh_b200_dot_d": (C.c_int, [c_i64, c_dp, c_dp, P(C.c_double), c_vp]),
        "cuddh_b200_dot_f": (C.c_int, [c_i64, c_dp, c_dp, P(C.c_float), c_vp]),
        "cuddh_b200_dist_d": (C.c_int, [c_i64, c_dp, c_dp, P(C.c_double), c_vp]),
        "cuddh_b200_dist_f": (C.c_int, [c_i64, c_dp, c_dp, P(C.c_float), c_vp]),
        "cuddh_b200_copy_d": (C.c_int, [c_i64, c_dp, c_dp, c_vp]),
        "cuddh_b200_copy_f": (C.c_int, [c_i64, c_dp, c_dp, c_vp]),
        "cuddh_b200_copy_i": (C.c_int, [c_i64, c_dp, c_dp, c_vp]),
        "cuddh_b200_scal_d": (C.c_int, [c_i64, C.c_double, c_dp, c_vp]),
        "cuddh_b200_scal_f": (C.c_int, [c_i64, C.c_float, c_dp, c_vp]),
        "cuddh_b200_fill_d": (C.c_int, [c_i64, C.c_double, c_dp, c_vp]),
        "cuddh_b200_fill_f": (C.c_int, [c_i64, C.c_float, c_dp, c_vp]),
        "cuddh_b200_fill_i": (C.c_int, [c_i64, C.c_int, c_dp, c_vp]),
        "cuddh_b200_gmres_d": (C.c_int, [c_i64, c_dp, c_vp, c_vp, c_dp, c_vp, c_vp, C.c_int, C.c_int, C.c_double, C.c_int,
                                         C.c_double, P(SolverOut), c_vp, c_vp, C.c_int, c_vp]),
        "cuddh_b200_gmres_f": (C.c_int, [c_i64, c_dp, c_vp, c_vp, c_dp, C.c_int, C.c_int, C.c_float, C.c_int, C.c_double,
                                         P(SolverOut), c_vp, c_vp, C.c_int, c_vp]),
        "cuddh_b200_gmres_d_ex": (C.c_int, [c_i64, c_dp, c_vp, c_vp, c_dp, c_vp, c_vp, C.c_int, C.c_int, C.c_double, C.c_int,
                                            C.c_double, P(GmresOptions), P(SolverOut), c_vp, c_vp, C.c_int, P(GmresStats), c_vp]),
        "cuddh_b200_gmres_f_ex": (C.c_int, [c_i64, c_dp, c_vp, c_vp, c_dp, C.c_int, C.c_int, C.c_float, C.c_int, C.c_double,
                                            P(GmresOptions), P(SolverOut), c_vp, c_vp, C.c_int, P(GmresStats), c_vp]),
        "cuddh_b200_operator_as_apply": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_as_apply": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_set_option": (C.c_int, [C.c_char_p, c_i64]),
        "cuddh_b200_get_option": (c_i64, [C.c_char_p]),
        "cuddh_b200_comm_unique_id": (C.c_int, [c_vp]),
        "cuddh_b200_comm_create": (C.c_int, [c_vp, C.c_int, C.c_int, P(c_vp)]),
        "cuddh_b200_comm_wrap": (C.c_int, [c_vp, C.c_int, C.c_int, P(c_vp)]),
        "cuddh_b200_comm_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_comm_allreduce_d": (C.c_int, [c_vp, c_dp, c_i64, c_vp]),
        "cuddh_b200_slab_create": (C.c_int, [c_vp, C.c_int, C.c_int, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp, P(c_vp)]),
        "cuddh_b200_slab_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_slab_bytes": (c_i64, [c_vp]),
        "cuddh_b200_slab_uses_peer_memory": (C.c_int, [c_vp]),
        "cuddh_b200_slab_exchange": (C.c_int, [c_vp, c_dp, c_vp]),
        "cuddh_b200_slab_mask": (c_vp, [c_vp]),
        "cuddh_b200_helmholtz_apply_slab": (C.c_int, [c_vp, c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_slab_bind": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_slab_as_apply": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_kernel_kind": (C.c_int, [c_vp]),
        "cuddh_b200_ddh_dist_create": (C.c_int, [c_vp, c_vp, C.c_int, C.c_int, P(c_vp)]),
        "cuddh_b200_ddh_dist_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_ddh_dist_info": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_ddh_dist_get_array": (C.c_int, [c_vp, C.c_char_p, c_vp, c_i64, P(c_i64)]),
        "cuddh_b200_ddh_dist_mask": (c_vp, [c_vp]),
        "cuddh_b200_ddh_dist_buffers": (C.c_int, [c_vp, P(c_vp), P(c_vp)]),
        "cuddh_b200_ddh_dist_rhs": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_dist_action": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_dist_apply_T": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_dist_postprocess": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_dist_as_apply": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_create": (C.c_int, [C.c_double, c_vp, c_vp, C.c_int, C.c_int, C.c_int, P(c_vp)]),
        "cuddh_b200_ddh_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_ddh_size": (c_i64, [c_vp]),
        "cuddh_b200_ddh_rhs": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_action": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_postprocess": (C.c_int, [c_vp, c_dp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_apply_T_range": (C.c_int, [c_vp, c_dp, c_dp, C.c_int, C.c_int, c_vp]),
        "cuddh_b200_ddh_rhs_range": (C.c_int, [c_vp, c_dp, c_dp, C.c_int, C.c_int, c_vp]),
        "cuddh_b200_ddh_postprocess_range": (C.c_int, [c_vp, c_dp, c_dp, c_dp, C.c_int, C.c_int, c_vp]),
        "cuddh_b200_ddh_info": (C.c_int, [c_vp, c_vp, P(C.c_double)]),
        "cuddh_b200_ddh_get_array": (C.c_int, [c_vp, C.c_char_p, c_vp, c_i64, P(c_i64)]),
        "cuddh_b200_ddh_flops": (C.c_double, [c_vp]),
        "cuddh_b200_ddh_transfer_slots": (C.c_int, [c_vp, c_vp, c_vp, c_i64, P(C.c_int)]),
        "cuddh_b200_ddh_transfer_orphans": (C.c_int, [c_vp, c_vp, c_i64, P(c_i64)]),
        "cuddh_b200_ddh_transfer_create": (C.c_int, [c_vp, c_i64, c_vp, P(c_vp)]),
        "cuddh_b200_ddh_transfer_destroy": (C.c_int, [c_vp]),
        "cuddh_b200_ddh_transfer_action": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_transfer_as_apply": (C.c_int, [c_vp, c_dp, c_dp, c_vp]),
        "cuddh_b200_ddh_transfer_info": (C.c_int, [c_vp, c_vp]),
        "cuddh_b200_ddh_transfer_get_block": (C.c_int, [c_vp, C.c_int, c_vp]),
        "cuddh_b200_ddh_transfer_action_batch": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp]),
        "cuddh_b200_ddh_transfer_as_apply_batch": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, c_vp]),
        "cuddh_b200_gmres_f_batch": (C.c_int, [c_i64, C.c_int, c_vp, c_vp, c_vp, c_vp, C.c_int, C.c_int, C.c_float, C.c_double,
                                               c_vp, c_vp, c_vp, C.c_int, c_vp]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return sig


SIGNATURES = None


def load():
    """Load the shared library (once). Raises if it has not been built: run __graft_entry__.build()."""
    global _lib, SIGNATURES
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CuddhError("libcuddh_b200.so is missing (%s): build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                             "or `make -C cuddhelmholtz_b200/csrc`. There is no CPU fallback." % LIB_PATH)
        _lib = C.CDLL(LIB_PATH)
        SIGNATURES = _proto(_lib)
    return _lib


def check(status):
    if status != 0:
        msg = load().cuddh_b200_last_error()
        raise CuddhError("cuddh_b200 error %d: %s" % (status, (msg or b"").decode()))
