"""ctypes binding of libdiffsound_sm100.so (the C-ABI in include/diffsound_sm100.h).

There is no fallback: if the shared library is missing the import raises, and
every wrapper raises RuntimeError(ds_last_error()) on a non-zero return code.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libdiffsound_sm100.so")

_lib = None

i32p = C.c_void_p
f64p = C.c_void_p
f32p = C.c_void_p
i64p = C.c_void_p
ptr = C.c_void_p
i64 = C.c_int64
cint = C.c_int
dbl = C.c_double


class LobpcgOpts(C.Structure):
    _fields_ = [("nev", C.c_int), ("maxit", C.c_int), ("cheb_degree", C.c_int), ("tol", C.c_double),
                ("sigma", C.c_double), ("cheb_ratio", C.c_double), ("n_rigid", C.c_int), ("verbose", C.c_int),
                ("smooth_steps", C.c_int), ("coarse_degree", C.c_int), ("smooth_ratio", C.c_double),
                ("coarse_ratio", C.c_double), ("nested", C.c_int), ("nested_tol", C.c_double),
                ("nested_degree", C.c_int), ("coords", C.c_void_p), ("locked", C.c_void_p), ("n_locked", C.c_int), ("precond_fp64", C.c_int), ("ortho_w", C.c_int),
                ("fixed", C.c_void_p)]


class PmgLevel(C.Structure):
    _fields_ = [("brow", C.c_void_p), ("bcol", C.c_void_p), ("n_nodes", C.c_int64), ("nnzb", C.c_int64),
                ("Kval", C.c_void_p), ("Mblk", C.c_void_p), ("parents", C.c_void_p), ("rptr", C.c_void_p),
                ("rlist", C.c_void_p), ("coords", C.c_void_p), ("fixed", C.c_void_p)]


# name -> (restype, argtypes); mirrors include/diffsound_sm100.h one to one
SIGNATURES = {
    "ds_version": (cint, []),
    "ds_last_error": (C.c_char_p, []),
    "ds_workspace_create": (cint, [C.POINTER(C.c_void_p)]),
    "ds_workspace_destroy": (cint, [ptr]),
    "ds_workspace_bytes": (i64, [ptr]),
    "ds_pattern_count": (cint, [ptr, i32p, i64, cint, i64, C.POINTER(C.c_int64), ptr]),
    "ds_pattern_fill": (cint, [ptr, i64, i32p, i32p, i32p, i32p, i32p, ptr]),
    "ds_pattern_expand_csr": (cint, [i32p, i32p, i64, i64, i64p, i64p, ptr]),
    "ds_assemble_km": (cint, [f32p, i32p, i64, cint, i64, dbl, dbl, f64p, f64p, i32p, i32p, i32p, i32p, i64,
                              f64p, f64p, f64p, ptr]),
    "ds_assemble_km_tets": (cint, [f32p, i32p, i64, cint, i64, dbl, dbl, f64p, f64p, i32p, i32p, i32p, i32p, i32p, cint, i64,
                                   f64p, f64p, f64p, ptr]),
    "ds_assemble_km_field": (cint, [f32p, i32p, i64, cint, i64, f64p, f64p, f32p, f64p, f32p, i32p, i32p, i32p, i32p, i64,
                                    f64p, f64p, f64p, ptr]),
    "ds_assemble_km_tets_field": (cint, [f32p, i32p, i64, cint, i64, f64p, f64p, f32p, f64p, f32p, i32p, i32p, i32p, i32p,
                                         i32p, cint, i64, f64p, f64p, f64p, ptr]),
    "ds_assemble_km_tensor": (cint, [f32p, i32p, i64, cint, i64, f64p, f32p, f64p, f32p, i32p, i32p, i32p, i32p, i64,
                                     f64p, f64p, f64p, ptr]),
    "ds_assemble_km_tets_tensor": (cint, [f32p, i32p, i64, cint, i64, f64p, f32p, f64p, f32p, i32p, i32p, i32p, i32p, i32p,
                                          cint, i64, f64p, f64p, f64p, ptr]),
    "ds_mass_expand": (cint, [i32p, i64, i64, f64p, f64p, ptr]),
    "ds_fix_nodes_km": (cint, [i32p, i32p, i64, i64, ptr, f64p, f64p, ptr]),
    "ds_support_km": (cint, [f32p, i32p, i64, cint, i64, i32p, i32p, i64, f64p, f64p, i32p, i32p, i32p, i64, i32p, i32p,
                             i32p, i64, f64p, ptr]),
    "ds_support_grad": (cint, [f32p, i32p, i64, cint, i64, i32p, i32p, i64, f64p, f64p, f64p, i64, cint, f64p, i32p, i32p,
                               i32p, i64, f64p, f64p, f64p, ptr]),
    "ds_support_energies": (cint, [f32p, i32p, i64, cint, i64, i32p, i32p, i64, f64p, f64p, f64p, i64, cint, f64p, ptr]),
    "ds_assemble_mass_coo": (cint, [f64p, i32p, i64, cint, f64p, dbl, f64p, i32p, i32p, ptr]),
    "ds_spmm_km": (cint, [i32p, i32p, i64, f64p, f64p, dbl, f64p, i64, cint, dbl, dbl, f64p, i64, f64p, i64, ptr]),
    "ds_spmm_k_and_m": (cint, [i32p, i32p, i64, f64p, f64p, f64p, i64, cint, f64p, i64, f64p, i64, ptr]),
    "ds_gram_scratch_elems": (i64, [cint, cint]),
    "ds_gram_f64": (cint, [f64p, i64, cint, f64p, i64, cint, i64, f64p, i64, f64p, ptr]),
    "ds_gram_sym2_scratch_elems": (i64, []),
    "ds_gram_sym2_f64": (cint, [f64p, f64p, f64p, i64, i64, C.POINTER(C.c_int), cint, f64p, f64p, i64, f64p, ptr]),
    "ds_rr_update_f64": (cint, [f64p, f64p, f64p, i64, cint, cint, f64p, f64p, cint, i64, i64, f64p, f64p, f64p, i64, ptr]),
    "ds_block_gemm_f64": (cint, [f64p, i64, cint, f64p, i64, cint, i64, dbl, f64p, i64, ptr]),
    "ds_eigh_scratch_elems": (i64, [cint]),
    "ds_eigh_generalized_f64": (cint, [f64p, f64p, cint, i64, dbl, f64p, f64p, i64, f64p, ptr, ptr]),
    "ds_lobpcg": (cint, [ptr, i32p, i32p, i64, f64p, f64p, C.POINTER(PmgLevel), f64p, cint, C.POINTER(LobpcgOpts),
                         f64p, f64p, C.POINTER(C.c_int64), ptr]),
    "ds_k32_record_bytes": (i64, [i64]),
    "ds_k32_pack": (cint, [i32p, i32p, i64, i64, f64p, f64p, dbl, ptr, f32p, ptr]),
    "ds_unique_rows3_count": (cint, [ptr, f32p, i64, C.POINTER(C.c_int64), ptr]),
    "ds_unique_rows3_fill": (cint, [ptr, ptr, ptr, ptr]),
    "ds_spmm32": (cint, [cint, i32p, ptr, i64, cint, f32p, f32p, f32p, f32p, f32p, dbl, dbl, i32p, ptr]),
    "ds_spmm32_chunk_count": (cint, [i64]),
    "ds_cheb32_solve": (cint, [i32p, ptr, f32p, i64, i64, f32p, cint, cint, dbl, dbl, cint, f32p, f32p, C.POINTER(cint), ptr]),
    "ds_spmm32_chunks": (cint, [i32p, i64, i32p, ptr]),
    "ds_k32_pack_slab": (cint, [i32p, i32p, i64, i64, i64, f64p, f64p, dbl, ptr, ptr, f32p, ptr]),
    "ds_spmm32_rowpart": (cint, [cint, i32p, ptr, i64, cint, C.POINTER(C.c_void_p), cint, cint, f32p, f32p, f32p, f32p,
                                 dbl, dbl, ptr]),
    "ds_peer_alloc": (cint, [i64, C.POINTER(C.c_void_p), C.POINTER(C.c_ubyte)]),
    "ds_peer_open": (cint, [C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]),
    "ds_peer_close": (cint, [ptr]),
    "ds_peer_free": (cint, [ptr]),
    "ds_pmg_coarse_count": (cint, [ptr, i32p, i64, i64, i32p, C.POINTER(C.c_int64), ptr]),
    "ds_pmg_coarse_fill": (cint, [ptr, f32p, i32p, i64, i64, i32p, i64, i32p, f32p, i32p, i32p, i32p, ptr]),
    "ds_pmg_restrict32": (cint, [i32p, i32p, i64, f32p, cint, f32p, ptr]),
    "ds_pmg_prolong_add32": (cint, [i32p, i64, f32p, cint, f32p, ptr]),
    "ds_corner_incidence": (cint, [ptr, i32p, i64, cint, cint, i64, i32p, i32p, ptr]),
    "ds_eigval_grad_shape": (cint, [f32p, i32p, i64, cint, i64, dbl, dbl, f64p, f64p, f64p, i64, cint, f64p, f64p,
                                    i32p, i32p, f64p, f32p, ptr]),
    "ds_eigval_grad_shape_field": (cint, [f32p, i32p, i64, cint, i64, f64p, f64p, f32p, f64p, f64p, f64p, i64, cint, f64p,
                                          f64p, i32p, i32p, f64p, f32p, ptr]),
    "ds_material_field_grad": (cint, [f32p, i32p, i64, cint, f32p, dbl, f64p, i64, cint, f64p, f64p, f64p, ptr]),
    "ds_element_energies": (cint, [f32p, i32p, i64, cint, f32p, dbl, f64p, i64, cint, f64p, f64p, f32p, f64p, f64p, ptr]),
    "ds_eigval_grad_shape_tensor": (cint, [f32p, i32p, i64, cint, i64, f64p, f32p, f64p, f64p, f64p, i64, cint, f64p, f64p,
                                           i32p, i32p, f64p, f32p, ptr]),
    "ds_elasticity_field_grad": (cint, [f32p, i32p, i64, cint, f32p, dbl, f64p, i64, cint, f64p, f64p, f64p, f64p, ptr]),
    "ds_element_energies_tensor": (cint, [f32p, i32p, i64, cint, f32p, dbl, f64p, i64, cint, f64p, f32p, f64p, f64p, ptr]),
    "ds_quadform_scratch_elems": (i64, [cint]),
    "ds_eigval_quadforms_material": (cint, [f32p, i32p, i64, cint, f64p, dbl, f64p, i64, cint, f64p, f64p, ptr]),
    "ds_synth_scratch_elems": (i64, [i64, cint, i64]),
    "ds_modal_synth_fwd": (cint, [f32p, f32p, f32p, i64, cint, i64, dbl, f32p, f32p, ptr]),
    "ds_force_fir": (cint, [f32p, f32p, i64, i64, cint, cint, f32p, ptr]),
    "ds_filtered_noise_fwd": (cint, [f32p, f32p, i64, cint, cint, cint, i64, dbl, f32p, ptr]),
    "ds_filtered_noise_bwd": (cint, [f32p, f32p, f32p, i64, cint, cint, cint, i64, dbl, f32p, ptr]),
    "ds_stft_frames": (cint, [i64, cint]),
    "ds_stft_power": (cint, [f32p, i64, i64, cint, cint, f32p, ptr]),
    "ds_mss_scratch_elems": (i64, [i64, i64, cint, cint]),
    "ds_mss_loss_fwd": (cint, [f32p, f32p, i64, i64, cint, cint, cint, dbl, dbl, f32p, f64p, ptr]),
    "ds_mss_loss_bwd": (cint, [f32p, f32p, i64, i64, cint, cint, cint, dbl, dbl, f64p, dbl, f32p, f32p, cint, ptr]),
    "ds_prof_read_work": (cint, [cint, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "ds_gram_strip_scratch_elems": (i64, []),
    "ds_gram_strip_f64": (cint, [f64p, f64p, i64, cint, f64p, i64, cint, i64, f64p, f64p, i64, f64p, ptr]),
    "ds_rr_update2_f64": (cint, [f64p, f64p, f64p, i64, cint, cint, cint, f64p, i64, i64, f64p, f64p, f64p, i64, ptr]),
    "ds_gram_algebra_scratch_elems": (i64, []),
    "ds_gram_algebra_f64": (cint, [f64p, f64p, f64p, f64p, i64, f64p, i64, f64p, cint, f64p, ptr]),
    "ds_fp64_peak": (cint, [cint, cint, cint, f64p, C.POINTER(C.c_double), ptr]),
    "ds_mtet_count": (cint, [ptr, f32p, dbl, i64p, i64, i64, C.POINTER(C.c_int64), ptr]),
    "ds_mtet_fill": (cint, [ptr, i64p, i64p, i64p, i64p, ptr]),
    "ds_compact_ids_count": (cint, [ptr, i64p, i64, i64, C.POINTER(C.c_int64), ptr]),
    "ds_compact_ids_fill": (cint, [ptr, i64p, i64p, i64p, ptr]),
    "ds_tet_components_count": (cint, [ptr, i64p, i64, i64, i32p, C.POINTER(C.c_int64), ptr]),
    "ds_tet_components_fill": (cint, [ptr, i64p, i64p, i64p, ptr]),
    "ds_mesh_sdf": (cint, [ptr, f32p, i64, i64p, i64, f32p, i64, cint, f32p, ptr]),
    "ds_mesh_sdf_nearest": (cint, [ptr, f32p, i64, i64p, i64, f32p, i64, cint, f32p, i32p, ptr]),
    "ds_mesh_sdf_backward": (cint, [ptr, f32p, i64, i64p, i64, f32p, i64, i32p, f32p, f32p, f32p, f32p, ptr]),
    "ds_mesh_winding_number": (cint, [ptr, f32p, i64, i64p, i64, f32p, i64, cint, f32p, ptr]),
    "ds_mesh_sdf_winding": (cint, [ptr, f32p, i64, i64p, i64, f32p, i64, cint, f32p, i32p, ptr]),
    "ds_stuff_edges_count": (cint, [ptr, ptr, i64, i64, i64, C.POINTER(C.c_int64), ptr]),
    "ds_stuff_edges_fill": (cint, [ptr, ptr, i64p, i64p, ptr]),
    "ds_stuff_count": (cint, [ptr, ptr, i64, i64, i64, C.POINTER(C.c_double), dbl, i64p, f64p, i64, C.POINTER(C.c_int64), ptr]),
    "ds_stuff_fill": (cint, [ptr, ptr, i64p, f64p, i64p, f32p, ptr]),
    "ds_tet_boundary_count": (cint, [ptr, f32p, i64, i32p, i64, cint, C.POINTER(C.c_int64), ptr]),
    "ds_tet_boundary_fill": (cint, [ptr, i32p, i32p, i32p, ptr]),
    "ds_modal_gains": (cint, [ptr, f32p, i64, i32p, i64, cint, i32p, i32p, i32p, i64, f32p, i32p, f32p, i64, f64p, i64, cint,
                              f32p, f32p, ptr]),
    "ds_modal_gains_backward": (cint, [ptr, f32p, i64, i32p, i64, cint, i32p, i32p, i32p, i64, f32p, i32p, f32p, i64, f64p,
                                       i64, cint, f32p, f32p, f32p, ptr]),
    "ds_lobpcg_residual": (cint, [f64p, f64p, i64, cint, i64, f64p, f64p, i64, f64p, f64p, ptr]),
    "ds_gather_cols_f32": (cint, [f64p, i64, C.POINTER(C.c_int), cint, cint, i64, f32p, ptr]),
    "ds_widen_f32": (cint, [f32p, cint, i64, f64p, i64, ptr]),
    "ds_jacobi32": (cint, [f32p, f32p, i64, cint, dbl, f32p, ptr]),
    "ds_spmm_dual_z32": (cint, [i32p, i32p, i64, i64, i32p, f64p, f64p, f32p, cint, f64p, i64, f64p, i64, ptr]),
    "ds_pmg_restrict32_range": (cint, [i32p, i32p, i64, f32p, cint, i64, i64, f32p, ptr]),
    "ds_pmg_prolong64": (cint, [i32p, i64, f64p, i64, cint, f64p, i64, ptr]),
    "ds_gram_insert_f64": (cint, [f64p, f64p, i64, f64p, f64p, i64, cint, cint, ptr]),
    "ds_sym_upper_f64": (cint, [f64p, f64p, i64, cint, ptr]),
    "ds_eigh_generalized_idx_f64": (cint, [f64p, f64p, cint, i64, C.POINTER(C.c_int), dbl, f64p, f64p, i64, f64p, ptr, ptr]),
    "ds_prof_enable": (cint, [cint]),
    "ds_prof_reserve": (cint, [cint]),
    "ds_prof_enable_classes": (cint, [C.c_uint32]),
    "ds_prof_reset": (cint, []),
    "ds_prof_num_classes": (cint, []),
    "ds_launch_count": (i64, []),
    "ds_prof_class_name": (C.c_char_p, [cint]),
    "ds_prof_read": (cint, [cint, C.POINTER(C.c_double), C.POINTER(C.c_int64)]),
    "ds_modal_synth_bwd": (cint, [f32p, f32p, f32p, f32p, i64, cint, i64, dbl, f32p, f32p, f32p, f32p, ptr]),
}


def load():
    """Load the shared library (once) and set the ctypes prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: build it with `python -m diffsound_b200.build` "
            "(nvcc, sm_100a). There is no CPU or PyTorch fallback for this path.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        except AttributeError:
            if os.environ.get("DIFFSOUND_PARTIAL_LIB") == "1":   # bring-up only
                continue
            raise
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error():
    return load().ds_last_error().decode(errors="replace")


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what} failed (code {rc}): {last_error()}")
