"""ctypes binding of libmgb200.so (C ABI declared in include/mgb200.h).

The library is built in-tree by `learnmultigrid_b200._lib.build()` (nvcc, sm_100a only).  There is no CPU
fallback: every compute entry point raises if the library is missing or no CUDA device is present.
"""
import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmgb200.so")
CSRC = os.path.join(_HERE, "csrc")

c_i32p = ctypes.c_void_p      # device pointers travel as integers
c_f64p = ctypes.c_void_p
c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_dbl = ctypes.c_double
c_vp = ctypes.c_void_p

MG_SMOOTH_JACOBI, MG_SMOOTH_MCGS, MG_SMOOTH_LEXGS, MG_SMOOTH_CHEBY = 0, 1, 2, 3
MG_COARSE_DENSE, MG_COARSE_BCR = 0, 1
MG_LEVEL_PROPER_COLORING, MG_LEVEL_NONZERO_DIAG = 1, 2
SLICE_IRREGULAR = -2 ** 31


class MgError(RuntimeError):
    pass


class mg_sell(ctypes.Structure):
    _fields_ = [("nrows", c_i64), ("ncols", c_i64), ("nslices", c_i64),
                ("d_slice_ptr", c_vp), ("d_cols", c_vp), ("d_vals", c_vp), ("max_slice_len", c_i64),
                ("uniform_len", c_i64), ("d_slice_rec", c_vp), ("d_rec_table", c_vp),
                ("nrec", ctypes.c_int32), ("n_spec", ctypes.c_int32), ("h_spec_row", ctypes.POINTER(c_i64)),
                ("h_spec_rec", ctypes.POINTER(ctypes.c_int32)), ("d_val_idx", c_vp), ("d_val_table", c_vp),
                ("d_rec_vals", c_vp), ("h_spec_vals", ctypes.POINTER(c_dbl))]


class mg_bcr(ctypes.Structure):
    _fields_ = [("n", c_i64), ("n_pad", c_i64), ("m", c_i64), ("nb", c_i64),
                ("nlevels", ctypes.c_int32), ("pad_", ctypes.c_int32),
                ("d_GL", c_vp * 32), ("d_GU", c_vp * 32), ("d_Dinv", c_vp * 32), ("d_HL", c_vp * 32),
                ("d_HU", c_vp * 32), ("na", c_i64 * 32), ("d_last_inv", c_vp), ("d_f", c_vp), ("d_x", c_vp), ("tail_na", c_i64), ("d_tail", c_vp),
                ("d_perm", c_vp)]


MG_MAX_RANKS = 8


class mg_comm(ctypes.Structure):
    _fields_ = [("rank", ctypes.c_int32), ("world", ctypes.c_int32), ("max_sites", ctypes.c_int32),
                ("dry_run", ctypes.c_int32), ("region_bytes", c_i64), ("d_arena", c_vp * MG_MAX_RANKS),
                ("timeout_s", c_dbl), ("site", ctypes.c_int32), ("all_pairs", ctypes.c_int32),
                ("bump_send", c_i64 * MG_MAX_RANKS), ("bump_recv", c_i64 * MG_MAX_RANKS)]


class mg_xfer(ctypes.Structure):
    _fields_ = [("npeers", ctypes.c_int32), ("pad_", ctypes.c_int32), ("peer", ctypes.c_int32 * MG_MAX_RANKS),
                ("d_send_idx", c_vp * MG_MAX_RANKS), ("send_off", c_i64 * MG_MAX_RANKS),
                ("send_cnt", c_i64 * MG_MAX_RANKS), ("d_recv_idx", c_vp * MG_MAX_RANKS),
                ("recv_off", c_i64 * MG_MAX_RANKS), ("recv_cnt", c_i64 * MG_MAX_RANKS)]


class mg_dist_level(ctypes.Structure):
    _fields_ = [("n_halo", c_i64), ("ncolors", ctypes.c_int32), ("pad_", ctypes.c_int32),
                ("xfer_color", ctypes.POINTER(mg_xfer)), ("xfer_all", ctypes.POINTER(mg_xfer)),
                ("xfer_gather", ctypes.POINTER(mg_xfer)), ("d_gather_tmp", c_vp), ("d_gather_self_idx", c_vp),
                ("n_gather_own", c_i64), ("d_mask_A", c_vp), ("d_mask_Q", c_vp), ("d_mask_QT", c_vp)]


class mg_bcr_dist(ctypes.Structure):
    _fields_ = [("fwd_j0", c_i64 * 32), ("fwd_j1", c_i64 * 32), ("fwd_xfer", ctypes.POINTER(mg_xfer) * 32),
                ("bwd_j0", c_i64 * 32), ("bwd_j1", c_i64 * 32), ("bwd_xfer", ctypes.POINTER(mg_xfer) * 32),
                ("tail_i0", c_i64), ("tail_i1", c_i64), ("tail_xfer", ctypes.POINTER(mg_xfer))]


class mg_dist_norm(ctypes.Structure):
    _fields_ = [("d_partials", c_vp), ("d_local", c_vp), ("d_slots", c_vp), ("d_norm2", c_vp),
                ("after", ctypes.c_int32), ("pad_", ctypes.c_int32)]


class mg_pcg(ctypes.Structure):
    _fields_ = [("d_x", c_vp), ("d_p", c_vp), ("d_Ap", c_vp), ("d_scalars", c_vp), ("d_partials", c_vp),
                ("d_slots", c_vp)]


class mg_gmres(ctypes.Structure):
    _fields_ = [("d_x", c_vp), ("d_V", c_vp), ("d_Z", c_vp), ("ld", c_i64), ("restart", ctypes.c_int32),
                ("pad_", ctypes.c_int32), ("d_H", c_vp), ("d_g", c_vp), ("d_cs", c_vp), ("d_sn", c_vp), ("d_y", c_vp),
                ("d_scalars", c_vp), ("d_partials", c_vp), ("d_slots", c_vp)]


class mg_level(ctypes.Structure):
    _fields_ = [("n", c_i64), ("A", mg_sell), ("d_dinv", c_vp),
                ("ncolors", ctypes.c_int32), ("h_color_ptr", ctypes.POINTER(c_i64)),
                ("d_csr_indptr", c_vp), ("d_csr_indices", c_vp), ("d_csr_values", c_vp),
                ("d_lex_level_ptr", c_vp), ("d_lex_level_rows", c_vp), ("lex_nlevels", c_i64),
                ("Q", mg_sell), ("QT", mg_sell),
                ("d_x", c_vp), ("d_b", c_vp), ("d_r", c_vp), ("d_tmp", c_vp),
                ("coarse_kind", ctypes.c_int32), ("d_coarse_inv", c_vp), ("coarse_bcr", c_vp),
                ("dist", ctypes.POINTER(mg_dist_level)), ("coarse_bcr_dist", ctypes.POINTER(mg_bcr_dist)),
                ("flags", ctypes.c_uint32), ("pad_", ctypes.c_uint32), ("d_diag", c_vp),
                ("cheb_degree", ctypes.c_int32), ("pad2_", ctypes.c_int32), ("h_cheb_coef", ctypes.POINTER(c_dbl))]


class mg_cycle_params(ctypes.Structure):
    _fields_ = [("smoother", ctypes.c_int32), ("nu_pre", ctypes.c_int32), ("nu_post", ctypes.c_int32),
                ("omega", c_dbl), ("zero_guess_skip", ctypes.c_int32), ("reverse_post", ctypes.c_int32),
                ("x0_zero", ctypes.c_int32), ("pad_", ctypes.c_int32)]


# name -> (restype, argtypes).  tests/test_abi.py checks that every function declared in include/mgb200.h is
# listed here and exported by the built library.
_SIGNATURES = {
    "mg_version": (c_int, []),
    "mg_last_error": (ctypes.c_char_p, []),
    "mg_struct_size": (c_i64, [c_int]),
    "mg_set_pdl": (c_int, [c_int]),
    "mg_device_info": (c_int, [ctypes.POINTER(c_int), ctypes.POINTER(c_i64), ctypes.POINTER(c_int)]),
    "mg_spmv_csr": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_residual_csr": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_jacobi_sweep_csr": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_dbl, c_vp]),
    "mg_gs_multicolor_sweep_csr": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(c_i64), c_vp,
                                           c_int, c_vp]),
    "mg_gs_lex_sweep_csr": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_int, c_vp]),
    "mg_prolong_correct_csr": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_sell_spmv": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp]),
    "mg_sell_slice_offsets": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp]),
    "mg_set_implied_min_rows": (c_i64, [c_i64]),
    "mg_tri_boxes_2d": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int32, c_vp, c_vp, c_vp]),
    "mg_tri_incidence_2d": (c_int, [c_i64, c_vp, c_vp, c_vp, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp]),
    "mg_tri_pairs_2d": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_value_dict_workspace": (c_i64, []),
    "mg_value_dict_build": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(c_int), c_vp]),
    "mg_set_value_dict": (c_int, [c_int]),
    "mg_set_implied_values": (c_int, [c_int]),
    "mg_set_short_rows_per_thread": (c_int, [c_int]),
    "mg_set_short_min_rows": (c_i64, [c_i64]),
    "mg_level_inspect": (c_int, [ctypes.POINTER(mg_sell), c_int, c_vp, c_vp, c_vp, c_vp]),
    "mg_sell_residual_rows": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "mg_sell_gs_rows_tail": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_i64, c_i64, c_int, c_vp, c_vp,
                                     ctypes.POINTER(c_int), c_vp]),
    "mg_sell_gs_tail_ok": (c_int, [ctypes.POINTER(mg_sell), c_i64, c_i64]),
    "mg_sell_gs_zero_first": (c_int, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_sell_prolong_correct_rows": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp, c_i64, c_i64, c_vp]),
    "mg_vcycle_norm": (c_int, [ctypes.POINTER(mg_level), c_int, ctypes.POINTER(mg_cycle_params), c_vp, c_vp, c_vp]),
    "mg_set_cycle_fusion": (c_int, [c_int]),
    "mg_pcg_start": (c_int, [c_vp, ctypes.POINTER(mg_level), ctypes.POINTER(mg_pcg), c_vp]),
    "mg_pcg_iterate": (c_int, [c_vp, ctypes.POINTER(mg_level), c_int, ctypes.POINTER(mg_cycle_params),
                               ctypes.POINTER(mg_pcg), c_int, c_vp]),
    "mg_gmres_start": (c_int, [c_vp, ctypes.POINTER(mg_level), ctypes.POINTER(mg_gmres), c_vp]),
    "mg_gmres_iterate": (c_int, [c_vp, ctypes.POINTER(mg_level), c_int, ctypes.POINTER(mg_cycle_params),
                                 ctypes.POINTER(mg_gmres), c_int, c_vp]),
    "mg_gmres_finish": (c_int, [ctypes.POINTER(mg_level), ctypes.POINTER(mg_cycle_params), ctypes.POINTER(mg_gmres),
                                c_int, c_vp]),
    "mg_krylov_partials": (c_i64, [c_i64, ctypes.c_int32]),
    "mg_multi_dot": (c_int, [c_i64, c_vp, c_i64, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp]),
    "mg_multi_axpy_norm": (c_int, [c_i64, c_vp, c_i64, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_scale_inv": (c_int, [c_i64, c_vp, c_vp, c_vp]),
    "mg_gmres_solve_update": (c_int, [c_i64, c_vp, ctypes.c_int32, c_vp, ctypes.c_int32, c_vp, c_vp, c_i64, c_vp,
                                      c_vp]),
    "mg_set_implied_columns": (c_int, [c_int]),
    "mg_set_implied_transfers": (c_int, [c_int]),
    "mg_sell_residual": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp, c_vp]),
    "mg_sell_residual_norm2": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_norm_workspace_size": (c_i64, [c_i64]),
    "mg_set_tma_min_rows": (c_i64, [c_i64]),
    "mg_sell_halo_mask": (c_int, [ctypes.POINTER(mg_sell), c_i64, c_vp, c_vp]),
    "mg_set_fused_exchange": (c_int, [c_int]),
    "mg_set_wide_min_len": (c_i64, [c_i64]),
    "mg_set_wide_max_rows": (c_i64, [c_i64]),
    "mg_sell_jacobi": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp, c_vp, c_dbl, c_vp]),
    "mg_sell_chebyshev": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp, c_vp, c_vp, c_dbl, c_dbl, c_int, c_vp]),
    "mg_chebyshev_zero_first": (c_int, [c_i64, c_dbl, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_sell_gs_rows": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_i64, c_i64, c_vp]),
    "mg_sell_prolong_correct": (c_int, [ctypes.POINTER(mg_sell), c_vp, c_vp, c_vp, c_vp]),
    "mg_dot": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_axpby": (c_int, [c_i64, c_dbl, c_vp, c_dbl, c_vp, c_vp, c_vp]),
    "mg_fill": (c_int, [c_i64, c_dbl, c_vp, c_vp]),
    "mg_gather": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_scatter": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_dense_inverse": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_dense_inverse_workspace": (c_i64, [c_i64]),
    "mg_dense_gemv": (c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_bcr_blocks_from_csr": (c_int, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_dense_inverse_batched": (c_int, [c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "mg_dense_gemm_batched": (c_int, [c_i64, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_dbl, c_dbl, c_vp]),
    "mg_bcr_solve": (c_int, [ctypes.POINTER(mg_bcr), c_vp, c_vp, c_vp]),
    "mg_bcr_solve_dist": (c_int, [ctypes.POINTER(mg_comm), ctypes.POINTER(mg_bcr), ctypes.POINTER(mg_bcr_dist), c_vp,
                                  c_vp, c_vp]),
    "mg_csr_to_dense": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_scan_workspace_size": (c_i64, [c_i64]),
    "mg_exclusive_scan_i32": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "mg_spgemm_symbolic": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp]),
    "mg_spgemm_numeric": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_vp, c_vp,
                                  c_vp, c_vp]),
    "mg_csr_compact_nonzeros": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_sort_workspace_size": (c_i64, [c_i64]),
    "mg_stable_argsort_i32": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_int, c_vp, c_i64, c_vp]),
    "mg_csr_transpose_workspace": (c_i64, [c_i64]),
    "mg_csr_transpose": (c_int, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_invert_permutation": (c_int, [c_i64, c_vp, c_vp, c_vp]),
    "mg_csr_row_lengths": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_csr_permute": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_sell_layout": (c_int, [c_i64, c_vp, c_vp, c_vp, ctypes.POINTER(c_i64), ctypes.POINTER(c_i64),
                               ctypes.POINTER(c_i64), c_vp, c_i64, c_vp]),
    "mg_sell_fill": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_extract_dinv": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_comm_alloc": (c_int, [c_i64, ctypes.POINTER(c_vp)]),
    "mg_comm_free": (c_int, [c_vp]),
    "mg_comm_export": (c_int, [c_vp, ctypes.c_char_p]),
    "mg_comm_import": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_vp)]),
    "mg_comm_unmap": (c_int, [c_vp]),
    "mg_comm_arena_bytes": (c_i64, [ctypes.c_int32, ctypes.c_int32, c_i64]),
    "mg_comm_init": (c_int, [ctypes.POINTER(mg_comm), c_vp]),
    "mg_comm_begin": (c_int, [ctypes.POINTER(mg_comm)]),
    "mg_comm_exchange": (c_int, [ctypes.POINTER(mg_comm), ctypes.POINTER(mg_xfer), c_vp, c_vp, c_vp]),
    "mg_comm_allreduce_sum": (c_int, [ctypes.POINTER(mg_comm), c_vp, c_vp, c_vp, c_vp]),
    "mg_comm_allreduce_sum_n": (c_int, [ctypes.POINTER(mg_comm), c_vp, ctypes.c_int32, c_vp, c_vp, c_vp]),
    "mg_comm_end": (c_int, [ctypes.POINTER(mg_comm), c_vp]),
    "mg_comm_error": (c_int, [ctypes.POINTER(mg_comm), ctypes.POINTER(ctypes.c_int32), c_vp]),
    "mg_csr_remap_cols": (c_int, [c_i64, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_assemble_p1_2d": (c_int, [c_i64, c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_assemble_load_p1_2d": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_coo_fold_sum": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_vector_from_runs": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_coupling_pairs_p1_2d": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_csr_dirichlet_count": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_csr_dirichlet_fill": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_coarsen": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_compact": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_extract_patches": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_count_variants": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_extract_variants": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_contributions": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_fold": (c_int, [c_i64, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_emit": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_row_normalise": (c_int, [c_i64, c_vp, c_vp, c_vp]),
    "mg_nn_cut_count": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_nn_cut_fill": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_amg_strength_count": (c_int, [c_i64, c_vp, c_vp, c_vp, c_dbl, c_vp, c_vp]),
    "mg_amg_strength_fill": (c_int, [c_i64, c_vp, c_vp, c_vp, c_dbl, c_vp, c_vp, c_vp, c_vp]),
    "mg_amg_pmis": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_amg_promote": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_amg_interp_count": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_amg_interp_fill": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                   ctypes.POINTER(c_i64), c_vp]),
    "mg_sa_diagonal": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_sa_strength_count": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_dbl, c_vp, c_vp]),
    "mg_sa_strength_fill": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_dbl, c_vp, c_vp, c_vp, c_vp]),
    "mg_sa_mis2": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_sa_aggregate": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, ctypes.POINTER(c_i64), c_vp]),
    "mg_sa_aggregate_norm": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp]),
    "mg_sa_tentative_fill": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_sa_smooth_scale": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_dbl, c_vp, c_vp]),
    "mg_host_greedy_color": (c_int, [c_i64, c_vp, c_vp, c_vp]),
    "mg_host_greedy_color_block": (c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_int]),
    "mg_host_lex_levels": (c_i64, [c_i64, c_vp, c_vp, c_vp]),
    "mg_color_workspace_size": (c_i64, [c_i64]),
    "mg_csr_coloring_flags": (c_int, [c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_color_first_fit": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_vp]),
    "mg_vcycle": (c_int, [ctypes.POINTER(mg_level), c_int, ctypes.POINTER(mg_cycle_params), c_vp]),
    "mg_vcycle_dist": (c_int, [ctypes.POINTER(mg_comm), ctypes.POINTER(mg_level), c_int,
                               ctypes.POINTER(mg_cycle_params), ctypes.POINTER(mg_dist_norm), c_vp]),
    "mg_last_launch_count": (c_i64, []),
    "mg_graph_begin": (c_int, [c_vp]),
    "mg_graph_end": (c_int, [c_vp, ctypes.POINTER(c_vp)]),
    "mg_graph_launch": (c_int, [c_vp, c_vp]),
    "mg_graph_destroy": (c_int, [c_vp]),
}

# serial host emulations of device code, exported by libmgb200_testing.so only (csrc/Makefile): the CPU test-suite checks
# the NN patch logic, the per-pair coupling integration and the colouring rounds through them; nothing in the product
# calls load_testing()
_TESTING_SIGNATURES = {
    "mg_host_coupling_pairs_p1_2d": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_host_nn_coarsen": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_host_nn_extract_patches": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "mg_host_nn_contributions": (c_int, [c_i64, c_vp, c_vp, c_vp, ctypes.c_int32, c_vp, c_vp, c_vp, c_vp]),
    "mg_host_color_rounds": (c_int, [c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
}

_lib = None
_testing_lib = None


def build(force=False, verbose=False):
    """Compile csrc/*.cu for sm_100a into learnmultigrid_b200/libmgb200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC, "-j8"]
    if force:
        cmd.append("-B")
    out = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if out.returncode != 0:
        raise MgError("building libmgb200.so failed:\n" + out.stdout)
    if verbose:
        print(out.stdout)
    return LIB_PATH


def load():
    """Load libmgb200.so and install the prototypes.  Fails loudly if it is missing: no fallback exists."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MgError("libmgb200.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'`"
                      % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)      # AttributeError here = header / library mismatch
        fn.restype = res
        fn.argtypes = args
    if os.environ.get("MGB_PDL", "1") == "0":
        lib.mg_set_pdl(0)
    if os.environ.get("MGB_FUSED_EXCHANGE", "1") == "0":
        lib.mg_set_fused_exchange(0)
    if os.environ.get("MGB_IMPLIED_COLUMNS", "1") == "0":
        lib.mg_set_implied_columns(0)
    if os.environ.get("MGB_IMPLIED_TRANSFERS", "1") == "0":
        lib.mg_set_implied_transfers(0)
    if "MGB_IMPLIED_MIN_ROWS" in os.environ:
        lib.mg_set_implied_min_rows(int(os.environ["MGB_IMPLIED_MIN_ROWS"]))
    if os.environ.get("MGB_VALUE_DICT", "1") == "0":
        lib.mg_set_value_dict(0)
    if os.environ.get("MGB_IMPLIED_VALUES", "1") == "0":
        lib.mg_set_implied_values(0)
    if "MGB_SHORT_ROWS" in os.environ:
        lib.mg_set_short_rows_per_thread(int(os.environ["MGB_SHORT_ROWS"]))
    if os.environ.get("MGB_CYCLE_FUSION", "1") == "0":
        lib.mg_set_cycle_fusion(0)
    if "MGB_WIDE_MIN_LEN" in os.environ:
        lib.mg_set_wide_min_len(int(os.environ["MGB_WIDE_MIN_LEN"]))
    if "MGB_WIDE_MAX_ROWS" in os.environ:
        lib.mg_set_wide_max_rows(int(os.environ["MGB_WIDE_MAX_ROWS"]))
    _lib = lib
    return lib


def load_testing():
    """libmgb200_testing.so: the product library plus the `mg_host_*` emulations (test infrastructure)."""
    global _testing_lib
    if _testing_lib is not None:
        return _testing_lib
    path = os.path.join(os.path.dirname(LIB_PATH), "libmgb200_testing.so")
    if not os.path.exists(path):
        raise MgError("libmgb200_testing.so is not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'`" % path)
    lib = ctypes.CDLL(path)
    for table in (_SIGNATURES, _TESTING_SIGNATURES):
        for name, (res, args) in table.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
    _testing_lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().mg_last_error().decode("utf-8", "replace")
        raise MgError("libmgb200 %s failed (status %d): %s" % (what, rc, msg))


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise MgError("learnmultigrid_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def ptr(t):
    """device pointer of a torch tensor (or None -> NULL)"""
    return None if t is None else t.data_ptr()


def stream_handle(torch):
    return torch.cuda.current_stream().cuda_stream
