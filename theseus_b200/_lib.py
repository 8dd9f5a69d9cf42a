"""ctypes binding of libthb200.so (the C ABI declared in include/thb200.h).

There is NO fallback: if the library is missing or a call fails, a RuntimeError is raised.  The
library is plain C ABI (device pointers, sizes, cudaStream_t) -- torch is only used by the caller
for device memory and streams.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.environ.get("THB200_LIB") or os.path.join(_HERE, "lib", "libthb200.so")  # override: kernel-variant experiments
_lib = None

c_i32, c_i64, c_f64, c_f32, c_vp = C.c_int32, C.c_int64, C.c_double, C.c_float, C.c_void_p


class CostGroup(C.Structure):
    _fields_ = [("kind", c_i32), ("weight_kind", c_i32), ("K", c_i32), ("dim", c_i32),
                ("x0", c_vp), ("x1", c_vp), ("aux", c_vp), ("w", c_vp), ("bstride", c_vp),
                ("a_off", c_vp), ("a_stride", c_vp), ("bp", c_vp), ("row0", c_vp),
                ("aux2", c_vp), ("aux3", c_vp), ("aux4", c_vp), ("bstride2", c_vp),
                ("robust_kind", c_i32), ("reserved0", c_i32), ("log_radius", c_vp), ("bstride_lr", c_vp),
                ("x2", c_vp), ("x3", c_vp), ("bstride3", c_vp), ("sdf_rows", c_i32), ("sdf_cols", c_i32)]


class VarTable(C.Structure):
    _fields_ = [("N", c_i32), ("x", c_vp), ("out", c_vp), ("kind", c_vp), ("col", c_vp), ("dof", c_vp)]


class GramPlan(C.Structure):
    _fields_ = [("num_entries", c_i64), ("ent_blk", c_vp), ("ent_p", c_vp), ("ent_q", c_vp),
                ("blk_out", c_vp), ("blk_ld", c_vp), ("blk_mirror", c_vp), ("blk_cptr", c_vp),
                ("c_off", c_vp), ("c_stride", c_vp), ("c_rows", c_vp), ("c_bpa", c_vp), ("c_bpb", c_vp),
                ("n", c_i64), ("col_cptr", c_vp), ("cc_off", c_vp), ("cc_stride", c_vp), ("cc_rows", c_vp),
                ("cc_row0", c_vp), ("num_blocks", c_i64), ("blk_rows", c_vp), ("blk_cols", c_vp),
                ("num_segments", c_i64), ("segments", c_vp), ("blk_order", c_vp)]


def make_gram_plan(arrs, dev):
    """thb_gram_plan from structure.build_gram_plan's arrays (`arrs`) and their device copies (`dev`)."""
    return GramPlan(
        num_entries=int(arrs["ent_blk"].shape[0]), ent_blk=dev["ent_blk"].data_ptr(), ent_p=dev["ent_p"].data_ptr(),
        ent_q=dev["ent_q"].data_ptr(), blk_out=dev["blk_out"].data_ptr(), blk_ld=dev["blk_ld"].data_ptr(),
        blk_mirror=dev["blk_mirror"].data_ptr(), blk_cptr=dev["blk_cptr"].data_ptr(), c_off=dev["c_off"].data_ptr(),
        c_stride=dev["c_stride"].data_ptr(), c_rows=dev["c_rows"].data_ptr(), c_bpa=dev["c_bpa"].data_ptr(),
        c_bpb=dev["c_bpb"].data_ptr(), n=int(arrs["n"]), col_cptr=dev["col_cptr"].data_ptr(),
        cc_off=dev["cc_off"].data_ptr(), cc_stride=dev["cc_stride"].data_ptr(), cc_rows=dev["cc_rows"].data_ptr(),
        cc_row0=dev["cc_row0"].data_ptr(), num_blocks=int(arrs["blk_out"].shape[0]), blk_rows=dev["blk_rows"].data_ptr(),
        blk_cols=dev["blk_cols"].data_ptr(), num_segments=int(arrs["segments"].shape[0]), segments=arrs["segments"].ctypes.data,
        blk_order=dev["blk_order"].data_ptr())


class SparsePlanStruct(C.Structure):
    _fields_ = [("N", c_i32), ("num_levels", c_i32), ("max_dim", c_i32), ("reserved", c_i32),
                ("n", c_i64), ("data_size", c_i64), ("winv_size", c_i64)] + [(k, c_vp) for k in (
                    "dims", "col_start", "pstart", "winv_off", "diag_off", "up_a", "up_b", "up_k",
                    "u_ptr", "u_tgt", "u_r", "u_c", "u_ld", "u_p0", "u_p1",
                    "f_ptr", "f_off", "f_dim", "f_w", "f_col",
                    "t_ptr", "t_off", "t_r", "t_dim", "t_w",
                    "s_ptr", "s_col", "fr_ptr", "fr_off", "fr_k", "bc_ptr", "bc_off", "bc_i")]


class SparseLanePlanStruct(C.Structure):
    _fields_ = [("N", c_i64), ("n", c_i64), ("data_size", c_i64), ("diag_size", c_i64), ("num_launches", c_i64)] + [(k, c_vp) for k in (
        "launches", "dims", "col_start", "pstart", "dl_off", "diag_off", "up_a", "up_b", "up_k", "u_tgt", "u_p0", "u_p1",
        "t_off", "t_diag", "t_dl", "t_pstart", "s_col", "fr_ptr", "fr_off", "fr_p", "fr_d", "bc_ptr", "bc_off", "bc_p", "bc_d")]


# name -> (restype, argtypes); every symbol declared in include/thb200.h
_PG, _PV, _PP = C.POINTER(CostGroup), C.POINTER(VarTable), C.POINTER(GramPlan)
_PS = C.POINTER(SparsePlanStruct)
_PL = C.POINTER(SparseLanePlanStruct)


class SparseLaneRootStruct(C.Structure):
    _fields_ = [("num_blocks", c_i64), ("num_cols", c_i64), ("nt", c_i64), ("root_start", c_i64), ("num_segments", c_i64)] + [(k, c_vp) for k in (
        "segments", "rb_off", "rb_row", "rb_col", "rb_di", "rb_dj", "rf_p0", "rf_p1", "root_cols", "root_dims")]


class SparseLaneTilesStruct(C.Structure):
    _fields_ = [("num_tiles", c_i64), ("num_steps", c_i64), ("tile_tgt", c_vp), ("step_ptr", c_vp), ("step_src", c_vp)]


class SparseLanePiecesStruct(C.Structure):
    _fields_ = [("num_pieces", c_i64), ("num_launches", c_i64)] + [(k, c_vp) for k in (
        "launches", "first", "width", "fr_ext_end", "bc_int_end", "order")]


class FrontPlanStruct(C.Structure):
    """thb_front_plan (include/thb200.h): multifrontal block-sparse Cholesky, arrays of theseus_b200/frontal.py."""
    _fields_ = [("S", c_i64), ("n", c_i64), ("data_size", c_i64), ("arena_size", c_i64), ("varena_size", c_i64)] + [(k, c_vp) for k in (
        "f_w", "f_b", "f_first", "f_class", "f_wpad", "f_np", "f_cb_ld", "f_depth", "f_panel_off", "f_cb_off", "f_fr_off", "f_u_off",
        "child_ptr", "child_list", "rel_ptr", "f_rel", "rows_ptr", "f_rows", "sched", "perm", "c_jw", "c_sp_ptr", "c_sp", "c_inv_ptr", "c_inv", "fd", "pc", "pmap")]


_PF = C.POINTER(FrontPlanStruct)
_PR = C.POINTER(SparseLaneRootStruct)
_PPIECES = C.POINTER(SparseLanePiecesStruct)
_PT = C.POINTER(SparseLaneTilesStruct)
SIGNATURES = {
    "thb_version": (c_i32, []),
    "thb_compiled_arch": (c_i32, []),
    "thb_launch_count": (c_i64, []),
    "thb_linearize_group_f64": (c_i32, [_PG, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "thb_linearize_group_f32": (c_i32, [_PG, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "thb_error_num_chunks": (c_i32, [c_i32]),
    "thb_error_group_f64": (c_i32, [_PG, c_i64, c_vp, c_vp]),
    "thb_error_group_f32": (c_i32, [_PG, c_i64, c_vp, c_vp]),
    "thb_error_reduce_f64": (c_i32, [c_vp, c_i32, c_i64, c_vp, c_vp]),
    "thb_error_reduce_f32": (c_i32, [c_vp, c_i32, c_i64, c_vp, c_vp]),
    "thb_retract_f64": (c_i32, [_PV, c_i64, c_vp, c_i64, c_f64, c_vp, c_vp]),
    "thb_retract_f32": (c_i32, [_PV, c_i64, c_vp, c_i64, c_f32, c_vp, c_vp]),
    "thb_commit_f64": (c_i32, [_PV, c_i64, c_vp, c_vp]),
    "thb_commit_f32": (c_i32, [_PV, c_i64, c_vp, c_vp]),
    "thb_gram_f64": (c_i32, [_PP, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "thb_gram_f32": (c_i32, [_PP, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_i64, c_vp, c_vp, c_vp]),
    "thb_fill_zero": (c_i32, [c_vp, c_i64, c_vp]),
    "thb_potrf_workspace_bytes": (c_i64, [c_i64, c_i64]),
    "thb_potrf_f64": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp]),
    "thb_potrs_f64": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp]),
    "thb_potrf_potrs_f64": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_i64, c_vp, c_i64, c_vp]),
    "thb_sparse_damp_f64": (c_i32, [_PS, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_factor_f64": (c_i32, [_PS, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_solve_f64": (c_i32, [_PS, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_symbolic_create": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_i32, c_vp]),
    "thb_symbolic_destroy": (None, [c_vp]),
    "thb_symbolic_array_count": (c_i64, [c_vp, C.c_char_p]),
    "thb_symbolic_array_elem_bytes": (c_i32, [c_vp, C.c_char_p]),
    "thb_symbolic_array_copy": (c_i32, [c_vp, C.c_char_p, c_vp, c_i64]),
    "thb_symbolic_stat": (C.c_double, [c_vp, C.c_char_p]),
    "thb_sparse_lane_padded_batch": (c_i64, [c_i64]),
    "thb_sparse_lane_gram_f64": (c_i32, [_PP, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "thb_sparse_lane_damp_f64": (c_i32, [_PL, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_factor_f64": (c_i32, [_PL, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_factor_tiled_f64": (c_i32, [_PL, _PT, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_solve_f64": (c_i32, [_PL, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_forward_f64": (c_i32, [_PL, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_backward_f64": (c_i32, [_PL, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_piece_forward_f64": (c_i32, [_PL, _PPIECES, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_piece_backward_f64": (c_i32, [_PL, _PPIECES, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_root_gather_f64": (c_i32, [_PR, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_root_rhs_f64": (c_i32, [_PL, _PR, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_sparse_lane_root_scatter_f64": (c_i32, [_PL, _PR, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_gram_dense_f64": (c_i32, [c_vp, c_vp, c_i64, c_i64, c_i64, c_vp]),
    "thb_front_small_smem_bytes": (c_i64, [c_i32, c_i32, c_i32]),
    "thb_front_factor_f64": (c_i32, [_PF, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "thb_front_solve_f64": (c_i32, [_PF, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "thb_potrf_partial_workspace_bytes": (c_i64, [c_i64, c_i64]),
    "thb_potrf_partial_inplace_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_i32, c_i32, c_i32, c_vp, c_i64, c_vp, c_i64, c_vp]),
    "thb_solve_backward_f64": (c_i32, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_vp]),
    "thb_lm_control_f64": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_i64, c_f64, c_vp, c_vp, c_vp, c_i32, c_f64, c_f64, c_f64,
                                   c_vp, c_vp, c_vp, c_vp]),
    "thb_lm_control_f32": (c_i32, [c_vp, c_vp, c_vp, c_i64, c_i64, c_f32, c_vp, c_vp, c_vp, c_i32, c_f32, c_f32, c_f32,
                                   c_vp, c_vp, c_vp, c_vp]),
    "thb_mat_vec_f64": (c_i32, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "thb_tmat_vec_f64": (c_i32, [c_i64, c_i64, c_i64, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp]),
}
for _sfx, _ in (("f64", c_f64), ("f32", c_f32)):
    SIGNATURES[f"thb_se3_exp_{_sfx}"] = (c_i32, [c_vp, c_vp, c_i64, c_vp])
    SIGNATURES[f"thb_se3_log_{_sfx}"] = (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp])
    SIGNATURES[f"thb_se3_adjoint_{_sfx}"] = (c_i32, [c_vp, c_vp, c_i64, c_vp])
    SIGNATURES[f"thb_se3_inverse_{_sfx}"] = (c_i32, [c_vp, c_vp, c_i64, c_vp])
    SIGNATURES[f"thb_se3_compose_{_sfx}"] = (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp])
    SIGNATURES[f"thb_se3_jexp_{_sfx}"] = (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp])
    SIGNATURES[f"thb_so3_jexp_{_sfx}"] = (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp])
    for _g in ("so3", "se2"):
        SIGNATURES[f"thb_{_g}_exp_{_sfx}"] = (c_i32, [c_vp, c_vp, c_i64, c_vp])
        SIGNATURES[f"thb_{_g}_log_{_sfx}"] = (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp])
        SIGNATURES[f"thb_{_g}_adjoint_{_sfx}"] = (c_i32, [c_vp, c_vp, c_i64, c_vp])
        SIGNATURES[f"thb_{_g}_inverse_{_sfx}"] = (c_i32, [c_vp, c_vp, c_i64, c_vp])
        SIGNATURES[f"thb_{_g}_compose_{_sfx}"] = (c_i32, [c_vp, c_vp, c_vp, c_i64, c_vp])


def lib_path():
    return _LIB_PATH


def load():
    """Load libthb200.so (after torch, so the CUDA runtime already mapped by torch is shared)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(_LIB_PATH):
        raise RuntimeError(
            f"libthb200.so not found at {_LIB_PATH}: build it with `python -m theseus_b200.build` "
            "(theseus_b200 has no CPU or PyTorch fallback for its compute path)")
    import torch  # noqa: F401  (maps libcudart first)
    lib = C.CDLL(_LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if a declared symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


# Kernel launches replayed from captured CUDA graphs (optimizer cuda_graph=True) do not pass through the library's entry points;
# the optimizer adds (kernels in the captured body) per replay here so that launch accounting stays truthful.
replayed_launches = 0


def total_launches() -> int:
    """Kernels of libthb200 launched in this process so far: direct launches (thb_launch_count) + graph replays."""
    return int(load().thb_launch_count()) + replayed_launches


def check(rc, what):
    if rc != 0:
        kind = "invalid argument" if rc < 0 else "CUDA error"
        raise RuntimeError(f"libthb200: {what} failed with {kind} code {rc}")


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    return None if t is None else C.c_void_p(t.data_ptr())
