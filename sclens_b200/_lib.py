"""ctypes binding of libsclens_b200.so (include/sclens_b200.h).  There is no CPU fallback:
a missing library or a missing sm_100 GPU raises."""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsclens_b200.so")

SCL_GRAM_FP16, SCL_GRAM_FP16X3 = 0, 1
SCL_ERR_NOSIGNAL = -6


class SclError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libsclens_b200 error {code}: {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [("device", C.c_int32), ("gram_mode", C.c_int32), ("cta_group", C.c_int32), ("verbose", C.c_int32),
                ("seed", C.c_uint64), ("subspace_extra", C.c_int32), ("subspace_degree", C.c_int32),
                ("exact_perturb", C.c_int32), ("gram_chunk_kb", C.c_int32), ("gram_tc_diag", C.c_int32),
                ("no_refine", C.c_int32), ("centering", C.c_int32), ("reserved", C.c_int32 * 3)]


class SignalInfo(C.Structure):
    _fields_ = [("N", C.c_int32), ("M", C.c_int32), ("nm", C.c_int32), ("n_signal", C.c_int32), ("n_Lmp", C.c_int32),
                ("mp_iters", C.c_int32), ("pass_", C.c_int32), ("gram_mode_used", C.c_int32),
                ("lambda_c", C.c_double), ("b_plus", C.c_double), ("b_minus", C.c_double), ("ks_static", C.c_double),
                ("t_ingest_ms", C.c_double), ("t_normalize_ms", C.c_double), ("t_null_ms", C.c_double),
                ("t_gram_ms", C.c_double), ("t_syevd_ms", C.c_double), ("t_fit_ms", C.c_double),
                ("t_backproject_ms", C.c_double)]


class RobustInfo(C.Structure):
    _fields_ = [("n_search", C.c_int32), ("n_perturb", C.c_int32), ("min_pc", C.c_int32), ("n_robust", C.c_int32),
                ("n_add", C.c_int64), ("p_sel", C.c_double), ("p_th", C.c_double), ("t_baseline_ms", C.c_double),
                ("t_search_ms", C.c_double), ("t_search_syevd_ms", C.c_double), ("t_perturb_ms", C.c_double),
                ("t_score_ms", C.c_double), ("t_outputs_ms", C.c_double), ("n_subspace_fallbacks", C.c_int32),
                ("reserved", C.c_int32)]


class QcParams(C.Structure):
    _fields_ = [("min_tp_c", C.c_double), ("min_tp_g", C.c_double), ("max_tp_c", C.c_double), ("max_tp_g", C.c_double),
                ("min_genes_per_cell", C.c_int32), ("max_genes_per_cell", C.c_int32), ("min_cells_per_gene", C.c_int32),
                ("reserved", C.c_int32), ("mito_percent", C.c_double), ("ribo_percent", C.c_double)]


class Profile(C.Structure):
    _fields_ = [("gram_gemm_ms", C.c_double), ("other_gemm_ms", C.c_double), ("densify_ms", C.c_double),
                ("stats_ms", C.c_double), ("sparse_ms", C.c_double), ("syevd_ms", C.c_double),
                ("gram_gemm_launches", C.c_int64), ("other_gemm_launches", C.c_int64), ("densify_launches", C.c_int64),
                ("sparse_calls", C.c_int64), ("syevd_calls", C.c_int64), ("gram_alg_flops", C.c_double),
                ("other_gemm_flops", C.c_double), ("densify_alg_bytes", C.c_double), ("sparse_alg_bytes", C.c_double),
                ("kernel_launches", C.c_int64), ("refine_ms", C.c_double), ("small_ms", C.c_double),
                ("stats_alg_bytes", C.c_double), ("stats_calls", C.c_int64), ("comm_ms", C.c_double),
                ("comm_bytes", C.c_double)]


class UmapParams(C.Structure):
    _fields_ = [("n_neighbors", C.c_int32), ("n_components", C.c_int32), ("n_epochs", C.c_int32), ("metric", C.c_int32),
                ("init", C.c_int32), ("neg_sample_rate", C.c_int32), ("spectral_maxiter", C.c_int32),
                ("reserved0", C.c_int32), ("min_dist", C.c_double), ("spread", C.c_double), ("learning_rate", C.c_double),
                ("repulsion_strength", C.c_double), ("local_connectivity", C.c_double), ("seed", C.c_uint64),
                ("reserved", C.c_int32 * 4)]


class UmapInfo(C.Structure):
    _fields_ = [("a", C.c_double), ("b", C.c_double), ("graph_nnz", C.c_int64), ("spectral_iters", C.c_int32),
                ("init_fallback", C.c_int32), ("t_knn_ms", C.c_double), ("t_graph_ms", C.c_double),
                ("t_init_ms", C.c_double), ("t_layout_ms", C.c_double), ("reserved", C.c_int32 * 4)]


_u32p = C.POINTER(C.c_uint32)
_f32p = C.POINTER(C.c_float)
_f64p = C.POINTER(C.c_double)
_u16p = C.POINTER(C.c_uint16)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_hp = C.c_void_p

# name -> argtypes; every symbol include/sclens_b200.h declares
SIGNATURES = {
    "scl_version": [],
    "scl_create": [C.POINTER(_hp), C.POINTER(Config)],
    "scl_destroy": [_hp],
    "scl_last_error": [_hp],
    "scl_get_profile": [_hp, C.POINTER(Profile)],
    "scl_reset_profile": [_hp],
    "scl_timer_start": [_hp],
    "scl_timer_stop": [_hp, _f64p],
    "scl_nccl_unique_id": [C.POINTER(C.c_uint8)],
    "scl_comm_init": [_hp, C.POINTER(C.c_uint8), C.c_int32, C.c_int32],
    "scl_plan_replicates": [C.c_int32, C.c_int32, C.c_int32, _i32p, _i32p],
    "scl_plan_gram_shard": [C.c_int64, C.c_int32, C.c_int32, _i64p, _i64p],
    "scl_plan_pass_task": [C.c_int32, C.c_int32, C.c_int32, _i32p, _i32p],
    "scl_plan_search_wave": [C.c_int32, C.c_int32, C.c_int32, _i32p],
    "scl_set_counts_csc": [_hp, C.c_int32, C.c_int32, C.c_int64, _u32p, _u32p, _f32p, C.c_int32],
    "scl_set_zero_candidates": [_hp, C.c_int64, _u32p, _u32p, C.c_int32],
    "scl_set_null_draws": [_hp, C.c_int64, _u32p, _u32p, C.c_int32],
    "scl_set_noise_baseline": [_hp, C.c_double],
    "scl_push_search_sample": [_hp, C.c_int64, _u32p, C.c_int32],
    "scl_push_perturb_sample": [_hp, C.c_int64, _u32p, C.c_int32],
    "scl_clear_draws": [_hp],
    "scl_op_preprocess": [_hp, C.c_int32, C.c_int32, C.c_int64, _u32p, _u32p, _f32p, C.c_int32, C.POINTER(C.c_uint8),
                          C.POINTER(QcParams), _i32p, _i32p, _i64p, _i32p, _i32p],
    "scl_get_counts_csc": [_hp, _u32p, _u32p, _f32p],
    "scl_run_signal": [_hp, C.POINTER(SignalInfo)],
    "scl_run_robustness": [_hp, C.c_double, C.c_double, C.c_int32, C.POINTER(RobustInfo)],
    "scl_run_pass": [_hp, C.c_double, C.c_double, C.c_int32, C.POINTER(SignalInfo), C.POINTER(RobustInfo)],
    "scl_get_L": [_hp, _f32p],
    "scl_get_Lmp": [_hp, _f32p],
    "scl_get_signal_ev": [_hp, _f32p],
    "scl_get_signal_evec": [_hp, _f32p],
    "scl_get_gene_basis": [_hp, _f32p],
    "scl_get_rec_vals": [_hp, _f64p, _f64p, _f64p, _f64p, _f64p],
    "scl_get_scores": [_hp, _f32p, _f64p, _f64p],
    "scl_get_sig_id": [_hp, _i32p],
    "scl_get_null_csc": [_hp, _i64p, _u32p, _u32p, _f32p],
    "scl_get_search_trace": [_hp, _f64p, _f64p],
    "scl_get_perturbed_evec": [_hp, C.c_int32, _f32p, _f32p],
    "scl_op_normalize": [_hp, C.c_int32, C.c_int32, C.c_int64, _u32p, _u32p, _f32p, C.c_int32, C.c_int64, _u16p, _u16p,
                         _f64p, _f64p, _f64p, _f64p, _f64p],
    "scl_op_gram": [_hp, C.c_int32, C.c_int64, C.c_int64, _u16p, _u16p, C.c_float, _f32p],
    "scl_op_gemm_tn": [_hp, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_int64, _u16p, _u16p, _u16p, _u16p,
                       C.c_float, C.c_int32, _f32p],
    "scl_op_syevd": [_hp, C.c_int32, _f32p, _f32p, _f32p, _f64p],
    "scl_op_syevd_tri": [_hp, C.c_int32, _f32p, C.c_int32, C.c_int32, _f32p, _f32p, _f64p],
    "scl_op_mp_fit": [_f32p, C.c_int32, _f32p, C.c_int32, _f64p],
    "scl_op_permute_null": [_hp, C.c_int32, C.c_int32, C.c_int64, _u32p, _u32p, _f32p, _u32p, _u32p, _i64p, _u32p,
                            _u32p, _f32p],
    "scl_op_perturb_merge": [_hp, C.c_int32, C.c_int32, C.c_int64, _u32p, _u32p, _f32p, C.c_int64, _u32p, _u32p,
                             C.c_int32, _u32p, _u32p, _f32p],
    "scl_op_corr_colabsmax": [_hp, C.c_int32, C.c_int32, C.c_int32, _f32p, _f32p, _f32p],
    "scl_op_topk_subspace": [_hp, C.c_int32, _f32p, C.c_int32, _f32p, _f32p, _i32p],
    "scl_op_scores": [_hp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _f32p, _f32p, C.c_double, _f32p, _f64p, _f64p,
                      _i32p, _i32p],
    "scl_op_draw_zero_candidates": [_hp, C.c_uint64, _i64p, _u32p, _u32p],
    "scl_op_zero_candidate_draws": [C.c_uint64, C.c_int64, C.c_int32, C.c_int32, _u32p, _u32p],
    "scl_op_noise_baseline": [_hp, C.c_int32, C.c_int32, C.c_uint64, _f64p],
    "scl_op_draw_subset": [_hp, C.c_int64, C.c_uint64, _u32p, _u32p],
    "scl_op_scores_from_pairs": [_f32p, C.c_int32, C.c_int32, C.c_double, _f64p, _f64p, _i32p, _i32p],
    "scl_op_denoise": [_hp, C.c_int32, C.c_int32, C.c_int32, _f32p, _f32p, _f64p, _f64p, _f64p, _f64p, _f64p, C.c_int32,
                       C.c_void_p],
    "scl_op_knn": [_hp, C.c_int32, C.c_int32, _f32p, C.c_int32, C.c_int32, _i32p, _f32p],
    "scl_op_umap": [_hp, C.c_int32, C.c_int32, _f32p, C.POINTER(UmapParams), _f32p, _f32p, C.POINTER(UmapInfo)],
    "scl_get_umap_graph": [_hp, _i64p, _u32p, _u32p, _f32p],
    "scl_get_umap_knn": [_hp, _i32p, _f32p],
    "scl_umap_fit_ab": [C.c_double, C.c_double, _f64p, _f64p],
    "scl_bench_gram": [_hp, C.c_int32, C.c_int64, C.c_int32, C.c_int32, C.c_int32, _f64p, _f64p],
    "scl_bench_syevd": [_hp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _f64p],
    "scl_bench_syevd_concurrent": [_hp, C.c_int32, C.c_int32, C.c_int32, _f64p],
    "scl_debug_set_eig_api": [C.c_int32],
    "scl_debug_last_solve": [_hp, _f64p],
    "scl_debug_eig_stage_totals": [_hp, _f64p],
    "scl_debug_set_two_stage": [C.c_int32, C.c_int32, C.c_int32],
    "scl_debug_two_stage": [_hp, C.c_int32, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, C.POINTER(C.c_int32)],
    "scl_debug_set_tuning": [C.c_int32, C.c_int32, C.c_int32],
    "scl_bench_normalize": [_hp, C.c_int32, C.c_int32, C.c_int32, _f64p, _f64p, _f64p],
}

_lib = None


def load() -> C.CDLL:
    """Load the shared library (raises if it has not been built: no fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(f"{LIB_PATH} not found - run `python -m sclens_b200.build` (there is no CPU fallback)")
        lib = C.CDLL(LIB_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.argtypes = args
            fn.restype = C.c_char_p if name == "scl_last_error" else C.c_int32
        _lib = lib
    return _lib


def ptr(a, ctype):
    if a is None:
        return None
    return a.ctypes.data_as(C.POINTER(ctype))


def as_u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def as_f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)
