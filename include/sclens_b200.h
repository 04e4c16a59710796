/*
 * sclens_b200.h - C ABI of libsclens_b200.so, the B200-native drop-in for the
 * signal-detection hot path of Mathbiomed/scLENS:  scLENS.sclens(pre_df; device_="gpu")
 * (reference: src/scLENS.jl:649-832 and the helpers it calls, :239-608).
 *
 * The reference has no FFI: its only backend seam is the `device_` string keyword that
 * branches into CUDA.jl library calls at src/scLENS.jl:335-343 (_wishart_matrix),
 * :365-369 (corr_mat), :377 (_get_eigen), :505 / :558 / :561 (back-projection) and
 * :814-816 (gene_basis).  A per-function shim would inherit the reference's seven PCIe
 * crossings per get_eigvec call, so the boundary sits one level up: a handle owns all
 * device state of one sclens() call; counts go in once (CSC), results come out once.
 * Function-level entry points (scl_op_*) expose the individual stages for unit parity.
 *
 * Conventions: every function returns 0 on success, <0 on error (no exceptions cross the
 * boundary, no CPU fallback exists); scl_last_error() gives the message.  All pointers are
 * HOST pointers owned by the caller and are never retained after the call returns.
 * Matrices are column-major (Julia layout) unless stated.  Indices passed in are
 * `index_base`-based (1 from Julia, 0 from C/Python); indices returned are 0-based.
 * A handle is not thread-safe; distinct handles are independent.
 */
#ifndef SCLENS_B200_H
#define SCLENS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define SCL_API __attribute__((visibility("default")))
#else
#define SCL_API
#endif

typedef struct scl_handle scl_handle;

enum {
  SCL_OK = 0,
  SCL_ERR_INVALID = -1,   /* bad argument / call order */
  SCL_ERR_CUDA = -2,      /* CUDA runtime / driver error */
  SCL_ERR_CUSOLVER = -3,  /* cuSOLVER error or non-convergence (reference NaN fallback :379-381 is an error here) */
  SCL_ERR_NOGPU = -4,     /* no sm_100 device: there is no CPU fallback */
  SCL_ERR_NCCL = -5,
  SCL_ERR_NOSIGNAL = -6,  /* scl_run_robustness called with zero signals (:780-784) */
  SCL_ERR_GRAPH = -7      /* a clustering input graph is not a symmetric CSR with sorted columns and finite positive weights */
};

/* Gram operand precision. FP16: one tcgen05 kind::f16 pass. FP16X3: hi/lo split, three
 * passes into the same TMEM accumulator (~fp32 accuracy; reference is FP32 SGEMM :337). */
enum { SCL_GRAM_FP16 = 0, SCL_GRAM_FP16X3 = 1 };

typedef struct {
  int32_t device;        /* CUDA device ordinal */
  int32_t gram_mode;     /* SCL_GRAM_* */
  int32_t cta_group;     /* 0 = library default, 1 or 2 = force tcgen05 cta_group */
  int32_t verbose;       /* 1: print the reference's progress lines (:539, :713, :762, :807) */
  uint64_t seed;         /* seed of the device-side draws when none are injected */
  int32_t subspace_extra;/* oversampling columns of the block subspace iteration (0 = default) */
  int32_t subspace_degree;/* Chebyshev degree per sweep (0 = default) */
  int32_t exact_perturb; /* 1: full syevd per replicate exactly as :775 (parity studies) */
  int32_t gram_chunk_kb; /* 64-element k-blocks the tensor core accumulates before the chunk is promoted into the
                            round-to-nearest FP32 sum (0 = library default; numerics studies) */
  int32_t gram_tc_diag;  /* numerics studies. 0: exact Float64 Gram diagonal + calibration of the tensor core's
                            accumulation bias (default); 1: the raw tensor-core result; 2: exact diagonal only */
  int32_t no_refine;     /* 1: return the FP32 eigensolver's eigenvalues as they are (no Float64 Rayleigh-quotient refinement) */
  int32_t centering;     /* 0: centering="mean" (default, :677-696); 1: centering="median" (:294-299, :653-654): per-gene median of
                            log1p(x / r_i) over all cells as the centre, rows rescaled to the mean row norm, no re-centring */
  int32_t reserved[3];
} scl_config;

typedef struct {
  int32_t N, M, nm;          /* cells, genes, min(N,M) */
  int32_t n_signal;          /* sum(L .> lambda_c)                     (:539/:578) */
  int32_t n_Lmp;             /* length(L_mp)                           (:458) */
  int32_t mp_iters;          /* fixed-point iterations of _mp_calculation (:436-455) */
  int32_t pass;              /* mp_check :pass                         (:486) */
  int32_t gram_mode_used;    /* SCL_GRAM_* actually used (guard band may escalate) */
  double lambda_c, b_plus, b_minus, ks_static;
  double t_ingest_ms, t_normalize_ms, t_null_ms, t_gram_ms, t_syevd_ms, t_fit_ms, t_backproject_ms;
} scl_signal_info;

typedef struct {
  int32_t n_search;          /* sparsity-search iterations executed    (:725-761) */
  int32_t n_perturb;         /* replicates run                         (:771-778) */
  int32_t min_pc;            /* ceil(1.5 * n_signal)                   (:770) */
  int32_t n_robust;          /* length(sig_id)                         (:806) */
  int64_t n_add;             /* round((1-p_)*M*N) at the selected p_   (:772) */
  double p_sel;              /* "Selected perturb sparisty"            (:762) */
  double p_th;               /* noise baseline                         (:712) */
  double t_baseline_ms, t_search_ms, t_search_syevd_ms, t_perturb_ms, t_score_ms, t_outputs_ms;
  int32_t n_subspace_fallbacks; /* replicates whose block subspace iteration gave up and took the exact solve of :775 */
  int32_t reserved;
} scl_robust_info;

/* Kernel-class timings (CUDA events on the library's stream) and algorithmic work counters,
 * accumulated since scl_reset_profile; what bench.py's roofline figures are computed from. */
typedef struct {
  double gram_gemm_ms, other_gemm_ms, densify_ms, stats_ms, sparse_ms, syevd_ms;
  int64_t gram_gemm_launches, other_gemm_launches, densify_launches, sparse_calls, syevd_calls;
  double gram_alg_flops;      /* sum of n(n+1)K over Gram launches (SYRK-minimal, SURVEY.md 8d) */
  double other_gemm_flops;    /* sum of 2mnk */
  double densify_alg_bytes;   /* sum of 8 nnz + 4(M+1) + N*M*s_out */
  double sparse_alg_bytes;    /* 20 nnz per null permutation, 8 nnz + 12 n_add per merge */
  int64_t kernel_launches;    /* kernels of this library launched by the process since load */
  double refine_ms;           /* Float64 Rayleigh-quotient refinement of the data spectrum */
  double small_ms;            /* calibration, reductions, collectives and other small kernels */
  double stats_alg_bytes;     /* statistics line passes: 40 nnz per normalisation (4 nnz row sums, 3 x 8 nnz, 12 nnz patch pass) */
  int64_t stats_calls;        /* normalisations (one set of statistics passes each) */
  double comm_ms;             /* NCCL collectives on the library stream (Gram all-reduce, broadcasts of results) */
  double comm_bytes;          /* payload bytes of those collectives as this rank sees them */
} scl_profile;

/* ---- lifecycle --------------------------------------------------------------------- */
SCL_API int32_t scl_version(void);
SCL_API int32_t scl_create(scl_handle** out, const scl_config* cfg);
SCL_API int32_t scl_destroy(scl_handle* h);
SCL_API const char* scl_last_error(scl_handle* h);   /* h may be NULL: last scl_create error */
SCL_API int32_t scl_get_profile(scl_handle* h, scl_profile* out);
SCL_API int32_t scl_reset_profile(scl_handle* h);
/* CUDA-event stopwatch on the handle's stream (the stream every kernel of the path is launched on). */
SCL_API int32_t scl_timer_start(scl_handle* h);
SCL_API int32_t scl_timer_stop(scl_handle* h, double* ms);

/* ---- multi-GPU plumbing (one process per GPU; SURVEY.md 8e) ------------------------- */
/* 128-byte NCCL unique id, created on rank 0 and distributed by the host language. */
SCL_API int32_t scl_nccl_unique_id(uint8_t out_id[128]);
SCL_API int32_t scl_comm_init(scl_handle* h, const uint8_t id[128], int32_t rank, int32_t world);
/* Pure host logic (testable without a GPU): which replicates / search steps a rank owns. */
SCL_API int32_t scl_plan_replicates(int32_t n_perturb, int32_t world, int32_t rank, int32_t* out_ids, int32_t* out_n);
SCL_API int32_t scl_plan_search_wave(int32_t wave, int32_t world, int32_t rank, int32_t* out_step);
/* Task list of scl_run_pass: wave `wave` gives rank `rank` task t = wave * world + rank; t = 0 data matrix, 1 null matrix,
 * 2 reference basis of the binarised matrix, t >= 3 the sparsity-search steps in order (out_search_step, else -1) - except
 * that with world >= 3 the slot t = world (rank 0, wave 1) is the Float64 refinement of the data spectrum and the steps
 * after it move down by one. */
SCL_API int32_t scl_plan_pass_task(int32_t wave, int32_t world, int32_t rank, int32_t* out_task, int32_t* out_search_step);
/* Block [k0, k1) of the Gram contraction axis (cells when N > M; padded length ld = K rounded up to 8) a rank
 * densifies and contracts before the partial Gram matrices are summed with ncclAllReduce. */
SCL_API int32_t scl_plan_gram_shard(int64_t K, int32_t world, int32_t rank, int64_t* out_k0, int64_t* out_k1);

/* ---- inputs ------------------------------------------------------------------------ */
/* df2sparr output (:90-120): SparseMatrixCSC{Float32,UInt32}, N cells x M genes, canonical
 * order, strictly positive values. */
SCL_API int32_t scl_set_counts_csc(scl_handle* h, int32_t N, int32_t M, int64_t nnz,
                           const uint32_t* colptr, const uint32_t* rowval, const float* nzval,
                           int32_t index_base);

/* ---- injected draws (optional; SURVEY.md 8c "draw injection") ------------------------ */
/* z_idx1/z_idx2 of :668-673. */
SCL_API int32_t scl_set_zero_candidates(scl_handle* h, int64_t n, const uint32_t* z_idx1, const uint32_t* z_idx2, int32_t index_base);
/* shuffle(nz_val) as a gather permutation (:275) and row_i (:247), both of length nnz. */
SCL_API int32_t scl_set_null_draws(scl_handle* h, int64_t n, const uint32_t* perm, const uint32_t* rows, int32_t index_base);
SCL_API int32_t scl_set_noise_baseline(scl_handle* h, double p_th);                       /* :709-712 */
SCL_API int32_t scl_push_search_sample(scl_handle* h, int64_t n, const uint32_t* sple_idx, int32_t index_base);  /* :731 */
SCL_API int32_t scl_push_perturb_sample(scl_handle* h, int64_t n, const uint32_t* sple_idx, int32_t index_base); /* :772 */
SCL_API int32_t scl_clear_draws(scl_handle* h);

/* ---- QC on the device (SURVEY.md 8f rank 3) ------------------------------------------- */
/* Thresholds of scLENS.preprocess (:160-162), same names, same defaults in the host mirrors. */
typedef struct {
  double min_tp_c, min_tp_g, max_tp_c, max_tp_g;      /* total counts per cell / gene: strict bounds (:186-187, :193-194) */
  int32_t min_genes_per_cell, max_genes_per_cell;     /* >= / < ; max 0 = off (:195, :213) */
  int32_t min_cells_per_gene, reserved;               /* >= (:188) */
  double mito_percent, ribo_percent;                  /* Float32 share strictly below percent/100; 0 = off (:198-211) */
} scl_qc_params;
/* preprocess (:160-236) on raw counts (N cells x M genes, CSC): cell / gene filters, drop of genes left empty, stable sort
 * of the survivors by their Float32 mean.  gene_flags[j]: bit 0 = mitochondrial name (r"^(?i)mt-." :196), bit 1 = ribosomal
 * (r"^(?i)RP[SL]." :197) - the caller matches the names.  Outputs: *n_cells / *n_genes / *out_nnz (0 cells: "There is no high
 * quality cells and genes" :231-234), fc_idx (kept cells, ascending, 0-based, capacity N) and gene_idx (kept genes in output
 * order, capacity M).  The filtered matrix becomes the handle's counts, as if passed to scl_set_counts_csc; read it back
 * with scl_get_counts_csc. */
SCL_API int32_t scl_op_preprocess(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr, const uint32_t* rowval,
                                  const float* nzval, int32_t index_base, const uint8_t* gene_flags, const scl_qc_params* p,
                                  int32_t* n_cells, int32_t* n_genes, int64_t* out_nnz, int32_t* fc_idx, int32_t* gene_idx);
/* The handle's counts as canonical 0-based CSC (colptr M+1, rowval / nzval nnz). */
SCL_API int32_t scl_get_counts_csc(scl_handle* h, uint32_t* colptr, uint32_t* rowval, float* nzval);

/* ---- the path ---------------------------------------------------------------------- */
/* :664-706: normalise, null matrix, get_sigev, mp_check. */
SCL_API int32_t scl_run_signal(scl_handle* h, scl_signal_info* out);
/* :709-819: noise baseline, sparsity search, perturbations, robustness scores, outputs. */
SCL_API int32_t scl_run_robustness(scl_handle* h, double th, double p_step, int32_t n_perturb, scl_robust_info* out);

/* Both stages as ONE call (:664-819).  On one GPU it is scl_run_signal followed by scl_run_robustness (skipped, with a
 * zeroed scl_robust_info, when there is no signal).  After scl_comm_init it is one pass shared by all ranks: cell-sharded
 * Gram matrices reduced to the rank that solves them, and the pass's eigensolves - data, null, binarised reference, search
 * steps - dealt to the ranks wave by wave.  Every rank must call it with the same arguments and ends with the same results.
 * n_perturb = 0 runs the signal stage alone (rout is zeroed). */
SCL_API int32_t scl_run_pass(scl_handle* h, double th, double p_step, int32_t n_perturb, scl_signal_info* sout,
                             scl_robust_info* rout);

/* ---- results (caller-allocated; sizes from the info structs) ------------------------- */
SCL_API int32_t scl_get_L(scl_handle* h, float* L /* nm, ascending, unfiltered (:378) */);
SCL_API int32_t scl_get_Lmp(scl_handle* h, float* L_mp /* n_Lmp */);
SCL_API int32_t scl_get_signal_ev(scl_handle* h, float* nL /* n_signal, descending */);
SCL_API int32_t scl_get_signal_evec(scl_handle* h, float* nV /* N x n_signal col-major, unit columns */);
SCL_API int32_t scl_get_gene_basis(scl_handle* h, float* g /* n_signal x M col-major (:813-819) */);
SCL_API int32_t scl_get_rec_vals(scl_handle* h, double* TGC /*N*/, double* mat2_mean /*M*/, double* mat2_std /*M*/,
                         double* norm_tgc /*N*/, double* cent /*M*/);                 /* :676-695 */
SCL_API int32_t scl_get_scores(scl_handle* h, float* b_ /* n_signal x C(n_perturb,2) col-major */,
                       double* m_scores /*n_signal*/, double* sd_scores /*n_signal*/); /* :795-803 */
SCL_API int32_t scl_get_sig_id(scl_handle* h, int32_t* sig_id /* n_robust, 0-based */);
SCL_API int32_t scl_get_null_csc(scl_handle* h, int64_t* nnz, uint32_t* colptr /*M+1*/, uint32_t* rowval, float* nzval);
SCL_API int32_t scl_get_search_trace(scl_handle* h, double* p /*n_search*/, double* second_smallest /*n_search*/);
SCL_API int32_t scl_get_perturbed_evec(scl_handle* h, int32_t replicate, float* nV /* N x min_pc */, float* nL /* min_pc */);

/* ---- function-level operators (host in / host out; unit parity) ---------------------- */
/* logn_scale(pre_scale(X)) (:650-652, :677-696).  layout 0: gene-major = column-major N x M
 * (Julia), 1: cell-major.  out_hi/out_lo are IEEE binary16 bit patterns (lo may be NULL);
 * ld = leading dimension in elements (multiple of 8). Statistic outputs may be NULL. */
SCL_API int32_t scl_op_normalize(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr,
                         const uint32_t* rowval, const float* nzval, int32_t layout, int64_t ld,
                         uint16_t* out_hi, uint16_t* out_lo,
                         double* TGC, double* mat2_mean, double* mat2_std, double* norm_tgc, double* cent);
/* _wishart_matrix (:332-344): G = A * A^T * scale, A = rows x K row-major binary16 (hi [+ lo]). */
SCL_API int32_t scl_op_gram(scl_handle* h, int32_t rows, int64_t K, int64_t ld, const uint16_t* a_hi, const uint16_t* a_lo,
                    float scale, float* G /* rows x rows, full symmetric */);
/* C[m,n] = alpha * sum_k A[m,k] B[n,k]; A m x K, B n x K row-major binary16; C col-major m x n
 * when c_colmajor else row-major. */
SCL_API int32_t scl_op_gemm_tn(scl_handle* h, int32_t m, int32_t n, int64_t K, int64_t lda, int64_t ldb,
                       const uint16_t* a_hi, const uint16_t* a_lo, const uint16_t* b_hi, const uint16_t* b_lo,
                       float alpha, int32_t c_colmajor, float* C);
/* _get_eigen (:375-382) on this library's own eigensolver (scl_op_syevd_tri with all vectors or none), ascending.  V may be
 * NULL (values only); ms (may be NULL): milliseconds of the solve. */
SCL_API int32_t scl_op_syevd(scl_handle* h, int32_t n, const float* A, float* L, float* V, double* ms);
/* The own eigensolver, the path scl_run_* use: the two-stage solver (dense -> band -> tridiagonal, Float64 Sturm multisection +
 * twisted factorisation, back-transformations Q2 and Q1, no library call); orders below 256 or a panel that cannot be factored:
 * own one-stage tridiagonalisation (cusolverDnSsytrd where it declines) + cusolverDnSormtr.  L: all n
 * eigenvalues ascending; V: the eigenvectors with ascending 0-based indices [v0, v1) as the columns of an n x (v1 - v0) column-major
 * array (vector v at V + (v - v0) n; v0 == v1: values only, V may be NULL).  out (may be NULL): out[0..2] = milliseconds of [reduction to tridiagonal form, tridiagonal eigenproblem, back-transformation + copy], out[3..5] =
 * [eigenvalue clusters re-solved by inverse iteration, eigenvalues in such clusters, 1 if the solve fell back to Ssyevd]. */
SCL_API int32_t scl_op_syevd_tri(scl_handle* h, int32_t n, const float* A, int32_t v0, int32_t v1, float* L, float* V, double out[6]);
/* _mp_calculation + _tw + mp_check (:424-487) on host doubles. out: [lambda_c,b_plus,b_minus,
 * ks_static, n_Lmp, mp_iters, pass, n_signal]. */
SCL_API int32_t scl_op_mp_fit(const float* L, int32_t nL, const float* Lr, int32_t nLr, double out[8]);
/* random_nz (:261-289) with injected draws -> canonical CSC (duplicates summed). */
SCL_API int32_t scl_op_permute_null(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr,
                            const uint32_t* rowval, const float* nzval, const uint32_t* perm, const uint32_t* rows,
                            int64_t* out_nnz, uint32_t* out_colptr, uint32_t* out_rowval, float* out_val);
/* sparse(vcat(...)) of :735 (binarise=1) / :774 (binarise=0) -> canonical CSC. */
SCL_API int32_t scl_op_perturb_merge(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr,
                             const uint32_t* rowval, const float* nzval, int64_t n_add, const uint32_t* add_row,
                             const uint32_t* add_col, int32_t binarise,
                             uint32_t* out_colptr, uint32_t* out_rowval, float* out_val);
/* d_arr of :742: for each column j of W (n x nw), max_i |<V[:,i], W[:,j]>| over the nv columns of V. */
SCL_API int32_t scl_op_corr_colabsmax(scl_handle* h, int32_t n, int32_t nv, int32_t nw, const float* V, const float* W, float* d);
/* Leading k eigenpairs of a symmetric n x n matrix by block Chebyshev subspace iteration. */
SCL_API int32_t scl_op_topk_subspace(scl_handle* h, int32_t n, const float* G, int32_t k, float* L /*k*/, float* V /* n x k */,
                             int32_t* iters);
/* robustness scoring (:786-806) on host-provided vectors: nV N x k, sets n_perturb x (N x min_pc). */
SCL_API int32_t scl_op_scores(scl_handle* h, int32_t N, int32_t k, int32_t min_pc, int32_t n_perturb, const float* nV,
                      const float* nV_sets, double th, float* b_, double* m_scores, double* sd_scores,
                      int32_t* sig_id, int32_t* n_robust);

/* ---- device-side draws of a production run (no injected draws), exposed for their own tests ----------------------- */
/* z_idx1 / z_idx2 of :668-673 drawn on the device from the handle's counts with `seed`: nnz uniform grid positions,
 * minus the stored entries, distinct in first-occurrence order.  *n = number of candidates; z1 / z2 (0-based rows / columns,
 * capacity >= nnz) may be NULL to ask for the count only.  The handle keeps the draw as its zero-candidate set. */
SCL_API int32_t scl_op_draw_zero_candidates(scl_handle* h, uint64_t seed, int64_t* n, uint32_t* z1, uint32_t* z2);
/* The uniform draws behind it, restated on the host (pure function of seed and draw index): rows[t], cols[t] of draw t. */
SCL_API int32_t scl_op_zero_candidate_draws(uint64_t seed, int64_t n_draws, int32_t N, int32_t M, uint32_t* rows, uint32_t* cols);
/* p_th of :709-712 drawn on the device: mean over n_rep of max |N(0, 1/nm)| over nm samples. */
SCL_API int32_t scl_op_noise_baseline(scl_handle* h, int32_t nm, int32_t n_rep, uint64_t seed, double* p_th);
/* sample(1:n_cand, n_take, replace=false) of :731 / :772 on the handle's zero candidates: the (row, col) pairs taken. */
SCL_API int32_t scl_op_draw_subset(scl_handle* h, int64_t n_take, uint64_t seed, uint32_t* rows, uint32_t* cols);

/* Host tail of the scoring (:797-806) on a k x n_pairs (column-major) table of pairwise similarities: Tukey fence,
 * median, corrected std, robust set {median > cos(th degrees)}.  Pure host code (testable without a GPU). */
SCL_API int32_t scl_op_scores_from_pairs(const float* b_, int32_t k, int32_t n_pairs, double th, double* m_scores,
                                 double* sd_scores, int32_t* sig_id, int32_t* n_robust);
/* get_denoised_df (:889-931) from the entries of the result Dict: pca_n1 N x r (the :pca_n1 columns), g_mat r x M
 * (= gene_basis[sig_id, :]), rec_vals TGC / mat2_mean / mat2_std / norm_tgc / cent_.  out: N x M column-major, Float64
 * (out_f32 = 0, as the reference's DataFrame) or Float32.  Replaces the cu()/mul! of :893-896 and the host broadcasts
 * of :921-927 by one fused kernel. */
SCL_API int32_t scl_op_denoise(scl_handle* h, int32_t N, int32_t M, int32_t r, const float* pca_n1, const float* g_mat,
                       const double* TGC, const double* mat2_mean, const double* mat2_std, const double* norm_tgc,
                       const double* cent, int32_t out_f32, void* out);

/* ---- apply_umap! (:863-873, UMAP.jl UMAP_) on the device ------------------------------------------------------------ */
/* Parameters of UMAP_ with its defaults in the host mirrors: n_neighbors 15, n_components 2, n_epochs 300, metric 1
 * (0 = euclidean, 1 = cosine), init 0 (0 = spectral, 1 = random), neg_sample_rate 5, spectral_maxiter 100, min_dist 0.1,
 * spread 1, learning_rate 1, repulsion_strength 1, local_connectivity 1, seed 0. */
typedef struct {
  int32_t n_neighbors;       /* k: 1 <= k <= 64, k < N */
  int32_t n_components;      /* nc: 1 <= nc <= 16 */
  int32_t n_epochs;          /* >= 0; 0 returns the start */
  int32_t metric;            /* 0 euclidean, 1 cosine (1/2 |x^ - y^|^2 of unit rows; a zero row is at distance 1) */
  int32_t init;              /* 0 spectral (random start when the iteration does not converge), 1 uniform in [-10, 10] */
  int32_t neg_sample_rate;   /* negative samples per fired edge */
  int32_t spectral_maxiter;  /* outer iterations of the spectral block iteration (degree-8 Chebyshev filter each) */
  int32_t reserved0;
  double min_dist, spread, learning_rate, repulsion_strength, local_connectivity;
  uint64_t seed;             /* every draw is a hash of (seed, stream, epoch, vertex, slot) */
  int32_t reserved[4];
} scl_umap_params;

typedef struct {
  double a, b;               /* fitted 1 / (1 + a x^(2b)) */
  int64_t graph_nnz;         /* stored entries of the symmetric fuzzy graph */
  int32_t spectral_iters;    /* outer iterations of the spectral start (0 when not run) */
  int32_t init_fallback;     /* 1: the spectral start did not converge and the random start was taken */
  double t_knn_ms, t_graph_ms, t_init_ms, t_layout_ms;   /* CUDA events on the handle's stream */
  int32_t reserved[4];
} scl_umap_info;

/* Exact k nearest neighbours of the rows of X (N x d column-major), self excluded, ascending in (distance, index):
 * idx / dist are N x k row-major ([i * k + s], 0-based).  metric as in scl_umap_params. */
SCL_API int32_t scl_op_knn(scl_handle* h, int32_t N, int32_t d, const float* X, int32_t k, int32_t metric, int32_t* idx,
                           float* dist);
/* UMAP_(X', nc) of apply_umap!: kNN, fuzzy graph, start, layout.  init_embedding (N x nc column-major) replaces the
 * computed start when not NULL (with n_epochs = 0 each stage can be checked on its own).  embedding: N x nc column-major.
 * The kNN and the graph stay on the handle (scl_get_umap_knn, scl_get_umap_graph).  Same seed, same bits. */
SCL_API int32_t scl_op_umap(scl_handle* h, int32_t N, int32_t d, const float* X, const scl_umap_params* p,
                            const float* init_embedding, float* embedding, scl_umap_info* info);
/* The fuzzy graph of the last scl_op_umap: symmetric N x N CSR, sorted columns, 0-based.  Call with NULL arrays for *nnz. */
SCL_API int32_t scl_get_umap_graph(scl_handle* h, int64_t* nnz, uint32_t* rowptr /* N+1 */, uint32_t* colidx, float* val);
/* The kNN of the last scl_op_umap (N x k row-major, as scl_op_knn). */
SCL_API int32_t scl_get_umap_knn(scl_handle* h, int32_t* idx, float* dist);
/* The a / b fit of UMAP_ (Levenberg-Marquardt on the host, Float64).  Pure host code. */
SCL_API int32_t scl_umap_fit_ab(double min_dist, double spread, double* a, double* b);

/* ---- clustering (scICE clustering!: Leiden trials over resolutions, IC of each cluster count) on the device ---------- */
/* Leiden with the modularity objective and resolution gamma (RB configuration model).  Weights are fixed point
 * round(w 2^shift) (at least 1), shift <= 32 from the largest weight and nnz; every trial's draws hash (seed, trial).
 * Defaults in the host mirrors: n_trials 50, max_iterations 10, max_sweeps 64, theta 0.01, seed 0. */
typedef struct {
  int32_t n_trials;          /* T >= 1 trials per resolution */
  int32_t max_iterations;    /* >= 1: restarts from the last labels until one changes no label */
  int32_t max_sweeps;        /* >= 1: local-moving sweeps per level (a level that reaches it is counted in capped_levels) */
  int32_t reserved0;
  double theta;              /* > 0: randomness of the refinement (probability ~ exp(gain / theta), leidenalg's 0.01) */
  uint64_t seed;
  int32_t reserved[4];
} scl_leiden_params;

typedef struct {
  int32_t max_levels;        /* most levels of one iteration of one trial */
  int32_t max_iterations;    /* most iterations of one trial */
  int32_t capped_levels;     /* levels whose local moving stopped at max_sweeps */
  int32_t weight_shift;      /* the fixed-point exponent */
  int64_t copy_levels;       /* sum over trials and iterations of the levels run */
  double t_validate_ms, t_move_ms, t_refine_ms, t_aggregate_ms, t_labels_ms;   /* CUDA events / host clock around synchronised work */
  int32_t reserved[4];
} scl_leiden_info;

/* Resolution search of the clustering: for every k in [k_min, k_max] the resolution whose trials most often give exactly k
 * clusters, and the IC of those trials.  Defaults: k_min 2, k_max 20, n_trials 50, max_rounds 12, n_grid 16, max_widen 4,
 * gamma_lo 0.01, gamma_hi 10, and the Leiden defaults above. */
typedef struct {
  int32_t k_min, k_max;      /* 1 <= k_min <= k_max <= N */
  int32_t n_trials;          /* >= 2 */
  int32_t max_rounds;        /* >= 0 bisection / widening rounds after the start grid */
  int32_t n_grid;            /* >= 2 log-spaced resolutions of the start grid on [gamma_lo, gamma_hi] */
  int32_t max_widen;         /* decades the search may add below gamma_lo and above gamma_hi */
  int32_t max_iterations, max_sweeps;
  double gamma_lo, gamma_hi, theta;
  uint64_t seed;
  int32_t reserved[4];
} scl_cluster_params;

typedef struct {
  int32_t n_rounds;          /* batches run, the start grid included */
  int32_t n_evaluated;       /* resolutions evaluated */
  int32_t n_found;           /* cluster counts in [k_min, k_max] found */
  int32_t weight_shift;
  int64_t copy_levels;
  double t_validate_ms, t_leiden_ms, t_ecs_ms, t_total_ms;
  int32_t reserved[4];
} scl_cluster_info;

/* R x T Leiden trials on an N-vertex graph.  rowptr (N+1) / colidx / val (nnz): symmetric CSR, sorted columns, 0-based,
 * finite positive weights (validated on the device: SCL_ERR_GRAPH otherwise); rowptr == NULL takes the fuzzy graph of
 * the handle's last scl_op_umap.  labels: [R][T][N] (ids 0..k-1 by cluster size, descending, ties by smallest member),
 * n_clusters / modularity: [R][T].  A trial's labels do not depend on the other trials of the batch. */
SCL_API int32_t scl_op_leiden(scl_handle* h, int32_t N, int64_t nnz, const uint32_t* rowptr, const uint32_t* colidx,
                              const double* val, int32_t R, const double* resolutions, const scl_leiden_params* p,
                              int32_t* labels, int32_t* n_clusters, double* modularity, scl_leiden_info* info);
/* T x T element-centric similarity (row-major) of T labelings [T][N] with ids in [0, N). */
SCL_API int32_t scl_op_label_ecs(scl_handle* h, int32_t T, int32_t N, const int32_t* labels, double* ecs);
/* The whole search (graph as scl_op_leiden).  Per k = k_min + i: found[i] (0 / 1), gamma[i], share[i] (fraction of the
 * trials at gamma[i] with exactly k clusters), ic[i] (1 / p^T S p over all trials at gamma[i]) and labels[i][N] (of the
 * trials with exactly k clusters, the one with the largest ECS row sum, ties to the lowest); entries of a k not found are 0 / NaN / -1.  eval_gamma / eval_mode
 * (capacity eval_cap, may be NULL) receive the evaluated resolutions and their modal cluster counts in evaluation order. */
SCL_API int32_t scl_op_cluster(scl_handle* h, int32_t N, int64_t nnz, const uint32_t* rowptr, const uint32_t* colidx,
                               const double* val, const scl_cluster_params* p, int32_t* found, double* gamma, double* share,
                               double* ic, int32_t* labels, int32_t eval_cap, double* eval_gamma, int32_t* eval_mode,
                               scl_cluster_info* info);
/* One planning step of the search (host only): from n evaluated (gamma, modal count) pairs, the next resolutions (at most
 * k_max - k_min + 3, ascending; *n_out = 0 when the search is done). */
SCL_API int32_t scl_cluster_plan(int32_t n, const double* gammas, const int32_t* modes, const scl_cluster_params* p,
                                 double* out, int32_t* n_out);

/* ---- kernel-level timing harness (device-resident synthetic operands; used by bench.py and the ncu captures) ---- */
/* Gram / GEMM kernel alone: rows x K binary16 operand generated on the device; mode bit0 = split (hi+lo) operands,
 * bit1 = full GEMM instead of the syrk schedule; chunk_kb = k-blocks per accumulation chunk (0 = default).
 * ms_avg: CUDA-event time per launch on the handle's stream; checksum: mean diagonal of the result. */
SCL_API int32_t scl_bench_gram(scl_handle* h, int32_t rows, int64_t K, int32_t mode, int32_t chunk_kb, int32_t reps,
                       double* ms_avg, double* checksum);
/* Normalisation kernels on the handle's counts (:677-696): statistics pre-passes and the fused densify writer. */
/* Timing study of the library eigensolvers on an n x n Wishart matrix generated on the device (CUDA events around the
 * solver call).  mode 0: Ssyevd with vectors (what the path calls), 1: values only, 2: Ssyevdx with the vectors of the
 * il..iu smallest eigenvalues (1-based, inclusive), 3: Xsyevd (64-bit API) with vectors, 4: Ssytrd alone (the
 * tridiagonalisation half of a one-stage solve), 5: Sormtr alone (back-transformation of an n x n block), 6 / 7 / 8: the
 * own tridiagonal stage with all vectors / the vectors il..iu / values only.  mode + 16: solve the data Gram matrix of the
 * last scl_run_signal (needs n == nm) instead of the synthetic one. */
SCL_API int32_t scl_bench_syevd(scl_handle* h, int32_t n, int32_t mode, int32_t il, int32_t iu, double* ms);
/* `nsolves` independent solves on the own eigensolver (as scl_op_syevd; mode 0: with vectors, 1: values only) of n x n
 * Wishart matrices issued at the same time from `nsolves` host threads, each with its own stream and solver; ms_wall = host
 * wall time until all are done (after one untimed round).  Answers whether independent eigensolves (sparsity-search steps)
 * overlap on ONE GPU. */
SCL_API int32_t scl_bench_syevd_concurrent(scl_handle* h, int32_t n, int32_t nsolves, int32_t mode, double* ms_wall);
/* Test hook (process-wide): on != 0 makes the own eigensolver take the one-stage path at every order, 0 restores the
 * choice by order. */
SCL_API int32_t scl_debug_force_one_stage(int32_t on);
/* Stage times of the handle's last own-path eigensolve, milliseconds: out[0..4] = dense->band, band->tridiagonal, tridiagonal
 * eigenproblem, stage-2 back-transformation, stage-1 back-transformation (all 0 unless the two-stage path ran); out[5] = 1 when
 * the two-stage path produced the result; out[6] = number of two-stage solves of this handle that fell back to one stage;
 * out[7] = number of own-path solves that fell back to cusolverDnSsyevd. */
SCL_API int32_t scl_debug_last_solve(scl_handle* h, double out[8]);
/* Totals over the handle's two-stage solves since scl_reset_profile, milliseconds: out[0..4] = the five stages as above; out[5] =
 * number of two-stage solves; out[6] = eigenvector columns back-transformed; out[7] = solves that fell back to one stage. */
SCL_API int32_t scl_debug_eig_stage_totals(scl_handle* h, double out[8]);
/* The stages of the two-stage reduction one by one on a host matrix A (n x n, symmetric, n a multiple of 4), for the stage-wise
 * parity tests: AB (n x 128, band storage AB[j*128 + (i-j)]) after dense -> band; d (n), e (n-1) after band -> tridiagonal;
 * Q2 (n x n, column v at Q2 + v*n) = the stage-2 transformation applied to the identity; Q (same layout) = Q1 Q2.  Any output
 * pointer may be NULL.  flags[0] = panel failure flag, flags[1] = number of panels. */
SCL_API int32_t scl_debug_two_stage(scl_handle* h, int32_t n, const float* A, float* AB, float* d, float* e, float* Q2, float* Q,
                                    int32_t flags[2]);
/* The Float64 Rayleigh-Ritz refinement of the eigenvalues on its own, as the pipeline runs it after an eigensolve: G (n x n,
 * symmetric) and V (n x n, the eigenvectors as rows, any scaling, ascending order), n >= 2.  L (n) = the refined eigenvalues,
 * ascending; stats (may be NULL): stats[0] = number of clusters solved as Rayleigh-Ritz blocks, stats[1] = size of the largest
 * (1 when there is none). */
SCL_API int32_t scl_debug_refine(scl_handle* h, int32_t n, const float* G, const float* V, float* L, int32_t stats[2]);
/* The Gram matrix with the exact diagonal and the tensor-core bias calibration, as the pipeline forms it: the syrk of scl_op_gram
 * (operand layout and scale as there; the handle's cta_group and gram_chunk_kb), the calibration samples, the diagonal set to
 * scale * diag (diag: rows Float64 sums of squares), the fitted factor and the diagonal scaled by it.  Calibrates at every
 * rows >= 2 (the pipeline from 64 on).  G (rows x rows) = the result; factor (may be NULL) = the common factor 1 - delta. */
SCL_API int32_t scl_debug_gram_calibrated(scl_handle* h, int32_t rows, int64_t K, int64_t ld, const uint16_t* a_hi, const uint16_t* a_lo,
                                          float scale, const double* diag, float* G, double* factor);
/* The tcgen05 GEMM on its own with every launch field given: C = alpha * A B' (A: m x K, B: n x K, binary16 rows of lda / ldb
 * elements; a_lo / b_lo: the low-order parts of split mode, both or neither).  All operand and result pointers are DEVICE
 * pointers (16-byte aligned); the call synchronises its stream before it returns.  epi: 0 Store C[i*ldc + j], 1
 * StoreTransposed C[j*ldc + i], 2 ColAbsMax C[j] = max(C[j], max_i |alpha (A B')_ij|) (C pre-filled by the caller).  syrk: A
 * and B the same operand (m == n), lower tile triangle mirrored (Store only).  splits > 1: split-K partial s at C +
 * s*split_stride; reduce_out (may be NULL): then also reduce_out[e] = reduce_scale * sum_s partial_s[e] for e <
 * split_stride, as the pipeline reduces its partials.  chunk_kb: k-blocks of 64 per tensor-core accumulation chain (0: the
 * default).  launch (may be NULL) = the launch as resolved: block_n, tile-splits, units (CTAs, or CTA pairs with
 * cta_group 2), effective splits, chunk_kb, chunked, the most tile-splits one unit takes.  Returns SCL_ERR_INVALID, and
 * launches nothing, for inconsistent arguments. */
SCL_API int32_t scl_debug_gemm(scl_handle* h, int32_t m, int32_t n, int64_t K, const uint16_t* a_hi, const uint16_t* a_lo, int64_t lda,
                               const uint16_t* b_hi, const uint16_t* b_lo, int64_t ldb, float alpha, int32_t epi, int32_t syrk,
                               int32_t splits, int64_t split_stride, int32_t chunk_kb, int32_t cta_group, float* C, int64_t ldc,
                               float* reduce_out, float reduce_scale, int32_t launch[7]);
/* Tuning studies only (process-wide).  stat_variant: launch shape of the statistics passes (0-7: line passes,
 * 8: strip passes; < 0 keeps the current one).  stat_heavy: line length above which a whole CTA takes a line
 * (<= 0 keeps).  writer: dense writer, -1 automatic, 0 register/overlay writer, 1 TMA bulk-store writer, 2 / 3
 * TMA bulk-store writer with one / two cp.async-staged entries per thread and line (<= -2 keeps).  Every writer and every
 * line-pass variant (0-7) gives identical results; the strip passes (8) and another stat_heavy sum the Float64
 * statistics in another order, which can change their last bits. */
SCL_API int32_t scl_debug_set_tuning(int32_t stat_variant, int32_t stat_heavy, int32_t writer);
SCL_API int32_t scl_bench_normalize(scl_handle* h, int32_t layout, int32_t with_lo, int32_t reps, double* ms_stats,
                            double* ms_densify, double* alg_bytes_densify);

#ifdef __cplusplus
}
#endif
#endif /* SCLENS_B200_H */
