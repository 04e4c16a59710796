// State of one sclens() call: everything lives on the device between the two run stages.
#pragma once
#include <deque>
#include <memory>
#include <string>
#include <vector>
#include "../../include/sclens_b200.h"
#include "common.cuh"
#include "eigen.h"
#include "prof.h"

struct scl_handle {
  scl_config cfg{};
  std::string err;
  cudaStream_t st = nullptr;
  std::unique_ptr<scl::Solver> solver;
  int world = 1, rank = 0;
  void* nccl = nullptr;   // ncclComm_t
  scl::Prof prof;
  scl::DBuf<double> gram_factor;   // common factor (1 - delta) of the Gram matrix gram_of() produced last
  cudaEvent_t t0 = nullptr, t1 = nullptr;

  // inputs
  scl::SpMat X;
  bool have_X = false;
  // injected draws
  bool have_zc = false;
  scl::DBuf<uint32_t> z1, z2;
  size_t n_cand = 0;
  bool have_null_draws = false;
  scl::DBuf<uint32_t> null_perm, null_rows;
  bool have_pth = false;
  double p_th = 0;
  std::vector<std::vector<uint32_t>> search_sples, perturb_sples;   // indexed by search step / replicate

  // signal stage results
  bool signal_done = false;
  scl_signal_info sinfo{};
  scl::NormStats S_main;
  scl::SpMat Xnull;
  std::vector<float> L, Lmp, nL;
  scl::DBuf<float> d_nV;          // [n_signal][N]  (== column-major N x n_signal)
  std::vector<double> rec_tgc, rec_mean, rec_std, rec_l2, rec_cent;

  // work buffers kept between calls (a second pass over the same handle allocates nothing)
  scl::DBuf<__half> ws_op_hi, ws_op_lo;     // dense Gram operand (hi, optional lo)
  scl::DBuf<__half> ws_vr_hi, ws_vr_lo;     // reference eigenbasis of the binarised matrix (search loop)
  scl::DBuf<float> ws_G, ws_G2, ws_W, ws_W2, ws_Gkeep;
  scl::SpMat ws_Xp;                         // perturbed matrix of the current search step / replicate
  scl::NormStats ws_Sp, ws_Sn;              // its statistics; the null matrix's statistics

  // robustness stage results
  bool robust_done = false;
  scl_robust_info rinfo{};
  std::vector<double> trace_p, trace_d;
  scl::DBuf<float> d_sets;        // [n_perturb][min_pc][N]
  std::vector<float> set_L;       // [n_perturb][min_pc]
  std::vector<float> b_;          // n_signal x n_pairs, column-major
  std::vector<double> m_scores, sd_scores;
  std::vector<int32_t> sig_id;
  std::vector<float> gene_basis;  // [M][n_signal] (== column-major n_signal x M)

  // apply_umap: kNN ([N][k], ascending (distance, index)) and fuzzy graph (symmetric CSR, sorted columns) of the last call
  int uk_N = 0, uk_k = 0;
  scl::DBuf<int32_t> uk_idx;
  scl::DBuf<float> uk_dist;
  bool have_umap_graph = false;
  int ug_N = 0;
  size_t ug_nnz = 0;
  scl::DBuf<uint32_t> ug_rowptr, ug_col, ug_rev;   // ug_rev[e]: position of the reverse edge of e
  scl::DBuf<float> ug_val;
  scl::DBuf<double> ug_deg;
};

namespace scl {
// refine.cu
void refine_eigenvalues(const float* dG, const float* dV, int n, float* dW, cudaStream_t st);
// pipeline.cu
void run_signal(scl_handle* h);
void run_robustness(scl_handle* h, double th, double p_step, int n_perturb);
void run_pass(scl_handle* h, double th, double p_step, int n_perturb);
int pass_refine_task(int world);
int pass_task_step(int task, int refine_task);
void score_from_pairs(const std::vector<float>& b_, int k, int n_pairs, double th, std::vector<double>& m,
                      std::vector<double>& sd, std::vector<int32_t>& sig);
void plan_gram_shard(int64_t K, int64_t ld, int world, int rank, int64_t* k0, int64_t* k1);
// umap.cu
// exact kNN of the N x d column-major device matrix dX: d_idx / d_dist [N][k], self excluded, ascending (distance, index)
void knn_device(const float* dX, int N, int d, int k, int metric, int32_t* d_idx, float* d_dist, cudaStream_t st);
void umap_fit_ab(double min_dist, double spread, double* a, double* b);
uint64_t umap_stream_key(uint64_t seed, uint32_t stream, uint32_t epoch);
// d_init: N x nc column-major start (null: computed start); d_emb: N x nc column-major result
void umap_run(scl_handle* h, const float* dX, int N, int d, const scl_umap_params& p, const float* d_init, float* d_emb,
              scl_umap_info* info);
// preprocess.cu
bool preprocess_device(const SpMat& X, const uint8_t* d_gene_flags, const scl_qc_params& p, std::vector<int32_t>& fc_idx,
                       std::vector<int32_t>& gene_idx, SpMat& out, cudaStream_t st);
// shared building blocks (also used by the scl_op_* entry points)
// shard=true (and world > 1): every rank contracts its own slice of the long axis (cells when N > M) and the
// partial Gram matrices are summed with ncclAllReduce
void gram_of(scl_handle* h, const SpMat& A, NormStats& S, DBuf<__half>& hi, DBuf<__half>& lo, float* dG, int nm,
             float scale, bool split, bool shard = false, int reduce_root = -1);
void corr_colabsmax(scl_handle* h, const float* dV, int nv, const float* dW, int nw, int n, float* d_out);
void topk_subspace(scl_handle* h, const float* dG, int n, int k, float* dL, float* dV, int* iters);
void score_sets(scl_handle* h, int N, int k, int min_pc, int n_perturb, const float* d_nV, const float* d_sets,
                double th, std::vector<float>& b_, std::vector<double>& m, std::vector<double>& sd,
                std::vector<int32_t>& sig);
}  // namespace scl
