#pragma once
#include <cuda_runtime.h>
#include <vector>

namespace scl {

struct Solver {
  struct Impl;
  Impl* impl;
  explicit Solver(cudaStream_t st);
  ~Solver();
  Solver(const Solver&) = delete;
  Solver& operator=(const Solver&) = delete;
  // syevd_tri with all vectors (vectors = true) or none: eigenvalues ascending in dW, eigenvectors overwrite dA (col-major)
  void syevd(float* dA, int n, float* dW, bool vectors, cudaStream_t st);
  void dsyevd_small(double* dA, int n, double* dW, cudaStream_t st);
  // The own eigensolver: reduction to tridiagonal form -> Float64 multisection + twisted factorisation (tridiag.cu) ->
  // back-transformation.  All n eigenvalues ascending in dW; the eigenvectors with ascending indices [v0, v1) in rows
  // [v0, v1) of dA's memory (v0 == v1: values only); the other rows of dA are overwritten with scratch.  Orders >= 4 kBand take
  // the two-stage reduction, smaller ones the one-stage path.  Falls back to Ssyevd on a kept copy of the matrix (all
  // vectors) when the tridiagonal stage fails; returns true when it did not have to.
  bool syevd_tri(float* dA, int n, float* dW, int v0, int v1, cudaStream_t st);
  // one stage: own tridiagonalisation (sytrd.cu; cusolverDnSsytrd where it declines), tridiag.cu, cusolverDnSormtr
  bool syevd_tri_one_stage(float* dA, int n, float* dW, int v0, int v1, cudaStream_t st);
  // two-stage reduction (sy2sb.cu, sb2st.cu, backtrans.cu) with the same contract; a panel that cannot be factored or a failed
  // tridiagonal stage falls back to syevd_tri_one_stage
  bool syevd_2stage(float* dA, int n, float* dW, int v0, int v1, cudaStream_t st);
  double ts_ms[5] = {0, 0, 0, 0, 0};   // last two-stage solve: dense->band, band->tridiagonal, tridiagonal eigenproblem, Q2, Q1 + copy
  bool tri_two_stage = false;
  // totals over the two-stage solves since the last reset: the five stages above, [5] solves, [6] eigenvector columns back-transformed
  double ts_total[7] = {0, 0, 0, 0, 0, 0, 0};
  int ts_fallbacks = 0;
  // milliseconds of the last syevd_tri call: [0] reduction to tridiagonal form, [1] eigenvalues + eigenvectors of T,
  // [2] back-transformation + copy
  double tri_ms[3] = {0, 0, 0};
  int tri_clusters = 0, tri_clustered = 0, tri_fallbacks = 0;
  bool tri_own_sytrd = false;   // the last syevd_tri call tridiagonalised with sytrd.cu
  // timing study of the library's symmetric eigensolvers on an n x n matrix (overwritten); returns milliseconds.
  // mode 0: Ssyevd vectors, 1: Ssyevd values only, 2: Ssyevdx vectors of the il..iu smallest, 3: Xsyevd (64-bit API) vectors
  double bench(float* dA, int n, float* dW, int mode, int il, int iu, cudaStream_t st);
};

struct TridiagStats {
  int clusters = 0, clustered = 0;   // groups of eigenvalues closer than 1e-9 |T| and how many eigenvalues they hold
};
// tridiag.cu: all eigenvalues (ascending; Float64 w64 and Float32 w32) of the symmetric tridiagonal (d32, e32) and the unit
// eigenvectors with ascending indices [v0, v1) as rows of Z; false when they came out non-finite / too degenerate
bool tridiag_eigen(const float* d32, const float* e32, int n, double* w64, float* w32, int v0, int v1, float* Z,
                   long long ldz, cudaStream_t st, TridiagStats* stats);

// sytrd.cu: own Householder tridiagonalisation (persistent cooperative kernel), output as ssytrd('L'); false = not handled
bool sytrd_lower(float* dA, int n, int lda, float* d_d, float* d_e, float* d_tau, cudaStream_t st);
// test hook (process-wide): syevd_tri takes the one-stage path at every order, so that path is tested at orders >= 4 kBand
void force_one_stage(bool on);

struct MpFit {
  std::vector<float> L_mp;
  double lambda_c, b_plus, b_minus, gamma, ks_static;
  int iters, n_signal;
  bool pass;
};
// _mp_calculation(L, Lr) + _tw + mp_check; caller passes Lr already without its largest value (:537)
MpFit mp_fit(const float* L, int nL, const float* Lr, int nLr);

}  // namespace scl
