// Block building blocks of the Chebyshev subspace iterations (subspace.cu): tall-skinny Float64 Gram products,
// row combinations and Cholesky QR of blocks stored vector-major ([rows][n], each vector contiguous).  Shared by the
// perturbation-stage eigensolver (subspace.cu) and the spectral start of the UMAP layout (umap.cu).
#pragma once
#include <cstdint>
#include <vector>
#include "common.cuh"

struct scl_handle;

namespace scl {

// splitmix64 finaliser: the counter-based hash behind the device-side draws
__host__ __device__ inline uint64_t mix64s(uint64_t x) {
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27; x *= 0x94d049bb133111ebull;
  x ^= x >> 31;
  return x;
}

struct BlockCtx {
  scl_handle* h;
  cudaStream_t st;
  int n;
  size_t ldn;
  const __half *g_hi, *g_lo;
  // true: gram_ts sums its per-CTA partial products in a fixed order (bitwise reproducible); false: Float64 atomics
  bool fixed_order = false;
};

// S[ra][rb] = A[ra][n] * B[rb][n]^T (Float64)
void gram_ts(const BlockCtx& c, const float* A, int ra, const float* B, int rb, double* dS);
// out[c][t] = beta * base[c][t] + alpha * sum_r Tt[c][r] * wgt[r] * In[r][t]   (wgt may be null)
void combine_rows(const BlockCtx& c, const float* In, int rin, const double* dTt, int rout, double alpha, const float* base,
                  double beta, float* out, const double* wgt = nullptr);
// host Cholesky S = R^T R (upper), returns Tt[c][r] = (R^-1)[r][c]; false when not positive definite
bool chol_inverse_t(std::vector<double>& S, int b, std::vector<double>& Tt);
// Q[rows][n] <- orthonormal basis of its row space (Cholesky QR, Float64 Gram); tmp is scratch [rows][n]
void chol_qr(const BlockCtx& c, float* Q, int rows, float* tmp, int passes);
// res[r] = | Z_r - theta_r Q_r |_2 (fixed-order reduction)
void residual_norms(const BlockCtx& c, const float* Z, const float* Q, const double* dTheta, int rows, double* dRes);

}  // namespace scl
