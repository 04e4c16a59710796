// Stage 1 of the two-stage eigensolver: symmetric dense -> symmetric band (half bandwidth kBand), lower storage.
//
// Per panel (kBand columns, the m rows below the band):
//   1. CholeskyQR with a Float64 Gram matrix: G = P'P (k_dot64: per-slab partials, fixed-order sum), R = chol(G).  The
//      Gram matrix is exact to Float64 rounding of Float32 products, so the factor is good for panels with condition
//      numbers up to ~1e7 - no column-by-column Householder sweep (2 kBand grid-wide reductions) over the panel.
//   2. Householder reconstruction (Ballard, Demmel, Grigori, Jacquelin, Nguyen, Solomonik 2015): with Q = P R^-1, the LU
//      factorisation Q1 - S = L U of the top kBand x kBand block (S = the sign matrix that makes every pivot >= 1 in
//      modulus) gives the unit lower trapezoidal V = [L; P2 (U R)^-1] of the compact WY form Q = (I - V T V')[I; 0] S.
//      All kBand x kBand work runs in Float64 in one CTA (k_panel_factor); the rows below are ONE slab product with the
//      kBand x kBand matrix (U R)^-1.
//   3. T is recomputed from the V actually stored: inv(T) = striu(V'V) + diag(V'V)/2 (k_tfactor), so I - V T V' is
//      orthogonal to working precision whatever rounding V suffered; the band receives R' = S R.
//   4. Two-sided update of the trailing matrix, lower triangle only: Y = A22 V (k_symm_tc: every lower tile is used
//      for its rows and, transposed, for its columns), Z = Y T, S2 = T'(V'Z), W = Z - V S2 / 2, A22 -= V W' + W V' (k_syr2k_tc).
// The two large products (k_symm_tc, k_syr2k_tc) run on the tensor-core tile engines of sgemm_tile.cuh: split binary16 for a
// matrix that passes half_range_ok, three-term TF32 otherwise; the panel-sized products run on its FP32 engine.  Every
// reduction has a fixed order.
#include <algorithm>
#include <cmath>
#include <vector>
#include "common.cuh"
#include "sgemm_tile.cuh"
#include "tmp.cuh"
#include "twostage.h"

namespace scl {
namespace {

constexpr int B = kBand;
// rows per CTA of the panel dot products (a multiple of 64): fewer rows = more CTAs on these short kernels, which sit on the
// critical path of every panel, against more partial matrices for the single-CTA kernels that sum them
constexpr int kSlab = 256;

// part[p][c1][c2] = sum over the rows of slab p of X[c1][i] * Y[c2][i].  F64 = true: every product accumulated in Float64 (the
// panel Gram matrix, whose Cholesky factor squares the panel's condition number).  F64 = false: Float32 accumulation over 64
// rows at a time, the 64-row sums added in Float64 (V'V and V'Z, which enter T and W at working precision only; the
// Float64 pipe of this part is an order of magnitude slower than the Float32 one).
template <bool F64>
__global__ void __launch_bounds__(256) k_dot64(const float* __restrict__ X, long long ldx, const float* __restrict__ Y,
                                               long long ldy, int rows, int slab, double* __restrict__ part) {
  // F64: 32-row chunks converted to Float64 once, on the way into shared memory (a conversion per use was 16 per element
  // and cost more than the multiply-adds); FP32: 64-row chunks
  constexpr int RC = F64 ? 32 : B;
  __shared__ __align__(16) unsigned char raw[2 * B * 33 * 8];
  const int tid = (int)threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int base = (int)blockIdx.x * slab, end = min(rows, base + slab);
  double acc[4][4];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
  for (int r0 = base; r0 < end; r0 += RC) {
    __syncthreads();
    if constexpr (F64) {
      double (*Xd)[33] = reinterpret_cast<double (*)[33]>(raw);
      double (*Yd)[33] = Xd + B;
      for (int e = tid; e < B * RC; e += 256) {
        const int c = e / RC, i = e % RC;
        const bool ok = r0 + i < end;
        Xd[c][i] = ok ? (double)X[(long long)c * ldx + r0 + i] : 0.0;
        Yd[c][i] = ok ? (double)Y[(long long)c * ldy + r0 + i] : 0.0;
      }
      __syncthreads();
#pragma unroll 4
      for (int r = 0; r < RC; ++r) {
        double xa[4], yb[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) xa[a] = Xd[ty + 16 * a][r];
#pragma unroll
        for (int b = 0; b < 4; ++b) yb[b] = Yd[tx + 16 * b][r];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) acc[a][b] = fma(xa[a], yb[b], acc[a][b]);
      }
    } else {
      float (*Xs)[B + 1] = reinterpret_cast<float (*)[B + 1]>(raw);
      float (*Ys)[B + 1] = Xs + B;
      for (int e = tid; e < B * B; e += 256) {
        const int c = e / B, i = e % B;
        const bool ok = r0 + i < end;
        Xs[c][i] = ok ? X[(long long)c * ldx + r0 + i] : 0.f;
        Ys[c][i] = ok ? Y[(long long)c * ldy + r0 + i] : 0.f;
      }
      __syncthreads();
      float fa[4][4];
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) fa[a][b] = 0.f;
#pragma unroll 8
      for (int r = 0; r < B; ++r) {
        float xa[4], yb[4];
#pragma unroll
        for (int a = 0; a < 4; ++a) xa[a] = Xs[ty + 16 * a][r];
#pragma unroll
        for (int b = 0; b < 4; ++b) yb[b] = Ys[tx + 16 * b][r];
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
          for (int b = 0; b < 4; ++b) fa[a][b] = fmaf(xa[a], yb[b], fa[a][b]);
      }
#pragma unroll
      for (int a = 0; a < 4; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] += (double)fa[a][b];
    }
  }
  double* out = part + (size_t)blockIdx.x * B * B;
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) out[(ty + 16 * a) * B + tx + 16 * b] = acc[a][b];
}

// out[e] = sum over the slabs p (in order) of part[p][e]: sixteen CTAs instead of the single CTA of the small-matrix kernel that
// consumes the sum (which otherwise spends most of its time reading nslab x 32 KB)
__global__ void __launch_bounds__(256) k_sum_dparts(const double* __restrict__ part, int nslab, double* __restrict__ out) {
  const int e = (int)blockIdx.x * 256 + (int)threadIdx.x;
  double s0 = 0.0, s1 = 0.0;
  int p = 0;
  for (; p + 1 < nslab; p += 2) {
    s0 += part[(size_t)p * B * B + e];
    s1 += part[(size_t)(p + 1) * B * B + e];
  }
  if (p < nslab) s0 += part[(size_t)p * B * B + e];
  out[e] = s0 + s1;
}

typedef double (*Mat65)[B + 1];

__device__ void sum_parts(const double* part, int nslab, Mat65 G) {
  for (int e = (int)threadIdx.x; e < B * B; e += (int)blockDim.x) {
    double s = 0;
    for (int p = 0; p < nslab; ++p) s += part[(size_t)p * B * B + e];
    G[e / B][e % B] = s;
  }
}

// M = inverse of the upper triangular U (both kBand x kBand, Float64 in shared memory); thread c < kBand owns column c
__device__ void invert_upper(Mat65 U, Mat65 M) {
  const int c = (int)threadIdx.x;
  if (c < B) {
    for (int r = B - 1; r > c; --r) M[r][c] = 0.0;
    M[c][c] = 1.0 / U[c][c];
    for (int r = c - 1; r >= 0; --r) {
      double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
      int k = r + 1;
      for (; k + 3 <= c; k += 4) {
        s0 = fma(U[r][k], M[k][c], s0);
        s1 = fma(U[r][k + 1], M[k + 1][c], s1);
        s2 = fma(U[r][k + 2], M[k + 2][c], s2);
        s3 = fma(U[r][k + 3], M[k + 3][c], s3);
      }
      for (; k <= c; ++k) s0 = fma(U[r][k], M[k][c], s0);
      M[r][c] = -((s0 + s1) + (s2 + s3)) / U[r][r];
    }
  }
}

// CholeskyQR + Householder reconstruction of one panel's kBand x kBand quantities (see the file header).
//   part / nslab : partial Gram matrices P'P
//   Ptop         : top kBand x kBand block of the panel inside A (read: P1; written: V1 = L, unit lower)
//   AB, c0       : band storage and the panel's first column: receives R' = S R
//   Mout         : (U R)^-1, row-major Float32 (the rows of V below the top block are P2 * Mout)
__global__ void __launch_bounds__(256) k_panel_factor(const double* __restrict__ part, int nslab, float* Ptop, long long lda,
                                                      float* AB, int c0, float* Mout, int* fail) {
  extern __shared__ __align__(16) double sm[];
  Mat65 G = reinterpret_cast<Mat65>(sm);
  Mat65 X = G + B;
  Mat65 U = X + B;
  __shared__ double S[B], D0[B];
  __shared__ int bad;
  const int tid = (int)threadIdx.x;
  sum_parts(part, nslab, G);
  for (int e = tid; e < B * B; e += 256) {
    const int i = e % B, c = e / B;
    X[i][c] = (double)Ptop[i + (long long)c * lda];
  }
  if (tid == 0) bad = 0;
  __syncthreads();
  if (tid < B) D0[tid] = G[tid][tid];
  __syncthreads();
  // Cholesky G = R'R, R in the upper triangle of G
  for (int j = 0; j < B; ++j) {
    if (tid == 0) {
      double p = G[j][j];
      if (!(p > 1e-13 * D0[j]) || !(p > 0.0)) {
        bad = 1;
        p = D0[j] > 0.0 ? D0[j] : 1.0;
      }
      G[j][j] = sqrt(p);
    }
    __syncthreads();
    if (tid > j && tid < B) G[j][tid] /= G[j][j];
    __syncthreads();
    for (int e = tid; e < B * B; e += 256) {
      const int r = e / B, c = e % B;
      if (r > j && c >= r) G[r][c] -= G[j][r] * G[j][c];
    }
    __syncthreads();
  }
  // X = P1 R^-1
  for (int c = 0; c < B; ++c) {
    if (tid < B) X[tid][c] /= G[c][c];
    __syncthreads();
    for (int e = tid; e < B * B; e += 256) {
      const int i = e % B, c2 = e / B;
      if (c2 > c) X[i][c2] -= X[i][c] * G[c][c2];
    }
    __syncthreads();
  }
  // LU with signs: X - S = L U
  for (int j = 0; j < B; ++j) {
    if (tid == 0) {
      const double p = X[j][j];
      S[j] = p >= 0.0 ? -1.0 : 1.0;
      X[j][j] = p - S[j];
    }
    __syncthreads();
    if (tid > j && tid < B) X[tid][j] /= X[j][j];
    __syncthreads();
    for (int e = tid; e < B * B; e += 256) {
      const int i = e % B, c = e / B;
      if (i > j && c > j) X[i][c] -= X[i][j] * X[j][c];
    }
    __syncthreads();
  }
  // V1 = L (unit lower), R' = S R into the band, U R
  for (int e = tid; e < B * B; e += 256) {
    const int i = e % B, c = e / B;
    Ptop[i + (long long)c * lda] = i > c ? (float)X[i][c] : (i == c ? 1.f : 0.f);
    const int r = e / B, cc = e % B;
    if (r <= cc) {
      AB[(size_t)(c0 + cc) * kLdab + (B + r - cc)] = (float)(S[r] * G[r][cc]);
      double s = 0;
      for (int k = r; k <= cc; ++k) s = fma(X[r][k], G[k][cc], s);
      U[r][cc] = s;
    } else {
      U[r][cc] = 0.0;
    }
  }
  __syncthreads();
  invert_upper(U, X);   // X no longer needed: L is in global memory, U R is in U
  __syncthreads();
  for (int e = tid; e < B * B; e += 256) {
    const int r = e / B, c = e % B;
    Mout[e] = r <= c ? (float)X[r][c] : 0.f;
  }
  if (tid == 0 && bad) atomicExch(fail, 1);
}

// T (row-major Float32) of I - V T V' from the partial Gram matrices V'V
__global__ void __launch_bounds__(256) k_tfactor(const double* __restrict__ part, int nslab, float* Tout) {
  extern __shared__ __align__(16) double sm[];
  Mat65 G = reinterpret_cast<Mat65>(sm);
  Mat65 M = G + B;
  const int tid = (int)threadIdx.x;
  sum_parts(part, nslab, G);
  __syncthreads();
  for (int e = tid; e < B * B; e += 256) {
    const int r = e / B, c = e % B;
    if (r == c) G[r][c] *= 0.5;
    else if (r > c) G[r][c] = 0.0;
  }
  __syncthreads();
  invert_upper(G, M);
  __syncthreads();
  for (int e = tid; e < B * B; e += 256) {
    const int r = e / B, c = e % B;
    Tout[e] = r <= c ? (float)M[r][c] : 0.f;
  }
}

// S2 = T' (V'Z), symmetrised, row-major Float32
__global__ void __launch_bounds__(256) k_sfactor(const double* __restrict__ part, int nslab, const float* __restrict__ T,
                                                 float* Sout) {
  extern __shared__ __align__(16) double sm[];
  Mat65 G = reinterpret_cast<Mat65>(sm);
  Mat65 Tm = G + B;
  Mat65 S = Tm + B;
  const int tid = (int)threadIdx.x;
  sum_parts(part, nslab, G);
  for (int e = tid; e < B * B; e += 256) Tm[e / B][e % B] = (double)T[e];
  __syncthreads();
  for (int e = tid; e < B * B; e += 256) {
    const int a = e / B, c = e % B;
    double s = 0;
    for (int k = 0; k <= a; ++k) s = fma(Tm[k][a], G[k][c], s);
    S[a][c] = s;
  }
  __syncthreads();
  for (int e = tid; e < B * B; e += 256) {
    const int a = e / B, c = e % B;
    Sout[e] = (float)(0.5 * (S[a][c] + S[c][a]));
  }
}

// Out[c][i] = (Add ? Add[c][i] : 0) + alpha * sum_c' In[c'][i] * Mat[c'][c]   for the rows of the CTA's 128-row block.
// In/Out/Add: kBand vectors of `rows` entries (vector c at + c * ld); Mat: kBand x kBand row-major.  In-place use
// (Out == In or Out == Add) is safe: a CTA reads exactly the rows it writes and finishes reading first.
__global__ void __launch_bounds__(256, 2) k_panel_mul(const float* In, long long ldin, const float* __restrict__ Mat, float* Out,
                                                      long long ldout, int rows, float alpha, const float* Add, long long ldadd,
                                                      int transposed_out) {
  __shared__ __align__(16) float smem[tile::Smem<64>::floats];
  const int i0 = (int)blockIdx.x * tile::TM;
  tile::Acc<64> acc;
  acc.clear();
  tile::mac<64>(acc, tile::opnd(In + i0, ldin, 0, rows - i0, B), tile::opnd(Mat, B, 0, B, B), B, smem);
#pragma unroll
  for (int b = 0; b < 4; ++b) {
    const int c = tile::Acc<64>::col(b);
#pragma unroll
    for (int a = 0; a < 8; ++a) {
      const int i = i0 + tile::Acc<64>::row(a);
      if (i < rows) {
        float v = alpha * acc.v[a][b];
        if (Add) v += Add[(long long)c * ldadd + i];
        if (transposed_out) Out[(long long)i * ldout + c] = v;
        else Out[(long long)c * ldout + i] = v;
      }
    }
  }
}

// Ypart[s][c][i] = sum over k in chunk s of A22sym(i, k) * V[c][k]: the trailing matrix is read from its lower triangle
// (tiles left of the diagonal as stored, the diagonal tile mirrored element by element, tiles below the diagonal transposed),
// on the tensor-core tile engine ENG (1: three-term TF32, 2: split binary16)
template <int ENG>
__global__ void __launch_bounds__(256, 2) k_symm_tc(const float* __restrict__ A22, long long lda, int m, const float* __restrict__ V,
                                                    long long ldv, float* __restrict__ Ypart, long long ldy, int chunk) {
  __shared__ __align__(16) unsigned char smem[tile::SmemE<ENG, 64>::bytes];
  const int i0 = (int)blockIdx.x * tile::TM;
  const int ka = (int)blockIdx.y * chunk, kb = min(m, ka + chunk);
  tile::AccT<64> acc;
  acc.clear();
  const int mi = m - i0;
  {  // tiles left of the diagonal tile
    const int k1 = min(kb, i0);
    if (k1 > ka)
      tile::mac_e<ENG, 64, 0, 1>(acc, tile::opnd(A22 + i0 + (long long)ka * lda, lda, 0, mi, k1 - ka), tile::opnd(V + ka, ldv, 1, B, k1 - ka),
                       k1 - ka, smem);
  }
  if (ka <= i0 && i0 < kb) {  // the diagonal tile (chunk boundaries are multiples of the tile size)
    const int kl = min(tile::TM, mi);
    tile::mac_e<ENG, 64, 0, 1>(acc, tile::opnd(A22 + i0 + (long long)i0 * lda, lda, 2, mi, kl), tile::opnd(V + i0, ldv, 1, B, kl), kl, smem);
  }
  {  // tiles below the diagonal tile, read transposed
    const int k3 = max(ka, i0 + tile::TM);
    if (kb > k3)
      tile::mac_e<ENG, 64, 1, 1>(acc, tile::opnd(A22 + k3 + (long long)i0 * lda, lda, 1, mi, kb - k3), tile::opnd(V + k3, ldv, 1, B, kb - k3),
                       kb - k3, smem);
  }
  float* out = Ypart + (size_t)blockIdx.y * B * ldy;
#pragma unroll
  for (int nt = 0; nt < tile::AccT<64>::NTL; ++nt)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int i = i0 + tile::AccT<64>::row(mt, e), c = tile::AccT<64>::col(nt, e);
        if (i < m) out[(long long)c * ldy + i] = acc.v[mt][nt][e];
      }
}

__global__ void k_sum_parts(const float* __restrict__ part, int nparts, size_t stride, size_t n, float* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int p = 0; p < nparts; ++p) s += part[(size_t)p * stride + i];
  out[i] = s;
}

// A22 -= V W' + W V', lower triangle, one 128 x 128 tile per CTA, on the tensor-core tile engine ENG.  The tile is formed
// transposed (columns j of the trailing matrix on the rows of the accumulator, rows i on its columns), so a thread's two
// adjacent outputs are adjacent in memory.
template <int ENG>
__global__ void __launch_bounds__(256, 2) k_syr2k_tc(float* A22, long long lda, int m, const float* __restrict__ V, long long ldv,
                                                     const float* __restrict__ W, long long ldw, int mode) {
  __shared__ __align__(16) unsigned char smem[tile::SmemE<ENG, 128>::bytes];
  // mode 0: linear tile index -> (I, J), J <= I.  mode 1: the first tile column only (J = 0).  mode 2: everything else.
  const int t = (int)blockIdx.x;
  int I, J;
  if (mode == 1) {
    I = t;
    J = 0;
  } else {
    I = (int)((sqrtf(8.f * (float)t + 1.f) - 1.f) * 0.5f);
    while ((I + 1) * (I + 2) / 2 <= t) ++I;
    while (I * (I + 1) / 2 > t) --I;
    J = t - I * (I + 1) / 2;
    if (mode == 2) {
      ++I;
      ++J;
    }
  }
  const int i0 = I * tile::TM, j0 = J * tile::TM;
  tile::AccT<128> acc;
  acc.clear();
  tile::mac_e<ENG, 128, 0, 0>(acc, tile::opnd(W + j0, ldw, 0, m - j0, B), tile::opnd(V + i0, ldv, 0, m - i0, B), B, smem);
  tile::mac_e<ENG, 128, 0, 0>(acc, tile::opnd(V + j0, ldv, 0, m - j0, B), tile::opnd(W + i0, ldw, 0, m - i0, B), B, smem);
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int j = j0 + tile::AccT<128>::row(mt, 2 * h);
      if (j >= m) continue;
      float* col = A22 + (long long)j * lda;
#pragma unroll
      for (int nt = 0; nt < tile::AccT<128>::NTL; ++nt) {
        const int i = i0 + tile::AccT<128>::col(nt, 0);
        if (i + 1 < m && i >= j) {
          float2 c = *reinterpret_cast<float2*>(col + i);
          c.x -= acc.v[mt][nt][2 * h];
          c.y -= acc.v[mt][nt][2 * h + 1];
          *reinterpret_cast<float2*>(col + i) = c;
        } else {
          if (i < m && i >= j) col[i] -= acc.v[mt][nt][2 * h];
          if (i + 1 < m && i + 1 >= j) col[i + 1] -= acc.v[mt][nt][2 * h + 1];
        }
      }
    }
}

// the last, short panel (2 <= m < kBand rows): plain Householder QR of the m x kBand block, the two-sided update of the m x m
// trailing block and T, all in one CTA.  V is stored zero-padded to kBand columns (T likewise), so the back-transformation
// treats it like any other panel.
__global__ void __launch_bounds__(64) k_tail_panel(float* A, long long lda, int n, int c0, float* AB, float* Tout) {
  extern __shared__ __align__(16) double sm[];
  Mat65 P = reinterpret_cast<Mat65>(sm);   // m x kBand block
  Mat65 V = P + B;                         // m x (m - 1), zero-padded
  Mat65 C = V + B;                         // trailing m x m block, full symmetric
  Mat65 T = C + B;
  __shared__ double tau[B], w[B], vv[B];
  __shared__ double s_beta, s_dot;
  const int tid = (int)threadIdx.x;
  const int r0 = c0 + B, m = n - r0;
  for (int e = tid; e < B * B; e += 64) {
    const int i = e % B, c = e / B;
    P[i][c] = i < m ? (double)A[(r0 + i) + (long long)(c0 + c) * lda] : 0.0;
    V[i][c] = 0.0;
    T[i][c] = 0.0;
    double v = 0.0;
    if (i < m && c < m) v = i >= c ? (double)A[(r0 + i) + (long long)(r0 + c) * lda] : (double)A[(r0 + c) + (long long)(r0 + i) * lda];
    C[i][c] = v;
  }
  if (tid < B) tau[tid] = 0.0;
  __syncthreads();
  for (int j = 0; j + 1 < m; ++j) {
    if (tid == 0) {
      double xn = 0;
      for (int i = j + 1; i < m; ++i) xn += P[i][j] * P[i][j];
      const double alpha = P[j][j];
      if (xn == 0.0) {
        tau[j] = 0.0;
        s_beta = alpha;
        vv[j] = 1.0;
        for (int i = j + 1; i < m; ++i) vv[i] = 0.0;
      } else {
        const double beta = -copysign(sqrt(alpha * alpha + xn), alpha);
        tau[j] = (beta - alpha) / beta;
        const double sc = 1.0 / (alpha - beta);
        vv[j] = 1.0;
        for (int i = j + 1; i < m; ++i) vv[i] = P[i][j] * sc;
        s_beta = beta;
      }
    }
    __syncthreads();
    // apply H_j to the block from the left: columns j+1.., thread per column
    if (tid > j) {
      double s = 0;
      for (int i = j; i < m; ++i) s += vv[i] * P[i][tid];
      s *= tau[j];
      for (int i = j; i < m; ++i) P[i][tid] -= vv[i] * s;
    }
    if (tid == j) {
      P[j][j] = s_beta;
      for (int i = j + 1; i < m; ++i) P[i][j] = 0.0;
    }
    if (tid >= j && tid < m) V[tid][j] = vv[tid];
    __syncthreads();
    // two-sided update of the trailing block with H_j (acts on its rows/columns j..m-1)
    if (tid < m) {
      double s = 0;
      for (int i = j; i < m; ++i) s += C[tid][i] * vv[i];
      w[tid] = tau[j] * s;
    }
    __syncthreads();
    if (tid == 0) {
      double s = 0;
      for (int i = j; i < m; ++i) s += w[i] * vv[i];
      s_dot = s;
    }
    __syncthreads();
    if (tid < m) {
      const double vi = tid >= j ? vv[tid] : 0.0;
      w[tid] -= 0.5 * tau[j] * s_dot * vi;
    }
    __syncthreads();
    if (tid < m) {
      const double vi = tid >= j ? vv[tid] : 0.0;
      for (int c = 0; c < m; ++c) {
        const double vc = c >= j ? vv[c] : 0.0;
        C[tid][c] -= vi * w[c] + w[tid] * vc;
      }
    }
    __syncthreads();
  }
  // T: forward columnwise larft
  for (int j = 0; j + 1 < m; ++j) {
    if (tid < j) {
      double s = 0;
      for (int i = j; i < m; ++i) s += V[i][tid] * V[i][j];
      w[tid] = s;
    }
    __syncthreads();
    if (tid < j) {
      double s = 0;
      for (int k = tid; k < j; ++k) s += T[tid][k] * w[k];
      T[tid][j] = -tau[j] * s;
    }
    if (tid == j) T[j][j] = tau[j];
    __syncthreads();
  }
  for (int e = tid; e < B * B; e += 64) {
    const int i = e % B, c = e / B;
    if (i < m) {
      A[(r0 + i) + (long long)(c0 + c) * lda] = (float)V[i][c];
      if (i <= c) AB[(size_t)(c0 + c) * kLdab + (B + i - c)] = (float)P[i][c];
      if (c < m && i >= c) A[(r0 + i) + (long long)(r0 + c) * lda] = (float)C[i][c];
    }
    Tout[e] = (float)T[e / B][e % B];
  }
  __syncthreads();
  // V T, transposed into the upper triangle of A like every other panel's
  for (int e = tid; e < B * B; e += 64) {
    const int i = e / B, c = e % B;
    if (i < m) {
      double s = 0;
      for (int k = 0; k <= c; ++k) s += V[i][k] * T[k][c];
      A[(c0 + c) + (long long)(r0 + i) * lda] = (float)s;
    }
  }
}

// diagonal blocks of the reduced matrix -> band storage (the sub-diagonal blocks were written by the panel kernels)
__global__ void k_extract_band(const float* __restrict__ A, long long lda, int n, int npanels, float* __restrict__ AB) {
  const int j = (int)blockIdx.x;
  const int kb = j / B, c0 = kb * B;
  const int last = kb < npanels ? min(n - 1, c0 + B - 1) : min(n - 1, j + B);
  for (int i = j + (int)threadIdx.x; i <= last; i += (int)blockDim.x) AB[(size_t)j * kLdab + (i - j)] = A[i + (long long)j * lda];
}

}  // namespace

namespace {
__global__ void __launch_bounds__(256) k_frob2(const float* __restrict__ A, int n, long long lda, double* __restrict__ out) {
  double s = 0.0;
  for (int c = (int)blockIdx.x; c < n; c += (int)gridDim.x) {
    const float* col = A + (long long)c * lda;
    for (int i = (int)threadIdx.x; i < n; i += 256) s += (double)col[i] * (double)col[i];
  }
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  __shared__ double ws[8];
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int w = 0; w < 8; ++w) t += ws[w];
    atomicAdd(out, t);
  }
}
}  // namespace

// May stage 1 multiply in split binary16?  Every quantity it forms is bounded by a small multiple of the Frobenius norm (an
// invariant of the reduction), so the norm must stay clear of binary16's overflow; and the absolute floor of the split
// (1.5e-11 per entry) must stay below FP32 rounding of the matrix as a whole.  One pass over the matrix and one synchronisation.
bool half_range_ok(const float* A, int n, long long lda, cudaStream_t st) {
  Tmp<double> acc(1, st);
  SCL_CUDA(cudaMemsetAsync(acc.p, 0, sizeof(double), st));
  k_frob2<<<std::min(n, 4 * sm_count()), 256, 0, st>>>(A, n, lda, acc.p);
  double f2 = 0.0;
  SCL_CUDA(cudaMemcpyAsync(&f2, acc.p, sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  count_launches(1);
  const double f = std::sqrt(f2);
  return std::isfinite(f) && f <= 1024.0 && f >= (double)n / 8192.0;
}

int sy2sb_lower(float* A, int n, long long lda, float* AB, float* T1, int* d_fail, cudaStream_t st, const Sy2sbAux* aux, bool half_ok) {
  SCL_REQUIRE((lda & 3) == 0 && ((uintptr_t)A & 15) == 0 && lda >= n, "sy2sb: leading dimension must be a multiple of 4");
  const long long ldy = ((long long)n + 3) & ~3LL;
  const int max_slabs = (n + kSlab - 1) / kSlab + 1;
  const int max_split = 16;
  Tmp<double> part((size_t)max_slabs * B * B, st), psum((size_t)B * B, st);
  Tmp<float> Mbuf(B * B, st), Sbuf(B * B, st), Ypart((size_t)max_split * B * ldy, st), Y((size_t)B * ldy, st), Z((size_t)B * ldy, st);
  SCL_CUDA(cudaMemsetAsync(AB, 0, (size_t)n * kLdab * sizeof(float), st));
  const size_t sm3 = 3 * B * (B + 1) * sizeof(double), sm2 = 2 * B * (B + 1) * sizeof(double), sm4 = 4 * B * (B + 1) * sizeof(double);
  static bool attr_done = false;
  if (!attr_done) {
    SCL_CUDA(cudaFuncSetAttribute(k_panel_factor, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm3));
    SCL_CUDA(cudaFuncSetAttribute(k_tfactor, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2));
    SCL_CUDA(cudaFuncSetAttribute(k_sfactor, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm3));
    SCL_CUDA(cudaFuncSetAttribute(k_tail_panel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm4));
    attr_done = true;
  }
  const int slots = 2 * sm_count();
  const int eng = half_ok ? 2 : 1;   // split binary16 only for a matrix within its range
  long launches = 0;
  // factorisation of panel k (full-size panels only) on stream s: V in place, T, V T into the upper triangle, R' into the band
  auto factor = [&](int k, cudaStream_t s) {
    const int c0 = k * B, r0 = c0 + B, m = n - r0;
    float* Pp = A + r0 + (long long)c0 * lda;
    float* Tk = T1 + (size_t)k * B * B;
    const int nslab = (m + kSlab - 1) / kSlab, ntile = (m + tile::TM - 1) / tile::TM;
    k_dot64<true><<<nslab, 256, 0, s>>>(Pp, lda, Pp, lda, m, kSlab, part.p);
    k_sum_dparts<<<B * B / 256, 256, 0, s>>>(part.p, nslab, psum.p);
    k_panel_factor<<<1, 256, sm3, s>>>(psum.p, 1, Pp, lda, AB, c0, Mbuf.p, d_fail);
    if (m > B) {
      const int nt2 = (m - B + tile::TM - 1) / tile::TM;
      k_panel_mul<<<nt2, 256, 0, s>>>(Pp + B, lda, Mbuf.p, Pp + B, lda, m - B, 1.f, nullptr, 0, 0);
    }
    k_dot64<false><<<nslab, 256, 0, s>>>(Pp, lda, Pp, lda, m, kSlab, part.p);
    k_sum_dparts<<<B * B / 256, 256, 0, s>>>(part.p, nslab, psum.p);
    k_tfactor<<<1, 256, sm2, s>>>(psum.p, 1, Tk);
    // V T for the back-transformation, transposed into the (otherwise unused) upper triangle of A: (V T)[i][c] at A(c0 + c, r0 + i)
    k_panel_mul<<<ntile, 256, 0, s>>>(Pp, lda, Tk, A + c0 + (long long)r0 * lda, lda, m, 1.f, nullptr, 0, 1);
    launches += 8;
  };
  int k = 0;
  bool factored = false;   // panel k was factored ahead (look-ahead) and the main stream already waits for it
  for (;; ++k) {
    const int c0 = k * B, r0 = c0 + B, m = n - r0;
    if (m <= 1) break;
    float* Pp = A + r0 + (long long)c0 * lda;        // the panel = V afterwards: vector c at Pp + c * lda
    float* A22 = A + r0 + (long long)r0 * lda;
    float* Tk = T1 + (size_t)k * B * B;
    if (m < B) {
      k_tail_panel<<<1, 64, sm4, st>>>(A, lda, n, c0, AB, Tk);
      ++launches;
      ++k;
      break;
    }
    const int nslab = (m + kSlab - 1) / kSlab;
    const int ntile = (m + tile::TM - 1) / tile::TM;
    if (!factored) factor(k, st);
    factored = false;
    // Y = A22 V, split over the contraction so that the grid covers the SMs several times over
    int split = std::max(1, std::min(max_split, (4 * slots + ntile - 1) / ntile));
    int chunk = ((m + split - 1) / split + tile::TM - 1) / tile::TM * tile::TM;
    chunk = std::max(chunk, 2 * tile::TM);
    split = (m + chunk - 1) / chunk;
    if (eng == 2) k_symm_tc<2><<<dim3(ntile, split), 256, 0, st>>>(A22, lda, m, Pp, lda, Ypart.p, ldy, chunk);
    else k_symm_tc<1><<<dim3(ntile, split), 256, 0, st>>>(A22, lda, m, Pp, lda, Ypart.p, ldy, chunk);
    const size_t ny = (size_t)B * ldy;
    k_sum_parts<<<(unsigned)((ny + 255) / 256), 256, 0, st>>>(Ypart.p, split, ny, ny, Y.p);
    k_panel_mul<<<ntile, 256, 0, st>>>(Y.p, ldy, Tk, Z.p, ldy, m, 1.f, nullptr, 0, 0);
    k_dot64<false><<<nslab, 256, 0, st>>>(Pp, lda, Z.p, ldy, m, kSlab, part.p);
    k_sum_dparts<<<B * B / 256, 256, 0, st>>>(part.p, nslab, psum.p);
    k_sfactor<<<1, 256, sm3, st>>>(psum.p, 1, Tk, Sbuf.p);
    k_panel_mul<<<ntile, 256, 0, st>>>(Pp, lda, Sbuf.p, Z.p, ldy, m, -0.5f, Z.p, ldy, 0);
    launches += 8;
    // look-ahead: the first tile column of the update holds the next panel; once it is done the next panel is factored on the
    // auxiliary stream (one or a few CTAs per kernel) while the main stream updates the rest of the trailing matrix
    const bool ahead = aux && aux->stream && ntile >= 4 && m - B >= B;
    if (ahead) {
      if (eng == 2) k_syr2k_tc<2><<<ntile, 256, 0, st>>>(A22, lda, m, Pp, lda, Z.p, ldy, 1);
      else k_syr2k_tc<1><<<ntile, 256, 0, st>>>(A22, lda, m, Pp, lda, Z.p, ldy, 1);
      SCL_CUDA(cudaEventRecord(aux->ready, st));
      SCL_CUDA(cudaStreamWaitEvent(aux->stream, aux->ready, 0));
      factor(k + 1, aux->stream);
      SCL_CUDA(cudaEventRecord(aux->done, aux->stream));
      if (eng == 2) k_syr2k_tc<2><<<(ntile - 1) * ntile / 2, 256, 0, st>>>(A22, lda, m, Pp, lda, Z.p, ldy, 2);
      else k_syr2k_tc<1><<<(ntile - 1) * ntile / 2, 256, 0, st>>>(A22, lda, m, Pp, lda, Z.p, ldy, 2);
      SCL_CUDA(cudaStreamWaitEvent(st, aux->done, 0));
      factored = true;
      ++launches;
    } else {
      if (eng == 2) k_syr2k_tc<2><<<ntile * (ntile + 1) / 2, 256, 0, st>>>(A22, lda, m, Pp, lda, Z.p, ldy, 0);
      else k_syr2k_tc<1><<<ntile * (ntile + 1) / 2, 256, 0, st>>>(A22, lda, m, Pp, lda, Z.p, ldy, 0);
    }
    ++launches;
  }
  k_extract_band<<<n, 64, 0, st>>>(A, lda, n, k, AB);
  SCL_CUDA(cudaGetLastError());
  count_launches((int)launches + 1);
  return k;
}

}  // namespace scl
