// apply_umap! (src/scLENS.jl:863-873, UMAP.jl 0.1.11 UMAP_) on the device: exact kNN, fuzzy simplicial set, spectral
// start and the SGD layout, for the N x r matrix :pca_n1 (r = number of robust signals, a handful).
//
// kNN.  r is a handful, so the pairwise distances are not a tcgen05 GEMM: a tensor-core tile would spend its K = 16
// slots on < 10 real dimensions, and binary16 operands would reorder near neighbours (distances agree only to ~1e-3).
// Each thread owns one query (held in registers), a CTA streams candidate tiles through shared memory (read as float4
// broadcasts) and computes squared distances in FP32 with fmaf; a candidate is inserted into the thread's sorted top-k
// only when it beats the current k-th, which after the first tiles almost never happens.  Order is lexicographic in
// (distance, index), so the result does not depend on how the candidates are tiled; at small N the candidate range is
// split across CTAs (grid.y) and the sorted partial lists are merged.  Cosine: rows normalised on the way in, distance
// 1/2 |x^ - y^|^2 (= 1 - cos, no cancellation for near-duplicates); a zero row is at distance 1 from everything.
//
// Graph.  smooth_knn_dists per row in Float64 (rho = local-connectivity distance, sigma by 64-step bisection), memberships
// w_ij, then the fuzzy union A + A^T - A o A^T as CSR with sorted columns: every row holds its own k neighbours (value
// combined with the reverse membership when the edge is mutual) plus the incoming edges that are not mutual; a warp
// ranks each row's distinct columns.  No FP atomics; the incoming slots are claimed with integer atomics and the rank
// pass makes the result independent of that order.
//
// Spectral start.  Top nc + 1 eigenvectors of S = D^-1/2 A D^-1/2 by a Chebyshev-filtered block iteration on a CSR x
// block SpMM; the known top vector D^1/2 1 / |.| is projected out of every product, so components of a disconnected
// graph (eigenvalue 1 repeated) are found like any other vector.  Gram products, Cholesky QR and the Rayleigh-Ritz
// rotations are the subspace.cu building blocks with fixed-order reductions.
//
// Layout.  One kernel per epoch, positions ping-pong between two buffers; a thread gathers everything that moves its
// vertex (own fired edges, their negative samples, the reverse draws of its incoming edges): no atomics, no races, the
// same seed gives the same bits.  Every draw is a counter-based hash of (seed, stream, epoch, vertex, slot).
#include <algorithm>
#include <cmath>
#include "handle.h"
#include "subspace.h"
#include "tmp.cuh"

namespace scl {

namespace {

constexpr int kQ = 128;          // queries per CTA (one per thread)
constexpr int kMaxK = 64;
constexpr int kMaxSplits = 32;
constexpr int kMaxNc = 16;

// ---- draws ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t draw_bits(uint64_t key, uint32_t vertex, uint32_t slot) {
  return mix64s(mix64s(key ^ (((uint64_t)vertex << 32) | slot)));
}
__device__ __forceinline__ float draw_unit(uint64_t key, uint32_t vertex, uint32_t slot) {
  return (float)(draw_bits(key, vertex, slot) >> 40) * (1.0f / 16777216.0f);
}

// ---- kNN -------------------------------------------------------------------------------------------------------------
// X column-major N x d -> Xr row-major [N][dp] (dp = d rounded up to 4, zero padded), cosine: unit rows, zero flags
__global__ void k_knn_prep(const float* __restrict__ X, int N, int d, int dp, int cosine, float* __restrict__ Xr,
                           uint8_t* __restrict__ zero) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  double s = 0;
  for (int t = 0; t < d; ++t) { const double v = X[(size_t)t * N + i]; s += v * v; }
  const double inv = (cosine && s > 0) ? 1.0 / sqrt(s) : 1.0;
  for (int t = 0; t < dp; ++t) Xr[(size_t)i * dp + t] = t < d ? (float)(X[(size_t)t * N + i] * inv) : 0.f;
  if (zero) zero[i] = s > 0 ? 0 : 1;
}

__device__ __forceinline__ bool lex_less(float da, int ia, float db, int ib) { return da < db || (da == db && ia < ib); }

// DR > 0: query in DR registers (dp <= DR); DR == 0: query in shared memory [dp][kQ]
template <int DR>
__global__ void __launch_bounds__(kQ) k_knn(const float* __restrict__ Xr, const uint8_t* __restrict__ zero, int N, int dp,
                                            int k, int tile, int per_split, float* __restrict__ pd, int* __restrict__ pi) {
  extern __shared__ float4 sm4[];
  float* sc = reinterpret_cast<float*>(sm4);                 // [tile][dp]
  uint8_t* sz = reinterpret_cast<uint8_t*>(sc + (size_t)tile * dp);   // [tile]
  float* sq = sc + (size_t)tile * dp + (tile + 3) / 4;       // DR == 0: [dp][kQ]
  const int tid = threadIdx.x;
  const int qi = blockIdx.x * kQ + tid;
  const bool live = qi < N;
  float q[DR > 0 ? DR : 1];
  if constexpr (DR > 0) {
#pragma unroll
    for (int t = 0; t < DR; ++t) q[t] = (live && t < dp) ? Xr[(size_t)qi * dp + t] : 0.f;
  } else {
    for (int t = 0; t < dp; ++t) sq[t * kQ + tid] = live ? Xr[(size_t)qi * dp + t] : 0.f;
  }
  const bool qzero = zero && live && zero[qi];
  float bd[kMaxK];
  int bi[kMaxK];
  int cnt = 0;
  float kd = INFINITY;
  int ki = 0x7fffffff;
  const int c0 = blockIdx.y * per_split, c1 = min(N, c0 + per_split);
  for (int base = c0; base < c1; base += tile) {
    const int tl = min(tile, c1 - base);
    __syncthreads();
    const float4* src = reinterpret_cast<const float4*>(Xr + (size_t)base * dp);
    for (int e = tid; e < tl * dp / 4; e += kQ) sm4[e] = src[e];
    if (zero)
      for (int e = tid; e < tl; e += kQ) sz[e] = zero[base + e];
    __syncthreads();
    if (!live) continue;
    for (int c = 0; c < tl; ++c) {
      const int j = base + c;
      const float* cv = sc + (size_t)c * dp;
      float acc = 0.f;
      if constexpr (DR > 0) {
#pragma unroll
        for (int t = 0; t < DR; t += 4) {
          if (t < dp) {
            const float4 v = *reinterpret_cast<const float4*>(cv + t);
            float e0 = q[t] - v.x, e1 = q[t + 1] - v.y, e2 = q[t + 2] - v.z, e3 = q[t + 3] - v.w;
            acc = fmaf(e0, e0, acc); acc = fmaf(e1, e1, acc); acc = fmaf(e2, e2, acc); acc = fmaf(e3, e3, acc);
          }
        }
      } else {
        for (int t = 0; t < dp; t += 4) {
          const float4 v = *reinterpret_cast<const float4*>(cv + t);
          float e0 = sq[t * kQ + tid] - v.x, e1 = sq[(t + 1) * kQ + tid] - v.y, e2 = sq[(t + 2) * kQ + tid] - v.z,
                e3 = sq[(t + 3) * kQ + tid] - v.w;
          acc = fmaf(e0, e0, acc); acc = fmaf(e1, e1, acc); acc = fmaf(e2, e2, acc); acc = fmaf(e3, e3, acc);
        }
      }
      if (zero && (qzero || sz[c])) acc = 2.f;   // cosine distance 1 (= acc / 2)
      if (j == qi) continue;
      if (cnt < k || lex_less(acc, j, kd, ki)) {
        int p = cnt < k ? cnt++ : k - 1;
        while (p > 0 && lex_less(acc, j, bd[p - 1], bi[p - 1])) { bd[p] = bd[p - 1]; bi[p] = bi[p - 1]; --p; }
        bd[p] = acc; bi[p] = j;
        if (cnt == k) { kd = bd[k - 1]; ki = bi[k - 1]; }
      }
    }
  }
  if (!live) return;
  const size_t o = ((size_t)blockIdx.y * N + qi) * k;
  for (int s = 0; s < k; ++s) {
    pd[o + s] = s < cnt ? bd[s] : INFINITY;
    pi[o + s] = s < cnt ? bi[s] : 0x7fffffff;
  }
}

// merge the sorted per-split lists [S][N][k] of squared distances; final distance sqrt (euclidean) or half (cosine)
__global__ void k_knn_merge(const float* __restrict__ pd, const int* __restrict__ pi, int N, int k, int S, int cosine,
                            int32_t* __restrict__ idx, float* __restrict__ dist) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  int head[kMaxSplits];
  for (int s = 0; s < S; ++s) head[s] = 0;
  for (int o = 0; o < k; ++o) {
    int best = 0;
    float bdv = INFINITY;
    int biv = 0x7fffffff;
    for (int s = 0; s < S; ++s) {
      if (head[s] >= k) continue;
      const size_t e = ((size_t)s * N + i) * k + head[s];
      if (lex_less(pd[e], pi[e], bdv, biv)) { bdv = pd[e]; biv = pi[e]; best = s; }
    }
    ++head[best];
    idx[(size_t)i * k + o] = biv;
    dist[(size_t)i * k + o] = cosine ? 0.5f * bdv : sqrtf(bdv);
  }
}

// ---- fuzzy graph -----------------------------------------------------------------------------------------------------
// smooth_knn_dists + memberships: w[i][s] = exp(-max(0, d_is - rho_i) / sigma_i)   (Float64)
__global__ void k_smooth_knn(const float* __restrict__ dist, int N, int k, double local_connectivity, double* __restrict__ w) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const float* d = dist + (size_t)i * k;
  // rho: the local_connectivity-th smallest non-zero distance, interpolated (local_connectivity = 1: the first)
  int nz0 = 0;
  while (nz0 < k && !(d[nz0] > 0.f)) ++nz0;
  const int nnz = k - nz0;
  double rho = 0;
  const int index = (int)floor(local_connectivity);
  const double interp = local_connectivity - index;
  if (nnz >= local_connectivity) {
    if (index > 0) {
      rho = d[nz0 + index - 1];
      if (interp > 1e-5) rho += interp * ((double)d[nz0 + index] - d[nz0 + index - 1]);
    } else {
      rho = interp * d[nz0];
    }
  } else if (nnz > 0) {
    rho = d[k - 1];
  }
  const double target = log2((double)k);
  double lo = 0, mid = 1, hi = INFINITY;
  for (int it = 0; it < 64; ++it) {
    double psum = 0;
    for (int s = 0; s < k; ++s) psum += exp(-fmax((double)d[s] - rho, 0.0) / mid);
    if (fabs(psum - target) < 1e-5) break;
    if (psum > target) {
      hi = mid;
      mid = (lo + hi) / 2;
    } else {
      lo = mid;
      mid = isinf(hi) ? mid * 2 : (lo + hi) / 2;
    }
  }
  for (int s = 0; s < k; ++s) w[(size_t)i * k + s] = exp(-fmax((double)d[s] - rho, 0.0) / mid);
}

__device__ __forceinline__ int find_in_row(const int32_t* __restrict__ knn, int k, int row, int v) {
  for (int t = 0; t < k; ++t)
    if (knn[(size_t)row * k + t] == v) return t;
  return -1;
}

// row lengths: k own entries + incoming edges that are not mutual
__global__ void k_union_count(const int32_t* __restrict__ knn, int N, int k, uint32_t* __restrict__ cnt) {
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= (size_t)N * k) return;
  const int i = (int)(e / k), j = knn[e];
  if (find_in_row(knn, k, j, i) < 0) atomicAdd(&cnt[j], 1u);
}

__global__ void k_union_fill(const int32_t* __restrict__ knn, const double* __restrict__ w, int N, int k,
                             const uint32_t* __restrict__ ptr, uint32_t* __restrict__ cursor, uint32_t* __restrict__ tcol,
                             double* __restrict__ tval) {
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= (size_t)N * k) return;
  const int i = (int)(e / k), s = (int)(e % k), j = knn[e];
  const double a = w[e];
  const int t = find_in_row(knn, k, j, i);
  const double b = t >= 0 ? w[(size_t)j * k + t] : 0.0;
  tcol[ptr[i] + s] = (uint32_t)j;
  tval[ptr[i] + s] = a + b - a * b;
  if (t < 0) {
    const uint32_t slot = ptr[j] + k + atomicAdd(&cursor[j], 1u);
    tcol[slot] = (uint32_t)i;
    tval[slot] = a;
  }
}

// one warp per row: the distinct columns of the row ranked into ascending order
__global__ void k_union_sort(const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ tcol, const double* __restrict__ tval,
                             int N, uint32_t* __restrict__ col, float* __restrict__ val) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= N) return;
  const uint32_t b = ptr[warp], L = ptr[warp + 1] - b;
  for (uint32_t t = lane; t < L; t += 32) {
    const uint32_t c = tcol[b + t];
    uint32_t rank = 0;
    for (uint32_t u = 0; u < L; ++u) rank += tcol[b + u] < c;
    col[b + rank] = c;
    val[b + rank] = (float)tval[b + t];
  }
}

// position of the reverse edge (j, i) of every stored (i, j); degrees D_i (Float64, fixed order)
__global__ void k_graph_aux(const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ col, const float* __restrict__ val,
                            int N, uint32_t* __restrict__ rev, double* __restrict__ deg) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  double s = 0;
  for (uint32_t e = ptr[i]; e < ptr[i + 1]; ++e) {
    const uint32_t j = col[e];
    uint32_t lo = ptr[j], hi = ptr[j + 1];
    while (lo < hi) {
      const uint32_t m = (lo + hi) / 2;
      if (col[m] < (uint32_t)i) lo = m + 1; else hi = m;
    }
    rev[e] = lo;
    s += val[e];
  }
  deg[i] = s;
}

// ---- spectral start --------------------------------------------------------------------------------------------------
// S values (A_ij / sqrt(D_i D_j)) and the known top eigenvector v0 = D^1/2 1 / |D^1/2 1|
__global__ void k_norm_graph(const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ col, const float* __restrict__ val,
                             const double* __restrict__ deg, double inv_norm, int N, float* __restrict__ sval, float* __restrict__ v0) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const double di = deg[i] > 0 ? 1.0 / sqrt(deg[i]) : 0.0;
  for (uint32_t e = ptr[i]; e < ptr[i + 1]; ++e) {
    const double dj = deg[col[e]] > 0 ? 1.0 / sqrt(deg[col[e]]) : 0.0;
    sval[e] = (float)((double)val[e] * di * dj);
  }
  v0[i] = (float)(sqrt(deg[i]) * inv_norm);
}

// CSR x block: Y[c][i] = s1 * ((S X)[c][i] - cshift * X[c][i]) - s2 * Xp[c][i]   (Xp may be null)
__global__ void k_spmm(const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ col, const float* __restrict__ sval, int N,
                       int b, const float* __restrict__ X, float cshift, float s1, float s2, const float* __restrict__ Xp,
                       float* __restrict__ Y) {
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= (size_t)N * b) return;
  const int c = (int)(e / N), i = (int)(e % N);
  const float* x = X + (size_t)c * N;
  float acc = 0.f;
  for (uint32_t t = ptr[i]; t < ptr[i + 1]; ++t) acc = fmaf(sval[t], x[col[t]], acc);
  float y = s1 * (acc - cshift * x[i]);
  if (Xp) y -= s2 * Xp[e];
  Y[e] = y;
}

__global__ void k_start_from_block(const float* __restrict__ Q, int N, int nc, float scale, uint64_t key_noise,
                                   float* __restrict__ P) {
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= (size_t)N * nc) return;
  const int i = (int)(e / nc), c = (int)(e % nc);
  const uint64_t h1 = draw_bits(key_noise, i, 2 * c), h2 = draw_bits(key_noise, i, 2 * c + 1);
  const double u1 = ((double)(h1 >> 40) + 1.0) * (1.0 / 16777217.0), u2 = (double)(h2 >> 40) * (1.0 / 16777216.0);
  const double g = sqrt(-2.0 * log(u1)) * cos(2.0 * M_PI * u2);
  P[e] = (float)((double)Q[(size_t)c * N + i] * scale + 1e-4 * g);
}

__global__ void k_random_start(int N, int nc, uint64_t key, float* __restrict__ P) {
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= (size_t)N * nc) return;
  const int i = (int)(e / nc), c = (int)(e % nc);
  P[e] = (float)((double)(draw_bits(key, i, c) >> 40) * (1.0 / 16777216.0) * 20.0 - 10.0);
}

// ---- layout ----------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float clip4(float v) { return fminf(4.f, fmaxf(-4.f, v)); }

__global__ void __launch_bounds__(128) k_layout_epoch(const uint32_t* __restrict__ ptr, const uint32_t* __restrict__ col,
                                                      const float* __restrict__ pval, const uint32_t* __restrict__ rev, int N,
                                                      int nc, const float* __restrict__ P, float* __restrict__ Pn,
                                                      uint64_t key_fire, uint64_t key_neg, float alpha, float a, float b,
                                                      float gamma, int neg_rate) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  float xi[kMaxNc], g[kMaxNc];
#pragma unroll
  for (int c = 0; c < kMaxNc; ++c) { xi[c] = c < nc ? P[(size_t)i * nc + c] : 0.f; g[c] = 0.f; }
  const uint32_t rb = ptr[i], re = ptr[i + 1];
  for (uint32_t e = rb; e < re; ++e) {
    const uint32_t j = col[e], r = rev[e];
    const bool f1 = draw_unit(key_fire, i, e - rb) <= pval[e];
    const bool f2 = draw_unit(key_fire, j, r - ptr[j]) <= pval[r];
    if (!f1 && !f2) continue;
    float xj[kMaxNc];
    float sd = 0.f;
#pragma unroll
    for (int c = 0; c < kMaxNc; ++c) {
      xj[c] = c < nc ? P[(size_t)j * nc + c] : 0.f;
      const float df = xi[c] - xj[c];
      sd = fmaf(df, df, sd);
    }
    const float delta = sd > 0.f ? (-2.f * a * b * powf(sd, b - 1.f)) / (1.f + a * powf(sd, b)) : 0.f;
    if (f1) {
#pragma unroll
      for (int c = 0; c < kMaxNc; ++c) g[c] += clip4(delta * (xi[c] - xj[c]));
      for (int t = 0; t < neg_rate; ++t) {
        const uint64_t h = draw_bits(key_neg, i, (e - rb) * (uint32_t)neg_rate + t);
        const int kk = (int)(((h >> 32) * (uint64_t)N) >> 32);
        if (kk == i) continue;
        float xk[kMaxNc];
        float sk = 0.f;
#pragma unroll
        for (int c = 0; c < kMaxNc; ++c) {
          xk[c] = c < nc ? P[(size_t)kk * nc + c] : 0.f;
          const float df = xi[c] - xk[c];
          sk = fmaf(df, df, sk);
        }
        const float dn = sk > 0.f ? (2.f * gamma * b) / ((1e-3f + sk) * (1.f + a * powf(sk, b))) : 0.f;
#pragma unroll
        for (int c = 0; c < kMaxNc; ++c) g[c] += dn > 0.f ? clip4(dn * (xi[c] - xk[c])) : 4.f;
      }
    }
    if (f2) {
#pragma unroll
      for (int c = 0; c < kMaxNc; ++c) g[c] -= clip4(delta * (xj[c] - xi[c]));
    }
  }
  for (int c = 0; c < nc; ++c) Pn[(size_t)i * nc + c] = xi[c] + alpha * g[c];
}

__global__ void k_to_colmajor(const float* __restrict__ P, int N, int nc, float* __restrict__ out) {
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= (size_t)N * nc) return;
  const int c = (int)(e / N), i = (int)(e % N);
  out[e] = P[(size_t)i * nc + c];
}

__global__ void k_from_colmajor(const float* __restrict__ in, int N, int nc, float* __restrict__ P) {
  const size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (e >= (size_t)N * nc) return;
  const int c = (int)(e / N), i = (int)(e % N);
  P[(size_t)i * nc + c] = in[e];
}

inline int blocks(size_t n, int t) { return (int)((n + t - 1) / t); }

// cyclic Jacobi on a small symmetric matrix (row-major b x b); eigenvalues descending, V row c = eigenvector c
void jacobi_desc(std::vector<double> A, int b, std::vector<double>& w, std::vector<double>& V) {
  std::vector<double> E((size_t)b * b, 0.0);
  for (int i = 0; i < b; ++i) E[(size_t)i * b + i] = 1.0;
  for (int sweep = 0; sweep < 100; ++sweep) {
    double off = 0, tot = 0;
    for (int p = 0; p < b; ++p)
      for (int q = 0; q < b; ++q) (p == q ? tot : off) += A[(size_t)p * b + q] * A[(size_t)p * b + q];
    if (off <= 1e-30 * (tot + off) || off == 0) break;
    for (int p = 0; p < b - 1; ++p)
      for (int q = p + 1; q < b; ++q) {
        const double apq = A[(size_t)p * b + q];
        if (apq == 0) continue;
        const double th = (A[(size_t)q * b + q] - A[(size_t)p * b + p]) / (2 * apq);
        const double t = (th >= 0 ? 1.0 : -1.0) / (std::fabs(th) + std::sqrt(th * th + 1));
        const double cs = 1 / std::sqrt(t * t + 1), sn = t * cs;
        for (int k = 0; k < b; ++k) {   // columns p, q
          const double akp = A[(size_t)k * b + p], akq = A[(size_t)k * b + q];
          A[(size_t)k * b + p] = cs * akp - sn * akq;
          A[(size_t)k * b + q] = sn * akp + cs * akq;
        }
        for (int k = 0; k < b; ++k) {   // rows p, q
          const double apk = A[(size_t)p * b + k], aqk = A[(size_t)q * b + k];
          A[(size_t)p * b + k] = cs * apk - sn * aqk;
          A[(size_t)q * b + k] = sn * apk + cs * aqk;
        }
        for (int k = 0; k < b; ++k) {   // eigenvector rows
          const double ep = E[(size_t)p * b + k], eq = E[(size_t)q * b + k];
          E[(size_t)p * b + k] = cs * ep - sn * eq;
          E[(size_t)q * b + k] = sn * ep + cs * eq;
        }
      }
  }
  std::vector<int> ord(b);
  for (int i = 0; i < b; ++i) ord[i] = i;
  std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return A[(size_t)x * b + x] > A[(size_t)y * b + y]; });
  w.resize(b);
  V.resize((size_t)b * b);
  for (int c = 0; c < b; ++c) {
    w[c] = A[(size_t)ord[c] * b + ord[c]];
    std::copy(E.begin() + (size_t)ord[c] * b, E.begin() + (size_t)(ord[c] + 1) * b, V.begin() + (size_t)c * b);
  }
}

struct StageTimer {
  cudaEvent_t a, b;
  cudaStream_t st;
  explicit StageTimer(cudaStream_t s) : st(s) {
    SCL_CUDA(cudaEventCreate(&a));
    SCL_CUDA(cudaEventCreate(&b));
    SCL_CUDA(cudaEventRecord(a, st));
  }
  ~StageTimer() { cudaEventDestroy(a); cudaEventDestroy(b); }
  double stop() {
    SCL_CUDA(cudaEventRecord(b, st));
    SCL_CUDA(cudaEventSynchronize(b));
    float ms = 0;
    SCL_CUDA(cudaEventElapsedTime(&ms, a, b));
    SCL_CUDA(cudaEventRecord(a, st));
    return ms;
  }
};

}  // namespace

uint64_t umap_stream_key(uint64_t seed, uint32_t stream, uint32_t epoch) {
  return mix64s(mix64s(seed ^ (0x9e3779b97f4a7c15ull * (stream + 1ull))) ^ epoch);
}

// ---- host entry points -----------------------------------------------------------------------------------------------
void knn_device(const float* dX, int N, int d, int k, int metric, int32_t* d_idx, float* d_dist, cudaStream_t st) {
  SCL_REQUIRE(k >= 1 && k <= kMaxK && k < N, "kNN: need 1 <= k <= 64 and k < N");
  SCL_REQUIRE(d >= 1 && d <= 1024, "kNN: dimension out of range");
  const int dp = (d + 3) / 4 * 4;
  const bool cosine = metric == 1;
  Tmp<float> Xr((size_t)N * dp, st);
  Tmp<uint8_t> zf(cosine ? N : 1, st);
  k_knn_prep<<<blocks(N, 256), 256, 0, st>>>(dX, N, d, dp, cosine, Xr.p, cosine ? zf.p : nullptr);
  const int bx = (N + kQ - 1) / kQ;
  const int tile = dp <= 64 ? 128 : std::max(8, (32768 / (dp * 4)) / 4 * 4);
  int S = std::min(kMaxSplits, std::max(1, (2 * sm_count() + bx - 1) / bx));
  int per = (N + S - 1) / S;
  per = (per + tile - 1) / tile * tile;
  S = (N + per - 1) / per;
  Tmp<float> pd((size_t)S * N * k, st);
  Tmp<int> pi((size_t)S * N * k, st);
  const size_t smem = (size_t)tile * dp * 4 + (tile + 3) / 4 * 4 + (dp <= 64 ? 0 : (size_t)dp * kQ * 4);
  dim3 grid(bx, S);
  const uint8_t* z = cosine ? zf.p : nullptr;
#define SCL_KNN(DRV)                                                                                            \
  do {                                                                                                          \
    SCL_CUDA(cudaFuncSetAttribute(k_knn<DRV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));         \
    k_knn<DRV><<<grid, kQ, smem, st>>>(Xr.p, z, N, dp, k, tile, per, pd.p, pi.p);                               \
  } while (0)
  if (dp <= 8) SCL_KNN(8);
  else if (dp <= 16) SCL_KNN(16);
  else if (dp <= 32) SCL_KNN(32);
  else if (dp <= 64) SCL_KNN(64);
  else SCL_KNN(0);
#undef SCL_KNN
  k_knn_merge<<<blocks(N, 128), 128, 0, st>>>(pd.p, pi.p, N, k, S, cosine, d_idx, d_dist);
  count_launches(3);
  SCL_CUDA(cudaGetLastError());
}

// fuzzy union graph of the handle's kNN (h->uk_*) into h->ug_*
static void build_graph(scl_handle* h, int N, int k, double local_connectivity) {
  cudaStream_t st = h->st;
  Tmp<double> w((size_t)N * k, st);
  k_smooth_knn<<<blocks(N, 128), 128, 0, st>>>(h->uk_dist.p, N, k, local_connectivity, w.p);
  Tmp<uint32_t> cnt(N + 1, st), tptr(N + 1, st), cursor(N + 1, st);
  SCL_CUDA(cudaMemsetAsync(cursor.p, 0, (N + 1) * sizeof(uint32_t), st));
  std::vector<uint32_t> kk(N, (uint32_t)k);
  SCL_CUDA(cudaMemcpyAsync(cnt.p, kk.data(), N * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  const size_t Nk = (size_t)N * k;
  k_union_count<<<blocks(Nk, 256), 256, 0, st>>>(h->uk_idx.p, N, k, cnt.p);
  exclusive_scan(cnt.p, tptr.p, N, st);
  uint32_t nnz = 0;
  SCL_CUDA(cudaMemcpyAsync(&nnz, tptr.p + N, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  Tmp<uint32_t> tcol(nnz, st);
  Tmp<double> tval(nnz, st);
  k_union_fill<<<blocks(Nk, 256), 256, 0, st>>>(h->uk_idx.p, w.p, N, k, tptr.p, cursor.p, tcol.p, tval.p);
  h->ug_rowptr.ensure(N + 1);
  h->ug_col.ensure(nnz);
  h->ug_val.ensure(nnz);
  h->ug_rev.ensure(nnz);
  h->ug_deg.ensure(N);
  SCL_CUDA(cudaMemcpyAsync(h->ug_rowptr.p, tptr.p, (N + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
  k_union_sort<<<blocks((size_t)N * 32, 256), 256, 0, st>>>(tptr.p, tcol.p, tval.p, N, h->ug_col.p, h->ug_val.p);
  k_graph_aux<<<blocks(N, 128), 128, 0, st>>>(h->ug_rowptr.p, h->ug_col.p, h->ug_val.p, N, h->ug_rev.p, h->ug_deg.p);
  count_launches(6);
  SCL_CUDA(cudaGetLastError());
  h->ug_nnz = nnz;
  h->ug_N = N;
  h->have_umap_graph = true;
}

// eigenvectors 2..nc+1 of the normalised Laplacian, scaled to max 10 plus 1e-4 N(0,1) noise, into P [N][nc];
// false when the iteration did not converge in maxiter outer iterations
static bool spectral_start(scl_handle* h, int N, int nc, int maxiter, uint64_t seed, float* P, int* iters) {
  cudaStream_t st = h->st;
  const int b = std::min(nc + 8, N - 1);
  *iters = 0;
  if (b < nc || N < 3) return false;
  const uint32_t* ptr = h->ug_rowptr.p;
  const uint32_t* col = h->ug_col.p;
  Tmp<float> sval(std::max<size_t>(h->ug_nnz, 1), st), v0(N, st);
  std::vector<double> deg(N);
  SCL_CUDA(cudaMemcpyAsync(deg.data(), h->ug_deg.p, N * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  double tot = 0;
  for (double x : deg) tot += x;
  if (!(tot > 0)) return false;
  k_norm_graph<<<blocks(N, 128), 128, 0, st>>>(ptr, col, h->ug_val.p, h->ug_deg.p, 1.0 / std::sqrt(tot), N, sval.p, v0.p);
  BlockCtx c{h, st, N, (size_t)N, nullptr, nullptr, true};
  const size_t bn = (size_t)b * N;
  Tmp<float> Q(bn, st), Z(bn, st), Y0(bn, st), Y1(bn, st), Y2(bn, st);
  Tmp<double> dC(b, st), dH((size_t)b * b, st), dTt((size_t)b * b, st), dTheta(b, st), dRes(b, st);
  k_random_start<<<blocks(bn, 256), 256, 0, st>>>(b, N, umap_stream_key(seed, 5, 0), Q.p);   // [b][N] in [-10, 10]
  auto deflate = [&](float* Y) {      // Y -= (Y v0) v0^T
    gram_ts(c, Y, b, v0.p, 1, dC.p);
    combine_rows(c, v0.p, 1, dC.p, b, -1.0, Y, 1.0, Y);
  };
  auto spmm = [&](const float* X, float cs, float s1, float s2, const float* Xp, float* Y) {
    k_spmm<<<blocks(bn, 256), 256, 0, st>>>(ptr, col, sval.p, N, b, X, cs, s1, s2, Xp, Y);
    count_launches(1);
  };
  deflate(Q.p);
  chol_qr(c, Q.p, b, Z.p, 2);
  std::vector<double> H((size_t)b * b), w, V, Tt((size_t)b * b), res(b);
  double cut = -1.0, top = 1.0;
  const int degree = 8;
  bool converged = false;
  int it = 0;
  for (; it < maxiter; ++it) {
    if (it > 0) {
      // Chebyshev filter damping [-1, cut], scaled three-term recurrence
      const double e = (cut + 1.0) / 2.0, cc = (cut - 1.0) / 2.0;
      double sigma = e / (top - cc);
      const double tau = 2.0 / sigma;
      deflate(Q.p);
      spmm(Q.p, (float)cc, (float)(sigma / e), 0.f, nullptr, Y1.p);
      SCL_CUDA(cudaMemcpyAsync(Y0.p, Q.p, bn * sizeof(float), cudaMemcpyDeviceToDevice, st));
      float *xp = Y0.p, *y = Y1.p, *yn = Y2.p;
      for (int i = 2; i <= degree; ++i) {
        const double sigma_new = 1.0 / (tau - sigma);
        deflate(y);
        spmm(y, (float)cc, (float)(2.0 * sigma_new / e), (float)(sigma * sigma_new), xp, yn);
        float* t = xp; xp = y; y = yn; yn = t;
        sigma = sigma_new;
      }
      SCL_CUDA(cudaMemcpyAsync(Q.p, y, bn * sizeof(float), cudaMemcpyDeviceToDevice, st));
      deflate(Q.p);
      chol_qr(c, Q.p, b, Z.p, 2);
    }
    // Rayleigh-Ritz
    spmm(Q.p, 0.f, 1.f, 0.f, nullptr, Z.p);
    deflate(Z.p);
    gram_ts(c, Q.p, b, Z.p, b, dH.p);
    SCL_CUDA(cudaMemcpyAsync(H.data(), dH.p, H.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < b; ++i)
      for (int j = i + 1; j < b; ++j) H[(size_t)i * b + j] = H[(size_t)j * b + i] = 0.5 * (H[(size_t)i * b + j] + H[(size_t)j * b + i]);
    jacobi_desc(H, b, w, V);
    // Tt[c][r] = V[c][r]: new vector c = sum_r V[c][r] old r
    std::copy(V.begin(), V.end(), Tt.begin());
    SCL_CUDA(cudaMemcpyAsync(dTt.p, Tt.data(), Tt.size() * sizeof(double), cudaMemcpyHostToDevice, st));
    SCL_CUDA(cudaMemcpyAsync(dTheta.p, w.data(), b * sizeof(double), cudaMemcpyHostToDevice, st));
    combine_rows(c, Q.p, b, dTt.p, b, 1.0, nullptr, 0.0, Y0.p);
    combine_rows(c, Z.p, b, dTt.p, b, 1.0, nullptr, 0.0, Y1.p);
    residual_norms(c, Y1.p, Y0.p, dTheta.p, b, dRes.p);
    SCL_CUDA(cudaMemcpyAsync(res.data(), dRes.p, b * sizeof(double), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaMemcpyAsync(Q.p, Y0.p, bn * sizeof(float), cudaMemcpyDeviceToDevice, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    double rmax = 0;
    for (int i = 0; i < nc; ++i) rmax = std::max(rmax, res[i]);
    if (rmax <= 1e-4) { converged = true; ++it; break; }
    cut = std::max(w[b - 1], -1.0);        // damp everything below the block's smallest Ritz value
    top = std::max(w[0], cut + 1e-3);       // scale of the recurrence: the largest Ritz value
  }
  *iters = it;
  if (!converged) return false;
  // scale by 10 / max over the nc vectors
  std::vector<float> Qh((size_t)nc * N);
  SCL_CUDA(cudaMemcpyAsync(Qh.data(), Q.p, Qh.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  float mx = -INFINITY, amx = 0;
  for (float v : Qh) { mx = std::max(mx, v); amx = std::max(amx, std::fabs(v)); }
  const float m = mx > 0 ? mx : amx;
  if (!(m > 0)) return false;
  k_start_from_block<<<blocks((size_t)N * nc, 256), 256, 0, st>>>(Q.p, N, nc, 10.0f / m, umap_stream_key(seed, 4, 0), P);
  count_launches(2);
  SCL_CUDA(cudaGetLastError());
  return true;
}

// least-squares fit of 1 / (1 + a x^(2b)) to the UMAP membership curve on 300 points of [0, 3 spread]
// (Levenberg-Marquardt from (1, 1), Float64)
void umap_fit_ab(double min_dist, double spread, double* a_out, double* b_out) {
  const int n = 300;
  std::vector<double> x(n), y(n);
  for (int i = 0; i < n; ++i) {
    x[i] = 3.0 * spread * i / (n - 1);
    y[i] = x[i] >= min_dist ? std::exp(-(x[i] - min_dist) / spread) : 1.0;
  }
  auto cost = [&](double a, double b) {
    double s = 0;
    for (int i = 0; i < n; ++i) {
      const double r = 1.0 / (1.0 + a * std::pow(x[i], 2 * b)) - y[i];
      s += r * r;
    }
    return s;
  };
  double a = 1, b = 1, lam = 1e-3, f = cost(a, b);
  for (int it = 0; it < 10000; ++it) {
    double JTJ[3] = {0, 0, 0}, g[2] = {0, 0};
    for (int i = 0; i < n; ++i) {
      const double xp = x[i] > 0 ? std::pow(x[i], 2 * b) : 0.0;
      const double den = 1.0 + a * xp;
      const double r = 1.0 / den - y[i];
      const double ja = -xp / (den * den);
      const double jb = x[i] > 0 ? -a * xp * 2.0 * std::log(x[i]) / (den * den) : 0.0;
      JTJ[0] += ja * ja; JTJ[1] += ja * jb; JTJ[2] += jb * jb;
      g[0] += ja * r; g[1] += jb * r;
    }
    bool accepted = false;
    while (lam < 1e30) {
      const double m00 = JTJ[0] * (1 + lam), m11 = JTJ[2] * (1 + lam), m01 = JTJ[1];
      const double det = m00 * m11 - m01 * m01;
      const double da = -(m11 * g[0] - m01 * g[1]) / det, db = -(m00 * g[1] - m01 * g[0]) / det;
      const double an = std::max(0.0, a + da), bn = b + db;
      const double fn = cost(an, bn);
      if (fn <= f) {
        const double step = std::fabs(an - a) + std::fabs(bn - b);
        a = an; b = bn;
        const bool done = step <= 1e-15 * (std::fabs(a) + std::fabs(b)) || f - fn <= 1e-30;
        f = fn;
        lam = std::max(lam / 10, 1e-15);
        accepted = !done;
        break;
      }
      lam *= 10;
    }
    if (!accepted) break;
  }
  *a_out = a;
  *b_out = b;
}

void umap_run(scl_handle* h, const float* dX, int N, int d, const scl_umap_params& p, const float* d_init, float* d_emb,
              scl_umap_info* info) {
  cudaStream_t st = h->st;
  const int k = p.n_neighbors, nc = p.n_components;
  *info = scl_umap_info{};
  StageTimer tm(st);
  h->uk_idx.ensure((size_t)N * k);
  h->uk_dist.ensure((size_t)N * k);
  h->uk_N = N;
  h->uk_k = k;
  knn_device(dX, N, d, k, p.metric, h->uk_idx.p, h->uk_dist.p, st);
  info->t_knn_ms = tm.stop();
  build_graph(h, N, k, p.local_connectivity);
  info->graph_nnz = (int64_t)h->ug_nnz;
  info->t_graph_ms = tm.stop();
  double a, b;
  umap_fit_ab(p.min_dist, p.spread, &a, &b);
  info->a = a;
  info->b = b;
  Tmp<float> P0((size_t)N * nc, st), P1((size_t)N * nc, st);
  if (d_init) {
    k_from_colmajor<<<blocks((size_t)N * nc, 256), 256, 0, st>>>(d_init, N, nc, P0.p);
    count_launches(1);
  } else {
    bool ok = false;
    if (p.init == 0) {
      int iters = 0;
      ok = spectral_start(h, N, nc, p.spectral_maxiter, p.seed, P0.p, &iters);
      info->spectral_iters = iters;
      if (!ok) {
        info->init_fallback = 1;
        std::fprintf(stderr, "sclens_b200 apply_umap: spectral start did not converge in %d iterations; falling back to "
                             "a random start\n", iters);
      }
    }
    if (!ok) {
      k_random_start<<<blocks((size_t)N * nc, 256), 256, 0, st>>>(N, nc, umap_stream_key(p.seed, 3, 0), P0.p);
      count_launches(1);
    }
  }
  SCL_CUDA(cudaGetLastError());
  info->t_init_ms = tm.stop();
  float *cur = P0.p, *nxt = P1.p;
  for (int e = 0; e < p.n_epochs; ++e) {
    const float alpha = (float)(p.learning_rate * (1.0 - (double)e / p.n_epochs));
    k_layout_epoch<<<blocks(N, 128), 128, 0, st>>>(h->ug_rowptr.p, h->ug_col.p, h->ug_val.p, h->ug_rev.p, N, nc, cur, nxt,
                                                    umap_stream_key(p.seed, 1, e), umap_stream_key(p.seed, 2, e), alpha,
                                                    (float)a, (float)b, (float)p.repulsion_strength, p.neg_sample_rate);
    std::swap(cur, nxt);
  }
  count_launches(p.n_epochs + 1);
  k_to_colmajor<<<blocks((size_t)N * nc, 256), 256, 0, st>>>(cur, N, nc, d_emb);
  SCL_CUDA(cudaGetLastError());
  info->t_layout_ms = tm.stop();
}

}  // namespace scl
