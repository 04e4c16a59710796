// Float64 Rayleigh-quotient refinement of the eigenvalues returned by the FP32 eigensolver.
//
// cusolverDnSsyevd (the reference's solver, src/scLENS.jl:377) is backward stable in FP32: every eigenvalue carries
// an ABSOLUTE error of order eps32 * |G| (measured 1.9e-5 on the 10k x 10k benchmark Gram, whose largest
// eigenvalue is 21), i.e. 2e-4 RELATIVE at the lower Marchenko-Pastur edge - above the 1e-4 contract although the
// matrix itself is good to 3e-5.  The Rayleigh quotient of a computed eigenvector is accurate to second order in
// the eigenvector error, so   rho_i = v_i' G v_i / v_i' v_i   evaluated in Float64 from the FP32 eigenvectors and
// the FP32 Gram matrix recovers the eigenvalues of G to ~1e-6 relative.  One n x n x n Float64 contraction per
// sclens() call (only the data matrix's spectrum is an output), ~1 % of the eigensolver's time.
//
// Kernel: classic register-tiled GEMM  Z = V * G  (G symmetric, so both operands are read K-major), 128 x 128
// output tile per CTA, 8 x 8 per thread, FP32 operands staged in shared memory and widened in registers, FP64
// accumulation; the epilogue contracts the tile of Z with the matching tile of V, so Z is never written.
#include <algorithm>
#include <cmath>
#include <cstdlib>
#include "common.cuh"
#include "tmp.cuh"

namespace scl {

namespace {

constexpr int kTile = 128;
constexpr int kStepK = 16;
constexpr int kRqThreads = 256;
constexpr int kBand = 8;          // H = V G V' is evaluated on its diagonals 0..kBand
constexpr int kMaxCluster = 96;

// part[(i * n_tiles + tc) * (kBand+1) + d] = sum over c in column tile tc of (V G)[i][c] * V[i+d][c]
__global__ void __launch_bounds__(kRqThreads)
k_rq_partial(const float* __restrict__ V, const float* __restrict__ G, int n, int n_tiles, double* __restrict__ part) {
  __shared__ __align__(16) float As[2][kStepK][kTile];   // V tile, [k][row]
  __shared__ __align__(16) float Bs[2][kStepK][kTile];   // G tile, [k][col]
  const int tid = threadIdx.x;
  const int tr = blockIdx.y, tc = blockIdx.x;
  const int row0 = tr * kTile, col0 = tc * kTile;
  const int tx = tid & 15, ty = tid >> 4;                // 16 x 16 threads
  // global -> shared: thread loads rows lr and lr + 64 (of both operands), 4 consecutive k
  const int lr = tid & 63, lk = (tid >> 6) * 4;          // 64 rows x 4 k-groups of 4
  double acc[8][8];
#pragma unroll
  for (int a = 0; a < 8; ++a)
#pragma unroll
    for (int b = 0; b < 8; ++b) acc[a][b] = 0.0;

  auto load = [&](int kb, float4 (&va)[2], float4 (&vb)[2]) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = row0 + lr + 64 * h, c = col0 + lr + 64 * h, k = kb + lk;
      float t[4] = {0.f, 0.f, 0.f, 0.f}, u[4] = {0.f, 0.f, 0.f, 0.f};
      if (r < n) {
        if (k + 3 < n && (n & 3) == 0) {
          const float4 q = *reinterpret_cast<const float4*>(V + (size_t)r * n + k);
          t[0] = q.x; t[1] = q.y; t[2] = q.z; t[3] = q.w;
        } else {
          for (int q = 0; q < 4; ++q) if (k + q < n) t[q] = V[(size_t)r * n + k + q];
        }
      }
      if (c < n) {
        if (k + 3 < n && (n & 3) == 0) {
          const float4 q = *reinterpret_cast<const float4*>(G + (size_t)c * n + k);
          u[0] = q.x; u[1] = q.y; u[2] = q.z; u[3] = q.w;
        } else {
          for (int q = 0; q < 4; ++q) if (k + q < n) u[q] = G[(size_t)c * n + k + q];
        }
      }
      va[h] = make_float4(t[0], t[1], t[2], t[3]);
      vb[h] = make_float4(u[0], u[1], u[2], u[3]);
    }
  };
  auto stash = [&](int buf, const float4 (&va)[2], const float4 (&vb)[2]) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = lr + 64 * h;
      As[buf][lk + 0][r] = va[h].x; As[buf][lk + 1][r] = va[h].y; As[buf][lk + 2][r] = va[h].z; As[buf][lk + 3][r] = va[h].w;
      Bs[buf][lk + 0][r] = vb[h].x; Bs[buf][lk + 1][r] = vb[h].y; Bs[buf][lk + 2][r] = vb[h].z; Bs[buf][lk + 3][r] = vb[h].w;
    }
  };

  float4 va[2], vb[2];
  load(0, va, vb);
  stash(0, va, vb);
  __syncthreads();
  int buf = 0;
  for (int kb = 0; kb < n; kb += kStepK, buf ^= 1) {
    const bool more = kb + kStepK < n;
    if (more) load(kb + kStepK, va, vb);
#pragma unroll
    for (int k = 0; k < kStepK; ++k) {
      // rows ty*4..+3 and 64+ty*4..+3; columns tx*4..+3 and 64+tx*4..+3 (conflict-free float4 reads)
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][k][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][k][64 + tx * 4]);
      const double a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const double b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fma(a[i], b[j], acc[i][j]);
    }
    if (more) stash(buf ^ 1, va, vb);
    __syncthreads();
  }
  // epilogue: contract the tile of Z = V G with rows r, r+1, ..., r+kBand of V over this tile's columns (a band of
  // H = V G V'), reducing over the 16 threads that share the rows
  for (int d = 0; d <= kBand; ++d) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int r = row0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      const int rr = r + d;
      double s = 0.0;
      if (rr < n) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int c = col0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
          if (c < n) s = fma(acc[i][j], (double)V[(size_t)rr * n + c], s);
        }
      }
#pragma unroll
      for (int o = 8; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);   // lanes of one ty: 16 consecutive
      if (tx == 0 && r < n) part[((size_t)r * n_tiles + tc) * (kBand + 1) + d] = s;
    }
  }
}

// vv[i] = |v_i|^2  (one warp per eigenvector)
__global__ void __launch_bounds__(256) k_row_norm2(const float* __restrict__ V, int n, double* __restrict__ vv) {
  const int lane = threadIdx.x & 31;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  if (i >= n) return;
  double s = 0.0;
  for (int c = lane; c < n; c += 32) {
    const double x = (double)V[(size_t)i * n + c];
    s = fma(x, x, s);
  }
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (lane == 0) vv[i] = s;
}

// Hb[i][d] = v_i' G v_{i+d} / (|v_i| |v_{i+d}|)   (sum of the tile partials in a fixed order)
__global__ void __launch_bounds__(256) k_band_finish(const double* __restrict__ part, const double* __restrict__ vv, int n,
                                                     int n_tiles, double* __restrict__ Hb) {
  const long long w = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (w >= (long long)n * (kBand + 1)) return;
  const int i = (int)(w / (kBand + 1)), d = (int)(w % (kBand + 1));
  double s = 0.0;
  if (i + d < n) {
    for (int t = 0; t < n_tiles; ++t) s += part[((size_t)i * n_tiles + t) * (kBand + 1) + d];
    s /= sqrt(vv[i] * vv[i + d]);
  }
  Hb[w] = s;
}

// eigenvalues of a small dense symmetric matrix (row-major m x m, destroyed) by cyclic Jacobi rotations
void jacobi_eigenvalues(std::vector<double>& a, int m, std::vector<double>& ev) {
  for (int sweep = 0; sweep < 60; ++sweep) {
    double off = 0, diag = 0;
    for (int p = 0; p < m; ++p) {
      diag += a[(size_t)p * m + p] * a[(size_t)p * m + p];
      for (int q = p + 1; q < m; ++q) off += a[(size_t)p * m + q] * a[(size_t)p * m + q];
    }
    if (off <= 1e-30 * diag) break;
    for (int p = 0; p < m; ++p)
      for (int q = p + 1; q < m; ++q) {
        const double apq = a[(size_t)p * m + q];
        if (apq == 0.0) continue;
        const double theta = (a[(size_t)q * m + q] - a[(size_t)p * m + p]) / (2.0 * apq);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double c = 1.0 / std::sqrt(t * t + 1.0), sn = t * c;
        for (int k = 0; k < m; ++k) {   // columns p, q
          const double akp = a[(size_t)k * m + p], akq = a[(size_t)k * m + q];
          a[(size_t)k * m + p] = c * akp - sn * akq;
          a[(size_t)k * m + q] = sn * akp + c * akq;
        }
        for (int k = 0; k < m; ++k) {   // rows p, q
          const double apk = a[(size_t)p * m + k], aqk = a[(size_t)q * m + k];
          a[(size_t)p * m + k] = c * apk - sn * aqk;
          a[(size_t)q * m + k] = sn * apk + c * aqk;
        }
      }
  }
  ev.resize(m);
  for (int p = 0; p < m; ++p) ev[p] = a[(size_t)p * m + p];
  std::sort(ev.begin(), ev.end());
}

}  // namespace

// dV: eigenvectors as rows of memory (cuSOLVER's column-major result), dG: the matrix they belong to (symmetric).
// dW (ascending FP32 eigenvalues) is overwritten by the refined eigenvalues, ascending.  stats (optional): [0] number of
// clusters solved as Rayleigh-Ritz blocks, [1] size of the largest (1 when there is none).
void refine_eigenvalues(const float* dG, const float* dV, int n, float* dW, cudaStream_t st, int* stats) {
  const int n_tiles = (n + kTile - 1) / kTile;
  const int nb = kBand + 1;
  Tmp<double> part((size_t)n * n_tiles * nb, st), vv(n, st), dHb((size_t)n * nb, st);
  count_launches(3);
  k_rq_partial<<<dim3(n_tiles, n_tiles), kRqThreads, 0, st>>>(dV, dG, n, n_tiles, part.p);
  k_row_norm2<<<(n * 32 + 255) / 256, 256, 0, st>>>(dV, n, vv.p);
  k_band_finish<<<(unsigned)(((long long)n * nb + 255) / 256), 256, 0, st>>>(part.p, vv.p, n, n_tiles, dHb.p);
  SCL_CUDA(cudaGetLastError());
  std::vector<double> Hb((size_t)n * nb);
  SCL_CUDA(cudaMemcpyAsync(Hb.data(), dHb.p, Hb.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  auto H = [&](int i, int j) -> double {   // i <= j <= i + kBand
    return Hb[(size_t)i * nb + (j - i)];
  };
  // Rayleigh quotients H_ii are exact to second order in the eigenvector error - except inside a cluster of
  // eigenvalues closer than the solver's backward error, where the computed vectors are an arbitrary rotation
  // of the true ones: there the Rayleigh-Ritz values of the cluster (eigenvalues of H restricted to it) are.
  // i and j are linked when the rotation angle |H_ij / (H_jj - H_ii)| is not negligible.
  std::vector<double> out(n);
  std::vector<double> blk, ev;
  const bool trace = getenv("SCL_TRACE") != nullptr;
  int n_clusters = 0, max_cluster = 1;
  int i = 0;
  while (i < n) {
    int hi = i;                                    // cluster = [i, hi]
    for (int a = i; a <= hi && hi - i + 1 < kMaxCluster; ++a)
      for (int b = std::max(a + 1, hi + 1); b <= std::min(n - 1, a + kBand); ++b)
        if (std::fabs(H(a, b)) > 0.02 * std::fabs(H(b, b) - H(a, a))) hi = std::max(hi, b);
    hi = std::min(hi, i + kMaxCluster - 1);
    const int m = hi - i + 1;
    if (m == 1) {
      out[i] = H(i, i);
    } else {
      blk.assign((size_t)m * m, 0.0);
      for (int a = 0; a < m; ++a)
        for (int b = a; b < m && b - a <= kBand; ++b) blk[(size_t)a * m + b] = blk[(size_t)b * m + a] = H(i + a, i + b);
      jacobi_eigenvalues(blk, m, ev);
      for (int a = 0; a < m; ++a) out[i + a] = ev[a];
      if (trace && (m > 8 || ev[0] < -1e-4)) {
        fprintf(stderr, "[scl] refine: cluster [%d,%d] size %d, H_ii %.6g .. %.6g -> ritz %.6g .. %.6g\n", i, hi, m, H(i, i),
                H(hi, hi), ev[0], ev[m - 1]);
      }
      ++n_clusters;
      max_cluster = std::max(max_cluster, m);
    }
    i = hi + 1;
  }
  if (trace) {
    fprintf(stderr, "[scl] refine: n=%d, %d clusters (largest %d); H_00 %.6g H_11 %.6g H_22 %.6g H_01 %.3g H_12 %.3g; vv0 %.9g\n", n,
            n_clusters, max_cluster, H(0, 0), H(1, 1), H(2, 2), H(0, 1), H(1, 2), 0.0);
  }
  if (stats) { stats[0] = n_clusters; stats[1] = max_cluster; }
  std::sort(out.begin(), out.end());
  std::vector<float> outf(n);
  for (int q = 0; q < n; ++q) outf[q] = (float)out[q];
  SCL_CUDA(cudaMemcpyAsync(dW, outf.data(), n * sizeof(float), cudaMemcpyHostToDevice, st));
  SCL_CUDA(cudaStreamSynchronize(st));
}

}  // namespace scl
