// Leading-k eigenpairs of a symmetric PSD matrix by Chebyshev-filtered block subspace
// iteration with locking (replaces the full syevd of get_eigvec, src/scLENS.jl:489-524, in
// the perturbation stage :771-778, where only the first ceil(1.5*n_signal) vectors are kept).
//
// The n x n products G*Q run on the tcgen05 GEMM (split binary16 operands, ~FP32 accuracy);
// the tall-skinny b x b reductions, Cholesky-QR and Rayleigh-Ritz rotations accumulate in
// Float64.  Blocks are stored vector-major ([b][n], each vector contiguous), which is the
// K-major layout the GEMM wants for its B operand.
//
// Per sweep: degree-d Chebyshev filter damping [0, cut] -> orthogonalise against the locked
// vectors -> CholQR2 -> Rayleigh-Ritz -> lock converged leading pairs.  The degree adapts so
// the filter's dynamic range over the active block stays below kAmpLimit (the block is
// stored in FP32, so a larger range would wash out the weakest wanted direction).
#include <algorithm>
#include <cmath>
#include "handle.h"
#include "subspace.h"
#include "tmp.cuh"

namespace scl {

namespace {

constexpr int kSlab = 64;
constexpr double kAmpLimit = 2.0e3;
// G's off-diagonal entries are ~1/sqrt(n) of its diagonal: scaled by 2^6 before the binary16 hi/lo split so
// their low-order parts stay normal numbers (diagonal ~O(1..30) -> <= 2e3, far below 65504)
constexpr float kGScale = 64.f;

inline size_t round8(size_t x) { return (x + 7) / 8 * 8; }

__global__ void k_random_rows(float* __restrict__ q, int rows, int n, uint64_t seed) {
  size_t total = (size_t)rows * n;
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    uint64_t h = mix64s(seed ^ mix64s(i));
    float u1 = ((uint32_t)(h >> 40) + 1u) * (1.0f / 16777217.0f);
    float u2 = (uint32_t)(h & 0xffffffu) * (1.0f / 16777216.0f);
    q[i] = sqrtf(-2.f * logf(u1)) * cospif(2.f * u2);
  }
}

// S[ra][rb] += A[ra][n] * B[rb][n]^T over one slab of kSlab positions per CTA (Float64).
// smem: sA[kSlab][pa], sB[kSlab][pb] (position-major so the 4x4 register tiles read float4).
__global__ void __launch_bounds__(256) k_gram_ts(const float* __restrict__ A, int ra, const float* __restrict__ B, int rb,
                                                 int n, double* __restrict__ S, double* __restrict__ part) {
  extern __shared__ float sm[];
  const int pa = ((ra + 3) / 4) * 4 + 4, pb = ((rb + 3) / 4) * 4 + 4;
  float* sA = sm;
  float* sB = (A == B) ? sA : sm + (size_t)kSlab * pa;
  const int t0 = blockIdx.x * kSlab;
  const int tl = min(kSlab, n - t0);
  for (int i = threadIdx.x; i < kSlab * pa; i += blockDim.x) sA[i] = 0.f;
  if (A != B)
    for (int i = threadIdx.x; i < kSlab * pb; i += blockDim.x) sB[i] = 0.f;
  __syncthreads();
  for (int i = threadIdx.x; i < ra * kSlab; i += blockDim.x) {
    int r = i / kSlab, t = i % kSlab;
    if (t < tl) sA[t * pa + r] = A[(size_t)r * n + t0 + t];
  }
  if (A != B)
    for (int i = threadIdx.x; i < rb * kSlab; i += blockDim.x) {
      int r = i / kSlab, t = i % kSlab;
      if (t < tl) sB[t * pb + r] = B[(size_t)r * n + t0 + t];
    }
  __syncthreads();
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int pbb = (A == B) ? pa : pb;
  for (int i0 = 0; i0 < ra; i0 += 64)
    for (int j0 = 0; j0 < rb; j0 += 64) {
      const int i = i0 + ty * 4, j = j0 + tx * 4;
      if (i >= ra || j >= rb) continue;
      double acc[4][4] = {};
      for (int t = 0; t < tl; ++t) {
        const float4 a = *reinterpret_cast<const float4*>(&sA[t * pa + i]);
        const float4 b = *reinterpret_cast<const float4*>(&sB[t * pbb + j]);
        const double av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
        for (int u = 0; u < 4; ++u)
#pragma unroll
          for (int v = 0; v < 4; ++v) acc[u][v] += av[u] * bv[v];
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
#pragma unroll
        for (int v = 0; v < 4; ++v)
          if (i + u < ra && j + v < rb) {
            if (part) part[(size_t)blockIdx.x * ra * rb + (size_t)(i + u) * rb + j + v] = acc[u][v];
            else atomicAdd(&S[(size_t)(i + u) * rb + j + v], acc[u][v]);
          }
    }
}

// S[e] = sum over CTAs of part[cta][e], CTAs in ascending order
__global__ void k_sum_parts(const double* __restrict__ part, int nparts, size_t ne, double* __restrict__ S) {
  for (size_t e = blockIdx.x * (size_t)blockDim.x + threadIdx.x; e < ne; e += (size_t)gridDim.x * blockDim.x) {
    double s = 0;
    for (int p = 0; p < nparts; ++p) s += part[(size_t)p * ne + e];
    S[e] = s;
  }
}

// out[c][t] = beta * base[c][t] + alpha * sum_r Tt[c][r] * In[r][t]   (Float64 accumulation)
__global__ void __launch_bounds__(256) k_combine_rows(const float* __restrict__ In, int rin, const double* __restrict__ Tt,
                                                      int rout, int n, double alpha, const float* __restrict__ base,
                                                      double beta, float* __restrict__ out,
                                                      const double* __restrict__ wgt) {
  extern __shared__ float sIn[];   // [rin][kSlab]
  const int t0 = blockIdx.x * kSlab;
  const int tl = min(kSlab, n - t0);
  for (int i = threadIdx.x; i < rin * kSlab; i += blockDim.x) {
    int r = i / kSlab, t = i % kSlab;
    sIn[i] = t < tl ? In[(size_t)r * n + t0 + t] : 0.f;
  }
  __syncthreads();
  const int t = threadIdx.x % kSlab, g = threadIdx.x / kSlab;   // 4 row groups
  if (t >= tl) return;
  for (int c = g; c < rout; c += 4) {
    const double* trow = Tt + (size_t)c * rin;
    double acc = 0;
    if (wgt) {
      for (int r = 0; r < rin; ++r) acc += trow[r] * wgt[r] * (double)sIn[r * kSlab + t];
    } else {
      for (int r = 0; r < rin; ++r) acc += trow[r] * (double)sIn[r * kSlab + t];
    }
    double v = alpha * acc;
    if (base) v += beta * (double)base[(size_t)c * n + t0 + t];
    out[(size_t)c * n + t0 + t] = (float)v;
  }
}

// Chebyshev recurrence step: out = (Z - c*Y) * s1 - s2 * Xp     (Xp may be null when s2 == 0)
__global__ void k_cheb_step(const float* __restrict__ Z, const float* __restrict__ Y, const float* __restrict__ Xp,
                            float c, float s1, float s2, size_t total, float* __restrict__ out) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < total; i += stride) {
    float v = (Z[i] - c * Y[i]) * s1;
    if (Xp) v -= s2 * Xp[i];
    out[i] = v;
  }
}

// res[r] = | Z_r - theta_r Q_r |_2
__global__ void __launch_bounds__(256) k_residuals(const float* __restrict__ Z, const float* __restrict__ Q,
                                                   const double* __restrict__ theta, int rows, int n,
                                                   double* __restrict__ res) {
  __shared__ double red[8];
  for (int r = blockIdx.x; r < rows; r += gridDim.x) {
    const double th = theta[r];
    double s = 0;
    for (int t = threadIdx.x; t < n; t += blockDim.x) {
      double d = (double)Z[(size_t)r * n + t] - th * (double)Q[(size_t)r * n + t];
      s += d * d;
    }
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0;
      for (int w = 0; w < 8; ++w) t += red[w];
      res[r] = sqrt(t);
    }
  }
}

}  // namespace

using Ctx = BlockCtx;

void gram_ts(const Ctx& c, const float* A, int ra, const float* B, int rb, double* dS) {
  const int pa = ((ra + 3) / 4) * 4 + 4, pb = ((rb + 3) / 4) * 4 + 4;
  size_t smem = (size_t)kSlab * (A == B ? pa : pa + pb) * sizeof(float);
  SCL_CUDA(cudaFuncSetAttribute(k_gram_ts, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  const int grid = (c.n + kSlab - 1) / kSlab;
  if (c.fixed_order) {
    const size_t ne = (size_t)ra * rb;
    Tmp<double> part((size_t)grid * ne, c.st);
    k_gram_ts<<<grid, 256, smem, c.st>>>(A, ra, B, rb, c.n, dS, part.p);
    k_sum_parts<<<(int)std::min<size_t>((ne + 255) / 256, 148 * 4), 256, 0, c.st>>>(part.p, grid, ne, dS);
    count_launches(2);
  } else {
    SCL_CUDA(cudaMemsetAsync(dS, 0, (size_t)ra * rb * sizeof(double), c.st));
    k_gram_ts<<<grid, 256, smem, c.st>>>(A, ra, B, rb, c.n, dS, nullptr);
    count_launches(1);
  }
  SCL_CUDA(cudaGetLastError());
}

void combine_rows(const Ctx& c, const float* In, int rin, const double* dTt, int rout, double alpha, const float* base,
                  double beta, float* out, const double* wgt) {
  size_t smem = (size_t)rin * kSlab * sizeof(float);
  SCL_CUDA(cudaFuncSetAttribute(k_combine_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  k_combine_rows<<<(c.n + kSlab - 1) / kSlab, 256, smem, c.st>>>(In, rin, dTt, rout, c.n, alpha, base, beta, out, wgt);
  count_launches(1);
  SCL_CUDA(cudaGetLastError());
}

void residual_norms(const Ctx& c, const float* Z, const float* Q, const double* dTheta, int rows, double* dRes) {
  k_residuals<<<std::min(rows, 148 * 4), 256, 0, c.st>>>(Z, Q, dTheta, rows, c.n, dRes);
  count_launches(1);
  SCL_CUDA(cudaGetLastError());
}

// Z[rows][n] = (G * Q^T)^T through the tensor-core GEMM (split operands)
static void apply_G(const Ctx& c, const float* Q, int rows, float* Z) {
  Tmp<__half> q_hi((size_t)rows * c.ldn, c.st), q_lo((size_t)rows * c.ldn, c.st);
  strided_split_f32_to_f16(Q, rows, c.n, c.n, (int64_t)c.ldn, q_hi.p, q_lo.p, c.st);
  const int cg = c.h->cfg.cta_group == 1 ? 1 : 2;
  GemmArgs g;
  g.A.hi = c.g_hi; g.A.lo = c.g_lo; g.A.rows = c.n; g.A.K = c.n; g.A.ld = (int64_t)c.ldn;
  g.B.hi = q_hi.p; g.B.lo = q_lo.p; g.B.rows = rows; g.B.K = c.n; g.B.ld = (int64_t)c.ldn;
  g.epi = Epilogue::StoreTransposed;
  g.ldc = c.n;
  g.cta_group = cg;
  const float inv_scale = 1.f / kGScale;
  // split-K so the machine is filled: pick the split count with the fewest waves per unit of work
  const int units = sm_count() / cg;
  const int tiles = (c.n + 128 * cg - 1) / (128 * cg);
  const int kblocks = (c.n + 63) / 64;
  int best = 1;
  double best_cost = 1e30;
  for (int s = 1; s <= 16 && s * 8 <= kblocks; ++s) {
    double cost = std::ceil((double)tiles * s / units) / s + 0.02 * s;
    if (cost < best_cost) { best_cost = cost; best = s; }
  }
  ProfScope ps(&c.h->prof, c.st, PK_OTHER_GEMM);
  c.h->prof.other_gemm_flops += 2.0 * (double)c.n * c.n * rows;
  if (best == 1) {
    g.C = Z; g.alpha = inv_scale;
    gemm_umma(g, c.st);
  } else {
    const size_t elems = (size_t)rows * c.n;
    Tmp<float> part((size_t)best * elems, c.st);
    g.C = part.p; g.splits = best; g.split_stride = (int64_t)elems;
    gemm_umma(g, c.st);
    reduce_splits(part.p, best, (int64_t)elems, elems, inv_scale, Z, c.st);
  }
}

bool chol_inverse_t(std::vector<double>& S, int b, std::vector<double>& Tt) {
  std::vector<double> R((size_t)b * b, 0.0);
  for (int j = 0; j < b; ++j) {
    double d = S[(size_t)j * b + j];
    for (int k = 0; k < j; ++k) d -= R[(size_t)k * b + j] * R[(size_t)k * b + j];
    if (!(d > 0)) return false;
    const double rjj = std::sqrt(d);
    R[(size_t)j * b + j] = rjj;
    for (int i = j + 1; i < b; ++i) {
      double s = S[(size_t)j * b + i];
      for (int k = 0; k < j; ++k) s -= R[(size_t)k * b + j] * R[(size_t)k * b + i];
      R[(size_t)j * b + i] = s / rjj;
    }
  }
  // invert the upper-triangular R by back substitution, column by column
  std::vector<double> Ri((size_t)b * b, 0.0);
  for (int c = 0; c < b; ++c) {
    Ri[(size_t)c * b + c] = 1.0 / R[(size_t)c * b + c];
    for (int r = c - 1; r >= 0; --r) {
      double s = 0;
      for (int k = r + 1; k <= c; ++k) s += R[(size_t)r * b + k] * Ri[(size_t)k * b + c];
      Ri[(size_t)r * b + c] = -s / R[(size_t)r * b + r];
    }
  }
  Tt.assign((size_t)b * b, 0.0);
  for (int c = 0; c < b; ++c)
    for (int r = 0; r <= c; ++r) Tt[(size_t)c * b + r] = Ri[(size_t)r * b + c];
  return true;
}

void chol_qr(const Ctx& c, float* Q, int rows, float* tmp, int passes) {
  Tmp<double> dS((size_t)rows * rows, c.st), dT((size_t)rows * rows, c.st);
  std::vector<double> S((size_t)rows * rows), Tt;
  for (int p = 0; p < passes; ++p) {
    gram_ts(c, Q, rows, Q, rows, dS.p);
    SCL_CUDA(cudaMemcpyAsync(S.data(), dS.p, S.size() * sizeof(double), cudaMemcpyDeviceToHost, c.st));
    SCL_CUDA(cudaStreamSynchronize(c.st));
    if (!chol_inverse_t(S, rows, Tt)) {
      // rank-deficient block: regularise relative to the largest diagonal and retry once
      double mx = 0;
      for (int i = 0; i < rows; ++i) mx = std::max(mx, S[(size_t)i * rows + i]);
      for (int i = 0; i < rows; ++i) S[(size_t)i * rows + i] += 1e-10 * mx;
      if (!chol_inverse_t(S, rows, Tt)) throw Error(SCL_ERR_CUSOLVER, "subspace iteration: block lost rank (CholQR failed)");
    }
    SCL_CUDA(cudaMemcpyAsync(dT.p, Tt.data(), Tt.size() * sizeof(double), cudaMemcpyHostToDevice, c.st));
    combine_rows(c, Q, rows, dT.p, rows, 1.0, nullptr, 0.0, tmp);
    SCL_CUDA(cudaMemcpyAsync(Q, tmp, (size_t)rows * c.n * sizeof(float), cudaMemcpyDeviceToDevice, c.st));
    SCL_CUDA(cudaStreamSynchronize(c.st));
  }
}

void topk_subspace(scl_handle* h, const float* dG, int n, int k, float* dL, float* dV, int* iters_out) {
  cudaStream_t st = h->st;
  const int extra = h->cfg.subspace_extra > 0 ? h->cfg.subspace_extra : 64;
  const int dmax = h->cfg.subspace_degree > 0 ? h->cfg.subspace_degree : 30;
  int b = std::min(256, ((k + extra + 31) / 32) * 32);
  SCL_REQUIRE(k >= 1 && k + 16 <= b, "too many vectors requested for the block subspace iteration (use exact_perturb)");
  SCL_REQUIRE(b * 2 <= n, "matrix too small for the block subspace iteration (use exact_perturb)");
  Ctx c;
  c.h = h; c.st = st; c.n = n; c.ldn = round8((size_t)n);
  Tmp<__half> g_hi((size_t)n * c.ldn, st), g_lo((size_t)n * c.ldn, st);
  strided_split_f32_to_f16(dG, n, n, n, (int64_t)c.ldn, g_hi.p, g_lo.p, st, kGScale);
  c.g_hi = g_hi.p; c.g_lo = g_lo.p;

  const size_t bn = (size_t)b * n;
  Tmp<float> Q(bn, st), Z(bn, st), Y0(bn, st), Y1(bn, st), Y2(bn, st), Vlock((size_t)k * n, st);
  Tmp<double> dH((size_t)b * b, st), dW(b, st), dTt((size_t)b * b, st), dTheta(b, st), dRes(b, st), dC((size_t)k * b, st),
      dShift(k, st);
  std::vector<double> shift(k);
  std::vector<double> Hh((size_t)b * b), Wh(b), Tt((size_t)b * b), theta(b), res(b), Llock;
  int nlock = 0;

  k_random_rows<<<148 * 4, 256, 0, st>>>(Q.p, b, n, mix64s(h->cfg.seed ^ 0x73756273ull));
  SCL_CUDA(cudaGetLastError());
  chol_qr(c, Q.p, b, Z.p, 2);

  double cut = 0, top = 0, theta_max = 0;
  int sweeps = 0, gemms = 0;
  const double tol = 3e-5;
  const int max_sweeps = 60;
  for (; sweeps < max_sweeps; ++sweeps) {
    const int ba = b - nlock;
    float* Qa = Q.p;   // active block lives in rows [0, ba)
    if (sweeps > 0) {
      // ---- Chebyshev filter of degree d damping [0, cut] (scaled three-term recurrence)
      const double e = cut / 2.0, cc = cut / 2.0;
      const double x_top = std::max(1.0 + 1e-6, (top - cc) / e);
      int d = (int)std::floor(std::acosh(kAmpLimit) / std::acosh(x_top));
      d = std::max(2, std::min(dmax, d));
      if (sweeps == 1) d = std::min(d, 3);   // Ritz values of the random start are poor bounds
      double sigma = e / (top - cc);
      const double tau = 2.0 / sigma;
      const size_t total = (size_t)ba * n;
      const int grid = (int)std::min<size_t>((total + 255) / 256, 148 * 16);
      // Locked eigenpairs are deflated from the operator, G' = G - sum_l (theta_l - cc) v_l v_l^T, which moves
      // them to the centre of the damped interval: without this the filter re-amplifies the ~1e-7 component the
      // FP32 active block keeps along a locked signal direction by T_d(x_l)/T_d(x_top) (1e20 at degree 30).
      for (int l = 0; l < nlock; ++l) shift[l] = Llock[l] - cc;
      if (nlock) SCL_CUDA(cudaMemcpyAsync(dShift.p, shift.data(), nlock * sizeof(double), cudaMemcpyHostToDevice, st));
      auto apply_deflated = [&](const float* y) {
        apply_G(c, y, ba, Z.p); ++gemms;
        if (nlock) {
          gram_ts(c, y, ba, Vlock.p, nlock, dC.p);                                   // C[ba][nlock] = y * Vlock^T
          combine_rows(c, Vlock.p, nlock, dC.p, ba, -1.0, Z.p, 1.0, Z.p, dShift.p);  // Z -= C diag(shift) Vlock
        }
      };
      apply_deflated(Qa);
      k_cheb_step<<<grid, 256, 0, st>>>(Z.p, Qa, nullptr, (float)cc, (float)(sigma / e), 0.f, total, Y1.p);
      count_launches(d);
      SCL_CUDA(cudaMemcpyAsync(Y0.p, Qa, total * sizeof(float), cudaMemcpyDeviceToDevice, st));
      float *xp = Y0.p, *y = Y1.p, *yn = Y2.p;
      for (int i = 2; i <= d; ++i) {
        const double sigma_new = 1.0 / (tau - sigma);
        apply_deflated(y);
        k_cheb_step<<<grid, 256, 0, st>>>(Z.p, y, xp, (float)cc, (float)(2.0 * sigma_new / e), (float)(sigma * sigma_new),
                                          total, yn);
        float* t = xp; xp = y; y = yn; yn = t;
        sigma = sigma_new;
      }
      SCL_CUDA(cudaGetLastError());
      SCL_CUDA(cudaMemcpyAsync(Qa, y, total * sizeof(float), cudaMemcpyDeviceToDevice, st));
      // ---- keep the active block orthogonal to the locked vectors (two passes)
      for (int pass = 0; pass < 2 && nlock > 0; ++pass) {
        gram_ts(c, Qa, ba, Vlock.p, nlock, dC.p);   // C[ba][nlock] = Qa * Vlock^T  == Tt[c][l]
        combine_rows(c, Vlock.p, nlock, dC.p, ba, -1.0, Qa, 1.0, Z.p);
        SCL_CUDA(cudaMemcpyAsync(Qa, Z.p, total * sizeof(float), cudaMemcpyDeviceToDevice, st));
      }
      chol_qr(c, Qa, ba, Z.p, 2);
    }
    // ---- Rayleigh-Ritz on the active block
    apply_G(c, Qa, ba, Z.p); ++gemms;
    gram_ts(c, Qa, ba, Z.p, ba, dH.p);
    SCL_CUDA(cudaMemcpyAsync(Hh.data(), dH.p, (size_t)ba * ba * sizeof(double), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < ba; ++i)
      for (int j = i + 1; j < ba; ++j) {
        double s = 0.5 * (Hh[(size_t)i * ba + j] + Hh[(size_t)j * ba + i]);
        Hh[(size_t)i * ba + j] = Hh[(size_t)j * ba + i] = s;
      }
    SCL_CUDA(cudaMemcpyAsync(dH.p, Hh.data(), (size_t)ba * ba * sizeof(double), cudaMemcpyHostToDevice, st));
    h->solver->dsyevd_small(dH.p, ba, dW.p, st);
    SCL_CUDA(cudaMemcpyAsync(Hh.data(), dH.p, (size_t)ba * ba * sizeof(double), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaMemcpyAsync(Wh.data(), dW.p, ba * sizeof(double), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    // eigenvector j (ascending) is column j of the column-major result == row j of memory; reverse to descending
    for (int cidx = 0; cidx < ba; ++cidx) {
      const int src = ba - 1 - cidx;
      theta[cidx] = Wh[src];
      std::copy(Hh.begin() + (size_t)src * ba, Hh.begin() + (size_t)(src + 1) * ba, Tt.begin() + (size_t)cidx * ba);
    }
    SCL_CUDA(cudaMemcpyAsync(dTt.p, Tt.data(), (size_t)ba * ba * sizeof(double), cudaMemcpyHostToDevice, st));
    SCL_CUDA(cudaMemcpyAsync(dTheta.p, theta.data(), ba * sizeof(double), cudaMemcpyHostToDevice, st));
    combine_rows(c, Qa, ba, dTt.p, ba, 1.0, nullptr, 0.0, Y0.p);    // Q <- Ritz vectors
    combine_rows(c, Z.p, ba, dTt.p, ba, 1.0, nullptr, 0.0, Y1.p);   // Z <- G * Ritz vectors
    residual_norms(c, Y1.p, Y0.p, dTheta.p, ba, dRes.p);
    SCL_CUDA(cudaMemcpyAsync(res.data(), dRes.p, ba * sizeof(double), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaMemcpyAsync(Qa, Y0.p, (size_t)ba * n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    if (nlock == 0) theta_max = std::max(theta_max, theta[0]);
    // ---- lock the converged leading pairs (contiguous prefix only, so order is preserved)
    int newly = 0;
    while (nlock + newly < k && newly < ba - 16 && res[newly] <= tol * std::max(theta[newly], 1e-3 * theta_max)) ++newly;
    if (newly > 0) {
      SCL_CUDA(cudaMemcpyAsync(Vlock.p + (size_t)nlock * n, Qa, (size_t)newly * n * sizeof(float), cudaMemcpyDeviceToDevice, st));
      for (int i = 0; i < newly; ++i) Llock.push_back(theta[i]);
      // shift the remaining active vectors to the front
      SCL_CUDA(cudaMemcpyAsync(Y0.p, Qa + (size_t)newly * n, (size_t)(ba - newly) * n * sizeof(float), cudaMemcpyDeviceToDevice, st));
      SCL_CUDA(cudaMemcpyAsync(Qa, Y0.p, (size_t)(ba - newly) * n * sizeof(float), cudaMemcpyDeviceToDevice, st));
      nlock += newly;
    }
    if (nlock >= k) { ++sweeps; break; }
    const int ba2 = b - nlock;
    top = theta[newly];              // largest unconverged Ritz value
    cut = theta[newly + ba2 - 1];    // smallest Ritz value of the active block
    if (!(cut > 0)) cut = 1e-6 * theta_max;
    if (top <= cut) top = cut * (1 + 1e-3);
  }
  if (nlock < k) throw Error(SCL_ERR_CUSOLVER, "block subspace iteration did not converge in " + std::to_string(max_sweeps) + " sweeps");
  std::vector<float> Lf(k);
  for (int i = 0; i < k; ++i) Lf[i] = (float)Llock[i];
  SCL_CUDA(cudaMemcpyAsync(dL, Lf.data(), k * sizeof(float), cudaMemcpyHostToDevice, st));
  SCL_CUDA(cudaMemcpyAsync(dV, Vlock.p, (size_t)k * n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  if (iters_out) *iters_out = gemms;
  (void)sweeps;
}

}  // namespace scl
