// Symmetric eigensolves (_get_eigen, src/scLENS.jl:375-382) on the own solver: the two-stage reduction (twostage.h) or the
// one-stage path (sytrd.cu), the Float64 tridiagonal stage (tridiag.cu) and the back-transformations.  cuSOLVER serves the
// one-stage path where the own kernels decline (Ssytrd, Sormtr), the last resort (Ssyevd) and the timing study of the
// library solvers.  Also the scalar Marchenko-Pastur / Tracy-Widom fit (:390-487).
#include <cusolverDn.h>
#include <algorithm>
#include <cmath>
#include <atomic>
#include "common.cuh"
#include "eigen.h"
#include "tmp.cuh"
#include "twostage.h"

namespace scl {

#define SCL_SOLVER(x)                                                                         \
  do {                                                                                        \
    cusolverStatus_t s_ = (x);                                                                \
    if (s_ != CUSOLVER_STATUS_SUCCESS)                                                        \
      throw scl::Error(-3, std::string(#x) + ": cusolver status " + std::to_string((int)s_)); \
  } while (0)

struct Solver::Impl {
  cusolverDnHandle_t h = nullptr;
  DBuf<float> work;
  DBuf<float> tri_d, tri_e, tri_tau, tri_z, tri_keep, tri_pad;   // own tridiagonal stage: T, reflector scalars, vectors, matrix copy, padded copy
  DBuf<double> tri_w;
  // two-stage path (twostage.h): band, panel T factors, stage-2 reflectors and their scalars, matrix copy for the fallback
  DBuf<float> ts_AB, ts_T1, ts_V2, ts_tau2, ts_keep;
  DBuf<int> ts_fail;
  Sy2sbAux ts_aux;
  DBuf<double> dwork;
  DBuf<int> info;
};

static std::atomic<bool> g_force_one_stage{false};
void force_one_stage(bool on) { g_force_one_stage.store(on, std::memory_order_relaxed); }

Solver::Solver(cudaStream_t st) : impl(new Impl) {
  SCL_SOLVER(cusolverDnCreate(&impl->h));
  SCL_SOLVER(cusolverDnSetStream(impl->h, st));
  impl->info.ensure(1);
}
Solver::~Solver() {
  if (impl->ts_aux.stream) {
    cudaStreamDestroy(impl->ts_aux.stream);
    cudaEventDestroy(impl->ts_aux.ready);
    cudaEventDestroy(impl->ts_aux.done);
  }
  if (impl->h) cusolverDnDestroy(impl->h);
  delete impl;
}

// Two-stage solve: dense -> band -> tridiagonal, Float64 tridiagonal stage, Z = Q1 Q2 E.  Same contract as
// syevd_tri; a panel that cannot be factored (rank-deficient panel) or a failed tridiagonal stage falls back, loudly and
// counted, to the one-stage path on a kept copy.
bool Solver::syevd_2stage(float* dA, int n, float* dW, int v0, int v1, cudaStream_t st) {
  const int m = v1 - v0;
  const size_t nn = (size_t)n * n;
  const long long lda = ((long long)n + 3) & ~3LL, ldz = lda;
  const int nlev = sb2st_levels(n);
  const long long ldv2 = (long long)nlev * kBand, ldt2 = nlev;
  cudaEvent_t ev[6];
  for (auto& e : ev) SCL_CUDA(cudaEventCreate(&e));
  impl->tri_d.ensure(n); impl->tri_e.ensure(n); impl->tri_w.ensure(n);
  impl->ts_keep.ensure(nn);
  impl->ts_AB.ensure((size_t)n * kLdab);
  impl->ts_T1.ensure((size_t)(n / kBand + 2) * kBand * kBand);
  impl->ts_fail.ensure(1);
  SCL_CUDA(cudaMemcpyAsync(impl->ts_keep.p, dA, nn * sizeof(float), cudaMemcpyDeviceToDevice, st));
  SCL_CUDA(cudaMemsetAsync(impl->ts_fail.p, 0, sizeof(int), st));
  float* Aq = dA;
  if (lda != n) {
    impl->tri_pad.ensure((size_t)lda * n);
    SCL_CUDA(cudaMemsetAsync(impl->tri_pad.p, 0, (size_t)lda * n * sizeof(float), st));
    SCL_CUDA(cudaMemcpy2DAsync(impl->tri_pad.p, (size_t)lda * sizeof(float), dA, (size_t)n * sizeof(float), (size_t)n * sizeof(float),
                               (size_t)n, cudaMemcpyDeviceToDevice, st));
    Aq = impl->tri_pad.p;
  }
  if (m) {
    impl->tri_z.ensure((size_t)m * ldz);
    impl->ts_V2.ensure((size_t)n * ldv2);
    impl->ts_tau2.ensure((size_t)n * ldt2);
    SCL_CUDA(cudaMemsetAsync(impl->ts_V2.p, 0, (size_t)n * ldv2 * sizeof(float), st));
    SCL_CUDA(cudaMemsetAsync(impl->ts_tau2.p, 0, (size_t)n * ldt2 * sizeof(float), st));
  }
  SCL_CUDA(cudaEventRecord(ev[0], st));
  if (!impl->ts_aux.stream) {
    int lo = 0, hi = 0;
    SCL_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));
    SCL_CUDA(cudaStreamCreateWithPriority(&impl->ts_aux.stream, cudaStreamNonBlocking, hi));
    SCL_CUDA(cudaEventCreateWithFlags(&impl->ts_aux.ready, cudaEventDisableTiming));
    SCL_CUDA(cudaEventCreateWithFlags(&impl->ts_aux.done, cudaEventDisableTiming));
  }
  const bool half_ok = half_range_ok(Aq, n, lda, st);
  const int npanels = sy2sb_lower(Aq, n, lda, impl->ts_AB.p, impl->ts_T1.p, impl->ts_fail.p, st, &impl->ts_aux, half_ok);
  SCL_CUDA(cudaEventRecord(ev[1], st));
  sb2st(impl->ts_AB.p, n, impl->tri_d.p, impl->tri_e.p, m > 0, impl->ts_V2.p, ldv2, impl->ts_tau2.p, ldt2, st);
  SCL_CUDA(cudaEventRecord(ev[2], st));
  TridiagStats ts;
  bool ok = tridiag_eigen(impl->tri_d.p, impl->tri_e.p, n, impl->tri_w.p, dW, v0, v1, impl->tri_z.p, ldz, st, &ts);
  SCL_CUDA(cudaEventRecord(ev[3], st));
  tri_clusters = ts.clusters;
  tri_clustered = ts.clustered;
  if (ok && m) {
    apply_q2(impl->ts_V2.p, ldv2, impl->ts_tau2.p, ldt2, n, impl->tri_z.p, ldz, m, st);
    SCL_CUDA(cudaEventRecord(ev[4], st));
    apply_q1(Aq, n, lda, impl->ts_T1.p, npanels, impl->tri_z.p, ldz, m, st);
    unit_vectors(impl->tri_z.p, ldz, n, m, st);
    SCL_CUDA(cudaMemcpy2DAsync(dA + (size_t)v0 * n, (size_t)n * sizeof(float), impl->tri_z.p, (size_t)ldz * sizeof(float),
                               (size_t)n * sizeof(float), (size_t)m, cudaMemcpyDeviceToDevice, st));
  } else {
    SCL_CUDA(cudaEventRecord(ev[4], st));
  }
  SCL_CUDA(cudaEventRecord(ev[5], st));
  int fail = 0;
  SCL_CUDA(cudaMemcpyAsync(&fail, impl->ts_fail.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  for (int i = 0; i < 5; ++i) {
    float t = 0;
    cudaEventElapsedTime(&t, ev[i], ev[i + 1]);
    ts_ms[i] = t;
  }
  if (!fail && ok) {
    for (int i = 0; i < 5; ++i) ts_total[i] += ts_ms[i];
    ts_total[5] += 1.0;
    ts_total[6] += (double)m;
  }
  tri_ms[0] = ts_ms[0] + ts_ms[1];
  tri_ms[1] = ts_ms[2];
  tri_ms[2] = ts_ms[3] + ts_ms[4];
  for (auto& e : ev) cudaEventDestroy(e);
  tri_own_sytrd = true;
  tri_two_stage = true;
  if (fail || !ok) {
    ++ts_fallbacks;
    fprintf(stderr, "[scl] two-stage reduction failed (panel flag %d, tridiagonal stage %s); this solve takes the one-stage path\n", fail,
            ok ? "ok" : "failed");
    SCL_CUDA(cudaMemcpyAsync(dA, impl->ts_keep.p, nn * sizeof(float), cudaMemcpyDeviceToDevice, st));
    tri_two_stage = false;
    return syevd_tri_one_stage(dA, n, dW, v0, v1, st);
  }
  return true;
}

// Measured at n = 20 000 (all vectors / smallest half / values only): two-stage 1.71 / 1.29 / 0.62 s; one-stage (own
// tridiagonalisation + own tridiagonal stage + Sormtr) 2.42 / 2.25 / 2.03 s; Ssyevd 3.65 s on the 68k x 20k data Gram matrix.
bool Solver::syevd_tri(float* dA, int n, float* dW, int v0, int v1, cudaStream_t st) {
  SCL_REQUIRE(n >= 2 && 0 <= v0 && v0 <= v1 && v1 <= n, "bad eigenvector index range");
  tri_two_stage = false;
  if (n >= 4 * kBand && !g_force_one_stage.load(std::memory_order_relaxed)) return syevd_2stage(dA, n, dW, v0, v1, st);
  return syevd_tri_one_stage(dA, n, dW, v0, v1, st);
}

bool Solver::syevd_tri_one_stage(float* dA, int n, float* dW, int v0, int v1, cudaStream_t st) {
  const int m = v1 - v0;
  const size_t nn = (size_t)n * n;
  cudaEvent_t ev[4];
  for (auto& e : ev) SCL_CUDA(cudaEventCreate(&e));
  impl->tri_d.ensure(n); impl->tri_e.ensure(n); impl->tri_tau.ensure(n); impl->tri_w.ensure(n);
  impl->tri_keep.ensure(nn);
  if (m) impl->tri_z.ensure((size_t)m * n);
  SCL_CUDA(cudaMemcpyAsync(impl->tri_keep.p, dA, nn * sizeof(float), cudaMemcpyDeviceToDevice, st));
  // the own tridiagonalisation reads 16-byte groups of rows: a matrix whose order is not a multiple of 4 is reduced in a copy
  // with a padded leading dimension (the reflectors stay there for Sormtr)
  float* Aq = dA;
  int lda = n;
  if (n & 3) {
    lda = (n + 3) & ~3;
    impl->tri_pad.ensure((size_t)lda * n);
    SCL_CUDA(cudaMemsetAsync(impl->tri_pad.p, 0, (size_t)lda * n * sizeof(float), st));
    SCL_CUDA(cudaMemcpy2DAsync(impl->tri_pad.p, (size_t)lda * sizeof(float), dA, (size_t)n * sizeof(float), (size_t)n * sizeof(float),
                               (size_t)n, cudaMemcpyDeviceToDevice, st));
    Aq = impl->tri_pad.p;
  }
  int lw1 = 0, lw2 = 0;
  SCL_SOLVER(cusolverDnSsytrd_bufferSize(impl->h, CUBLAS_FILL_MODE_LOWER, n, Aq, lda, impl->tri_d.p, impl->tri_e.p, impl->tri_tau.p, &lw1));
  if (m)
    SCL_SOLVER(cusolverDnSormtr_bufferSize(impl->h, CUBLAS_SIDE_LEFT, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_N, n, m, Aq, lda,
                                           impl->tri_tau.p, impl->tri_z.p, n, &lw2));
  impl->work.ensure((size_t)std::max(lw1, lw2) + 1);
  SCL_CUDA(cudaEventRecord(ev[0], st));
  tri_own_sytrd = sytrd_lower(Aq, n, lda, impl->tri_d.p, impl->tri_e.p, impl->tri_tau.p, st);
  if (!tri_own_sytrd)
    SCL_SOLVER(cusolverDnSsytrd(impl->h, CUBLAS_FILL_MODE_LOWER, n, Aq, lda, impl->tri_d.p, impl->tri_e.p, impl->tri_tau.p,
                                impl->work.p, lw1, impl->info.p));
  else
    SCL_CUDA(cudaMemsetAsync(impl->info.p, 0, sizeof(int), st));
  SCL_CUDA(cudaEventRecord(ev[1], st));
  TridiagStats ts;
  bool ok = tridiag_eigen(impl->tri_d.p, impl->tri_e.p, n, impl->tri_w.p, dW, v0, v1, impl->tri_z.p, n, st, &ts);
  SCL_CUDA(cudaEventRecord(ev[2], st));
  tri_clusters = ts.clusters;
  tri_clustered = ts.clustered;
  int info = 0;
  if (ok && m) {
    SCL_SOLVER(cusolverDnSormtr(impl->h, CUBLAS_SIDE_LEFT, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_N, n, m, Aq, lda, impl->tri_tau.p,
                                impl->tri_z.p, n, impl->work.p, lw2, impl->info.p));
    SCL_CUDA(cudaMemcpyAsync(dA + (size_t)v0 * n, impl->tri_z.p, (size_t)m * n * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  SCL_CUDA(cudaEventRecord(ev[3], st));
  SCL_CUDA(cudaMemcpyAsync(&info, impl->info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  for (int i = 0; i < 3; ++i) {
    float t = 0;
    cudaEventElapsedTime(&t, ev[i], ev[i + 1]);
    tri_ms[i] = t;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  if (info != 0) ok = false;
  if (!ok) {
    // loud, not silent: counted, and reported by the timing entry points
    ++tri_fallbacks;
    fprintf(stderr, "[scl] own tridiagonal stage failed (info=%d); this solve falls back to cusolverDnSsyevd\n", info);
    SCL_CUDA(cudaMemcpyAsync(dA, impl->tri_keep.p, nn * sizeof(float), cudaMemcpyDeviceToDevice, st));
    int lwork = 0;
    const cusolverEigMode_t jobz = m ? CUSOLVER_EIG_MODE_VECTOR : CUSOLVER_EIG_MODE_NOVECTOR;
    SCL_SOLVER(cusolverDnSsyevd_bufferSize(impl->h, jobz, CUBLAS_FILL_MODE_UPPER, n, dA, n, dW, &lwork));
    impl->work.ensure((size_t)lwork);
    SCL_SOLVER(cusolverDnSsyevd(impl->h, jobz, CUBLAS_FILL_MODE_UPPER, n, dA, n, dW, impl->work.p, lwork, impl->info.p));
    SCL_CUDA(cudaMemcpyAsync(&info, impl->info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    if (info != 0) throw Error(-3, "cusolverDnSsyevd did not converge, info=" + std::to_string(info));
  }
  return ok;
}

// A (n x n, symmetric, full) is overwritten by the eigenvectors when vectors=true.
void Solver::syevd(float* dA, int n, float* dW, bool vectors, cudaStream_t st) { syevd_tri(dA, n, dW, 0, vectors ? n : 0, st); }

void Solver::dsyevd_small(double* dA, int n, double* dW, cudaStream_t st) {
  int lwork = 0;
  SCL_SOLVER(cusolverDnDsyevd_bufferSize(impl->h, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, n, dA, n, dW, &lwork));
  impl->dwork.ensure((size_t)lwork);
  SCL_SOLVER(cusolverDnDsyevd(impl->h, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, n, dA, n, dW, impl->dwork.p,
                              lwork, impl->info.p));
  int info = 0;
  SCL_CUDA(cudaMemcpyAsync(&info, impl->info.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  if (info != 0) throw Error(-3, "cusolverDnDsyevd did not converge, info=" + std::to_string(info));
}

double Solver::bench(float* dA, int n, float* dW, int mode, int il, int iu, cudaStream_t st) {
  cudaEvent_t e0, e1;
  SCL_CUDA(cudaEventCreate(&e0));
  SCL_CUDA(cudaEventCreate(&e1));
  int info = 0;
  if (mode == 0 || mode == 1) {
    const cusolverEigMode_t jobz = mode == 0 ? CUSOLVER_EIG_MODE_VECTOR : CUSOLVER_EIG_MODE_NOVECTOR;
    int lwork = 0;
    SCL_SOLVER(cusolverDnSsyevd_bufferSize(impl->h, jobz, CUBLAS_FILL_MODE_UPPER, n, dA, n, dW, &lwork));
    impl->work.ensure((size_t)lwork);
    SCL_CUDA(cudaEventRecord(e0, st));
    SCL_SOLVER(cusolverDnSsyevd(impl->h, jobz, CUBLAS_FILL_MODE_UPPER, n, dA, n, dW, impl->work.p, lwork, impl->info.p));
  } else if (mode == 2) {
    int lwork = 0, meig = 0;
    SCL_SOLVER(cusolverDnSsyevdx_bufferSize(impl->h, CUSOLVER_EIG_MODE_VECTOR, CUSOLVER_EIG_RANGE_I, CUBLAS_FILL_MODE_UPPER, n,
                                            dA, n, 0.f, 0.f, il, iu, &meig, dW, &lwork));
    impl->work.ensure((size_t)lwork);
    SCL_CUDA(cudaEventRecord(e0, st));
    SCL_SOLVER(cusolverDnSsyevdx(impl->h, CUSOLVER_EIG_MODE_VECTOR, CUSOLVER_EIG_RANGE_I, CUBLAS_FILL_MODE_UPPER, n, dA, n,
                                 0.f, 0.f, il, iu, &meig, dW, impl->work.p, lwork, impl->info.p));
  } else if (mode == 9) {
    // own tridiagonalisation (sytrd.cu) alone
    Tmp<float> d(n, st), e(n, st), tau(n, st);
    SCL_CUDA(cudaEventRecord(e0, st));
    if (!sytrd_lower(dA, n, n, d.p, e.p, tau.p, st)) throw Error(-1, "sytrd_lower does not handle this size (order must be a multiple of 4 here)");
    SCL_CUDA(cudaMemsetAsync(impl->info.p, 0, sizeof(int), st));
  } else if (mode >= 6 && mode <= 8) {
    // own tridiagonal stage: 6 = all vectors, 7 = vectors il..iu (1-based inclusive), 8 = values only
    const int v0 = mode == 7 ? il - 1 : 0, v1 = mode == 6 ? n : (mode == 7 ? iu : 0);
    SCL_CUDA(cudaEventRecord(e0, st));
    syevd_tri(dA, n, dW, v0, v1, st);
  } else if (mode == 4 || mode == 5) {
    // the two library halves of a one-stage solve, timed apart: 4 = Ssytrd (tridiagonalisation) alone, 5 = Sormtr
    // (back-transformation of an n x n block by the reflectors of a previous Ssytrd) alone
    Tmp<float> d(n, st), e(n, st), tau(n, st);
    int lw1 = 0, lw2 = 0;
    SCL_SOLVER(cusolverDnSsytrd_bufferSize(impl->h, CUBLAS_FILL_MODE_LOWER, n, dA, n, d.p, e.p, tau.p, &lw1));
    Tmp<float> Cm(mode == 5 ? (size_t)n * n : 1, st);
    if (mode == 5)
      SCL_SOLVER(cusolverDnSormtr_bufferSize(impl->h, CUBLAS_SIDE_LEFT, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_N, n, n, dA, n, tau.p,
                                             Cm.p, n, &lw2));
    impl->work.ensure((size_t)std::max(lw1, lw2));
    if (mode == 4) SCL_CUDA(cudaEventRecord(e0, st));
    SCL_SOLVER(cusolverDnSsytrd(impl->h, CUBLAS_FILL_MODE_LOWER, n, dA, n, d.p, e.p, tau.p, impl->work.p, lw1, impl->info.p));
    if (mode == 5) {
      SCL_CUDA(cudaMemsetAsync(Cm.p, 0, (size_t)n * n * sizeof(float), st));
      SCL_CUDA(cudaEventRecord(e0, st));
      SCL_SOLVER(cusolverDnSormtr(impl->h, CUBLAS_SIDE_LEFT, CUBLAS_FILL_MODE_LOWER, CUBLAS_OP_N, n, n, dA, n, tau.p, Cm.p, n,
                                  impl->work.p, lw2, impl->info.p));
      SCL_CUDA(cudaEventRecord(e1, st));
      SCL_CUDA(cudaEventSynchronize(e1));
    }
  } else {
    cusolverDnParams_t params = nullptr;
    SCL_SOLVER(cusolverDnCreateParams(&params));
    size_t wd = 0, wh = 0;
    SCL_SOLVER(cusolverDnXsyevd_bufferSize(impl->h, params, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, (int64_t)n,
                                           CUDA_R_32F, dA, (int64_t)n, CUDA_R_32F, dW, CUDA_R_32F, &wd, &wh));
    impl->work.ensure(wd / sizeof(float) + 1);
    std::vector<unsigned char> hbuf(wh + 1);
    SCL_CUDA(cudaEventRecord(e0, st));
    SCL_SOLVER(cusolverDnXsyevd(impl->h, params, CUSOLVER_EIG_MODE_VECTOR, CUBLAS_FILL_MODE_UPPER, (int64_t)n, CUDA_R_32F, dA,
                                (int64_t)n, CUDA_R_32F, dW, CUDA_R_32F, impl->work.p, wd, hbuf.data(), wh, impl->info.p));
    SCL_CUDA(cudaEventRecord(e1, st));
    SCL_CUDA(cudaEventSynchronize(e1));   // the host buffer must outlive the call
    cusolverDnDestroyParams(params);
  }
  SCL_CUDA(cudaEventRecord(e1, st));
  SCL_CUDA(cudaEventSynchronize(e1));
  float ms = 0;
  SCL_CUDA(cudaEventElapsedTime(&ms, e0, e1));
  SCL_CUDA(cudaMemcpy(&info, impl->info.p, sizeof(int), cudaMemcpyDeviceToHost));
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  if (info != 0) throw Error(-3, "eigensolver timing study: info=" + std::to_string(info));
  return (double)ms;
}

// ---- Marchenko-Pastur / Tracy-Widom (host, Float64 on the Float32 eigenvalues) ------------
namespace {
struct MpParams {
  double m1, m2, gamma, b_plus, b_minus;
};
MpParams mp_parameters(const std::vector<double>& L) {   // _mp_parameters :390-408
  MpParams p{};
  double s1 = 0, s2 = 0;
  for (double v : L) { s1 += v; s2 += v * v; }
  const double n = (double)L.size();
  p.m1 = s1 / n;
  p.m2 = s2 / n;
  p.gamma = p.m2 / (p.m1 * p.m1) - 1.0;
  const double sg = std::sqrt(p.gamma);
  p.b_plus = p.m1 * (1 + sg) * (1 + sg);
  p.b_minus = p.m1 * (1 - sg) * (1 - sg);
  return p;
}
std::vector<double> window(const std::vector<double>& L, double lo, double hi) {
  std::vector<double> out;
  for (double v : L)
    if (lo < v && v < hi) out.push_back(v);   // strict both sides (:431)
  return out;
}
}  // namespace

MpFit mp_fit(const float* L, int nL, const float* Lr, int nLr) {
  SCL_REQUIRE(nL > 1 && nLr > 1, "too few eigenvalues for the MP fit");
  std::vector<double> Ld(L, L + nL), Lrd(Lr, Lr + nLr);
  MpFit out{};
  // _mp_calculation :424-459
  MpParams pr = mp_parameters(Lrd);
  double b_plus = pr.b_plus, b_minus = pr.b_minus;
  std::vector<double> Lu = window(Ld, b_minus, b_plus);
  SCL_REQUIRE(!Lu.empty(), "no eigenvalue inside the null-matrix MP window");
  MpParams q = mp_parameters(Lu);
  double new_b_plus = q.b_plus, new_b_minus = q.b_minus;
  int iter = 0;
  const double eps = 1e-6, eta = 1.0;
  const int max_iter = 10000;
  while (true) {
    double loss = (1 - new_b_plus / b_plus) * (1 - new_b_plus / b_plus);
    ++iter;
    if (loss <= eps || iter == max_iter) break;
    double gradient = new_b_plus - b_plus;
    new_b_plus = b_plus + eta * gradient;
    Lu = window(Ld, new_b_minus, new_b_plus);
    b_plus = new_b_plus;
    b_minus = new_b_minus;
    SCL_REQUIRE(!Lu.empty(), "MP window became empty");
    q = mp_parameters(Lu);
    new_b_plus = q.b_plus;
    new_b_minus = q.b_minus;
  }
  out.b_plus = new_b_plus;
  out.b_minus = new_b_minus;
  out.iters = iter;
  for (int i = 0; i < nL; ++i)
    if (new_b_minus < (double)L[i] && (double)L[i] < new_b_plus) out.L_mp.push_back(L[i]);
  SCL_REQUIRE(out.L_mp.size() > 1, "MP fit selected fewer than two eigenvalues");
  // _tw :461-467
  std::vector<double> Lmpd(out.L_mp.begin(), out.L_mp.end());
  MpParams pm = mp_parameters(Lmpd);
  const double gamma = pm.gamma;
  const double p = (double)nL / gamma;
  const double sigma = 1.0 / std::pow(p, 2.0 / 3.0) * std::pow(gamma, 5.0 / 6.0) * std::pow(1 + std::sqrt(gamma), 4.0 / 3.0);
  out.lambda_c = pm.m1 * (1 + std::sqrt(gamma)) * (1 + std::sqrt(gamma)) + sigma;
  out.gamma = gamma;
  out.n_signal = 0;
  for (int i = 0; i < nL; ++i)
    if ((double)L[i] > out.lambda_c) ++out.n_signal;   // strict (:541)
  // mp_check :469-487
  {
    double mn = *std::min_element(Lmpd.begin(), Lmpd.end()) - 1, mx = *std::max_element(Lmpd.begin(), Lmpd.end()) + 1;
    const int nb = 99;
    std::vector<double> edges(nb + 1), cnt(nb, 0.0);
    for (int i = 0; i <= nb; ++i) edges[i] = mn + (mx - mn) * (double)i / (double)nb;
    for (double v : Lmpd) {
      int b = (int)std::floor((v - mn) / (mx - mn) * nb);
      b = std::max(0, std::min(nb - 1, b));
      // guard the floating-point edge: bin i is [e_i, e_i+1)
      while (b > 0 && v < edges[b]) --b;
      while (b < nb - 1 && v >= edges[b + 1]) ++b;
      cnt[b] += 1;
    }
    const double tot = (double)Lmpd.size();
    double acc = 0, acc2 = 0, D = 0;
    std::vector<double> c2(nb);
    const double sg = std::sqrt(pm.gamma);
    (void)sg;
    for (int i = 0; i < nb; ++i) {
      double x = 0.5 * (edges[i] + edges[i + 1]);
      double pdf = 0;
      if (pm.b_minus < x && x < pm.b_plus)
        pdf = std::sqrt((pm.b_plus - x) * (x - pm.b_minus)) / (2 * pm.m1 * M_PI * pm.gamma * x);
      acc2 += pdf;
      c2[i] = acc2;
    }
    const double mxc = *std::max_element(c2.begin(), c2.end());
    for (int i = 0; i < nb; ++i) {
      acc += cnt[i] / tot;
      D = std::max(D, std::fabs(acc - c2[i] / mxc));
    }
    const double c_alpha = std::sqrt(-0.5 * std::log(0.05));
    out.ks_static = D;
    out.pass = D <= c_alpha * std::sqrt((double)(nb + nb) / nb / nb);
  }
  return out;
}

}  // namespace scl
