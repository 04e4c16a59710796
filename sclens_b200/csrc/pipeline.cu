// Orchestration of the sclens() path on one GPU (src/scLENS.jl:649-832): everything between
// "counts in" and "results out" stays device-resident.  Stage boundaries follow the
// reference: run_signal == :664-706, run_robustness == :709-819.
#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include "nccl_dyn.h"
#include "handle.h"
#include "tmp.cuh"

namespace scl {

std::atomic<long long> g_kernel_launches{0};

void Prof::resolve() {
  for (auto& e : pending) {
    cudaEventSynchronize(e.b);
    float t = 0;
    cudaEventElapsedTime(&t, e.a, e.b);
    ms[e.kind] += t;
    calls[e.kind] += 1;
    cudaEventDestroy(e.a);
    cudaEventDestroy(e.b);
  }
  pending.clear();
}
void Prof::reset() {
  resolve();
  *this = Prof();
}

namespace {

inline size_t round8(size_t x) { return (x + 7) / 8 * 8; }

// Unit vectors in dimension n have entries ~1/sqrt(n); scaled by 2^10 before the binary16 hi/lo split their
// low-order parts stay normal numbers (|entry| <= 1 -> <= 1024, far below 65504).  Undone through alpha.
constexpr float kUnitScale = 1024.f;

#define SCL_NCCL(x)                                                                                   \
  do {                                                                                                \
    ncclResult_t r_ = (x);                                                                            \
    if (r_ != ncclSuccess) throw scl::Error(SCL_ERR_NCCL, std::string(#x) + ": " + nccl_api().GetErrorString(r_)); \
  } while (0)

inline bool multi(const scl_handle* h) { return h->world > 1 && h->nccl != nullptr; }

struct Timer {
  cudaEvent_t a, b;
  cudaStream_t st;
  explicit Timer(cudaStream_t s) : st(s) {
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, st);
  }
  ~Timer() {
    cudaEventDestroy(a);
    cudaEventDestroy(b);
  }
  double stop() {
    cudaEventRecord(b, st);
    cudaEventSynchronize(b);
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventRecord(a, st);
    return ms;
  }
};

// rows of `src` (stride ld_src, may be negative to walk backwards) -> dst rows (stride ld_dst)
__global__ void k_copy_rows(const float* __restrict__ src, long long ld_src, float* __restrict__ dst, long long ld_dst,
                            int rows, int cols) {
  for (int r = blockIdx.y; r < rows; r += gridDim.y)
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < cols; c += gridDim.x * blockDim.x)
      dst[(long long)r * ld_dst + c] = src[(long long)r * ld_src + c];
}

__global__ void k_gather_rows(const float* __restrict__ src, const int* __restrict__ row_idx, float* __restrict__ dst,
                              int rows, long long cols) {
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    const float* s = src + (long long)row_idx[r] * cols;
    for (long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x; c < cols; c += (long long)gridDim.x * blockDim.x)
      dst[(long long)r * cols + c] = s[c];
  }
}

// unit-normalise every row (one block per row), Float64 accumulation  (mapslices(s -> s/norm(s)) :505, :558)
__global__ void __launch_bounds__(256) k_normalize_rows(float* __restrict__ a, int rows, long long cols) {
  __shared__ double red[8];
  for (int r = blockIdx.x; r < rows; r += gridDim.x) {
    float* p = a + (long long)r * cols;
    double s = 0;
    for (long long c = threadIdx.x; c < cols; c += blockDim.x) s += (double)p[c] * (double)p[c];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
    __syncthreads();
    double t = 0;
    for (int w = 0; w < 8; ++w) t += red[w];
    const float inv = (float)(1.0 / sqrt(t));
    for (long long c = threadIdx.x; c < cols; c += blockDim.x) p[c] *= inv;
  }
}

void copy_rows(const float* src, long long ld_src, float* dst, long long ld_dst, int rows, int cols, cudaStream_t st) {
  if (!rows) return;
  count_launches(1);
  dim3 grid((unsigned)std::min((cols + 255) / 256, 64), (unsigned)std::min(rows, 65535));
  k_copy_rows<<<grid, 256, 0, st>>>(src, ld_src, dst, ld_dst, rows, cols);
  SCL_CUDA(cudaGetLastError());
}

void normalize_rows(float* a, int rows, long long cols, cudaStream_t st) {
  if (!rows) return;
  count_launches(1);
  k_normalize_rows<<<std::min(rows, 148 * 8), 256, 0, st>>>(a, rows, cols);
  SCL_CUDA(cudaGetLastError());
}

int cta_group_of(const scl_handle* h) { return h->cfg.cta_group == 1 ? 1 : 2; }

// number of split-K partitions that fills the machine for a GEMM with `tiles` output tiles
int pick_splits(int tiles, int64_t K, int cta_group) {
  int units = sm_count() / cta_group;
  int kblocks = (int)((K + 63) / 64);
  int s = std::max(1, units / std::max(1, tiles));
  return std::max(1, std::min(s, std::max(1, kblocks / 4)));
}

// C (fp32, host-visible layout given by epi) = alpha * A * B^T through split-K partials.
void gemm_splitk(scl_handle* h, const GemmOperand& A, const GemmOperand& B, bool syrk, float alpha, Epilogue epi,
                 float* dC, int64_t ldc, size_t c_elems) {
  const int cg = cta_group_of(h);
  const int tile_m = 128 * cg;
  const int tiles = ((A.rows + tile_m - 1) / tile_m) * ((B.rows + 255) / 256);
  const int splits = pick_splits(tiles, A.K, cg);
  GemmArgs g;
  g.A = A; g.B = B; g.syrk = syrk; g.epi = epi; g.ldc = ldc; g.cta_group = cg;
  ProfScope ps(&h->prof, h->st, PK_OTHER_GEMM);
  h->prof.other_gemm_flops += 2.0 * A.rows * (double)B.rows * (double)A.K;
  if (splits == 1) {
    g.alpha = alpha; g.C = dC; g.splits = 1;
    gemm_umma(g, h->st);
    return;
  }
  Tmp<float> part((size_t)splits * c_elems, h->st);
  SCL_CUDA(cudaMemsetAsync(part.p, 0, (size_t)splits * c_elems * sizeof(float), h->st));
  g.alpha = 1.f; g.C = part.p; g.splits = splits; g.split_stride = (int64_t)c_elems;
  gemm_umma(g, h->st);
  reduce_splits(part.p, splits, (int64_t)c_elems, c_elems, alpha, dC, h->st);
}

// ---- calibration of the tensor core's accumulation bias -----------------------------------
// tcgen05 accumulates in FP32 with truncation: every partial sum is pulled towards zero, so a Gram matrix
// comes out as (1 - delta) * G with delta ~ 3e-8 per MMA of the accumulation chain (measured, profiles/
// r1_diag_eig_error_*.txt), uniformly over the off-diagonal entries.  Together with the exact Float64 diagonal
// that is a relative diagonal excess delta, which moves an eigenvalue by delta * (mean diagonal - lambda) - ten
// times delta at the lower Marchenko-Pastur edge.  delta is measured per Gram matrix from kCalibSamples
// off-diagonal entries evaluated exactly (Float64 dot products of the binary16 operand rows); the diagonal is
// scaled by (1 - delta) so the whole matrix carries one common factor, which is divided out of the eigenvalues.
// (kCalibSamples: handle.h)

__device__ __forceinline__ void calib_pair(int s, int rows, int& i, int& j) {
  uint64_t h = (uint64_t)(s + 1) * 0x9E3779B97F4A7C15ull;
  h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32;
  i = (int)((h & 0xffffffffull) % (uint64_t)rows);
  j = (int)((h >> 32) % (uint64_t)(rows - 1));
  if (j >= i) ++j;   // j != i
}

// ex[s] = sum_k a_i[k] a_j[k] over [k0, k0 + Ks) exactly as the tensor core would form it without rounding
// (hi*hi, plus hi*lo + lo*hi in split mode); rows are zero padded up to a multiple of 8 elements
__global__ void __launch_bounds__(256) k_sample_dots(const __half* __restrict__ hi, const __half* __restrict__ lo,
                                                     long long ld, long long k0, long long Ks, int rows,
                                                     double* __restrict__ ex) {
  __shared__ double red[8];
  int i, j;
  calib_pair(blockIdx.x, rows, i, j);
  const __half* ai = hi + (long long)i * ld + k0;
  const __half* aj = hi + (long long)j * ld + k0;
  const __half* li = lo ? lo + (long long)i * ld + k0 : nullptr;
  const __half* lj = lo ? lo + (long long)j * ld + k0 : nullptr;
  const long long n8 = (Ks + 7) / 8;
  double acc = 0;
  for (long long c = threadIdx.x; c < n8; c += blockDim.x) {
    const uint4 u = *reinterpret_cast<const uint4*>(ai + c * 8), v = *reinterpret_cast<const uint4*>(aj + c * 8);
    const __half2* x = reinterpret_cast<const __half2*>(&u);
    const __half2* y = reinterpret_cast<const __half2*>(&v);
    uint4 ul = make_uint4(0, 0, 0, 0), vl = ul;
    if (lo) { ul = *reinterpret_cast<const uint4*>(li + c * 8); vl = *reinterpret_cast<const uint4*>(lj + c * 8); }
    const __half2* xl = reinterpret_cast<const __half2*>(&ul);
    const __half2* yl = reinterpret_cast<const __half2*>(&vl);
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float2 a = __half22float2(x[q]), b = __half22float2(y[q]);
      acc += (double)a.x * (double)b.x + (double)a.y * (double)b.y;
      if (lo) {
        const float2 al = __half22float2(xl[q]), bl = __half22float2(yl[q]);
        acc += (double)a.x * (double)bl.x + (double)al.x * (double)b.x + (double)a.y * (double)bl.y + (double)al.y * (double)b.y;
      }
    }
  }
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0;
    for (int w = 0; w < 8; ++w) t += red[w];
    ex[blockIdx.x] = t;
  }
}

// factor[0] = 1 + least-squares slope of (G_tc - G_exact) on G_exact over the samples  (= 1 - delta)
__global__ void __launch_bounds__(256) k_fit_shrink(const float* __restrict__ G, int n, double inv_scale,
                                                    const double* __restrict__ ex, int S, double* __restrict__ factor) {
  __shared__ double rx[8], ry[8];
  double sxx = 0, sxy = 0;
  for (int s = threadIdx.x; s < S; s += blockDim.x) {
    int i, j;
    calib_pair(s, n, i, j);
    const double e = ex[s], t = (double)G[(size_t)i * n + j] * inv_scale;
    sxx += e * e;
    sxy += (t - e) * e;
  }
  for (int o = 16; o; o >>= 1) { sxx += __shfl_xor_sync(0xffffffffu, sxx, o); sxy += __shfl_xor_sync(0xffffffffu, sxy, o); }
  if ((threadIdx.x & 31) == 0) { rx[threadIdx.x >> 5] = sxx; ry[threadIdx.x >> 5] = sxy; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int w = 0; w < 8; ++w) { a += rx[w]; b += ry[w]; }
    double f = a > 0 ? 1.0 + b / a : 1.0;
    if (!(f > 0.999 && f < 1.001)) f = 1.0;   // a bias this large is not the effect being calibrated
    factor[0] = f;
  }
}

__global__ void k_scale_diagonal(float* __restrict__ G, int n, const double* __restrict__ factor) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) G[(size_t)i * n + i] = (float)((double)G[(size_t)i * n + i] * factor[0]);
}

__global__ void k_unscale_values(float* __restrict__ w, int n, const double* __restrict__ factor) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) w[i] = (float)((double)w[i] / factor[0]);
}

// lower triangle (row r: columns 0..r) of an n x n matrix <-> packed array of n(n+1)/2 floats.  The partial Gram
// matrices of the ranks travel packed (SURVEY.md 8e): half the bytes of the square over NVLink.
__global__ void k_pack_lower(const float* __restrict__ G, int n, float* __restrict__ P) {
  for (int r = blockIdx.y; r < n; r += gridDim.y) {
    const float* src = G + (size_t)r * n;
    float* dst = P + (size_t)r * (r + 1) / 2;
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c <= r; c += gridDim.x * blockDim.x) dst[c] = src[c];
  }
}
// square tiles: element (r, c), r >= c, is written to (r, c) and (c, r) through a padded shared-memory transpose
__global__ void __launch_bounds__(256) k_unpack_lower_mirror(const float* __restrict__ P, int n, float* __restrict__ G) {
  __shared__ float t[32][33];
  const int tr = blockIdx.y, tc = blockIdx.x;
  if (tc > tr) return;
  const int r0 = tr * 32, c0 = tc * 32, tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  for (int i = ty; i < 32; i += 8) {
    const int r = r0 + i, c = c0 + tx;
    float v = 0.f;
    if (r < n && c <= r) {
      v = P[(size_t)r * (r + 1) / 2 + c];
      G[(size_t)r * n + c] = v;
    }
    t[i][tx] = v;
  }
  __syncthreads();
  for (int i = ty; i < 32; i += 8) {
    const int c = c0 + i, r = r0 + tx;   // mirrored element (c, r) = value at (r, c)
    if (r < n && c < r) G[(size_t)c * n + r] = t[tx][i];
  }
}

double quantile7(const std::vector<double>& sorted, double p) {
  const size_t n = sorted.size();
  if (n == 1) return sorted[0];
  double hh = (double)(n - 1) * p;
  size_t lo = (size_t)std::floor(hh);
  if (lo >= n - 1) return sorted[n - 1];
  return sorted[lo] + (hh - (double)lo) * (sorted[lo + 1] - sorted[lo]);
}

}  // namespace

// The three calibration steps of gram_of(), shared with scl_debug_gram_calibrated.
// ex[s] = exact dot product of sample pair s over the operand columns [k0, k0 + Ks) (hi, plus the cross terms with lo)
void calib_sample_dots(const __half* hi, const __half* lo, long long ld, long long k0, long long Ks, int rows, double* ex,
                       cudaStream_t st) {
  count_launches(1);
  k_sample_dots<<<kCalibSamples, 256, 0, st>>>(hi, lo, ld, k0, Ks, rows, ex);
  SCL_CUDA(cudaGetLastError());
}
// factor[0] = 1 - delta from the samples of G (= scale * operand operand'), 1 when the fit falls outside (0.999, 1.001)
void calib_fit(const float* G, int n, float scale, const double* ex, double* factor, cudaStream_t st) {
  count_launches(1);
  k_fit_shrink<<<1, 256, 0, st>>>(G, n, 1.0 / (double)scale, ex, kCalibSamples, factor);
  SCL_CUDA(cudaGetLastError());
}
// G[i][i] *= factor[0]: the exact diagonal takes the common factor of the tensor-core off-diagonal
void calib_scale_diagonal(float* G, int n, const double* factor, cudaStream_t st) {
  count_launches(1);
  k_scale_diagonal<<<(n + 255) / 256, 256, 0, st>>>(G, n, factor);
  SCL_CUDA(cudaGetLastError());
}

// Contraction-axis block of rank `rank`: whole 64-element k-blocks, ceil(kblocks / world) per rank, the last rank also
// takes the zero padding up to ld.  Blocks are disjoint and cover [0, ld); a rank beyond the data gets an empty block.
void plan_gram_shard(int64_t K, int64_t ld, int world, int rank, int64_t* k0, int64_t* k1) {
  const int64_t kblocks = (K + 63) / 64, per = (kblocks + world - 1) / world;
  *k0 = std::min<int64_t>(ld, (int64_t)rank * per * 64);     // clamped to ld (a multiple of 8), never to K: a rank whose
  *k1 = std::min<int64_t>(ld, (int64_t)(rank + 1) * per * 64);  // block starts beyond the data gets the empty block [ld, ld)
  if (rank == world - 1) *k1 = ld;
}

// ---------------------------------------------------------------------------------------
// normalise A and form its Wishart matrix on the smaller side:  dG = operand * operand^T * scale
void gram_of(scl_handle* h, const SpMat& A, NormStats& S, DBuf<__half>& hi, DBuf<__half>& lo, float* dG, int nm,
             float scale, bool split, bool shard, int reduce_root) {
  const bool gene_side = A.N > A.M;                 // contract over cells (N > M) or over genes
  {
    ProfScope ps(&h->prof, h->st, PK_STATS);
    S.centering = h->cfg.centering;
    compute_norm_stats(A, S, h->st);
    ensure_patch(A, S, gene_side ? 0 : 1, h->st);
    h->prof.stats_alg_bytes += 40.0 * (double)A.nnz;   // 4 nnz (row sums) + 3 x 8 nnz + 12 nnz (patch pass)
    h->prof.stats_norms += 1;
  }
  const int rows = gene_side ? A.M : A.N;
  const int64_t K = gene_side ? A.N : A.M;
  const size_t ld = round8((size_t)K);
  SCL_REQUIRE(rows == nm, "Gram size mismatch");
  // Multi-GPU: rank g owns the g-th block of the contraction axis (a cell block when N > M).  It densifies and
  // contracts only that block - the operand buffer holds just that slice (rows x (k1 - k0)) - and the partial Gram
  // matrices are summed over NVLink (SURVEY.md 8e).
  int64_t k0 = 0, k1 = (int64_t)ld;
  const bool sharded = shard && multi(h);
  if (sharded) plan_gram_shard(K, (int64_t)ld, h->world, h->rank, &k0, &k1);
  const bool have_work = k1 > k0;
  const size_t lds = sharded ? (size_t)std::max<int64_t>(8, k1 - k0) : ld;   // row stride of the operand buffer
  hi.ensure((size_t)rows * lds);
  if (split) lo.ensure((size_t)rows * lds);
  // exact Gram diagonal: the tensor core's truncating FP32 accumulation biases long same-sign sums low; the
  // diagonal (the only systematically same-sign sum) comes from the statistics passes in Float64 instead
  if (have_work) {
    {
      ProfScope ps(&h->prof, h->st, PK_DENSIFY);
      densify(A, S, gene_side ? 0 : 1, ld, hi.p, split ? lo.p : nullptr, h->st, k0, k1, sharded ? lds : 0);
      const double frac = (double)(k1 - k0) / (double)ld;
      h->prof.densify_alg_bytes += frac * (8.0 * (double)A.nnz + (double)A.N * A.M * (split ? 4.0 : 2.0)) + 4.0 * (A.M + 1);
    }
    const int64_t Ks = std::min<int64_t>(K, k1) - k0;
    GemmArgs g;
    const int64_t o0 = sharded ? 0 : k0;   // a slice buffer starts at the rank's first position
    g.A.hi = hi.p + o0; g.A.lo = split ? lo.p + o0 : nullptr; g.A.rows = rows; g.A.K = Ks; g.A.ld = (int64_t)lds;
    g.B = g.A;
    g.syrk = true;
    g.alpha = scale;
    g.C = dG;
    g.ldc = nm;
    g.cta_group = cta_group_of(h);
    g.chunk_kb = h->cfg.gram_chunk_kb;
    {
      ProfScope ps(&h->prof, h->st, PK_GRAM_GEMM);
      gemm_umma(g, h->st);
      h->prof.gram_alg_flops += (double)rows * (rows + 1.0) * (double)Ks;
    }
  } else {
    SCL_CUDA(cudaMemsetAsync(dG, 0, (size_t)nm * nm * sizeof(float), h->st));
  }
  // exact values of the calibration samples over this rank's part of the contraction
  const bool calibrate = h->cfg.gram_tc_diag == 0 && nm >= 64;
  Tmp<double> ex(kCalibSamples, h->st);
  h->gram_factor.ensure(4);
  if (calibrate) {
    ProfScope ps(&h->prof, h->st, PK_SMALL);
    if (have_work)
      calib_sample_dots(hi.p, split ? lo.p : nullptr, (long long)lds, (long long)(sharded ? 0 : k0),
                        (long long)(std::min<int64_t>(K, k1) - k0), rows, ex.p, h->st);
    else
      SCL_CUDA(cudaMemsetAsync(ex.p, 0, kCalibSamples * sizeof(double), h->st));
  }
  if (sharded) {
    // packed lower triangle, summed in FP32 (rank order fixed by NCCL's algorithm choice for a given world size); to the
    // one rank that solves this matrix when the caller names it, to every rank otherwise
    ProfScope ps(&h->prof, h->st, PK_COMM);
    const size_t np = (size_t)nm * (nm + 1) / 2;
    Tmp<float> packed(np, h->st);
    count_launches(2);
    k_pack_lower<<<dim3(8, (unsigned)std::min(nm, 16384)), 256, 0, h->st>>>(dG, nm, packed.p);
    SCL_CUDA(cudaGetLastError());
    if (reduce_root >= 0) {
      SCL_NCCL(nccl_api().Reduce(packed.p, packed.p, np, ncclFloat, ncclSum, reduce_root, (ncclComm_t)h->nccl, h->st));
      if (calibrate) SCL_NCCL(nccl_api().Reduce(ex.p, ex.p, kCalibSamples, ncclDouble, ncclSum, reduce_root, (ncclComm_t)h->nccl, h->st));
    } else {
      SCL_NCCL(nccl_api().AllReduce(packed.p, packed.p, np, ncclFloat, ncclSum, (ncclComm_t)h->nccl, h->st));
      if (calibrate) SCL_NCCL(nccl_api().AllReduce(ex.p, ex.p, kCalibSamples, ncclDouble, ncclSum, (ncclComm_t)h->nccl, h->st));
    }
    const unsigned nt = (unsigned)((nm + 31) / 32);
    k_unpack_lower_mirror<<<dim3(nt, nt), 256, 0, h->st>>>(packed.p, nm, dG);
    SCL_CUDA(cudaGetLastError());
    h->prof.comm_bytes += 4.0 * (double)np + (calibrate ? 8.0 * kCalibSamples : 0.0);
  }
  // every rank holds the complete statistics, so the full-length diagonal is written after the reduction
  if (h->cfg.gram_tc_diag != 1) {
    ProfScope ps(&h->prof, h->st, PK_STATS);
    set_gram_diagonal(dG, nm, gram_diagonal(A, S, gene_side, h->st), (double)scale, h->st);
  }
  if (calibrate) {
    ProfScope ps(&h->prof, h->st, PK_SMALL);
    calib_fit(dG, nm, scale, ex.p, h->gram_factor.p, h->st);
    calib_scale_diagonal(dG, nm, h->gram_factor.p, h->st);
  } else {
    const double one = 1.0;
    SCL_CUDA(cudaMemcpyAsync(h->gram_factor.p, &one, sizeof(double), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  }
}

// eigenvalues of the matrix gram_of() produced last (slot 0) or of one whose factor was saved -> eigenvalues of the Gram
// matrix itself
void unscale_eigenvalues(scl_handle* h, float* dW, int n, int slot = 0) {
  count_launches(1);
  k_unscale_values<<<(n + 255) / 256, 256, 0, h->st>>>(dW, n, h->gram_factor.p + slot);
  SCL_CUDA(cudaGetLastError());
}
// keep the factor of the Gram matrix gram_of() produced last while other matrices are formed (slots 1..3)
void save_gram_factor(scl_handle* h, int slot) {
  SCL_CUDA(cudaMemcpyAsync(h->gram_factor.p + slot, h->gram_factor.p, sizeof(double), cudaMemcpyDeviceToDevice, h->st));
}

// d[j] = max_i |<V_i, W_j>|  (:742) with V pre-converted to binary16 hi/lo rows
static void corr_colabsmax_pre(scl_handle* h, const GemmOperand& V, const float* dW, int nw, int n, float* d_out) {
  const size_t ld = (size_t)V.ld;
  Tmp<__half> w_hi((size_t)nw * ld, h->st), w_lo((size_t)nw * ld, h->st);
  strided_split_f32_to_f16(dW, nw, n, n, (int64_t)ld, w_hi.p, w_lo.p, h->st, kUnitScale);
  SCL_CUDA(cudaMemsetAsync(d_out, 0, (size_t)nw * sizeof(float), h->st));
  GemmArgs g;
  g.alpha = 1.f / (kUnitScale * kUnitScale);
  g.A = V;
  g.B.hi = w_hi.p; g.B.lo = w_lo.p; g.B.rows = nw; g.B.K = n; g.B.ld = (int64_t)ld;
  g.epi = Epilogue::ColAbsMax;
  g.C = d_out;
  g.ldc = 0;
  g.cta_group = cta_group_of(h);
  ProfScope ps(&h->prof, h->st, PK_OTHER_GEMM);
  gemm_umma(g, h->st);
  h->prof.other_gemm_flops += 2.0 * V.rows * (double)nw * n;
}

void corr_colabsmax(scl_handle* h, const float* dV, int nv, const float* dW, int nw, int n, float* d_out) {
  const size_t ld = round8((size_t)n);
  Tmp<__half> v_hi((size_t)nv * ld, h->st), v_lo((size_t)nv * ld, h->st);
  strided_split_f32_to_f16(dV, nv, n, n, (int64_t)ld, v_hi.p, v_lo.p, h->st, kUnitScale);
  GemmOperand V;
  V.hi = v_hi.p; V.lo = v_lo.p; V.rows = nv; V.K = n; V.ld = (int64_t)ld;
  corr_colabsmax_pre(h, V, dW, nw, n, d_out);
}

// out[k][N] = normalise_rows( Vk[k][M] * Xtilde^T )  i.e. columns X*v / |X*v|  (:503-505, :556-558)
// dVrows: pointer to the first wanted eigenvector, ld_v elements between consecutive wanted ones
static void back_project(scl_handle* h, const SpMat& A, NormStats& S, const float* dVrows, long long ld_v, int k,
                         float* d_out) {
  const int N = A.N, M = A.M;
  const size_t ldm = round8((size_t)M);
  Tmp<__half> x_hi((size_t)N * ldm, h->st), x_lo((size_t)N * ldm, h->st);
  densify(A, S, 1, ldm, x_hi.p, x_lo.p, h->st);
  Tmp<__half> v_hi((size_t)k * ldm, h->st), v_lo((size_t)k * ldm, h->st);
  strided_split_f32_to_f16(dVrows, k, M, ld_v, (int64_t)ldm, v_hi.p, v_lo.p, h->st, kUnitScale);   // rows are normalised afterwards
  GemmArgs g;
  g.A.hi = x_hi.p; g.A.lo = x_lo.p; g.A.rows = N; g.A.K = M; g.A.ld = (int64_t)ldm;
  g.B.hi = v_hi.p; g.B.lo = v_lo.p; g.B.rows = k; g.B.K = M; g.B.ld = (int64_t)ldm;
  g.epi = Epilogue::StoreTransposed;
  g.C = d_out;
  g.ldc = N;
  g.cta_group = cta_group_of(h);
  {
    ProfScope ps(&h->prof, h->st, PK_OTHER_GEMM);
    gemm_umma(g, h->st);
    h->prof.other_gemm_flops += 2.0 * N * (double)M * k;
  }
  normalize_rows(d_out, k, N, h->st);
}

// ---------------------------------------------------------------------------------------
namespace {

// rec_vals (:676-695) and the ascending spectrum :L of the data matrix to the host
void fetch_signal_outputs(scl_handle* h, const float* dW, int nm, bool sorted_needed) {
  cudaStream_t st = h->st;
  const int N = h->X.N, M = h->X.M;
  h->L.resize(nm);
  SCL_CUDA(cudaMemcpyAsync(h->L.data(), dW, nm * sizeof(float), cudaMemcpyDeviceToHost, st));
  h->rec_tgc.resize(N); h->rec_l2.resize(N); h->rec_mean.resize(M); h->rec_std.resize(M); h->rec_cent.resize(M);
  SCL_CUDA(cudaMemcpyAsync(h->rec_tgc.data(), h->S_main.tgc.p, N * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaMemcpyAsync(h->rec_l2.data(), h->S_main.l2.p, N * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaMemcpyAsync(h->rec_mean.data(), h->S_main.ybar.p, M * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaMemcpyAsync(h->rec_std.data(), h->S_main.sigma.p, M * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaMemcpyAsync(h->rec_cent.data(), h->S_main.cent.p, M * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  for (float v : h->L)
    if (!std::isfinite(v)) throw Error(SCL_ERR_CUSOLVER, "non-finite eigenvalue (the reference's CPU fallback :379-381 is an error here)");
  // Rayleigh quotients of neighbouring bulk eigenvectors can swap by ~1e-6 relative: :L is ascending (:378); the
  // signal eigenvalues are far apart, so their pairing with the eigenvectors is untouched
  if (sorted_needed) std::sort(h->L.begin(), h->L.end());
}

// MP / TW fit (:537-538/:576-577) from :L and the null spectrum; Lr[1:end-1] drops the largest null eigenvalue
void fit_signal(scl_handle* h, const std::vector<float>& Lr) {
  scl_signal_info& info = h->sinfo;
  const int nm = info.nm;
  auto c0 = std::chrono::steady_clock::now();
  MpFit fit = mp_fit(h->L.data(), nm, Lr.data(), nm - 1);
  info.t_fit_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - c0).count();
  h->Lmp = fit.L_mp;
  info.n_signal = fit.n_signal;
  info.n_Lmp = (int)fit.L_mp.size();
  info.mp_iters = fit.iters;
  info.pass = fit.pass ? 1 : 0;
  info.lambda_c = fit.lambda_c;
  info.b_plus = fit.b_plus;
  info.b_minus = fit.b_minus;
  info.ks_static = fit.ks_static;
  if (h->cfg.verbose) printf("(Using gpu) number of signal ev: %d\n", info.n_signal);
  const int k = info.n_signal;
  h->nL.resize(k);
  for (int i = 0; i < k; ++i) h->nL[i] = h->L[nm - 1 - i];
}

// signal eigenvectors, descending (:541-551), as cell-space unit vectors (:556-558).  top: eigenvector of the largest
// eigenvalue, the next ones ld_top floats further (negative: walking backwards through the solver's ascending rows)
void project_signal(scl_handle* h, const float* top, long long ld_top) {
  const int N = h->X.N, M = h->X.M, k = h->sinfo.n_signal;
  h->d_nV.ensure((size_t)std::max(1, k) * N);
  if (k > 0) {
    if (N > M)
      back_project(h, h->X, h->S_main, top, ld_top, k, h->d_nV.p);
    else
      copy_rows(top, ld_top, h->d_nV.p, N, k, N, h->st);
  }
}

void make_null_matrix(scl_handle* h) {
  const SpMat& X = h->X;
  ProfScope ps(&h->prof, h->st, PK_SPARSE);
  if (h->have_null_draws)
    permute_null(X, h->null_perm.p, h->null_rows.p, h->Xnull, h->st);
  else
    draw_null_device(X, h->cfg.seed, h->Xnull, h->st);
  h->prof.sparse_alg_bytes += 20.0 * (double)X.nnz;
  SCL_REQUIRE(h->Xnull.N == X.N && h->Xnull.M == X.M, "null matrix shape");
}

}  // namespace

void run_signal(scl_handle* h) {
  SCL_REQUIRE(h->have_X, "scl_set_counts_csc must be called first");
  cudaStream_t st = h->st;
  const SpMat& X = h->X;
  const int N = X.N, M = X.M, nm = std::min(N, M);
  const bool split = h->cfg.gram_mode == SCL_GRAM_FP16X3;
  scl_signal_info& info = h->sinfo;
  info = scl_signal_info{};
  info.N = N; info.M = M; info.nm = nm;
  info.gram_mode_used = h->cfg.gram_mode;
  h->signal_done = false;
  h->robust_done = false;

  DBuf<__half>&op_hi = h->ws_op_hi, &op_lo = h->ws_op_lo;
  DBuf<float>&G = h->ws_G, &W = h->ws_W;
  G.ensure((size_t)nm * nm);
  W.ensure(nm);
  Timer tm(st);
  // --- data matrix: normalise (:677-696), Gram (:529/:569), eigen (:530/:570)
  gram_of(h, X, h->S_main, op_hi, op_lo, G.p, nm, 1.0f / (float)M, split, /*shard=*/true);
  info.t_normalize_ms = 0;  // fused into the Gram timing below (one stream); see bench for per-kernel times
  info.t_gram_ms += tm.stop();
  // the FP32 solver's eigenvalues carry an absolute error ~eps32*|G|; the spectrum of the data matrix is an output
  // (:L, :L_mp), so it is refined by Float64 Rayleigh quotients of the computed eigenvectors (refine.cu)
  const bool refine = !h->cfg.no_refine;
  DBuf<float>& Gkeep = h->ws_Gkeep;
  if (refine) {
    Gkeep.ensure((size_t)nm * nm);
    SCL_CUDA(cudaMemcpyAsync(Gkeep.p, G.p, (size_t)nm * nm * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  { ProfScope ps(&h->prof, st, PK_SYEVD); h->solver->syevd(G.p, nm, W.p, true, st); }
  info.t_syevd_ms += tm.stop();
  if (refine) {
    ProfScope ps(&h->prof, st, PK_REFINE);
    refine_eigenvalues(Gkeep.p, G.p, nm, W.p, st);
  }
  unscale_eigenvalues(h, W.p, nm);
  fetch_signal_outputs(h, W.p, nm, refine);
  tm.stop();

  // --- null matrix (:701) and its spectrum (:531-532/:571-572)
  make_null_matrix(h);
  info.t_null_ms += tm.stop();
  {
    NormStats& Sn = h->ws_Sn;
    DBuf<float>&G2 = h->ws_G2, &W2 = h->ws_W2;
    G2.ensure((size_t)nm * nm);
    W2.ensure(nm);
    gram_of(h, h->Xnull, Sn, op_hi, op_lo, G2.p, nm, 1.0f / (float)M, split, /*shard=*/true);
    info.t_gram_ms += tm.stop();
    { ProfScope ps(&h->prof, st, PK_SYEVD); h->solver->syevd(G2.p, nm, W2.p, false, st); }
    unscale_eigenvalues(h, W2.p, nm);
    info.t_syevd_ms += tm.stop();
    std::vector<float> Lr(nm);
    SCL_CUDA(cudaMemcpyAsync(Lr.data(), W2.p, nm * sizeof(float), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    fit_signal(h, Lr);
  }
  tm.stop();
  project_signal(h, G.p + (size_t)(nm - 1) * nm, -(long long)nm);
  SCL_CUDA(cudaStreamSynchronize(st));
  info.t_backproject_ms = tm.stop();
  h->prof.resolve();
  h->signal_done = true;
}

// Host tail of the robustness scoring (:797-806), pure host code: per signal, Tukey fence (type-7 quartiles,
// q1 - 1.5 iqr <= b <= q3 + 1.5 iqr) over its n_pairs pairwise similarities, median and corrected standard deviation of
// what is left, and the robust set {i : median_i > cos(th)}.  b_ is k x n_pairs column-major.
void score_from_pairs(const std::vector<float>& b_, int k, int n_pairs, double th, std::vector<double>& m_scores,
                      std::vector<double>& sd_scores, std::vector<int32_t>& sig) {
  const double th_ = std::cos(th * M_PI / 180.0);
  m_scores.assign(k, 0.0);
  sd_scores.assign(k, 0.0);
  sig.clear();
  for (int i = 0; i < k; ++i) {
    std::vector<double> row(n_pairs);
    for (int q = 0; q < n_pairs; ++q) row[q] = (double)b_[(size_t)q * k + i];
    std::vector<double> srt = row;
    std::sort(srt.begin(), srt.end());
    const double q1 = quantile7(srt, 0.25), q3 = quantile7(srt, 0.75), iqr = q3 - q1;
    std::vector<double> f;
    for (double v : srt)
      if (q1 - 1.5 * iqr <= v && v <= q3 + 1.5 * iqr) f.push_back(v);
    const size_t n = f.size();
    double med = n ? ((n & 1) ? f[n / 2] : 0.5 * (f[n / 2 - 1] + f[n / 2])) : NAN;
    double mean = 0;
    for (double v : f) mean += v;
    mean /= (double)std::max<size_t>(1, n);
    double ss = 0;
    for (double v : f) ss += (v - mean) * (v - mean);
    m_scores[i] = med;
    sd_scores[i] = n > 1 ? std::sqrt(ss / (double)(n - 1)) : NAN;
    if (med > th_) sig.push_back(i);
  }
}

// ---------------------------------------------------------------------------------------
// Robustness scoring (:786-806).  d_nV: [k][N]; d_sets: [n_perturb][min_pc][N].
void score_sets(scl_handle* h, int N, int k, int min_pc, int n_perturb, const float* d_nV, const float* d_sets,
                double th, std::vector<float>& b_, std::vector<double>& m_scores, std::vector<double>& sd_scores,
                std::vector<int32_t>& sig) {
  cudaStream_t st = h->st;
  const size_t ld = round8((size_t)N);
  const int P = n_perturb, tot = P * min_pc;
  // |nV' * nV_set[r]| for all r at once (:788)
  Tmp<__half> a_hi((size_t)k * ld, st), a_lo((size_t)k * ld, st), s_hi((size_t)tot * ld, st), s_lo((size_t)tot * ld, st);
  strided_split_f32_to_f16(d_nV, k, N, N, (int64_t)ld, a_hi.p, a_lo.p, st, kUnitScale);
  strided_split_f32_to_f16(d_sets, tot, N, N, (int64_t)ld, s_hi.p, s_lo.p, st, kUnitScale);
  GemmOperand A, B;
  A.hi = a_hi.p; A.lo = a_lo.p; A.rows = k; A.K = N; A.ld = (int64_t)ld;
  B.hi = s_hi.p; B.lo = s_lo.p; B.rows = tot; B.K = N; B.ld = (int64_t)ld;
  Tmp<float> c1((size_t)k * tot, st);
  gemm_splitk(h, A, B, false, 1.f / (kUnitScale * kUnitScale), Epilogue::Store, c1.p, tot, (size_t)k * tot);
  std::vector<float> hc1((size_t)k * tot);
  SCL_CUDA(cudaMemcpyAsync(hc1.data(), c1.p, hc1.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  std::vector<int> rows((size_t)P * k);   // row (r*k + i) of the gathered stack = sets[r][a_b[i,r]]
  for (int r = 0; r < P; ++r)
    for (int i = 0; i < k; ++i) {
      int best = 0;
      float bv = -1.f;
      for (int j = 0; j < min_pc; ++j) {
        float v = std::fabs(hc1[(size_t)i * tot + (size_t)r * min_pc + j]);
        if (v > bv) { bv = v; best = j; }   // first maximum (argmax, Appendix A14)
      }
      rows[(size_t)r * k + i] = r * min_pc + best;
    }
  // sub_nVset stack and all pairwise |sub_i' sub_j| (:790-795)
  const int R = P * k;
  Tmp<int> d_rows(R, st);
  SCL_CUDA(cudaMemcpyAsync(d_rows.p, rows.data(), R * sizeof(int), cudaMemcpyHostToDevice, st));
  Tmp<float> sub((size_t)R * N, st);
  {
    dim3 grid((unsigned)std::min((N + 255) / 256, 64), (unsigned)std::min(R, 65535));
    k_gather_rows<<<grid, 256, 0, st>>>(d_sets, d_rows.p, sub.p, R, N);
    count_launches(1);
    SCL_CUDA(cudaGetLastError());
  }
  Tmp<__half> u_hi((size_t)R * ld, st), u_lo((size_t)R * ld, st);
  strided_split_f32_to_f16(sub.p, R, N, N, (int64_t)ld, u_hi.p, u_lo.p, st, kUnitScale);
  GemmOperand U;
  U.hi = u_hi.p; U.lo = u_lo.p; U.rows = R; U.K = N; U.ld = (int64_t)ld;
  Tmp<float> c2((size_t)R * R, st);
  gemm_splitk(h, U, U, true, 1.f / (kUnitScale * kUnitScale), Epilogue::Store, c2.p, R, (size_t)R * R);
  std::vector<float> hc2((size_t)R * R);
  SCL_CUDA(cudaMemcpyAsync(hc2.data(), c2.p, hc2.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  const int n_pairs = P * (P - 1) / 2;
  b_.assign((size_t)k * n_pairs, 0.f);
  int pair = 0;
  for (int a = 0; a < P; ++a)
    for (int b = a + 1; b < P; ++b, ++pair)
      for (int i = 0; i < k; ++i) {
        float mx = 0.f;
        for (int j = 0; j < k; ++j) mx = std::max(mx, std::fabs(hc2[(size_t)(a * k + i) * R + (size_t)(b * k + j)]));
        b_[(size_t)pair * k + i] = mx;   // column-major k x n_pairs
      }
  score_from_pairs(b_, k, n_pairs, th, m_scores, sd_scores, sig);
}

// ---------------------------------------------------------------------------------------
namespace {

// additions (row, col) for one perturbation: injected sample indices (indexed by search step / replicate) or a
// device draw keyed by the same index, so every rank of a multi-GPU run derives identical draws
void make_additions(scl_handle* h, const std::vector<std::vector<uint32_t>>& injected, size_t index, size_t n_add,
                    uint64_t draw_seed, uint32_t* d_row, uint32_t* d_col) {
  if (index < injected.size()) {
    const std::vector<uint32_t>& s = injected[index];
    SCL_REQUIRE(s.size() == n_add, "injected sample has the wrong length for this sparsity step");
    for (uint32_t v : s) SCL_REQUIRE((size_t)v < h->n_cand, "injected sample index outside the zero-candidate pool");
    Tmp<uint32_t> d_idx(n_add, h->st);
    SCL_CUDA(cudaMemcpyAsync(d_idx.p, s.data(), n_add * sizeof(uint32_t), cudaMemcpyHostToDevice, h->st));
    gather_pairs(h->z1.p, h->z2.p, d_idx.p, n_add, d_row, d_col, h->st);
    SCL_CUDA(cudaStreamSynchronize(h->st));
  } else {
    draw_subset_device(h->z1.p, h->z2.p, h->n_cand, n_add, draw_seed, d_row, d_col, h->st);
  }
}

// L .> 0 (:495) read in exact arithmetic: the Gram of a column-centred N x M matrix with N <= M has
// one exactly-zero eigenvalue that FP32 returns as +-1e-7; the reference keeps or drops that vector by
// the sign of rounding noise.  An eigenvalue below 1e-5 * max(L) is treated as not positive here and
// in the oracle (DESIGN.md, deviations).  L is ascending.
int first_positive(const std::vector<float>& L) {
  const float thr = 1e-5f * L.back();
  int i = 0;
  while (i < (int)L.size() && !(L[i] > thr)) ++i;
  return i;
}

}  // namespace

namespace {

// reference loop state of the sparsity search (:722-760): second-smallest values are fed in step order, whoever evaluated
// them (this rank sequentially, or the ranks of a wave speculatively) - the outcome is the sequential loop's
struct SearchState {
  double p_step, p_th;
  int tank_n = 5;
  std::vector<double> tank2;            // row 2 of tank_ (second smallest of d_arr per step)
  std::vector<double> p_of_step{0.999};
  double p_ = 0.999;
  int step = 0;
  bool stop = false;
  double p_at(int s_) {
    while ((int)p_of_step.size() <= s_) p_of_step.push_back(p_of_step.back() - p_step);   // :760, same rounding drift
    return p_of_step[s_];
  }
  // the sequential loop reaches step s only if no earlier step stopped it: every earlier p_ was >= 0.9 (:756)
  bool reachable(int s_) { return s_ == 0 || p_at(s_ - 1) >= 0.9; }
  long long n_add(int s_, int N, int M) { return (long long)std::nearbyint((1.0 - p_at(s_)) * (double)M * (double)N); }   // :726
  // d2 >= 0: second-smallest of d_arr; -1: the candidate pool is smaller than this step's additions (:727-730)
  void feed(scl_handle* h, int s_, double d2) {
    if (stop) return;
    p_ = p_at(s_);
    if (d2 == -1.0) {
      p_ += p_step;
      stop = true;
      return;
    }
    SCL_REQUIRE(d2 >= 0, "sparsity search consumed a step that was never evaluated");
    tank2.push_back(d2);
    h->trace_p.push_back(p_);
    h->trace_d.push_back(d2);
    if (h->cfg.verbose) printf("%.9g\n", d2);
    ++step;
    int below = 0;
    const int cnt = (int)tank2.size() < tank_n ? (int)tank2.size() : tank_n;
    for (int q = 0; q < cnt; ++q)
      if (tank2[tank2.size() - 1 - q] < p_th) ++below;
    if (below > tank_n - 1 || p_ < 0.9) {                    // :756
      p_ += (double)(tank_n - 1) * p_step;
      stop = true;
    }
  }
};

// device state shared by the search steps of one pass
struct SearchCtx {
  float bin_scale = 0;
  int n_2 = 0, nw = 0;
  GemmOperand Vr;
  std::vector<float> Lh;
};

// noise baseline (:709-713), zero candidates (:668-673), buffers of the perturbed matrices
void robust_prepare(scl_handle* h) {
  cudaStream_t st = h->st;
  const SpMat& X = h->X;
  const int nm = std::min(X.N, X.M);
  scl_robust_info& info = h->rinfo;
  info = scl_robust_info{};
  h->robust_done = false;
  const double p_th = h->have_pth ? h->p_th : noise_baseline_device(nm, 5000, h->cfg.seed, st);
  info.p_th = p_th;
  if (h->cfg.verbose) printf("spth_: %.17g\n", p_th);
  if (!h->have_zc) h->n_cand = draw_zero_candidates_device(X, h->cfg.seed, h->z1, h->z2, st);
  h->ws_G.ensure((size_t)nm * nm);
  h->ws_W.ensure(nm);
  // the perturbed matrices gain up to ~2-3 % of the grid in stored entries before the search stops (p_ ~ 0.98):
  // size their buffers once instead of growing them step by step
  const size_t cap = X.nnz + (size_t)(0.03 * (double)X.N * (double)X.M) + 1024;
  h->ws_Xp.reserve(cap);
  h->ws_Sp.reserve(cap);
  h->trace_p.clear();
  h->trace_d.clear();
}

// reference basis of the binarised matrix (:717-721): Gram matrix into ws_G and its full eigenbasis in place
void binref_solve(scl_handle* h, SearchCtx& c) {
  cudaStream_t st = h->st;
  const SpMat& X = h->X;
  const int N = X.N, M = X.M, nm = std::min(N, M);
  const bool split = h->cfg.gram_mode == SCL_GRAM_FP16X3;
  perturb_merge(X, nullptr, nullptr, 0, true, h->ws_Xp, st);
  gram_of(h, h->ws_Xp, h->ws_Sp, h->ws_op_hi, h->ws_op_lo, h->ws_G.p, nm, c.bin_scale, split);
  { ProfScope ps(&h->prof, st, PK_SYEVD); h->solver->syevd(h->ws_G.p, nm, h->ws_W.p, true, st); }
}

// The reference basis keeps the complete eigenbasis (oracle get_eigvec(keep_null=True); DESIGN.md, deviations): null
// directions of the binarised matrix are kept, as in the reference whenever their eigenvalues round positive, so their
// perturbed counterparts are not mistaken for delocalised vectors.  hi/lo binary16 rows, the GEMM's K-major operand.
void binref_operand(scl_handle* h, SearchCtx& c, bool convert) {
  const int nm = std::min(h->X.N, h->X.M);
  const size_t ldv = round8((size_t)nm);
  h->ws_vr_hi.ensure((size_t)nm * ldv);
  h->ws_vr_lo.ensure((size_t)nm * ldv);
  if (convert) strided_split_f32_to_f16(h->ws_G.p, nm, nm, nm, (int64_t)ldv, h->ws_vr_hi.p, h->ws_vr_lo.p, h->st, kUnitScale);
  c.Vr.hi = h->ws_vr_hi.p; c.Vr.lo = h->ws_vr_lo.p; c.Vr.rows = nm; c.Vr.K = nm; c.Vr.ld = (int64_t)ldv;
}

void search_ctx_init(scl_handle* h, SearchCtx& c) {
  const int N = h->X.N, M = h->X.M, nm = std::min(N, M);
  c.bin_scale = 1.0f / (float)(N > M ? N : M);   // transposed call when N > M (Appendix A9)
  c.n_2 = (int)std::nearbyint((double)nm / 2.0);   // round(Int, .) ties-to-even (:722); the reference basis is complete
  c.nw = c.n_2 + 1;                                // nV_2[:, end-n_2:end] (Appendix A13)
  c.Lh.assign(nm, 0.f);
  SCL_REQUIRE(c.nw >= 5, "too few noise vectors");
}

// heavy part of search step s_ (:726-740): additions, merge, normalise, Gram, eigenvectors of the nw smallest positive
// eigenvalues, left in rows [i0, i0 + nw) of ws_G.  Returns i0, or -1 when the candidate pool is exhausted (:727-730).
int search_step_solve(scl_handle* h, SearchCtx& c, SearchState& ss, int s_, scl_robust_info& info, Timer& tm, double& t_gram) {
  cudaStream_t st = h->st;
  const SpMat& X = h->X;
  const int N = X.N, M = X.M, nm = std::min(N, M), nw = c.nw;
  const bool split = h->cfg.gram_mode == SCL_GRAM_FP16X3;
  const long long nnzidx = ss.n_add(s_, N, M);
  if ((long long)h->n_cand < nnzidx) return -1;
  DBuf<float>&G = h->ws_G, &W = h->ws_W;
  SpMat& Xp = h->ws_Xp;
  NormStats& Sp = h->ws_Sp;
  tm.stop();
  Tmp<uint32_t> a_row((size_t)std::max<long long>(1, nnzidx), st), a_col((size_t)std::max<long long>(1, nnzidx), st);
  make_additions(h, h->search_sples, (size_t)s_, (size_t)nnzidx, h->cfg.seed + 0x5eed0000ull + (uint64_t)s_, a_row.p, a_col.p);
  {
    ProfScope ps(&h->prof, st, PK_SPARSE);
    perturb_merge(X, a_row.p, a_col.p, (size_t)nnzidx, true, Xp, st);
    h->prof.sparse_alg_bytes += 8.0 * (double)X.nnz + 12.0 * (double)nnzidx;
  }
  gram_of(h, Xp, Sp, h->ws_op_hi, h->ws_op_lo, G.p, nm, c.bin_scale, split);
  t_gram += tm.stop();
  int i0 = -1;
  // vectors of the index range this step reads only (the nw smallest positive eigenpairs plus a margin for non-positive
  // eigenvalues); all eigenvalues come back, so the "positive" threshold is exact
  const int iu = std::min(nm, nw + 64);
  { ProfScope ps(&h->prof, st, PK_SYEVD); h->solver->syevd_tri(G.p, nm, W.p, 0, iu, st); }
  SCL_CUDA(cudaMemcpyAsync(c.Lh.data(), W.p, nm * sizeof(float), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  const int j = first_positive(c.Lh);
  if (j + nw <= iu) {
    i0 = j;
  } else {   // more than 64 non-positive eigenvalues: rebuild the Gram matrix and take the full solve below
    gram_of(h, Xp, Sp, h->ws_op_hi, h->ws_op_lo, G.p, nm, c.bin_scale, split);
  }
  if (i0 < 0) {
    { ProfScope ps(&h->prof, st, PK_SYEVD); h->solver->syevd(G.p, nm, W.p, true, st); }
    SCL_CUDA(cudaMemcpyAsync(c.Lh.data(), W.p, nm * sizeof(float), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    i0 = first_positive(c.Lh);
    SCL_REQUIRE(nm - i0 >= c.n_2 + 1, "perturbed matrix has too few positive eigenvalues");
  }
  info.t_search_syevd_ms += tm.stop();
  return i0;
}

// d_arr of :742 for the vectors search_step_solve left in ws_G; returns its second-smallest value (:747-748)
double search_step_corr(scl_handle* h, SearchCtx& c, int i0) {
  cudaStream_t st = h->st;
  const int nm = std::min(h->X.N, h->X.M), nw = c.nw;
  Tmp<float> d_d(nw, st);
  corr_colabsmax_pre(h, c.Vr, h->ws_G.p + (size_t)i0 * nm, nw, nm, d_d.p);
  std::vector<float> d_host(nw);
  SCL_CUDA(cudaMemcpyAsync(d_host.data(), d_d.p, nw * sizeof(float), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  std::partial_sort(d_host.begin(), d_host.begin() + 5, d_host.end());
  return (double)d_host[1];
}

// every rank learns whether any rank failed in the section just finished; all of them throw together instead of leaving
// the healthy ones blocked in the next collective
void sync_errors(scl_handle* h, const std::string& mine) {
  if (!multi(h)) {
    if (!mine.empty()) throw Error(SCL_ERR_INVALID, mine);
    return;
  }
  Tmp<int> flag(1, h->st);
  const int f = mine.empty() ? 0 : 1 + h->rank;
  SCL_CUDA(cudaMemcpyAsync(flag.p, &f, sizeof(int), cudaMemcpyHostToDevice, h->st));
  SCL_NCCL(nccl_api().AllReduce(flag.p, flag.p, 1, ncclInt, ncclMax, (ncclComm_t)h->nccl, h->st));
  int any = 0;
  SCL_CUDA(cudaMemcpyAsync(&any, flag.p, sizeof(int), cudaMemcpyDeviceToHost, h->st));
  SCL_CUDA(cudaStreamSynchronize(h->st));
  if (!mine.empty()) throw Error(SCL_ERR_INVALID, mine);
  if (any) throw Error(SCL_ERR_NCCL, "rank " + std::to_string(any - 1) + " failed in this stage of the cooperative pass; all ranks abort");
}

// perturbations (:767-778), robustness scores (:786-807), gene_basis (:813-819)
void robust_tail(scl_handle* h, double th, int n_perturb, double p_, Timer& tm) {
  cudaStream_t st = h->st;
  const SpMat& X = h->X;
  const int N = X.N, M = X.M, nm = std::min(N, M);
  const bool split = h->cfg.gram_mode == SCL_GRAM_FP16X3;
  scl_robust_info& info = h->rinfo;
  DBuf<__half>&op_hi = h->ws_op_hi, &op_lo = h->ws_op_lo;
  DBuf<float>&G = h->ws_G, &W = h->ws_W;
  SpMat& Xp = h->ws_Xp;
  NormStats& Sp = h->ws_Sp;
  std::vector<float> Lh(nm);
  const int k = h->sinfo.n_signal;
  // :776 takes min(min_pc, number of positive eigenpairs) columns per replicate; a replicate with fewer gets zero
  // columns for the rest (a zero column never wins an argmax of |.|, so the scores are the reference's)
  const int min_pc = std::min((int)std::ceil((double)k * 1.5), nm);
  const long long n_add = (long long)std::nearbyint((1.0 - p_) * (double)M * (double)N);     // :772
  SCL_REQUIRE((long long)h->n_cand >= n_add, "zero-candidate pool smaller than the perturbation size");
  info.min_pc = min_pc;
  info.n_add = n_add;
  info.n_perturb = n_perturb;
  h->d_sets.ensure((size_t)n_perturb * min_pc * N);
  h->set_L.assign((size_t)n_perturb * min_pc, 0.f);
  // the block subspace iteration needs room for its block (k + 64 vectors, at most 256, at most n / 2); anything else -
  // tiny matrices, signal-rich inputs, a replicate that does not converge - takes the exact solve the reference makes
  const int sub_b = std::min(256, ((min_pc + (h->cfg.subspace_extra > 0 ? h->cfg.subspace_extra : 64) + 31) / 32) * 32);
  const bool can_subspace = min_pc + 16 <= sub_b && sub_b * 2 <= nm;
  const bool exact = h->cfg.exact_perturb != 0 || !can_subspace;
  Tmp<float> topL(min_pc, st), topV((size_t)min_pc * nm, st);
  Tmp<float> setL_dev((size_t)n_perturb * min_pc, st);
  std::string err;
  try {
    for (int r = 0; r < n_perturb; ++r) {
      if (multi(h) && r % h->world != h->rank) continue;   // replicate r belongs to rank r mod G (scl_plan_replicates)
      Tmp<uint32_t> a_row((size_t)std::max<long long>(1, n_add), st), a_col((size_t)std::max<long long>(1, n_add), st);
      make_additions(h, h->perturb_sples, (size_t)r, (size_t)n_add, h->cfg.seed + 0xbeef0000ull + (uint64_t)r, a_row.p, a_col.p);
      {
        ProfScope ps(&h->prof, st, PK_SPARSE);
        perturb_merge(X, a_row.p, a_col.p, (size_t)n_add, false, Xp, st);                        // :774
        h->prof.sparse_alg_bytes += 8.0 * (double)X.nnz + 12.0 * (double)n_add;
      }
      gram_of(h, Xp, Sp, op_hi, op_lo, G.p, nm, 1.0f / (float)M, split);                         // :775 -> :492/:512
      float* set_r = h->d_sets.p + (size_t)r * min_pc * N;
      const float* vec0 = nullptr;
      long long ldvec = 0;
      int have = min_pc;
      bool solved = false;
      if (!exact) {
        try {
          int iters = 0;
          topk_subspace(h, G.p, nm, min_pc, topL.p, topV.p, &iters);
          unscale_eigenvalues(h, topL.p, min_pc);
          SCL_CUDA(cudaMemcpyAsync(&h->set_L[(size_t)r * min_pc], topL.p, min_pc * sizeof(float), cudaMemcpyDeviceToHost, st));
          vec0 = topV.p;
          ldvec = nm;
          solved = true;
        } catch (const Error& e) {
          if (e.code != SCL_ERR_CUSOLVER) throw;
          ++info.n_subspace_fallbacks;   // did not converge / lost rank: the Gram matrix is intact, solve it exactly
        }
      }
      if (!solved) {
        {
          ProfScope ps(&h->prof, st, PK_SYEVD);
          h->solver->syevd_tri(G.p, nm, W.p, nm - min_pc, nm, st);
        }
        unscale_eigenvalues(h, W.p, nm);
        SCL_CUDA(cudaMemcpyAsync(Lh.data(), W.p, nm * sizeof(float), cudaMemcpyDeviceToHost, st));
        SCL_CUDA(cudaStreamSynchronize(st));
        have = std::min(min_pc, nm - first_positive(Lh));
        for (int i = 0; i < have; ++i) h->set_L[(size_t)r * min_pc + i] = Lh[nm - 1 - i];
        vec0 = G.p + (size_t)(nm - 1) * nm;
        ldvec = -(long long)nm;
      }
      if (have < min_pc) SCL_CUDA(cudaMemsetAsync(set_r + (size_t)have * N, 0, (size_t)(min_pc - have) * N * sizeof(float), st));
      if (have > 0) {
        if (N > M)
          back_project(h, Xp, Sp, vec0, ldvec, have, set_r);
        else
          copy_rows(vec0, ldvec, set_r, N, have, N, st);
      }
    }
    SCL_CUDA(cudaStreamSynchronize(st));
  } catch (const std::exception& e) {
    err = e.what();
  }
  sync_errors(h, err);
  if (multi(h)) {
    // every rank scores all replicates: N x min_pc blocks travel once over NVLink from their owner
    ProfScope ps(&h->prof, st, PK_COMM);
    SCL_CUDA(cudaMemcpyAsync(setL_dev.p, h->set_L.data(), h->set_L.size() * sizeof(float), cudaMemcpyHostToDevice, st));
    SCL_NCCL(nccl_api().GroupStart());
    for (int r = 0; r < n_perturb; ++r) {
      float* set_r = h->d_sets.p + (size_t)r * min_pc * N;
      SCL_NCCL(nccl_api().Broadcast(set_r, set_r, (size_t)min_pc * N, ncclFloat, r % h->world, (ncclComm_t)h->nccl, st));
      SCL_NCCL(nccl_api().Broadcast(setL_dev.p + (size_t)r * min_pc, setL_dev.p + (size_t)r * min_pc, (size_t)min_pc, ncclFloat,
                             r % h->world, (ncclComm_t)h->nccl, st));
    }
    SCL_NCCL(nccl_api().GroupEnd());
    SCL_CUDA(cudaMemcpyAsync(h->set_L.data(), setL_dev.p, h->set_L.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    h->prof.comm_bytes += 4.0 * (double)n_perturb * min_pc * (N + 1);
  }
  info.t_perturb_ms = tm.stop();

  // --- robustness scores (:786-807)
  score_sets(h, N, k, min_pc, n_perturb, h->d_nV.p, h->d_sets.p, th, h->b_, h->m_scores, h->sd_scores, h->sig_id);
  info.n_robust = (int)h->sig_id.size();
  if (h->cfg.verbose) printf("Number of filtered signal: %d\n", info.n_robust);
  info.t_score_ms = tm.stop();

  // --- gene_basis = diag(1/sqrt(nL)) * nV' * scaled_X / sqrt(M)   (:813-819)
  {
    const size_t ldn = round8((size_t)N);
    Tmp<__half> x_hi((size_t)M * ldn, st), x_lo((size_t)M * ldn, st), v_hi((size_t)k * ldn, st), v_lo((size_t)k * ldn, st);
    densify(X, h->S_main, 0, ldn, x_hi.p, x_lo.p, st);
    strided_split_f32_to_f16(h->d_nV.p, k, N, N, (int64_t)ldn, v_hi.p, v_lo.p, st, kUnitScale);
    Tmp<float> gb((size_t)M * k, st);
    GemmArgs g;
    g.A.hi = x_hi.p; g.A.lo = x_lo.p; g.A.rows = M; g.A.K = N; g.A.ld = (int64_t)ldn;
    g.B.hi = v_hi.p; g.B.lo = v_lo.p; g.B.rows = k; g.B.K = N; g.B.ld = (int64_t)ldn;
    g.epi = Epilogue::Store;
    g.alpha = 1.0f / std::sqrt((float)M) / kUnitScale;
    g.C = gb.p;
    g.ldc = k;
    g.cta_group = cta_group_of(h);
    {
      ProfScope ps(&h->prof, st, PK_OTHER_GEMM);
      gemm_umma(g, st);
      h->prof.other_gemm_flops += 2.0 * M * (double)N * k;
    }
    h->gene_basis.resize((size_t)M * k);
    SCL_CUDA(cudaMemcpyAsync(h->gene_basis.data(), gb.p, h->gene_basis.size() * sizeof(float), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    for (int j = 0; j < M; ++j)
      for (int i = 0; i < k; ++i) h->gene_basis[(size_t)j * k + i] /= std::sqrt(h->nL[i]);
  }
  info.t_outputs_ms = tm.stop();
  h->prof.resolve();
  h->robust_done = true;
}

}  // namespace

void run_robustness(scl_handle* h, double th, double p_step, int n_perturb) {
  SCL_REQUIRE(h->signal_done, "scl_run_signal must succeed first");
  if (h->sinfo.n_signal == 0) throw Error(SCL_ERR_NOSIGNAL, "warning: There is no signal");
  SCL_REQUIRE(n_perturb >= 2, "n_perturb must be >= 2");
  cudaStream_t st = h->st;
  scl_robust_info& info = h->rinfo;
  Timer tm(st);
  robust_prepare(h);
  info.t_baseline_ms = tm.stop();

  // --- reference basis of the binarised matrix (:717-721)
  SearchCtx c;
  search_ctx_init(h, c);
  binref_solve(h, c);
  binref_operand(h, c, true);
  info.t_search_syevd_ms += tm.stop();

  // --- sparsity search (:715-762)
  // Steps are independent given their draws; only the stop rule is sequential.  With G ranks, wave w evaluates
  // steps w*G .. w*G+G-1 speculatively (rank g takes step w*G+g, p_ = 0.999 - step*p_step accumulated exactly as
  // the reference's repeated `p_ -= p_step`), the second-smallest values are gathered, and the stop rule is applied
  // in step order - the result is identical to the sequential loop (SURVEY.md 8e).  G = 1 is the plain loop.
  // (scl_run_pass spreads the three solves above over the ranks as well.)
  const int G_ = multi(h) ? h->world : 1;
  SearchState ss;
  ss.p_step = p_step;
  ss.p_th = info.p_th;
  Tmp<double> wave_dev(G_, st);
  double t_gram = 0;
  for (int wave = 0; !ss.stop; ++wave) {
    const int my_step = wave * G_ + (multi(h) ? h->rank : 0);
    double my_d2 = -2.0;   // not evaluated: the sequential loop cannot reach this step
    std::string err;
    try {
      if (ss.reachable(my_step)) {
        const int i0 = search_step_solve(h, c, ss, my_step, info, tm, t_gram);
        my_d2 = i0 < 0 ? -1.0 : search_step_corr(h, c, i0);
      }
    } catch (const std::exception& e) {
      err = e.what();
    }
    std::vector<double> wave_d2(G_, my_d2);
    if (G_ > 1) {
      sync_errors(h, err);
      SCL_CUDA(cudaMemcpyAsync(wave_dev.p + h->rank, &my_d2, sizeof(double), cudaMemcpyHostToDevice, st));
      SCL_NCCL(nccl_api().AllGather(wave_dev.p + h->rank, wave_dev.p, 1, ncclDouble, (ncclComm_t)h->nccl, st));
      SCL_CUDA(cudaMemcpyAsync(wave_d2.data(), wave_dev.p, G_ * sizeof(double), cudaMemcpyDeviceToHost, st));
      SCL_CUDA(cudaStreamSynchronize(st));
    } else if (!err.empty()) {
      throw Error(SCL_ERR_INVALID, err);
    }
    for (int g = 0; g < G_; ++g) ss.feed(h, wave * G_ + g, wave_d2[g]);   // the reference's loop body, in step order
  }
  info.n_search = ss.step;
  info.p_sel = ss.p_;
  info.t_search_ms = t_gram + tm.stop();
  if (h->cfg.verbose) printf("Selected perturb sparisty: %.17g\n", ss.p_);
  robust_tail(h, th, n_perturb, ss.p_, tm);
}

// Task list of the shared pass: 0 data, 1 null, 2 reference basis, then the search steps - with one slot taken out for the
// Float64 refinement of the data spectrum when there are at least three ranks: the first slot of wave 1, which is rank 0's
// (the rank that holds the data matrix's eigenvectors), so the refinement does not lengthen wave 0 and costs rank 0 one
// search step instead.  Fewer ranks refine right after the data solve (their rank 0 reuses the buffer in wave 1).
int pass_refine_task(int world) { return world >= 3 ? world : -1; }
int pass_task_step(int task, int refine_task) {
  if (task < 3 || task == refine_task) return -1;
  return task - 3 - ((refine_task >= 0 && task > refine_task) ? 1 : 0);
}

// One complete sclens() pass (:664-819).  One rank: run_signal, then run_robustness.  Several ranks: ONE pass shared by all
// of them - the Gram matrices of the data and null matrices are contracted cell block by cell block on every rank and
// reduced (packed triangle) to the rank that solves them, and the pass's eigensolves form one task list
//   [data, null, binarised reference, search step 0, search step 1, ...]          task t -> rank t mod G, wave t div G
// so that the three solves that used to run redundantly on every rank share a wave with the first search steps.  What a
// later task needs from an earlier one travels once over NVLink: the two spectra (for the MP/TW fit every rank repeats),
// the k signal eigenvectors, and the reference basis as binary16 hi/lo rows.  Search steps keep their eigenvectors until the
// basis has arrived.  The stop rule consumes the steps in order, so the outcome is the sequential loop's.
void run_pass(scl_handle* h, double th, double p_step, int n_perturb) {
  const bool signal_only = n_perturb == 0;   // the signal stage alone (:664-706), still shared by the ranks
  if (!multi(h)) {
    run_signal(h);
    h->rinfo = scl_robust_info{};
    if (h->sinfo.n_signal == 0 || signal_only) return;   // :780-784
    run_robustness(h, th, p_step, n_perturb);
    return;
  }
  SCL_REQUIRE(h->have_X, "scl_set_counts_csc must be called first");
  SCL_REQUIRE(n_perturb >= 2 || signal_only, "n_perturb must be >= 2 (or 0 for the signal stage alone)");
  cudaStream_t st = h->st;
  const SpMat& X = h->X;
  const int N = X.N, M = X.M, nm = std::min(N, M), G_ = h->world, me = h->rank;
  const bool split = h->cfg.gram_mode == SCL_GRAM_FP16X3;
  scl_signal_info& sinfo = h->sinfo;
  sinfo = scl_signal_info{};
  sinfo.N = N; sinfo.M = M; sinfo.nm = nm;
  sinfo.gram_mode_used = h->cfg.gram_mode;
  h->signal_done = false;
  const int r_data = 0, r_null = 1 % G_, r_bin = 2 % G_;
  const bool refine = !h->cfg.no_refine;
  DBuf<float>&G = h->ws_G, &W = h->ws_W, &G2 = h->ws_G2, &W2 = h->ws_W2;
  G.ensure((size_t)nm * nm); W.ensure(nm); G2.ensure((size_t)nm * nm); W2.ensure(nm);
  Timer tm(st);
  std::string err;
  SearchCtx c;
  SearchState ss;
  scl_robust_info& rinfo = h->rinfo;
  double t_gram = 0;
  // --- cooperative part: both sharded Gram matrices, the draws every rank repeats identically
  try {
    gram_of(h, X, h->S_main, h->ws_op_hi, h->ws_op_lo, G.p, nm, 1.0f / (float)M, split, /*shard=*/true, r_data);
    save_gram_factor(h, 1);
    if (me == r_data && refine) {
      h->ws_Gkeep.ensure((size_t)nm * nm);
      SCL_CUDA(cudaMemcpyAsync(h->ws_Gkeep.p, G.p, (size_t)nm * nm * sizeof(float), cudaMemcpyDeviceToDevice, st));
    }
    make_null_matrix(h);
    sinfo.t_null_ms = tm.stop();
    gram_of(h, h->Xnull, h->ws_Sn, h->ws_op_hi, h->ws_op_lo, G2.p, nm, 1.0f / (float)M, split, /*shard=*/true, r_null);
    save_gram_factor(h, 2);
    sinfo.t_gram_ms = tm.stop();
    if (!signal_only) {
      robust_prepare(h);
      rinfo.t_baseline_ms = tm.stop();
      search_ctx_init(h, c);
      binref_operand(h, c, false);
    } else {
      rinfo = scl_robust_info{};
    }
    ss.p_step = p_step;
    ss.p_th = rinfo.p_th;
  } catch (const std::exception& e) {
    err = e.what();
  }
  sync_errors(h, err);

  Tmp<double> wave_dev(G_, st);
  bool have_fit = false, have_basis = false;
  const int refine_task = (refine && !signal_only) ? pass_refine_task(G_) : -1;
  std::vector<float> Lr(nm);
  for (int wave = 0; !ss.stop; ++wave) {
    const int task = wave * G_ + me;
    int i0 = -2;            // search step of this rank in this wave: -2 none / unreachable, -1 pool exhausted, >= 0 solved
    const int my_step = pass_task_step(task, refine_task);
    err.clear();
    try {
      if (task == 0) {                  // data matrix (:530/:570)
        { ProfScope ps(&h->prof, st, PK_SYEVD); h->solver->syevd(G.p, nm, W.p, true, st); }
        sinfo.t_syevd_ms += tm.stop();
        if (refine && refine_task < 0) {
          ProfScope ps(&h->prof, st, PK_REFINE);
          refine_eigenvalues(h->ws_Gkeep.p, G.p, nm, W.p, st);
        }
        if (refine_task < 0) unscale_eigenvalues(h, W.p, nm, 1);
      }
      if (task == refine_task) {        // Float64 refinement of the data spectrum, in the slot after the data solve's wave
        ProfScope ps(&h->prof, st, PK_REFINE);
        refine_eigenvalues(h->ws_Gkeep.p, G.p, nm, W.p, st);
        unscale_eigenvalues(h, W.p, nm, 1);
      }
      if (task == 1) {                  // null matrix, values only (:531-532/:571-572)
        { ProfScope ps(&h->prof, st, PK_SYEVD); h->solver->syevd(G2.p, nm, W2.p, false, st); }
        unscale_eigenvalues(h, W2.p, nm, 2);
        sinfo.t_syevd_ms += tm.stop();
      }
      if (task == 2 && !signal_only) {  // reference basis of the binarised matrix (:717-721)
        tm.stop();
        binref_solve(h, c);
        rinfo.t_search_syevd_ms += tm.stop();
      }
      if (!signal_only && my_step >= 0 && ss.reachable(my_step)) i0 = search_step_solve(h, c, ss, my_step, rinfo, tm, t_gram);
      SCL_CUDA(cudaStreamSynchronize(st));
    } catch (const std::exception& e) {
      err = e.what();
    }
    sync_errors(h, err);
    err.clear();
    double my_d2 = i0 == -1 ? -1.0 : -2.0;
    try {
      // --- what later tasks need from this wave's, in task order
      const bool fit_now = !have_fit && wave >= (refine_task >= 0 ? refine_task / G_ : 1 / G_);   // data (refined) and null spectra are in
      const bool basis_now = !signal_only && !have_basis && wave >= 2 / G_;   // task 2 is done (wave 0 when G >= 3, wave 1 when G = 2)
      if (fit_now) {
        ProfScope ps(&h->prof, st, PK_COMM);
        SCL_NCCL(nccl_api().Broadcast(W.p, W.p, nm, ncclFloat, r_data, (ncclComm_t)h->nccl, st));
        SCL_NCCL(nccl_api().Broadcast(W2.p, W2.p, nm, ncclFloat, r_null, (ncclComm_t)h->nccl, st));
        h->prof.comm_bytes += 8.0 * nm;
      }
      if (fit_now) {
        fetch_signal_outputs(h, W.p, nm, refine);
        SCL_CUDA(cudaMemcpyAsync(Lr.data(), W2.p, nm * sizeof(float), cudaMemcpyDeviceToHost, st));
        SCL_CUDA(cudaStreamSynchronize(st));
        fit_signal(h, Lr);
        const int k = sinfo.n_signal;
        // the k leading eigenvectors leave the solving rank before its buffer is reused (G = 2: by the reference basis)
        Tmp<float> top((size_t)std::max(1, k) * nm, st);
        if (k > 0) {
          if (me == r_data) copy_rows(G.p + (size_t)(nm - 1) * nm, -(long long)nm, top.p, nm, k, nm, st);
          ProfScope ps(&h->prof, st, PK_COMM);
          SCL_NCCL(nccl_api().Broadcast(top.p, top.p, (size_t)k * nm, ncclFloat, r_data, (ncclComm_t)h->nccl, st));
          h->prof.comm_bytes += 4.0 * (double)k * nm;
        }
        tm.stop();
        project_signal(h, top.p, (long long)nm);
        SCL_CUDA(cudaStreamSynchronize(st));
        sinfo.t_backproject_ms = tm.stop();
        h->signal_done = true;
        have_fit = true;
      }
      if (basis_now) {
        if (me == r_bin) binref_operand(h, c, true);
        ProfScope ps(&h->prof, st, PK_COMM);
        const size_t cnt = (size_t)nm * (size_t)c.Vr.ld;
        SCL_NCCL(nccl_api().Broadcast(h->ws_vr_hi.p, h->ws_vr_hi.p, cnt, ncclHalf, r_bin, (ncclComm_t)h->nccl, st));
        SCL_NCCL(nccl_api().Broadcast(h->ws_vr_lo.p, h->ws_vr_lo.p, cnt, ncclHalf, r_bin, (ncclComm_t)h->nccl, st));
        SCL_CUDA(cudaStreamSynchronize(st));
        h->prof.comm_bytes += 4.0 * (double)cnt;
        have_basis = true;
      }
      if (i0 >= 0) {
        SCL_REQUIRE(have_basis, "search step finished before the reference basis");
        tm.stop();
        my_d2 = search_step_corr(h, c, i0);
        t_gram += tm.stop();
      }
    } catch (const std::exception& e) {
      err = e.what();
    }
    sync_errors(h, err);
    if (have_fit && (sinfo.n_signal == 0 || signal_only)) {   // :780-784: nothing to test (or nothing asked for)
      h->prof.resolve();
      return;
    }
    std::vector<double> wave_d2(G_, -2.0);
    SCL_CUDA(cudaMemcpyAsync(wave_dev.p + me, &my_d2, sizeof(double), cudaMemcpyHostToDevice, st));
    SCL_NCCL(nccl_api().AllGather(wave_dev.p + me, wave_dev.p, 1, ncclDouble, (ncclComm_t)h->nccl, st));
    SCL_CUDA(cudaMemcpyAsync(wave_d2.data(), wave_dev.p, G_ * sizeof(double), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    for (int g = 0; g < G_; ++g) {
      const int s_ = pass_task_step(wave * G_ + g, refine_task);
      if (s_ >= 0) ss.feed(h, s_, wave_d2[g]);
    }
  }
  rinfo.n_search = ss.step;
  rinfo.p_sel = ss.p_;
  rinfo.t_search_ms = t_gram + tm.stop();
  if (h->cfg.verbose) printf("Selected perturb sparisty: %.17g\n", ss.p_);
  robust_tail(h, th, n_perturb, ss.p_, tm);
}

}  // namespace scl
