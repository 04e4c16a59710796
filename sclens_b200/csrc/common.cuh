// Shared declarations of libsclens_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>
#include <vector>
#include "prof.h"

namespace scl {

struct Error : std::runtime_error {
  int code;
  Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#define SCL_CUDA(x)                                                                        \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess)                                                                 \
      throw scl::Error(-2, std::string(#x) + ": " + cudaGetErrorString(e_) + " @" +        \
                               __FILE__ + ":" + std::to_string(__LINE__));                 \
  } while (0)

#define SCL_REQUIRE(cond, msg)                                                             \
  do {                                                                                     \
    if (!(cond)) throw scl::Error(-1, std::string(msg) + " (" #cond ")");                  \
  } while (0)

// Device buffer, grows on demand, freed with the handle.
template <typename T>
struct DBuf {
  T* p = nullptr;
  size_t cap = 0;
  DBuf() = default;
  DBuf(const DBuf&) = delete;
  DBuf& operator=(const DBuf&) = delete;
  ~DBuf() { release(); }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  T* ensure(size_t n) {
    if (n > cap) {
      // a buffer that has to grow again is growing with the problem (the perturbed matrices of the sparsity
      // search gain ~1 % of entries per step): cudaFree/cudaMalloc cost ~10 ms per 100 MB, so leave headroom
      const bool regrow = p != nullptr;
      release();
      size_t want = regrow ? n + n / 2 + 64 : n + n / 16 + 64;
      SCL_CUDA(cudaMalloc(&p, want * sizeof(T)));
      cap = want;
    }
    return p;
  }
  void swap(DBuf& o) {
    std::swap(p, o.p);
    std::swap(cap, o.cap);
  }
};

// Canonical device sparse matrix: CSC (gene lines) plus its CSR mirror (cell lines).
// 0-based; both orientations sorted inside a line.
struct SpMat {
  int N = 0, M = 0;
  size_t nnz = 0;
  DBuf<uint32_t> colptr, rowval, rowptr, colidx;
  DBuf<float> val, rval;
  // capacity for nnz_cap stored entries in both orientations (no-op when already large enough)
  void reserve(size_t nnz_cap) {
    rowval.ensure(nnz_cap); val.ensure(nnz_cap); colidx.ensure(nnz_cap); rval.ensure(nnz_cap);
  }
  void swap(SpMat& o) {
    std::swap(N, o.N); std::swap(M, o.M); std::swap(nnz, o.nnz);
    colptr.swap(o.colptr); rowval.swap(o.rowval); rowptr.swap(o.rowptr); colidx.swap(o.colidx);
    val.swap(o.val); rval.swap(o.rval);
  }
};

// Per-matrix normalisation statistics (SURVEY.md Appendix C), all Float64 on device.
struct NormStats {
  DBuf<double> tgc, l2, inv_s;      // per cell: r_i, l_i, 1/s_i
  DBuf<float> inv_s_f;              // float copy streamed by the densify kernels
  DBuf<double> ybar, sigma, mu, cent;  // per gene
  DBuf<float> mu_f, cent_f, inv_sigma_f;
  DBuf<double> scalars;             // [0]=|mu|^2 [1]=mean(l) [2]=sum(1/s) [3]=sum(1/s^2) [4]=mu.c [5]=|c|^2
  DBuf<double> sumsq_gene, sumsq_cell;   // exact sums of squares of the normalised matrix's columns / rows
  // parameters gathered per stored entry by the statistics passes, packed so one 32-byte sector holds them all
  DBuf<double2> cell_par;           // {1/r_i, 1/s_i}
  DBuf<double4> gene_par;           // {1/sigma_j, mu_j, c_j, -}
  DBuf<double> red_partial;         // scratch of the multi-block reductions
  DBuf<unsigned int> red_counter;
  // final value (z_ij - mu_j)/s_i - c_j of every stored entry, in CSC / CSR order: the writer's sparse patch for the
  // gene-major / cell-major layout, computed on first use (ensure_patch)
  DBuf<float> patch_csc, patch_csr;
  bool have_patch[2] = {false, false};
  // strip passes: offsets of every line's entries inside every strip, [0] gene lines (CSC) x cell strips, [1] cell
  // lines (CSR) x gene strips (shared with the dense writer), and the per-(line, strip) partial sums
  DBuf<uint32_t> off[2];
  int off_strips[2] = {0, 0};
  bool off_valid[2] = {false, false};
  DBuf<double> strip_partial;
  // centering="median" (:294-299, :653-654): per-gene median of y = log1p(x / r_i) over ALL cells replaces the mean as the
  // centre and there is no final re-centring (c_j = 0); everything downstream reads mu_j and c_j and is unchanged
  int centering = 0;                // 0 mean (default path), 1 median
  DBuf<double> median;
  void reserve(size_t nnz_cap) {
    patch_csc.ensure(nnz_cap); patch_csr.ensure(nnz_cap);
  }
};

struct Workspace;  // sparse scratch, defined in sparse.cu

// ---- sparse.cu ----
// out[0..n] = exclusive scan of in[0..n-1], out[n] = total (one CTA)
void exclusive_scan(const uint32_t* in, uint32_t* out, int n, cudaStream_t st);
void build_csr_mirror(SpMat& A, cudaStream_t st);
void upload_csc(SpMat& A, int N, int M, size_t nnz, const uint32_t* colptr, const uint32_t* rowval,
                const float* val, int index_base, cudaStream_t st);
// out = canonical( base (+ optional value override) + COO additions with value 1 )
void perturb_merge(const SpMat& base, const uint32_t* d_add_row, const uint32_t* d_add_col, size_t n_add,
                   bool binarise, SpMat& out, cudaStream_t st);
// out = canonical( (rows[t], col(t), val[perm[t]]) ) : duplicates summed
void permute_null(const SpMat& base, const uint32_t* d_perm, const uint32_t* d_rows, SpMat& out, cudaStream_t st);
// device-side draws (Feistel bijections; see draws.cu)
void draw_null_device(const SpMat& base, uint64_t seed, SpMat& out, cudaStream_t st);
size_t draw_zero_candidates_device(const SpMat& base, uint64_t seed, DBuf<uint32_t>& z1, DBuf<uint32_t>& z2,
                                   cudaStream_t st);
// grid position (row + N * col) of the t-th uniform draw behind draw_zero_candidates_device, on the host (tests)
uint64_t zero_candidate_position_host(uint64_t seed, uint64_t t, uint64_t grid);
void draw_subset_device(const uint32_t* z1, const uint32_t* z2, size_t n_cand, size_t n_take, uint64_t seed,
                        uint32_t* out_row, uint32_t* out_col, cudaStream_t st);
void gather_pairs(const uint32_t* z1, const uint32_t* z2, const uint32_t* d_idx, size_t n, uint32_t* out_row,
                  uint32_t* out_col, cudaStream_t st);
double noise_baseline_device(int nm, int n_rep, uint64_t seed, cudaStream_t st);

// ---- normalize.cu ----
void compute_norm_stats(const SpMat& A, NormStats& S, cudaStream_t st);
// sparse patch of the writer for `layout` (and, for layout 1, the cell-side Gram diagonal); no-op when already present
void ensure_patch(const SpMat& A, NormStats& S, int layout, cudaStream_t st);
// layout 0: gene-major out[M][ld] (column-major N x M); 1: cell-major out[N][ld]
// [pos0,pos1): range of positions of every line to emit (default: the whole padded line) - the cell block of a rank
void densify(const SpMat& A, NormStats& S, int layout, size_t ld, __half* out_hi, __half* out_lo,
             cudaStream_t st, long long pos0 = 0, long long pos1 = -1, size_t slice_stride = 0);
// slice_stride != 0: out_hi / out_lo hold ONLY the positions [pos0, pos1) of every line, slice_stride elements apart
void set_norm_tuning(int stat_variant, int stat_heavy, int writer);
// exact Float64 Gram diagonal (unscaled) of the normalised matrix on its gene side / cell side
const double* gram_diagonal(const SpMat& A, NormStats& S, bool gene_side, cudaStream_t st);
void set_gram_diagonal(float* G, int n, const double* sumsq, double scale, cudaStream_t st);

// ---- denoise.cu ----
void denoise(const float* dA, const float* dG, int r, int N, int M, const double* cent, const double* sigma,
             const double* ybar, const double* l2, double mean_l, double mean_tgc, void* d_out, bool out_f32,
             cudaStream_t st);

// ---- gemm_umma.cu ----
struct GemmOperand {
  const __half* hi = nullptr;
  const __half* lo = nullptr;  // optional low-order part (split mode)
  int rows = 0;                // logical rows
  int64_t K = 0;               // contraction length
  int64_t ld = 0;              // elements between rows (multiple of 8)
};
enum class Epilogue : int { Store = 0, StoreTransposed = 1, ColAbsMax = 2 };
struct GemmArgs {
  GemmOperand A, B;
  bool syrk = false;        // B == A, lower-triangular tile schedule, mirrored store
  float alpha = 1.f;
  Epilogue epi = Epilogue::Store;
  float* C = nullptr;       // Store: C[m*ldc+n]; StoreTransposed: C[n*ldc+m]; ColAbsMax: C[n] (pre-zeroed)
  int64_t ldc = 0;
  int splits = 1;           // split-K: partial s written at C + s*split_stride (caller reduces)
  int64_t split_stride = 0;
  int cta_group = 2;        // 1 or 2
  int chunk_kb = 0;         // k-blocks (of 64) per tensor-core accumulation chunk; 0 = default (64, or 21 in split mode)
};
void gemm_umma(const GemmArgs& a, cudaStream_t st);
void split_f32_to_f16(const float* in, size_t n, __half* hi, __half* lo, cudaStream_t st);
// pre_scale (a power of two) is applied before rounding so the low-order part of small entries (unit vectors in
// high dimension: ~1/sqrt(n)) stays in the normal binary16 range; the caller divides alpha by it
void strided_split_f32_to_f16(const float* in, int rows, int64_t cols, int64_t ld_in, int64_t ld_out, __half* hi,
                              __half* lo, cudaStream_t st, float pre_scale = 1.f);
void fill_random_f16(__half* out, size_t n, uint32_t seed, float scale, cudaStream_t st);   // ~N(0, scale^2), bench harness
void reduce_splits(const float* part, int splits, int64_t stride, size_t n, float scale, float* out, cudaStream_t st);
int sm_count();

}  // namespace scl
