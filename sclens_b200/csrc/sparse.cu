// Integer-exact sparse plumbing on device: CSR mirror, line canonicalisation (sort + sum
// duplicates), the perturbation merge of src/scLENS.jl:735/:774 and the null-matrix
// permutation of :239-289.  All HBM-bound; no sorting library is used - a line (one gene
// column or one cell row) is scattered into a dense shared-memory strip and compacted in
// index order, which is exactly the semantics of Julia's sparse(I,J,V) (duplicates summed,
// (col,row) order).
#include <chrono>
#include <cstdlib>
#include "common.cuh"
#include "tmp.cuh"

namespace scl {

static constexpr int kCanonChunk = 8192;  // positions per shared-memory strip (32 KB)
static constexpr int kCanonThreads = 256;

// ---------------------------------------------------------------------------------------
__global__ void k_fill_u32(uint32_t* p, uint32_t v, size_t n) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] = v;
}

// out[0..n] = exclusive scan of in[0..n-1]; out[n] = total.  One block.
__global__ void __launch_bounds__(1024) k_exclusive_scan(const uint32_t* __restrict__ in, uint32_t* __restrict__ out, int n) {
  __shared__ uint32_t part[1024];
  int tid = threadIdx.x;
  int chunk = (n + 1023) / 1024;
  int b = tid * chunk, e = min(n, b + chunk);
  uint32_t s = 0;
  for (int i = b; i < e; ++i) s += in[i];
  part[tid] = s;
  __syncthreads();
  for (int off = 1; off < 1024; off <<= 1) {
    uint32_t v = tid >= off ? part[tid - off] : 0;
    __syncthreads();
    part[tid] += v;
    __syncthreads();
  }
  uint32_t run = tid ? part[tid - 1] : 0;
  for (int i = b; i < e; ++i) {
    uint32_t v = in[i];
    out[i] = run;
    run += v;
  }
  if (tid == 1023) out[n] = part[1023];
}

__global__ void k_count_index(const uint32_t* __restrict__ idx, size_t n, uint32_t* __restrict__ cnt) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) atomicAdd(&cnt[idx[i]], 1u);
}

// One block per CSC column (grid-stride): scatter entries into row buckets.
__global__ void k_scatter_to_rows(const uint32_t* __restrict__ colptr, const uint32_t* __restrict__ rowval,
                                  const float* __restrict__ val, int M, const uint32_t* __restrict__ rowptr,
                                  uint32_t* __restrict__ cursor, uint32_t* __restrict__ out_col,
                                  float* __restrict__ out_val) {
  for (int j = blockIdx.x; j < M; j += gridDim.x) {
    uint32_t b = colptr[j], e = colptr[j + 1];
    for (uint32_t t = b + threadIdx.x; t < e; t += blockDim.x) {
      uint32_t r = rowval[t];
      uint32_t slot = atomicAdd(&cursor[r], 1u);
      uint32_t dst = rowptr[r] + slot;
      out_col[dst] = (uint32_t)j;
      out_val[dst] = val[t];
    }
  }
}

// Canonicalise lines: every line l owns the input segment [in_ptr[l], in_ptr[l+1]) of
// (pos,val) pairs in arbitrary order, possibly with duplicate pos.  Output is sorted by pos
// with duplicates summed.  COUNT_ONLY writes the distinct count per line to out_cnt.
template <bool COUNT_ONLY>
__global__ void __launch_bounds__(kCanonThreads) k_canon(const uint32_t* __restrict__ in_ptr,
                                                        const uint32_t* __restrict__ in_pos,
                                                        const float* __restrict__ in_val,
                                                        const uint32_t* __restrict__ out_ptr,
                                                        uint32_t* __restrict__ out_pos, float* __restrict__ out_val,
                                                        uint32_t* __restrict__ out_cnt, int n_lines, int line_len) {
  __shared__ float acc[kCanonChunk];
  __shared__ uint32_t warp_cnt[kCanonThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr int kWarps = kCanonThreads / 32;
  constexpr int kPerWarp = kCanonChunk / kWarps;  // 1024 positions per warp
  for (int l = blockIdx.x; l < n_lines; l += gridDim.x) {
    const uint32_t sb = in_ptr[l], se = in_ptr[l + 1];
    uint32_t written = 0;  // uniform across the block
    if (sb == se) {
      if (COUNT_ONLY && tid == 0) out_cnt[l] = 0;
      continue;
    }
    const uint32_t ob = COUNT_ONLY ? 0u : out_ptr[l];
    for (int base = 0; base < line_len; base += kCanonChunk) {
      const int len = min(kCanonChunk, line_len - base);
      for (int i = tid; i < kCanonChunk; i += kCanonThreads) acc[i] = 0.f;
      __syncthreads();
      for (uint32_t t = sb + tid; t < se; t += kCanonThreads) {
        uint32_t p = in_pos[t];
        if (p >= (uint32_t)base && p < (uint32_t)(base + len)) atomicAdd(&acc[p - base], in_val[t]);
      }
      __syncthreads();
      // pass 1: per-warp distinct counts over its 1024-position strip
      uint32_t c = 0;
      const int w0 = warp * kPerWarp;
      for (int i = 0; i < kPerWarp; i += 32) c += __popc(__ballot_sync(0xffffffffu, acc[w0 + i + lane] != 0.f));
      if (lane == 0) warp_cnt[warp] = c;
      __syncthreads();
      uint32_t wbase = 0, total = 0;
      for (int w = 0; w < kWarps; ++w) {
        uint32_t v = warp_cnt[w];
        if (w < warp) wbase += v;
        total += v;
      }
      if (!COUNT_ONLY) {
        uint32_t run = ob + written + wbase;
        for (int i = 0; i < kPerWarp; i += 32) {
          float v = acc[w0 + i + lane];
          uint32_t m = __ballot_sync(0xffffffffu, v != 0.f);
          if (v != 0.f) {
            uint32_t dst = run + __popc(m & ((1u << lane) - 1u));
            out_pos[dst] = (uint32_t)(base + w0 + i + lane);
            out_val[dst] = v;
          }
          run += __popc(m);
        }
      }
      written += total;
      __syncthreads();
    }
    if (COUNT_ONLY && tid == 0) out_cnt[l] = written;
  }
}

static inline int grid_for(size_t n, int threads, int cap = 148 * 16) {
  size_t g = (n + threads - 1) / threads;
  if (g < 1) g = 1;
  if (g > (size_t)cap) g = cap;
  return (int)g;
}

void exclusive_scan(const uint32_t* in, uint32_t* out, int n, cudaStream_t st) {
  k_exclusive_scan<<<1, 1024, 0, st>>>(in, out, n);
  SCL_CUDA(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------
void build_csr_mirror(SpMat& A, cudaStream_t st) {
  count_launches(4);
  const int N = A.N, M = A.M;
  const size_t nnz = A.nnz;
  A.rowptr.ensure(N + 1);
  A.colidx.ensure(nnz ? nnz : 1);
  A.rval.ensure(nnz ? nnz : 1);
  Tmp<uint32_t> cnt(N + 1, st), cursor(N + 1, st), tcol(nnz ? nnz : 1, st);
  Tmp<float> tval(nnz ? nnz : 1, st);
  SCL_CUDA(cudaMemsetAsync(cnt.p, 0, (N + 1) * sizeof(uint32_t), st));
  SCL_CUDA(cudaMemsetAsync(cursor.p, 0, (N + 1) * sizeof(uint32_t), st));
  if (nnz) k_count_index<<<grid_for(nnz, 256), 256, 0, st>>>(A.rowval.p, nnz, cnt.p);
  exclusive_scan(cnt.p, A.rowptr.p, N, st);
  if (nnz) {
    k_scatter_to_rows<<<min(M, 148 * 8), 128, 0, st>>>(A.colptr.p, A.rowval.p, A.val.p, M, A.rowptr.p, cursor.p,
                                                        tcol.p, tval.p);
    k_canon<false><<<min(N, 148 * 8), kCanonThreads, 0, st>>>(A.rowptr.p, tcol.p, tval.p, A.rowptr.p, A.colidx.p,
                                                              A.rval.p, nullptr, N, M);
  }
  SCL_CUDA(cudaGetLastError());
}

__global__ void k_rebase(uint32_t* p, size_t n, uint32_t base) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) p[i] -= base;
}

// canonical-form check of an uploaded CSC, one warp per column: monotone column pointers ending at nnz, rows inside
// [0, N) and strictly increasing inside a column, strictly positive finite values.  flag[0] = first kind of violation seen.
__global__ void __launch_bounds__(256) k_validate_csc(const uint32_t* __restrict__ colptr, const uint32_t* __restrict__ rowval,
                                                      const float* __restrict__ val, int N, int M, size_t nnz, int* __restrict__ flag) {
  const int lane = threadIdx.x & 31;
  for (int j = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < M; j += (gridDim.x * blockDim.x) >> 5) {
    const uint32_t b = colptr[j], e = colptr[j + 1];
    if (b > e || (size_t)e > nnz || (j == 0 && b != 0) || (j == M - 1 && (size_t)e != nnz)) {
      if (lane == 0) atomicCAS(flag, 0, 1);
      continue;
    }
    for (uint32_t t = b + lane; t < e; t += 32) {
      const uint32_t r = rowval[t];
      const float v = val[t];
      if (r >= (uint32_t)N) atomicCAS(flag, 0, 2);
      else if (t > b && rowval[t - 1] >= r) atomicCAS(flag, 0, 3);
      if (!(v > 0.f) || !(v < 3.0e38f)) atomicCAS(flag, 0, 4);
    }
  }
}

void validate_csc(const SpMat& A, cudaStream_t st) {
  Tmp<int> flag(1, st);
  SCL_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), st));
  count_launches(1);
  k_validate_csc<<<std::min((A.M + 7) / 8, 148 * 16), 256, 0, st>>>(A.colptr.p, A.rowval.p, A.val.p, A.N, A.M, A.nnz, flag.p);
  SCL_CUDA(cudaGetLastError());
  int f = 0;
  SCL_CUDA(cudaMemcpyAsync(&f, flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  static const char* what[] = {"", "column pointers are not monotone from 0 to nnz", "a row index is outside [0, N)",
                               "row indices are not strictly increasing inside a column", "a stored value is not a positive finite number"};
  if (f) throw Error(-1 /*SCL_ERR_INVALID*/, std::string("counts are not a canonical CSC matrix: ") + what[f]);
}

void upload_csc(SpMat& A, int N, int M, size_t nnz, const uint32_t* colptr, const uint32_t* rowval, const float* val,
                int index_base, cudaStream_t st) {
  A.N = N; A.M = M; A.nnz = nnz;
  A.colptr.ensure(M + 1);
  A.rowval.ensure(nnz ? nnz : 1);
  A.val.ensure(nnz ? nnz : 1);
  SCL_CUDA(cudaMemcpyAsync(A.colptr.p, colptr, (M + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  if (nnz) {
    SCL_CUDA(cudaMemcpyAsync(A.rowval.p, rowval, nnz * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    SCL_CUDA(cudaMemcpyAsync(A.val.p, val, nnz * sizeof(float), cudaMemcpyHostToDevice, st));
  }
  if (index_base) {
    k_rebase<<<grid_for(M + 1, 256), 256, 0, st>>>(A.colptr.p, M + 1, (uint32_t)index_base);
    if (nnz) k_rebase<<<grid_for(nnz, 256), 256, 0, st>>>(A.rowval.p, nnz, (uint32_t)index_base);
  }
  SCL_CUDA(cudaGetLastError());
  count_launches(index_base ? 2 : 0);
  validate_csc(A, st);          // before anything indexes with it: the mirror builder and every line pass trust the form
  build_csr_mirror(A, st);
}

// ---------------------------------------------------------------------------------------
__global__ void k_merged_counts(const uint32_t* __restrict__ colptr, const uint32_t* __restrict__ addcnt, int M,
                                uint32_t* __restrict__ cnt) {
  int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < M) cnt[j] = (colptr[j + 1] - colptr[j]) + addcnt[j];
}

__global__ void k_copy_base(const uint32_t* __restrict__ colptr, const uint32_t* __restrict__ rowval,
                            const float* __restrict__ val, int M, const uint32_t* __restrict__ newptr, bool binarise,
                            uint32_t* __restrict__ out_row, float* __restrict__ out_val) {
  for (int j = blockIdx.x; j < M; j += gridDim.x) {
    uint32_t b = colptr[j], e = colptr[j + 1], nb = newptr[j];
    for (uint32_t t = b + threadIdx.x; t < e; t += blockDim.x) {
      out_row[nb + (t - b)] = rowval[t];
      out_val[nb + (t - b)] = binarise ? 1.f : val[t];
    }
  }
}

__global__ void k_scatter_additions(const uint32_t* __restrict__ add_row, const uint32_t* __restrict__ add_col,
                                    size_t n_add, const uint32_t* __restrict__ colptr,
                                    const uint32_t* __restrict__ newptr, uint32_t* __restrict__ cursor,
                                    uint32_t* __restrict__ out_row, float* __restrict__ out_val) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n_add; i += stride) {
    uint32_t j = add_col[i];
    uint32_t slot = atomicAdd(&cursor[j], 1u);
    uint32_t dst = newptr[j] + (colptr[j + 1] - colptr[j]) + slot;
    out_row[dst] = add_row[i];
    out_val[dst] = 1.f;
  }
}

// ---- bitmap merge -----------------------------------------------------------------------
// The perturbed matrices of :735/:774 are the (sorted) base lines plus a set of ones at zero positions.
// One CTA per line: base and added positions are marked in two shared-memory bitmaps of line_len bits; a
// block-wide prefix sum over the word popcounts gives every set bit its output slot, so the merged line comes
// out sorted without sorting anything, and the base values are found by their rank in the base bitmap.
// Additions that hit a stored position or each other (impossible for draws from the zero candidates) raise
// `flag`, and the caller falls back to the general canonicalisation.
static constexpr int kMergeThreads = 256;

__global__ void k_count_adds(const uint32_t* __restrict__ add_row, const uint32_t* __restrict__ add_col, size_t n_add,
                             uint32_t* __restrict__ cnt_col, uint32_t* __restrict__ cnt_row) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n_add; i += stride) {
    atomicAdd(&cnt_col[add_col[i]], 1u);
    atomicAdd(&cnt_row[add_row[i]], 1u);
  }
}

// bucket_col[aptr_col[c] + k] = row, bucket_row[aptr_row[r] + k] = col  (unordered inside a bucket)
__global__ void k_bucket_adds(const uint32_t* __restrict__ add_row, const uint32_t* __restrict__ add_col, size_t n_add,
                              const uint32_t* __restrict__ aptr_col, const uint32_t* __restrict__ aptr_row,
                              uint32_t* __restrict__ cur_col, uint32_t* __restrict__ cur_row,
                              uint32_t* __restrict__ bucket_col, uint32_t* __restrict__ bucket_row) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n_add; i += stride) {
    const uint32_t r = add_row[i], c = add_col[i];
    bucket_col[aptr_col[c] + atomicAdd(&cur_col[c], 1u)] = r;
    bucket_row[aptr_row[r] + atomicAdd(&cur_row[r], 1u)] = c;
  }
}

__global__ void k_add_ptrs(const uint32_t* __restrict__ a, const uint32_t* __restrict__ b, int n, uint32_t* __restrict__ out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = a[i] + b[i];
}

// One CTA per line.  Shared memory: base bitmap, added bitmap, and the exclusive prefix of their word popcounts
// (4 arrays of `words` 32-bit entries).  Every stored entry and every addition then knows its output slot from two
// popcounts - slot = (entries before it in the base line) + (additions before its position) - so the base line is read and
// the merged line written by consecutive threads at consecutive (base) / monotone (merged) addresses: no per-bit loops, no
// sorting, coalesced traffic.  Additions (12 % of a line at the largest perturbation) scatter into the gaps.
__global__ void __launch_bounds__(kMergeThreads)
k_merge_lines(const uint32_t* __restrict__ base_ptr, const uint32_t* __restrict__ base_idx,
              const float* __restrict__ base_val, const uint32_t* __restrict__ add_ptr,
              const uint32_t* __restrict__ add_pos, const uint32_t* __restrict__ out_ptr, uint32_t* __restrict__ out_idx,
              float* __restrict__ out_val, int n_lines, int line_len, int binarise, int* __restrict__ flag) {
  extern __shared__ uint32_t bm[];   // [4][words]: base bits, added bits, prefix of base popcounts, prefix of added popcounts
  __shared__ unsigned long long warp_tot[kMergeThreads / 32];
  const int words = (line_len + 31) >> 5;
  uint32_t* bmB = bm;
  uint32_t* bmA = bm + words;
  uint32_t* pfB = bm + 2 * words;
  uint32_t* pfA = bm + 3 * words;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int wpt = (words + kMergeThreads - 1) / kMergeThreads;   // contiguous words per thread
  for (int l = blockIdx.x; l < n_lines; l += gridDim.x) {
    const uint32_t bb = base_ptr[l], be = base_ptr[l + 1], ab = add_ptr[l], ae = add_ptr[l + 1], ob = out_ptr[l];
    if (ae == ab) {   // nothing added to this line: copy
#pragma unroll 4
      for (uint32_t t = bb + tid; t < be; t += kMergeThreads) {
        out_idx[ob + (t - bb)] = base_idx[t];
        out_val[ob + (t - bb)] = binarise ? 1.f : base_val[t];
      }
      continue;
    }
    for (int w = tid; w < 2 * words; w += kMergeThreads) bm[w] = 0u;
    __syncthreads();
    // four independent loads per thread in flight (a line is a few thousand entries over 256 threads: without this a thread
    // waits for one 4-byte load at a time)
    for (uint32_t t0 = bb + tid; t0 < be; t0 += 4 * kMergeThreads) {
      uint32_t p[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t t = t0 + u * kMergeThreads;
        p[u] = t < be ? base_idx[t] : 0xffffffffu;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (p[u] != 0xffffffffu) atomicOr(&bmB[p[u] >> 5], 1u << (p[u] & 31));
    }
    bool bad = false;
    for (uint32_t t = ab + tid; t < ae; t += kMergeThreads) {
      const uint32_t p = add_pos[t];
      if (p >= (uint32_t)line_len) { bad = true; continue; }
      const uint32_t bit = 1u << (p & 31);
      if (atomicOr(&bmA[p >> 5], bit) & bit) bad = true;       // the same position added twice
    }
    __syncthreads();
    // exclusive prefix of the word popcounts, both bitmaps at once: (added << 32) | base
    const int w0 = min(words, tid * wpt), w1 = min(words, w0 + wpt);
    unsigned long long cnt = 0;
    for (int w = w0; w < w1; ++w) {
      const uint32_t B = bmB[w], A = bmA[w];
      if (B & A) bad = true;                                     // an addition on a stored position
      cnt += ((unsigned long long)__popc(A) << 32) | (unsigned long long)__popc(B);
    }
    unsigned long long incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += v;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    unsigned long long run = incl - cnt;
    for (int q = 0; q < warp; ++q) run += warp_tot[q];
    for (int w = w0; w < w1; ++w) {
      pfB[w] = (uint32_t)(run & 0xffffffffull);
      pfA[w] = (uint32_t)(run >> 32);
      run += ((unsigned long long)__popc(bmA[w]) << 32) | (unsigned long long)__popc(bmB[w]);
    }
    if (bad) atomicOr(flag, 1);
    __syncthreads();
    // stored entries: slot = rank in the base line + additions at smaller positions
    for (uint32_t t0 = bb + tid; t0 < be; t0 += 4 * kMergeThreads) {
      uint32_t p[4];
      float v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const uint32_t t = t0 + u * kMergeThreads;
        const bool ok = t < be;
        p[u] = ok ? base_idx[t] : 0xffffffffu;
        v[u] = (ok && !binarise) ? base_val[t] : 1.f;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        if (p[u] == 0xffffffffu) continue;
        const uint32_t t = t0 + u * kMergeThreads, w = p[u] >> 5, low = (1u << (p[u] & 31)) - 1u;
        const uint32_t slot = (t - bb) + pfA[w] + __popc(bmA[w] & low);
        out_idx[ob + slot] = p[u];
        out_val[ob + slot] = v[u];
      }
    }
    // additions: slot = additions at smaller positions + stored entries at smaller positions; value 1 (:735, :774)
    for (uint32_t t = ab + tid; t < ae; t += kMergeThreads) {
      const uint32_t p = add_pos[t];
      if (p >= (uint32_t)line_len) continue;
      const uint32_t w = p >> 5, low = (1u << (p & 31)) - 1u;
      const uint32_t slot = pfA[w] + __popc(bmA[w] & low) + pfB[w] + __popc(bmB[w] & low);
      out_idx[ob + slot] = p;
      out_val[ob + slot] = 1.f;
    }
    __syncthreads();   // bitmaps, prefixes and warp_tot are reused by the next line
  }
}

static void perturb_merge_general(const SpMat& base, const uint32_t* d_add_row, const uint32_t* d_add_col, size_t n_add,
                                  bool binarise, SpMat& out, cudaStream_t st);

void perturb_merge(const SpMat& base, const uint32_t* d_add_row, const uint32_t* d_add_col, size_t n_add,
                   bool binarise, SpMat& out, cudaStream_t st) {
  const int N = base.N, M = base.M;
  const size_t nnz = base.nnz + n_add;
  const size_t smem_c = (size_t)4 * ((N + 31) / 32) * sizeof(uint32_t), smem_r = (size_t)4 * ((M + 31) / 32) * sizeof(uint32_t);
  if (smem_c > 200 * 1024 || smem_r > 200 * 1024) {   // a line's bitmaps must fit in shared memory
    perturb_merge_general(base, d_add_row, d_add_col, n_add, binarise, out, st);
    return;
  }
  count_launches(n_add ? 8 : 4);
  static const bool trace = getenv("SCL_TRACE") != nullptr;
  auto now = [] { return std::chrono::steady_clock::now(); };
  auto ms_since = [&](std::chrono::steady_clock::time_point t) { return std::chrono::duration<double, std::milli>(now() - t).count(); };
  const auto t_begin = now();
  out.N = N; out.M = M; out.nnz = nnz;
  out.colptr.ensure(M + 1); out.rowptr.ensure(N + 1);
  out.rowval.ensure(nnz ? nnz : 1); out.val.ensure(nnz ? nnz : 1);
  out.colidx.ensure(nnz ? nnz : 1); out.rval.ensure(nnz ? nnz : 1);
  Tmp<uint32_t> cnt((size_t)M + N + 2, st), aptr((size_t)M + N + 2, st), cur((size_t)M + N + 2, st);
  Tmp<uint32_t> bucket_col(n_add ? n_add : 1, st), bucket_row(n_add ? n_add : 1, st);
  Tmp<int> flag(1, st);
  uint32_t *cnt_col = cnt.p, *cnt_row = cnt.p + M + 1, *aptr_col = aptr.p, *aptr_row = aptr.p + M + 1;
  uint32_t *cur_col = cur.p, *cur_row = cur.p + M + 1;
  const double t_alloc = ms_since(t_begin);
  SCL_CUDA(cudaMemsetAsync(cnt.p, 0, ((size_t)M + N + 2) * sizeof(uint32_t), st));
  SCL_CUDA(cudaMemsetAsync(cur.p, 0, ((size_t)M + N + 2) * sizeof(uint32_t), st));
  SCL_CUDA(cudaMemsetAsync(flag.p, 0, sizeof(int), st));
  if (n_add) k_count_adds<<<grid_for(n_add, 256), 256, 0, st>>>(d_add_row, d_add_col, n_add, cnt_col, cnt_row);
  exclusive_scan(cnt_col, aptr_col, M, st);
  exclusive_scan(cnt_row, aptr_row, N, st);
  if (n_add)
    k_bucket_adds<<<grid_for(n_add, 256), 256, 0, st>>>(d_add_row, d_add_col, n_add, aptr_col, aptr_row, cur_col, cur_row,
                                                        bucket_col.p, bucket_row.p);
  k_add_ptrs<<<(M + 256) / 256, 256, 0, st>>>(base.colptr.p, aptr_col, M + 1, out.colptr.p);
  k_add_ptrs<<<(N + 256) / 256, 256, 0, st>>>(base.rowptr.p, aptr_row, N + 1, out.rowptr.p);
  SCL_CUDA(cudaFuncSetAttribute(k_merge_lines, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  k_merge_lines<<<min(M, 148 * 8), kMergeThreads, smem_c, st>>>(base.colptr.p, base.rowval.p, base.val.p, aptr_col,
                                                                bucket_col.p, out.colptr.p, out.rowval.p, out.val.p, M, N,
                                                                binarise ? 1 : 0, flag.p);
  k_merge_lines<<<min(N, 148 * 8), kMergeThreads, smem_r, st>>>(base.rowptr.p, base.colidx.p, base.rval.p, aptr_row,
                                                                bucket_row.p, out.rowptr.p, out.colidx.p, out.rval.p, N, M,
                                                                binarise ? 1 : 0, flag.p);
  SCL_CUDA(cudaGetLastError());
  int bad = 0;
  const double t_launch = ms_since(t_begin);
  SCL_CUDA(cudaMemcpyAsync(&bad, flag.p, sizeof(int), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  if (trace)
    fprintf(stderr, "[scl] perturb_merge n_add=%zu: alloc %.3f ms, launched at %.3f ms, done at %.3f ms, fallback=%d\n", n_add,
            t_alloc, t_launch, ms_since(t_begin), bad);
  if (bad) perturb_merge_general(base, d_add_row, d_add_col, n_add, binarise, out, st);   // sparse(I,J,V) sums them
}

// General path: any additions (coinciding with stored entries or with each other); lines are canonicalised.
static void perturb_merge_general(const SpMat& base, const uint32_t* d_add_row, const uint32_t* d_add_col, size_t n_add,
                                  bool binarise, SpMat& out, cudaStream_t st) {
  count_launches(n_add ? 6 : 4);
  const int N = base.N, M = base.M;
  const size_t nnz = base.nnz + n_add;
  out.N = N; out.M = M;
  out.colptr.ensure(M + 1);
  Tmp<uint32_t> addcnt(M + 1, st), cnt(M + 1, st), tptr(M + 1, st), cursor(M + 1, st), trow(nnz ? nnz : 1, st);
  Tmp<float> tval(nnz ? nnz : 1, st);
  SCL_CUDA(cudaMemsetAsync(addcnt.p, 0, (M + 1) * sizeof(uint32_t), st));
  SCL_CUDA(cudaMemsetAsync(cursor.p, 0, (M + 1) * sizeof(uint32_t), st));
  if (n_add) k_count_index<<<grid_for(n_add, 256), 256, 0, st>>>(d_add_col, n_add, addcnt.p);
  k_merged_counts<<<(M + 255) / 256, 256, 0, st>>>(base.colptr.p, addcnt.p, M, cnt.p);
  exclusive_scan(cnt.p, tptr.p, M, st);
  k_copy_base<<<min(M, 148 * 8), 128, 0, st>>>(base.colptr.p, base.rowval.p, base.val.p, M, tptr.p, binarise,
                                               trow.p, tval.p);
  if (n_add)
    k_scatter_additions<<<grid_for(n_add, 256), 256, 0, st>>>(d_add_row, d_add_col, n_add, base.colptr.p,
                                                              tptr.p, cursor.p, trow.p, tval.p);
  // duplicates are summed, so the canonical lines can be shorter than the staged ones: count, scan, emit
  k_canon<true><<<min(M, 148 * 8), kCanonThreads, 0, st>>>(tptr.p, trow.p, tval.p, nullptr, nullptr, nullptr, cnt.p, M, N);
  exclusive_scan(cnt.p, out.colptr.p, M, st);
  uint32_t total = 0;
  SCL_CUDA(cudaMemcpyAsync(&total, out.colptr.p + M, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  out.nnz = total;
  out.rowval.ensure(total ? total : 1);
  out.val.ensure(total ? total : 1);
  k_canon<false><<<min(M, 148 * 8), kCanonThreads, 0, st>>>(tptr.p, trow.p, tval.p, out.colptr.p, out.rowval.p,
                                                            out.val.p, nullptr, M, N);
  SCL_CUDA(cudaGetLastError());
  build_csr_mirror(out, st);
}

// ---------------------------------------------------------------------------------------
__global__ void k_gather_f32(const float* __restrict__ src, const uint32_t* __restrict__ perm, size_t n,
                             float* __restrict__ dst) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) dst[i] = src[perm[i]];
}

// Shared tail of the null-matrix builders: (trow, tval) hold, per base column segment, the
// new rows and shuffled values; canonicalise with duplicate summation.
static void finish_null(const SpMat& base, const uint32_t* trow, const float* tval, SpMat& out, cudaStream_t st) {
  count_launches(3);
  const int N = base.N, M = base.M;
  out.N = N; out.M = M;
  out.colptr.ensure(M + 1);
  Tmp<uint32_t> cnt(M + 1, st);
  k_canon<true><<<min(M, 148 * 8), kCanonThreads, 0, st>>>(base.colptr.p, trow, tval, nullptr, nullptr, nullptr, cnt.p,
                                                           M, N);
  exclusive_scan(cnt.p, out.colptr.p, M, st);
  uint32_t total = 0;
  SCL_CUDA(cudaMemcpyAsync(&total, out.colptr.p + M, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  out.nnz = total;
  out.rowval.ensure(total ? total : 1);
  out.val.ensure(total ? total : 1);
  k_canon<false><<<min(M, 148 * 8), kCanonThreads, 0, st>>>(base.colptr.p, trow, tval, out.colptr.p, out.rowval.p,
                                                            out.val.p, nullptr, M, N);
  SCL_CUDA(cudaGetLastError());
  build_csr_mirror(out, st);
}

void permute_null(const SpMat& base, const uint32_t* d_perm, const uint32_t* d_rows, SpMat& out, cudaStream_t st) {
  count_launches(1);
  const size_t nnz = base.nnz;
  Tmp<float> tval(nnz ? nnz : 1, st);
  if (nnz) k_gather_f32<<<grid_for(nnz, 256), 256, 0, st>>>(base.val.p, d_perm, nnz, tval.p);
  finish_null(base, d_rows, tval.p, out, st);
}

// ---------------------------------------------------------------------------------------
// Device-side draws.  A keyed Feistel network on ceil(log2 n) bits with cycle walking is a
// bijection of [0,n): perm(t) is computed independently per element, so a random
// permutation / a without-replacement sample costs one pass and no sort.
__host__ __device__ inline uint64_t mix64(uint64_t x) {
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ull;
  x ^= x >> 27; x *= 0x94d049bb133111ebull;
  x ^= x >> 31;
  return x;
}

struct Feistel {
  uint64_t n;
  uint32_t half_bits;   // bits per half
  uint64_t keys[8];
  __host__ static Feistel make(uint64_t n, uint64_t seed) {
    Feistel f;
    f.n = n;
    uint32_t bits = 2;
    while (bits < 64 && (1ull << bits) < n) ++bits;
    if (bits & 1) ++bits;
    f.half_bits = bits / 2;
    for (int r = 0; r < 8; ++r) f.keys[r] = mix64(seed + 0x9e3779b97f4a7c15ull * (uint64_t)(r + 1));
    return f;
  }
  __host__ __device__ inline uint64_t encrypt(uint64_t x) const {
    const uint64_t mask = (1ull << half_bits) - 1ull;
    uint64_t L = x >> half_bits, R = x & mask;
#pragma unroll
    for (int r = 0; r < 8; ++r) {
      uint64_t F = mix64(R ^ keys[r]) & mask;
      uint64_t nl = R;
      R = L ^ F;
      L = nl;
    }
    return (L << half_bits) | R;
  }
  __host__ __device__ inline uint64_t operator()(uint64_t t) const {
    uint64_t x = encrypt(t);
    while (x >= n) x = encrypt(x);
    return x;
  }
};

// Null matrix, aligned semantics: gene j receives count_j distinct uniformly random rows
// (:247) and globally shuffled values (:275).  One block per gene; rows are drawn by
// rejection against a shared-memory bitmap (the complement is drawn for dense genes).
__global__ void __launch_bounds__(256) k_null_rows(const uint32_t* __restrict__ colptr, int N, int M, uint64_t seed,
                                                   uint32_t* __restrict__ out_row) {
  extern __shared__ uint32_t bitmap[];  // ceil(N/32) words
  __shared__ uint32_t accepted;
  __shared__ uint32_t warp_cnt[8];
  const int words = (N + 31) / 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int j = blockIdx.x; j < M; j += gridDim.x) {
    const uint32_t b = colptr[j], cnt = colptr[j + 1] - b;
    if (cnt == 0) continue;
    const bool complement = cnt > (uint32_t)N / 2;
    const uint32_t target = complement ? (uint32_t)N - cnt : cnt;
    for (int w = tid; w < words; w += blockDim.x) bitmap[w] = 0;
    if (tid == 0) accepted = 0;
    __syncthreads();
    uint64_t ctr = 0;
    // rounds of proposals: at most `remaining` threads propose, so the count never overshoots
    while (true) {
      __syncthreads();
      const uint32_t have = accepted;
      __syncthreads();
      if (have >= target) break;
      if ((uint32_t)tid < target - have) {
        uint64_t h = mix64(seed ^ mix64(((uint64_t)j << 32) ^ (ctr * blockDim.x + tid)));
        uint32_t r = (uint32_t)(((h >> 32) * (uint64_t)N) >> 32);
        uint32_t bit = 1u << (r & 31);
        uint32_t prev = atomicOr(&bitmap[r >> 5], bit);
        if (!(prev & bit)) atomicAdd(&accepted, 1u);
      }
      ++ctr;
    }
    // emit rows in ascending order (set bits, or clear bits when the complement was drawn)
    uint32_t run = 0;
    for (int w0 = 0; w0 < words; w0 += blockDim.x) {
      int w = w0 + tid;
      uint32_t bits = 0;
      if (w < words) {
        bits = bitmap[w];
        if (complement) bits = ~bits;
        int valid = N - w * 32;
        if (valid < 32) bits &= (valid <= 0) ? 0u : ((1u << valid) - 1u);
      }
      uint32_t c = __popc(bits);
      // block exclusive prefix of c
      uint32_t incl = c;
      for (int o = 1; o < 32; o <<= 1) {
        uint32_t v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
      }
      if (lane == 31) warp_cnt[warp] = incl;
      __syncthreads();
      uint32_t wb = 0, tot = 0;
      for (int q = 0; q < 8; ++q) {
        uint32_t v = warp_cnt[q];
        if (q < warp) wb += v;
        tot += v;
      }
      uint32_t dst = b + run + wb + incl - c;
      while (bits) {
        int k = __ffs(bits) - 1;
        bits &= bits - 1;
        out_row[dst++] = (uint32_t)(w * 32 + k);
      }
      run += tot;
      __syncthreads();
    }
  }
}

__global__ void k_feistel_gather_f32(const float* __restrict__ src, Feistel f, float* __restrict__ dst) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < f.n; i += stride) dst[i] = src[f(i)];
}

void draw_null_device(const SpMat& base, uint64_t seed, SpMat& out, cudaStream_t st) {
  count_launches(2);
  const size_t nnz = base.nnz;
  SCL_REQUIRE(nnz > 0, "empty matrix");
  // k_null_rows emits every gene's rows ascending and distinct, so the canonical CSC of the null matrix is
  // written in place: same column pointers, new rows, values moved by one keyed bijection of [0, nnz)
  out.N = base.N; out.M = base.M; out.nnz = nnz;
  out.colptr.ensure(base.M + 1);
  out.rowval.ensure(nnz);
  out.val.ensure(nnz);
  SCL_CUDA(cudaMemcpyAsync(out.colptr.p, base.colptr.p, (base.M + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
  size_t smem = ((size_t)base.N + 31) / 32 * sizeof(uint32_t);
  SCL_REQUIRE(smem <= 200 * 1024, "N too large for the shared-memory row bitmap");
  SCL_CUDA(cudaFuncSetAttribute(k_null_rows, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  k_null_rows<<<min(base.M, 148 * 4), 256, smem, st>>>(base.colptr.p, base.N, base.M, mix64(seed ^ 0x6e756c6cull),
                                                      out.rowval.p);
  Feistel f = Feistel::make(nnz, mix64(seed ^ 0x73687566ull));
  k_feistel_gather_f32<<<grid_for(nnz, 256), 256, 0, st>>>(base.val.p, f, out.val.p);
  SCL_CUDA(cudaGetLastError());
  build_csr_mirror(out, st);
}

// Zero candidates (:668-673), the reference's own recipe on the device: nnz independent uniform grid positions (draw t
// is a pure function of (seed, t): counter-based, no state), minus the non-zero set (binary search in the gene's sorted
// row list), de-duplicated keeping the FIRST occurrence, in draw order - `setdiff(sample_idx, z_idset)`.  First occurrence
// is decided deterministically: an open-addressing table holds, per drawn position, the smallest draw index that hit it
// (the table stores draw indices only - the position of a stored draw is recomputed from its index).
__host__ __device__ inline uint64_t zc_position(uint64_t seed, uint64_t t, uint64_t grid) {
  const uint64_t h = mix64(seed ^ mix64(t + 0x632be59bd9b4e019ull));
#ifdef __CUDA_ARCH__
  return __umul64hi(h, grid);
#else
  return (uint64_t)(((unsigned __int128)h * grid) >> 64);
#endif
}

__global__ void k_zc_insert(uint64_t seed, uint64_t grid, size_t n_draw, uint32_t* __restrict__ table, uint32_t mask) {
  size_t t = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; t < n_draw; t += stride) {
    const uint64_t pos = zc_position(seed, t, grid);
    uint32_t slot = (uint32_t)mix64(pos) & mask;
    while (true) {
      const uint32_t cur = atomicCAS(table + slot, 0xffffffffu, (uint32_t)t);
      if (cur == 0xffffffffu) break;                                   // claimed an empty slot
      if (zc_position(seed, cur, grid) == pos) {                       // the slot of this position: keep the earliest draw
        atomicMin(table + slot, (uint32_t)t);
        break;
      }
      slot = (slot + 1) & mask;
    }
  }
}

__global__ void k_zero_cand_flags(const uint32_t* __restrict__ colptr, const uint32_t* __restrict__ rowval, int N,
                                  uint64_t seed, uint64_t grid, const uint32_t* __restrict__ table, uint32_t mask, size_t T,
                                  uint32_t* __restrict__ cand_row, uint32_t* __restrict__ cand_col,
                                  uint32_t* __restrict__ block_cnt) {
  __shared__ uint32_t wc[8];
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  bool keep = false;
  uint32_t r = 0, c = 0;
  if (i < T) {
    const uint64_t g = zc_position(seed, i, grid);
    c = (uint32_t)(g / (uint64_t)N);
    r = (uint32_t)(g % (uint64_t)N);
    uint32_t lo = colptr[c], hi = colptr[c + 1];
    while (lo < hi) {
      uint32_t mid = (lo + hi) >> 1;
      if (rowval[mid] < r) lo = mid + 1; else hi = mid;
    }
    keep = !(lo < colptr[c + 1] && rowval[lo] == r);
    if (keep) {   // first occurrence of this position among the draws?
      uint32_t slot = (uint32_t)mix64(g) & mask;
      while (true) {
        const uint32_t cur = table[slot];
        if (cur == 0xffffffffu) { keep = false; break; }               // cannot happen: every draw was inserted
        if (zc_position(seed, cur, grid) == g) { keep = cur == (uint32_t)i; break; }
        slot = (slot + 1) & mask;
      }
    }
    cand_row[i] = keep ? r : 0xffffffffu;
    cand_col[i] = c;
  }
  uint32_t m = __ballot_sync(0xffffffffu, keep);
  if ((threadIdx.x & 31) == 0) wc[threadIdx.x >> 5] = __popc(m);
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t s = 0;
    for (int q = 0; q < 8; ++q) s += wc[q];
    block_cnt[blockIdx.x] = s;
  }
}

__global__ void k_zero_cand_compact(const uint32_t* __restrict__ cand_row, const uint32_t* __restrict__ cand_col,
                                    size_t T, const uint32_t* __restrict__ block_off, uint32_t* __restrict__ z1,
                                    uint32_t* __restrict__ z2) {
  __shared__ uint32_t wc[8];
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  uint32_t r = i < T ? cand_row[i] : 0xffffffffu;
  bool keep = r != 0xffffffffu;
  uint32_t m = __ballot_sync(0xffffffffu, keep);
  int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) wc[warp] = __popc(m);
  __syncthreads();
  uint32_t wb = 0;
  for (int q = 0; q < warp; ++q) wb += wc[q];
  if (keep) {
    uint32_t dst = block_off[blockIdx.x] + wb + __popc(m & ((1u << lane) - 1u));
    z1[dst] = r;
    z2[dst] = cand_col[i];
  }
}

size_t draw_zero_candidates_device(const SpMat& base, uint64_t seed, DBuf<uint32_t>& z1, DBuf<uint32_t>& z2,
                                   cudaStream_t st) {
  count_launches(4);
  const uint64_t grid = (uint64_t)base.N * (uint64_t)base.M;
  const size_t T = base.nnz;                        // the reference draws length(nz_val) pairs (:669)
  SCL_REQUIRE(T > 0 && T < 0xffffffffull, "empty matrix, or too many stored entries for 32-bit draw indices");
  const uint64_t key = mix64(seed ^ 0x7a65726full);
  size_t cap = 1;
  while (cap < 2 * T) cap <<= 1;                    // load factor <= 1/2
  SCL_REQUIRE(cap <= (1ull << 32), "draw table too large");
  const uint32_t mask = (uint32_t)(cap - 1);
  Tmp<uint32_t> table(cap, st);
  SCL_CUDA(cudaMemsetAsync(table.p, 0xff, cap * sizeof(uint32_t), st));
  k_zc_insert<<<grid_for(T, 256), 256, 0, st>>>(key, grid, T, table.p, mask);
  const int threads = 256;
  const size_t blocks = (T + threads - 1) / threads;
  SCL_REQUIRE(blocks < (1ull << 31), "too many candidate blocks");
  Tmp<uint32_t> crow(T, st), ccol(T, st), bcnt(blocks + 1, st), boff(blocks + 1, st);
  k_zero_cand_flags<<<(unsigned)blocks, threads, 0, st>>>(base.colptr.p, base.rowval.p, base.N, key, grid, table.p, mask, T,
                                                          crow.p, ccol.p, bcnt.p);
  exclusive_scan(bcnt.p, boff.p, (int)blocks, st);
  uint32_t total = 0;
  SCL_CUDA(cudaMemcpyAsync(&total, boff.p + blocks, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  z1.ensure(total ? total : 1);
  z2.ensure(total ? total : 1);
  k_zero_cand_compact<<<(unsigned)blocks, threads, 0, st>>>(crow.p, ccol.p, T, boff.p, z1.p, z2.p);
  SCL_CUDA(cudaGetLastError());
  return total;
}

// the draw the kernels make, restated for the tests: grid position of draw t (host)
uint64_t zero_candidate_position_host(uint64_t seed, uint64_t t, uint64_t grid) {
  return zc_position(mix64(seed ^ 0x7a65726full), t, grid);
}

// sample(1:n_cand, n_take, replace=false) (:731, :772) as the first n_take images of a keyed
// bijection of [0,n_cand); gathers the (row,col) pairs directly.
__global__ void k_subset_pairs(const uint32_t* __restrict__ z1, const uint32_t* __restrict__ z2, Feistel f,
                               size_t n_take, uint32_t* __restrict__ out_row, uint32_t* __restrict__ out_col) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n_take; i += stride) {
    uint64_t s = f(i);
    out_row[i] = z1[s];
    out_col[i] = z2[s];
  }
}

void draw_subset_device(const uint32_t* z1, const uint32_t* z2, size_t n_cand, size_t n_take, uint64_t seed,
                        uint32_t* out_row, uint32_t* out_col, cudaStream_t st) {
  SCL_REQUIRE(n_take <= n_cand, "sample larger than the candidate pool");
  if (!n_take) return;
  count_launches(1);
  Feistel f = Feistel::make(n_cand, seed);
  k_subset_pairs<<<grid_for(n_take, 256), 256, 0, st>>>(z1, z2, f, n_take, out_row, out_col);
  SCL_CUDA(cudaGetLastError());
}

__global__ void k_gather_pairs(const uint32_t* __restrict__ z1, const uint32_t* __restrict__ z2,
                               const uint32_t* __restrict__ idx, size_t n, uint32_t* __restrict__ out_row,
                               uint32_t* __restrict__ out_col) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    uint32_t s = idx[i];
    out_row[i] = z1[s];
    out_col[i] = z2[s];
  }
}

void gather_pairs(const uint32_t* z1, const uint32_t* z2, const uint32_t* d_idx, size_t n, uint32_t* out_row,
                  uint32_t* out_col, cudaStream_t st) {
  if (!n) return;
  count_launches(1);
  k_gather_pairs<<<grid_for(n, 256), 256, 0, st>>>(z1, z2, d_idx, n, out_row, out_col);
  SCL_CUDA(cudaGetLastError());
}

// Noise baseline (:709-712): mean over n_rep blocks of max_{nm} |N(0,1/nm)|.
__global__ void __launch_bounds__(256) k_noise_baseline(int nm, uint64_t seed, double* __restrict__ out_max) {
  __shared__ float red[8];
  const uint64_t rep = blockIdx.x;
  float m = 0.f;
  for (int i = threadIdx.x; i < (nm + 1) / 2; i += blockDim.x) {
    uint64_t h = mix64(seed ^ mix64((rep << 32) ^ (uint64_t)i));
    float u1 = ((uint32_t)(h >> 40) + 1u) * (1.0f / 16777217.0f);   // (0,1]
    float u2 = (uint32_t)(h & 0xffffffu) * (1.0f / 16777216.0f);
    float rad = sqrtf(-2.f * logf(u1));
    float s, c;
    sincospif(2.f * u2, &s, &c);
    m = fmaxf(m, fabsf(rad * c));
    if (2 * i + 1 < nm) m = fmaxf(m, fabsf(rad * s));
  }
  for (int o = 16; o; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int q = 1; q < 8; ++q) m = fmaxf(m, red[q]);
    out_max[rep] = (double)m;
  }
}

double noise_baseline_device(int nm, int n_rep, uint64_t seed, cudaStream_t st) {
  count_launches(1);
  Tmp<double> mx(n_rep, st);
  k_noise_baseline<<<n_rep, 256, 0, st>>>(nm, mix64(seed ^ 0x70746821ull), mx.p);
  SCL_CUDA(cudaGetLastError());
  std::vector<double> h(n_rep);
  SCL_CUDA(cudaMemcpyAsync(h.data(), mx.p, n_rep * sizeof(double), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  double s = 0;
  for (double v : h) s += v;
  return s / n_rep * sqrt(1.0 / nm);
}

}  // namespace scl
