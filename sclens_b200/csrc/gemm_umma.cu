// tcgen05 / TMEM / TMA GEMM for sm_100a:  C[m,n] = alpha * sum_k A[m,k] * B[n,k]
// ("TN": both operands K-major binary16, FP32 accumulation in tensor memory).
//
// Serves every dense contraction of the sclens() path:
//   * Wishart/Gram  X^T X / size(X,2)  (src/scLENS.jl:332-344)  -> syrk mode: lower-triangular
//     tile schedule, result mirrored so the full symmetric matrix is materialised exactly once
//   * corr_mat |V^T W| column maxima (:363-373, :742)           -> ColAbsMax epilogue
//   * back-projection X * V diag(1/sqrt(L)) (:503-505, :556-558), gene_basis (:814-816),
//     subspace-iteration products                                -> Store / StoreTransposed
//
// Structure (one persistent CTA, or CTA pair with cta_group::2, per SM):
//   warp 0   TMA producer   cp.async.bulk.tensor 128B-swizzled tiles into a multi-stage ring
//   warp 1   MMA issuer     one thread issues tcgen05.mma (M=128*cta_group, N<=256, K=16)
//   warp 2   TMEM allocator 512 columns = two accumulator stages of 256 FP32 columns
//   warps 4-7 epilogue      tcgen05.ld -> registers -> global (overlaps the next tile's MMAs)
// Optional split precision: operands arrive as hi+lo binary16 pairs and three MMAs
// (hi*hi + hi*lo + lo*hi) accumulate into the same TMEM tile (~FP32 accuracy).
#include <cuda.h>
#include "common.cuh"
#include "tmp.cuh"

namespace scl {

namespace {

constexpr int kBlockK = 64;                 // binary16 elements per 128-byte swizzle row
constexpr int kTileRowsA = 128;             // A rows per CTA (UMMA M = 128 * cta_group)
constexpr int kMaxBlockN = 256;             // UMMA N
constexpr int kThreads = 256;
constexpr int kEpiWarp0 = 4;
constexpr uint32_t kTmemCols = 512;
constexpr int kSmemBudget = 192 * 1024;     // operand ring
constexpr int kEpiPitch = 36;               // floats per row of an epilogue warp's 32 x 32 staging block (16-byte rows)
constexpr int kEpiStageBytes = 4 * 32 * kEpiPitch * 4;

struct Tile {
  int tm, tn, split, diag;  // diag: tile touches the diagonal band (syrk)
};

struct KParams {
  const Tile* tiles;
  int n_tiles;
  int m_rows, n_rows;
  int k_blocks_total;   // ceil(K / 64)
  int splits;
  int block_n;          // UMMA N (multiple of 16, <= 256)
  int chunk_kb;         // k-blocks accumulated by the tensor core before the chunk is promoted into the FP32 sum
  int chunked;          // 1: TMEM columns [0,256) = chunk accumulator, [256,512) = running FP32 sum (one stage)
                        // 0: the whole K range fits one chunk; two accumulator stages overlap epilogue and MMAs
  int syrk;
  int epi;
  float alpha;
  float* C;
  long long ldc;
  long long split_stride;
};

// ---- PTX wrappers ---------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t addr = smem_u32(bar);
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "WAIT_LOOP:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra DONE;\n\t"
      "bra WAIT_LOOP;\n\t"
      "DONE:\n\t"
      "}" ::"r"(addr), "r"(parity) : "memory");
}
// arrive on the barrier at the same offset in CTA `cta` of the cluster
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t* bar, uint32_t cta) {
  asm volatile(
      "{\n\t"
      ".reg .b32 remote;\n\t"
      "mapa.shared::cluster.u32 remote, %0, %1;\n\t"
      "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [remote];\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(cta) : "memory");
}
__device__ __forceinline__ void mbar_arrive_local(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int CG>
__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
  if constexpr (CG == 1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
  } else {
    // both CTAs of the pair signal the leader's barrier (peer bit cleared)
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], "
        "[%2];" ::"r"(smem_u32(dst)),
        "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & 0xFEFFFFFFu), "r"(c0), "r"(c1)
        : "memory");
  }
}

template <int CG>
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
  if constexpr (CG == 1) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}

// tcgen05.commit: the barrier is signalled once all previously issued MMAs have retired.
template <int CG>
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  if constexpr (CG == 1) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
  } else {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"((uint16_t)3)
        : "memory");
  }
}

template <int CG>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t cols) {
  if constexpr (CG == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  } else {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
  }
}
template <int CG>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t cols) {
  if constexpr (CG == 1)
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
  else
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(cols) : "memory");
}

__device__ __forceinline__ void tmem_ld_32x32b_x32_nowait(uint32_t taddr, uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}

// K-major, 128-byte swizzle shared-memory matrix descriptor (8-row groups 1024 B apart).
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);   // start address
  d |= (uint64_t)0 << 16;                       // leading byte offset (unused for swizzled K-major)
  d |= (uint64_t)(1024 >> 4) << 32;             // stride byte offset
  d |= (uint64_t)1 << 46;                       // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                       // SWIZZLE_128B
  return d;
}

// kind::f16 instruction descriptor: F16 x F16 -> F32, both operands K-major.
__device__ __forceinline__ uint32_t make_idesc(uint32_t M, uint32_t N) {
  uint32_t d = 0;
  d |= 1u << 4;            // c_format = F32
  d |= 0u << 7;            // a_format = F16
  d |= 0u << 10;           // b_format = F16
  d |= (N >> 3) << 17;     // n_dim
  d |= (M >> 4) << 24;     // m_dim
  return d;
}

template <int CG, bool SPLIT>
struct Cfg {
  static constexpr int kRowsB = kMaxBlockN / CG;                  // B rows held by one CTA
  static constexpr int kBytesA = kTileRowsA * 128;                // 16 KB
  static constexpr int kBytesB = kRowsB * 128;                    // 32 KB (cta_group 1) / 16 KB (cta_group 2)
  static constexpr int kStageBytes = (kBytesA + kBytesB) * (SPLIT ? 2 : 1);
  static constexpr int kStages = kSmemBudget / kStageBytes;
  static constexpr int kSmemBytes = kStages * kStageBytes + kEpiStageBytes + 1024 /*align*/ + 256 /*barriers*/;
};

// ---- epilogue output paths ---------------------------------------------------------------
// A warp holds a 32 x 32 block of the result: lane = row (TMEM lane), x[i] = column i.
// Row-major destinations go through a per-warp shared-memory transpose so that every store
// instruction writes whole 128-byte row segments; column-major destinations (the syrk mirror,
// StoreTransposed) are already contiguous across lanes.
struct EpiBlock {
  float* stg;      // this warp's staging block [32][kEpiPitch]
  int lane;
  int row0;        // global row of lane 0
  int gc0;         // global column of x[0]
  int m_rows, n_rows;
};

// dst[(row0 + r) * ldc + gc0 + c] = x_r[c]   for c <= r - diag_shift when lower_only (diag_shift = gc0 - row0)
__device__ __forceinline__ void store_rowmajor(const EpiBlock& e, const float (&x)[32], float* __restrict__ C, long long ldc,
                                               bool lower_only) {
#pragma unroll
  for (int i = 0; i < 32; i += 4)
    *reinterpret_cast<float4*>(e.stg + e.lane * kEpiPitch + i) = make_float4(x[i], x[i + 1], x[i + 2], x[i + 3]);
  __syncwarp();
  float* base = C + (long long)e.row0 * ldc + e.gc0;
  const bool full = e.row0 + 32 <= e.m_rows && e.gc0 + 32 <= e.n_rows;
  const bool interior = !lower_only || e.gc0 + 31 <= e.row0;
  if (full && interior && (ldc & 3) == 0 && (reinterpret_cast<uintptr_t>(base) & 15) == 0) {
    const int rr = e.lane >> 3, cc = (e.lane & 7) * 4;     // 4 rows x 128 bytes per instruction
#pragma unroll
    for (int r = 0; r < 32; r += 4)
      *reinterpret_cast<float4*>(base + (long long)(r + rr) * ldc + cc) =
          *reinterpret_cast<const float4*>(e.stg + (r + rr) * kEpiPitch + cc);
  } else {
    const int c = e.gc0 + e.lane;
#pragma unroll 4
    for (int r = 0; r < 32; ++r) {
      const int gr = e.row0 + r;
      if (gr < e.m_rows && c < e.n_rows && (!lower_only || c <= gr)) base[(long long)r * ldc + e.lane] = e.stg[r * kEpiPitch + e.lane];
    }
  }
  __syncwarp();
}

// dst[(gc0 + c) * ldc + row0 + lane] = x[c]   (strict: skip c == row when strict_upper, the diagonal is written once)
__device__ __forceinline__ void store_colmajor(const EpiBlock& e, const float (&x)[32], float* __restrict__ C, long long ldc,
                                               bool strict_lower_src) {
  const int r = e.row0 + e.lane;
  if (r >= e.m_rows) return;
  float* base = C + (long long)e.gc0 * ldc + r;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    const int c = e.gc0 + i;
    if (c < e.n_rows && (!strict_lower_src || c < r)) base[(long long)i * ldc] = x[i];
  }
}

template <int CG, bool SPLIT>
__global__ void __launch_bounds__(kThreads, 1)
k_gemm_umma(const __grid_constant__ CUtensorMap mapA_hi, const __grid_constant__ CUtensorMap mapA_lo,
            const __grid_constant__ CUtensorMap mapB_hi, const __grid_constant__ CUtensorMap mapB_lo, const KParams p) {
  using C = Cfg<CG, SPLIT>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  float* epi_stage = reinterpret_cast<float*>(smem + C::kStages * C::kStageBytes);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + C::kStages * C::kStageBytes + kEpiStageBytes);
  uint64_t* full_bar = bars;                       // [kStages]
  uint64_t* empty_bar = bars + C::kStages;         // [kStages]
  uint64_t* tmem_full = bars + 2 * C::kStages;     // [2]
  uint64_t* tmem_empty = bars + 2 * C::kStages + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * C::kStages + 4);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = CG == 2 ? cluster_ctarank() : 0u;
  const bool leader = rank == 0;
  const int unit = CG == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;      // CTA or CTA pair
  const int n_units = CG == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA_hi)) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB_hi)) : "memory");
    if (SPLIT) {
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapA_lo)) : "memory");
      asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&mapB_lo)) : "memory");
    }
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < C::kStages; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&tmem_full[s], 1);
      mbar_init(&tmem_empty[s], CG * 4);   // one arrival per epilogue warp of every CTA in the group
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc<CG>(tmem_slot, kTmemCols);
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int block_n = p.block_n;
  const int rows_b = block_n / CG;                      // B rows this CTA loads
  const uint32_t stage_tx = (uint32_t)((C::kBytesA + rows_b * 128) * (SPLIT ? 2 : 1) * CG);
  const int kb_per_split = (p.k_blocks_total + p.splits - 1) / p.splits;
  const int n_acc = p.chunked ? 1 : 2;                  // accumulator stages the MMA issuer rotates through

  if (warp == 0 && lane == 0) {
    // ===================== TMA producer =====================
    int stage = 0;
    uint32_t phase = 0;
    for (int it = unit; it < p.n_tiles; it += n_units) {
      const Tile t = p.tiles[it];
      const int kb0 = t.split * kb_per_split;
      const int kb1 = min(p.k_blocks_total, kb0 + kb_per_split);
      const int row_a = t.tm * (kTileRowsA * CG) + (int)rank * kTileRowsA;
      const int row_b = t.tn * block_n + (int)rank * rows_b;
      for (int kb = kb0; kb < kb1; ++kb) {
        mbar_wait(&empty_bar[stage], phase ^ 1);
        uint8_t* s = smem + stage * C::kStageBytes;
        if (leader) mbar_arrive_expect_tx(&full_bar[stage], stage_tx);
        tma_load_2d<CG>(&mapA_hi, &full_bar[stage], s, kb * kBlockK, row_a);
        tma_load_2d<CG>(&mapB_hi, &full_bar[stage], s + C::kBytesA, kb * kBlockK, row_b);
        if (SPLIT) {
          tma_load_2d<CG>(&mapA_lo, &full_bar[stage], s + C::kBytesA + C::kBytesB, kb * kBlockK, row_a);
          tma_load_2d<CG>(&mapB_lo, &full_bar[stage], s + 2 * C::kBytesA + C::kBytesB, kb * kBlockK, row_b);
        }
        if (++stage == C::kStages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1 && lane == 0 && leader) {
    // ===================== MMA issuer (leader CTA only) =====================
    const uint32_t idesc = make_idesc(kTileRowsA * CG, (uint32_t)block_n);
    int stage = 0;
    uint32_t phase = 0;
    int accum = 0;
    uint32_t accum_phase = 0;
    for (int it = unit; it < p.n_tiles; it += n_units) {
      const Tile t = p.tiles[it];
      const int kb0 = t.split * kb_per_split;
      const int kb1 = min(p.k_blocks_total, kb0 + kb_per_split);
      // An empty split-K partition (the last ones when splits does not divide the k-blocks) takes no accumulator stage:
      // no wait, no commit, no phase advance - the epilogue skips it alike and writes its zeros from registers.
      if (kb1 <= kb0) continue;
      // The tensor core accumulates in FP32 with truncation towards zero: every partial sum shrinks by ~1e-7 of its
      // magnitude per MMA (more for coherent same-sign sums than for random-sign ones).  The truncation is symmetric in
      // sign - accumulating alternate chunks with the operand negated (instruction-descriptor bit 13) and subtracting
      // them changed the measured bias by < 15 %, so that is not done.  At most chunk_kb k-blocks are accumulated by the
      // tensor core; the epilogue warps then add the chunk into a running FP32 sum (round-to-nearest) that lives in the
      // other half of tensor memory; the remaining uniform shrink is calibrated out by the caller (pipeline.cu).
      int kb = kb0;
      do {
        const int kend = min(kb1, kb + p.chunk_kb);
        mbar_wait(&tmem_empty[accum], accum_phase ^ 1);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(accum * kMaxBlockN);
        uint32_t first = 1;
        for (; kb < kend; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * C::kStageBytes);
          const uint64_t a_hi = make_smem_desc(sa);
          const uint64_t b_hi = make_smem_desc(sa + C::kBytesA);
          const uint64_t a_lo = make_smem_desc(sa + C::kBytesA + C::kBytesB);
          const uint64_t b_lo = make_smem_desc(sa + 2 * C::kBytesA + C::kBytesB);
#pragma unroll
          for (int k = 0; k < kBlockK / 16; ++k) {
            const uint64_t adv = (uint64_t)(k * 32 >> 4);   // 16 elements = 32 bytes along K inside the swizzle atom
            umma_f16<CG>(tmem_d, a_hi + adv, b_hi + adv, idesc, first ? 0u : 1u);
            first = 0;
            if (SPLIT) {
              umma_f16<CG>(tmem_d, a_hi + adv, b_lo + adv, idesc, 1u);
              umma_f16<CG>(tmem_d, a_lo + adv, b_hi + adv, idesc, 1u);
            }
          }
          umma_commit<CG>(&empty_bar[stage]);     // frees the smem slot in every CTA of the group
          if (++stage == C::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit<CG>(&tmem_full[accum]);
        if (++accum == n_acc) { accum = 0; accum_phase ^= 1; }
      } while (kb < kb1);
    }
  } else if (warp >= kEpiWarp0) {
    // ===================== epilogue =====================
    const int q = warp - kEpiWarp0;                    // TMEM lane quarter
    int accum = 0;
    uint32_t accum_phase = 0;
    EpiBlock e;
    e.stg = epi_stage + q * 32 * kEpiPitch;
    e.lane = lane;
    e.m_rows = p.m_rows;
    e.n_rows = p.n_rows;
    const uint32_t lane_sel = (uint32_t)(q * 32) << 16;
    for (int it = unit; it < p.n_tiles; it += n_units) {
      const Tile t = p.tiles[it];
      const int kb0 = t.split * kb_per_split;
      const int kb1 = min(p.k_blocks_total, kb0 + kb_per_split);
      e.row0 = t.tm * (kTileRowsA * CG) + (int)rank * kTileRowsA + q * 32;
      const int r = e.row0 + lane;                       // global row of this thread
      const int col0 = t.tn * block_n;
      float* Cs = p.C + (long long)t.split * p.split_stride;
      const bool row_ok = r < p.m_rows;
      // columns of this tile the warp has to produce: inside the matrix and (syrk) not strictly above the diagonal
      int n_cols = min(block_n, p.n_rows - col0);
      if (p.syrk) n_cols = min(n_cols, e.row0 + 32 - col0);
      if (e.row0 >= p.m_rows) n_cols = 0;
      // an empty split-K partition: no accumulator stage (as in the issuer), zeros from registers
      const bool have = kb1 > kb0;
      int kb = kb0;
      do {   // one pass per accumulation chunk
        const bool first_chunk = kb == kb0;
        kb = min(kb1, kb + p.chunk_kb);
        const bool last_chunk = kb >= kb1;
        if (have) {
          mbar_wait(&tmem_full[accum], accum_phase);
          tc_fence_after();
        }
        const uint32_t t_chunk = tmem_base + lane_sel + (uint32_t)(accum * kMaxBlockN);
        const uint32_t t_sum = tmem_base + lane_sel + (uint32_t)kMaxBlockN;     // chunked mode only
        if (p.chunked && have) {
          // fold the chunk into the running sum, then hand the chunk accumulator back before any global store
          for (int c0 = 0; c0 < n_cols; c0 += 32) {
            uint32_t v[32];
            tmem_ld_32x32b_x32_nowait(t_chunk + (uint32_t)c0, v);
            if (!first_chunk) {
              uint32_t s[32];
              tmem_ld_32x32b_x32_nowait(t_sum + (uint32_t)c0, s);
              tmem_ld_wait();
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) + __uint_as_float(s[i]));
            } else {
              tmem_ld_wait();
            }
            tmem_st_32x32b_x32(t_sum + (uint32_t)c0, v);
          }
          tmem_st_wait();
        }
        auto release = [&]() {
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (CG == 2) mbar_arrive_cluster(&tmem_empty[accum], 0); else mbar_arrive_local(&tmem_empty[accum]);
          }
        };
        if (p.chunked && have) release();
        if (last_chunk) {
          const uint32_t t_src = p.chunked ? t_sum : t_chunk;
          for (int c0 = 0; c0 < n_cols; c0 += 32) {
            uint32_t v[32];
            if (have) {
              tmem_ld_32x32b_x32_nowait(t_src + (uint32_t)c0, v);
              tmem_ld_wait();
            } else {
#pragma unroll
              for (int i = 0; i < 32; ++i) v[i] = 0u;
            }
            e.gc0 = col0 + c0;
            float x[32];
#pragma unroll
            for (int i = 0; i < 32; ++i) x[i] = __uint_as_float(v[i]) * p.alpha;
            if (p.epi == (int)Epilogue::ColAbsMax) {
#pragma unroll
              for (int i = 0; i < 32; ++i) {
                float a = row_ok ? fabsf(x[i]) : 0.f;
#pragma unroll
                for (int o = 16; o; o >>= 1) a = fmaxf(a, __shfl_xor_sync(0xffffffffu, a, o));
                if (lane == 0 && e.gc0 + i < p.n_rows) atomicMax(reinterpret_cast<int*>(Cs) + e.gc0 + i, __float_as_int(a));
              }
            } else if (p.syrk) {
              store_rowmajor(e, x, Cs, p.ldc, /*lower_only=*/true);
              store_colmajor(e, x, Cs, p.ldc, /*strict_lower_src=*/true);      // mirror, from the same value
            } else if (p.epi == (int)Epilogue::Store) {
              store_rowmajor(e, x, Cs, p.ldc, false);
            } else {  // StoreTransposed: C[n * ldc + m]
              store_colmajor(e, x, Cs, p.ldc, false);
            }
          }
        }
        if (have) {
          if (!p.chunked) release();
          if (++accum == n_acc) { accum = 0; accum_phase ^= 1; }
        }
      } while (kb < kb1);
    }
  }

  __syncwarp();
  tc_fence_before();
  if (CG == 2) cluster_sync_all(); else __syncthreads();
  if (warp == 2) tmem_dealloc<CG>(tmem_base, kTmemCols);
}

// ---- host side ------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

PFN_encodeTiled get_encode() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    SCL_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
    SCL_REQUIRE(p != nullptr && q == cudaDriverEntryPointSuccess, "cuTensorMapEncodeTiled unavailable");
    fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

CUtensorMap make_map(const __half* base, int rows, int64_t K, int64_t ld, int box_rows) {
  SCL_REQUIRE(ld % 8 == 0, "operand leading dimension must be a multiple of 8 elements (16 bytes)");
  SCL_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0, "operand base must be 16-byte aligned");
  CUtensorMap m;
  cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(__half)};
  cuuint32_t box[2] = {(cuuint32_t)kBlockK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = get_encode()(&m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) throw Error(-2, "cuTensorMapEncodeTiled failed: " + std::to_string((int)r));
  return m;
}

// Tile order: 8x8 super-tiles so the ~74-148 tiles in flight share operand row blocks in L2.
std::vector<Tile> build_tiles(int tiles_m, int tiles_n, int splits, bool syrk, int tile_m, int tile_n) {
  std::vector<Tile> out;
  constexpr int S = 8;
  for (int sm = 0; sm < tiles_m; sm += S)
    for (int sn = 0; sn < tiles_n; sn += S)
      for (int tm = sm; tm < std::min(tiles_m, sm + S); ++tm)
        for (int tn = sn; tn < std::min(tiles_n, sn + S); ++tn) {
          int diag = 0;
          if (syrk) {
            long long row_hi = (long long)(tm + 1) * tile_m - 1, col_lo = (long long)tn * tile_n;
            if (col_lo > row_hi) continue;   // entirely above the diagonal
            diag = 1;
          }
          for (int s = 0; s < splits; ++s) out.push_back(Tile{tm, tn, s, diag});
        }
  return out;
}

template <int CG, bool SPLIT>
void launch(const GemmArgs& a, cudaStream_t st, GemmLaunch* info) {
  using C = Cfg<CG, SPLIT>;
  const int tile_m = kTileRowsA * CG;
  int block_n = kMaxBlockN;
  if (!a.syrk) {
    block_n = std::min(kMaxBlockN, ((a.B.rows + 31) / 32) * 32);
    if (block_n < 32) block_n = 32;
  }
  const int tiles_m = (a.A.rows + tile_m - 1) / tile_m;
  const int tiles_n = (a.B.rows + block_n - 1) / block_n;
  const int kblocks = (int)((a.A.K + kBlockK - 1) / kBlockK);
  int splits = std::max(1, std::min(a.splits, kblocks));
  std::vector<Tile> tiles = build_tiles(tiles_m, tiles_n, splits, a.syrk, tile_m, block_n);
  SCL_REQUIRE(!tiles.empty(), "empty GEMM");
  Tmp<Tile> d_tiles(tiles.size(), st);
  SCL_CUDA(cudaMemcpyAsync(d_tiles.p, tiles.data(), tiles.size() * sizeof(Tile), cudaMemcpyHostToDevice, st));

  CUtensorMap mA_hi = make_map(a.A.hi, a.A.rows, a.A.K, a.A.ld, kTileRowsA);
  CUtensorMap mB_hi = make_map(a.B.hi, a.B.rows, a.B.K, a.B.ld, block_n / CG);
  CUtensorMap mA_lo = mA_hi, mB_lo = mB_hi;
  if (SPLIT) {
    mA_lo = make_map(a.A.lo, a.A.rows, a.A.K, a.A.ld, kTileRowsA);
    mB_lo = make_map(a.B.lo, a.B.rows, a.B.K, a.B.ld, block_n / CG);
  }
  KParams p;
  p.tiles = d_tiles.p;
  p.n_tiles = (int)tiles.size();
  p.m_rows = a.A.rows;
  p.n_rows = a.B.rows;
  p.k_blocks_total = kblocks;
  p.splits = splits;
  p.block_n = block_n;
  // Chunks of equal length, at most `want` k-blocks each (default 64 = 256 MMAs, 21 in split mode = 252 MMAs:
  // a truncation bias below ~2e-5 relative on a coherent sum).  ColAbsMax operands are unit vectors with
  // random-sign products: one chunk.
  {
    const int kbs = (kblocks + splits - 1) / splits;
    const int want = a.epi == Epilogue::ColAbsMax ? (1 << 30) : (a.chunk_kb > 0 ? a.chunk_kb : (SPLIT ? 21 : 64));
    const int n_chunks = std::max(1, (kbs + want - 1) / want);
    p.chunk_kb = std::max(1, (kbs + n_chunks - 1) / n_chunks);
    p.chunked = n_chunks > 1 ? 1 : 0;
  }
  p.syrk = a.syrk ? 1 : 0;
  p.epi = (int)a.epi;
  p.alpha = a.alpha;
  p.C = a.C;
  p.ldc = a.ldc;
  p.split_stride = a.split_stride;

  auto kern = k_gemm_umma<CG, SPLIT>;
  SCL_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, C::kSmemBytes));
  const int sms = sm_count();
  int units = CG == 2 ? sms / 2 : sms;
  units = std::min(units, (int)tiles.size());
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(units * CG);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = C::kSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CG;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  SCL_CUDA(cudaLaunchKernelEx(&cfg, kern, mA_hi, mA_lo, mB_hi, mB_lo, p));
  count_launches(1);
  if (info) {
    info->block_n = block_n;
    info->n_tiles = p.n_tiles;
    info->units = units;
    info->splits = splits;
    info->chunk_kb = p.chunk_kb;
    info->chunked = p.chunked;
    info->max_per_unit = (p.n_tiles + units - 1) / units;
  }
}

// ---- small elementwise helpers ----------------------------------------------------------
__global__ void k_split_f32(const float* __restrict__ in, size_t n, __half* __restrict__ hi, __half* __restrict__ lo) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    float x = in[i];
    __half h = __float2half_rn(x);
    hi[i] = h;
    if (lo) lo[i] = __float2half_rn(x - __half2float(h));
  }
}

__global__ void k_strided_split_f32(const float* __restrict__ in, int rows, long long cols, long long ld_in,
                                    long long ld_out, __half* __restrict__ hi, __half* __restrict__ lo, float pre_scale) {
  for (int r = blockIdx.y; r < rows; r += gridDim.y) {
    for (long long c = blockIdx.x * (long long)blockDim.x + threadIdx.x; c < ld_out; c += (long long)gridDim.x * blockDim.x) {
      float x = c < cols ? in[(long long)r * ld_in + c] * pre_scale : 0.f;
      __half h = __float2half_rn(x);
      hi[(long long)r * ld_out + c] = h;
      if (lo) lo[(long long)r * ld_out + c] = __float2half_rn(x - __half2float(h));
    }
  }
}

__global__ void k_fill_random_f16(__half* __restrict__ out, size_t n, uint32_t seed, float scale) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  const size_t stride = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += stride) {
    uint64_t h = (i + 1) * 0x9E3779B97F4A7C15ull ^ ((uint64_t)seed << 32);
    h ^= h >> 29; h *= 0xBF58476D1CE4E5B9ull; h ^= h >> 32;
    // sum of four 16-bit uniforms, centred: variance 4/12 -> scaled to unit variance
    const float u = (float)(h & 0xffff) + (float)((h >> 16) & 0xffff) + (float)((h >> 32) & 0xffff) + (float)(h >> 48);
    out[i] = __float2half_rn((u * (1.0f / 65536.f) - 2.0f) * 1.7320508f * scale);
  }
}

__global__ void k_reduce_splits(const float* __restrict__ part, int splits, long long stride, size_t n, float scale,
                                float* __restrict__ out) {
  size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  size_t step = (size_t)gridDim.x * blockDim.x;
  for (; i < n; i += step) {
    float s = 0.f;
    for (int k = 0; k < splits; ++k) s += part[(size_t)k * stride + i];
    out[i] = s * scale;
  }
}

}  // namespace

int sm_count() {
  static int n = 0;
  if (!n) {
    int dev = 0;
    SCL_CUDA(cudaGetDevice(&dev));
    SCL_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
  }
  return n;
}

void gemm_umma(const GemmArgs& a, cudaStream_t st, GemmLaunch* info) {
  SCL_REQUIRE(a.A.hi && a.B.hi && a.C, "null GEMM operand");
  SCL_REQUIRE(a.A.K == a.B.K, "contraction lengths differ");
  const bool split = a.A.lo != nullptr && a.B.lo != nullptr;
  if (a.cta_group == 1) {
    if (split) launch<1, true>(a, st, info); else launch<1, false>(a, st, info);
  } else {
    if (split) launch<2, true>(a, st, info); else launch<2, false>(a, st, info);
  }
}

void split_f32_to_f16(const float* in, size_t n, __half* hi, __half* lo, cudaStream_t st) {
  if (!n) return;
  count_launches(1);
  int grid = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
  k_split_f32<<<grid, 256, 0, st>>>(in, n, hi, lo);
  SCL_CUDA(cudaGetLastError());
}

void strided_split_f32_to_f16(const float* in, int rows, int64_t cols, int64_t ld_in, int64_t ld_out, __half* hi,
                              __half* lo, cudaStream_t st, float pre_scale) {
  if (!rows) return;
  count_launches(1);
  dim3 grid((unsigned)std::min<int64_t>((ld_out + 255) / 256, 64), (unsigned)std::min(rows, 65535));
  k_strided_split_f32<<<grid, 256, 0, st>>>(in, rows, cols, ld_in, ld_out, hi, lo, pre_scale);
  SCL_CUDA(cudaGetLastError());
}

void fill_random_f16(__half* out, size_t n, uint32_t seed, float scale, cudaStream_t st) {
  if (!n) return;
  count_launches(1);
  k_fill_random_f16<<<148 * 8, 256, 0, st>>>(out, n, seed, scale);
  SCL_CUDA(cudaGetLastError());
}

void reduce_splits(const float* part, int splits, int64_t stride, size_t n, float scale, float* out, cudaStream_t st) {
  if (!n) return;
  count_launches(1);
  int grid = (int)std::min<size_t>((n + 255) / 256, 148 * 16);
  k_reduce_splits<<<grid, 256, 0, st>>>(part, splits, stride, n, scale, out);
  SCL_CUDA(cudaGetLastError());
}

}  // namespace scl
