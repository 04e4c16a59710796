// Back-transformation of the two-stage eigensolver: Z <- Q1 Q2 Z for the eigenvectors Z of the tridiagonal matrix.
//
// Q2 (stage-2 reflectors, one per sweep and chase level, kBand long, consecutive sweeps shifted by one row): the reflectors
// of kBand consecutive sweeps at one level form a parallelogram V (2 kBand - 1 rows x kBand columns) and are applied as
// one block I - V T V'.  Generation order is sweep-major; reflectors (s, k) and (s', k') with s < s', k < k' act on disjoint
// rows, so inside a group of sweeps the product may be taken level by level, and the eigenvectors see: groups descending,
// levels ascending inside a group (oracle/two_stage_ref.py: apply_q2 == apply_q2_plain).  Every eigenvector is independent:
// a warp owns 16 vectors, keeps their 128-row window in registers and walks all blocks (k_q2_apply_h, split binary16 on
// mma.sync).
// Q1 (stage-1 panels, V T stored by stage 1 in the upper triangle of A): for 64 vectors or more, eight panels at a time as one
// block reflector on the tcgen05 GEMM of gemm_umma.cu (apply_q1_umma); for fewer, Z[r0:] -= (V T) (V' Z[r0:]) panel by panel,
// last panel first, on the split-binary16 tile engine of sgemm_tile.cuh.
#include <cuda_fp16.h>
#include <algorithm>
#include "common.cuh"
#include "sgemm_tile.cuh"
#include "tmp.cuh"
#include "twostage.h"

namespace scl {

namespace {

constexpr int B = kBand;

static_assert(B == 64, "the register-stationary kernel is written for a half bandwidth of 64");

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "Q2_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra Q2_DONE;\n\t"
      "bra Q2_WAIT;\n\t"
      "Q2_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
               "l"(src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

__device__ __forceinline__ void ld_rows(float (&r)[4], const float* za, const float* zb, bool oka, bool okb, int row, int n) {
  float2 u = make_float2(0.f, 0.f), v = u;
  if (row + 1 < n) {
    if (oka) u = *reinterpret_cast<const float2*>(za + row);
    if (okb) v = *reinterpret_cast<const float2*>(zb + row);
  } else if (row < n) {
    if (oka) u.x = za[row];
    if (okb) v.x = zb[row];
  }
  r[0] = u.x; r[1] = u.y; r[2] = v.x; r[3] = v.y;
}
__device__ __forceinline__ void st_rows(const float (&r)[4], float* za, float* zb, bool oka, bool okb, int row, int n) {
  if (row + 1 < n) {
    if (oka) *reinterpret_cast<float2*>(za + row) = make_float2(r[0], r[1]);
    if (okb) *reinterpret_cast<float2*>(zb + row) = make_float2(r[2], r[3]);
  } else if (row < n) {
    if (oka) za[row] = r[0];
    if (okb) zb[row] = r[2];
  }
}

// ---------------------------------------------------------------------------------------------------------------- Q2
// The window of a slab never leaves the register file.  A warp owns 16 eigenvectors and keeps their 128-row window as the
// accumulator fragments of sixteen m16n8 tiles (vectors = the M dimension, window rows = N).  A 16-row step of the window is
// two accumulator tiles, and their registers (tile i | tile i + 1), converted to binary16, are the A fragment of the next
// product as they stand (natural k order).  So  X' = Z' V  ->  X2' = X' T'  ->  Z' -= X2' V'  chain through registers: no
// shared-memory window, no CTA-wide barrier, and the only operands that come from shared memory are the reflector block and
// its T factor.  Those are the same for every warp and every vector, so a pre-pass (k_q2_images_h) writes them once, already
// split and already in the shared-memory layout, and one elected thread streams one 40 KB image per block through a
// four-stage cp.async.bulk ring (mbarrier full / empty pairs); warps never wait for each other except through that ring.
// Split binary16: x = hi + lo / 2048, hi = half(x), lo = half((x - hi) 2048), 22 significant bits; the factor keeps lo out of
// the subnormal range, and values below 6e-5 (eigenvector entries never need more) keep an absolute error of 1.5e-11.
// Everything that is multiplied is O(1) or smaller: eigenvector entries, reflectors (|v| <= 1), T (|tau| <= 2), X, X2.
// Measured on B200 (scripts/mma_rate.cu), the warp-level tensor path issues one mma.sync per 8 cycles and sub-partition for
// m16n8k8 TF32 and for m16n8k16 FP16 alike, so a binary16 step contracts twice as many terms in the same time as the
// three-term TF32 split of the same 22 bits (254 / 440 ms against 380 / 558 ms for the smallest half / all vectors at
// n = 20 000).
// B fragments come from the image by ldmatrix: plain for the first product and for T (pairs along the window rows of one
// reflector), transposed for the last product (pairs along the reflectors of one window row); one ldmatrix.x4 fetches the hi
// and lo fragments of a step.  Image of a block: binary16 planes P hi, P lo (64 rows of 88: 8 zeros, the 72 entries of the
// nine steps, 8 zeros - the zeros serve the half steps that stick out of the band), T hi, T lo (64 rows of 72); row pitches of
// 176 and 144 bytes spread the eight 16-byte rows of an ldmatrix over all banks.
// Accumulation: the tensor core adds with truncation, so the leading term a_hi b_hi of every step starts from a zero
// accumulator and is added to the running sum with a rounded FP32 add; the two cross terms, 2^-11 of it, are chained in
// tensor-core accumulators of their own (their truncation is 2^-35 of the result), which also keeps the dependent chains short.
constexpr int kPRowH = 88, kTRowH = 72;
constexpr int kPPlaneH = B * kPRowH, kTPlaneH = B * kTRowH;        // halves per plane
constexpr int kBlkHalves = 2 * kPPlaneH + 2 * kTPlaneH;            // 20 480 halves = 40 960 bytes
constexpr int kBlkBytesH = kBlkHalves * 2;
constexpr int kStagesH = 4;
constexpr float kLoScale = 2048.f, kLoInv = 1.f / 2048.f;

// Pre-pass: T factor of block (G, k) (forward columnwise larft on the Gram matrix of its reflectors), then the block's image at
// its place in processing order (groups descending, levels ascending: block index (q - G)(q - G + 1) / 2 + k with q = the last
// group).
__global__ void __launch_bounds__(256) k_q2_images_h(const float* __restrict__ V2, long long ldv2, const float* __restrict__ tau2,
                                                     long long ldt2, int n, int q, __half* __restrict__ Img) {
  const int k = (int)blockIdx.x, G = (int)blockIdx.y, s0 = G * B;
  if (s0 + 1 + B * k > n - 2) return;
  __shared__ float Vc[B][B + 1], T[B][B + 1];
  __shared__ float tau[B];
  const int tid = (int)threadIdx.x;
  for (int e = tid; e < B * B; e += 256) {
    const int j = e / B, i = e % B, s = s0 + j;
    Vc[j][i] = s < n - 2 ? V2[(size_t)s * ldv2 + (size_t)k * B + i] : 0.f;
    if (j <= i) T[j][i] = 0.f;
  }
  if (tid < B) tau[tid] = s0 + tid < n - 2 ? tau2[(size_t)(s0 + tid) * ldt2 + k] : 0.f;
  __syncthreads();
  for (int e = tid; e < B * B; e += 256) {
    const int a = e / B, b = e % B;
    if (a < b) {
      const int sh = b - a;
      float s = 0.f;
      for (int i = 0; i + sh < B; ++i) s = fmaf(Vc[a][i + sh], Vc[b][i], s);
      T[b][a] = s;
    }
  }
  __syncthreads();
  for (int j = 0; j < B; ++j) {
    if (tid < j) {
      float s = 0.f;
      for (int qq = tid; qq < j; ++qq) s = fmaf(T[tid][qq], T[j][qq], s);
      T[tid][j] = -tau[j] * s;
    } else if (tid == j) {
      T[j][j] = tau[j];
    }
    __syncthreads();
  }
  __half* img = Img + ((size_t)(q - G) * (q - G + 1) / 2 + k) * kBlkHalves;
  for (int e = tid; e < B * kPRowH; e += 256) {
    const int c = e / kPRowH, up = e % kPRowH;
    const int i = up - 8 - (c & 7) - 1;   // entry up holds window row 8 (c / 8) + up - 8 = entry i of reflector c
    const float x = (i >= 0 && i < B) ? Vc[c][i] : 0.f;
    const __half hi = __float2half_rn(x);
    img[e] = hi;
    img[kPPlaneH + e] = __float2half_rn((x - __half2float(hi)) * kLoScale);
  }
  for (int e = tid; e < B * kTRowH; e += 256) {
    const int c = e / kTRowH, u = e % kTRowH;
    const float x = (u < B && c <= u) ? T[c][u] : 0.f;
    const __half hi = __float2half_rn(x);
    img[2 * kPPlaneH + e] = hi;
    img[2 * kPPlaneH + kTPlaneH + e] = __float2half_rn((x - __half2float(hi)) * kLoScale);
  }
}

struct Q2HArgs {
  const __half* Img;
  float* Z;
  long long ldz;
  int n, mvec, q, tiles, base, extra;
};

__device__ __forceinline__ void mma_f16_zero(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%10,%10,%10,%10};"
      : "=f"(d[0]), "=f"(d[1]), "=f"(d[2]), "=f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]), "f"(0.f));
}
__device__ __forceinline__ void mma_f16(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
template <bool kTrans>
__device__ __forceinline__ void ldsm4(uint32_t (&bh)[2], uint32_t (&bl)[2], uint32_t addr) {
  if (kTrans)
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(bh[0]), "=r"(bh[1]), "=r"(bl[0]), "=r"(bl[1]) : "r"(addr));
  else
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(bh[0]), "=r"(bh[1]), "=r"(bl[0]), "=r"(bl[1]) : "r"(addr));
}
// one accumulator tile (rows g | g + 8, columns 2t, 2t + 1) as the two half-fragments (hi, lo) of a 16-deep A operand
__device__ __forceinline__ void pack_hl(const float (&r)[4], uint32_t (&h)[2], uint32_t (&l)[2]) {
  const __half2 h0 = __floats2half2_rn(r[0], r[1]), h1 = __floats2half2_rn(r[2], r[3]);
  const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
  const __half2 l0 = __floats2half2_rn((r[0] - f0.x) * kLoScale, (r[1] - f0.y) * kLoScale);
  const __half2 l1 = __floats2half2_rn((r[2] - f1.x) * kLoScale, (r[3] - f1.y) * kLoScale);
  h[0] = *reinterpret_cast<const uint32_t*>(&h0);
  h[1] = *reinterpret_cast<const uint32_t*>(&h1);
  l[0] = *reinterpret_cast<const uint32_t*>(&l0);
  l[1] = *reinterpret_cast<const uint32_t*>(&l1);
}
// acc += sign * a_hi b_hi from a zero accumulator; cross (+)= a_lo b_hi + a_hi b_lo (both carry the factor 2048)
template <bool kFirst>
__device__ __forceinline__ void mma_step_h(float (&acc)[4], float (&cross)[4], const uint32_t (&ah)[4], const uint32_t (&al)[4],
                                           const uint32_t (&bh)[2], const uint32_t (&bl)[2], float sign) {
  float d[4];
  mma_f16_zero(d, ah, bh);
  if (kFirst) mma_f16_zero(cross, al, bh);
  else mma_f16(cross, al, bh);
  mma_f16(cross, ah, bl);
  acc[0] = fmaf(sign, d[0], acc[0]); acc[1] = fmaf(sign, d[1], acc[1]); acc[2] = fmaf(sign, d[2], acc[2]); acc[3] = fmaf(sign, d[3], acc[3]);
}

template <int MAXW>
__global__ void __launch_bounds__(MAXW * 32, 1) k_q2_apply_h(Q2HArgs a) {
  extern __shared__ __align__(16) float sm[];
  __half* smh = reinterpret_cast<__half*>(sm);
  uint64_t* full = reinterpret_cast<uint64_t*>(smh + kStagesH * kBlkHalves);
  uint64_t* empty = full + kStagesH;
  const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5, g = lane >> 2, t = lane & 3;
  const int cta = (int)blockIdx.x;
  const int ntile = a.base + (cta < a.extra ? 1 : 0);
  const int tile0 = cta * a.base + min(cta, a.extra);
  if (tid == 0) {
    for (int s = 0; s < kStagesH; ++s) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], (uint32_t)ntile);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  if (warp >= ntile) return;
  const int q = a.q, n = a.n;
  const int nblk = (q + 1) * (q + 2) / 2;
  if (tid == 0) {
    for (int b = 0; b < kStagesH - 1 && b < nblk; ++b) {
      mbar_arrive_expect_tx(&full[b], kBlkBytesH);
      bulk_g2s(smh + b * kBlkHalves, a.Img + (size_t)b * kBlkHalves, kBlkBytesH, &full[b]);
    }
  }
  const int va = (tile0 + warp) * 16 + g, vb = va + 8;
  const bool oka = va < a.mvec, okb = vb < a.mvec;
  float* za = a.Z + (size_t)(oka ? va : 0) * a.ldz;
  float* zb = a.Z + (size_t)(okb ? vb : 0) * a.ldz;
  // ldmatrix row addresses of this lane (bytes, relative to a stage): matrix m = lane / 8 (0, 1: hi plane, 2, 3: lo plane; odd:
  // the second half of the 16-deep step), row r = lane % 8
  const int lm = lane >> 3, lr = lane & 7;
  const uint32_t offP = 2u * (uint32_t)((lm >> 1) * kPPlaneH + lr * kPRowH + (lm & 1) * 8);                        // first product
  const uint32_t offT = 2u * (uint32_t)(2 * kPPlaneH + (lm >> 1) * kTPlaneH + lr * kTRowH + (lm & 1) * 8);          // T product
  const uint32_t offU = 2u * (uint32_t)((lm >> 1) * kPPlaneH + ((lm & 1) * 8 + lr) * kPRowH - (lm & 1) * 8);        // last product
  const uint32_t sm0 = smem_u32(smh);
  float z[16][4];
  int b = 0;
  for (int G = q; G >= 0; --G) {
    const int nl = q - G + 1;
    int R0 = B * G;
#pragma unroll
    for (int i = 0; i < 16; ++i) ld_rows(z[i], za, zb, oka, okb, R0 + 8 * i + 2 * t, n);
    for (int k = 0; k < nl; ++k, ++b, R0 += B) {
      const int s = b % kStagesH;
      if (tid == 0 && b + kStagesH - 1 < nblk) {   // refill the stage block b - 1 used, once every warp has released it
        const int s2 = (b + kStagesH - 1) % kStagesH;
        if (b >= 1) mbar_wait(&empty[s2], (uint32_t)(((b - 1) / kStagesH) & 1));
        mbar_arrive_expect_tx(&full[s2], kBlkBytesH);
        bulk_g2s(smh + s2 * kBlkHalves, a.Img + (size_t)(b + kStagesH - 1) * kBlkHalves, kBlkBytesH, &full[s2]);
      }
      __syncwarp();
      const bool more = k + 1 < nl;
      if (more) {
        const int v = (tile0 + warp) * 16 + (lane >> 1);
        const int r = R0 + 128 + ((lane & 1) ? 63 : 0);
        if (v < a.mvec && r < n) {
          const float* pz = a.Z + (size_t)v * a.ldz + r;
          asm volatile("prefetch.global.L2 [%0];" ::"l"(pz));
          if (!(lane & 1) && r + 32 < n) asm volatile("prefetch.global.L2 [%0];" ::"l"(pz + 32));
        }
      }
      mbar_wait(&full[s], (uint32_t)((b / kStagesH) & 1));
      const uint32_t st0 = sm0 + (uint32_t)s * kBlkBytesH;
      // ---- X'[vec][c] = sum_w Z'[vec][w] V[w][c]: the 16 rows of tiles (i, i + 1) meet the reflector tiles j = i - 2 s, s = 0 .. 4
      float x[8][4], xc[8][4];
#pragma unroll
      for (int j = 0; j < 8; ++j) x[j][0] = x[j][1] = x[j][2] = x[j][3] = 0.f;
      {
        uint32_t ph[2], pl[2];
        pack_hl(z[0], ph, pl);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          uint32_t qh[2] = {0u, 0u}, ql[2] = {0u, 0u};
          if (i + 1 < 16) pack_hl(z[i + 1], qh, ql);
          const uint32_t ah[4] = {ph[0], ph[1], qh[0], qh[1]}, al[4] = {pl[0], pl[1], ql[0], ql[1]};
#pragma unroll
          for (int sq = 0; sq < 5; ++sq) {
            const int j = i - 2 * sq;
            if (j >= 0 && j <= 7) {
              uint32_t bh[2], bl[2];
              ldsm4<false>(bh, bl, st0 + offP + 2u * (uint32_t)(8 * j * kPRowH + 8 + 16 * sq));
              if (sq == 0) mma_step_h<true>(x[j], xc[j], ah, al, bh, bl, 1.f);
              else mma_step_h<false>(x[j], xc[j], ah, al, bh, bl, 1.f);
            }
          }
          ph[0] = qh[0]; ph[1] = qh[1]; pl[0] = ql[0]; pl[1] = ql[1];
        }
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        x[j][0] = fmaf(xc[j][0], kLoInv, x[j][0]); x[j][1] = fmaf(xc[j][1], kLoInv, x[j][1]);
        x[j][2] = fmaf(xc[j][2], kLoInv, x[j][2]); x[j][3] = fmaf(xc[j][3], kLoInv, x[j][3]);
      }
      // ---- X2'[vec][c] = sum_{c' >= c} X'[vec][c'] T[c][c']: 16 columns c' per step
      float x2[8][4];
#pragma unroll
      for (int j = 0; j < 8; ++j) x2[j][0] = x2[j][1] = x2[j][2] = x2[j][3] = 0.f;
#pragma unroll
      for (int kb = 0; kb < 4; ++kb) {
        uint32_t h0[2], l0[2], h1[2], l1[2];
        pack_hl(x[2 * kb], h0, l0);
        pack_hl(x[2 * kb + 1], h1, l1);
        const uint32_t ah[4] = {h0[0], h0[1], h1[0], h1[1]}, al[4] = {l0[0], l0[1], l1[0], l1[1]};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (j <= 2 * kb + 1) {
            uint32_t bh[2], bl[2];
            ldsm4<false>(bh, bl, st0 + offT + 2u * (uint32_t)(8 * j * kTRowH + 16 * kb));
            float dm[4], dc[4];
            mma_f16_zero(dm, ah, bh);
            mma_f16_zero(dc, al, bh);
            mma_f16(dc, ah, bl);
            x2[j][0] += fmaf(dc[0], kLoInv, dm[0]); x2[j][1] += fmaf(dc[1], kLoInv, dm[1]);
            x2[j][2] += fmaf(dc[2], kLoInv, dm[2]); x2[j][3] += fmaf(dc[3], kLoInv, dm[3]);
          }
        }
      }
      // ---- Z'[vec][w] -= sum_c X2'[vec][c] V[w][c]: row tile i meets the 16-reflector steps kb with 0 <= i - 2 kb <= 9
      {
        uint32_t x2h[8][2], x2l[8][2];
#pragma unroll
        for (int j = 0; j < 8; ++j) pack_hl(x2[j], x2h[j], x2l[j]);
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          float zc[4];
          bool first = true;
#pragma unroll
          for (int kb = 0; kb < 4; ++kb) {
            const int d = i - 2 * kb;
            if (d >= 0 && d <= 9) {
              const uint32_t ah[4] = {x2h[2 * kb][0], x2h[2 * kb][1], x2h[2 * kb + 1][0], x2h[2 * kb + 1][1]};
              const uint32_t al[4] = {x2l[2 * kb][0], x2l[2 * kb][1], x2l[2 * kb + 1][0], x2l[2 * kb + 1][1]};
              uint32_t bh[2], bl[2];
              ldsm4<true>(bh, bl, st0 + offU + 2u * (uint32_t)(16 * kb * kPRowH + 8 + 8 * d));
              if (first) mma_step_h<true>(z[i], zc, ah, al, bh, bl, -1.f);
              else mma_step_h<false>(z[i], zc, ah, al, bh, bl, -1.f);
              first = false;
            }
          }
          z[i][0] = fmaf(zc[0], -kLoInv, z[i][0]); z[i][1] = fmaf(zc[1], -kLoInv, z[i][1]);
          z[i][2] = fmaf(zc[2], -kLoInv, z[i][2]); z[i][3] = fmaf(zc[3], -kLoInv, z[i][3]);
        }
      }
      __syncwarp();
      if (lane == 0) mbar_arrive(&empty[s]);
#pragma unroll
      for (int i = 0; i < 8; ++i) st_rows(z[i], za, zb, oka, okb, R0 + 8 * i + 2 * t, n);
      if (more) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
#pragma unroll
          for (int e = 0; e < 4; ++e) z[i][e] = z[i + 8][e];
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) ld_rows(z[i + 8], za, zb, oka, okb, R0 + 128 + 8 * i + 2 * t, n);
      } else {
#pragma unroll
        for (int i = 8; i < 16; ++i) st_rows(z[i], za, zb, oka, okb, R0 + 8 * i + 2 * t, n);
      }
    }
  }
}

// unit length again: the tensor core adds with truncation, so every block update comes back a few 1e-8 short, which shortens a
// vector by ~1e-7 n / 64 over the whole of Q2 (measured 4e-6 at n = 2531) while turning it by far less
__global__ void __launch_bounds__(256) k_unit_vectors(float* __restrict__ Z, long long ldz, int n, int mvec) {
  const int v = (int)blockIdx.x * 8 + ((int)threadIdx.x >> 5), lane = (int)threadIdx.x & 31;
  if (v >= mvec) return;
  float* z = Z + (size_t)v * ldz;
  double s = 0.0;
  for (int i = lane; i < n; i += 32) s += (double)z[i] * (double)z[i];
#pragma unroll
  for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if (!(s > 0.0)) return;
  const float f = (float)(1.0 / sqrt(s));
  for (int i = lane; i < n; i += 32) z[i] *= f;
}

// ---------------------------------------------------------------------------------------------------------------- Q1
// Panel by panel on the split-binary16 tile engine of sgemm_tile.cuh: eigenvector slabs, reflector panels and their products
// are O(1).  Xpart[s][c][vec] = sum over rows i of chunk s of V[c][i] * Z[vec][r0 + i]
__global__ void __launch_bounds__(256, 2) k_q1_x_tc(const float* __restrict__ Vp, long long lda, int m, const float* __restrict__ Zr,
                                                    long long ldz, int mvec, float* __restrict__ Xpart, long long ldx, int chunk) {
  __shared__ __align__(16) unsigned char smem[tile::SmemE<2, 64>::bytes];
  const int vec0 = (int)blockIdx.x * tile::TM;
  const int ka = (int)blockIdx.y * chunk, kl = min(m, ka + chunk) - ka;
  tile::AccT<64> acc;
  acc.clear();
  tile::mac_e<2, 64, 1, 1>(acc, tile::opnd(Zr + (long long)vec0 * ldz + ka, ldz, 1, mvec - vec0, kl), tile::opnd(Vp + ka, lda, 1, B, kl), kl, smem);
  float* out = Xpart + (size_t)blockIdx.y * B * ldx;
#pragma unroll
  for (int nt = 0; nt < tile::AccT<64>::NTL; ++nt)
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int v = vec0 + tile::AccT<64>::row(mt, e), c = tile::AccT<64>::col(nt, e);
        if (v < mvec) out[(long long)c * ldx + v] = acc.v[mt][nt][e];
      }
}

__global__ void k_sum_parts32(const float* __restrict__ part, int nparts, size_t stride, size_t n, float* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int p = 0; p < nparts; ++p) s += part[(size_t)p * stride + i];
  out[i] = s;
}

// Z[vec][r0 + i] -= sum_c X[c][vec] (V T)[i][c] (VTt: the panel's V T as sy2sb left it, element (i, c) at VTt[c + i * lda]):
// vectors on the rows of the tile, matrix rows on its columns, so that a thread's two adjacent outputs are adjacent in memory
__global__ void __launch_bounds__(256, 2) k_q1_z_tc(const float* __restrict__ VTt, long long lda, int m, const float* __restrict__ Xp,
                                                    long long ldx, int mvec, float* Zr, long long ldz) {
  __shared__ __align__(16) unsigned char smem[tile::SmemE<2, 128>::bytes];
  const int i0 = (int)blockIdx.x * tile::TM, vec0 = (int)blockIdx.y * tile::TM;
  tile::AccT<128> acc;
  acc.clear();
  tile::mac_e<2, 128, 0, 1>(acc, tile::opnd(Xp + vec0, ldx, 0, mvec - vec0, B), tile::opnd(VTt + (long long)i0 * lda, lda, 1, m - i0, B), B, smem);
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int v = vec0 + tile::AccT<128>::row(mt, 2 * h);
      if (v >= mvec) continue;
      float* zc = Zr + (long long)v * ldz;
#pragma unroll
      for (int nt = 0; nt < tile::AccT<128>::NTL; ++nt) {
        const int i = i0 + tile::AccT<128>::col(nt, 0);
        if (i + 1 < m) {
          float2 z = *reinterpret_cast<float2*>(zc + i);
          z.x -= acc.v[mt][nt][2 * h];
          z.y -= acc.v[mt][nt][2 * h + 1];
          *reinterpret_cast<float2*>(zc + i) = z;
        } else if (i < m) {
          zc[i] -= acc.v[mt][nt][2 * h];
        }
      }
    }
}

// ---------------------------------------------------------------------------------------- Q1 on the tcgen05 GEMM
// Eight panels at a time: H_a H_a+1 ... H_a+7 Z = Z - (VT)_blk X with X_j = V_j' Z - sum_{l > j} (V_j' V_l T_l) X_l, j descending.
// Y = V_blk' Z (512 x vectors, contraction over the rows) and Z -= (VT)_blk X (contraction over the 512 reflectors) are two
// large products on gemm_umma.cu in split binary16 (hi hi + hi lo + lo hi, FP32 accumulation in TMEM); the couplings come from
// the Gram matrix V_blk' V_blk (one more product) and the recursion runs per vector in the 512-dimensional space.  Operands are
// converted once per block; powers of two keep their low-order parts in binary16's normal range.
constexpr int kQ1Panels = 8;
constexpr float kScV = 1024.f, kScVT = 64.f, kScZ = 1024.f, kScX = 256.f;
// k-blocks per accumulation chunk of the two large products (profiles/r2_two_stage_stage_times_20000.txt compares 2, 4 and 8)
constexpr int kQ1ChunkKb = 4;

// V of the block's panels as (hi, lo) binary16, reflector-major [ncols][ldk] over the rows r0 .. n; zero above a panel's first row
__global__ void __launch_bounds__(256) k_q1_conv_v(const float* __restrict__ A, long long lda, int n, int c0, int r0, long long ldk,
                                                   __half* __restrict__ hi, __half* __restrict__ lo) {
  const int c = (int)blockIdx.y;
  const int rj = c0 + (c / B) * B + B;   // first row of the panel that holds column c
  const float* col = A + (long long)(c0 + c) * lda;
  for (long long k = (long long)blockIdx.x * 256 + threadIdx.x; k < ldk; k += (long long)gridDim.x * 256) {
    const long long i = r0 + k;
    const float x = (i < n && i >= rj) ? col[i] * kScV : 0.f;
    const __half h = __float2half_rn(x);
    hi[(long long)c * ldk + k] = h;
    lo[(long long)c * ldk + k] = __float2half_rn(x - __half2float(h));
  }
}
// (V T) of the block's panels, row-major [m][ldo]: element (i, c) sits at A[(c0 + c) + i lda] for i >= the panel's first row
__global__ void __launch_bounds__(256) k_q1_conv_vt(const float* __restrict__ A, long long lda, int n, int c0, int ncols, int r0,
                                                    long long ldo, __half* __restrict__ hi, __half* __restrict__ lo) {
  const long long i = r0 + (long long)blockIdx.x;
  if (i >= n) return;
  const float* row = A + i * lda + c0;
  for (int c = (int)threadIdx.x; c < ldo; c += 256) {
    const int rj = c0 + (c / B) * B + B;
    const float x = (c < ncols && i >= rj) ? row[c] * kScVT : 0.f;
    const __half h = __float2half_rn(x);
    hi[(long long)blockIdx.x * ldo + c] = h;
    lo[(long long)blockIdx.x * ldo + c] = __float2half_rn(x - __half2float(h));
  }
}
// St[j][l][c'][c] = sum_d G[64 j + c][64 l + d] T_l[d][c']   (l > j)
__global__ void __launch_bounds__(256) k_q1_couplings(const float* __restrict__ G, int ldg, const float* __restrict__ T1, int np,
                                                      float* __restrict__ St) {
  const int l = (int)blockIdx.x, j = (int)blockIdx.y;
  if (l <= j || l >= np) return;
  __shared__ float Gs[B][B + 1], Ts[B][B + 1];
  for (int e = (int)threadIdx.x; e < B * B; e += 256) {
    Gs[e / B][e % B] = G[(long long)(B * j + e / B) * ldg + B * l + e % B];
    Ts[e / B][e % B] = T1[(size_t)l * B * B + e];
  }
  __syncthreads();
  float* out = St + ((size_t)j * np + l) * B * B;
  for (int e = (int)threadIdx.x; e < B * B; e += 256) {
    const int cp = e / B, c = e % B;
    float acc = 0.f;
#pragma unroll 8
    for (int d = 0; d < B; ++d) acc = fmaf(Gs[c][d], Ts[d][cp], acc);
    out[cp * B + c] = acc;
  }
}
// X_j = Y_j - sum_{l > j} S_jl X_l, j = np - 2 .. 0, in place on Y [np 64][ldy]; one thread per vector
__global__ void __launch_bounds__(128) k_q1_recursion(float* __restrict__ Y, long long ldy, int mvec, int np, const float* __restrict__ St) {
  extern __shared__ __align__(16) float Ss[];   // [np - 1 - j][c'][c]
  const int v = (int)blockIdx.x * 128 + (int)threadIdx.x;
  for (int j = np - 2; j >= 0; --j) {
    const int nl = np - 1 - j;
    __syncthreads();
    for (int e = (int)threadIdx.x; e < nl * B * B / 4; e += 128)
      reinterpret_cast<float4*>(Ss)[e] = reinterpret_cast<const float4*>(St + ((size_t)j * np + j + 1) * B * B)[e];
    __syncthreads();
    if (v < mvec) {
      float acc[B];
#pragma unroll
      for (int c = 0; c < B; ++c) acc[c] = Y[(long long)(B * j + c) * ldy + v];
      for (int l = 0; l < nl; ++l) {
        const float* Yl = Y + (long long)(B * (j + 1 + l)) * ldy + v;
        const float* Sl = Ss + (size_t)l * B * B;
        for (int cp = 0; cp < B; ++cp) {
          const float xl = Yl[(long long)cp * ldy];
#pragma unroll
          for (int c4 = 0; c4 < B / 4; ++c4) {
            const float4 sv = *reinterpret_cast<const float4*>(Sl + cp * B + 4 * c4);
            acc[4 * c4 + 0] = fmaf(-sv.x, xl, acc[4 * c4 + 0]);
            acc[4 * c4 + 1] = fmaf(-sv.y, xl, acc[4 * c4 + 1]);
            acc[4 * c4 + 2] = fmaf(-sv.z, xl, acc[4 * c4 + 2]);
            acc[4 * c4 + 3] = fmaf(-sv.w, xl, acc[4 * c4 + 3]);
          }
        }
      }
#pragma unroll
      for (int c = 0; c < B; ++c) Y[(long long)(B * j + c) * ldy + v] = acc[c];
    }
  }
}
// X [ncols][ldy] (FP32) -> (hi, lo) binary16, vector-major [mvec][ldo]
__global__ void __launch_bounds__(256) k_q1_conv_x(const float* __restrict__ X, long long ldy, int mvec, int ncols, long long ldo,
                                                   __half* __restrict__ hi, __half* __restrict__ lo) {
  __shared__ float tl[32][33];
  const int v0 = (int)blockIdx.x * 32, c0 = (int)blockIdx.y * 32;
  const int tx = (int)threadIdx.x & 31, ty = (int)threadIdx.x >> 5;
  for (int r = ty; r < 32; r += 8) {
    const int c = c0 + r, v = v0 + tx;
    tl[r][tx] = (c < ncols && v < mvec) ? X[(long long)c * ldy + v] * kScX : 0.f;
  }
  __syncthreads();
  for (int r = ty; r < 32; r += 8) {
    const int v = v0 + r, c = c0 + tx;
    if (v < mvec && c < ldo) {
      const float x = tl[tx][r];
      const __half h = __float2half_rn(x);
      hi[(long long)v * ldo + c] = h;
      lo[(long long)v * ldo + c] = __float2half_rn(x - __half2float(h));
    }
  }
}
// Z[v][r0 + k] += U[v][k]
__global__ void __launch_bounds__(256) k_q1_add(float* __restrict__ Z, long long ldz, int r0, const float* __restrict__ U, long long ldu,
                                                int m, int mvec) {
  for (int v = (int)blockIdx.y; v < mvec; v += (int)gridDim.y) {
    float* z = Z + (long long)v * ldz + r0;
    const float* u = U + (long long)v * ldu;
    for (int k = ((int)blockIdx.x * 256 + (int)threadIdx.x) * 4; k < m; k += (int)gridDim.x * 1024) {
      if (k + 3 < m) {
        float4 a = *reinterpret_cast<float4*>(z + k);
        const float4 b = *reinterpret_cast<const float4*>(u + k);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
        *reinterpret_cast<float4*>(z + k) = a;
      } else {
        for (int q = k; q < m; ++q) z[q] += u[q];
      }
    }
  }
}

}  // namespace

void apply_q2(const float* V2, long long ldv2, const float* tau2, long long ldt2, int n, float* Z, long long ldz, int mvec,
              cudaStream_t st) {
  if (mvec <= 0 || n <= 2) return;
  const int nsweeps = n - 2;
  const int ngroups = (nsweeps + B - 1) / B;
  const int nlev = sb2st_levels(n);
  const int q = (n - 3) / B;   // last group; group G has q - G + 1 levels
  const size_t nblk = (size_t)(q + 1) * (q + 2) / 2;
  Tmp<__half> Img(nblk * kBlkHalves, st);
  k_q2_images_h<<<dim3(nlev, ngroups), 256, 0, st>>>(V2, ldv2, tau2, ldt2, n, q, Img.p);
  SCL_CUDA(cudaGetLastError());
  // 16-vector tiles, one warp each; at most 12 warps per CTA (registers are granted to a CTA in units of four warps: 255 per
  // thread up to 8 warps, 168 up to 12), as few waves as that allows
  const int tiles = (mvec + 15) / 16, sms = sm_count();
  const int waves = (tiles + sms * 12 - 1) / (sms * 12);
  const int grid = std::min(tiles, sms * waves);
  const int base = tiles / grid, extra = tiles % grid;
  const int warps = base + (extra ? 1 : 0);
  const size_t smem = (size_t)kStagesH * kBlkBytesH + 2 * kStagesH * sizeof(uint64_t);
  Q2HArgs a{Img.p, Z, ldz, n, mvec, q, tiles, base, extra};
  if (warps <= 8) {
    SCL_CUDA(cudaFuncSetAttribute(k_q2_apply_h<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_q2_apply_h<8><<<grid, warps * 32, smem, st>>>(a);
  } else {
    SCL_CUDA(cudaFuncSetAttribute(k_q2_apply_h<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    k_q2_apply_h<12><<<grid, warps * 32, smem, st>>>(a);
  }
  SCL_CUDA(cudaGetLastError());
  count_launches(2);
}

void unit_vectors(float* Z, long long ldz, int n, int mvec, cudaStream_t st) {
  if (mvec <= 0) return;
  k_unit_vectors<<<(mvec + 7) / 8, 256, 0, st>>>(Z, ldz, n, mvec);
  SCL_CUDA(cudaGetLastError());
  count_launches(1);
}

static void apply_q1_umma(const float* A, int n, long long lda, const float* T1, int npanels, float* Z, long long ldz, int mvec,
                          cudaStream_t st) {
  const int nblocks = (npanels + kQ1Panels - 1) / kQ1Panels;
  const long long ldk_max = (((long long)n + 7) & ~7LL), ldo = kQ1Panels * B;
  const long long ldy = ((long long)mvec + 7) & ~7LL;
  Tmp<__half> vh((size_t)ldo * ldk_max, st), vl((size_t)ldo * ldk_max, st), th((size_t)ldk_max * ldo, st), tl((size_t)ldk_max * ldo, st);
  Tmp<__half> zh((size_t)mvec * ldk_max, st), zl((size_t)mvec * ldk_max, st), xh((size_t)mvec * ldo, st), xl((size_t)mvec * ldo, st);
  Tmp<float> Y((size_t)ldo * ldy, st), G((size_t)ldo * ldo, st), St((size_t)kQ1Panels * kQ1Panels * B * B, st), U((size_t)mvec * ldk_max, st);
  const size_t rec_smem = (size_t)(kQ1Panels - 1) * B * B * sizeof(float);
  SCL_CUDA(cudaFuncSetAttribute(k_q1_recursion, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rec_smem));
  long launches = 0;
  for (int b = nblocks - 1; b >= 0; --b) {
    const int a = b * kQ1Panels, np = std::min(kQ1Panels, npanels - a);
    const int c0 = a * B, r0 = c0 + B, m = n - r0, ncols = np * B;
    if (m < 1) continue;
    const long long ldk = ((long long)m + 7) & ~7LL;
    k_q1_conv_v<<<dim3((unsigned)std::min<long long>((ldk + 255) / 256, 64), ncols), 256, 0, st>>>(A, lda, n, c0, r0, ldk, vh.p, vl.p);
    k_q1_conv_vt<<<m, 256, 0, st>>>(A, lda, n, c0, ncols, r0, ldo, th.p, tl.p);
    strided_split_f32_to_f16(Z + r0, mvec, m, ldz, ldk, zh.p, zl.p, st, kScZ);
    GemmArgs g;
    // Y = V' Z
    g.A.hi = vh.p; g.A.lo = vl.p; g.A.rows = ncols; g.A.K = m; g.A.ld = ldk;
    g.B.hi = zh.p; g.B.lo = zl.p; g.B.rows = mvec; g.B.K = m; g.B.ld = ldk;
    g.alpha = 1.f / (kScV * kScZ);
    g.chunk_kb = kQ1ChunkKb;   // short tensor-core chains: the accumulator truncates, 3e-8 per MMA of a chain, one-sided
    g.epi = Epilogue::Store;
    g.C = Y.p; g.ldc = ldy;
    gemm_umma(g, st);
    if (np > 1) {
      GemmArgs s2;
      s2.A.hi = vh.p; s2.A.lo = vl.p; s2.A.rows = ncols; s2.A.K = m; s2.A.ld = ldk;
      s2.B = s2.A;
      s2.syrk = true;
      s2.alpha = 1.f / (kScV * kScV);
      s2.C = G.p; s2.ldc = ldo;
      gemm_umma(s2, st);
      k_q1_couplings<<<dim3(np, np), 256, 0, st>>>(G.p, (int)ldo, T1 + (size_t)a * B * B, np, St.p);
      k_q1_recursion<<<(mvec + 127) / 128, 128, rec_smem, st>>>(Y.p, ldy, mvec, np, St.p);
      launches += 3;
    }
    k_q1_conv_x<<<dim3((mvec + 31) / 32, (unsigned)(ldo / 32)), 256, 0, st>>>(Y.p, ldy, mvec, ncols, ldo, xh.p, xl.p);
    // U = - X' (VT)'
    GemmArgs u;
    u.A.hi = xh.p; u.A.lo = xl.p; u.A.rows = mvec; u.A.K = ncols; u.A.ld = ldo;
    u.B.hi = th.p; u.B.lo = tl.p; u.B.rows = m; u.B.K = ncols; u.B.ld = ldo;
    u.alpha = -1.f / (kScX * kScVT);
    u.chunk_kb = kQ1ChunkKb;
    u.C = U.p; u.ldc = ldk;
    gemm_umma(u, st);
    k_q1_add<<<dim3((unsigned)std::min((m + 1023) / 1024, 64), (unsigned)std::min(mvec, 65535)), 256, 0, st>>>(Z, ldz, r0, U.p, ldk, m, mvec);
    launches += 7;
  }
  SCL_CUDA(cudaGetLastError());
  count_launches((int)launches);
}

void apply_q1(const float* A, int n, long long lda, const float* T1, int npanels, float* Z, long long ldz, int mvec,
              cudaStream_t st) {
  if (mvec <= 0 || npanels <= 0) return;
  if (mvec >= 64) {   // a handful of vectors is not worth the block machinery: panel by panel below
    apply_q1_umma(A, n, lda, T1, npanels, Z, ldz, mvec, st);
    return;
  }
  const long long ldx = ((long long)mvec + 3) & ~3LL;
  const int max_split = 16;
  Tmp<float> Xpart((size_t)max_split * B * ldx, st), Xp((size_t)B * ldx, st);
  const int vt = (mvec + tile::TM - 1) / tile::TM;
  const int slots = 2 * sm_count();
  for (int k = npanels - 1; k >= 0; --k) {
    const int c0 = k * B, r0 = c0 + B, m = n - r0;
    if (m < 1) continue;
    const float* Vp = A + r0 + (long long)c0 * lda;
    int split = std::max(1, std::min(max_split, (4 * slots + vt - 1) / vt));
    int chunk = ((m + split - 1) / split + tile::KT - 1) / tile::KT * tile::KT;
    chunk = std::max(chunk, 4 * tile::KT);
    split = (m + chunk - 1) / chunk;
    const size_t nx = (size_t)B * ldx;
    k_q1_x_tc<<<dim3(vt, split), 256, 0, st>>>(Vp, lda, m, Z + r0, ldz, mvec, Xpart.p, ldx, chunk);
    k_sum_parts32<<<(unsigned)((nx + 255) / 256), 256, 0, st>>>(Xpart.p, split, nx, nx, Xp.p);
    k_q1_z_tc<<<dim3((m + tile::TM - 1) / tile::TM, vt), 256, 0, st>>>(A + c0 + (long long)r0 * lda, lda, m, Xp.p, ldx, mvec, Z + r0, ldz);
  }
  SCL_CUDA(cudaGetLastError());
  count_launches(3 * npanels);
}

}  // namespace scl
