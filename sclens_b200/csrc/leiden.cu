// Clustering of the cell graph on the device: batched Leiden trials (modularity with resolution, the RB configuration
// model), the element-centric similarity (ECS) of labelings and the inconsistency coefficient (IC) of scICE.
//
// Weights.  Every edge weight becomes an unsigned 64-bit fixed-point integer round(w 2^s) (at least 1), with s <= 32 chosen
// from the largest weight and nnz so that 2m < 2^62.  Degrees, community totals and coarse weights are then exact integer
// sums: integer atomics give the same bits in any order, so nothing needs a sort or a fixed reduction tree.  Gains are
// evaluated in Float64 from those integers with explicit round-to-nearest operations (no FMA contraction).
// oracle/leiden_ref.py restates the algorithm step for step (hashes, integer weights, gain expression, tie rules), and
// tests/test_leiden_gpu.py compares the labels bit for bit.
//
// Batch.  R resolutions x T trials run as one disjoint union of G = R T copies.  Level 0 reads the caller's CSR through
// (copy, vertex) = divmod(global id, N); from level 1 on the coarse graphs of all copies form one CSR.  A copy's draws are
// hashes of its own key (seed, trial) and of copy-local vertex ids, and communities never span copies, so a trial gives
// the same labels alone or inside any batch.
//
// One level.  (1) Local moving in sweeps of two sub-rounds: a hash bit of (key, iteration, level, sweep, vertex) picks the
// sub-round of each vertex; a vertex of the sub-round sums its row per neighbouring community (warp, open-addressing
// table) and moves to the best strictly positive gain against the totals of the sub-round's start (ties: smaller id; a
// singleton enters a singleton only when that one's id is smaller); totals are rebuilt with integer atomics.  The level
// ends after a sweep without a move or at max_sweeps.  (2) Refinement from singletons inside each community, one sweep of
// two sub-rounds: a well-connected singleton of the sub-round joins a well-connected subset of its community whose members
// are not movers in the sub-round, or stays, drawn with probability exp(gain / theta) (Gumbel-max race over the
// candidates with gain >= 0, staying has gain 0).  (3) Aggregation of the refined subsets (renumbered per copy by a prefix
// sum) into a CSR with sorted columns, summed integer weights and self-loops; the coarse partition is the local-moving one.
// A copy stops at a level whose local moving moved no vertex and whose refinement merged nothing; an iteration restarts from its labels on the original graph until one
// changes no label (max_iterations).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <numeric>
#include "handle.h"
#include "leiden.h"
#include "subspace.h"
#include "tmp.cuh"

namespace scl {

namespace {

constexpr uint32_t kEmpty = 0xffffffffu;
constexpr int kWarps = 4;              // warps per CTA of the row kernels
constexpr int kCap = 512;              // shared-memory table slots per warp (rows up to kCap / 2 entries)
constexpr int kMaxLevels = 256;
constexpr int64_t kBatchVertices = (int64_t)1 << 27;   // copies x vertices of one device batch (~16 GB of state)

inline int blocks(size_t n, int t) { return (int)std::min<size_t>((n + t - 1) / t, 1u << 30); }

// ---- draws -----------------------------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint64_t step_key(uint64_t copy_key, uint32_t stream, uint32_t iter, uint32_t level,
                                                      uint32_t sweep) {
  return mix64s(mix64s(copy_key ^ (0x9e3779b97f4a7c15ull * (stream + 1ull))) ^
                (((uint64_t)iter << 48) | ((uint64_t)level << 32) | sweep));
}
__device__ __forceinline__ uint64_t draw_bits(uint64_t key, uint32_t a, uint32_t b) {
  return mix64s(mix64s(key ^ (((uint64_t)a << 32) | b)));
}
// Gumbel(0, 1) from the 53 high bits: u in (0, 1)
__device__ __forceinline__ double gumbel(uint64_t key, uint32_t a, uint32_t b) {
  const double u = __dmul_rn(__dadd_rn((double)(draw_bits(key, a, b) >> 11), 0.5), 1.1102230246251565e-16);
  return -log(-log(u));
}

// ---- graph of one level ----------------------------------------------------------------------------------------------
struct LGraph {
  int level0;
  uint32_t N0;                                   // level 0: vertices of the shared graph, v = copy * N0 + i
  const uint32_t* rp0;
  const uint32_t* col0;
  const uint64_t* w0;
  const uint64_t* rp;                            // level >= 1: batch CSR with global vertex ids
  const uint32_t* col;
  const uint64_t* w;
  const uint32_t* copy;                          // level >= 1: copy of every vertex
  const uint32_t* voff;                          // [G + 1] first vertex of every copy
};
__device__ __forceinline__ uint32_t copy_of(const LGraph& g, uint32_t v) { return g.level0 ? v / g.N0 : g.copy[v]; }
__device__ __forceinline__ void row_of(const LGraph& g, uint32_t v, uint64_t& b, uint64_t& e, uint32_t& base) {
  if (g.level0) {
    const uint32_t i = v % g.N0;
    b = g.rp0[i]; e = g.rp0[i + 1]; base = v - i;
  } else {
    b = g.rp[v]; e = g.rp[v + 1]; base = 0;
  }
}
__device__ __forceinline__ uint32_t col_at(const LGraph& g, uint64_t t, uint32_t base) { return base + (g.level0 ? g.col0[t] : g.col[t]); }
__device__ __forceinline__ uint64_t w_at(const LGraph& g, uint64_t t) { return g.level0 ? g.w0[t] : g.w[t]; }

// ---- per-warp open-addressing table (shared or global memory: generic pointers) --------------------------------------
struct Tab {
  uint32_t* key;
  unsigned long long* val;
  uint32_t mask;
};
__device__ __forceinline__ uint32_t tab_size_for(uint64_t len) {
  uint32_t s = 32;
  while (s < 2 * len) s <<= 1;
  return s;
}
__device__ __forceinline__ void tab_clear(const Tab& t, int lane) {
  for (uint32_t i = lane; i <= t.mask; i += 32) { t.key[i] = kEmpty; t.val[i] = 0; }
  __syncwarp();
}
__device__ __forceinline__ void tab_add(const Tab& t, uint32_t k, uint64_t w) {
  uint32_t h = (k * 0x9E3779B1u) & t.mask;
  while (true) {
    const uint32_t old = atomicCAS(&t.key[h], kEmpty, k);
    if (old == kEmpty || old == k) { atomicAdd(&t.val[h], (unsigned long long)w); return; }
    h = (h + 1) & t.mask;
  }
}
// best (score, id): larger score, then smaller id
__device__ __forceinline__ void warp_best(double& s, uint32_t& id) {
  for (int o = 16; o; o >>= 1) {
    const double s2 = __shfl_xor_sync(0xffffffffu, s, o);
    const uint32_t i2 = __shfl_xor_sync(0xffffffffu, id, o);
    if (s2 > s || (s2 == s && i2 < id)) { s = s2; id = i2; }
  }
}

struct Tables {          // where a warp's table lives: shared (small rows) or a global slice (long rows)
  uint32_t* gkey;
  unsigned long long* gval;
  uint32_t gslots;       // slots per global slice (0: shared kernel)
};

// Which table a warp uses for a row of len entries; false when another kernel handles the row.
__device__ __forceinline__ bool pick_table(const Tables& T, uint64_t len, uint32_t* skey, unsigned long long* sval, int wib,
                                           uint32_t gwarp, Tab& t) {
  const uint32_t need = tab_size_for(len);
  if (T.gslots == 0) {
    if (need > kCap) return false;
    t.key = skey + wib * kCap; t.val = sval + wib * kCap; t.mask = need - 1;
  } else {
    if (need <= kCap) return false;
    t.key = T.gkey + (size_t)gwarp * T.gslots; t.val = T.gval + (size_t)gwarp * T.gslots; t.mask = need - 1;
  }
  return true;
}

struct CopyPar {
  const double* gamma;     // [G]
  const uint64_t* key;     // [G]
  const uint8_t* active;   // [G]
};

// ---- local moving ----------------------------------------------------------------------------------------------------
// score of community c for v: w(v, c) - (gamma k_v) (K_c / 2m); the expression the oracle restates
__device__ __forceinline__ double move_score(uint64_t w, double gk, uint64_t K, double inv2m) {
  return __dsub_rn((double)w, __dmul_rn(gk, __dmul_rn((double)K, inv2m)));
}

__device__ __forceinline__ uint64_t warp_sum_u64(uint64_t x) {
  for (int o = 16; o; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
  return x;
}

// one warp per vertex of the sub-round; comm_new starts as a copy of comm and only movers are written
__global__ void __launch_bounds__(kWarps * 32) k_move(LGraph g, uint32_t n, CopyPar cp, const uint32_t* __restrict__ comm,
                                                      const unsigned long long* __restrict__ K, const uint32_t* __restrict__ csize,
                                                      const unsigned long long* __restrict__ deg, uint32_t* __restrict__ comm_new,
                                                      double inv2m, uint32_t iter, uint32_t level, uint32_t sweep, uint32_t sub,
                                                      unsigned int* __restrict__ moved, Tables T) {
  __shared__ uint32_t skey[kWarps * kCap];
  __shared__ unsigned long long sval[kWarps * kCap];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t gw = blockIdx.x * kWarps + wib, nw = gridDim.x * kWarps;
  for (uint32_t v = gw; v < n; v += nw) {
    const uint32_t c = copy_of(g, v);
    if (!cp.active[c]) continue;
    const uint32_t vl = v - g.voff[c];
    if ((uint32_t)(draw_bits(step_key(cp.key[c], 7, iter, level, sweep), vl, 0) & 1) != sub) continue;
    uint64_t b, e;
    uint32_t base;
    row_of(g, v, b, e, base);
    Tab t;
    if (!pick_table(T, e - b, skey, sval, wib, gw, t)) continue;
    tab_clear(t, lane);
    for (uint64_t q = b + lane; q < e; q += 32) {
      const uint32_t x = col_at(g, q, base);
      if (x != v) tab_add(t, comm[x], w_at(g, q));
    }
    __syncwarp();
    const uint32_t a = comm[v];
    const uint64_t kv = deg[v];
    const double gk = __dmul_rn(cp.gamma[c], (double)kv);
    const bool single = csize[a] == 1;
    double best = -INFINITY;
    uint32_t bid = kEmpty;
    uint64_t wa = 0;
    for (uint32_t i = lane; i <= t.mask; i += 32) {
      const uint32_t k = t.key[i];
      if (k == kEmpty) continue;
      if (k == a) { wa = t.val[i]; continue; }
      if (single && csize[k] == 1 && k > a) continue;
      const double s = move_score(t.val[i], gk, K[k], inv2m);
      if (s > best || (s == best && k < bid)) { best = s; bid = k; }
    }
    wa = warp_sum_u64(wa);
    warp_best(best, bid);
    const double stay = move_score(wa, gk, K[a] - kv, inv2m);
    if (lane == 0 && bid != kEmpty && best > stay) {
      comm_new[v] = bid;
      atomicAdd(&moved[c], 1u);
    }
    __syncwarp();
  }
}

// totals of a partition: tot[p[v]] += deg[v], cnt[p[v]] += 1 (tot / cnt zeroed by the caller)
__global__ void k_totals(const uint32_t* __restrict__ p, const unsigned long long* __restrict__ deg, uint32_t n,
                         unsigned long long* __restrict__ tot, uint32_t* __restrict__ cnt) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  atomicAdd(&tot[p[v]], deg[v]);
  atomicAdd(&cnt[p[v]], 1u);
}

// ---- refinement ------------------------------------------------------------------------------------------------------
// ext[s] = w(S, C - S) of every refined subset S (zeroed by the caller)
__global__ void k_ext(LGraph g, uint32_t n, const uint32_t* __restrict__ comm, const uint32_t* __restrict__ ref,
                      unsigned long long* __restrict__ ext) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  uint64_t b, e;
  uint32_t base;
  row_of(g, v, b, e, base);
  const uint32_t a = comm[v], r = ref[v];
  uint64_t acc = 0;
  for (uint64_t q = b; q < e; ++q) {
    const uint32_t x = col_at(g, q, base);
    if (x != v && comm[x] == a && ref[x] != r) acc += w_at(g, q);
  }
  if (acc) atomicAdd(&ext[r], (unsigned long long)acc);
}

// well connected: w(S, C - S) >= gamma K_S (K_C - K_S) / 2m
__device__ __forceinline__ bool well_connected(uint64_t ext, double gamma, uint64_t KS, uint64_t KC, double inv2m) {
  return (double)ext >= __dmul_rn(__dmul_rn(gamma, (double)KS), __dmul_rn((double)(KC - KS), inv2m));
}

__global__ void __launch_bounds__(kWarps * 32) k_refine(LGraph g, uint32_t n, CopyPar cp, const uint32_t* __restrict__ comm,
                                                        const unsigned long long* __restrict__ K,
                                                        const unsigned long long* __restrict__ deg,
                                                        const uint32_t* __restrict__ ref, const unsigned long long* __restrict__ Kr,
                                                        const uint32_t* __restrict__ rsize,
                                                        const unsigned long long* __restrict__ ext, uint32_t* __restrict__ ref_new,
                                                        double inv2m, double ctheta, uint32_t iter, uint32_t level, uint32_t sub,
                                                        Tables T) {
  __shared__ uint32_t skey[kWarps * kCap];
  __shared__ unsigned long long sval[kWarps * kCap];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t gw = blockIdx.x * kWarps + wib, nw = gridDim.x * kWarps;
  for (uint32_t v = gw; v < n; v += nw) {
    const uint32_t c = copy_of(g, v);
    if (!cp.active[c]) continue;
    const uint32_t o = g.voff[c], vl = v - o;
    const uint64_t k8 = step_key(cp.key[c], 8, iter, level, 0);
    if ((uint32_t)(draw_bits(k8, vl, 0) & 1) != sub) continue;
    if (ref[v] != v || rsize[v] != 1) continue;
    const uint32_t a = comm[v];
    const uint64_t kv = deg[v];
    const double gamma = cp.gamma[c];
    const double gk = __dmul_rn(gamma, (double)kv);
    if (!well_connected(ext[v], gamma, kv, K[a], inv2m)) continue;
    uint64_t b, e;
    uint32_t base;
    row_of(g, v, b, e, base);
    Tab t;
    if (!pick_table(T, e - b, skey, sval, wib, gw, t)) continue;
    tab_clear(t, lane);
    for (uint64_t q = b + lane; q < e; q += 32) {
      const uint32_t x = col_at(g, q, base);
      if (x != v && comm[x] == a) tab_add(t, ref[x], w_at(g, q));
    }
    __syncwarp();
    const uint64_t k9 = step_key(cp.key[c], 9, iter, level, sub);
    double best = gumbel(k9, vl, vl);     // staying: gain 0
    uint32_t bid = v;
    for (uint32_t i = lane; i <= t.mask; i += 32) {
      const uint32_t S = t.key[i];
      if (S == kEmpty) continue;
      if (rsize[S] == 1 && (uint32_t)(draw_bits(k8, S - o, 0) & 1) == sub) continue;   // a singleton of this sub-round
      const uint64_t KS = Kr[S];
      if (!well_connected(ext[S], gamma, KS, K[a], inv2m)) continue;
      const double gain = move_score(t.val[i], gk, KS, inv2m);
      if (!(gain >= 0.0)) continue;
      const double s = __dadd_rn(__dmul_rn(gain, ctheta), gumbel(k9, vl, S - o));
      if (s > best || (s == best && S < bid)) { best = s; bid = S; }
    }
    warp_best(best, bid);
    if (lane == 0 && bid != v) ref_new[v] = bid;
    __syncwarp();
  }
}

// ---- aggregation -----------------------------------------------------------------------------------------------------
__global__ void k_live_count(LGraph g, uint32_t n, const uint32_t* __restrict__ rsize, unsigned int* __restrict__ cnt) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n && rsize[s] > 0) atomicAdd(&cnt[copy_of(g, s)], 1u);
}

__global__ void k_live_flag(LGraph g, uint32_t n, const uint32_t* __restrict__ rsize, const uint8_t* __restrict__ active,
                            uint32_t* __restrict__ flag) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n) flag[s] = (rsize[s] > 0 && active[copy_of(g, s)]) ? 1u : 0u;
}

// labels of the copies that finish at this level: level-0 id space, copy * N0 + local community id
__global__ void k_record(const uint32_t* __restrict__ map0, const uint32_t* __restrict__ comm, const uint32_t* __restrict__ voff,
                         const uint8_t* __restrict__ finish, uint32_t N0, size_t n0, uint32_t* __restrict__ fin) {
  const size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (v >= n0) return;
  const uint32_t c = (uint32_t)(v / N0);
  if (finish[c]) fin[v] = c * N0 + (comm[map0[v]] - voff[c]);
}

__global__ void k_coarse_nodes(LGraph g, uint32_t n, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ nid,
                               const uint32_t* __restrict__ comm, const unsigned long long* __restrict__ Kr,
                               const uint32_t* __restrict__ rsize, uint32_t* __restrict__ ccopy, unsigned long long* __restrict__ cdeg,
                               uint32_t* __restrict__ cmin, uint32_t* __restrict__ mcnt) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n || !flag[s]) return;
  const uint32_t t = nid[s];
  ccopy[t] = copy_of(g, s);
  cdeg[t] = Kr[s];
  mcnt[t] = rsize[s];
  atomicMin(&cmin[comm[s]], t);
}

__global__ void k_coarse_comm(uint32_t n, const uint32_t* __restrict__ flag, const uint32_t* __restrict__ nid,
                              const uint32_t* __restrict__ comm, const uint32_t* __restrict__ cmin, uint32_t* __restrict__ ccomm) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s < n && flag[s]) ccomm[nid[s]] = cmin[comm[s]];
}

__global__ void k_map0(uint32_t* __restrict__ map0, const uint32_t* __restrict__ ref, const uint32_t* __restrict__ nid,
                       const uint8_t* __restrict__ active, uint32_t N0, size_t n0) {
  const size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (v < n0 && active[v / N0]) map0[v] = nid[ref[map0[v]]];
}

__global__ void k_members(LGraph g, uint32_t n, const uint8_t* __restrict__ active, const uint32_t* __restrict__ ref,
                          const uint32_t* __restrict__ nid, const uint32_t* __restrict__ mptr, uint32_t* __restrict__ mcur,
                          uint32_t* __restrict__ mem, unsigned long long* __restrict__ rbound) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n || !active[copy_of(g, v)]) return;
  const uint32_t t = nid[ref[v]];
  mem[mptr[t] + atomicAdd(&mcur[t], 1u)] = v;
  uint64_t b, e;
  uint32_t base;
  row_of(g, v, b, e, base);
  atomicAdd(&rbound[t], (unsigned long long)(e - b));
}

// one warp per coarse node: phase 0 counts its distinct coarse neighbours, phase 1 writes them (unsorted) at rp[t]
__global__ void __launch_bounds__(kWarps * 32) k_coarse_rows(LGraph g, uint32_t nc, const uint32_t* __restrict__ mptr,
                                                             const uint32_t* __restrict__ mem, const unsigned long long* __restrict__ rbound,
                                                             const uint32_t* __restrict__ ref, const uint32_t* __restrict__ nid,
                                                             int phase, unsigned long long* __restrict__ dcnt,
                                                             const unsigned long long* __restrict__ rp, uint32_t* __restrict__ tcol,
                                                             unsigned long long* __restrict__ tw, Tables T) {
  __shared__ uint32_t skey[kWarps * kCap];
  __shared__ unsigned long long sval[kWarps * kCap];
  const int wib = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t gw = blockIdx.x * kWarps + wib, nw = gridDim.x * kWarps;
  for (uint32_t s = gw; s < nc; s += nw) {
    Tab t;
    if (!pick_table(T, rbound[s], skey, sval, wib, gw, t)) continue;
    tab_clear(t, lane);
    for (uint32_t m = mptr[s]; m < mptr[s + 1]; ++m) {
      const uint32_t u = mem[m];
      uint64_t b, e;
      uint32_t base;
      row_of(g, u, b, e, base);
      for (uint64_t q = b + lane; q < e; q += 32) tab_add(t, nid[ref[col_at(g, q, base)]], w_at(g, q));
    }
    __syncwarp();
    uint64_t pos = phase ? rp[s] : 0;
    for (uint32_t i0 = 0; i0 <= t.mask; i0 += 32) {
      const uint32_t k = t.key[i0 + lane];
      const unsigned bal = __ballot_sync(0xffffffffu, k != kEmpty);
      if (phase && k != kEmpty) {
        const uint64_t p = pos + __popc(bal & ((1u << lane) - 1));
        tcol[p] = k;
        tw[p] = t.val[i0 + lane];
      }
      pos += __popc(bal);
    }
    if (!phase && lane == 0) dcnt[s] = pos;
    __syncwarp();
  }
}

// one warp per coarse row: rank the distinct columns into ascending order
__global__ void k_rank_rows(uint32_t nc, const unsigned long long* __restrict__ rp, const uint32_t* __restrict__ tcol,
                            const unsigned long long* __restrict__ tw, uint32_t* __restrict__ col, unsigned long long* __restrict__ w) {
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const uint32_t nw = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t s = warp; s < nc; s += nw) {
    const uint64_t b = rp[s], L = rp[s + 1] - b;
    for (uint64_t q = lane; q < L; q += 32) {
      const uint32_t c = tcol[b + q];
      uint64_t r = 0;
      for (uint64_t u = 0; u < L; ++u) r += tcol[b + u] < c;
      col[b + r] = c;
      w[b + r] = tw[b + q];
    }
  }
}

__global__ void k_row_len_max(LGraph g, uint32_t n, unsigned long long* __restrict__ out) {   // out[0] max, out[1] long rows
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n) return;
  uint64_t b, e;
  uint32_t base;
  row_of(g, v, b, e, base);
  if (e - b > kCap / 2) { atomicMax(&out[0], (unsigned long long)(e - b)); atomicAdd(&out[1], 1ull); }
}

__global__ void k_bound_max(const unsigned long long* __restrict__ rb, uint32_t n, unsigned long long* __restrict__ out) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v < n && rb[v] > kCap / 2) { atomicMax(&out[0], rb[v]); atomicAdd(&out[1], 1ull); }
}

// ---- level 0, labels, restart, modularity ----------------------------------------------------------------------------
__global__ void k_expand(const unsigned long long* __restrict__ deg0, uint32_t N0, size_t n0, unsigned long long* __restrict__ deg,
                         uint32_t* __restrict__ comm, uint32_t* __restrict__ map0) {
  const size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (v >= n0) return;
  deg[v] = deg0[v % N0];
  map0[v] = (uint32_t)v;
  comm[v] = (uint32_t)v;
}

__global__ void k_restart_min(const uint32_t* __restrict__ fin, const uint8_t* __restrict__ active, uint32_t N0, size_t n0,
                              uint32_t* __restrict__ cmin) {
  const size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (v < n0 && active[v / N0]) atomicMin(&cmin[fin[v]], (uint32_t)v);
}
__global__ void k_restart_set(const uint32_t* __restrict__ fin, const uint32_t* __restrict__ cmin, size_t n0, uint32_t* __restrict__ comm) {
  const size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (v < n0) comm[v] = cmin[fin[v]] == kEmpty ? (uint32_t)v : cmin[fin[v]];
}

// intra-cluster weight of every copy on the original graph
__global__ void k_win(const uint32_t* __restrict__ rp, const uint32_t* __restrict__ col, const uint64_t* __restrict__ w,
                      const uint32_t* __restrict__ fin, uint32_t N0, size_t n0, unsigned long long* __restrict__ win) {
  const size_t v = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (v >= n0) return;
  const uint32_t c = (uint32_t)(v / N0), i = (uint32_t)(v % N0);
  const size_t base = (size_t)c * N0;
  const uint32_t l = fin[v];
  uint64_t acc = 0;
  for (uint32_t q = rp[i]; q < rp[i + 1]; ++q)
    if (fin[base + col[q]] == l) acc += w[q];
  if (acc) atomicAdd(&win[c], (unsigned long long)acc);
}

// ---- multi-block exclusive scan: out[0..n) exclusive, out[n] total --------------------------------------------------
constexpr int kScanB = 1024, kScanItems = 8;
template <typename T>
__global__ void __launch_bounds__(kScanB) k_scan_block(const T* __restrict__ in, size_t n, T* __restrict__ out, T* __restrict__ bsum) {
  __shared__ T part[kScanB];
  const size_t b0 = (size_t)blockIdx.x * kScanB * kScanItems + (size_t)threadIdx.x * kScanItems;
  T loc[kScanItems];
  T s = 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i) { loc[i] = b0 + i < n ? in[b0 + i] : 0; s += loc[i]; }
  part[threadIdx.x] = s;
  __syncthreads();
  for (int off = 1; off < kScanB; off <<= 1) {
    const T v = threadIdx.x >= off ? part[threadIdx.x - off] : 0;
    __syncthreads();
    part[threadIdx.x] += v;
    __syncthreads();
  }
  T run = threadIdx.x ? part[threadIdx.x - 1] : 0;
#pragma unroll
  for (int i = 0; i < kScanItems; ++i)
    if (b0 + i < n) { out[b0 + i] = run; run += loc[i]; }
  if (threadIdx.x == kScanB - 1) bsum[blockIdx.x] = part[kScanB - 1];
}
template <typename T>
__global__ void k_scan_add(T* __restrict__ out, size_t n, const T* __restrict__ boff) {
  const size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] += boff[i / ((size_t)kScanB * kScanItems)];
}
template <typename T>
void scan(const T* in, T* out, size_t n, cudaStream_t st) {
  const size_t per = (size_t)kScanB * kScanItems;
  const size_t nb = std::max<size_t>(1, (n + per - 1) / per);
  Tmp<T> bsum(nb + 1, st), boff(nb + 1, st);
  k_scan_block<T><<<(unsigned)nb, kScanB, 0, st>>>(in, n, out, bsum.p);
  if (nb > 1) {
    scan(bsum.p, boff.p, nb, st);
    k_scan_add<T><<<blocks(n, 256), 256, 0, st>>>(out, n, boff.p);
    SCL_CUDA(cudaMemcpyAsync(out + n, boff.p + nb, sizeof(T), cudaMemcpyDeviceToDevice, st));
  } else {
    SCL_CUDA(cudaMemcpyAsync(out + n, bsum.p, sizeof(T), cudaMemcpyDeviceToDevice, st));
  }
  count_launches(nb > 1 ? 2 : 1);
  SCL_CUDA(cudaGetLastError());
}

// ---- graph validation and fixed point --------------------------------------------------------------------------------
enum : unsigned { kBadPtr = 1, kBadCol = 2, kBadVal = 4, kBadSym = 8 };

__global__ void k_check_ptr(const uint32_t* __restrict__ rp, int N, size_t nnz, unsigned int* __restrict__ bad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i > N) return;
  if ((i == 0 && rp[0] != 0) || (i == N && rp[N] != nnz) || (i < N && rp[i] > rp[i + 1])) atomicOr(bad, kBadPtr);
}

template <typename V>
__global__ void k_check_rows(const uint32_t* __restrict__ rp, const uint32_t* __restrict__ col, const V* __restrict__ val, int N,
                             unsigned int* __restrict__ bad, unsigned long long* __restrict__ maxbits) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  unsigned f = 0;
  double mx = 0;
  for (uint32_t q = rp[i]; q < rp[i + 1]; ++q) {
    if (col[q] >= (uint32_t)N || (q > rp[i] && col[q] <= col[q - 1])) f |= kBadCol;
    const double x = (double)val[q];
    if (!(x > 0) || !isfinite(x)) f |= kBadVal; else mx = fmax(mx, x);
  }
  if (f) atomicOr(bad, f);
  atomicMax(maxbits, (unsigned long long)__double_as_longlong(mx));   // positive doubles order as their bits
}

template <typename V>
__global__ void k_check_sym(const uint32_t* __restrict__ rp, const uint32_t* __restrict__ col, const V* __restrict__ val, int N,
                            unsigned int* __restrict__ bad) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  for (uint32_t q = rp[i]; q < rp[i + 1]; ++q) {
    const uint32_t j = col[q];
    uint32_t lo = rp[j], hi = rp[j + 1];
    while (lo < hi) {
      const uint32_t m = (lo + hi) / 2;
      if (col[m] < (uint32_t)i) lo = m + 1; else hi = m;
    }
    if (lo == rp[j + 1] || col[lo] != (uint32_t)i || val[lo] != val[q]) { atomicOr(bad, kBadSym); return; }
  }
}

template <typename V>
__global__ void k_to_fixed(const uint32_t* __restrict__ rp, const V* __restrict__ val, int N, int shift, uint64_t* __restrict__ w,
                           unsigned long long* __restrict__ deg) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  uint64_t s = 0;
  for (uint32_t q = rp[i]; q < rp[i + 1]; ++q) {
    const uint64_t x = (uint64_t)llrint(ldexp((double)val[q], shift));
    w[q] = x ? x : 1;
    s += w[q];
  }
  deg[i] = s;
}

// ---- ECS -------------------------------------------------------------------------------------------------------------
constexpr int kEcsThreads = 256;
constexpr int kEcsSmem = 8192;   // contingency cells in shared memory

// ECS of one trial pair per CTA.  Up to kEcsSmem cells the contingency table is dense in shared memory; above, the
// non-zero cells (at most N) are counted in an open-addressing table of gslots >= 2N slots in a global slice, so the
// work and memory stay O(N) however many clusters the labelings have.
__device__ __forceinline__ double ecs_term(double x, double A, double B) {
  return x * (1.0 - 0.5 * (x * fabs(1.0 / A - 1.0 / B) + (A - x) / A + (B - x) / B));
}

__global__ void __launch_bounds__(kEcsThreads) k_ecs(const int32_t* __restrict__ lab, int N, const int* __restrict__ kk,
                                                     const int* __restrict__ soff, const int* __restrict__ sz,
                                                     const int2* __restrict__ pairs, int p0, unsigned long long* __restrict__ gkey,
                                                     uint32_t* __restrict__ gcnt, uint32_t gslots, double* __restrict__ out) {
  __shared__ uint32_t stab[kEcsSmem];
  __shared__ double red[kEcsThreads];
  const int2 pr = pairs[p0 + blockIdx.x];
  const int kb = kk[pr.y];
  const size_t cells = (size_t)kk[pr.x] * kb;
  const int32_t* la = lab + (size_t)pr.x * N;
  const int32_t* lb = lab + (size_t)pr.y * N;
  const int* sa = sz + soff[pr.x];
  const int* sb = sz + soff[pr.y];
  double acc = 0;
  if (cells <= kEcsSmem) {
    for (size_t c = threadIdx.x; c < cells; c += kEcsThreads) stab[c] = 0;
    __syncthreads();
    for (int v = threadIdx.x; v < N; v += kEcsThreads) atomicAdd(&stab[(size_t)la[v] * kb + lb[v]], 1u);
    __syncthreads();
    for (size_t c = threadIdx.x; c < cells; c += kEcsThreads)
      if (stab[c]) acc += ecs_term(stab[c], sa[c / kb], sb[c % kb]);
  } else {
    unsigned long long* key = gkey + (size_t)blockIdx.x * gslots;
    uint32_t* cnt = gcnt + (size_t)blockIdx.x * gslots;
    const unsigned long long empty = ~0ull;
    for (uint32_t c = threadIdx.x; c < gslots; c += kEcsThreads) { key[c] = empty; cnt[c] = 0; }
    __syncthreads();
    for (int v = threadIdx.x; v < N; v += kEcsThreads) {
      const unsigned long long k = (unsigned long long)la[v] * kb + lb[v];
      uint32_t h = (uint32_t)(mix64s(k) & (gslots - 1));
      while (true) {
        const unsigned long long old = atomicCAS(&key[h], empty, k);
        if (old == empty || old == k) { atomicAdd(&cnt[h], 1u); break; }
        h = (h + 1) & (gslots - 1);
      }
    }
    __syncthreads();
    for (uint32_t c = threadIdx.x; c < gslots; c += kEcsThreads)
      if (cnt[c]) acc += ecs_term(cnt[c], sa[key[c] / kb], sb[key[c] % kb]);
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  for (int o = kEcsThreads / 2; o; o >>= 1) {
    if (threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[p0 + blockIdx.x] = red[0] / N;
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

template <typename T>
void to_host(std::vector<T>& h, const T* d, size_t n, cudaStream_t st) {
  h.resize(n);
  if (n) SCL_CUDA(cudaMemcpyAsync(h.data(), d, n * sizeof(T), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
}
template <typename T>
void to_dev(T* d, const std::vector<T>& h, cudaStream_t st) {
  if (!h.empty()) SCL_CUDA(cudaMemcpyAsync(d, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, st));
}

// Global table slices for the rows a shared table cannot hold; n_long rows, the longest max_len entries.
struct LongTables {
  DBuf<uint32_t> key;
  DBuf<unsigned long long> val;
  Tables get(unsigned long long max_len, unsigned long long n_long, int* grid) {
    if (n_long == 0) return Tables{nullptr, nullptr, 0};
    uint32_t slots = 32;
    while (slots < 2 * max_len) slots <<= 1;
    const size_t budget_slots = (size_t)1 << 28;                       // 3 GiB of slices at most
    size_t warps = std::min<size_t>({(size_t)n_long, (size_t)sm_count() * 16, std::max<size_t>(1, budget_slots / slots)});
    warps = (warps + kWarps - 1) / kWarps * kWarps;
    key.ensure(warps * slots);
    val.ensure(warps * slots);
    *grid = (int)(warps / kWarps);
    return Tables{key.p, val.p, slots};
  }
};

// canonical labels of one copy (raw ids in [base, base + N)): clusters by size descending, ties by smallest member;
// returns the cluster count
int canonical(const uint32_t* raw, uint32_t base, int N, int32_t* out, std::vector<int>& id, std::vector<int>& sizes) {
  id.assign(N, -1);
  sizes.clear();
  for (int i = 0; i < N; ++i) {
    int& c = id[raw[i] - base];
    if (c < 0) { c = (int)sizes.size(); sizes.push_back(0); }   // order of first appearance = order of smallest member
    ++sizes[c];
  }
  const int k = (int)sizes.size();
  std::vector<int> ord(k), rank(k);
  std::iota(ord.begin(), ord.end(), 0);
  std::stable_sort(ord.begin(), ord.end(), [&](int x, int y) { return sizes[x] > sizes[y]; });
  for (int r = 0; r < k; ++r) rank[ord[r]] = r;
  for (int i = 0; i < N; ++i) out[i] = rank[id[raw[i] - base]];
  return k;
}

}  // namespace

// ---- host entry points -----------------------------------------------------------------------------------------------
void leiden_prepare(const uint32_t* rp, const uint32_t* col, const double* val_f64, const float* val_f32, int N, size_t nnz,
                    FixGraph& g, cudaStream_t st) {
  SCL_REQUIRE(N >= 1 && nnz < (1ull << 32), "graph: need N >= 1 and nnz < 2^32");
  Tmp<unsigned int> bad(1, st);
  Tmp<unsigned long long> mx(1, st);
  SCL_CUDA(cudaMemsetAsync(bad.p, 0, sizeof(unsigned), st));
  SCL_CUDA(cudaMemsetAsync(mx.p, 0, sizeof(unsigned long long), st));
  unsigned hb = 0;
  k_check_ptr<<<blocks(N + 1, 256), 256, 0, st>>>(rp, N, nnz, bad.p);
  SCL_CUDA(cudaMemcpyAsync(&hb, bad.p, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  if (hb) throw Error(SCL_ERR_GRAPH, "graph: row pointers are not monotone from 0 to nnz");
  if (val_f64) k_check_rows<<<blocks(N, 128), 128, 0, st>>>(rp, col, val_f64, N, bad.p, mx.p);
  else k_check_rows<<<blocks(N, 128), 128, 0, st>>>(rp, col, val_f32, N, bad.p, mx.p);
  SCL_CUDA(cudaMemcpyAsync(&hb, bad.p, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  if (hb & kBadCol) throw Error(SCL_ERR_GRAPH, "graph: a column is out of range or a row is not strictly increasing");
  if (hb & kBadVal) throw Error(SCL_ERR_GRAPH, "graph: a weight is not finite and positive");
  if (val_f64) k_check_sym<<<blocks(N, 128), 128, 0, st>>>(rp, col, val_f64, N, bad.p);
  else k_check_sym<<<blocks(N, 128), 128, 0, st>>>(rp, col, val_f32, N, bad.p);
  unsigned long long mbits = 0;
  SCL_CUDA(cudaMemcpyAsync(&hb, bad.p, sizeof(unsigned), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaMemcpyAsync(&mbits, mx.p, sizeof(mbits), cudaMemcpyDeviceToHost, st));
  SCL_CUDA(cudaStreamSynchronize(st));
  count_launches(3);
  if (hb) throw Error(SCL_ERR_GRAPH, "graph: not symmetric (a reverse edge is missing or has another weight)");
  double maxw;
  std::memcpy(&maxw, &mbits, sizeof(maxw));
  g.N = N;
  g.nnz = nnz;
  g.shift = leiden_weight_shift(maxw, nnz);
  g.rp.ensure(N + 1);
  g.col.ensure(std::max<size_t>(nnz, 1));
  g.w.ensure(std::max<size_t>(nnz, 1));
  g.deg.ensure(N);
  SCL_CUDA(cudaMemcpyAsync(g.rp.p, rp, (N + 1) * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
  if (nnz) SCL_CUDA(cudaMemcpyAsync(g.col.p, col, nnz * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
  auto* dg = reinterpret_cast<unsigned long long*>(g.deg.p);
  if (val_f64) k_to_fixed<<<blocks(N, 128), 128, 0, st>>>(rp, val_f64, N, g.shift, g.w.p, dg);
  else k_to_fixed<<<blocks(N, 128), 128, 0, st>>>(rp, val_f32, N, g.shift, g.w.p, dg);
  SCL_CUDA(cudaGetLastError());
  std::vector<uint64_t> deg;
  to_host(deg, g.deg.p, N, st);
  g.two_m = 0;
  for (uint64_t d : deg) g.two_m += d;
}

int leiden_weight_shift(double maxw, size_t nnz) {
  int e = 0;
  std::frexp(maxw > 0 ? maxw : 1.0, &e);                     // maxw < 2^e
  int lg = 0;
  while (((size_t)1 << lg) < nnz + 1) ++lg;                   // nnz + 1 <= 2^lg
  return std::min(32, 61 - lg - e);
}

uint64_t leiden_copy_key(uint64_t seed, uint32_t trial) { return umap_stream_key(seed, 6, trial); }

void leiden_run(const FixGraph& gr, const double* gammas, int R, int T, int t0, uint64_t seed, int max_iterations, int max_sweeps,
                double theta, int32_t* labels, int32_t* nclu, double* modularity, LeidenStats* stats, cudaStream_t st) {
  SCL_REQUIRE(R >= 1 && T >= 1 && (int64_t)R * T * gr.N < (1ll << 31), "leiden: resolutions x trials x N must stay below 2^31");
  const int G = R * T;
  const uint32_t N0 = (uint32_t)gr.N;
  const size_t n0 = (size_t)G * N0;
  *stats = LeidenStats{};
  const double inv2m = gr.two_m ? 1.0 / (double)gr.two_m : 0.0;
  const double ctheta = std::ldexp(1.0 / theta, -gr.shift);
  std::vector<double> hg(G);
  std::vector<uint64_t> hk(G);
  for (int r = 0; r < R; ++r)
    for (int t = 0; t < T; ++t) { hg[r * T + t] = gammas[r]; hk[r * T + t] = leiden_copy_key(seed, (uint32_t)(t0 + t)); }
  Tmp<double> dgam(G, st);
  Tmp<uint64_t> dkey(G, st);
  Tmp<uint8_t> dact(G, st), dfinish(G, st);
  to_dev(dgam.p, hg, st);
  to_dev(dkey.p, hk, st);
  // per-level state (level-0 sized; coarse levels are smaller)
  using ull = unsigned long long;
  Tmp<uint32_t> comm(n0, st), comm_new(n0, st), csize(n0, st), ref(n0, st), ref_new(n0, st), rsize(n0, st);
  Tmp<ull> deg(n0, st), K(n0, st), Kr(n0, st), ext(n0, st);
  Tmp<uint32_t> map0(n0, st), fin(n0, st), cmin(n0, st), flag(n0 + 1, st), nid(n0 + 1, st);
  Tmp<uint32_t> voff(G + 1, st), cvoff(G + 1, st), ccopy(n0, st), mcnt(n0 + 1, st), mptr(n0 + 1, st), mcur(n0, st), mem(n0, st);
  Tmp<ull> cdeg(n0, st), rbound(n0, st), misc(2, st);
  Tmp<unsigned int> moved(G, st), cnt(G, st);
  Tmp<uint32_t> ccomm(n0, st), copyA(n0, st);
  DBuf<uint64_t> rpA, rpB, wA, wB, tw;
  DBuf<uint32_t> colA, colB, tcol;
  LongTables lt;
  std::vector<uint8_t> it_active(G, 1), lvl_active(G), finish(G);
  std::vector<int32_t> prev((size_t)G * N0, -1), cur((size_t)N0);
  std::vector<uint32_t> hfin;
  std::vector<unsigned> hmoved(G), hcnt(G);
  std::vector<uint64_t> lvl_moved(G);
  std::vector<uint32_t> hvoff(G + 1);
  std::vector<int> idbuf, sizes;
  std::vector<int> iters(G, 0);
  StageTimer tm(st);
  auto dev_bool = [&](uint8_t* d, const std::vector<uint8_t>& h) { to_dev(d, h, st); };
  for (int it = 0; it < max_iterations; ++it) {
    if (std::none_of(it_active.begin(), it_active.end(), [](uint8_t a) { return a != 0; })) break;
    for (int c = 0; c < G; ++c) if (it_active[c]) iters[c] = it + 1;
    stats->max_iterations = it + 1;
    // level 0
    k_expand<<<blocks(n0, 256), 256, 0, st>>>(reinterpret_cast<const ull*>(gr.deg.p), N0, n0, deg.p, comm.p, map0.p);
    dev_bool(dact.p, it_active);
    if (it > 0) {
      SCL_CUDA(cudaMemsetAsync(cmin.p, 0xff, n0 * sizeof(uint32_t), st));
      k_restart_min<<<blocks(n0, 256), 256, 0, st>>>(fin.p, dact.p, N0, n0, cmin.p);
      k_restart_set<<<blocks(n0, 256), 256, 0, st>>>(fin.p, cmin.p, n0, comm.p);
    }
    for (int c = 0; c <= G; ++c) hvoff[c] = (uint32_t)(c * N0);
    to_dev(voff.p, hvoff, st);
    lvl_active = it_active;
    uint32_t n = (uint32_t)n0;
    LGraph g{1, N0, gr.rp.p, gr.col.p, gr.w.p, nullptr, nullptr, nullptr, nullptr, voff.p};
    uint32_t* cur_copy = nullptr;
    for (int level = 0;; ++level) {
      stats->max_levels = std::max(stats->max_levels, level + 1);
      for (int c = 0; c < G; ++c) stats->copy_levels += lvl_active[c];
      // long rows of this level
      SCL_CUDA(cudaMemsetAsync(misc.p, 0, 2 * sizeof(ull), st));
      k_row_len_max<<<blocks(n, 256), 256, 0, st>>>(g, n, misc.p);
      std::vector<ull> hm;
      to_host(hm, misc.p, 2, st);
      int lgrid = 0;
      const Tables Tl = lt.get(hm[0], hm[1], &lgrid);
      const Tables Ts{nullptr, nullptr, 0};
      const int sgrid = std::max(1, std::min(blocks(n, kWarps), sm_count() * 64));
      const CopyPar cp{dgam.p, dkey.p, dact.p};
      // (1) local moving
      dev_bool(dact.p, lvl_active);
      std::vector<uint8_t> lm = lvl_active;
      std::fill(lvl_moved.begin(), lvl_moved.end(), 0);
      SCL_CUDA(cudaMemsetAsync(K.p, 0, n * sizeof(ull), st));
      SCL_CUDA(cudaMemsetAsync(csize.p, 0, n * sizeof(uint32_t), st));
      k_totals<<<blocks(n, 256), 256, 0, st>>>(comm.p, deg.p, n, K.p, csize.p);
      for (int sweep = 0;; ++sweep) {
        SCL_CUDA(cudaMemsetAsync(moved.p, 0, G * sizeof(unsigned), st));
        for (uint32_t sub = 0; sub < 2; ++sub) {
          SCL_CUDA(cudaMemcpyAsync(comm_new.p, comm.p, n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
          k_move<<<sgrid, kWarps * 32, 0, st>>>(g, n, cp, comm.p, K.p, csize.p, deg.p, comm_new.p, inv2m, it, level, sweep, sub,
                                                moved.p, Ts);
          if (Tl.gslots)
            k_move<<<lgrid, kWarps * 32, 0, st>>>(g, n, cp, comm.p, K.p, csize.p, deg.p, comm_new.p, inv2m, it, level, sweep,
                                                  sub, moved.p, Tl);
          std::swap(comm.p, comm_new.p);
          SCL_CUDA(cudaMemsetAsync(K.p, 0, n * sizeof(ull), st));
          SCL_CUDA(cudaMemsetAsync(csize.p, 0, n * sizeof(uint32_t), st));
          k_totals<<<blocks(n, 256), 256, 0, st>>>(comm.p, deg.p, n, K.p, csize.p);
          count_launches(Tl.gslots ? 3 : 2);
        }
        SCL_CUDA(cudaGetLastError());
        to_host(hmoved, moved.p, G, st);
        bool any = false;
        for (int c = 0; c < G; ++c) {
          if (!lm[c]) continue;
          lvl_moved[c] += hmoved[c];
          if (hmoved[c] == 0) lm[c] = 0;
          else if (sweep + 1 >= max_sweeps) { lm[c] = 0; ++stats->capped_levels; }
          any |= lm[c] != 0;
        }
        if (!any) break;
        dev_bool(dact.p, lm);
      }
      dev_bool(dact.p, lvl_active);
      stats->t_move_ms += tm.stop();
      // (2) refinement
      k_expand<<<blocks(n, 256), 256, 0, st>>>(deg.p, n, n, Kr.p, ref.p, ref_new.p);   // singletons: ref = v
      for (uint32_t sub = 0; sub <= 2; ++sub) {
        SCL_CUDA(cudaMemsetAsync(Kr.p, 0, n * sizeof(ull), st));
        SCL_CUDA(cudaMemsetAsync(rsize.p, 0, n * sizeof(uint32_t), st));
        SCL_CUDA(cudaMemsetAsync(ext.p, 0, n * sizeof(ull), st));
        k_totals<<<blocks(n, 256), 256, 0, st>>>(ref.p, deg.p, n, Kr.p, rsize.p);
        k_ext<<<blocks(n, 128), 128, 0, st>>>(g, n, comm.p, ref.p, ext.p);
        if (sub == 2) break;
        SCL_CUDA(cudaMemcpyAsync(ref_new.p, ref.p, n * sizeof(uint32_t), cudaMemcpyDeviceToDevice, st));
        k_refine<<<sgrid, kWarps * 32, 0, st>>>(g, n, cp, comm.p, K.p, deg.p, ref.p, Kr.p, rsize.p, ext.p, ref_new.p, inv2m,
                                                ctheta, it, level, sub, Ts);
        if (Tl.gslots)
          k_refine<<<lgrid, kWarps * 32, 0, st>>>(g, n, cp, comm.p, K.p, deg.p, ref.p, Kr.p, rsize.p, ext.p, ref_new.p, inv2m,
                                                  ctheta, it, level, sub, Tl);
        std::swap(ref.p, ref_new.p);
        count_launches(Tl.gslots ? 5 : 4);
      }
      SCL_CUDA(cudaGetLastError());
      stats->t_refine_ms += tm.stop();
      // (3) which copies merged anything
      SCL_CUDA(cudaMemsetAsync(cnt.p, 0, G * sizeof(unsigned), st));
      k_live_count<<<blocks(n, 256), 256, 0, st>>>(g, n, rsize.p, cnt.p);
      to_host(hcnt, cnt.p, G, st);
      bool any = false;
      for (int c = 0; c < G; ++c) {
        finish[c] = 0;
        if (!lvl_active[c]) continue;
        const bool still = hcnt[c] == hvoff[c + 1] - hvoff[c] && lvl_moved[c] == 0;   // neither moved nor merged
        if (still || level + 1 >= kMaxLevels) { finish[c] = 1; lvl_active[c] = 0; }
        any |= lvl_active[c] != 0;
      }
      dev_bool(dfinish.p, finish);
      k_record<<<blocks(n0, 256), 256, 0, st>>>(map0.p, comm.p, voff.p, dfinish.p, N0, n0, fin.p);
      count_launches(2);
      if (!any) { stats->t_aggregate_ms += tm.stop(); break; }
      // (4) aggregation of the refined subsets of the copies that go on
      dev_bool(dact.p, lvl_active);
      k_live_flag<<<blocks(n, 256), 256, 0, st>>>(g, n, rsize.p, dact.p, flag.p);
      scan<uint32_t>(flag.p, nid.p, n, st);
      uint32_t nc = 0;
      SCL_CUDA(cudaMemcpyAsync(&nc, nid.p + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      // coarse copy offsets: nid at the old offsets
      std::vector<uint32_t> hnid_at(G + 1);
      for (int c = 0; c <= G; ++c)
        SCL_CUDA(cudaMemcpyAsync(&hnid_at[c], nid.p + hvoff[c], sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
      SCL_CUDA(cudaStreamSynchronize(st));
      SCL_CUDA(cudaMemsetAsync(cmin.p, 0xff, n * sizeof(uint32_t), st));
      SCL_CUDA(cudaMemsetAsync(mcnt.p, 0, (nc + 1) * sizeof(uint32_t), st));
      k_coarse_nodes<<<blocks(n, 256), 256, 0, st>>>(g, n, flag.p, nid.p, comm.p, Kr.p, rsize.p, copyA.p, cdeg.p, cmin.p, mcnt.p);
      k_coarse_comm<<<blocks(n, 256), 256, 0, st>>>(n, flag.p, nid.p, comm.p, cmin.p, ccomm.p);
      k_map0<<<blocks(n0, 256), 256, 0, st>>>(map0.p, ref.p, nid.p, dact.p, N0, n0);
      scan<uint32_t>(mcnt.p, mptr.p, nc, st);
      SCL_CUDA(cudaMemsetAsync(mcur.p, 0, std::max<uint32_t>(nc, 1) * sizeof(uint32_t), st));
      SCL_CUDA(cudaMemsetAsync(rbound.p, 0, std::max<uint32_t>(nc, 1) * sizeof(ull), st));
      k_members<<<blocks(n, 256), 256, 0, st>>>(g, n, dact.p, ref.p, nid.p, mptr.p, mcur.p, mem.p, rbound.p);
      SCL_CUDA(cudaMemsetAsync(misc.p, 0, 2 * sizeof(ull), st));
      k_bound_max<<<blocks(nc, 256), 256, 0, st>>>(rbound.p, nc, misc.p);
      to_host(hm, misc.p, 2, st);
      int agrid = 0;
      const Tables Ta = lt.get(hm[0], hm[1], &agrid);
      const int cgrid = std::max(1, std::min(blocks(nc, kWarps), sm_count() * 64));
      Tmp<ull> dcnt(nc + 1, st);
      auto* rpN = &(rpA.p == g.rp ? rpB : rpA);
      auto* colN = &(colA.p == g.col ? colB : colA);
      auto* wN = &(wA.p == g.w ? wB : wA);
      rpN->ensure(nc + 1);
      ull* rpn = reinterpret_cast<ull*>(rpN->p);
      k_coarse_rows<<<cgrid, kWarps * 32, 0, st>>>(g, nc, mptr.p, mem.p, rbound.p, ref.p, nid.p, 0, dcnt.p, nullptr, nullptr,
                                                  nullptr, Ts);
      if (Ta.gslots)
        k_coarse_rows<<<agrid, kWarps * 32, 0, st>>>(g, nc, mptr.p, mem.p, rbound.p, ref.p, nid.p, 0, dcnt.p, nullptr, nullptr,
                                                    nullptr, Ta);
      scan<ull>(dcnt.p, rpn, nc, st);
      ull nnzc = 0;
      SCL_CUDA(cudaMemcpyAsync(&nnzc, rpn + nc, sizeof(ull), cudaMemcpyDeviceToHost, st));
      SCL_CUDA(cudaStreamSynchronize(st));
      tcol.ensure(std::max<ull>(nnzc, 1));
      tw.ensure(std::max<ull>(nnzc, 1));
      colN->ensure(std::max<ull>(nnzc, 1));
      wN->ensure(std::max<ull>(nnzc, 1));
      auto* twp = reinterpret_cast<ull*>(tw.p);
      k_coarse_rows<<<cgrid, kWarps * 32, 0, st>>>(g, nc, mptr.p, mem.p, rbound.p, ref.p, nid.p, 1, dcnt.p, rpn, tcol.p, twp, Ts);
      if (Ta.gslots)
        k_coarse_rows<<<agrid, kWarps * 32, 0, st>>>(g, nc, mptr.p, mem.p, rbound.p, ref.p, nid.p, 1, dcnt.p, rpn, tcol.p, twp, Ta);
      k_rank_rows<<<std::max(1, std::min(blocks((size_t)nc * 32, 256), sm_count() * 32)), 256, 0, st>>>(
          nc, rpn, tcol.p, twp, colN->p, reinterpret_cast<ull*>(wN->p));
      count_launches(14);
      SCL_CUDA(cudaGetLastError());
      // the coarse level becomes the current one
      std::swap(comm.p, ccomm.p);
      std::swap(deg.p, cdeg.p);
      std::swap(copyA.p, ccopy.p);
      cur_copy = ccopy.p;
      for (int c = 0; c <= G; ++c) hvoff[c] = hnid_at[c];
      to_dev(cvoff.p, hvoff, st);
      std::swap(voff.p, cvoff.p);
      n = nc;
      g = LGraph{0, N0, nullptr, nullptr, nullptr, rpN->p, colN->p, wN->p, cur_copy, voff.p};
      stats->t_aggregate_ms += tm.stop();
    }
    // labels of this iteration
    to_host(hfin, fin.p, n0, st);
    for (int c = 0; c < G; ++c) {
      if (!it_active[c]) continue;
      int32_t* out = labels + (size_t)c * N0;
      nclu[c] = canonical(hfin.data() + (size_t)c * N0, c * N0, (int)N0, out, idbuf, sizes);
      if (std::equal(out, out + N0, prev.data() + (size_t)c * N0)) it_active[c] = 0;
      else std::copy(out, out + N0, prev.data() + (size_t)c * N0);
    }
    stats->t_labels_ms += tm.stop();
  }
  // modularity on the original graph: sum_c [w_in(c) - gamma K_c^2 / 2m] / 2m
  Tmp<ull> win(G, st);
  SCL_CUDA(cudaMemsetAsync(win.p, 0, G * sizeof(ull), st));
  k_win<<<blocks(n0, 256), 256, 0, st>>>(gr.rp.p, gr.col.p, gr.w.p, fin.p, N0, n0, win.p);
  count_launches(1);
  std::vector<ull> hwin;
  std::vector<uint64_t> hdeg;
  to_host(hwin, win.p, G, st);
  to_host(hdeg, gr.deg.p, N0, st);
  std::vector<uint64_t> Kc;
  for (int c = 0; c < G; ++c) {
    const int32_t* l = labels + (size_t)c * N0;
    Kc.assign(nclu[c], 0);
    for (uint32_t i = 0; i < N0; ++i) Kc[l[i]] += hdeg[i];
    double s = 0;
    for (uint64_t x : Kc) { const double f = (double)x * inv2m; s += f * f; }
    modularity[c] = (double)hwin[c] * inv2m - hg[c] * s;
  }
  stats->t_labels_ms += tm.stop();
}

void leiden_batched(const FixGraph& g, const double* gammas, int R, int T, uint64_t seed, int max_iterations, int max_sweeps,
                    double theta, int32_t* labels, int32_t* nclu, double* modularity, LeidenStats* stats, cudaStream_t st) {
  // a trial's labels do not depend on its batch, so a batch larger than kBatchVertices copies x vertices runs in chunks:
  // whole resolutions when T x N fits, else chunks of trials of one resolution
  const int64_t N = g.N;
  SCL_REQUIRE(N < kBatchVertices, "leiden: N must stay below 2^27");
  *stats = LeidenStats{};
  auto add = [&](const LeidenStats& s) {
    stats->max_levels = std::max(stats->max_levels, s.max_levels);
    stats->max_iterations = std::max(stats->max_iterations, s.max_iterations);
    stats->capped_levels += s.capped_levels;
    stats->copy_levels += s.copy_levels;
    stats->t_move_ms += s.t_move_ms; stats->t_refine_ms += s.t_refine_ms;
    stats->t_aggregate_ms += s.t_aggregate_ms; stats->t_labels_ms += s.t_labels_ms;
  };
  LeidenStats s;
  if ((int64_t)T * N <= kBatchVertices) {
    const int rc = (int)std::max<int64_t>(1, kBatchVertices / ((int64_t)T * N));
    for (int r0 = 0; r0 < R; r0 += rc) {
      const int nr = std::min(rc, R - r0);
      const size_t o = (size_t)r0 * T;
      leiden_run(g, gammas + r0, nr, T, 0, seed, max_iterations, max_sweeps, theta, labels + o * N, nclu + o, modularity + o, &s, st);
      add(s);
    }
    return;
  }
  const int tc = (int)(kBatchVertices / N);
  for (int r = 0; r < R; ++r)
    for (int t0 = 0; t0 < T; t0 += tc) {
      const int nt = std::min(tc, T - t0);
      const size_t o = (size_t)r * T + t0;
      leiden_run(g, gammas + r, 1, nt, t0, seed, max_iterations, max_sweeps, theta, labels + o * N, nclu + o, modularity + o, &s, st);
      add(s);
    }
}

void label_ecs(const int32_t* labels, int T, int N, double* S, cudaStream_t st) {
  std::vector<int> kk(T), soff(T + 1, 0), sz;
  for (int t = 0; t < T; ++t) {
    int k = 0;
    for (int i = 0; i < N; ++i) {
      const int32_t l = labels[(size_t)t * N + i];
      SCL_REQUIRE(l >= 0 && l < N, "label_ecs: labels must lie in [0, N)");
      k = std::max(k, l + 1);
    }
    kk[t] = k;
    soff[t + 1] = soff[t] + k;
  }
  sz.assign(soff[T], 0);
  for (int t = 0; t < T; ++t)
    for (int i = 0; i < N; ++i) ++sz[soff[t] + labels[(size_t)t * N + i]];
  std::vector<int2> pairs;
  for (int a = 0; a < T; ++a)
    for (int b = a + 1; b < T; ++b) pairs.push_back(int2{a, b});
  for (int a = 0; a < T; ++a) S[(size_t)a * T + a] = 1.0;
  if (pairs.empty()) return;
  Tmp<int32_t> dl((size_t)T * N, st);
  Tmp<int> dk(T, st), doff(T + 1, st), dsz(std::max<size_t>(sz.size(), 1), st);
  Tmp<int2> dp(pairs.size(), st);
  Tmp<double> dout(pairs.size(), st);
  SCL_CUDA(cudaMemcpyAsync(dl.p, labels, (size_t)T * N * sizeof(int32_t), cudaMemcpyHostToDevice, st));
  to_dev(dk.p, kk, st);
  to_dev(doff.p, soff, st);
  to_dev(dsz.p, sz, st);
  to_dev(dp.p, pairs, st);
  bool big = false;
  for (const int2& p : pairs) big |= (size_t)kk[p.x] * kk[p.y] > (size_t)kEcsSmem;
  uint32_t gslots = 0;
  if (big) { gslots = 32; while (gslots < 2u * (uint32_t)N) gslots <<= 1; }
  const size_t chunk = big ? std::max<size_t>(1, std::min(pairs.size(), ((size_t)1 << 26) / gslots)) : pairs.size();
  Tmp<unsigned long long> gkey(big ? chunk * gslots : 1, st);
  Tmp<uint32_t> gcnt(big ? chunk * gslots : 1, st);
  for (size_t p0 = 0; p0 < pairs.size(); p0 += chunk) {
    const int nb = (int)std::min(chunk, pairs.size() - p0);
    k_ecs<<<nb, kEcsThreads, 0, st>>>(dl.p, N, dk.p, doff.p, dsz.p, dp.p, (int)p0, gkey.p, gcnt.p, gslots, dout.p);
    count_launches(1);
  }
  SCL_CUDA(cudaGetLastError());
  std::vector<double> h;
  to_host(h, dout.p, pairs.size(), st);
  for (size_t q = 0; q < pairs.size(); ++q) S[(size_t)pairs[q].x * T + pairs[q].y] = S[(size_t)pairs[q].y * T + pairs[q].x] = h[q];
}

std::vector<double> cluster_plan(const std::vector<double>& gam, const std::vector<int>& mode, int k_min, int k_max,
                                 double lo_limit, double hi_limit) {
  std::vector<double> out;
  if (gam.empty()) return out;
  std::vector<size_t> ord(gam.size());
  std::iota(ord.begin(), ord.end(), 0);
  std::sort(ord.begin(), ord.end(), [&](size_t a, size_t b) { return gam[a] < gam[b]; });
  const double g_lo = gam[ord.front()], g_hi = gam[ord.back()];
  // widen while an end of the target range is not bracketed
  if (mode[ord.front()] > k_min && g_lo / 10 >= lo_limit * (1 - 1e-9)) out.push_back(g_lo / 10);
  if (mode[ord.back()] < k_max && g_hi * 10 <= hi_limit * (1 + 1e-9)) out.push_back(g_hi * 10);
  for (int k = k_min; k <= k_max; ++k) {
    bool found = false;
    double lo = -1;
    for (size_t i : ord) {
      if (mode[i] == k) found = true;
      if (mode[i] < k) lo = gam[i];
    }
    if (found || lo < 0) continue;
    double hi = -1;
    for (size_t i : ord)
      if (gam[i] > lo && mode[i] > k) { hi = gam[i]; break; }
    if (hi < 0 || hi <= lo * (1 + 1e-9)) continue;
    out.push_back(std::sqrt(lo * hi));
  }
  std::sort(out.begin(), out.end());
  out.erase(std::unique(out.begin(), out.end()), out.end());
  return out;
}

}  // namespace scl
