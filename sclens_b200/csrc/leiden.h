// Device Leiden, label similarity and the resolution search (leiden.cu).
#pragma once
#include <vector>
#include "common.cuh"

namespace scl {

// A graph in the exact integer form every Leiden kernel reads: symmetric CSR, sorted columns, weights round(w 2^shift).
struct FixGraph {
  int N = 0;
  size_t nnz = 0;
  int shift = 0;
  uint64_t two_m = 0;
  DBuf<uint32_t> rp, col;
  DBuf<uint64_t> w, deg;
};

// Validate (on the device) and convert a CSR; val_f64 or val_f32 (exactly one non-null) are device pointers, as are rp /
// col.  Throws Error(SCL_ERR_GRAPH) for a graph that is not a symmetric CSR with sorted columns and finite positive weights.
void leiden_prepare(const uint32_t* rp, const uint32_t* col, const double* val_f64, const float* val_f32, int N, size_t nnz,
                    FixGraph& g, cudaStream_t st);

// Fixed-point exponent of a graph: the largest s <= 32 with nnz * maxw * 2^s < 2^61, so 2m < 2^62 after rounding.
int leiden_weight_shift(double maxw, size_t nnz);
// Key of trial t: every draw of the trial hashes it (stream 6 of umap_stream_key).
uint64_t leiden_copy_key(uint64_t seed, uint32_t trial);

struct LeidenStats {
  int max_levels = 0, max_iterations = 0, capped_levels = 0;
  int64_t copy_levels = 0;
  double t_move_ms = 0, t_refine_ms = 0, t_aggregate_ms = 0, t_labels_ms = 0;
};

// R resolutions x T trials (trial t uses the draws of trial t0 + t).  labels [R][T][N] (cluster ids by size, descending),
// nclu [R T], modularity [R T] on host.
void leiden_run(const FixGraph& g, const double* gammas, int R, int T, int t0, uint64_t seed, int max_iterations,
                int max_sweeps, double theta, int32_t* labels, int32_t* nclu, double* modularity, LeidenStats* stats,
                cudaStream_t st);

// leiden_run over a batch of any size, in chunks of at most 2^27 copies x vertices (identical results: a trial's labels do
// not depend on its batch).
void leiden_batched(const FixGraph& g, const double* gammas, int R, int T, uint64_t seed, int max_iterations, int max_sweeps,
                    double theta, int32_t* labels, int32_t* nclu, double* modularity, LeidenStats* stats, cudaStream_t st);

// T x T ECS matrix (row-major) of T labelings [T][N] with ids 0..k_t - 1.
void label_ecs(const int32_t* labels, int T, int N, double* S, cudaStream_t st);

// Next resolutions of the search from the (gamma, modal count) pairs evaluated so far; empty when done.
std::vector<double> cluster_plan(const std::vector<double>& gam, const std::vector<int>& mode, int k_min, int k_max,
                                 double lo_limit, double hi_limit);

}  // namespace scl
