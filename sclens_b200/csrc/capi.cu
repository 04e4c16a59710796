// extern "C" surface of libsclens_b200.so (see include/sclens_b200.h).
#include "nccl_dyn.h"
#include <chrono>
#include <cmath>
#include <cstring>
#include <thread>
#include "handle.h"
#include "tmp.cuh"
#include "twostage.h"

using namespace scl;

namespace {
thread_local std::string g_create_error;

template <typename F>
int32_t guard(scl_handle* h, F&& f) {
  try {
    f();
    return SCL_OK;
  } catch (const scl::Error& e) {
    if (h) h->err = e.what(); else g_create_error = e.what();
    return e.code;
  } catch (const std::exception& e) {
    if (h) h->err = e.what(); else g_create_error = e.what();
    return SCL_ERR_INVALID;
  }
}

void upload_u32(DBuf<uint32_t>& dst, const uint32_t* src, size_t n, int base, cudaStream_t st) {
  dst.ensure(n ? n : 1);
  if (!n) return;
  if (base == 0) {
    SCL_CUDA(cudaMemcpyAsync(dst.p, src, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
  } else {
    std::vector<uint32_t> tmp(src, src + n);
    for (auto& v : tmp) v -= (uint32_t)base;
    SCL_CUDA(cudaMemcpyAsync(dst.p, tmp.data(), n * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    SCL_CUDA(cudaStreamSynchronize(st));
  }
}

void download_csc(const SpMat& A, uint32_t* colptr, uint32_t* rowval, float* val, cudaStream_t st) {
  SCL_CUDA(cudaMemcpyAsync(colptr, A.colptr.p, (A.M + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
  if (A.nnz) {
    SCL_CUDA(cudaMemcpyAsync(rowval, A.rowval.p, A.nnz * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaMemcpyAsync(val, A.val.p, A.nnz * sizeof(float), cudaMemcpyDeviceToHost, st));
  }
  SCL_CUDA(cudaStreamSynchronize(st));
}
}  // namespace

extern "C" {

int32_t scl_version(void) { return 100; }

int32_t scl_create(scl_handle** out, const scl_config* cfg) {
  if (!out) return SCL_ERR_INVALID;
  *out = nullptr;
  scl_handle* h = nullptr;
  int32_t rc = guard(nullptr, [&] {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) throw Error(SCL_ERR_NOGPU, "no CUDA device: libsclens_b200 has no CPU fallback");
    scl_config c{};
    if (cfg) c = *cfg;
    SCL_REQUIRE(c.device >= 0 && c.device < ndev, "bad device ordinal");
    SCL_CUDA(cudaSetDevice(c.device));
    cudaDeviceProp prop;
    SCL_CUDA(cudaGetDeviceProperties(&prop, c.device));
    if (prop.major != 10) throw Error(SCL_ERR_NOGPU, std::string("sm_100 (B200) required, found sm_") + std::to_string(prop.major * 10 + prop.minor));
    h = new scl_handle;
    h->cfg = c;
    SCL_CUDA(cudaStreamCreateWithFlags(&h->st, cudaStreamNonBlocking));
    cudaMemPool_t pool;
    SCL_CUDA(cudaDeviceGetDefaultMemPool(&pool, c.device));
    uint64_t thr = UINT64_MAX;
    SCL_CUDA(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr));
    h->solver.reset(new Solver(h->st));
  });
  if (rc != SCL_OK) {
    delete h;
    return rc;
  }
  *out = h;
  return SCL_OK;
}

int32_t scl_destroy(scl_handle* h) {
  if (!h) return SCL_OK;
  cudaSetDevice(h->cfg.device);
  if (h->st) cudaStreamSynchronize(h->st);
  if (h->nccl) nccl_api().CommDestroy((ncclComm_t)h->nccl);
  h->prof.resolve();
  if (h->t0) { cudaEventDestroy(h->t0); cudaEventDestroy(h->t1); }
  h->solver.reset();
  if (h->st) cudaStreamDestroy(h->st);
  delete h;
  return SCL_OK;
}

const char* scl_last_error(scl_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int32_t scl_get_profile(scl_handle* h, scl_profile* out) {
  if (!h || !out) return SCL_ERR_INVALID;
  h->prof.resolve();
  const Prof& p = h->prof;
  out->gram_gemm_ms = p.ms[PK_GRAM_GEMM]; out->other_gemm_ms = p.ms[PK_OTHER_GEMM]; out->densify_ms = p.ms[PK_DENSIFY];
  out->stats_ms = p.ms[PK_STATS]; out->sparse_ms = p.ms[PK_SPARSE]; out->syevd_ms = p.ms[PK_SYEVD];
  out->gram_gemm_launches = p.calls[PK_GRAM_GEMM]; out->other_gemm_launches = p.calls[PK_OTHER_GEMM];
  out->densify_launches = p.calls[PK_DENSIFY]; out->sparse_calls = p.calls[PK_SPARSE]; out->syevd_calls = p.calls[PK_SYEVD];
  out->gram_alg_flops = p.gram_alg_flops; out->other_gemm_flops = p.other_gemm_flops;
  out->densify_alg_bytes = p.densify_alg_bytes; out->sparse_alg_bytes = p.sparse_alg_bytes;
  out->kernel_launches = g_kernel_launches.load();
  out->refine_ms = p.ms[PK_REFINE];
  out->small_ms = p.ms[PK_SMALL];
  out->stats_alg_bytes = p.stats_alg_bytes;
  out->stats_calls = p.stats_norms;
  out->comm_ms = p.ms[PK_COMM];
  out->comm_bytes = p.comm_bytes;
  return SCL_OK;
}

int32_t scl_reset_profile(scl_handle* h) {
  if (!h) return SCL_ERR_INVALID;
  h->prof.reset();
  if (h->solver) for (double& v : h->solver->ts_total) v = 0.0;
  return SCL_OK;
}

int32_t scl_timer_start(scl_handle* h) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    if (!h->t0) { SCL_CUDA(cudaEventCreate(&h->t0)); SCL_CUDA(cudaEventCreate(&h->t1)); }
    SCL_CUDA(cudaStreamSynchronize(h->st));
    SCL_CUDA(cudaEventRecord(h->t0, h->st));
  });
}

int32_t scl_timer_stop(scl_handle* h, double* ms) {
  if (!h || !ms || !h->t0) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaEventRecord(h->t1, h->st));
    SCL_CUDA(cudaEventSynchronize(h->t1));
    float t = 0;
    SCL_CUDA(cudaEventElapsedTime(&t, h->t0, h->t1));
    *ms = t;
  });
}

// ---- multi-GPU plumbing -----------------------------------------------------------------
int32_t scl_nccl_unique_id(uint8_t out_id[128]) {
  static_assert(sizeof(ncclUniqueId) == 128, "ncclUniqueId size");
  ncclUniqueId id;
  try {
    if (nccl_api().GetUniqueId(&id) != ncclSuccess) return SCL_ERR_NCCL;
  } catch (const Error&) {
    return SCL_ERR_NCCL;
  }
  std::memcpy(out_id, &id, 128);
  return SCL_OK;
}

int32_t scl_comm_init(scl_handle* h, const uint8_t id[128], int32_t rank, int32_t world) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(world >= 1 && rank >= 0 && rank < world, "bad rank/world");
    if (h->nccl && h->world == world && h->rank == rank) return;   // already this rank of this world: keep the communicator
    if (h->nccl) {                                                 // a different world: the old communicator goes first
      nccl_api().CommDestroy((ncclComm_t)h->nccl);
      h->nccl = nullptr;
    }
    h->world = world;
    h->rank = rank;
    if (world == 1) return;
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    ncclUniqueId uid;
    std::memcpy(&uid, id, 128);
    ncclComm_t comm;
    ncclResult_t r = nccl_api().CommInitRank(&comm, world, uid, rank);
    if (r != ncclSuccess) throw Error(SCL_ERR_NCCL, std::string("ncclCommInitRank: ") + nccl_api().GetErrorString(r));
    h->nccl = comm;
  });
}

int32_t scl_plan_replicates(int32_t n_perturb, int32_t world, int32_t rank, int32_t* out_ids, int32_t* out_n) {
  if (n_perturb < 0 || world < 1 || rank < 0 || rank >= world || !out_n) return SCL_ERR_INVALID;
  int n = 0;
  for (int r = rank; r < n_perturb; r += world) {
    if (out_ids) out_ids[n] = r;
    ++n;
  }
  *out_n = n;
  return SCL_OK;
}

int32_t scl_plan_search_wave(int32_t wave, int32_t world, int32_t rank, int32_t* out_step) {
  if (wave < 0 || world < 1 || rank < 0 || rank >= world || !out_step) return SCL_ERR_INVALID;
  *out_step = wave * world + rank;
  return SCL_OK;
}

int32_t scl_plan_pass_task(int32_t wave, int32_t world, int32_t rank, int32_t* out_task, int32_t* out_search_step) {
  if (wave < 0 || world < 1 || rank < 0 || rank >= world || !out_task) return SCL_ERR_INVALID;
  *out_task = wave * world + rank;
  if (out_search_step) *out_search_step = scl::pass_task_step(*out_task, scl::pass_refine_task(world));
  return SCL_OK;
}

int32_t scl_plan_gram_shard(int64_t K, int32_t world, int32_t rank, int64_t* out_k0, int64_t* out_k1) {
  if (K < 1 || world < 1 || rank < 0 || rank >= world || !out_k0 || !out_k1) return SCL_ERR_INVALID;
  scl::plan_gram_shard(K, (K + 7) / 8 * 8, world, rank, out_k0, out_k1);
  return SCL_OK;
}

// ---- inputs -------------------------------------------------------------------------------
int32_t scl_set_counts_csc(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr,
                           const uint32_t* rowval, const float* nzval, int32_t index_base) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(N > 1 && M > 1 && nnz > 0 && colptr && rowval && nzval, "bad CSC input");
    SCL_REQUIRE(index_base == 0 || index_base == 1, "index_base must be 0 or 1");
    SCL_REQUIRE((int64_t)colptr[M] - index_base == nnz, "colptr[M] does not match nnz");
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    upload_csc(h->X, N, M, (size_t)nnz, colptr, rowval, nzval, index_base, h->st);
    SCL_CUDA(cudaStreamSynchronize(h->st));
    h->have_X = true;
    h->signal_done = h->robust_done = false;
    h->have_zc = h->have_null_draws = h->have_pth = false;
    h->search_sples.clear();
    h->perturb_sples.clear();
  });
}

int32_t scl_set_zero_candidates(scl_handle* h, int64_t n, const uint32_t* z1, const uint32_t* z2, int32_t index_base) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_X && n >= 0 && (n == 0 || (z1 && z2)), "bad zero candidates");
    SCL_REQUIRE(index_base == 0 || index_base == 1, "index_base must be 0 or 1");
    for (int64_t t = 0; t < n; ++t)   // the merge kernels index lines with them
      SCL_REQUIRE(z1[t] - (uint32_t)index_base < (uint32_t)h->X.N && z2[t] - (uint32_t)index_base < (uint32_t)h->X.M,
                  "zero candidate outside the N x M grid");
    upload_u32(h->z1, z1, (size_t)n, index_base, h->st);
    upload_u32(h->z2, z2, (size_t)n, index_base, h->st);
    SCL_CUDA(cudaStreamSynchronize(h->st));
    h->n_cand = (size_t)n;
    h->have_zc = true;
  });
}

int32_t scl_set_null_draws(scl_handle* h, int64_t n, const uint32_t* perm, const uint32_t* rows, int32_t index_base) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_X && (size_t)n == h->X.nnz && perm && rows, "null draws must have length nnz");
    upload_u32(h->null_perm, perm, (size_t)n, index_base, h->st);
    upload_u32(h->null_rows, rows, (size_t)n, index_base, h->st);
    SCL_CUDA(cudaStreamSynchronize(h->st));
    h->have_null_draws = true;
  });
}

int32_t scl_set_noise_baseline(scl_handle* h, double p_th) {
  if (!h || !(p_th > 0)) return SCL_ERR_INVALID;
  h->p_th = p_th;
  h->have_pth = true;
  return SCL_OK;
}

static int32_t push_sample(scl_handle* h, int which, int64_t n, const uint32_t* s, int32_t base) {
  if (!h || n < 0 || (n > 0 && !s) || (base != 0 && base != 1)) return SCL_ERR_INVALID;
  std::vector<std::vector<uint32_t>>& q = which == 0 ? h->search_sples : h->perturb_sples;
  std::vector<uint32_t> v(s, s + n);
  if (base)
    for (auto& x : v) x -= (uint32_t)base;
  q.push_back(std::move(v));
  return SCL_OK;
}
int32_t scl_push_search_sample(scl_handle* h, int64_t n, const uint32_t* s, int32_t base) {
  return push_sample(h, 0, n, s, base);
}
int32_t scl_push_perturb_sample(scl_handle* h, int64_t n, const uint32_t* s, int32_t base) {
  return push_sample(h, 1, n, s, base);
}
int32_t scl_clear_draws(scl_handle* h) {
  if (!h) return SCL_ERR_INVALID;
  h->have_zc = h->have_null_draws = h->have_pth = false;
  h->search_sples.clear();
  h->perturb_sples.clear();
  return SCL_OK;
}

// ---- the path -----------------------------------------------------------------------------
int32_t scl_run_signal(scl_handle* h, scl_signal_info* out) {
  if (!h) return SCL_ERR_INVALID;
  int32_t rc = guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    run_signal(h);
  });
  if (rc == SCL_OK && out) *out = h->sinfo;
  return rc;
}

int32_t scl_run_robustness(scl_handle* h, double th, double p_step, int32_t n_perturb, scl_robust_info* out) {
  if (!h) return SCL_ERR_INVALID;
  int32_t rc = guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    run_robustness(h, th, p_step, n_perturb);
  });
  if (rc == SCL_OK && out) *out = h->rinfo;
  return rc;
}

int32_t scl_op_preprocess(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr, const uint32_t* rowval,
                          const float* nzval, int32_t index_base, const uint8_t* gene_flags, const scl_qc_params* p,
                          int32_t* n_cells, int32_t* n_genes, int64_t* out_nnz, int32_t* fc_idx, int32_t* gene_idx) {
  if (!h || !colptr || !rowval || !nzval || !gene_flags || !p || !n_cells || !n_genes || N < 1 || M < 1 || nnz < 1) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    SpMat raw;
    upload_csc(raw, N, M, (size_t)nnz, colptr, rowval, nzval, index_base, h->st);
    Tmp<uint8_t> flags(M, h->st);
    SCL_CUDA(cudaMemcpyAsync(flags.p, gene_flags, (size_t)M, cudaMemcpyHostToDevice, h->st));
    std::vector<int32_t> fc, gi;
    SpMat out;
    const bool any = preprocess_device(raw, flags.p, *p, fc, gi, out, h->st);
    *n_cells = any ? out.N : 0;
    *n_genes = any ? out.M : 0;
    if (out_nnz) *out_nnz = any ? (int64_t)out.nnz : 0;
    if (!any) return;
    if (fc_idx) std::memcpy(fc_idx, fc.data(), fc.size() * sizeof(int32_t));
    if (gene_idx) std::memcpy(gene_idx, gi.data(), gi.size() * sizeof(int32_t));
    h->X.swap(out);
    h->have_X = true;
    h->signal_done = h->robust_done = false;
    h->have_zc = h->have_null_draws = h->have_pth = false;
    h->search_sples.clear();
    h->perturb_sples.clear();
  });
}

int32_t scl_get_counts_csc(scl_handle* h, uint32_t* colptr, uint32_t* rowval, float* nzval) {
  if (!h || !colptr || !rowval || !nzval) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_X, "no counts on the handle");
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    download_csc(h->X, colptr, rowval, nzval, h->st);
  });
}

int32_t scl_run_pass(scl_handle* h, double th, double p_step, int32_t n_perturb, scl_signal_info* sout, scl_robust_info* rout) {
  if (!h) return SCL_ERR_INVALID;
  int32_t rc = guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    run_pass(h, th, p_step, n_perturb);
  });
  if (rc == SCL_OK && sout) *sout = h->sinfo;
  if (rc == SCL_OK && rout) *rout = h->rinfo;
  return rc;
}

// ---- results ------------------------------------------------------------------------------
#define NEED_SIGNAL() SCL_REQUIRE(h->signal_done, "scl_run_signal has not completed")
#define NEED_ROBUST() SCL_REQUIRE(h->robust_done, "scl_run_robustness has not completed")

int32_t scl_get_L(scl_handle* h, float* L) {
  if (!h || !L) return SCL_ERR_INVALID;
  return guard(h, [&] { NEED_SIGNAL(); std::memcpy(L, h->L.data(), h->L.size() * sizeof(float)); });
}
int32_t scl_get_Lmp(scl_handle* h, float* L) {
  if (!h || !L) return SCL_ERR_INVALID;
  return guard(h, [&] { NEED_SIGNAL(); std::memcpy(L, h->Lmp.data(), h->Lmp.size() * sizeof(float)); });
}
int32_t scl_get_signal_ev(scl_handle* h, float* nL) {
  if (!h || !nL) return SCL_ERR_INVALID;
  return guard(h, [&] { NEED_SIGNAL(); std::memcpy(nL, h->nL.data(), h->nL.size() * sizeof(float)); });
}
int32_t scl_get_signal_evec(scl_handle* h, float* nV) {
  if (!h || !nV) return SCL_ERR_INVALID;
  return guard(h, [&] {
    NEED_SIGNAL();
    size_t n = (size_t)h->sinfo.n_signal * h->sinfo.N;
    if (n) SCL_CUDA(cudaMemcpy(nV, h->d_nV.p, n * sizeof(float), cudaMemcpyDeviceToHost));
  });
}
int32_t scl_get_gene_basis(scl_handle* h, float* g) {
  if (!h || !g) return SCL_ERR_INVALID;
  return guard(h, [&] { NEED_ROBUST(); std::memcpy(g, h->gene_basis.data(), h->gene_basis.size() * sizeof(float)); });
}
int32_t scl_get_rec_vals(scl_handle* h, double* TGC, double* mean, double* sd, double* norm_tgc, double* cent) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    NEED_SIGNAL();
    if (TGC) std::memcpy(TGC, h->rec_tgc.data(), h->rec_tgc.size() * sizeof(double));
    if (mean) std::memcpy(mean, h->rec_mean.data(), h->rec_mean.size() * sizeof(double));
    if (sd) std::memcpy(sd, h->rec_std.data(), h->rec_std.size() * sizeof(double));
    if (norm_tgc) std::memcpy(norm_tgc, h->rec_l2.data(), h->rec_l2.size() * sizeof(double));
    if (cent) std::memcpy(cent, h->rec_cent.data(), h->rec_cent.size() * sizeof(double));
  });
}
int32_t scl_get_scores(scl_handle* h, float* b_, double* m, double* sd) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    NEED_ROBUST();
    if (b_) std::memcpy(b_, h->b_.data(), h->b_.size() * sizeof(float));
    if (m) std::memcpy(m, h->m_scores.data(), h->m_scores.size() * sizeof(double));
    if (sd) std::memcpy(sd, h->sd_scores.data(), h->sd_scores.size() * sizeof(double));
  });
}
int32_t scl_get_sig_id(scl_handle* h, int32_t* sig) {
  if (!h || !sig) return SCL_ERR_INVALID;
  return guard(h, [&] { NEED_ROBUST(); std::memcpy(sig, h->sig_id.data(), h->sig_id.size() * sizeof(int32_t)); });
}
int32_t scl_get_null_csc(scl_handle* h, int64_t* nnz, uint32_t* colptr, uint32_t* rowval, float* nzval) {
  if (!h || !nnz) return SCL_ERR_INVALID;
  return guard(h, [&] {
    NEED_SIGNAL();
    *nnz = (int64_t)h->Xnull.nnz;
    if (colptr && rowval && nzval) download_csc(h->Xnull, colptr, rowval, nzval, h->st);
  });
}
int32_t scl_get_search_trace(scl_handle* h, double* p, double* d) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    NEED_ROBUST();
    if (p) std::memcpy(p, h->trace_p.data(), h->trace_p.size() * sizeof(double));
    if (d) std::memcpy(d, h->trace_d.data(), h->trace_d.size() * sizeof(double));
  });
}
int32_t scl_get_perturbed_evec(scl_handle* h, int32_t r, float* nV, float* nL) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    NEED_ROBUST();
    SCL_REQUIRE(r >= 0 && r < h->rinfo.n_perturb, "replicate out of range");
    const size_t per = (size_t)h->rinfo.min_pc * h->sinfo.N;
    if (nV) SCL_CUDA(cudaMemcpy(nV, h->d_sets.p + (size_t)r * per, per * sizeof(float), cudaMemcpyDeviceToHost));
    if (nL) std::memcpy(nL, &h->set_L[(size_t)r * h->rinfo.min_pc], h->rinfo.min_pc * sizeof(float));
  });
}

// ---- function-level operators ---------------------------------------------------------------
int32_t scl_op_normalize(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr,
                         const uint32_t* rowval, const float* nzval, int32_t layout, int64_t ld, uint16_t* out_hi,
                         uint16_t* out_lo, double* TGC, double* mean, double* sd, double* norm_tgc, double* cent) {
  if (!h) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    SpMat A;
    NormStats S;
    S.centering = h->cfg.centering;
    upload_csc(A, N, M, (size_t)nnz, colptr, rowval, nzval, 0, h->st);
    compute_norm_stats(A, S, h->st);
    if (out_hi) {
      const size_t lines = layout == 1 ? N : M;
      Tmp<__half> hi(lines * (size_t)ld, h->st), lo(lines * (size_t)ld, h->st);
      densify(A, S, layout, (size_t)ld, hi.p, out_lo ? lo.p : nullptr, h->st);
      SCL_CUDA(cudaMemcpyAsync(out_hi, hi.p, lines * (size_t)ld * 2, cudaMemcpyDeviceToHost, h->st));
      if (out_lo) SCL_CUDA(cudaMemcpyAsync(out_lo, lo.p, lines * (size_t)ld * 2, cudaMemcpyDeviceToHost, h->st));
      SCL_CUDA(cudaStreamSynchronize(h->st));
    }
    auto dl = [&](double* dst, const double* src, size_t n) {
      if (dst) SCL_CUDA(cudaMemcpyAsync(dst, src, n * sizeof(double), cudaMemcpyDeviceToHost, h->st));
    };
    dl(TGC, S.tgc.p, N); dl(norm_tgc, S.l2.p, N); dl(mean, S.ybar.p, M); dl(sd, S.sigma.p, M); dl(cent, S.cent.p, M);
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_gram(scl_handle* h, int32_t rows, int64_t K, int64_t ld, const uint16_t* a_hi, const uint16_t* a_lo,
                    float scale, float* G) {
  if (!h || !a_hi || !G) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    const size_t n = (size_t)rows * (size_t)ld;
    Tmp<__half> hi(n, h->st), lo(n, h->st);
    Tmp<float> g((size_t)rows * rows, h->st);
    SCL_CUDA(cudaMemcpyAsync(hi.p, a_hi, n * 2, cudaMemcpyHostToDevice, h->st));
    if (a_lo) SCL_CUDA(cudaMemcpyAsync(lo.p, a_lo, n * 2, cudaMemcpyHostToDevice, h->st));
    GemmArgs a;
    a.A.hi = hi.p; a.A.lo = a_lo ? lo.p : nullptr; a.A.rows = rows; a.A.K = K; a.A.ld = ld;
    a.B = a.A;
    a.syrk = true; a.alpha = scale; a.C = g.p; a.ldc = rows;
    a.cta_group = h->cfg.cta_group == 1 ? 1 : 2;
    a.chunk_kb = h->cfg.gram_chunk_kb;
    gemm_umma(a, h->st);
    SCL_CUDA(cudaMemcpyAsync(G, g.p, (size_t)rows * rows * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

/* Kernel-level timing on device-resident synthetic operands (bench / ncu harness; no host data moves).
 * mode bit0: split (hi+lo) operands; bit1: plain GEMM A*B^T instead of the syrk schedule. */
int32_t scl_bench_gram(scl_handle* h, int32_t rows, int64_t K, int32_t mode, int32_t chunk_kb, int32_t reps,
                       double* ms_avg, double* checksum) {
  if (!h || rows <= 0 || K <= 0 || reps <= 0) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    const int64_t ld = (K + 7) / 8 * 8;
    const size_t n = (size_t)rows * (size_t)ld;
    const bool split = mode & 1;
    Tmp<__half> hi(n, h->st), lo(split ? n : 1, h->st);
    Tmp<float> g((size_t)rows * rows, h->st);
    fill_random_f16(hi.p, n, 0x1234u, 1.0f, h->st);
    if (split) fill_random_f16(lo.p, n, 0x9876u, 1.0f / 2048.f, h->st);
    GemmArgs a;
    a.A.hi = hi.p; a.A.lo = split ? lo.p : nullptr; a.A.rows = rows; a.A.K = K; a.A.ld = ld;
    a.B = a.A;
    a.syrk = !(mode & 2); a.alpha = 1.0f / (float)K; a.C = g.p; a.ldc = rows;
    a.cta_group = h->cfg.cta_group == 1 ? 1 : 2;
    a.chunk_kb = chunk_kb;
    gemm_umma(a, h->st);   // warm-up
    cudaEvent_t e0, e1;
    SCL_CUDA(cudaEventCreate(&e0));
    SCL_CUDA(cudaEventCreate(&e1));
    SCL_CUDA(cudaEventRecord(e0, h->st));
    for (int r = 0; r < reps; ++r) gemm_umma(a, h->st);
    SCL_CUDA(cudaEventRecord(e1, h->st));
    SCL_CUDA(cudaEventSynchronize(e1));
    float ms = 0;
    SCL_CUDA(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    if (ms_avg) *ms_avg = ms / reps;
    if (checksum) {
      std::vector<float> d(rows);
      SCL_CUDA(cudaMemcpy2DAsync(d.data(), sizeof(float), g.p, (size_t)(rows + 1) * sizeof(float), sizeof(float), rows,
                                 cudaMemcpyDeviceToHost, h->st));
      SCL_CUDA(cudaStreamSynchronize(h->st));
      double t = 0;
      for (float v : d) t += v;
      *checksum = t / rows;   // mean diagonal: ~E[x^2] of the synthetic operand
    }
  });
}

/* Times the normalisation kernels on the handle's counts: the statistics pre-passes and the fused densify writer
 * (layout 0 gene-major / 1 cell-major, with_lo: also emit the low-order binary16 part). */
// symmetric test matrix with a Marchenko-Pastur-like spectrum: G = B B^T / K from a random binary16 operand
int32_t scl_bench_syevd(scl_handle* h, int32_t n, int32_t mode, int32_t il, int32_t iu, double* ms) {
  if (!h || n < 8 || !ms) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    const int64_t K = 2 * (int64_t)n, ld = (K + 7) / 8 * 8;
    Tmp<__half> op((size_t)n * ld, h->st);
    Tmp<float> g((size_t)n * n, h->st), w(n, h->st);
    fill_random_f16(op.p, (size_t)n * ld, 0x5eedu, 1.0f, h->st);
    GemmArgs a;
    a.A.hi = op.p; a.A.rows = n; a.A.K = K; a.A.ld = ld;
    a.B = a.A;
    a.syrk = true; a.alpha = 1.0f / (float)K; a.C = g.p; a.ldc = n;
    a.cta_group = h->cfg.cta_group == 1 ? 1 : 2;
    gemm_umma(a, h->st);
    if (mode & 16) {   // the data Gram matrix of the last scl_run_signal instead of the synthetic one
      SCL_REQUIRE(h->signal_done && h->ws_Gkeep.p && h->sinfo.nm == n, "mode bit 4 needs a finished scl_run_signal of the same size");
      SCL_CUDA(cudaMemcpyAsync(g.p, h->ws_Gkeep.p, (size_t)n * n * sizeof(float), cudaMemcpyDeviceToDevice, h->st));
    }
    *ms = h->solver->bench(g.p, n, w.p, mode & 15, il, iu, h->st);
  });
}

int32_t scl_op_syevd_tri(scl_handle* h, int32_t n, const float* A, int32_t v0, int32_t v1, float* L, float* V, double* out_ms) {
  if (!h || !A || !L || n < 2 || v0 < 0 || v1 < v0 || v1 > n || (v1 > v0 && !V)) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    Tmp<float> g((size_t)n * n, h->st), w(n, h->st);
    SCL_CUDA(cudaMemcpyAsync(g.p, A, (size_t)n * n * sizeof(float), cudaMemcpyHostToDevice, h->st));
    const bool own = h->solver->syevd_tri(g.p, n, w.p, v0, v1, h->st);
    SCL_CUDA(cudaMemcpyAsync(L, w.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    if (v1 > v0)
      SCL_CUDA(cudaMemcpyAsync(V, g.p + (size_t)v0 * n, (size_t)(v1 - v0) * n * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
    if (out_ms) {
      for (int i = 0; i < 3; ++i) out_ms[i] = h->solver->tri_ms[i];
      out_ms[3] = (double)h->solver->tri_clusters;
      out_ms[4] = (double)h->solver->tri_clustered;
      out_ms[5] = own ? 0.0 : 1.0;
    }
  });
}

int32_t scl_op_draw_zero_candidates(scl_handle* h, uint64_t seed, int64_t* n, uint32_t* z1, uint32_t* z2) {
  if (!h || !n) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_X, "scl_set_counts_csc must be called first");
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    h->n_cand = draw_zero_candidates_device(h->X, seed, h->z1, h->z2, h->st);
    h->have_zc = true;
    *n = (int64_t)h->n_cand;
    if (z1) SCL_CUDA(cudaMemcpyAsync(z1, h->z1.p, h->n_cand * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
    if (z2) SCL_CUDA(cudaMemcpyAsync(z2, h->z2.p, h->n_cand * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_zero_candidate_draws(uint64_t seed, int64_t n_draws, int32_t N, int32_t M, uint32_t* rows, uint32_t* cols) {
  if (n_draws < 0 || N < 1 || M < 1 || !rows || !cols) return SCL_ERR_INVALID;
  const uint64_t grid = (uint64_t)N * (uint64_t)M;
  for (int64_t t = 0; t < n_draws; ++t) {
    const uint64_t g = zero_candidate_position_host(seed, (uint64_t)t, grid);
    rows[t] = (uint32_t)(g % (uint64_t)N);
    cols[t] = (uint32_t)(g / (uint64_t)N);
  }
  return SCL_OK;
}

int32_t scl_op_noise_baseline(scl_handle* h, int32_t nm, int32_t n_rep, uint64_t seed, double* p_th) {
  if (!h || nm < 1 || n_rep < 1 || !p_th) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    *p_th = noise_baseline_device(nm, n_rep, seed, h->st);
  });
}

int32_t scl_op_draw_subset(scl_handle* h, int64_t n_take, uint64_t seed, uint32_t* rows, uint32_t* cols) {
  if (!h || n_take < 0 || !rows || !cols) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_zc || h->n_cand > 0, "no zero candidates on the handle (scl_set_zero_candidates / scl_op_draw_zero_candidates)");
    SCL_REQUIRE((size_t)n_take <= h->n_cand, "sample larger than the candidate pool");
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    Tmp<uint32_t> r((size_t)std::max<int64_t>(1, n_take), h->st), c((size_t)std::max<int64_t>(1, n_take), h->st);
    draw_subset_device(h->z1.p, h->z2.p, h->n_cand, (size_t)n_take, seed, r.p, c.p, h->st);
    SCL_CUDA(cudaMemcpyAsync(rows, r.p, (size_t)n_take * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaMemcpyAsync(cols, c.p, (size_t)n_take * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_bench_syevd_concurrent(scl_handle* h, int32_t n, int32_t nsolves, int32_t mode, double* ms_wall) {
  if (!h || n < 8 || nsolves < 1 || nsolves > 8 || !ms_wall) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    const int64_t K = 2 * (int64_t)n, ld = (K + 7) / 8 * 8;
    Tmp<__half> op((size_t)n * ld, h->st);
    fill_random_f16(op.p, (size_t)n * ld, 0x5eedu, 1.0f, h->st);
    struct Lane {
      cudaStream_t st = nullptr;
      std::unique_ptr<Solver> solver;
      DBuf<float> g, w;
      std::string err;
    };
    std::vector<Lane> lanes(nsolves);
    for (auto& L : lanes) {
      SCL_CUDA(cudaStreamCreateWithFlags(&L.st, cudaStreamNonBlocking));
      L.solver.reset(new Solver(L.st));
      L.g.ensure((size_t)n * n);
      L.w.ensure(n);
    }
    auto fill = [&](Lane& L) {
      GemmArgs a;
      a.A.hi = op.p; a.A.rows = n; a.A.K = K; a.A.ld = ld;
      a.B = a.A;
      a.syrk = true; a.alpha = 1.0f / (float)K; a.C = L.g.p; a.ldc = n;
      a.cta_group = h->cfg.cta_group == 1 ? 1 : 2;
      gemm_umma(a, h->st);
    };
    // one warm-up solve per lane (workspace allocation, library initialisation), then the timed concurrent round
    for (int round = 0; round < 2; ++round) {
      for (auto& L : lanes) fill(L);
      SCL_CUDA(cudaStreamSynchronize(h->st));
      const auto t0 = std::chrono::steady_clock::now();
      std::vector<std::thread> th;
      for (auto& L : lanes)
        th.emplace_back([&L, n, mode, dev = h->cfg.device] {
          try {
            cudaSetDevice(dev);
            L.solver->syevd(L.g.p, n, L.w.p, mode == 0, L.st);
            cudaStreamSynchronize(L.st);
          } catch (const std::exception& e) { L.err = e.what(); }
        });
      for (auto& t : th) t.join();
      *ms_wall = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
      for (auto& L : lanes)
        if (!L.err.empty()) throw Error(SCL_ERR_CUSOLVER, L.err);
    }
    for (auto& L : lanes) { L.solver.reset(); cudaStreamDestroy(L.st); }
  });
}

int32_t scl_debug_set_eig_api(int32_t v) {
  scl::set_eig_api(v);
  return SCL_OK;
}

int32_t scl_debug_last_solve(scl_handle* h, double* out) {
  if (!h || !out || !h->solver) return SCL_ERR_INVALID;
  for (int i = 0; i < 5; ++i) out[i] = h->solver->tri_two_stage ? h->solver->ts_ms[i] : 0.0;
  out[5] = h->solver->tri_two_stage ? 1.0 : 0.0;
  out[6] = (double)h->solver->ts_fallbacks;
  out[7] = (double)h->solver->tri_fallbacks;
  return SCL_OK;
}

int32_t scl_debug_set_two_stage(int32_t q2_variant, int32_t stage1_engine, int32_t q1_engine) {
  scl::g_two_stage_override[0].store(q2_variant, std::memory_order_relaxed);
  scl::g_two_stage_override[1].store(stage1_engine, std::memory_order_relaxed);
  scl::g_two_stage_override[2].store(q1_engine, std::memory_order_relaxed);
  return SCL_OK;
}

int32_t scl_debug_eig_stage_totals(scl_handle* h, double* out) {
  if (!h || !out || !h->solver) return SCL_ERR_INVALID;
  for (int i = 0; i < 7; ++i) out[i] = h->solver->ts_total[i];
  out[7] = (double)h->solver->ts_fallbacks;
  return SCL_OK;
}

int32_t scl_debug_two_stage(scl_handle* h, int32_t n, const float* A, float* AB, float* d, float* e, float* Q2, float* Q,
                            int32_t* flags) {
  if (!h || !A || n < 8 || (n & 3)) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    cudaStream_t st = h->st;
    const size_t nn = (size_t)n * n;
    const int nlev = sb2st_levels(n);
    const long long ldv2 = (long long)nlev * kBand, ldt2 = nlev;
    Tmp<float> dA(nn, st), dAB((size_t)n * kLdab, st), T1((size_t)(n / kBand + 2) * kBand * kBand, st), dd(n, st), de(n, st);
    Tmp<float> V2((size_t)n * ldv2, st), tau2((size_t)n * ldt2, st), Z(nn, st);
    Tmp<int> fail(1, st);
    SCL_CUDA(cudaMemcpyAsync(dA.p, A, nn * sizeof(float), cudaMemcpyHostToDevice, st));
    SCL_CUDA(cudaMemsetAsync(fail.p, 0, sizeof(int), st));
    SCL_CUDA(cudaMemsetAsync(V2.p, 0, (size_t)n * ldv2 * sizeof(float), st));
    SCL_CUDA(cudaMemsetAsync(tau2.p, 0, (size_t)n * ldt2 * sizeof(float), st));
    const int npanels = sy2sb_lower(dA.p, n, n, dAB.p, T1.p, fail.p, st);
    if (AB) SCL_CUDA(cudaMemcpyAsync(AB, dAB.p, (size_t)n * kLdab * sizeof(float), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    sb2st(dAB.p, n, dd.p, de.p, true, V2.p, ldv2, tau2.p, ldt2, st);
    if (d) SCL_CUDA(cudaMemcpyAsync(d, dd.p, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (e) SCL_CUDA(cudaMemcpyAsync(e, de.p, (size_t)(n - 1) * sizeof(float), cudaMemcpyDeviceToHost, st));
    SCL_CUDA(cudaStreamSynchronize(st));
    if (Q2 || Q) {
      std::vector<float> eye(nn, 0.f);
      for (int i = 0; i < n; ++i) eye[(size_t)i * n + i] = 1.f;
      SCL_CUDA(cudaMemcpyAsync(Z.p, eye.data(), nn * sizeof(float), cudaMemcpyHostToDevice, st));
      apply_q2(V2.p, ldv2, tau2.p, ldt2, n, Z.p, n, n, st);
      if (Q2) SCL_CUDA(cudaMemcpyAsync(Q2, Z.p, nn * sizeof(float), cudaMemcpyDeviceToHost, st));
      SCL_CUDA(cudaStreamSynchronize(st));
      if (Q) {
        apply_q1(dA.p, n, n, T1.p, npanels, Z.p, n, n, st);
        SCL_CUDA(cudaMemcpyAsync(Q, Z.p, nn * sizeof(float), cudaMemcpyDeviceToHost, st));
      }
    }
    if (flags) {
      SCL_CUDA(cudaMemcpyAsync(&flags[0], fail.p, sizeof(int), cudaMemcpyDeviceToHost, st));
      flags[1] = npanels;
    }
    SCL_CUDA(cudaStreamSynchronize(st));
  });
}

int32_t scl_debug_set_tuning(int32_t stat_variant, int32_t stat_heavy, int32_t writer) {
  scl::set_norm_tuning(stat_variant, stat_heavy, writer);
  return SCL_OK;
}

int32_t scl_bench_normalize(scl_handle* h, int32_t layout, int32_t with_lo, int32_t reps, double* ms_stats,
                            double* ms_densify, double* alg_bytes_densify) {
  if (!h || reps <= 0) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_X, "scl_set_counts_csc must be called first");
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    const SpMat& X = h->X;
    const size_t line_len = layout == 1 ? X.M : X.N, lines = layout == 1 ? X.N : X.M;
    const size_t ld = (line_len + 7) / 8 * 8;
    Tmp<__half> hi(lines * ld, h->st), lo(with_lo ? lines * ld : 1, h->st);
    NormStats S;
    S.centering = h->cfg.centering;
    cudaEvent_t e0, e1, e2;
    SCL_CUDA(cudaEventCreate(&e0));
    SCL_CUDA(cudaEventCreate(&e1));
    SCL_CUDA(cudaEventCreate(&e2));
    double ts = 0, td = 0;
    for (int r = -1; r < reps; ++r) {   // r = -1: warm-up
      SCL_CUDA(cudaEventRecord(e0, h->st));
      compute_norm_stats(X, S, h->st);
      ensure_patch(X, S, layout, h->st);
      SCL_CUDA(cudaEventRecord(e1, h->st));
      densify(X, S, layout, ld, hi.p, with_lo ? lo.p : nullptr, h->st);
      SCL_CUDA(cudaEventRecord(e2, h->st));
      SCL_CUDA(cudaEventSynchronize(e2));
      float a = 0, b = 0;
      SCL_CUDA(cudaEventElapsedTime(&a, e0, e1));
      SCL_CUDA(cudaEventElapsedTime(&b, e1, e2));
      if (r >= 0) { ts += a; td += b; }
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1); cudaEventDestroy(e2);
    if (ms_stats) *ms_stats = ts / reps;
    if (ms_densify) *ms_densify = td / reps;
    if (alg_bytes_densify) *alg_bytes_densify = 8.0 * (double)X.nnz + 4.0 * (X.M + 1) + (double)X.N * X.M * (with_lo ? 4.0 : 2.0);
  });
}

int32_t scl_op_gemm_tn(scl_handle* h, int32_t m, int32_t n, int64_t K, int64_t lda, int64_t ldb, const uint16_t* a_hi,
                       const uint16_t* a_lo, const uint16_t* b_hi, const uint16_t* b_lo, float alpha,
                       int32_t c_colmajor, float* C) {
  if (!h || !a_hi || !b_hi || !C) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    const size_t na = (size_t)m * lda, nb = (size_t)n * ldb;
    const bool split = a_lo && b_lo;
    Tmp<__half> ah(na, h->st), al(na, h->st), bh(nb, h->st), bl(nb, h->st);
    Tmp<float> c((size_t)m * n, h->st);
    SCL_CUDA(cudaMemcpyAsync(ah.p, a_hi, na * 2, cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(bh.p, b_hi, nb * 2, cudaMemcpyHostToDevice, h->st));
    if (split) {
      SCL_CUDA(cudaMemcpyAsync(al.p, a_lo, na * 2, cudaMemcpyHostToDevice, h->st));
      SCL_CUDA(cudaMemcpyAsync(bl.p, b_lo, nb * 2, cudaMemcpyHostToDevice, h->st));
    }
    SCL_CUDA(cudaMemsetAsync(c.p, 0, (size_t)m * n * sizeof(float), h->st));
    GemmArgs a;
    a.A.hi = ah.p; a.A.lo = split ? al.p : nullptr; a.A.rows = m; a.A.K = K; a.A.ld = lda;
    a.B.hi = bh.p; a.B.lo = split ? bl.p : nullptr; a.B.rows = n; a.B.K = K; a.B.ld = ldb;
    a.alpha = alpha;
    a.epi = c_colmajor ? Epilogue::StoreTransposed : Epilogue::Store;
    a.C = c.p;
    a.ldc = c_colmajor ? m : n;
    a.cta_group = h->cfg.cta_group == 1 ? 1 : 2;
    gemm_umma(a, h->st);
    SCL_CUDA(cudaMemcpyAsync(C, c.p, (size_t)m * n * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_syevd(scl_handle* h, int32_t n, const float* A, float* L, float* V, double* ms) {
  if (!h || !A || !L) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    Tmp<float> a((size_t)n * n, h->st), w(n, h->st);
    SCL_CUDA(cudaMemcpyAsync(a.p, A, (size_t)n * n * sizeof(float), cudaMemcpyHostToDevice, h->st));
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0, h->st);
    h->solver->syevd(a.p, n, w.p, V != nullptr, h->st);
    cudaEventRecord(e1, h->st);
    cudaEventSynchronize(e1);
    float t = 0;
    cudaEventElapsedTime(&t, e0, e1);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    if (ms) *ms = t;
    SCL_CUDA(cudaMemcpyAsync(L, w.p, n * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    if (V) SCL_CUDA(cudaMemcpyAsync(V, a.p, (size_t)n * n * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_mp_fit(const float* L, int32_t nL, const float* Lr, int32_t nLr, double out[8]) {
  if (!L || !Lr || !out) return SCL_ERR_INVALID;
  return guard(nullptr, [&] {
    MpFit f = mp_fit(L, nL, Lr, nLr);
    out[0] = f.lambda_c; out[1] = f.b_plus; out[2] = f.b_minus; out[3] = f.ks_static;
    out[4] = (double)f.L_mp.size(); out[5] = f.iters; out[6] = f.pass ? 1 : 0; out[7] = f.n_signal;
  });
}

int32_t scl_op_permute_null(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr,
                            const uint32_t* rowval, const float* nzval, const uint32_t* perm, const uint32_t* rows,
                            int64_t* out_nnz, uint32_t* out_colptr, uint32_t* out_rowval, float* out_val) {
  if (!h || !out_nnz) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    SpMat A, R;
    upload_csc(A, N, M, (size_t)nnz, colptr, rowval, nzval, 0, h->st);
    if (perm && rows) {
      DBuf<uint32_t> dp, dr;
      upload_u32(dp, perm, (size_t)nnz, 0, h->st);
      upload_u32(dr, rows, (size_t)nnz, 0, h->st);
      permute_null(A, dp.p, dr.p, R, h->st);
      SCL_CUDA(cudaStreamSynchronize(h->st));
    } else {
      draw_null_device(A, h->cfg.seed, R, h->st);
    }
    *out_nnz = (int64_t)R.nnz;
    if (out_colptr && out_rowval && out_val) download_csc(R, out_colptr, out_rowval, out_val, h->st);
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_perturb_merge(scl_handle* h, int32_t N, int32_t M, int64_t nnz, const uint32_t* colptr,
                             const uint32_t* rowval, const float* nzval, int64_t n_add, const uint32_t* add_row,
                             const uint32_t* add_col, int32_t binarise, uint32_t* out_colptr, uint32_t* out_rowval,
                             float* out_val) {
  if (!h || !out_colptr) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    SpMat A, R;
    upload_csc(A, N, M, (size_t)nnz, colptr, rowval, nzval, 0, h->st);
    DBuf<uint32_t> dr, dc;
    upload_u32(dr, add_row, (size_t)n_add, 0, h->st);
    upload_u32(dc, add_col, (size_t)n_add, 0, h->st);
    perturb_merge(A, dr.p, dc.p, (size_t)n_add, binarise != 0, R, h->st);
    download_csc(R, out_colptr, out_rowval, out_val, h->st);
  });
}

int32_t scl_op_corr_colabsmax(scl_handle* h, int32_t n, int32_t nv, int32_t nw, const float* V, const float* W, float* d) {
  if (!h || !V || !W || !d) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    Tmp<float> dv((size_t)nv * n, h->st), dw((size_t)nw * n, h->st), dd(nw, h->st);
    SCL_CUDA(cudaMemcpyAsync(dv.p, V, (size_t)nv * n * sizeof(float), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(dw.p, W, (size_t)nw * n * sizeof(float), cudaMemcpyHostToDevice, h->st));
    corr_colabsmax(h, dv.p, nv, dw.p, nw, n, dd.p);
    SCL_CUDA(cudaMemcpyAsync(d, dd.p, nw * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_topk_subspace(scl_handle* h, int32_t n, const float* G, int32_t k, float* L, float* V, int32_t* iters) {
  if (!h || !G || !L || !V) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    Tmp<float> g((size_t)n * n, h->st), l(k, h->st), v((size_t)k * n, h->st);
    SCL_CUDA(cudaMemcpyAsync(g.p, G, (size_t)n * n * sizeof(float), cudaMemcpyHostToDevice, h->st));
    int it = 0;
    topk_subspace(h, g.p, n, k, l.p, v.p, &it);
    if (iters) *iters = it;
    SCL_CUDA(cudaMemcpyAsync(L, l.p, k * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaMemcpyAsync(V, v.p, (size_t)k * n * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_scores(scl_handle* h, int32_t N, int32_t k, int32_t min_pc, int32_t n_perturb, const float* nV,
                      const float* nV_sets, double th, float* b_, double* m_scores, double* sd_scores, int32_t* sig_id,
                      int32_t* n_robust) {
  if (!h || !nV || !nV_sets) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    const size_t ns = (size_t)n_perturb * min_pc * N;
    Tmp<float> dv((size_t)k * N, h->st), ds(ns, h->st);
    SCL_CUDA(cudaMemcpyAsync(dv.p, nV, (size_t)k * N * sizeof(float), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(ds.p, nV_sets, ns * sizeof(float), cudaMemcpyHostToDevice, h->st));
    std::vector<float> b;
    std::vector<double> m, sd;
    std::vector<int32_t> sig;
    score_sets(h, N, k, min_pc, n_perturb, dv.p, ds.p, th, b, m, sd, sig);
    if (b_) std::memcpy(b_, b.data(), b.size() * sizeof(float));
    if (m_scores) std::memcpy(m_scores, m.data(), m.size() * sizeof(double));
    if (sd_scores) std::memcpy(sd_scores, sd.data(), sd.size() * sizeof(double));
    if (sig_id) std::memcpy(sig_id, sig.data(), sig.size() * sizeof(int32_t));
    if (n_robust) *n_robust = (int32_t)sig.size();
  });
}

// host tail of the scoring (:797-806) on a given k x n_pairs similarity table: pure host code
int32_t scl_op_scores_from_pairs(const float* b_, int32_t k, int32_t n_pairs, double th, double* m_scores, double* sd_scores,
                                 int32_t* sig_id, int32_t* n_robust) {
  if (!b_ || k < 1 || n_pairs < 1 || !n_robust) return SCL_ERR_INVALID;
  return guard(nullptr, [&] {
    std::vector<float> b(b_, b_ + (size_t)k * n_pairs);
    std::vector<double> m, sd;
    std::vector<int32_t> sig;
    score_from_pairs(b, k, n_pairs, th, m, sd, sig);
    if (m_scores) std::memcpy(m_scores, m.data(), m.size() * sizeof(double));
    if (sd_scores) std::memcpy(sd_scores, sd.data(), sd.size() * sizeof(double));
    if (sig_id) std::memcpy(sig_id, sig.data(), sig.size() * sizeof(int32_t));
    *n_robust = (int32_t)sig.size();
  });
}

// get_denoised_df (:889-931) from the entries of the result Dict (all host pointers, Julia layouts)
int32_t scl_op_denoise(scl_handle* h, int32_t N, int32_t M, int32_t r, const float* pca_n1, const float* g_mat,
                       const double* TGC, const double* mat2_mean, const double* mat2_std, const double* norm_tgc,
                       const double* cent, int32_t out_f32, void* out) {
  if (!h || !pca_n1 || !g_mat || !TGC || !mat2_mean || !mat2_std || !norm_tgc || !cent || !out) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(N > 0 && M > 0 && r > 0, "bad shape");
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    double mean_tgc = 0, mean_l = 0;
    for (int i = 0; i < N; ++i) { mean_tgc += TGC[i]; mean_l += norm_tgc[i]; }
    mean_tgc /= (double)N;
    mean_l /= (double)N;
    SCL_REQUIRE(mean_l > 0, "norm_tgc must be positive");
    Tmp<float> dA((size_t)r * N, h->st), dG((size_t)r * M, h->st);
    Tmp<double> dc(M, h->st), ds(M, h->st), dy(M, h->st), dl(N, h->st);
    SCL_CUDA(cudaMemcpyAsync(dA.p, pca_n1, (size_t)r * N * sizeof(float), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(dG.p, g_mat, (size_t)r * M * sizeof(float), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(dc.p, cent, M * sizeof(double), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(ds.p, mat2_std, M * sizeof(double), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(dy.p, mat2_mean, M * sizeof(double), cudaMemcpyHostToDevice, h->st));
    SCL_CUDA(cudaMemcpyAsync(dl.p, norm_tgc, N * sizeof(double), cudaMemcpyHostToDevice, h->st));
    const size_t bytes = (size_t)N * M * (out_f32 ? sizeof(float) : sizeof(double));
    Tmp<unsigned char> dout(bytes, h->st);
    denoise(dA.p, dG.p, r, N, M, dc.p, ds.p, dy.p, dl.p, mean_l, mean_tgc, dout.p, out_f32 != 0, h->st);
    SCL_CUDA(cudaMemcpyAsync(out, dout.p, bytes, cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

// ---- apply_umap! -----------------------------------------------------------------------------------------------------
namespace {
void check_umap_input(int32_t N, int32_t d, const float* X, int32_t k, int32_t metric) {
  SCL_REQUIRE(X != nullptr, "X is NULL");
  SCL_REQUIRE(N >= 2 && d >= 1 && d <= 1024, "bad shape");
  SCL_REQUIRE(k >= 1 && k <= 64 && k < N, "need 1 <= n_neighbors <= 64 and n_neighbors < N");
  SCL_REQUIRE(metric == 0 || metric == 1, "metric must be 0 (euclidean) or 1 (cosine)");
  const size_t n = (size_t)N * d;
  for (size_t i = 0; i < n; ++i) SCL_REQUIRE(std::isfinite(X[i]), "X has a non-finite entry");
}
}  // namespace

int32_t scl_op_knn(scl_handle* h, int32_t N, int32_t d, const float* X, int32_t k, int32_t metric, int32_t* idx, float* dist) {
  if (!h || !idx || !dist) return SCL_ERR_INVALID;
  return guard(h, [&] {
    check_umap_input(N, d, X, k, metric);
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    Tmp<float> dX((size_t)N * d, h->st);
    Tmp<int32_t> di((size_t)N * k, h->st);
    Tmp<float> dd((size_t)N * k, h->st);
    SCL_CUDA(cudaMemcpyAsync(dX.p, X, (size_t)N * d * sizeof(float), cudaMemcpyHostToDevice, h->st));
    knn_device(dX.p, N, d, k, metric, di.p, dd.p, h->st);
    SCL_CUDA(cudaMemcpyAsync(idx, di.p, (size_t)N * k * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaMemcpyAsync(dist, dd.p, (size_t)N * k * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_op_umap(scl_handle* h, int32_t N, int32_t d, const float* X, const scl_umap_params* p, const float* init_embedding,
                    float* embedding, scl_umap_info* info) {
  if (!h || !p || !embedding || !info) return SCL_ERR_INVALID;
  return guard(h, [&] {
    const scl_umap_params& q = *p;
    check_umap_input(N, d, X, q.n_neighbors, q.metric);
    SCL_REQUIRE(q.n_components >= 1 && q.n_components <= 16, "n_components must be in [1, 16]");
    SCL_REQUIRE(q.n_epochs >= 0 && q.init >= 0 && q.init <= 1 && q.neg_sample_rate >= 0 && q.spectral_maxiter >= 0,
                "bad n_epochs / init / neg_sample_rate / spectral_maxiter");
    SCL_REQUIRE(std::isfinite(q.min_dist) && q.min_dist >= 0 && std::isfinite(q.spread) && q.spread > 0,
                "need min_dist >= 0 and spread > 0");
    SCL_REQUIRE(std::isfinite(q.learning_rate) && q.learning_rate > 0 && std::isfinite(q.repulsion_strength) &&
                q.repulsion_strength >= 0, "need learning_rate > 0 and repulsion_strength >= 0");
    SCL_REQUIRE(std::isfinite(q.local_connectivity) && q.local_connectivity >= 0 && q.local_connectivity <= q.n_neighbors,
                "need 0 <= local_connectivity <= n_neighbors");
    const size_t ne = (size_t)N * q.n_components;
    if (init_embedding)
      for (size_t i = 0; i < ne; ++i) SCL_REQUIRE(std::isfinite(init_embedding[i]), "init_embedding has a non-finite entry");
    SCL_CUDA(cudaSetDevice(h->cfg.device));
    h->have_umap_graph = false;
    Tmp<float> dX((size_t)N * d, h->st), dI(init_embedding ? ne : 1, h->st), dE(ne, h->st);
    SCL_CUDA(cudaMemcpyAsync(dX.p, X, (size_t)N * d * sizeof(float), cudaMemcpyHostToDevice, h->st));
    if (init_embedding) SCL_CUDA(cudaMemcpyAsync(dI.p, init_embedding, ne * sizeof(float), cudaMemcpyHostToDevice, h->st));
    umap_run(h, dX.p, N, d, q, init_embedding ? dI.p : nullptr, dE.p, info);
    SCL_CUDA(cudaMemcpyAsync(embedding, dE.p, ne * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_get_umap_graph(scl_handle* h, int64_t* nnz, uint32_t* rowptr, uint32_t* colidx, float* val) {
  if (!h || !nnz) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_umap_graph, "scl_op_umap has not completed");
    *nnz = (int64_t)h->ug_nnz;
    if (rowptr && colidx && val) {
      SCL_CUDA(cudaMemcpyAsync(rowptr, h->ug_rowptr.p, (h->ug_N + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
      SCL_CUDA(cudaMemcpyAsync(colidx, h->ug_col.p, h->ug_nnz * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->st));
      SCL_CUDA(cudaMemcpyAsync(val, h->ug_val.p, h->ug_nnz * sizeof(float), cudaMemcpyDeviceToHost, h->st));
      SCL_CUDA(cudaStreamSynchronize(h->st));
    }
  });
}

int32_t scl_get_umap_knn(scl_handle* h, int32_t* idx, float* dist) {
  if (!h || !idx || !dist) return SCL_ERR_INVALID;
  return guard(h, [&] {
    SCL_REQUIRE(h->have_umap_graph, "scl_op_umap has not completed");
    const size_t n = (size_t)h->uk_N * h->uk_k;
    SCL_CUDA(cudaMemcpyAsync(idx, h->uk_idx.p, n * sizeof(int32_t), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaMemcpyAsync(dist, h->uk_dist.p, n * sizeof(float), cudaMemcpyDeviceToHost, h->st));
    SCL_CUDA(cudaStreamSynchronize(h->st));
  });
}

int32_t scl_umap_fit_ab(double min_dist, double spread, double* a, double* b) {
  if (!a || !b || !std::isfinite(min_dist) || !(min_dist >= 0) || !std::isfinite(spread) || !(spread > 0)) return SCL_ERR_INVALID;
  return guard(nullptr, [&] { umap_fit_ab(min_dist, spread, a, b); });
}

}  // extern "C"
