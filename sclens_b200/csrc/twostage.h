// Two-stage symmetric eigensolver (replaces the one-stage tridiagonalisation inside _get_eigen, src/scLENS.jl:375-382):
//   stage 1  sy2sb.cu     dense -> band (half bandwidth kBand): CholeskyQR panels with Householder reconstruction, two-sided
//                         rank-2b updates - all matrix-matrix work, no matrix-vector products over the trailing matrix
//   stage 2  sb2st.cu     band -> tridiagonal by bulge chasing: one persistent kernel, sweeps pipelined through progress flags
//   (tridiag.cu)          eigenvalues / eigenvectors of T in Float64, as in the one-stage path
//   back     backtrans.cu Z = Q1 Q2 E: stage-2 reflectors in blocks of kBand sweeps x one chase level, stage-1 panels as I - V T V'
// The algebra is restated on the CPU in oracle/two_stage_ref.py (tests/test_two_stage_cpu.py).
#pragma once
#include <cuda_runtime.h>
#include "common.cuh"

namespace scl {

constexpr int kBand = 64;          // half bandwidth of the intermediate band matrix = panel width of stage 1
constexpr int kLdab = 2 * kBand;   // band storage: AB[j * kLdab + (i - j)], 0 <= i - j < 2 kBand (room for the bulge)

struct TwoStageTimes {
  double ms[6] = {0, 0, 0, 0, 0, 0};   // sy2sb, sb2st, tridiagonal eigenproblem, Q2, Q1, copies
};

// stage 1.  A: n x n column-major, leading dimension lda (multiple of 4, 16-byte aligned base), lower triangle read.  On
// return: the band in AB (zero outside the half bandwidth), the panels' reflectors V in A below the band (panel k: columns
// k kBand .. of A, rows (k+1) kBand .. n, unit lower trapezoidal, stored explicitly), their T factors in T1 [panel][kBand^2]
// (row-major).  *d_fail (device flag) is raised when a panel could not be factored (rank-deficient panel).
// Returns the number of panels.
// aux (optional): a second stream and two events for the look-ahead - the next panel is factored there while the main stream
// finishes the trailing update.
struct Sy2sbAux {
  cudaStream_t stream = nullptr;
  cudaEvent_t ready = nullptr, done = nullptr;
};
// half_ok: the matrix passed half_range_ok, so the products of the trailing update may run in split binary16 (engine 2)
int sy2sb_lower(float* A, int n, long long lda, float* AB, float* T1, int* d_fail, cudaStream_t st, const Sy2sbAux* aux = nullptr,
                bool half_ok = false);
bool half_range_ok(const float* A, int n, long long lda, cudaStream_t st);

// stage 2.  AB as above (destroyed).  d (n), e (n - 1).  With keep = true the reflector of sweep s, chase level k is stored at
// V2 + s * ldv2 + k * kBand (kBand floats, v[0] = 1) and its tau at tau2 + s * ldt2 + k.
void sb2st(float* AB, int n, float* d, float* e, bool keep, float* V2, long long ldv2, float* tau2, long long ldt2,
           cudaStream_t st);
inline int sb2st_levels(int n) { return (n + kBand - 1) / kBand + 1; }

// Z: mvec vectors of length n, vector-major (vector v at Z + v * ldz, ldz a multiple of 4).  Z <- Q2 Z.
void apply_q2(const float* V2, long long ldv2, const float* tau2, long long ldt2, int n, float* Z, long long ldz, int mvec,
              cudaStream_t st);
// Z <- Q1 Z with the panels left in A by sy2sb_lower
void apply_q1(const float* A, int n, long long lda, const float* T1, int npanels, float* Z, long long ldz, int mvec,
              cudaStream_t st);

// Engines of the matrix-matrix products, each chosen by the input (measured at n = 20 000; a / b = smallest half / all vectors):
//   stage 1   split binary16 on the mma.sync tile engine of sgemm_tile.cuh when the matrix passes half_range_ok, three-term
//             TF32 otherwise (304 vs 369 ms; FP32 FMA took 394 ms against 370 ms for TF32 in an earlier run)
//   Q2        register-stationary split binary16 (254 / 440 ms; three-term TF32 380 / 558 ms, a shared-memory window 818 / 1627 ms)
//   Q1        64 vectors or more: eight panels at a time on the tcgen05 GEMM of gemm_umma.cu in split binary16 (83 / 130 ms);
//             fewer: panel by panel on the split-binary16 tile engine (192 / 366 ms at this size, where it is not used; TF32
//             251 / 474 ms, FP32 FMA 252 / 487 ms)

// every vector scaled to unit length (after the back-transformation: the tensor-core products of apply_q2 lose ~1e-7 n / 64)
void unit_vectors(float* Z, long long ldz, int n, int mvec, cudaStream_t st);

}  // namespace scl
