// Grouped small-GEMM launcher (exact-fp32 FFMA path) used by the MLP forward/backward.
#pragma once
#include "common.cuh"
#include <cuda.h>     // CUtensorMap (type only; the encoder is resolved through the runtime)

namespace d4pg {

enum GemmMode {
  GEMM_FWD = 0,   // C[M,N] = A[M,K] . W[N,K]^T (+bias, act)      models.py:33-40,77-83
  GEMM_DX = 1,    // C[M,N] = dZ[M,K] . W[K,N]    (* act')         autograd of the above, ddpg.py:230,242
  GEMM_DW = 2     // C[M,N] = dZ[K,M]^T . X[K,N]  (+ column sums -> bias grad)
};
enum GemmEpi {
  EPI_NONE = 0, EPI_BIAS = 1, EPI_BIAS_RELU = 2, EPI_BIAS_TANH = 3,
  EPI_RELU_MASK = 4,   // C *= (aux > 0)
  EPI_TANH_MASK = 5    // C *= (1 - aux^2)
};

struct GemmProblem {
  const float* A; const float* A2; const float* Bm; const float* bias; const float* aux;
  float* C; float* bias_grad;
  int M, N, K, K1;
  int lda, lda2, ldb, ldc, ldaux;
  int mode, epi, flags;
  int tiles_m, tiles_n, tile_begin;
  // split-K (dW only, large batches): the contraction dim is cut into `ksplit` slices of `kslice`
  // (a multiple of every kernel's K chunk); slice CTAs accumulate into C with fp32 atomics, so C must
  // be zero beforehand (the learner clears the gradient buffer at the start of such a step).
  int ksplit, kslice;
};

constexpr int GEMM_MAX_PROBLEMS = 8;
enum GemmFlags { GEMM_A_VEC = 1, GEMM_B_VEC = 2, GEMM_A_TMA = 4, GEMM_B_TMA = 8, GEMM_ASYNC_OK = 16 };
struct GemmBatch {
  GemmProblem p[GEMM_MAX_PROBLEMS];
  int n;
  int total_tiles;
  // tcgen05 path only: TMA descriptors of the operands that qualify (16-B aligned rows, K-major)
  alignas(64) CUtensorMap tmap_a[GEMM_MAX_PROBLEMS];
  alignas(64) CUtensorMap tmap_b[GEMM_MAX_PROBLEMS];
  alignas(64) CUtensorMap tmap_a2[GEMM_MAX_PROBLEMS];   // concatenated tail of A (critic fc2's action columns)
  int all_tma;                                           // every operand of every problem is TMA-fed -> v2 kernel
  unsigned long long* trace;                             // optional %globaltimer phase stamps of CTA 0 (D4PG_TC_TRACE)
};

// host helpers ---------------------------------------------------------------------------
GemmProblem gemm_fwd(const float* X, int ldx, const float* X2, int ldx2, int K1, const float* W, int ldw,
                     const float* bias, float* Y, int ldy, int M, int N, int K, int epi);
GemmProblem gemm_dx(const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx,
                    int M, int N_in, int K_out, int epi, const float* aux, int ldaux);
GemmProblem gemm_dw(const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw,
                    float* db, int N_out, int K_in, int M_batch);
void gemm_batch_begin(GemmBatch& b);
void gemm_batch_add(GemmBatch& b, const GemmProblem& p);
int gemm_batch_launch(const GemmBatch& b, cudaStream_t st);                    // exact fp32 FFMA (32x32 tiles)
void gemm_batch_retile(GemmBatch& b, int bm, int bn);
bool gemm_batch_has_splitk(const GemmBatch& b);
void gemm_tc_prepare(GemmBatch& b);                                             // TMA eligibility + tensor maps
int gemm_tc_batch_launch(const GemmBatch& b, int passes, cudaStream_t st);      // tcgen05 (128x32 tiles)
// precision: 0 = fp32 FFMA, 1 = 3xTF32 tcgen05 (fp32-accurate), 2 = 1xTF32 tcgen05
int gemm_launch(GemmBatch& b, int precision, cudaStream_t st);

}  // namespace d4pg
