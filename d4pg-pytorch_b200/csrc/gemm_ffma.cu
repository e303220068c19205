// Exact-fp32 grouped GEMM for the actor/critic MLP layers (precision mode 0).
//
// Replaces the ATen/MKL nn.Linear forward calls of models.py:33-40,77-83 and their autograd
// backward (ddpg.py:230,242).  One launch runs up to 8 independent layer problems (the actor,
// critic and target networks advance in lock-step through the step's dependency levels), each
// tiled 32x32 so a 256x256x256 layer spreads over 64 CTAs: at batch 256 the whole step is
// latency-bound, so small tiles on many SMs beat big tiles on few.  Accumulation is plain FFMA
// in k order, i.e. a true fp32 dot product (needed for the 1e-5 parity of config 2).
#include "gemm_ffma_dev.cuh"
#include "mlp_chain.cuh"
#include <algorithm>

namespace d4pg {

template <bool ALLOW_SPLIT>
__global__ void __launch_bounds__(GEMM_THREADS, 2) gemm_ffma_kernel(const __grid_constant__ GemmBatch batch) {
  __shared__ __align__(16) float smem[2 * KC * LDS_A + 2 * KC * LDS_B];
  static_assert(2 * KC * LDS_A + 2 * KC * LDS_B >= GEMM_WARPS * BM * BN, "partial-tile buffer must fit");
  int pi = 0;
#pragma unroll
  for (int i = 1; i < GEMM_MAX_PROBLEMS; ++i)
    if (i < batch.n && int(blockIdx.x) >= batch.p[i].tile_begin) pi = i;
  const GemmProblem P = batch.p[pi];        // one copy into registers (no constant-bank reads in the loops)
  gemm_tile_dispatch<ALLOW_SPLIT>(P, smem, blockIdx.x - P.tile_begin);
}

// Every dW of a step in one launch (mlp_chain.cuh: GemmWideBatch).  Only the asynchronous dW tile is
// compiled in, which needs no staging registers: 3 CTAs per SM (304 tiles at config 2 are ONE wave; at
// 2 CTAs per SM the last 8 tiles were a second wave that doubled the launch's duration).
template <bool ALLOW_SPLIT>
__global__ void __launch_bounds__(GEMM_THREADS, 3) gemm_wide_kernel(const __grid_constant__ GemmWideBatch batch) {
  extern __shared__ __align__(16) float smem[];        // DW_SMEM_FLOATS
  int pi = 0;
#pragma unroll
  for (int i = 1; i < GEMM_WIDE_MAX; ++i)
    if (i < batch.n && int(blockIdx.x) >= batch.p[i].tile_begin) pi = i;
  const GemmProblem& P = batch.p[pi];
  const int tile = blockIdx.x - P.tile_begin;
  step_stamp(batch.trace, 6);
  if (ALLOW_SPLIT && P.ksplit > 1) {
    const int per_slice = P.tiles_m * P.tiles_n;
    const int ks = tile / per_slice, t2 = tile - ks * per_slice;
    const int tm = t2 / P.tiles_n, tn = t2 - tm * P.tiles_n;
    const int kbeg = ks * P.kslice;
    gemm_dw_tile_async<true>(P, smem, tm * BM, tn * BN, tn, kbeg, min(P.K, kbeg + P.kslice));
  } else {
    const int tm = tile / P.tiles_n, tn = tile - tm * P.tiles_n;
    gemm_dw_tile_async<false>(P, smem, tm * BM, tn * BN, tn, 0, P.K);
  }
  step_stamp(batch.trace, 6 + 16);
  if (batch.has_peer_sig) {                              // gradients of this rank complete -> tell the peers (system scope)
    __syncthreads();
    if (threadIdx.x == 0) peer_signal_last_cta(batch.peer_sig, gridDim.x);
  }
}

// ---- host side -------------------------------------------------------------------------------
GemmProblem gemm_fwd(const float* X, int ldx, const float* X2, int ldx2, int K1, const float* W, int ldw,
                     const float* bias, float* Y, int ldy, int M, int N, int K, int epi) {
  GemmProblem p{};
  p.A = X; p.lda = ldx; p.A2 = X2 ? X2 : X; p.lda2 = X2 ? ldx2 : ldx; p.K1 = X2 ? K1 : K;
  p.Bm = W; p.ldb = ldw; p.bias = bias; p.C = Y; p.ldc = ldy; p.M = M; p.N = N; p.K = K;
  p.mode = GEMM_FWD; p.epi = epi;
  return p;
}
GemmProblem gemm_dx(const float* dZ, int lddz, const float* W, int ldw, float* dX, int lddx,
                    int M, int N_in, int K_out, int epi, const float* aux, int ldaux) {
  GemmProblem p{};
  p.A = dZ; p.lda = lddz; p.A2 = dZ; p.lda2 = lddz; p.K1 = K_out;
  p.Bm = W; p.ldb = ldw; p.C = dX; p.ldc = lddx; p.M = M; p.N = N_in; p.K = K_out;
  p.mode = GEMM_DX; p.epi = epi; p.aux = aux; p.ldaux = ldaux;
  return p;
}
GemmProblem gemm_dw(const float* dZ, int lddz, const float* X, int ldx, float* dW, int lddw,
                    float* db, int N_out, int K_in, int M_batch) {
  GemmProblem p{};
  p.A = dZ; p.lda = lddz; p.A2 = dZ; p.lda2 = lddz; p.K1 = M_batch;
  p.Bm = X; p.ldb = ldx; p.C = dW; p.ldc = lddw; p.bias_grad = db;
  p.M = N_out; p.N = K_in; p.K = M_batch;
  p.mode = GEMM_DW; p.epi = EPI_NONE;
  return p;
}
void gemm_batch_begin(GemmBatch& b) { b.n = 0; b.total_tiles = 0; b.all_tma = 0; b.trace = nullptr; }
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }
static void prepare_problem(GemmProblem& p) {
  // 128-bit staging is legal when rows start 16-B aligned and the contiguous extent is a multiple of 4
  bool avec, bvec;
  if (p.mode == GEMM_DW) avec = aligned16(p.A) && p.lda % 4 == 0 && p.M % 4 == 0;
  else avec = aligned16(p.A) && p.lda % 4 == 0 && p.K1 % 4 == 0;
  if (p.mode == GEMM_FWD) bvec = aligned16(p.Bm) && p.ldb % 4 == 0 && p.K % 4 == 0;
  else bvec = aligned16(p.Bm) && p.ldb % 4 == 0 && p.N % 4 == 0;
  p.flags = (avec ? GEMM_A_VEC : 0) | (bvec ? GEMM_B_VEC : 0);
  if (p.mode == GEMM_DW && aligned16(p.A) && p.lda % 4 == 0 && aligned16(p.Bm) && p.ldb % 4 == 0) p.flags |= GEMM_ASYNC_OK;
  // dW over a large batch: 8 tiles x (B/32) serial chunks would leave the GPU idle -> split K
  p.ksplit = 1; p.kslice = p.K;
  if (p.mode == GEMM_DW && p.K >= 1024) {
    p.ksplit = std::min(8, cdiv(p.K, 512));
    p.kslice = cdiv(cdiv(p.K, p.ksplit), 64) * 64;
    p.ksplit = cdiv(p.K, p.kslice);
  }
  p.tiles_m = cdiv(p.M, BM); p.tiles_n = cdiv(p.N, BN);
}
void gemm_batch_add(GemmBatch& b, const GemmProblem& pin) {
  GemmProblem p = pin;
  prepare_problem(p);
  p.tile_begin = b.total_tiles;
  b.total_tiles += p.tiles_m * p.tiles_n * p.ksplit;
  b.p[b.n++] = p;
}
void gemm_batch_retile(GemmBatch& b, int bm, int bn) {
  b.total_tiles = 0;
  for (int i = 0; i < b.n; ++i) {
    GemmProblem& p = b.p[i];
    p.tiles_m = cdiv(p.M, bm); p.tiles_n = cdiv(p.N, bn); p.tile_begin = b.total_tiles;
    b.total_tiles += p.tiles_m * p.tiles_n * p.ksplit;
  }
}
void gemm_wide_begin(GemmWideBatch& b, const PeerSignal* sig) {
  b.n = 0; b.total_tiles = 0; b.trace = nullptr; b.has_peer_sig = sig ? 1 : 0;
  if (sig) b.peer_sig = *sig;
}
void gemm_wide_add(GemmWideBatch& b, const GemmProblem& pin) {
  if (b.n >= GEMM_WIDE_MAX) { b.n = GEMM_WIDE_MAX + 1; return; }      // reported by gemm_wide_launch
  GemmProblem p = pin;
  prepare_problem(p);
  p.tile_begin = b.total_tiles;
  b.total_tiles += p.tiles_m * p.tiles_n * p.ksplit;
  b.p[b.n++] = p;
}
int gemm_wide_launch(GemmWideBatch& b, cudaStream_t st) {
  D4PG_REQUIRE(b.n > 0 && b.n <= GEMM_WIDE_MAX, D4PG_EINVAL, "gemm_wide_launch: %d problems (max %d)", b.n, GEMM_WIDE_MAX);
  bool split = false;
  for (int i = 0; i < b.n; ++i) {
    split = split || b.p[i].ksplit > 1;
    D4PG_REQUIRE(b.p[i].mode == GEMM_DW && (b.p[i].flags & GEMM_ASYNC_OK), D4PG_ENOTSUP,
                 "gemm_wide_launch: problem %d is not a dW with 16-B aligned, 16-B pitched operands", i);
  }
  D4PG_MAX_CARVEOUT(gemm_wide_kernel<false>);
  D4PG_MAX_CARVEOUT(gemm_wide_kernel<true>);
  const size_t smem = DW_SMEM_FLOATS * sizeof(float);
  static bool smem_set = false;
  if (!smem_set) {
    D4PG_CUDA_OK(cudaFuncSetAttribute(gemm_wide_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    D4PG_CUDA_OK(cudaFuncSetAttribute(gemm_wide_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    smem_set = true;
  }
  b.trace = debug_trace_buffer() ? debug_trace_buffer() + STEP_TRACE_BASE : nullptr;
  if (split) gemm_wide_kernel<true><<<b.total_tiles, GEMM_THREADS, smem, st>>>(b);
  else gemm_wide_kernel<false><<<b.total_tiles, GEMM_THREADS, smem, st>>>(b);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}
bool gemm_batch_has_splitk(const GemmBatch& b) {
  for (int i = 0; i < b.n; ++i) if (b.p[i].ksplit > 1) return true;
  return false;
}
int gemm_launch(GemmBatch& b, int precision, cudaStream_t st) {
  if (precision == 0) return gemm_batch_launch(b, st);
  gemm_tc_prepare(b);                 // picks the kernel variant and tiles the problems accordingly
  return gemm_tc_batch_launch(b, precision == 1 ? 3 : 1, st);
}
int gemm_batch_launch(const GemmBatch& b, cudaStream_t st) {
  D4PG_REQUIRE(b.n > 0 && b.n <= GEMM_MAX_PROBLEMS, D4PG_EINVAL, "gemm_batch_launch: %d problems", b.n);
  for (int i = 0; i < b.n; ++i)     // a concatenated input must switch source on a K-chunk boundary
    D4PG_REQUIRE(b.p[i].mode != GEMM_FWD || b.p[i].K1 == b.p[i].K || b.p[i].K1 % KC == 0, D4PG_ENOTSUP,
                 "gemm_batch_launch: concat split K1=%d must be a multiple of %d", b.p[i].K1, KC);
  D4PG_MAX_CARVEOUT(gemm_ffma_kernel<false>);
  D4PG_MAX_CARVEOUT(gemm_ffma_kernel<true>);
  if (gemm_batch_has_splitk(b)) gemm_ffma_kernel<true><<<b.total_tiles, GEMM_THREADS, 0, st>>>(b);
  else gemm_ffma_kernel<false><<<b.total_tiles, GEMM_THREADS, 0, st>>>(b);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

}  // namespace d4pg
