// Tensor-core grouped GEMM for the actor/critic MLP layers (precision modes 1 = 3xTF32, 2 = 1xTF32).
//
// Same problem descriptors and epilogues as gemm_ffma.cu (models.py:33-40,77-83 forward, autograd
// backward of ddpg.py:230,242), but the contraction runs on the 5th-generation tensor cores:
//   * one CTA = one 128 x 32 output tile; fp32 accumulator in TMEM (32 columns x 128 lanes),
//   * operands staged per 32-deep K chunk into the canonical SWIZZLE_128B UMMA layouts
//     (all K-major: sources that are contiguous along the tile dim are transposed while staged),
//   * 3xTF32: every fp32 operand is split into hi = tf32(x) and lo = tf32(x - hi) while it is
//     staged; D += Ah*Bh + Ah*Bl + Al*Bh gives ~2^-21 relative accuracy, enough for the 1e-5
//     parity bar of config 2 (a single-pass TF32 or BF16 product is not),
//   * operands whose rows are 16-B aligned and K-contiguous (activations, 256-wide weights) are
//     fetched by TMA (cp.async.bulk.tensor, SWIZZLE_128B tensor maps, mbarrier complete_tx) one
//     chunk ahead of the MMAs and split hi/lo in place; ragged operands (|s|=17, the 262-wide
//     critic fc2 rows, transposed uses) are staged by the threads,
//   * a single elected thread issues tcgen05.mma; tcgen05.commit -> mbarrier releases the smem
//     stage (2-stage ring: staging of chunk c+1 overlaps the MMAs of chunk c),
//   * epilogue: tcgen05.ld (one TMEM lane = one output row per thread), bias / ReLU / tanh /
//     activation-derivative masks fused, 128-B row segments stored straight to global.
#include "gemm_ffma.cuh"
#include "tc_common.cuh"
#include <stdlib.h>

namespace d4pg {

using namespace tc;

constexpr int TC_BM = 128, TC_BN = 32, TC_KC = 32;
constexpr int TC_THREADS = 128;
constexpr uint32_t A_BYTES = TC_BM * 128;          // one K-chunk of A (hi or lo): 128 rows x 128 B
constexpr uint32_t B_BYTES = TC_BN * 128;          // one K-chunk of B: 32 rows x 128 B
constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;   // hi + lo for both operands
constexpr int TC_STAGES = 2;
constexpr int BAR_EMPTY = 0, BAR_FULL = TC_STAGES, BAR_DONE = 2 * TC_STAGES, TC_NBARS = 2 * TC_STAGES + 1;
constexpr uint32_t TC_SMEM = TC_STAGES * STAGE_BYTES + 1024 /*alignment slack*/;

// ---- staging into SWIZZLE_128B layouts with the hi/lo split ---------------------------------------
__device__ __forceinline__ void put_split(uint8_t* hi_base, uint8_t* lo_base, uint32_t off, float x) {
  const float h = tf32_hi(x);
  *reinterpret_cast<float*>(hi_base + off) = h;
  *reinterpret_cast<float*>(lo_base + off) = tf32_lo(x, h);
}
__device__ __forceinline__ void put_split4(uint8_t* hi_base, uint8_t* lo_base, uint32_t off, float4 v) {
  float4 h = make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w));
  float4 l = make_float4(tf32_lo(v.x, h.x), tf32_lo(v.y, h.y), tf32_lo(v.z, h.z), tf32_lo(v.w, h.w));
  *reinterpret_cast<float4*>(hi_base + off) = h;
  *reinterpret_cast<float4*>(lo_base + off) = l;
}

// K-major block: rows = M/N index, 32 k per row.  src(row, k) = src[row*ld + k].
template <int ROWS>
__device__ __forceinline__ void stage_kmajor(uint8_t* hi, uint8_t* lo, const float* __restrict__ src, int ld, bool vec,
                                             int row0, int nrows, int k0, int K, int tid) {
  if (vec) {
    // 8 float4 per row; a 16-B chunk keeps its position inside the 128-B row up to the XOR swizzle
#pragma unroll 4
    for (int e = tid; e < ROWS * 8; e += TC_THREADS) {
      const int r = e >> 3, q = e & 7, k = k0 + (q << 2);
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (row0 + r < nrows && k < K) v = __ldg(reinterpret_cast<const float4*>(src + size_t(row0 + r) * ld + k));
      put_split4(hi, lo, sw128_kmajor_off(r, q << 2), v);
    }
  } else {
#pragma unroll 4
    for (int e = tid; e < ROWS * 32; e += TC_THREADS) {
      const int r = e >> 5, kk = e & 31, k = k0 + kk;
      const float x = (row0 + r < nrows && k < K) ? __ldg(src + size_t(row0 + r) * ld + k) : 0.f;
      put_split(hi, lo, sw128_kmajor_off(r, kk), x);
    }
  }
}
// Transposing stage: the source is contiguous along the tile dim (src(k, col) = src[k*ld + col], as in
// dX's W[nout, kin] and dW's dZ[b, nout] / X[b, kin]); it is read coalesced along `col` and written
// into the SAME K-major layout with (row = col, k).  Keeping every operand K-major means a single
// UMMA descriptor form (validated by tests/probe/tc_probe.cu); tf32 MN-major operands would need the
// SWIZZLE_128B_BASE32B layout instead.
template <int COLS>
__device__ __forceinline__ void stage_transposed(uint8_t* hi, uint8_t* lo, const float* __restrict__ src, int ld, bool vec,
                                                 int col0, int ncols, int k0, int K, int tid) {
  if (vec) {
#pragma unroll 4
    for (int e = tid; e < 32 * (COLS / 4); e += TC_THREADS) {
      const int kk = e / (COLS / 4), col = (e % (COLS / 4)) << 2;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (k0 + kk < K && col0 + col < ncols) v = __ldg(reinterpret_cast<const float4*>(src + size_t(k0 + kk) * ld + col0 + col));
      put_split(hi, lo, sw128_kmajor_off(col, kk), v.x);
      put_split(hi, lo, sw128_kmajor_off(col + 1, kk), v.y);
      put_split(hi, lo, sw128_kmajor_off(col + 2, kk), v.z);
      put_split(hi, lo, sw128_kmajor_off(col + 3, kk), v.w);
    }
  } else {
#pragma unroll 4
    for (int e = tid; e < 32 * COLS; e += TC_THREADS) {
      const int kk = e / COLS, col = e % COLS;
      const float x = (k0 + kk < K && col0 + col < ncols) ? __ldg(src + size_t(k0 + kk) * ld + col0 + col) : 0.f;
      put_split(hi, lo, sw128_kmajor_off(col, kk), x);
    }
  }
}

// TMA landed raw fp32 in `hi`; rewrite it as hi and emit lo at the same (already swizzled) offsets
template <int BYTES>
__device__ __forceinline__ void split_in_place(uint8_t* hi, uint8_t* lo, int tid) {
#pragma unroll 4
  for (int e = tid; e < BYTES / 16; e += TC_THREADS) {
    const float4 v = *reinterpret_cast<const float4*>(hi + e * 16);
    put_split4(hi, lo, uint32_t(e) * 16u, v);
  }
}

template <int MODE>
__device__ __forceinline__ void tc_tile(const GemmProblem& P, const CUtensorMap* tmA, const CUtensorMap* tmB,
                                        uint8_t* smem, uint64_t* bars, uint32_t tmem_d,
                                        int m0, int n0, int tn, int passes) {
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  constexpr bool A_T = (MODE == GEMM_DW);       // source contiguous along the tile dim -> transposing stage
  constexpr bool B_T = (MODE != GEMM_FWD);
  const uint32_t idesc = make_idesc(FMT_TF32, false, false, TC_BM, TC_BN);
  const bool avec = (P.flags & GEMM_A_VEC) != 0, bvec = (P.flags & GEMM_B_VEC) != 0;
  const bool a_tma = (P.flags & GEMM_A_TMA) != 0, b_tma = (P.flags & GEMM_B_TMA) != 0;
  const int nchunks = (P.K + TC_KC - 1) / TC_KC;
  uint64_t* empty = bars + BAR_EMPTY;  // [TC_STAGES]  MMAs that read a stage have completed
  uint64_t* full = bars + BAR_FULL;    // [TC_STAGES]  TMA bytes of a stage have landed
  uint64_t* done = bars + BAR_DONE;    // all MMAs of the tile have completed

  // TMA for chunk c (thread 0): A from the main source only (the concat tail is staged by threads)
  auto issue_tma = [&](int c) {
    const int st = c % TC_STAGES, k0 = c * TC_KC;
    uint8_t* Ahi = smem + st * STAGE_BYTES;
    uint8_t* Bhi = Ahi + 2 * A_BYTES;
    const bool a_now = a_tma && k0 < P.K1, b_now = b_tma;
    if (!(a_now || b_now)) return;
    mbar_expect_tx(&full[st], (a_now ? A_BYTES : 0u) + (b_now ? B_BYTES : 0u));
    if (a_now) tma_load_2d(Ahi, tmA, &full[st], k0, m0);
    if (b_now) tma_load_2d(Bhi, tmB, &full[st], k0, n0);
  };
  if (tid == 0 && (a_tma || b_tma)) issue_tma(0);
  uint32_t full_parity[TC_STAGES] = {0u, 0u};      // per-stage phase of the TMA barrier (not every chunk uses it)

  for (int c = 0; c < nchunks; ++c) {
    const int st = c % TC_STAGES;
    uint8_t* Ahi = smem + st * STAGE_BYTES;
    uint8_t* Alo = Ahi + A_BYTES;
    uint8_t* Bhi = Alo + A_BYTES;
    uint8_t* Blo = Bhi + B_BYTES;
    const int k0 = c * TC_KC;
    // the other stage is reused by chunk c+1: wait until the MMAs of chunk c-1 have drained it, then
    // let the TMA of chunk c+1 fly while this chunk is staged / split / multiplied
    if (c + 1 < nchunks) {
      if (c + 1 >= TC_STAGES) mbar_wait(&empty[(c + 1) % TC_STAGES], (((c + 1) / TC_STAGES) - 1) & 1);
      if (tid == 0 && (a_tma || b_tma)) issue_tma(c + 1);
    }
    const bool a_now = a_tma && k0 < P.K1;
    // ---- thread-staged operands -----------------------------------------------------------------
    if (!a_now) {
      if (A_T) stage_transposed<TC_BM>(Ahi, Alo, P.A, P.lda, avec, m0, P.M, k0, P.K, tid);              // dZ[k*lda + m]
      else if (k0 >= P.K1) stage_kmajor<TC_BM>(Ahi, Alo, P.A2, P.lda2, false, m0, P.M, k0 - P.K1, P.K - P.K1, tid);
      else stage_kmajor<TC_BM>(Ahi, Alo, P.A, P.lda, avec, m0, P.M, k0, P.K1, tid);
    }
    if (!b_tma) {
      if (B_T) stage_transposed<TC_BN>(Bhi, Blo, P.Bm, P.ldb, bvec, n0, P.N, k0, P.K, tid);             // B[k*ldb + n]
      else stage_kmajor<TC_BN>(Bhi, Blo, P.Bm, P.ldb, bvec, n0, P.N, k0, P.K, tid);                     // W[n*ldb + k]
    }
    // ---- TMA-fed operands: wait for the bytes, split hi/lo in place --------------------------------
    if (a_now || b_tma) {
      mbar_wait(&full[st], full_parity[st]);
      full_parity[st] ^= 1u;
      if (passes > 1) {
        if (a_now) split_in_place<A_BYTES>(Ahi, Alo, tid);
        if (b_tma) split_in_place<B_BYTES>(Bhi, Blo, tid);
      }
    }
    fence_proxy_async();
    __syncthreads();
    if (tid == 0) {
      tc_fence_after_sync();
#pragma unroll 1
      for (int p = 0; p < passes; ++p) {
        const uint8_t* Ap = (p == 2) ? Alo : Ahi;
        const uint8_t* Bp = (p == 1) ? Blo : Bhi;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint64_t ad = make_smem_desc(smem_u32(Ap + ks * 32), 16, 1024);
          const uint64_t bd = make_smem_desc(smem_u32(Bp + ks * 32), 16, 1024);
          mma_tf32(tmem_d, ad, bd, idesc, (c | p | ks) != 0);
        }
      }
      mma_commit(&empty[st]);
      if (c == nchunks - 1) mma_commit(done);
    }
  }
  mbar_wait(done, 0);
  tc_fence_after_sync();

  // ---- epilogue: one TMEM lane (= output row) per thread, 32 columns ------------------------------
  float r[32];
  tmem_ld_32x32(tmem_d + (uint32_t(warp * 32) << 16), r);
  const int gi = m0 + warp * 32 + lane;
  if (gi < P.M) {
    float* crow = P.C + size_t(gi) * P.ldc + n0;
    const float* arow = P.aux ? P.aux + size_t(gi) * P.ldaux + n0 : nullptr;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      if (n0 + j >= P.N) break;
      float x = r[j];
      switch (P.epi) {
        case EPI_BIAS: x += __ldg(P.bias + n0 + j); break;
        case EPI_BIAS_RELU: x = fmaxf(x + __ldg(P.bias + n0 + j), 0.f); break;
        case EPI_BIAS_TANH: x = tanhf(x + __ldg(P.bias + n0 + j)); break;
        case EPI_RELU_MASK: x = (__ldg(arow + j) > 0.f) ? x : 0.f; break;
        case EPI_TANH_MASK: { const float t = __ldg(arow + j); x *= (1.f - t * t); } break;
        default: break;
      }
      crow[j] = x;
    }
  }
  // ---- dW: bias gradient = column sums of dZ (rows of A), exact fp32, tn == 0 tiles only -------------
  if (MODE == GEMM_DW && P.bias_grad != nullptr && tn == 0) {
    const int m = m0 + tid;                                   // 128 threads <-> 128 A rows
    if (m < P.M) {
      float s = 0.f;
      for (int k = 0; k < P.K; ++k) s += __ldg(P.A + size_t(k) * P.lda + m);    // coalesced across threads
      P.bias_grad[m] = s;
    }
  }
}

__global__ void __launch_bounds__(TC_THREADS) gemm_tc_kernel(const __grid_constant__ GemmBatch batch, int passes) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  __shared__ __align__(8) uint64_t bars[TC_NBARS];
  __shared__ uint32_t tmem_base_s;

  int pi = 0;
#pragma unroll
  for (int i = 1; i < GEMM_MAX_PROBLEMS; ++i)
    if (i < batch.n && int(blockIdx.x) >= batch.p[i].tile_begin) pi = i;
  const GemmProblem P = batch.p[pi];
  const int tile = blockIdx.x - P.tile_begin;
  const int tm = tile / P.tiles_n, tn = tile - tm * P.tiles_n;

  if (threadIdx.x < 32) tmem_alloc(&tmem_base_s, 32);
  if (threadIdx.x == 32) {
    for (int i = 0; i < TC_NBARS; ++i) mbar_init(&bars[i], 1);
    mbar_fence_init();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_d = tmem_base_s;

  const CUtensorMap* tmA = &batch.tmap_a[pi];
  const CUtensorMap* tmB = &batch.tmap_b[pi];
  if (P.mode == GEMM_FWD) tc_tile<GEMM_FWD>(P, tmA, tmB, smem, bars, tmem_d, tm * TC_BM, tn * TC_BN, tn, passes);
  else if (P.mode == GEMM_DX) tc_tile<GEMM_DX>(P, tmA, tmB, smem, bars, tmem_d, tm * TC_BM, tn * TC_BN, tn, passes);
  else tc_tile<GEMM_DW>(P, tmA, tmB, smem, bars, tmem_d, tm * TC_BM, tn * TC_BN, tn, passes);

  tc_fence_before_sync();
  __syncthreads();
  if (threadIdx.x < 32) tmem_dealloc(tmem_d, 32);
}

// =====================================================================================================
// v2: warp-specialised, every operand TMA-fed (needs 16-B row pitches -- the learner's own buffers).
//   warp 0      : TMA producer (one lane): S-deep ring of raw fp32 chunks, one mbarrier per stage
//   warp 1      : TMEM owner + the single MMA-issuing lane
//   warps 2..5  : "converters": split each landed chunk into tf32 hi (in place) / lo (2-stage ring),
//                 then the epilogue (each warp owns the TMEM lane quadrant warp%4)
// Operands that are contiguous along the tile dim (dX's W, dW's dZ and X) are loaded with the
// SWIZZLE_128B_ATOM_32B tensor-map mode and fed to the MMA as MN-major (SWIZZLE_128B_BASE32B
// descriptors, validated by tests/probe/tc_probe.cu); the split is layout-agnostic (flat float4).
// =====================================================================================================
constexpr int T2_BM = 128, T2_BN = 64, T2_KC = 32;
constexpr int T2_THREADS = 192;
constexpr int T2_STAGES = 6;
constexpr uint32_t T2_A_BYTES = T2_BM * 128, T2_B_BYTES = T2_BN * 128;          // 16 KB + 8 KB per chunk
constexpr uint32_t T2_STAGE = T2_A_BYTES + T2_B_BYTES;
constexpr uint32_t T2_SMEM = T2_STAGES * T2_STAGE + 2 * T2_STAGE + 1024;
constexpr int T2_FULL = 0, T2_CONV = T2_STAGES, T2_EMPTY = 2 * T2_STAGES, T2_LOEMPTY = 3 * T2_STAGES,
              T2_DONE = 3 * T2_STAGES + 2, T2_NBARS = 3 * T2_STAGES + 3;

__device__ __forceinline__ unsigned long long gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
#define TRACE(slot) do { if (batch.trace && blockIdx.x == 0) batch.trace[slot] = gtime(); } while (0)

__global__ void __launch_bounds__(T2_THREADS, 1) gemm_tc2_kernel(const __grid_constant__ GemmBatch batch, int passes) {
  extern __shared__ uint8_t smem_raw[];
  if (threadIdx.x == 0) TRACE(0);
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* lo_ring = smem + T2_STAGES * T2_STAGE;
  __shared__ __align__(8) uint64_t bars[T2_NBARS];
  __shared__ uint32_t tmem_base_s;

  int pi = 0;
#pragma unroll
  for (int i = 1; i < GEMM_MAX_PROBLEMS; ++i)
    if (i < batch.n && int(blockIdx.x) >= batch.p[i].tile_begin) pi = i;
  const GemmProblem P = batch.p[pi];
  const int tile = blockIdx.x - P.tile_begin;
  const int per_slice = P.tiles_m * P.tiles_n;
  const int kslice_id = tile / per_slice, tile2 = tile - kslice_id * per_slice;
  const int tm = tile2 / P.tiles_n, tn = tile2 - tm * P.tiles_n;
  const int m0 = tm * T2_BM, n0 = tn * T2_BN;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const bool a_mn = (P.mode == GEMM_DW), b_mn = (P.mode != GEMM_FWD);
  // split-K (dW over a large batch): this CTA contracts K chunks [c_beg, c_beg + nchunks)
  const int kbeg = kslice_id * P.kslice, kend = min(P.K, kbeg + P.kslice);
  const int c_beg = kbeg / T2_KC;
  const int nchunks = (kend - kbeg + T2_KC - 1) / T2_KC;
  const bool split = P.ksplit > 1;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < T2_NBARS; ++i) mbar_init(&bars[i], (i >= T2_CONV && i < T2_CONV + T2_STAGES) ? 4u : 1u);
    mbar_fence_init();
    tma_prefetch_desc(&batch.tmap_a[pi]);
    tma_prefetch_desc(&batch.tmap_b[pi]);
  }
  if (warp == 1) tmem_alloc(&tmem_base_s, 64);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_d = tmem_base_s;
  if (threadIdx.x == 0) TRACE(1);

  if (warp == 0) {
    // ================================ TMA producer ==================================================
    if (lane == 0) {
      for (int c = 0; c < nchunks; ++c) {
        const int s = c % T2_STAGES, k0 = (c_beg + c) * T2_KC;
        if (c >= T2_STAGES) mbar_wait(&bars[T2_EMPTY + s], ((c / T2_STAGES) - 1) & 1);
        uint8_t* Ad = smem + s * T2_STAGE;
        uint8_t* Bd = Ad + T2_A_BYTES;
        uint64_t* full = &bars[T2_FULL + s];
        mbar_expect_tx(full, T2_STAGE);
        if (a_mn) {
#pragma unroll
          for (int j = 0; j < 4; ++j) tma_load_2d(Ad + j * 4096, &batch.tmap_a[pi], full, m0 + 32 * j, k0);
        } else if (k0 >= P.K1) {
          tma_load_2d(Ad, &batch.tmap_a2[pi], full, k0 - P.K1, m0);
        } else {
          tma_load_2d(Ad, &batch.tmap_a[pi], full, k0, m0);
        }
        if (b_mn) {
#pragma unroll
          for (int j = 0; j < 2; ++j) tma_load_2d(Bd + j * 4096, &batch.tmap_b[pi], full, n0 + 32 * j, k0);
        } else {
          tma_load_2d(Bd, &batch.tmap_b[pi], full, k0, n0);
        }
        if (c == 0) TRACE(2);
      }
      TRACE(3);
    }
  } else if (warp == 1) {
    // ================================ MMA issuer =====================================================
    if (lane == 0) {
      const uint32_t idesc = make_idesc(FMT_TF32, a_mn, b_mn, T2_BM, T2_BN);
      // The issuing lane is a single thread: keep its per-MMA work to a couple of integer adds.  A
      // descriptor is (template with LBO/SBO/layout bits) + (byte address >> 4) in the low 14 bits;
      // stepping K by one MMA adds 32 B (K-major) or 1024 B (MN-major) to the start address.
      const uint64_t a_tmpl = a_mn ? make_smem_desc(0, 4096, 512, 1) : make_smem_desc(0, 16, 1024, 2);
      const uint64_t b_tmpl = b_mn ? make_smem_desc(0, 4096, 512, 1) : make_smem_desc(0, 16, 1024, 2);
      const uint32_t a_step = (a_mn ? 1024u : 32u) >> 4, b_step = (b_mn ? 1024u : 32u) >> 4;
      const uint32_t smem_base = smem_u32(smem) >> 4, lo_base = smem_u32(lo_ring) >> 4;
      for (int c = 0; c < nchunks; ++c) {
        const int s = c % T2_STAGES, l = c & 1;
        mbar_wait(&bars[(passes > 1 ? T2_CONV : T2_FULL) + s], (c / T2_STAGES) & 1);
        tc_fence_after_sync();
        const uint32_t ahi = smem_base + uint32_t(s) * (T2_STAGE >> 4), bhi = ahi + (T2_A_BYTES >> 4);
        const uint32_t alo = lo_base + uint32_t(l) * (T2_STAGE >> 4), blo = alo + (T2_A_BYTES >> 4);
#pragma unroll
        for (int ks = 0; ks < 4; ++ks)
          mma_tf32(tmem_d, a_tmpl + (ahi + ks * a_step), b_tmpl + (bhi + ks * b_step), idesc, (c | ks) != 0);
        if (passes > 1) {
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            mma_tf32(tmem_d, a_tmpl + (ahi + ks * a_step), b_tmpl + (blo + ks * b_step), idesc, true);
#pragma unroll
          for (int ks = 0; ks < 4; ++ks)
            mma_tf32(tmem_d, a_tmpl + (alo + ks * a_step), b_tmpl + (bhi + ks * b_step), idesc, true);
        }
        mma_commit(&bars[T2_EMPTY + s]);
        if (passes > 1) mma_commit(&bars[T2_LOEMPTY + l]);
        if (c == 0) TRACE(6);
      }
      mma_commit(&bars[T2_DONE]);
      TRACE(7);
    }
  } else {
    // ================================ converters, then epilogue =======================================
    const int t2 = tid - 64;                       // 0..127
    if (passes > 1) {
      for (int c = 0; c < nchunks; ++c) {
        const int s = c % T2_STAGES, l = c & 1;
        uint8_t* hi = smem + s * T2_STAGE;
        uint8_t* lo = lo_ring + l * T2_STAGE;
        mbar_wait(&bars[T2_FULL + s], (c / T2_STAGES) & 1);
        if (c == 0 && t2 == 0) TRACE(4);
        if (c >= 2) mbar_wait(&bars[T2_LOEMPTY + l], ((c >> 1) - 1) & 1);
        constexpr int PER = int(T2_STAGE / 16) / 128;        // 12 float4 per thread per chunk
        float4 v[PER];
#pragma unroll
        for (int q = 0; q < PER; ++q) v[q] = *reinterpret_cast<const float4*>(hi + (t2 + q * 128) * 16);
#pragma unroll
        for (int q = 0; q < PER; ++q) put_split4(hi, lo, uint32_t(t2 + q * 128) * 16u, v[q]);
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars[T2_CONV + s]);
        if (c == 0 && t2 == 0) TRACE(5);
      }
    }
    if (t2 == 0) TRACE(8);
    mbar_wait(&bars[T2_DONE], 0);
    tc_fence_after_sync();
    if (t2 == 0) TRACE(9);
    const int quad = warp & 3;
    const int gi = m0 + quad * 32 + lane;
#pragma unroll 1
    for (int half = 0; half < 2; ++half) {
      float r[32];
      tmem_ld_32x32(tmem_d + (uint32_t(quad * 32) << 16) + uint32_t(half * 32), r);
      const int nb = n0 + half * 32;
      if (gi < P.M && nb < P.N) {
        float* crow = P.C + size_t(gi) * P.ldc + nb;
        const float* arow = P.aux ? P.aux + size_t(gi) * P.ldaux + nb : nullptr;
        // 16-B row pitches: whole float4 groups inside [0, N) go out as 128-bit accesses
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const int j = j4 * 4;
          if (nb + j >= P.N) break;
          const bool full4 = (nb + j + 3 < P.N);
          float x[4] = {r[j], r[j + 1], r[j + 2], r[j + 3]};
          float ex[4] = {0.f, 0.f, 0.f, 0.f};
          if (P.epi == EPI_BIAS || P.epi == EPI_BIAS_RELU || P.epi == EPI_BIAS_TANH) {
            if (full4) { const float4 b4 = __ldg(reinterpret_cast<const float4*>(P.bias + nb + j)); ex[0] = b4.x; ex[1] = b4.y; ex[2] = b4.z; ex[3] = b4.w; }
            else for (int q = 0; q < 4; ++q) if (nb + j + q < P.N) ex[q] = __ldg(P.bias + nb + j + q);
          } else if (P.epi == EPI_RELU_MASK || P.epi == EPI_TANH_MASK) {
            if (full4) { const float4 a4 = __ldg(reinterpret_cast<const float4*>(arow + j)); ex[0] = a4.x; ex[1] = a4.y; ex[2] = a4.z; ex[3] = a4.w; }
            else for (int q = 0; q < 4; ++q) if (nb + j + q < P.N) ex[q] = __ldg(arow + j + q);
          }
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            switch (P.epi) {
              case EPI_BIAS: x[q] += ex[q]; break;
              case EPI_BIAS_RELU: x[q] = fmaxf(x[q] + ex[q], 0.f); break;
              case EPI_BIAS_TANH: x[q] = tanhf(x[q] + ex[q]); break;
              case EPI_RELU_MASK: x[q] = (ex[q] > 0.f) ? x[q] : 0.f; break;
              case EPI_TANH_MASK: x[q] *= (1.f - ex[q] * ex[q]); break;
              default: break;
            }
          }
          if (split) { for (int q = 0; q < 4; ++q) if (nb + j + q < P.N) atomicAdd(crow + j + q, x[q]); }   // C pre-zeroed
          else if (full4) *reinterpret_cast<float4*>(crow + j) = make_float4(x[0], x[1], x[2], x[3]);
          else for (int q = 0; q < 4; ++q) if (nb + j + q < P.N) crow[j + q] = x[q];
        }
      }
    }
    if (P.mode == GEMM_DW && P.bias_grad != nullptr && tn == 0) {       // bias gradient: column sums of dZ
      const int m = m0 + t2;
      if (m < P.M) {
        float sacc = 0.f;
        for (int k = kbeg; k < kend; ++k) sacc += __ldg(P.A + size_t(k) * P.lda + m);
        if (split) atomicAdd(P.bias_grad + m, sacc);
        else P.bias_grad[m] = sacc;
      }
    }
  }
  if (tid == 64) TRACE(10);
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_d, 64);
  if (threadIdx.x == 32) TRACE(11);
}

// ---- host: TMA descriptors -------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn get_encoder() {
  static EncodeTiledFn fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}
// [rows x inner] fp32, row pitch ld floats, box = 32 x box_rows, 128-B swizzle, zero fill out of bounds
static bool encode_kmajor(CUtensorMap* tm, const float* base, int inner, int rows, int ld, int box_rows) {
  EncodeTiledFn enc = get_encoder();
  if (!enc) return false;
  cuuint64_t dims[2] = {cuuint64_t(inner), cuuint64_t(rows)};
  cuuint64_t strides[1] = {cuuint64_t(ld) * 4};
  cuuint32_t box[2] = {32, cuuint32_t(box_rows)};
  cuuint32_t estr[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// [k rows x mn cols] fp32 source that is contiguous along the tile dim: box = 32 mn x 32 k rows,
// SWIZZLE_128B_ATOM_32B (what the MN-major tf32 UMMA descriptor expects)
static bool encode_mnmajor(CUtensorMap* tm, const float* base, int mn, int krows, int ld) {
  EncodeTiledFn enc = get_encoder();
  if (!enc) return false;
  cuuint64_t dims[2] = {cuuint64_t(mn), cuuint64_t(krows)};
  cuuint64_t strides[1] = {cuuint64_t(ld) * 4};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  return enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
static bool tma_ok(const float* p, int ld) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0 && ld % 4 == 0; }

// v2 eligibility: every operand of every problem can be described by a tensor map
static bool prepare_v2(GemmBatch& b) {
  for (int i = 0; i < b.n; ++i) {
    const GemmProblem& p = b.p[i];
    if (!tma_ok(p.A, p.lda) || !tma_ok(p.Bm, p.ldb)) return false;
    if (!tma_ok(p.C, p.ldc) || (p.aux && !tma_ok(p.aux, p.ldaux))) return false;      // 128-bit epilogue accesses
    if (p.bias && (reinterpret_cast<uintptr_t>(p.bias) & 15)) return false;
    bool ok;
    if (p.mode == GEMM_DW) ok = encode_mnmajor(&b.tmap_a[i], p.A, p.M, p.K, p.lda);
    else ok = encode_kmajor(&b.tmap_a[i], p.A, p.K1, p.M, p.lda, T2_BM);
    if (ok && p.mode == GEMM_FWD && p.K1 < p.K)
      ok = tma_ok(p.A2, p.lda2) && p.K1 % T2_KC == 0 && encode_kmajor(&b.tmap_a2[i], p.A2, p.K - p.K1, p.M, p.lda2, T2_BM);
    if (ok) ok = (p.mode == GEMM_FWD) ? encode_kmajor(&b.tmap_b[i], p.Bm, p.K, p.N, p.ldb, T2_BN)
                                      : encode_mnmajor(&b.tmap_b[i], p.Bm, p.N, p.K, p.ldb);
    if (!ok) return false;
  }
  return true;
}

// Decide per operand whether TMA may fetch it (K-contiguous source, 16-B aligned rows) and encode the maps.
static unsigned long long* g_trace = nullptr;
unsigned long long* debug_trace_buffer() {
  static const bool tracing = getenv("D4PG_TC_TRACE") != nullptr;
  if (tracing && !g_trace) { cudaMalloc(&g_trace, 512 * sizeof(unsigned long long)); cudaMemset(g_trace, 0, 512 * 8); }
  return tracing ? g_trace : nullptr;
}
void gemm_tc_prepare(GemmBatch& b) {
  b.trace = debug_trace_buffer();
  b.all_tma = prepare_v2(b) ? 1 : 0;
  if (b.all_tma) { gemm_batch_retile(b, T2_BM, T2_BN); return; }
  for (int i = 0; i < b.n; ++i) { b.p[i].ksplit = 1; b.p[i].kslice = b.p[i].K; }    // v1 kernel has no split-K
  gemm_batch_retile(b, TC_BM, TC_BN);
  for (int i = 0; i < b.n; ++i) {
    GemmProblem& p = b.p[i];
    p.flags &= ~(GEMM_A_TMA | GEMM_B_TMA);
    if (p.mode != GEMM_DW && tma_ok(p.A, p.lda) && encode_kmajor(&b.tmap_a[i], p.A, p.K1, p.M, p.lda, TC_BM))
      p.flags |= GEMM_A_TMA;
    if (p.mode == GEMM_FWD && tma_ok(p.Bm, p.ldb) && encode_kmajor(&b.tmap_b[i], p.Bm, p.K, p.N, p.ldb, TC_BN))
      p.flags |= GEMM_B_TMA;
  }
}

int gemm_tc_batch_launch(const GemmBatch& b, int passes, cudaStream_t st) {
  D4PG_REQUIRE(b.n > 0 && b.n <= GEMM_MAX_PROBLEMS, D4PG_EINVAL, "gemm_tc_batch_launch: %d problems", b.n);
  for (int i = 0; i < b.n; ++i)
    D4PG_REQUIRE(b.p[i].mode != GEMM_FWD || b.p[i].K1 == b.p[i].K || b.p[i].K1 % TC_KC == 0, D4PG_ENOTSUP,
                 "gemm_tc_batch_launch: concat split K1=%d must be a multiple of %d", b.p[i].K1, TC_KC);
  static bool attr_set = false;
  if (!attr_set) {
    D4PG_CUDA_OK(cudaFuncSetAttribute(gemm_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(TC_SMEM)));
    D4PG_CUDA_OK(cudaFuncSetAttribute(gemm_tc2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(T2_SMEM)));
    D4PG_MAX_CARVEOUT(gemm_tc_kernel);
    D4PG_MAX_CARVEOUT(gemm_tc2_kernel);
    attr_set = true;
  }
  if (b.all_tma) gemm_tc2_kernel<<<b.total_tiles, T2_THREADS, T2_SMEM, st>>>(b, passes);
  else gemm_tc_kernel<<<b.total_tiles, TC_THREADS, TC_SMEM, st>>>(b, passes);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

}  // namespace d4pg

// debug: %globaltimer (ns) phase stamps of CTA 0 of the last gemm_tc2 launch (D4PG_TC_TRACE=1)
extern "C" int32_t d4pg_debug_trace_read(unsigned long long* out, int32_t n) {
  if (!d4pg::g_trace || !out || n < 1 || n > 512) return D4PG_ESTATE;
  D4PG_CUDA_OK(cudaMemcpy(out, d4pg::g_trace, size_t(n) * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return D4PG_OK;
}
extern "C" int32_t d4pg_debug_tc_trace(unsigned long long* out16) {
  if (!d4pg::g_trace || !out16) return D4PG_ESTATE;
  D4PG_CUDA_OK(cudaMemcpy(out16, d4pg::g_trace, 32 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
  return D4PG_OK;
}
