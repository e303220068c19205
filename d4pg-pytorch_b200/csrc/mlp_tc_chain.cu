// tcgen05 cluster chains: every dependent layer of an actor/critic network chain in ONE launch, each layer a
// tcgen05.mma (UTCHMMA) tile with a TMEM accumulator, operands brought in by TMA bulk copies.
//
// Reference ops: actor.forward / critic.forward (models.py:32-41,76-88) for the five forward passes of
// DDPG.train (ddpg.py:205-208,236) and the two backward passes of ddpg.py:230,242 (dX only; dW is gemm_wide).
//
// Decomposition.  A thread-block CLUSTER of 8 CTAs owns 64 batch rows (UMMA M = 64) for a whole chain.  CTA r
// owns output features [32r, 32r+32) of every 256-wide layer (UMMA N = 32), so a layer is eight 64x32xK tiles
// and the layer-to-layer dependency is an all-gather of the 64x256 activation plane inside the cluster.
//
// Precision.  3xTF32: x = hi + lo, hi = x with the low 13 mantissa bits cleared, lo = tf32(x - hi);
// D += Al*Bh + Ah*Bl + Ah*Bh with fp32 accumulation in TMEM (~2^-21 relative, meets the 1e-5 parity bar).
// Nothing is split on the critical path:
//   * weights: hi/lo parts are PRE-PACKED once per step (tcc_pack_kernel, right after Adam changed them) into the
//     exact shared-memory image the MMA reads (K-major SWIZZLE_128B, 32x32 blocks) -- for the backward pass the
//     transposed image -- so a CTA's weight slice of a layer is ONE contiguous cp.async.bulk;
//   * activations: the epilogue that PRODUCES a layer output (tcgen05.ld -> bias/ReLU/tanh/mask) writes it three
//     times: row-major fp32 (for the loss kernel / dW), and as hi and lo images of its 64x32 tile = K-chunk r of
//     the next layer's A operand, already swizzled.  The consumers fetch chunk c with one 16-KB cp.async.bulk.
//
// Per CTA: warp 0 = loader (one lane issues every bulk copy: weight slice one slot ahead, A chunks into an
// 8-deep ring, completion on mbarriers by byte count), warp 1 = TMEM owner + the single MMA-issuing lane (12
// tcgen05.mma per 32-deep chunk and group; tcgen05.commit releases ring buffers and signals the accumulator),
// warps 2..9 = epilogue (lane quarter = warp % 4, 16 accumulator columns each).  A slot boundary is a cluster
// barrier (arrive.release / wait.acquire): outputs in L2 are visible, ring and weight buffers are free.
#include "mlp_tc_chain.cuh"
#include "tc_common.cuh"
#include <stdlib.h>
#include <string.h>

namespace d4pg {

using namespace tc;

// shared-memory map (bytes from the 1024-B aligned base)
constexpr uint32_t TCC_OFF_A = 0;
constexpr uint32_t TCC_OFF_W = TCC_ABUFS * TCC_A_CHUNK;
constexpr uint32_t TCC_OFF_BAR = TCC_OFF_W + TCC_MAX_CHUNKS * TCC_W_CHUNK;
constexpr uint32_t TCC_SMEM = TCC_OFF_BAR + 256 + 1024;      // barriers + alignment slack
constexpr int TCC_TMEM_COLS = TCC_MAX_GROUPS * 2 * TCC_BN; // one 128-lane x 64-column fp32 accumulator per group
constexpr int TCC_TRACE_PER_SLOT = 12;

__device__ __forceinline__ void tcc_cluster_arrive() { asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory"); }
__device__ __forceinline__ void tcc_cluster_wait() { asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory"); }
__device__ __forceinline__ unsigned tcc_ctarank() {
  unsigned r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ unsigned long long tcc_gtime() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// 1-D bulk copy global -> this CTA's shared memory, completion by byte count on an mbarrier
__device__ __forceinline__ void tcc_bulk_load(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
// Watchdog: every mbarrier wait of this kernel is bounded (~2 s of SM clocks).  A protocol bug then ends the launch
// with a trap and a record in HOST-mapped memory (readable after the context died: d4pg_debug_watchdog) instead of
// hanging the GPU.  record[0] = 1, [1] = code | slot << 8 | rank << 16 | parity << 24 | block << 32, [2] = seq / nact.
__device__ __forceinline__ void tcc_wait(uint64_t* bar, uint32_t parity, unsigned long long* dbg, unsigned code, unsigned aux) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  bool recorded = false;
  while (!mbar_try_wait(bar, parity)) {
    const long long dt = clock64() - t0;
    if (dt > 4000000000ll && !recorded) {
      recorded = true;
      if (dbg) {
        if (atomicCAS(dbg, 0ull, 1ull) == 0ull) {           // the first wait that timed out anywhere
          dbg[1] = (unsigned long long)code | ((unsigned long long)parity << 24) | ((unsigned long long)blockIdx.x << 32);
          dbg[2] = aux;
        }
        const unsigned kind = code & 0xFFu;                 // and the first one of every kind (5 kinds, 2 words each)
        if (kind < 6 && atomicCAS(dbg + 4 + 2 * kind, 0ull, 1ull) == 0ull) {
          dbg[4 + 2 * kind] = (unsigned long long)code | ((unsigned long long)parity << 24) | ((unsigned long long)blockIdx.x << 32);
          dbg[5 + 2 * kind] = aux;
        }
        __threadfence_system();
      }
    }
    if (dt > 5000000000ll) __trap();                        // every stuck waiter had time to leave its record
  }
}
#define TCC_CODE(kind, slot, rank) (unsigned(kind) | (unsigned(slot) << 8) | (unsigned(rank) << 16))
enum { WD_LOADER_DFULL = 2, WD_MMA_WFULL = 3, WD_MMA_FULL = 4, WD_EPI_DFULL = 5 };

// The MMA-issuing code runs WARP-UNIFORM (all 32 lanes execute the loop with identical values, so descriptors live in
// uniform registers) and only the instruction is predicated on an elected lane: measured on B200 (tests/probe/
// mma_probe2.cu) 25 cycles per 64x32x8 tcgen05.mma this way vs 50 from a single-lane branch and 150+ with per-thread
// integer arithmetic (R2UR round trips) in the loop.
// The descriptors are passed as their LOW words (start address >> 4 | LBO << 16); the high word of a K-major
// SWIZZLE_128B descriptor (SBO = 1024, version 1, layout 2) is the constant 0x40004040, so the compiler moves two
// instead of four values into uniform registers per instruction.
constexpr uint32_t TCC_DESC_HI = 0x40004040u;
constexpr uint32_t TCC_DESC_LO = 1u << 16;                 // LBO = 16 bytes (unused by swizzled K-major layouts)
__device__ __forceinline__ void tcc_mma_elect(uint32_t tmem_d, uint32_t adesc_lo, uint32_t bdesc_lo, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, q;\n\t.reg .b64 da, db;\n\t"
      "mov.b64 da, {%1, %5};\n\t"
      "mov.b64 db, {%2, %5};\n\t"
      "elect.sync _|q, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], da, db, %3, p;\n\t}"
      ::"r"(tmem_d), "r"(adesc_lo), "r"(bdesc_lo), "r"(idesc), "r"(accumulate), "r"(TCC_DESC_HI) : "memory");
}
__device__ __forceinline__ void tcc_commit_elect(uint64_t* bar) {
  asm volatile(
      "{\n\t.reg .pred q;\n\telect.sync _|q, 0xffffffff;\n\t"
      "@q tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(smem_u32(bar)) : "memory");
}

// 32 lanes x 16 columns of fp32 accumulators (no wait: several loads may be in flight, then tcc_tmem_ld_wait)
__device__ __forceinline__ void tcc_tmem_ld16(uint32_t taddr, float (&r)[16]) {
  uint32_t* u = reinterpret_cast<uint32_t*>(r);
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(u[0]), "=r"(u[1]), "=r"(u[2]), "=r"(u[3]), "=r"(u[4]), "=r"(u[5]), "=r"(u[6]), "=r"(u[7]),
        "=r"(u[8]), "=r"(u[9]), "=r"(u[10]), "=r"(u[11]), "=r"(u[12]), "=r"(u[13]), "=r"(u[14]), "=r"(u[15])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tcc_tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

__device__ __forceinline__ float4 tcc_hi4(float4 v) { return make_float4(tf32_hi(v.x), tf32_hi(v.y), tf32_hi(v.z), tf32_hi(v.w)); }
__device__ __forceinline__ float4 tcc_lo4(float4 v, float4 h) {
  return make_float4(tf32_lo(v.x, h.x), tf32_lo(v.y, h.y), tf32_lo(v.z, h.z), tf32_lo(v.w, h.w));
}

// [64 rows x 32 k] chunk of a row-major fp32 array -> hi / lo SWIZZLE_128B K-major images (256 epilogue threads)
__device__ __forceinline__ void tcc_convert_chunk(uint8_t* dst, const float* __restrict__ src, int ld, int k0, int ncols,
                                                  int m0, int B, int et) {
#pragma unroll
  for (int p = 0; p < 2; ++p) {
    const int e = et + p * 256, row = e >> 3, u = e & 7, k = k0 + (u << 2);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (m0 + row < B && k < ncols) {
      v = __ldg(reinterpret_cast<const float4*>(src + size_t(m0 + row) * ld + k));     // ld is a multiple of 4 >= ncols
      if (k + 1 >= ncols) v.y = 0.f;
      if (k + 2 >= ncols) v.z = 0.f;
      if (k + 3 >= ncols) v.w = 0.f;
    }
    const float4 h = tcc_hi4(v);
    const uint32_t off = sw128_kmajor_off(row, u << 2);
    *reinterpret_cast<float4*>(dst + off) = h;
    *reinterpret_cast<float4*>(dst + TCC_A_HALF + off) = tcc_lo4(v, h);
  }
}

__device__ __forceinline__ bool tcc_group_active(const TccSlot& S, int g, int n0) { return g < S.ngroups && n0 < S.g[g].N; }
__device__ __forceinline__ bool tcc_slot_active(const TccSlot& S, int n0) { return tcc_group_active(S, 0, n0) || tcc_group_active(S, 1, n0); }

// loader lane: the CTA's weight slices of one slot -> W buffer (one bulk copy per group)
__device__ __forceinline__ void tcc_issue_weights(const TccSlot& S, int rank, int n0, uint8_t* Wb, uint64_t* wfull) {
  const uint32_t gbytes = uint32_t(S.nchunks) * TCC_W_CHUNK;
  uint32_t bytes = 0;
#pragma unroll
  for (int g = 0; g < TCC_MAX_GROUPS; ++g)
    if (tcc_group_active(S, g, n0)) bytes += gbytes;
  mbar_expect_tx(wfull, bytes);
#pragma unroll
  for (int g = 0; g < TCC_MAX_GROUPS; ++g)
    if (tcc_group_active(S, g, n0)) tcc_bulk_load(Wb + g * gbytes, S.g[g].wimg + size_t(rank) * gbytes, gbytes, wfull);
}

__global__ void __cluster_dims__(TCC_CLUSTER, 1, 1) __launch_bounds__(TCC_THREADS, 1)
mlp_tc_chain_kernel(const __grid_constant__ TccArgs args) {
  extern __shared__ uint8_t tcc_smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(tcc_smem_raw) + 1023) & ~uintptr_t(1023));
  uint8_t* Ab = smem + TCC_OFF_A;        // [TCC_ABUFS] A-chunk buffers; buffer 8 doubles as the resident X chunk
  uint8_t* Xb = Ab + 8 * TCC_A_CHUNK;
  uint8_t* Wb = smem + TCC_OFF_W;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + TCC_OFF_BAR);
  uint64_t* full = bars;                 // [TCC_ABUFS]  bytes of the copy that starts at this buffer have landed
  uint64_t* wfull = bars + TCC_ABUFS;    // weight slices of the current slot have landed
  uint64_t* dfull = wfull + 1;           // all MMAs of the current slot have completed
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(dfull + 1);

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rank = int(tcc_ctarank());
  const int cid = blockIdx.x / TCC_CLUSTER;
  const int chain = cid / args.row_blocks, rb = cid - chain * args.row_blocks;
  const int m0 = rb * TCC_ROWS, B = args.B;
  const TccChain& CH = args.chain[chain];
  const int ns = CH.nslots;
  const int n0 = rank * TCC_BN;
  uint8_t* planes = args.xchg + (size_t(chain) * args.row_blocks + rb) * (size_t(TCC_PLANES) * TCC_PLANE_BYTES);
  const int npre = CH.pre ? (CH.precols + TCC_KC - 1) / TCC_KC : 0;
  const int passes = args.passes;
  unsigned long long* tr0 = (args.trace && int(blockIdx.x) == args.trace_cta) ? args.trace : nullptr;
  if (args.wait_epoch) {                 // host pipeline: the sample kernel of this step publishes per-CTA epochs
    if (tid < args.wait_n) {
      const unsigned long long target = (unsigned long long)(*reinterpret_cast<const volatile long long*>(args.wait_clock) + 1);
      unsigned long long v;
      do { asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(args.wait_epoch + tid) : "memory"); } while (v < target);
    }
    __syncthreads();
  }
  step_stamp(args.step_trace, args.step_slot);

  if (tid == 0) {
    for (int i = 0; i < TCC_ABUFS + 2; ++i) mbar_init(&bars[i], 1);
    mbar_fence_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, TCC_TMEM_COLS);
  if (warp >= 2) {
    const int et = tid - 64;
    if (CH.x0) tcc_convert_chunk(Xb, CH.x0, CH.x0ld, 0, CH.x0cols, m0, B, et);
    for (int p = 0; p < npre; ++p) tcc_convert_chunk(Ab + p * TCC_A_CHUNK, CH.pre, CH.preld, p * TCC_KC, CH.precols, m0, B, et);
    fence_proxy_async();
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_d = *tmem_slot;

  // the pre-converted chunks: complete the first phase of their `full` barriers (the MMA issuer waits on them like on a copy)
  if (tid == 0)
    for (int p = 0; p < npre; ++p) mbar_arrive(&full[p]);
  // per-role state.  fph: bit b = parity of the NEXT completion of full[b] this thread will wait for (MMA issuer)
  uint32_t fph = 0;
  int nact = 0;                          // slots this CTA took part in so far: phase of wfull / dfull
  if (warp == 0 && lane == 0 && tcc_slot_active(CH.slot[0], n0)) tcc_issue_weights(CH.slot[0], rank, n0, Wb, wfull);

  for (int l = 0; l < ns; ++l) {
    const TccSlot& S = CH.slot[l];
    const bool act0 = tcc_group_active(S, 0, n0), act1 = tcc_group_active(S, 1, n0);
    const bool active = act0 || act1;
    unsigned long long* tr = tr0 ? tr0 + TCC_TRACE_PER_SLOT * l : nullptr;
    bool arrived = false;                  // this thread already arrived on the slot's cluster barrier (hi epilogue warps)

    if (warp == 0) {
      // ============================== loader ==========================================================
      // Every A buffer is free here: the previous slot's MMAs completed before anyone passed the cluster barrier.
      if (lane == 0) {
        if (tr) tr[0] = tcc_gtime();
        if (active && S.nloads > 0) {
          // the cluster's generic-proxy stores to the planes (acquired by the barrier above) -> this thread's TMA reads
          asm volatile("fence.proxy.async.global;" ::: "memory");
          for (int i = 0; i < S.nloads; ++i) {
            const TccLoad L = S.ld[i];
            const uint32_t bytes = uint32_t(L.count) * TCC_A_CHUNK;
            mbar_expect_tx(&full[L.buf0], bytes);
            tcc_bulk_load(Ab + L.buf0 * TCC_A_CHUNK, planes + size_t(L.plane) * TCC_PLANE_BYTES + size_t(L.chunk0) * TCC_A_CHUNK,
                          bytes, &full[L.buf0]);
          }
        }
        if (tr) tr[1] = tcc_gtime();
        // next slot's weights travel while this slot's epilogue and the barrier run
        if (l + 1 < ns && tcc_slot_active(CH.slot[l + 1], n0)) {
          if (active) tcc_wait(dfull, nact & 1, args.watchdog, TCC_CODE(WD_LOADER_DFULL, l, rank), nact);  // the weight buffer is free
          tcc_issue_weights(CH.slot[l + 1], rank, n0, Wb, wfull);
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ============================== MMA issuer (warp-uniform, elected lane issues) =====================
      if (active) {
        // ONE instruction per 8-deep k-step computes all partial products of the 3xTF32 split: the A chunk holds the hi
        // image (64 rows) directly followed by the lo image (64 rows) = a 128-row operand, the weight chunk hi (32 rows)
        // then lo (32 rows) = a 64-row operand.  D[128 x 64] = [Ah; Al] . [Bh; Bl]^T: rows 0-63 / columns 0-31 = Ah.Bh,
        // columns 32-63 = Ah.Bl, rows 64-127 / columns 0-31 = Al.Bh (and Al.Bl, ~2^-22 relative, unused).  4 MMAs per
        // chunk instead of 12: the issue rate of tcgen05.mma (~50 cycles with fresh descriptors) is what bounds a slot.
        const uint32_t idesc = make_idesc(FMT_TF32, false, false, 2 * TCC_ROWS, 2 * TCC_BN);
        // (TCC_DESC_HI << 32 | TCC_DESC_LO) == make_smem_desc(0, 16, 1024, 2)
        const int nch = S.nchunks, boff = S.boff;
        const uint32_t wait_mask = S.wait_mask;
        const uint32_t gstride = (uint32_t(nch) * TCC_W_CHUNK) >> 4;
        const uint32_t w_base = (smem_u32(Wb) >> 4) | TCC_DESC_LO;
        const uint32_t a_base = ((smem_u32(Ab) >> 4) + uint32_t(boff) * (TCC_A_CHUNK >> 4)) | TCC_DESC_LO;
        // lane 0 waits, the warp re-converges on __syncwarp: the issue code below then runs provably converged, which is
        // what lets the compiler keep descriptors in the uniform datapath instead of R2UR round trips per instruction
        if (lane == 0) {
          tcc_wait(wfull, nact & 1, args.watchdog, TCC_CODE(WD_MMA_WFULL, l, rank), nact);
          if (tr) tr[2] = tcc_gtime();
        }
        __syncwarp();
        // Chunk c of the slot's K lives in A buffer c + boff (checked at launch) and every index below derives from
        // kernel parameters and the loop counter only.
        for (int c = 0; c < nch; ++c) {
          if ((wait_mask >> c) & 1u) {                    // first chunk of a bulk copy / a pre-converted chunk
            const int b = c + boff;
            if (lane == 0) {
              tcc_wait(&full[b], (fph >> b) & 1u, args.watchdog, TCC_CODE(WD_MMA_FULL, l, rank), b);
              if (tr && c == 0) tr[3] = tcc_gtime();
            }
            fph ^= 1u << b;
            __syncwarp();
          }
          tc_fence_after_sync();
          const uint32_t a_d = a_base + uint32_t(c) * (TCC_A_CHUNK >> 4);
          const uint32_t acc = c != 0;
#pragma unroll
          for (int g = 0; g < TCC_MAX_GROUPS; ++g) {
            if (!(g == 0 ? act0 : act1)) continue;
            const uint32_t b_d = w_base + g * gstride + uint32_t(c) * (TCC_W_CHUNK >> 4);
            const uint32_t d0 = tmem_d + uint32_t(g * 2 * TCC_BN);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) tcc_mma_elect(d0, a_d + 2 * ks, b_d + 2 * ks, idesc, ks ? 1u : acc);
          }
        }
        tcc_commit_elect(dfull);
        if (tr && lane == 0) tr[4] = tcc_gtime();
      }
      __syncwarp();
    } else {
      // ============================== epilogue ========================================================
      // TMEM lane quarter q = warp % 4.  Quarters 0/1 hold accumulator rows 0-63 (A hi image: Ah.Bh | Ah.Bl), quarters
      // 2/3 rows 64-127 (A lo image: Al.Bh): the "lo" warp of a pair hands its 32 x 16 partial sums to the "hi" warp
      // through shared memory (A buffer g: free, every MMA of the slot has completed), which adds the three partial
      // products, applies the epilogue and stores.  Pair = (q, q + 2) of one 16-column half: named barrier 1 + half * 2 + (q & 1).
      const int et = tid - 64;
      const int q = warp & 3, half = (warp - 2) >> 2;
      const bool hi_warp = q < 2;
      const int row = 32 * (q & 1) + lane;                 // batch row inside the cluster's 64-row block
      const int gi = m0 + row;
      const bool row_ok = gi < B;
      constexpr int SCP = 36;                              // scratch row pitch in floats (16-B aligned, spreads the banks)
      if (active) {
        // this thread's epilogue operands do not depend on the chain: fetch them before the accumulator is ready
        float eop[TCC_MAX_GROUPS][16];
#pragma unroll
        for (int g = 0; g < TCC_MAX_GROUPS; ++g) {
#pragma unroll
          for (int j = 0; j < 16; ++j) eop[g][j] = 0.f;
          if (!hi_warp || !(g == 0 ? act0 : act1)) continue;
          const TccGroup& G = S.g[g];
          const int npad = (G.N + 3) & ~3;
          const bool fwd = G.epi == EPI_BIAS || G.epi == EPI_BIAS_RELU || G.epi == EPI_BIAS_TANH;
          const bool msk = G.epi == EPI_RELU_MASK || G.epi == EPI_TANH_MASK;
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const int gj = n0 + half * 16 + 4 * i;
            if (gj >= npad) continue;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (fwd) v = __ldg(reinterpret_cast<const float4*>(G.bias + gj));
            else if (msk && row_ok) v = __ldg(reinterpret_cast<const float4*>(G.aux + size_t(gi) * G.ldaux + gj));
            eop[g][4 * i] = v.x; eop[g][4 * i + 1] = v.y; eop[g][4 * i + 2] = v.z; eop[g][4 * i + 3] = v.w;
          }
        }
        tcc_wait(dfull, nact & 1, args.watchdog, TCC_CODE(WD_EPI_DFULL, l, rank), nact);
        tc_fence_after_sync();
        if (tr && et == 0) tr[5] = tcc_gtime();
        // the resident X chunk is re-used for another array (critic fc2's action columns) now that this slot's MMAs are
        // done -- before any thread arrives on the slot's barrier
        if (S.xsrc) {
          tcc_convert_chunk(Xb, S.xsrc, S.xld, 0, S.xcols, m0, B, et);
          fence_proxy_async();                             // shared-memory writes -> the tensor core's async-proxy reads
        }
        const uint32_t tq = tmem_d + (uint32_t(32 * q) << 16) + uint32_t(half * 16);
        if (!hi_warp) {
          // ---- lo rows: Al.Bh partial sums -> scratch ---------------------------------------------------------
#pragma unroll
          for (int g = 0; g < TCC_MAX_GROUPS; ++g) {
            if (!(g == 0 ? act0 : act1)) continue;
            float t[16];
            tcc_tmem_ld16(tq + uint32_t(g * 2 * TCC_BN), t);
            tcc_tmem_ld_wait();
            float* sc = reinterpret_cast<float*>(Ab + g * TCC_A_CHUNK) + row * SCP + half * 16;
#pragma unroll
            for (int i = 0; i < 4; ++i) *reinterpret_cast<float4*>(sc + 4 * i) = make_float4(t[4 * i], t[4 * i + 1], t[4 * i + 2], t[4 * i + 3]);
          }
          asm volatile("bar.sync %0, 64;" ::"r"(1 + half * 2 + (q & 1)) : "memory");
        } else {
          // ---- hi rows: Ah.Bh + Ah.Bl (TMEM) + Al.Bh (scratch), epilogue, stores -----------------------------------
          float r[TCC_MAX_GROUPS][16], r2[TCC_MAX_GROUPS][16];
#pragma unroll
          for (int g = 0; g < TCC_MAX_GROUPS; ++g) {
            if (!(g == 0 ? act0 : act1)) continue;
            tcc_tmem_ld16(tq + uint32_t(g * 2 * TCC_BN), r[g]);
            tcc_tmem_ld16(tq + uint32_t(g * 2 * TCC_BN + TCC_BN), r2[g]);
          }
          tcc_tmem_ld_wait();
          if (tr && et == 64) tr[6] = tcc_gtime();
          asm volatile("bar.sync %0, 64;" ::"r"(1 + half * 2 + (q & 1)) : "memory");
          bool any_pub = false;
#pragma unroll
          for (int g = 0; g < TCC_MAX_GROUPS; ++g) {
            if (!(g == 0 ? act0 : act1)) continue;
            const TccGroup& G = S.g[g];
            const float* sc = reinterpret_cast<const float*>(Ab + g * TCC_A_CHUNK) + row * SCP + half * 16;
            const int epi = G.epi;
            float x16[16];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 t = *reinterpret_cast<const float4*>(sc + 4 * i);
              x16[4 * i] = t.x; x16[4 * i + 1] = t.y; x16[4 * i + 2] = t.z; x16[4 * i + 3] = t.w;
            }
            // the epilogue kind is decided ONCE per group, around whole loops (a per-element switch compiles to an
            // indirect branch per element: 32 BRX per group cost 1.7 us of a 5 us slot)
#pragma unroll
            for (int j = 0; j < 16; ++j) x16[j] = (r2[g][j] + x16[j]) + r[g][j];   // the two small cross terms first, then the leading product
            if (epi == EPI_BIAS || epi == EPI_BIAS_RELU || epi == EPI_BIAS_TANH) {
#pragma unroll
              for (int j = 0; j < 16; ++j) x16[j] += eop[g][j];
              if (epi == EPI_BIAS_RELU) {
#pragma unroll
                for (int j = 0; j < 16; ++j) x16[j] = fmaxf(x16[j], 0.f);
              } else if (epi == EPI_BIAS_TANH) {
#pragma unroll
                for (int j = 0; j < 16; ++j)
                  if (n0 + half * 16 + j < G.N) x16[j] = tanhf(x16[j]);             // warp-uniform guard: the 6 action columns only
              }
            } else if (epi == EPI_RELU_MASK) {
#pragma unroll
              for (int j = 0; j < 16; ++j) x16[j] = (eop[g][j] > 0.f) ? x16[j] : 0.f;
            } else if (epi == EPI_TANH_MASK) {
#pragma unroll
              for (int j = 0; j < 16; ++j) x16[j] *= (1.f - eop[g][j] * eop[g][j]);
            }
#pragma unroll
            for (int j = 0; j < 16; ++j) {
              const int gj = n0 + half * 16 + j;
              x16[j] = (row_ok && gj < G.N) ? x16[j] : 0.f; // pad rows / columns stay zero in the images
              r[g][j] = x16[j];                            // kept for the row-major store after the barrier arrive
            }
            if (G.pub >= 0) {
              // K-chunk `rank` of the consumers' A operand: the hi and lo images of this 64 x 32 tile are ONE contiguous
              // 16-KB block of the plane -> staged in shared memory (A buffer 2 + g, free) in the image layout and
              // written with a single TMA bulk store (scattered 16-B st.global cost 32 L2 transactions per warp store)
              any_pub = true;
              uint8_t* stg = Ab + (2 + g) * TCC_A_CHUNK;
              const uint32_t rbase = uint32_t((row >> 3) * 1024 + (row & 7) * 128);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const float4 v = make_float4(x16[4 * i], x16[4 * i + 1], x16[4 * i + 2], x16[4 * i + 3]);
                const float4 h = tcc_hi4(v);
                const uint32_t off = rbase + uint32_t((((half * 4 + i) ^ (row & 7)) & 7) << 4);
                *reinterpret_cast<float4*>(stg + off) = h;
                *reinterpret_cast<float4*>(stg + TCC_A_HALF + off) = tcc_lo4(v, h);
              }
            }
          }
          if (tr && et == 64) tr[7] = tcc_gtime();
          if (any_pub) {                                   // uniform over the hi warps (depends on the slot only)
            fence_proxy_async();                           // staged tiles (generic proxy) -> TMA store (async proxy)
            asm volatile("bar.sync 5, 128;" ::: "memory"); // the four hi warps
            if (et == 64) {
#pragma unroll
              for (int g = 0; g < TCC_MAX_GROUPS; ++g) {
                if (!(g == 0 ? act0 : act1) || S.g[g].pub < 0) continue;
                uint8_t* img = planes + size_t(S.g[g].pub) * TCC_PLANE_BYTES + size_t(rank) * TCC_A_CHUNK;
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;"
                             ::"l"(img), "r"(smem_u32(Ab + (2 + g) * TCC_A_CHUNK)), "r"(TCC_A_CHUNK) : "memory");
              }
              asm volatile("cp.async.bulk.commit_group;" ::: "memory");
              asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");      // writes complete: visible before the barrier arrive
            }
          }
          if (tr && et == 64) tr[8] = tcc_gtime();
          tc_fence_before_sync();                          // accumulator reads done before the next slot's MMAs overwrite it
          // The row-major outputs are read by later kernels only: they are stored AFTER this thread's barrier arrive, so
          // the cluster does not wait for them to drain.
          if (l + 1 < ns) { tcc_cluster_arrive(); arrived = true; }
#pragma unroll
          for (int g = 0; g < TCC_MAX_GROUPS; ++g) {
            if (!(g == 0 ? act0 : act1)) continue;
            const TccGroup& G = S.g[g];
            if (G.C && row_ok) {
              const int npad = (G.N + 3) & ~3;
              float* crow = G.C + size_t(gi) * G.ldc;
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int gj = n0 + half * 16 + 4 * i;
                if (gj < npad) *reinterpret_cast<float4*>(crow + gj) = make_float4(r[g][4 * i], r[g][4 * i + 1], r[g][4 * i + 2], r[g][4 * i + 3]);
              }
            }
          }
        }
        tc_fence_before_sync();                            // accumulator reads done before the next slot's MMAs overwrite it
      }
      if (!active && S.xsrc) {                             // (an inactive CTA did not read X in this slot)
        tcc_convert_chunk(Xb, S.xsrc, S.xld, 0, S.xcols, m0, B, et);
        fence_proxy_async();
      }
      if (tr && et == 0) tr[9] = tcc_gtime();
    }
    if (active) ++nact;
    if (l + 1 < ns) {
      if (!arrived) tcc_cluster_arrive();
      tcc_cluster_wait();
      if (tr && tid == 0) tr[10] = tcc_gtime();
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_d, TCC_TMEM_COLS);
  step_stamp(args.step_trace, args.step_slot + 16);
}

// ---- weight packing -------------------------------------------------------------------------------------
// One CTA per 32x32 block: 256 threads, one float4 of hi and lo each.
__global__ void __launch_bounds__(256) tcc_pack_kernel(const __grid_constant__ TccPackArgs args) {
  int ui = 0;
#pragma unroll 1
  for (int i = 1; i < args.n; ++i)
    if (int(blockIdx.x) >= args.use[i].block_begin) ui = i;
  const TccPackUse& U = args.use[ui];
  const int blk = blockIdx.x - U.block_begin;
  const int slice = blk / U.nchunks, chunk = blk - slice * U.nchunks;
  uint8_t* dst = args.dst + U.dst_off + size_t(blk) * TCC_W_CHUNK;
  const int tid = threadIdx.x;
  float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
  int j, u;
  if (U.mode == GEMM_FWD) {
    j = tid >> 3; u = tid & 7;                               // consecutive threads: consecutive 16-B units of a W row
    const int n = slice * TCC_BN + j, k = chunk * TCC_KC + 4 * u;
    if (n < U.N && k < U.K) {
      v = __ldg(reinterpret_cast<const float4*>(U.W + size_t(n) * U.ldw + k));   // row pitch is a multiple of 4 floats
      if (k + 1 >= U.K) v.y = 0.f;
      if (k + 2 >= U.K) v.z = 0.f;
      if (k + 3 >= U.K) v.w = 0.f;
    }
  } else {
    j = tid & 31; u = tid >> 5;                              // consecutive threads: consecutive columns n of a W row (coalesced)
    const int n = slice * TCC_BN + j, k = chunk * TCC_KC + 4 * u;
    if (n < U.N) {
      if (k < U.K) v.x = __ldg(U.W + size_t(k) * U.ldw + n);
      if (k + 1 < U.K) v.y = __ldg(U.W + size_t(k + 1) * U.ldw + n);
      if (k + 2 < U.K) v.z = __ldg(U.W + size_t(k + 2) * U.ldw + n);
      if (k + 3 < U.K) v.w = __ldg(U.W + size_t(k + 3) * U.ldw + n);
    }
  }
  const float4 h = tcc_hi4(v);
  const uint32_t off = sw128_kmajor_off(j, 4 * u);
  *reinterpret_cast<float4*>(dst + off) = h;
  *reinterpret_cast<float4*>(dst + TCC_W_HALF + off) = tcc_lo4(v, h);
}

static unsigned long long* g_tcc_watchdog_host = nullptr;
// allocated once per process, outside of any stream capture (tcc users call this at create time)
unsigned long long* tcc_watchdog_device() {
  static bool tried = false;
  static unsigned long long* dev = nullptr;
  if (!tried) {
    tried = true;
    unsigned long long* host = nullptr;
    if (cudaHostAlloc(reinterpret_cast<void**>(&host), 128, cudaHostAllocMapped) == cudaSuccess) {
      memset(host, 0, 128);
      if (cudaHostGetDevicePointer(reinterpret_cast<void**>(&dev), host, 0) != cudaSuccess) dev = nullptr;
      g_tcc_watchdog_host = host;
    }
    (void)cudaGetLastError();
  }
  return dev;
}
}  // namespace d4pg
// the watchdog record of the tcgen05 chain kernel (host-mapped memory: readable after a trapped launch killed the context)
extern "C" int32_t d4pg_debug_watchdog(unsigned long long* out16) {
  if (!out16) return D4PG_EINVAL;
  for (int i = 0; i < 16; ++i) out16[i] = d4pg::g_tcc_watchdog_host ? d4pg::g_tcc_watchdog_host[i] : 0ull;
  return D4PG_OK;
}
namespace d4pg {

void tcc_pack_begin(TccPackArgs& p, uint8_t* dst) { p.n = 0; p.total_blocks = 0; p.dst = dst; }
int tcc_pack_add(TccPackArgs& p, const float* W, int ldw, int mode, int N, int K) {
  if (p.n >= TCC_MAX_USES) return -1;
  TccPackUse& u = p.use[p.n];
  u.W = W; u.ldw = ldw; u.mode = mode; u.N = N; u.K = K;
  u.nslices = cdiv(N, TCC_BN); u.nchunks = cdiv(K, TCC_KC);
  u.block_begin = p.total_blocks;
  u.dst_off = (long long)(p.total_blocks) * TCC_W_CHUNK;
  p.total_blocks += u.nslices * u.nchunks;
  return p.n++;
}
long long tcc_pack_bytes(const TccPackArgs& p) { return (long long)(p.total_blocks) * TCC_W_CHUNK; }
// the set's images start `first_byte` into the buffer `dst` (dst_off of every use is relative to the set's own start)
void tcc_pack_set_base(TccPackArgs& p, uint8_t* dst, long long first_byte) { p.dst = dst + first_byte; }
int launch_tcc_pack(const TccPackArgs& p, cudaStream_t st) {
  D4PG_REQUIRE(p.n > 0 && p.dst, D4PG_EINVAL, "launch_tcc_pack: nothing to pack");
  tcc_pack_kernel<<<p.total_blocks, 256, 0, st>>>(p);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

// ---- chain construction -----------------------------------------------------------------------------------
int64_t tcc_xchg_floats(int B) {
  return int64_t(TCC_MAX_CHAINS) * cdiv(B, TCC_ROWS) * TCC_PLANES * (TCC_PLANE_BYTES / 4);
}
void tcc_args_begin(TccArgs& a, int B, uint8_t* xchg, int passes) {
  memset(&a, 0, sizeof(a));
  a.B = B; a.row_blocks = cdiv(B, TCC_ROWS); a.xchg = xchg; a.passes = passes;
}
void tcc_chain_x0(TccArgs& a, int c, const float* src, int ld, int cols) {
  a.chain[c].x0 = src; a.chain[c].x0ld = ld; a.chain[c].x0cols = cols;
}
void tcc_chain_pre(TccArgs& a, int c, const float* src, int ld, int cols) {
  a.chain[c].pre = src; a.chain[c].preld = ld; a.chain[c].precols = cols;
}
int tcc_slot_begin(TccArgs& a, int c) {
  if (c >= a.nchains) a.nchains = c + 1;
  TccChain& ch = a.chain[c];
  const int l = ch.nslots++;
  if (l < TCC_MAX_SLOTS) { ch.slot[l] = TccSlot{}; ch.slot[l].g[0].pub = ch.slot[l].g[1].pub = -1; }
  return l;
}
static void tcc_push_chunk(TccSlot& s, int kind, int plane, int chunk) {
  if (s.nchunks < TCC_MAX_CHUNKS) s.ch[s.nchunks] = TccChunk{short(kind), short(plane), short(chunk), 0};
  ++s.nchunks;
}
void tcc_slot_src_x(TccArgs& a, int c, int slot) { tcc_push_chunk(a.chain[c].slot[slot], TCC_SRC_X, 0, 0); }
void tcc_slot_src_pre(TccArgs& a, int c, int slot) {
  const int n = cdiv(a.chain[c].precols, TCC_KC);
  for (int i = 0; i < n; ++i) tcc_push_chunk(a.chain[c].slot[slot], TCC_SRC_PRE, 0, i);
}
void tcc_slot_src_plane(TccArgs& a, int c, int slot, int plane, int nchunks) {
  for (int i = 0; i < nchunks; ++i) tcc_push_chunk(a.chain[c].slot[slot], TCC_SRC_IMG, plane, i);
}
void tcc_slot_reconvert_x(TccArgs& a, int c, int slot, const float* src, int ld, int cols) {
  TccSlot& s = a.chain[c].slot[slot];
  s.xsrc = src; s.xld = ld; s.xcols = cols;
}
int tcc_slot_group(TccArgs& a, int c, int slot, const TccImage& img, int epi, const float* bias,
                   const float* aux, int ldaux, float* C, int ldc, int publish) {
  TccChain& ch = a.chain[c];
  TccSlot& s = ch.slot[slot];
  const int gi = s.ngroups++;
  if (gi >= TCC_MAX_GROUPS) return -1;
  TccGroup& g = s.g[gi];
  g.wimg = img.ptr; g.bias = bias; g.aux = aux; g.ldaux = ldaux; g.C = C; g.ldc = ldc;
  g.N = img.N; g.epi = epi; g.kchunks = img.kchunks;
  g.pub = publish ? ch.nplanes++ : -1;
  return g.pub;
}

// A chunks per bulk copy: fewer, larger copies are faster, but above 2 the first MMA of a slot waits longer
constexpr int TCC_LOAD_GROUP = 2;
int launch_mlp_tc_chain(TccArgs& a, cudaStream_t st) {
  D4PG_REQUIRE(a.nchains > 0 && a.nchains <= TCC_MAX_CHAINS, D4PG_EINVAL, "launch_mlp_tc_chain: %d chains", a.nchains);
  D4PG_REQUIRE(a.passes == 1 || a.passes == 3, D4PG_EINVAL, "launch_mlp_tc_chain: passes %d", a.passes);
  for (int c = 0; c < a.nchains; ++c) {
    TccChain& ch = a.chain[c];
    bool x_clobbered = false;
    D4PG_REQUIRE(ch.nslots > 0 && ch.nslots <= TCC_MAX_SLOTS, D4PG_EINVAL, "launch_mlp_tc_chain: chain %d has %d slots", c, ch.nslots);
    D4PG_REQUIRE(ch.nplanes <= TCC_PLANES, D4PG_ENOTSUP, "launch_mlp_tc_chain: chain %d publishes %d planes", c, ch.nplanes);
    D4PG_REQUIRE(!ch.x0 || (ch.x0cols <= TCC_KC && ch.x0ld % 4 == 0 && ch.x0ld >= ch.x0cols), D4PG_ENOTSUP, "launch_mlp_tc_chain: bad X source");
    D4PG_REQUIRE(!ch.pre || (ch.precols <= 8 * TCC_KC && ch.preld % 4 == 0 && ch.preld >= ch.precols), D4PG_ENOTSUP,
                 "launch_mlp_tc_chain: bad first-slot source");
    int planes_seen = 0;
    for (int l = 0; l < ch.nslots; ++l) {
      TccSlot& s = ch.slot[l];
      D4PG_REQUIRE(s.ngroups >= 1 && s.ngroups <= TCC_MAX_GROUPS, D4PG_EINVAL, "launch_mlp_tc_chain: slot %d has %d groups", l, s.ngroups);
      D4PG_REQUIRE(s.nchunks >= 1 && s.nchunks <= TCC_MAX_CHUNKS && s.ngroups * s.nchunks <= TCC_MAX_CHUNKS, D4PG_ENOTSUP,
                   "launch_mlp_tc_chain: slot %d: %d groups x %d chunks exceed the weight buffer", l, s.ngroups, s.nchunks);
      // A buffers are direct-mapped: the j-th non-resident chunk of a slot lives in buffer j (0..7); a 9th one takes
      // buffer 8, the resident X chunk's, if this slot does not read X (and X is dead from then on).  Consecutive
      // chunks of one plane in consecutive buffers travel as ONE bulk copy (at most TCC_LOAD_GROUP chunks each, so that the
      // MMAs of the first chunks overlap the arrival of the rest).
      int nring = 0;
      bool uses_x = false;
      for (int i = 0; i < s.nchunks; ++i) uses_x = uses_x || s.ch[i].kind == TCC_SRC_X;
      s.nloads = 0;
      for (int i = 0; i < s.nchunks; ++i) {
        TccChunk& k = s.ch[i];
        if (k.kind == TCC_SRC_IMG) D4PG_REQUIRE(k.plane >= 0 && k.plane < planes_seen && k.chunk < TCC_CLUSTER, D4PG_EINVAL,
                                                 "launch_mlp_tc_chain: slot %d reads plane %d before it is published", l, k.plane);
        if (k.kind == TCC_SRC_PRE) D4PG_REQUIRE(l == 0 && ch.pre && k.chunk == nring && nring < 8, D4PG_EINVAL, "launch_mlp_tc_chain: pre chunks belong to slot 0, in order");
        if (k.kind == TCC_SRC_X) {
          D4PG_REQUIRE(ch.x0 != nullptr && !x_clobbered, D4PG_EINVAL, "launch_mlp_tc_chain: slot %d reads X but the chain has none (or it was overwritten)", l);
          k.buf = 8;
          continue;
        }
        if (nring < 8) k.buf = short(nring);
        else {
          D4PG_REQUIRE(nring == 8 && !uses_x && k.kind == TCC_SRC_IMG, D4PG_ENOTSUP, "launch_mlp_tc_chain: slot %d needs more than 9 A buffers", l);
          k.buf = 8; x_clobbered = true;
        }
        ++nring;
        if (k.kind == TCC_SRC_IMG) {
          TccLoad* cur = s.nloads ? &s.ld[s.nloads - 1] : nullptr;
          if (cur && cur->plane == k.plane && cur->chunk0 + cur->count == k.chunk && cur->buf0 + cur->count == k.buf && cur->count < TCC_LOAD_GROUP) ++cur->count;
          else s.ld[s.nloads++] = TccLoad{k.plane, k.chunk, k.buf, 1};
        }
      }
      s.nacc = 1;
      // MMA-side view: chunk c <-> A buffer c + boff, wait on full[c + boff] where a copy (or a pre-converted chunk) starts
      s.boff = s.ch[0].buf;
      s.wait_mask = 0;
      for (int i = 0; i < s.nchunks; ++i) {
        D4PG_REQUIRE(s.ch[i].buf == s.boff + i, D4PG_ENOTSUP, "launch_mlp_tc_chain: slot %d: chunk %d is not in A buffer %d", l, i, s.boff + i);
        if (s.ch[i].kind == TCC_SRC_PRE) s.wait_mask |= 1u << i;
      }
      for (int i = 0; i < s.nloads; ++i) s.wait_mask |= 1u << (s.ld[i].buf0 - s.boff);
      for (int g = 0; g < s.ngroups; ++g) {
        const TccGroup& G = s.g[g];
        D4PG_REQUIRE(G.N > 0 && G.N <= TCC_CLUSTER * TCC_BN && G.wimg, D4PG_ENOTSUP, "launch_mlp_tc_chain: group width %d", G.N);
        D4PG_REQUIRE(G.kchunks == s.nchunks, D4PG_EINVAL, "launch_mlp_tc_chain: chain %d slot %d: A operand has %d chunks, the weight image %d", c, l, s.nchunks, G.kchunks);
        D4PG_REQUIRE(!G.C || (G.ldc % 4 == 0 && G.ldc >= ((G.N + 3) & ~3) && (reinterpret_cast<uintptr_t>(G.C) & 15) == 0), D4PG_EINVAL,
                     "launch_mlp_tc_chain: output pitch");
        const bool fwd = G.epi == EPI_BIAS || G.epi == EPI_BIAS_RELU || G.epi == EPI_BIAS_TANH;
        const bool msk = G.epi == EPI_RELU_MASK || G.epi == EPI_TANH_MASK;
        D4PG_REQUIRE(!fwd || (G.bias && (reinterpret_cast<uintptr_t>(G.bias) & 15) == 0), D4PG_EINVAL, "launch_mlp_tc_chain: bias");
        D4PG_REQUIRE(!msk || (G.aux && G.ldaux % 4 == 0 && (reinterpret_cast<uintptr_t>(G.aux) & 15) == 0), D4PG_EINVAL, "launch_mlp_tc_chain: mask operand");
        if (G.pub >= 0) ++planes_seen;
      }
      if (l == 0 && ch.pre) D4PG_REQUIRE(s.g[0].N > (TCC_CLUSTER - 1) * TCC_BN, D4PG_ENOTSUP, "launch_mlp_tc_chain: the first slot must span the cluster");
    }
  }
  static bool attr_set = false;
  if (!attr_set) {
    D4PG_CUDA_OK(cudaFuncSetAttribute(mlp_tc_chain_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(TCC_SMEM)));
    D4PG_CUDA_OK(cudaFuncSetAttribute(mlp_tc_chain_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, int(cudaSharedmemCarveoutMaxShared)));
    attr_set = true;
  }
  a.watchdog = tcc_watchdog_device();
  unsigned long long* dbg = debug_trace_buffer();
  a.trace = dbg ? dbg + (a.step_slot == 5 ? 384 : 256) : nullptr;
  a.step_trace = dbg ? dbg + STEP_TRACE_BASE : nullptr;
  { const char* e = getenv("D4PG_TRACE_CTA"); a.trace_cta = e ? atoi(e) : 0; if (a.trace_cta >= a.nchains * a.row_blocks * TCC_CLUSTER) a.trace_cta = 0; }
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(a.nchains * a.row_blocks * TCC_CLUSTER); cfg.blockDim = dim3(TCC_THREADS);
  cfg.dynamicSmemBytes = TCC_SMEM; cfg.stream = st;
  cfg.attrs = nullptr; cfg.numAttrs = 0;              // cluster shape is compiled in (__cluster_dims__)
  D4PG_CUDA_OK(cudaLaunchKernelEx(&cfg, mlp_tc_chain_kernel, a));
  return D4PG_OK;
}

}  // namespace d4pg
