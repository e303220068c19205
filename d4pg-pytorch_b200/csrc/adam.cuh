// Fused Adam + Polyak and the device-side step clock.
#pragma once
#include "common.cuh"

namespace d4pg {

// Per-step scalars produced on the device so a captured CUDA graph needs no host patching.
struct LearnerClock {
  // base counters: read by the step's FIRST kernel (sample), advanced by its LAST (adam)
  int64_t adam_step;     // completed Adam steps (state['step'] before this step)
  int64_t beta_t;        // LinearSchedule.t
  int64_t steps_done;    // Philox counter / bookkeeping
  int64_t reserved;
  // derived per-step scalars: written by the sample kernel, read by later kernels of the step
  float beta;            // PER beta for this step's IS weights
  float neg_step_size[2];   // -(lr/bc1) for actor, critic
  float bc2_sqrt;        // sqrt(1 - beta2^step)
  float pad;
  // ---- prefetch pipeline (cfg.prefetch): batch k+1 is sampled on a side branch while step k's backward
  // pass and Adam still run, so the sampler keeps its OWN counters (advanced by step k's loss kernel, which
  // runs after sample(k) and before sample(k+1)) and writes the derived scalars of step k into the slot of
  // the batch buffer it fills (a launch argument); Adam of that step reads the same slot.
  int64_t s_adam_step, s_beta_t, s_steps_done;
  float d_neg_step_size[2][2];
  float d_bc2_sqrt[2];
};

struct ClockParams {
  double lr_actor, lr_critic, beta1, beta2;
  double per_beta0, per_beta_final; int64_t per_beta_iters;
};

// prefetch pipeline: scalars of the step whose batch is being sampled, into its parity slot
__device__ __forceinline__ void clock_derive_pipelined(LearnerClock* c, const ClockParams& a, int slot) {
  const double step = double(c->s_adam_step + 1);
  const double bc1 = 1.0 - pow(a.beta1, step);
  const double bc2 = 1.0 - pow(a.beta2, step);
  c->d_neg_step_size[slot][0] = float(-(a.lr_actor / bc1));
  c->d_neg_step_size[slot][1] = float(-(a.lr_critic / bc1));
  c->d_bc2_sqrt[slot] = float(sqrt(bc2));
}
// executed by ONE thread of the step's first kernel
__device__ __forceinline__ void clock_derive(LearnerClock* c, const ClockParams& a) {
  const double step = double(c->adam_step + 1);                      // post-increment step count
  const double bc1 = 1.0 - pow(a.beta1, step);
  const double bc2 = 1.0 - pow(a.beta2, step);
  c->neg_step_size[0] = float(-(a.lr_actor / bc1));
  c->neg_step_size[1] = float(-(a.lr_critic / bc1));
  c->bc2_sqrt = float(sqrt(bc2));
}
// LinearSchedule.value() for clock t (prioritized_replay_memory.py:25-29)
__device__ __forceinline__ float clock_beta(const LearnerClock* c, const ClockParams& a, bool pipelined = false) {
  const double frac = fmin(double(pipelined ? c->s_beta_t : c->beta_t) / double(a.per_beta_iters), 1.0);
  return float(a.per_beta0 + frac * (a.per_beta_final - a.per_beta0));
}

constexpr int D4PG_MAX_PEERS = 8;
// Cross-rank signals are PUSHED: a rank that finished a phase stores its step count into slot [its rank] of every rank's
// inbox (one posted NVLink store each, after a system-scope fence), and waiters poll their own LOCAL inbox -- one one-way
// NVLink latency per hop instead of a remote-polling round trip.  Flag block of a rank, per signal kind k (64 u64 apart):
// [0] unused, [1] local count of this rank's own completions, [2] CTA ticket, [8 + r] inbox slot written by rank r.
struct PeerSignal {
  unsigned long long* local;                   // this rank's block for the signal kind
  unsigned long long* inbox[8];                // inbox[p] = &(rank p's block)[8 + my_rank]
  int world;
};
// called by thread 0 of every CTA of the producing kernel after a __syncthreads(): the last CTA publishes
__device__ __forceinline__ void peer_signal_last_cta(const PeerSignal& s, unsigned nblocks) {
  __threadfence();
  unsigned long long* f = s.local;
  if (atomicAdd(f + 2, 1ull) == nblocks - 1) {
    f[2] = 0ull;
    const unsigned long long v = f[1] + 1ull;
    f[1] = v;
    __threadfence_system();                    // ONE system-scope fence, then relaxed stores: fence + relaxed store = release;
    // (st.release.sys per peer put a MEMBAR.ALL.SYS in front of every one of the N flag stores)
    for (int p = 0; p < s.world; ++p) asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(s.inbox[p]), "l"(v) : "memory");
  }
}
// threads 0..world-1 of a CTA poll the LOCAL inbox until every rank published >= this rank's own count; then __syncthreads
__device__ __forceinline__ void peer_wait_all(const unsigned long long* block, int world) {
  const int r = threadIdx.x;
  if (r < world) {
    const unsigned long long target = __ldcg(block + 1);
    unsigned long long v;
    do {
      asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(block + 8 + r) : "memory");
    } while (v < target);
  }
  __syncthreads();
}

// x[r]: rank r's [2][n] gradient halves; red[r]: rank r's [n] REDUCED gradient (every slice written by the rank that owns
// it); flag[r] / flag2[r]: "gradient half of step k complete" / "my slice of step k is reduced and pushed to everyone"
struct PeerInfo {
  int world, rank; int64_t n;
  float* x[D4PG_MAX_PEERS]; float* red[D4PG_MAX_PEERS];
  unsigned long long* flag[D4PG_MAX_PEERS]; unsigned long long* flag2[D4PG_MAX_PEERS];
  // in-switch reduction (NVLS): mc = multicast mapping of every rank's [2][n] gradient buffer (multimem.ld_reduce on it
  // returns the sum over the ranks), mc_uc = this rank's own buffer through an ordinary mapping; null when not set up
  const float* mc; float* mc_uc;
};

// tcgen05 chains (mlp_tc_chain.cu): the updated weights are ALSO written as the tensor cores' forward operand images
// (hi / lo tf32 parts, 32 x 32 K-major SWIZZLE_128B blocks), for the online network and -- the Polyak output -- its
// target, so that the next step's forward chains need no separate pack launch.  One entry per weight matrix.
struct AdamImgLayer { int64_t w_off, w_end; int ld, nchunks; uint8_t* img; uint8_t* img_t; };
struct AdamSeg {
  float* p; const float* g; float* m; float* v; float* target; int64_t n;
  float* g_out; int64_t g_off;                 // peer mode: the summed gradient is also stored here; offset in the exchange half
  float neg_step_size; int clock_slot;        // clock_slot >= 0: read -step_size from the device clock
  AdamImgLayer imgl[4]; int nimg;              // nimg = 0: no images
};
struct AdamArgs {
  AdamSeg seg[2]; int nseg;
  float w1, w2, beta2, eps, bc2_sqrt, tau, one_minus_tau, grad_scale;
  LearnerClock* clock;                        // optional (learner): scalars in, counters advanced
  unsigned long long* trace;
  // fused all-reduce: g = sum over ranks r = 0..npeers-1 (fixed order: identical on every rank) of peer_g[r][g_off + i],
  // read over NVLink from IPC-mapped peer memory; the ranks were synchronised by comm_peer_barrier
  const float* peer_g[D4PG_MAX_PEERS]; int npeers;
  const float* mc_g;                          // non-null: g = multimem.ld_reduce over all ranks at mc_g + g_off + i (NVSwitch sums)
  int peer_reduced;                           // 1: seg.g already holds the reduced gradient (reduce-scatter + all-gather ran before);
                                              //    only wait for every rank's "slice pushed" flag.  0: sum the ranks' halves here
  // non-null: wait inside the kernel until every rank published step count >= this rank's local one
  // (the signal came from the dW kernel's last CTA); null: a barrier launch already ordered the ranks
  const unsigned long long* my_flags; int rank;   // this rank's flag block of the awaited signal kind (local inbox inside)
  int pipe_slot;                              // >= 0: the step's scalars are in this slot of the clock (prefetch pipeline)
  // fused tail (learner): deterministic batch means of the per-row losses -> out[0], out[1]
  const float* loss_rows; const float* pi_rows; int B; float inv_count; float* loss_out;
  int skip_tail;                              // 1: no loss means / clock advance in this launch (first of two Adam launches of a step)
};
int launch_adam(const AdamArgs& a, cudaStream_t st);


}  // namespace d4pg
