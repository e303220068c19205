// Cross-translation-unit internals of libd4pg_sm100.so (not part of the C ABI).
#pragma once
#include "common.cuh"
#include "adam.cuh"

struct d4pg_replay;
struct d4pg_comm;

namespace d4pg {

struct HeadsArgs {
  const float* target_logits; const float* q_logits; const float* pi_logits;
  const double* rewards; const uint8_t* dones;
  int B, N; int flags;
  int ld;                 // row pitch (floats) of every [B,N] array (>= N)
  double v_min, v_max, delta, discount, prio_eps;
  float grad_scale;
  float* m; int32_t* bins_l; int32_t* bins_u; float* target_probs; float* q_probs;
  float* loss_rows; float* td; float* prio; float* dlogits_q; float* pi_rows; float* dlogits_pi;
  // corrected-semantics switches (SURVEY.md section 8f.4; the reference does neither, H3 / H4):
  const float* is_weights;   // non-null: critic CE row i is scaled by the PER importance weight w_i
  int ce_priority;           // 1: priority = CE_i + eps instead of |sum_j m_ij q_ij| + eps
  unsigned long long* trace;
  int only_policy;               // 1: only the policy head (pi_rows, dlogits_pi) -- the second loss launch of the post-update-critic plan
  LearnerClock* sampler_clock;   // prefetch pipeline: thread 0 advances the sampler's counters (after sample(k), before sample(k+1))
};
int launch_heads(const HeadsArgs& a, int mode, cudaStream_t st);

constexpr int SAMPLE_ROWS = 32;      // batch rows per CTA of the sample + gather kernel (replay_dev.cuh)

// sample for the learner: per-step scalars come from device memory (graph replay safe)
int learner_sample(d4pg_replay* h, int B, int prioritized, const double* uniforms, const int32_t* positions,
                   uint64_t seed, LearnerClock* clock, const ClockParams& cp,
                   int32_t* idx, float* weights, float* s, float* a, double* r, float* s2, uint8_t* d,
                   int ld_obs, int ld_act, int pipe_slot, cudaStream_t st, bool dependent = false,
                   unsigned long long* done_epoch = nullptr);
// gate != nullptr: *gate is bumped (release) once the trees are complete -- by the update kernel itself when it can
int launch_tree_update(d4pg_replay* h, int B, const int32_t* idx, const float* prio, cudaStream_t st, unsigned long long* gate = nullptr);
int64_t replay_generation(const d4pg_replay* h);
// ingest gate (host pipeline): every gated learner step bumps the buffer's flag once (launch_gate_signal) and arms the
// gate after its launch; the next add / presample on the ingest stream first waits for flag >= number of armed steps
unsigned long long* replay_gate_flag(d4pg_replay* h);
void replay_arm_gate(d4pg_replay* h);
int replay_gate_consume(d4pg_replay* h, cudaStream_t st);
int launch_gate_signal(unsigned long long* flag, cudaStream_t st);
void trace_set_side_stream(cudaStream_t s);     // changes whenever the caller mutates the buffer
int comm_allreduce(d4pg_comm* c, float* buf, int64_t n, cudaStream_t st);
// fused all-reduce over IPC-mapped peer memory (comm.cu): x[r] = rank r's [2][n] gradient halves
bool comm_peer_info(d4pg_comm* c, PeerInfo* out);
PeerSignal comm_peer_signal(const PeerInfo& info, int kind);    // kind 0: gradient half complete, 1: reduced slice pushed
int comm_peer_barrier(d4pg_comm* c, cudaStream_t st);
// reduce-scatter + all-gather of the step's gradient over peer memory: this rank sums ITS slice of every rank's half
// `parity` (rank order) and pushes the result into every rank's reduced buffer; publishes flag2 when done
int comm_peer_reduce_scatter(d4pg_comm* c, int parity, cudaStream_t st);
// two-phase in-switch form: multimem.ld_reduce of this rank's slice, multimem.st into every rank's reduced buffer
// (mc_uc + 2n on each rank), then flag2
int comm_mc_reduce_bcast(d4pg_comm* c, int parity, cudaStream_t st);

}  // namespace d4pg
