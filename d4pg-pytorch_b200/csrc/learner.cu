// The learner: one DDPG.train() body (ddpg.py:200-255) as a fixed sequence of launches,
// captured once into a CUDA graph and replayed.  No host synchronisation inside a step; every
// per-step scalar (Adam bias corrections, PER beta, Philox counter) lives in device memory and
// is advanced by a one-thread clock kernel so the captured graph never needs patching.
//
// Step order (reference line -> launch):
//   ddpg.py:202  sample                       -> sample_gather_kernel (tree descent + row gather)
//   ddpg.py:205-208 target/online forwards    -> 7 grouped-GEMM levels (actor_target, critic_target,
//                                                critic, actor and critic(s, actor(s)) in lock-step)
//   ddpg.py:214-222 projection, CE loss, td   -> heads_kernel (also the policy head of ddpg.py:236-238)
//   ddpg.py:229-231 critic backward           -> grouped dX / dW levels (shared with the policy pass)
//   ddpg.py:236-243 policy backward           -> uses the PRE-update critic weights (SURVEY.md H7):
//                                                both backward passes run before any Adam update
//   ddpg.py:232,244,247,250 Adam x2, sync, Polyak -> one fused adam_polyak_kernel (2 segments)
//   ddpg.py:252-255 update_priorities         -> tree_write_kernel<TREE_UPDATE>
#include "common.cuh"
#include "gemm_ffma.cuh"
#include "adam.cuh"
#include <string.h>
#include <stdlib.h>
#include <new>
#include <string>
#include <vector>

#include "internal.cuh"
#include "mlp_chain.cuh"
#include "mlp_tc_chain.cuh"

namespace d4pg {

struct Workspace {
  // batch
  float *s, *a, *s2; double* r; uint8_t* done;
  // activations: [0]=actor_target [1]=critic_target [2]=critic [3]=actor [4]=critic on policy action
  float *h1[5], *h2[5], *h3[5], *out[5];
  // heads
  float *m, *q_probs, *target_probs, *dlogits_q, *dlogits_pi, *loss_rows, *pi_rows;
  // backward
  float *c_dz22, *c_dz2, *c_dz1, *p_dz22, *p_dz2, *a_dz3, *a_dz22, *a_dh2, *a_dz1;
  LearnerClock* clock;
  float* xchg;                     // exchange planes of the cluster-fused chain kernels (chain mode)
  unsigned long long* pipe_epoch;  // host pipeline: per-CTA completion epochs of the presample kernel (polled by the forward chains)
  // prefetch pipeline: the second half of the double-buffered batch, and the sampler's own index / weight buffers
  float *s_b, *a_b, *s2_b; double* r_b; uint8_t* done_b;
  int32_t* idx2[2]; float* wts2[2];
  int64_t total;
};

// Every 2-D plane has a row pitch that is a multiple of 4 floats (16-B rows): |s|=17 -> 20,
// |a|=6 -> 8, N=51 -> 52.  That makes every GEMM operand TMA- and float4-addressable.
static Workspace carve(float* base, int B, int S, int A, int N, bool chain, bool prefetch) {
  Workspace w{};
  int64_t off = 0;
  auto take = [&](int64_t n) { float* p = base ? base + off : nullptr; off += align4(n); return p; };
  const int H = D4PG_HIDDEN, Sp = pitch4(S), Ap = pitch4(A), Np = pitch4(N);
  w.s = take(int64_t(B) * Sp); w.a = take(int64_t(B) * Ap); w.s2 = take(int64_t(B) * Sp);
  w.r = reinterpret_cast<double*>(take(int64_t(B) * 2));
  w.done = reinterpret_cast<uint8_t*>(take((B + 3) / 4));
  for (int k = 0; k < 5; ++k) {
    if (k != 4) w.h1[k] = take(int64_t(B) * H);
    w.h2[k] = take(int64_t(B) * H); w.h3[k] = take(int64_t(B) * H);
  }
  w.out[0] = take(int64_t(B) * Ap); w.out[3] = take(int64_t(B) * Ap);
  w.out[1] = take(int64_t(B) * Np); w.out[2] = take(int64_t(B) * Np); w.out[4] = take(int64_t(B) * Np);
  w.m = take(int64_t(B) * Np); w.q_probs = take(int64_t(B) * Np); w.target_probs = take(int64_t(B) * Np);
  w.dlogits_q = take(int64_t(B) * Np); w.dlogits_pi = take(int64_t(B) * Np);
  w.loss_rows = take(B); w.pi_rows = take(B);
  w.c_dz22 = take(int64_t(B) * H); w.c_dz2 = take(int64_t(B) * H); w.c_dz1 = take(int64_t(B) * H);
  w.p_dz22 = take(int64_t(B) * H); w.p_dz2 = take(int64_t(B) * H);
  w.a_dz3 = take(int64_t(B) * Ap); w.a_dz22 = take(int64_t(B) * H); w.a_dh2 = take(int64_t(B) * H);
  w.a_dz1 = take(int64_t(B) * H);
  w.clock = reinterpret_cast<LearnerClock*>(take(sizeof(LearnerClock) / 4 + 4));
  w.xchg = chain ? take(std::max(chain_xchg_floats(B), tcc_xchg_floats(B))) : nullptr;
  w.pipe_epoch = reinterpret_cast<unsigned long long*>(take(2 * int64_t((B + SAMPLE_ROWS - 1) / SAMPLE_ROWS)));
  if (prefetch) {
    w.s_b = take(int64_t(B) * Sp); w.a_b = take(int64_t(B) * Ap); w.s2_b = take(int64_t(B) * Sp);
    w.r_b = reinterpret_cast<double*>(take(int64_t(B) * 2));
    w.done_b = reinterpret_cast<uint8_t*>(take((B + 3) / 4));
    for (int k = 0; k < 2; ++k) { w.idx2[k] = reinterpret_cast<int32_t*>(take(B)); w.wts2[k] = take(B); }
  }
  w.total = off;
  return w;
}
}  // namespace d4pg

using namespace d4pg;

struct d4pg_learner {
  d4pg_learner_config_t cfg;
  d4pg_learner_buffers_t buf;
  d4pg_replay* replay;
  d4pg_comm* comm;
  Workspace ws;
  NetDims da, dc;
  cudaGraphExec_t graph_exec[4];   // [batch parity * 2 + cold]; only [0] without the prefetch pipeline
  bool graph_ready[4];
  cudaGraphExec_t multi_exec[2];   // RUN_UNROLL warm steps in one graph, by starting batch parity (d4pg_learner_run)
  bool multi_ready[2];
  int pipe_par;                    // half of the double-buffered batch the NEXT step trains on
  int last_par;                    // ... the last step trained on
  bool prefetch_valid;             // that half already holds the next step's batch
  int64_t seen_gen;                // replay generation when it was sampled
  int64_t steps_done;
  int kernels_per_step;
  // profiling (d4pg_learner_profile_step): CUDA-event pair around every launch of an eager step
  cudaStream_t side; cudaEvent_t ev_fork, ev_join;
  ChainArgs chain_fwd_args, chain_bwd_args;
  // tcgen05 chains (precision >= 1): library-owned weight images + the per-step pack / chain descriptors
  // weight images: forward ones (packed at the start of a graph launch, then kept current by the Adam kernel) and the
  // transposed ones of the dX chains (packed every step on the side branch, off the critical path)
  uint8_t* tcc_images; TccPackArgs tcc_pack_fwd, tcc_pack_dx; TccImage tcc_img[32]; bool tcc_ok;
  cudaEvent_t ev_fork2, ev_join2;
  TccArgs tcc_fwd_args, tcc_bwd_args;
  GemmWideBatch dw_batch;
  // host-facing step: library-owned pinned staging, double-buffered by step parity (a buffer is rewritten only after
  // the H2D copy out of it, two steps earlier, has completed)
  double* host_u[4]; int32_t* host_pos[4]; float* host_losses; cudaEvent_t ev_in, ev_out, ev_h2d[4];
  int64_t host_steps;
  // results of the host-facing steps: {critic loss, actor loss, -, -} of step k land in ring slot k & 1 (async D2H queued
  // by the step itself), so a caller can read step k-1 while step k runs
  float* loss_ring[2]; cudaEvent_t ev_loss[2]; int64_t loss_steps;
  // host pipeline: library-owned ingest stream (adds + the presample of the next batch), the gate flag the step's
  // priority write-back bumps, how many gated steps were launched
  cudaStream_t ing; cudaEvent_t ev_ing; unsigned long long* gate_flag;
  bool images_dirty;               // parameters were written outside the library since the forward weight images were last current
  bool profiling;
  std::vector<cudaEvent_t> ev;
  std::vector<std::string> ev_name;
  std::vector<int> ev_reps;        // how many times the launch between the event pair was repeated
};

// step plan: 0 = one grouped launch per dependency level, 1 = cluster-fused chains (mlp_chain.cu exact fp32 /
// mlp_tc_chain.cu tcgen05).  The chain plans pay off while the batch fits one wave of clusters: measured
// on B200, batch 1024 (config 3) 409 us with chains vs 320 us per level, batch 4096 (config 5) 906 vs 733 us
// (tcgen05 levels), so batches above 512 rows always run plan 0.
static int step_plan(const d4pg_learner_config_t& c) { return c.batch > 512 ? 0 : c.chain; }
// prefetch pipeline: batch t+1 is sampled on a side branch of step t (device-side sampling only)
static bool prefetching(const d4pg_learner_config_t& c) { return c.prefetch != 0 && c.sample_mode == 1; }
// host pipeline (host-drawn uniforms / positions, cfg.prefetch): the host-facing step samples batch k on the library's
// ingest stream -- behind the caller's add(k), gated on step k-1's priority write-back -- while step k-1's backward
// pass, dW and Adam still run on the learner stream; the step graph then starts from the sampled batch.  Same double
// buffers and clock slots as the device prefetch pipeline; the order of tree operations is the reference's
// (update_priorities(k-1) -> add(k) -> sample(k), main.py / ddpg.py:200-255).
static bool host_pipe(const d4pg_learner_config_t& c) { return c.prefetch != 0 && c.sample_mode == 0 && c.use_graph != 0; }
static bool piped(const d4pg_learner_config_t& c) { return prefetching(c) || host_pipe(c); }
struct d4pg_learner;
static bool inline_wait(const d4pg_learner* L);     // the warm host-pipeline graph polls the sampler's epochs itself (tcgen05 chain plan)

// weight matrices as the tcgen05 chains consume them (F = forward image, D = transposed image for dX)
enum { U_A_F1, U_A_F2, U_A_F22, U_A_F3, U_A_D3, U_A_D22, U_A_D2, U_AT_F1, U_AT_F2, U_AT_F22, U_AT_F3,
       U_C_F1, U_C_F2, U_C_F22, U_C_F3, U_C_D3, U_C_D22, U_C_D2H, U_C_D2A, U_CT_F1, U_CT_F2, U_CT_F22, U_CT_F3, U_COUNT };

// tcgen05 chains need |s| <= 32 (one resident input chunk), |a| <= 32 (one K-tail chunk) and <= 256 atoms
static bool tcc_shapes_ok(const d4pg_learner_config_t& c) {
  return c.chain == 1 && c.batch <= 512 && c.precision >= 1 && c.obs_dim <= 32 && c.act_dim <= 32 && c.n_atoms <= 256;
}
static int tcc_setup(d4pg_learner* L) {
  L->tcc_ok = false; L->tcc_images = nullptr;
  const d4pg_learner_config_t& c = L->cfg;
  if (!tcc_shapes_ok(c)) return D4PG_OK;
  const d4pg_learner_buffers_t& b = L->buf;
  const NetDims& da = L->da; const NetDims& dc = L->dc;
  const int S = c.obs_dim, A = c.act_dim, N = c.n_atoms, H = D4PG_HIDDEN;
  TccPackArgs& pf = L->tcc_pack_fwd; TccPackArgs& pd = L->tcc_pack_dx;
  tcc_pack_begin(pf, nullptr); tcc_pack_begin(pd, nullptr);
  int use_of[U_COUNT]; bool is_dx[U_COUNT];
  auto add = [&](int id, const float* W, int ldw, int mode, int rows, int K) {
    is_dx[id] = mode == GEMM_DX;
    use_of[id] = tcc_pack_add(is_dx[id] ? pd : pf, W, ldw, mode, rows, K);
  };
  const float* Wn[2] = {b.actor, b.actor_target};
  for (int t = 0; t < 2; ++t) {
    const int base = t ? U_AT_F1 : U_A_F1;
    add(base + 0, Wn[t] + da.w_off[0], da.ld[0], GEMM_FWD, H, S);
    add(base + 1, Wn[t] + da.w_off[1], da.ld[1], GEMM_FWD, H, H);
    add(base + 2, Wn[t] + da.w_off[2], da.ld[2], GEMM_FWD, H, H);
    add(base + 3, Wn[t] + da.w_off[3], da.ld[3], GEMM_FWD, A, H);
  }
  add(U_A_D3, b.actor + da.w_off[3], da.ld[3], GEMM_DX, H, A);
  add(U_A_D22, b.actor + da.w_off[2], da.ld[2], GEMM_DX, H, H);
  add(U_A_D2, b.actor + da.w_off[1], da.ld[1], GEMM_DX, H, H);
  const float* Wm[2] = {b.critic, b.critic_target};
  for (int t = 0; t < 2; ++t) {
    const int base = t ? U_CT_F1 : U_C_F1;
    add(base + 0, Wm[t] + dc.w_off[0], dc.ld[0], GEMM_FWD, H, S);
    add(base + 1, Wm[t] + dc.w_off[1], dc.ld[1], GEMM_FWD, H, H + A);      // K = [h1 (256) | action]: 8 chunks + a tail chunk
    add(base + 2, Wm[t] + dc.w_off[2], dc.ld[2], GEMM_FWD, H, H);
    add(base + 3, Wm[t] + dc.w_off[3], dc.ld[3], GEMM_FWD, N, H);
  }
  add(U_C_D3, b.critic + dc.w_off[3], dc.ld[3], GEMM_DX, H, N);
  add(U_C_D22, b.critic + dc.w_off[2], dc.ld[2], GEMM_DX, H, H);
  add(U_C_D2H, b.critic + dc.w_off[1], dc.ld[1], GEMM_DX, H, H);
  add(U_C_D2A, b.critic + dc.w_off[1] + H, dc.ld[1], GEMM_DX, A, H);
  for (int i = 0; i < U_COUNT; ++i) D4PG_REQUIRE(use_of[i] >= 0, D4PG_ENOTSUP, "tcc_setup: too many weight images");
  const long long fwd_bytes = tcc_pack_bytes(pf), all_bytes = fwd_bytes + tcc_pack_bytes(pd);
  D4PG_CUDA_OK(cudaMalloc(&L->tcc_images, size_t(all_bytes)));
  D4PG_CUDA_OK(cudaMemset(L->tcc_images, 0, size_t(all_bytes)));
  tcc_pack_set_base(pf, L->tcc_images, 0);
  tcc_pack_set_base(pd, L->tcc_images, fwd_bytes);
  for (int i = 0; i < U_COUNT; ++i) L->tcc_img[i] = tcc_image(is_dx[i] ? pd : pf, use_of[i]);
  (void)tcc_watchdog_device();                         // allocate outside of any stream capture
  L->tcc_ok = true;
  return D4PG_OK;
}

// ---- tcgen05 chain builders (mlp_tc_chain.cu) ----------------------------------------------------------------------
struct TccCtx {
  d4pg_learner* L; const Workspace* w; const NetDims* da; const NetDims* dc;
  const float *Wa, *Wat, *Wc, *Wct;
  int B, S, A, N, Sp, Ap, Np;
};
// T: actor_target(s') -> critic_target(s', .)   (fc1 of both networks share the resident s' chunk)     ddpg.py:205-206
static void tcc_build_T(TccArgs& fa, int ci, const TccCtx& x) {
  const TccImage* U = x.L->tcc_img; const Workspace& w = *x.w; const NetDims& da = *x.da; const NetDims& dc = *x.dc;
  const int H = D4PG_HIDDEN;
  int l, p1, p2, pa;
  tcc_chain_x0(fa, ci, w.s2, x.Sp, x.S);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_x(fa, ci, l);
  p1 = tcc_slot_group(fa, ci, l, U[U_AT_F1], EPI_BIAS_RELU, x.Wat + da.b_off[0], nullptr, 0, nullptr, H, 1);
  p2 = tcc_slot_group(fa, ci, l, U[U_CT_F1], EPI_BIAS_RELU, x.Wct + dc.b_off[0], nullptr, 0, nullptr, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  p1 = tcc_slot_group(fa, ci, l, U[U_AT_F2], EPI_BIAS, x.Wat + da.b_off[1], nullptr, 0, nullptr, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  p1 = tcc_slot_group(fa, ci, l, U[U_AT_F22], EPI_BIAS_RELU, x.Wat + da.b_off[2], nullptr, 0, nullptr, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  pa = tcc_slot_group(fa, ci, l, U[U_AT_F3], EPI_BIAS_TANH, x.Wat + da.b_off[3], nullptr, 0, w.out[0], x.Ap, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p2, 8); tcc_slot_src_plane(fa, ci, l, pa, 1);
  p1 = tcc_slot_group(fa, ci, l, U[U_CT_F2], EPI_BIAS_RELU, x.Wct + dc.b_off[1], nullptr, 0, nullptr, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  p1 = tcc_slot_group(fa, ci, l, U[U_CT_F22], EPI_BIAS_RELU, x.Wct + dc.b_off[2], nullptr, 0, nullptr, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  tcc_slot_group(fa, ci, l, U[U_CT_F3], EPI_BIAS, x.Wct + dc.b_off[3], nullptr, 0, w.out[1], x.Np, 0);
}
// the actor's four layers on s (outputs kept row-major for its backward pass); returns the plane of its action output
static int tcc_build_actor(TccArgs& fa, int ci, const TccCtx& x, int* critic_h1_plane) {
  const TccImage* U = x.L->tcc_img; const Workspace& w = *x.w; const NetDims& da = *x.da; const NetDims& dc = *x.dc;
  const int H = D4PG_HIDDEN;
  int l, p1;
  tcc_chain_x0(fa, ci, w.s, x.Sp, x.S);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_x(fa, ci, l);
  p1 = tcc_slot_group(fa, ci, l, U[U_A_F1], EPI_BIAS_RELU, x.Wa + da.b_off[0], nullptr, 0, w.h1[3], H, 1);
  if (critic_h1_plane)       // critic fc1 on the same resident s chunk (h1 of critic(s, actor(s)); same values as chain Q's)
    *critic_h1_plane = tcc_slot_group(fa, ci, l, U[U_C_F1], EPI_BIAS_RELU, x.Wc + dc.b_off[0], nullptr, 0, nullptr, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  p1 = tcc_slot_group(fa, ci, l, U[U_A_F2], EPI_BIAS, x.Wa + da.b_off[1], nullptr, 0, w.h2[3], H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  p1 = tcc_slot_group(fa, ci, l, U[U_A_F22], EPI_BIAS_RELU, x.Wa + da.b_off[2], nullptr, 0, w.h3[3], H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  return tcc_slot_group(fa, ci, l, U[U_A_F3], EPI_BIAS_TANH, x.Wa + da.b_off[3], nullptr, 0, w.out[3], x.Ap, 1);
}
// P: actor(s) -> critic(s, actor(s))                                                                     ddpg.py:236-238
static void tcc_build_P(TccArgs& fa, int ci, const TccCtx& x) {
  const TccImage* U = x.L->tcc_img; const Workspace& w = *x.w; const NetDims& dc = *x.dc;
  const int H = D4PG_HIDDEN;
  int l, p1, p2 = -1;
  const int pa = tcc_build_actor(fa, ci, x, &p2);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p2, 8); tcc_slot_src_plane(fa, ci, l, pa, 1);
  p1 = tcc_slot_group(fa, ci, l, U[U_C_F2], EPI_BIAS_RELU, x.Wc + dc.b_off[1], nullptr, 0, w.h2[4], H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  p1 = tcc_slot_group(fa, ci, l, U[U_C_F22], EPI_BIAS_RELU, x.Wc + dc.b_off[2], nullptr, 0, w.h3[4], H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  tcc_slot_group(fa, ci, l, U[U_C_F3], EPI_BIAS, x.Wc + dc.b_off[3], nullptr, 0, w.out[4], x.Np, 0);
}
// critic(s, `act`): the resident chunk holds s for fc1, then the action rows (fc2's K tail)                ddpg.py:208
static void tcc_build_Q(TccArgs& fa, int ci, const TccCtx& x, const float* act, float* h1, float* h2, float* h3, float* logits) {
  const TccImage* U = x.L->tcc_img; const Workspace& w = *x.w; const NetDims& dc = *x.dc;
  const int H = D4PG_HIDDEN;
  int l, p1;
  tcc_chain_x0(fa, ci, w.s, x.Sp, x.S);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_x(fa, ci, l); tcc_slot_reconvert_x(fa, ci, l, act, x.Ap, x.A);
  p1 = tcc_slot_group(fa, ci, l, U[U_C_F1], EPI_BIAS_RELU, x.Wc + dc.b_off[0], nullptr, 0, h1, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8); tcc_slot_src_x(fa, ci, l);
  p1 = tcc_slot_group(fa, ci, l, U[U_C_F2], EPI_BIAS_RELU, x.Wc + dc.b_off[1], nullptr, 0, h2, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  p1 = tcc_slot_group(fa, ci, l, U[U_C_F22], EPI_BIAS_RELU, x.Wc + dc.b_off[2], nullptr, 0, h3, H, 1);
  l = tcc_slot_begin(fa, ci); tcc_slot_src_plane(fa, ci, l, p1, 8);
  tcc_slot_group(fa, ci, l, U[U_C_F3], EPI_BIAS, x.Wc + dc.b_off[3], nullptr, 0, logits, x.Np, 0);
}
// C: critic loss, dlogits_q -> fc3 -> fc2_2 -> fc2[:, :H]                                                  ddpg.py:230
static void tcc_build_bwd_C(TccArgs& ba, int ci, const TccCtx& x) {
  const TccImage* U = x.L->tcc_img; const Workspace& w = *x.w;
  const int H = D4PG_HIDDEN;
  int l, p1;
  tcc_chain_pre(ba, ci, w.dlogits_q, x.Np, x.N);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_pre(ba, ci, l);
  p1 = tcc_slot_group(ba, ci, l, U[U_C_D3], EPI_RELU_MASK, nullptr, w.h3[2], H, w.c_dz22, H, 1);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_plane(ba, ci, l, p1, 8);
  p1 = tcc_slot_group(ba, ci, l, U[U_C_D22], EPI_RELU_MASK, nullptr, w.h2[2], H, w.c_dz2, H, 1);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_plane(ba, ci, l, p1, 8);
  tcc_slot_group(ba, ci, l, U[U_C_D2H], EPI_RELU_MASK, nullptr, w.h1[2], H, w.c_dz1, H, 0);
}
// P: policy loss, dlogits_pi -> critic fc3 -> fc2_2 -> fc2[:, H:] (d action, tanh') -> actor fc3 -> fc2_2 -> fc2   ddpg.py:242
static void tcc_build_bwd_P(TccArgs& ba, int ci, const TccCtx& x) {
  const TccImage* U = x.L->tcc_img; const Workspace& w = *x.w;
  const int H = D4PG_HIDDEN;
  int l, p1;
  tcc_chain_pre(ba, ci, w.dlogits_pi, x.Np, x.N);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_pre(ba, ci, l);
  p1 = tcc_slot_group(ba, ci, l, U[U_C_D3], EPI_RELU_MASK, nullptr, w.h3[4], H, nullptr, H, 1);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_plane(ba, ci, l, p1, 8);
  p1 = tcc_slot_group(ba, ci, l, U[U_C_D22], EPI_RELU_MASK, nullptr, w.h2[4], H, nullptr, H, 1);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_plane(ba, ci, l, p1, 8);
  p1 = tcc_slot_group(ba, ci, l, U[U_C_D2A], EPI_TANH_MASK, nullptr, w.out[3], x.Ap, w.a_dz3, x.Ap, 1);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_plane(ba, ci, l, p1, 1);
  p1 = tcc_slot_group(ba, ci, l, U[U_A_D3], EPI_RELU_MASK, nullptr, w.h3[3], H, w.a_dz22, H, 1);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_plane(ba, ci, l, p1, 8);
  p1 = tcc_slot_group(ba, ci, l, U[U_A_D22], EPI_NONE, nullptr, nullptr, 0, w.a_dh2, H, 1);
  l = tcc_slot_begin(ba, ci); tcc_slot_src_plane(ba, ci, l, p1, 8);
  tcc_slot_group(ba, ci, l, U[U_A_D2], EPI_RELU_MASK, nullptr, w.h1[3], H, w.a_dz1, H, 0);
}

// idempotent launches (pure functions of their inputs) are repeated in profile mode
constexpr int PROFILE_REPS = 16;

// par: half of the double-buffered batch this step trains on; cold: sample it first (no valid prefetch)
// pack_fwd: re-pack the forward weight images first (start of a graph launch / eager step: the caller may have changed
// the parameters); later steps of one multi-step graph rely on the images the previous step's Adam kernel wrote
static int enqueue_step(d4pg_learner* L, cudaStream_t st, int par, bool cold, bool pack_fwd = true) {
  const d4pg_learner_config_t& c = L->cfg;
  const d4pg_learner_buffers_t& b = L->buf;
  Workspace w = L->ws;                               // local copy: the batch pointers follow `par`
  const bool pf = piped(c);
  int32_t* bidx = b.idx; float* bwts = b.weights;
  if (pf) {
    if (par) { w.s = w.s_b; w.a = w.a_b; w.s2 = w.s2_b; w.r = w.r_b; w.done = w.done_b; }
    bidx = w.idx2[par]; bwts = w.wts2[par];
  }
  const NetDims& da = L->da; const NetDims& dc = L->dc;
  const int B = c.batch, S = c.obs_dim, A = c.act_dim, N = c.n_atoms, H = D4PG_HIDDEN;
  const int Sp = pitch4(S), Ap = pitch4(A), Np = pitch4(N);          // activation row pitches
  const int* la = da.ld; const int* lc = dc.ld;                        // weight row pitches per layer
  int rc; int nk = 0;
#define LEVEL(gb) RUN(gemm_launch(gb, c.precision, st))
#define RUN(expr)                                                                          \
  do {                                                                                     \
    if (L->profiling) { cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);    \
      std::string nm0(#expr);                                                              \
      /* the loss kernel also advances the sampler clock under the prefetch pipeline: not idempotent there */ \
      const bool rep = nm0.rfind("gemm_launch", 0) == 0 || (nm0.rfind("launch_heads", 0) == 0 && !pf) || \
                       nm0.rfind("launch_mlp_chain", 0) == 0 || nm0.rfind("launch_mlp_tc_chain", 0) == 0; \
      cudaEventRecord(e0, st); rc = (expr);                                                \
      for (int _r = 1; rep && _r < PROFILE_REPS && rc == 0; ++_r) rc = (expr);             \
      cudaEventRecord(e1, st);                                                             \
      L->ev.push_back(e0); L->ev.push_back(e1); L->ev_reps.push_back(rep ? PROFILE_REPS : 1); \
      std::string nm(#expr); L->ev_name.push_back(nm.substr(0, nm.find('('))); }           \
    else rc = (expr);                                                                      \
    if (rc) return rc;                                                                     \
    ++nk;                                                                                  \
  } while (0)

  // 1. sample + gather (ddpg.py:187-197).  The same kernel derives this step's device-side
  //    scalars (Adam bias corrections, PER beta, Philox counter) from the learner clock.
  ClockParams cp{c.lr_actor, c.lr_critic, c.beta1, c.beta2, c.per_beta0, c.per_beta_final,
                 c.per_beta_iters > 0 ? c.per_beta_iters : 1};
  if (!pf || cold)
    RUN(learner_sample(L->replay, B, c.prioritized, c.sample_mode == 0 ? b.uniforms : nullptr,
                       (c.sample_mode == 0 && !c.prioritized) ? b.positions : nullptr,
                       c.philox_seed, w.clock, cp,
                       bidx, bwts, w.s, w.a, w.r, w.s2, w.done, Sp, Ap, pf ? par : -1, st));

  const float* Wa = b.actor; const float* Wat = b.actor_target; const float* Wc = b.critic; const float* Wct = b.critic_target;
  GemmBatch g;
  const int plan = step_plan(c);
  const bool tcc = plan == 1 && c.precision >= 1 && L->tcc_ok;       // tcgen05 cluster chains
  // corrected-semantics switch (SURVEY.md H7, loss_flags & 4): the actor gradient goes through the critic AFTER this
  // step's critic update (the reference uses the stale local copy, ddpg.py:229-247).  Two half steps: critic forward /
  // loss / backward / Adam, then the policy pass through the updated critic, actor backward / Adam.
  const bool h7 = (c.loss_flags & 4) != 0;
  D4PG_REQUIRE(!h7 || (tcc && c.world_size <= 1), D4PG_ENOTSUP, "post-update-critic actor gradient needs the tcgen05 chain plan (precision tf32x3 / tf32, chain plan, batch <= 512) on one GPU");
  const bool chain = plan == 1 && !tcc;
  const bool pre_ok = chain && c.precision == 0 && A <= 8;             // pre-layers: fp32 tile, |a| <= 8
  if (tcc) {
    // 2''. the same three forward chains on the tensor cores (mlp_tc_chain.cu): clusters of 8 CTAs own 64 rows,
    // every layer a tcgen05.mma tile.  The hi/lo weight images are re-packed first (Adam / Polyak changed them).
    if (pack_fwd) RUN(launch_tcc_pack(L->tcc_pack_fwd, st));
    // the transposed images of the dX chains are needed ~35 us from now: packed on the side branch
    D4PG_CUDA_OK(cudaEventRecord(L->ev_fork2, st));
    D4PG_CUDA_OK(cudaStreamWaitEvent(L->side, L->ev_fork2, 0));
    RUN(launch_tcc_pack(L->tcc_pack_dx, L->side));
    D4PG_CUDA_OK(cudaEventRecord(L->ev_join2, L->side));
    const TccImage* U = L->tcc_img;
    TccArgs& fa = L->tcc_fwd_args;
    tcc_args_begin(fa, B, reinterpret_cast<uint8_t*>(w.xchg), c.precision == 1 ? 3 : 1); fa.step_slot = 1;
    TccCtx cx{L, &w, &da, &dc, Wa, Wat, Wc, Wct, B, S, A, N, Sp, Ap, Np};
    tcc_build_T(fa, 0, cx);                                      // chain 0  T: actor_target(s') -> critic_target(s', .)
    if (h7) tcc_build_actor(fa, 1, cx, nullptr);                 // chain 1  (post-update plan) the actor alone; the critic pass follows the critic's Adam
    else tcc_build_P(fa, 1, cx);                                 // chain 1  P: actor(s) -> critic(s, actor(s))
    tcc_build_Q(fa, 2, cx, w.a, w.h1[2], w.h2[2], w.h3[2], w.out[2]);   // chain 2  Q: critic(s, a)
    if (host_pipe(c) && !cold && inline_wait(L)) {
      // warm host-pipeline variant: the batch comes from the ingest stream's sample kernel; instead of a stream event
      // (event + graph start: ~6 us after the sample ends) every CTA polls the epochs that kernel publishes
      fa.wait_epoch = w.pipe_epoch; fa.wait_clock = reinterpret_cast<const long long*>(&w.clock->steps_done);
      fa.wait_n = cdiv(B, SAMPLE_ROWS);
    }
    RUN(launch_mlp_tc_chain(fa, st));
  } else if (chain) {
    // 2'. the three forward chains of the step as ONE cluster launch (mlp_chain.cu):
    //   chain 0  T: actor_target(s') -> critic_target(s', .)      ddpg.py:205-206
    //   chain 1  P: actor(s) -> critic(s, actor(s))                ddpg.py:236-238 (fc1 of the critic is recomputed: K=|s|)
    //   chain 2  Q: critic(s, a)                                   ddpg.py:208
    // The block scheduler fills SMs in launch order: the two 8-layer chains come first so that each of their CTAs
    // gets an SM of its own, and the short 4-layer chain is the one that doubles up (measured with %smid: in the
    // order T,Q,P 38 SMs hosted a T and a P CTA while 52 SMs hosted a lone Q CTA; forward launch 49 us)
    ChainArgs& ca = L->chain_fwd_args;
    chain_args_begin(ca, B, w.xchg, c.precision);
    ChainSlot sl; int at3 = -1, ct1, q1, a3 = -1, c1;
    (void)at3; (void)a3;
    sl = chain_fwd(Wat + da.w_off[0], la[0], Wat + da.b_off[0], H, S, EPI_BIAS_RELU, w.h1[0], H, 1); chain_src_global(sl, w.s2, Sp); int t = chain_add(ca, 0, sl);
    sl = chain_fwd(Wat + da.w_off[1], la[1], Wat + da.b_off[1], H, H, EPI_BIAS, w.h2[0], H, 1); chain_src_plane(sl, t); t = chain_add(ca, 0, sl);
    sl = chain_fwd(Wat + da.w_off[2], la[2], Wat + da.b_off[2], H, H, EPI_BIAS_RELU, w.h3[0], H, 1); chain_src_plane(sl, t); t = chain_add(ca, 0, sl);
    // the 6-wide actor fc3 is a PRE-LAYER of the critic's fc2 slot (every CTA computes it for its 32 rows) instead of
    // a slot of its own, when it fits (|a| <= 8, fp32 tile); otherwise it is a slot that publishes 8 plane rows
    const int t22 = t;
    if (pre_ok) {
      sl = chain_fwd(Wct + dc.w_off[0], lc[0], Wct + dc.b_off[0], H, S, EPI_BIAS_RELU, w.h1[1], H, 1); chain_src_global(sl, w.s2, Sp); ct1 = chain_add(ca, 0, sl);
      sl = chain_fwd(Wct + dc.w_off[1], lc[1], Wct + dc.b_off[1], H, H + A, EPI_BIAS_RELU, w.h2[1], H, 1); chain_src_plane(sl, ct1);
      chain_pre_layer(sl, Wat + da.w_off[3], la[3], Wat + da.b_off[3], nullptr, 0, A, H, EPI_BIAS_TANH, w.out[0], Ap, t22, H, false);
      t = chain_add(ca, 0, sl);
    } else {
    sl = chain_fwd(Wat + da.w_off[3], la[3], Wat + da.b_off[3], A, H, EPI_BIAS_TANH, w.out[0], Ap, 1); chain_src_plane(sl, t); at3 = chain_add(ca, 0, sl);
    sl = chain_fwd(Wct + dc.w_off[0], lc[0], Wct + dc.b_off[0], H, S, EPI_BIAS_RELU, w.h1[1], H, 1); chain_src_global(sl, w.s2, Sp); ct1 = chain_add(ca, 0, sl);
    sl = chain_fwd(Wct + dc.w_off[1], lc[1], Wct + dc.b_off[1], H, H + A, EPI_BIAS_RELU, w.h2[1], H, 1); chain_src_plane(sl, ct1); chain_src2_plane(sl, H, at3); t = chain_add(ca, 0, sl);
    }
    sl = chain_fwd(Wct + dc.w_off[2], lc[2], Wct + dc.b_off[2], H, H, EPI_BIAS_RELU, w.h3[1], H, 1); chain_src_plane(sl, t); t = chain_add(ca, 0, sl);
    sl = chain_fwd(Wct + dc.w_off[3], lc[3], Wct + dc.b_off[3], N, H, EPI_BIAS, w.out[1], Np, 0); chain_src_plane(sl, t); chain_add(ca, 0, sl);

    sl = chain_fwd(Wc + dc.w_off[0], lc[0], Wc + dc.b_off[0], H, S, EPI_BIAS_RELU, w.h1[2], H, 1); chain_src_global(sl, w.s, Sp); q1 = chain_add(ca, 2, sl);
    sl = chain_fwd(Wc + dc.w_off[1], lc[1], Wc + dc.b_off[1], H, H + A, EPI_BIAS_RELU, w.h2[2], H, 1); chain_src_plane(sl, q1); chain_src2_global(sl, H, w.a, Ap); t = chain_add(ca, 2, sl);
    sl = chain_fwd(Wc + dc.w_off[2], lc[2], Wc + dc.b_off[2], H, H, EPI_BIAS_RELU, w.h3[2], H, 1); chain_src_plane(sl, t); t = chain_add(ca, 2, sl);
    sl = chain_fwd(Wc + dc.w_off[3], lc[3], Wc + dc.b_off[3], N, H, EPI_BIAS, w.out[2], Np, 0); chain_src_plane(sl, t); chain_add(ca, 2, sl);

    sl = chain_fwd(Wa + da.w_off[0], la[0], Wa + da.b_off[0], H, S, EPI_BIAS_RELU, w.h1[3], H, 1); chain_src_global(sl, w.s, Sp); t = chain_add(ca, 1, sl);
    sl = chain_fwd(Wa + da.w_off[1], la[1], Wa + da.b_off[1], H, H, EPI_BIAS, w.h2[3], H, 1); chain_src_plane(sl, t); t = chain_add(ca, 1, sl);
    sl = chain_fwd(Wa + da.w_off[2], la[2], Wa + da.b_off[2], H, H, EPI_BIAS_RELU, w.h3[3], H, 1); chain_src_plane(sl, t); t = chain_add(ca, 1, sl);
    const int a22 = t;
    if (pre_ok) {
      sl = chain_fwd(Wc + dc.w_off[0], lc[0], Wc + dc.b_off[0], H, S, EPI_BIAS_RELU, nullptr, H, 1); chain_src_global(sl, w.s, Sp); c1 = chain_add(ca, 1, sl);
      sl = chain_fwd(Wc + dc.w_off[1], lc[1], Wc + dc.b_off[1], H, H + A, EPI_BIAS_RELU, w.h2[4], H, 1); chain_src_plane(sl, c1);
      chain_pre_layer(sl, Wa + da.w_off[3], la[3], Wa + da.b_off[3], nullptr, 0, A, H, EPI_BIAS_TANH, w.out[3], Ap, a22, H, false);
      t = chain_add(ca, 1, sl);
    } else {
    sl = chain_fwd(Wa + da.w_off[3], la[3], Wa + da.b_off[3], A, H, EPI_BIAS_TANH, w.out[3], Ap, 1); chain_src_plane(sl, t); a3 = chain_add(ca, 1, sl);
    sl = chain_fwd(Wc + dc.w_off[0], lc[0], Wc + dc.b_off[0], H, S, EPI_BIAS_RELU, nullptr, H, 1); chain_src_global(sl, w.s, Sp); c1 = chain_add(ca, 1, sl);
    sl = chain_fwd(Wc + dc.w_off[1], lc[1], Wc + dc.b_off[1], H, H + A, EPI_BIAS_RELU, w.h2[4], H, 1); chain_src_plane(sl, c1); chain_src2_plane(sl, H, a3); t = chain_add(ca, 1, sl);
    }
    sl = chain_fwd(Wc + dc.w_off[2], lc[2], Wc + dc.b_off[2], H, H, EPI_BIAS_RELU, w.h3[4], H, 1); chain_src_plane(sl, t); t = chain_add(ca, 1, sl);
    sl = chain_fwd(Wc + dc.w_off[3], lc[3], Wc + dc.b_off[3], N, H, EPI_BIAS, w.out[4], Np, 0); chain_src_plane(sl, t); chain_add(ca, 1, sl);
    RUN(launch_mlp_chain(ca, st));
  } else {
  // 2. forward level 1: fc1 of actor_target(s'), critic_target(s'), critic(s), actor(s)
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_fwd(w.s2, Sp, nullptr, 0, 0, Wat + da.w_off[0], la[0], Wat + da.b_off[0], w.h1[0], H, B, H, S, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.s2, Sp, nullptr, 0, 0, Wct + dc.w_off[0], lc[0], Wct + dc.b_off[0], w.h1[1], H, B, H, S, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.s, Sp, nullptr, 0, 0, Wc + dc.w_off[0], lc[0], Wc + dc.b_off[0], w.h1[2], H, B, H, S, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.s, Sp, nullptr, 0, 0, Wa + da.w_off[0], la[0], Wa + da.b_off[0], w.h1[3], H, B, H, S, EPI_BIAS_RELU));
  LEVEL(g);
  // level 2: fc2 (actor: no activation, models.py:36; critic: cat(h1, a) + relu, models.py:80)
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_fwd(w.h1[0], H, nullptr, 0, 0, Wat + da.w_off[1], la[1], Wat + da.b_off[1], w.h2[0], H, B, H, H, EPI_BIAS));
  gemm_batch_add(g, gemm_fwd(w.h1[2], H, w.a, Ap, H, Wc + dc.w_off[1], lc[1], Wc + dc.b_off[1], w.h2[2], H, B, H, H + A, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.h1[3], H, nullptr, 0, 0, Wa + da.w_off[1], la[1], Wa + da.b_off[1], w.h2[3], H, B, H, H, EPI_BIAS));
  LEVEL(g);
  // level 3: fc2_2 + relu
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_fwd(w.h2[0], H, nullptr, 0, 0, Wat + da.w_off[2], la[2], Wat + da.b_off[2], w.h3[0], H, B, H, H, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.h2[2], H, nullptr, 0, 0, Wc + dc.w_off[2], lc[2], Wc + dc.b_off[2], w.h3[2], H, B, H, H, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.h2[3], H, nullptr, 0, 0, Wa + da.w_off[2], la[2], Wa + da.b_off[2], w.h3[3], H, B, H, H, EPI_BIAS_RELU));
  LEVEL(g);
  // level 4: fc3 (actor: tanh; critic: logits)
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_fwd(w.h3[0], H, nullptr, 0, 0, Wat + da.w_off[3], la[3], Wat + da.b_off[3], w.out[0], Ap, B, A, H, EPI_BIAS_TANH));
  gemm_batch_add(g, gemm_fwd(w.h3[2], H, nullptr, 0, 0, Wc + dc.w_off[3], lc[3], Wc + dc.b_off[3], w.out[2], Np, B, N, H, EPI_BIAS));
  gemm_batch_add(g, gemm_fwd(w.h3[3], H, nullptr, 0, 0, Wa + da.w_off[3], la[3], Wa + da.b_off[3], w.out[3], Ap, B, A, H, EPI_BIAS_TANH));
  LEVEL(g);
  // level 5: critic_target.fc2([h1t, a_t(s')]) and critic.fc2([h1, actor(s)]) (h1 of the critic is reused)
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_fwd(w.h1[1], H, w.out[0], Ap, H, Wct + dc.w_off[1], lc[1], Wct + dc.b_off[1], w.h2[1], H, B, H, H + A, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.h1[2], H, w.out[3], Ap, H, Wc + dc.w_off[1], lc[1], Wc + dc.b_off[1], w.h2[4], H, B, H, H + A, EPI_BIAS_RELU));
  LEVEL(g);
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_fwd(w.h2[1], H, nullptr, 0, 0, Wct + dc.w_off[2], lc[2], Wct + dc.b_off[2], w.h3[1], H, B, H, H, EPI_BIAS_RELU));
  gemm_batch_add(g, gemm_fwd(w.h2[4], H, nullptr, 0, 0, Wc + dc.w_off[2], lc[2], Wc + dc.b_off[2], w.h3[4], H, B, H, H, EPI_BIAS_RELU));
  LEVEL(g);
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_fwd(w.h3[1], H, nullptr, 0, 0, Wct + dc.w_off[3], lc[3], Wct + dc.b_off[3], w.out[1], Np, B, N, H, EPI_BIAS));
  gemm_batch_add(g, gemm_fwd(w.h3[4], H, nullptr, 0, 0, Wc + dc.w_off[3], lc[3], Wc + dc.b_off[3], w.out[4], Np, B, N, H, EPI_BIAS));
  LEVEL(g);

  }

  // 3. heads: softmaxes, projection, CE loss, td, priorities, logit gradients (ddpg.py:214-222,236-238)
  HeadsArgs ha{};
  ha.target_logits = w.out[1]; ha.q_logits = w.out[2]; ha.pi_logits = h7 ? nullptr : w.out[4];
  ha.rewards = w.r; ha.dones = w.done; ha.B = B; ha.N = N; ha.flags = 0; ha.ld = Np;
  ha.v_min = c.v_min; ha.v_max = c.v_max; ha.delta = (c.v_max - c.v_min) / double(N - 1);
  // live projection discounts with gamma even for n_steps>1 (SURVEY.md H5); mode 1 uses gamma**n (ddpg.py:24)
  ha.discount = (c.proj_mode == 1) ? pow(c.gamma, double(c.n_steps)) : c.gamma; ha.prio_eps = c.prio_eps;
  ha.grad_scale = 1.0f / (float(B) * float(c.world_size > 1 ? c.world_size : 1));
  ha.m = w.m; ha.target_probs = w.target_probs; ha.q_probs = w.q_probs;
  ha.loss_rows = w.loss_rows; ha.td = b.td; ha.prio = b.prio; ha.dlogits_q = w.dlogits_q;
  ha.pi_rows = w.pi_rows; ha.dlogits_pi = w.dlogits_pi;
  ha.is_weights = ((c.loss_flags & 1) && c.prioritized) ? bwts : nullptr;
  ha.sampler_clock = pf ? w.clock : nullptr;          // sample(t) is done, sample(t+1) not yet launched
  ha.ce_priority = (c.loss_flags & 2) ? 1 : 0;
  RUN(launch_heads(ha, c.proj_mode, st));

  // 4. priorities into the trees (ddpg.py:252-255): independent of the backward pass, so it runs
  //    on a forked branch (side stream -> parallel graph branch) and joins before the step ends
  if (c.prioritized || pf) {
    D4PG_CUDA_OK(cudaEventRecord(L->ev_fork, st));
    D4PG_CUDA_OK(cudaStreamWaitEvent(L->side, L->ev_fork, 0));
    // host pipeline: the write-back also opens the ingest gate of step k+1 (its tree add / presample wait for this step's
    // loss kernel -- which advanced the sampler clock -- and for the priorities)
    if (c.prioritized) RUN(launch_tree_update(L->replay, B, bidx, b.prio, L->side, host_pipe(c) ? L->gate_flag : nullptr));
    else if (host_pipe(c)) RUN(launch_gate_signal(L->gate_flag, L->side));
    if (prefetching(c)) {
      // 4'. the NEXT step's batch, sampled from the just-updated trees into the other half of the batch buffers
      // while this step's backward pass, dW and Adam run (it needs the trees, not the weights)
      const int q = par ^ 1;
      const Workspace& o = L->ws;
      RUN(learner_sample(L->replay, B, c.prioritized, nullptr, nullptr, c.philox_seed, w.clock, cp, o.idx2[q], o.wts2[q],
                         q ? o.s_b : o.s, q ? o.a_b : o.a, q ? o.r_b : o.r, q ? o.s2_b : o.s2, q ? o.done_b : o.done,
                         Sp, Ap, q, L->side));
    }
    if (pf) {                                          // the caller-visible copies of this step's indices / IS weights (off the
      // path to the next batch: after the write-back and the prefetch)
      D4PG_CUDA_OK(cudaMemcpyAsync(b.idx, bidx, size_t(B) * sizeof(int32_t), cudaMemcpyDeviceToDevice, L->side));
      if (b.weights && c.prioritized)
        D4PG_CUDA_OK(cudaMemcpyAsync(b.weights, bwts, size_t(B) * sizeof(float), cudaMemcpyDeviceToDevice, L->side));
    }
    D4PG_CUDA_OK(cudaEventRecord(L->ev_join, L->side));
  }

  float* Ga = b.grad_actor; float* Gc = b.grad_critic;
  // data parallel with IPC-mapped peers: this step's gradients go straight into this rank's half of the exchange
  // buffer (double-buffered by step parity), the Adam kernel sums all ranks' halves over NVLink
  PeerInfo peers{};
  const bool peer_mode = c.world_size > 1 && comm_peer_info(L->comm, &peers);
  const int gpar = pf ? par : int(L->steps_done & 1);
  const bool inline_sync_possible = chain || tcc;
  // Exchange shapes (D4PG_COMM_MODE=mc|mc2|pull|rs; default: "mc" from D4PG_COMM_MC_FROM = 3 ranks up when the communicator
  // set up a multicast object, else "pull"):
  //   "mc"   in-switch reduction: ONE hop and 1.15 MB inbound per rank -- the Adam kernel's multimem.ld_reduce over an NVLS
  //          multicast object returns the sum over all ranks, added by the NVSwitch (8 ranks: 101.6 us/step);
  //   "mc2"  its two-phase form: every rank ld_reduces its 1/N slice and multimem.st's it to everyone (2 x 1.15 MB per GPU
  //          whatever N), then a second flag hop (8 ranks: 100.9 us; 2 ranks: 98.9 vs 90.5 for "mc");
  //   "pull" one hop, every rank sums all N halves inside Adam (N x 1.15 MB inbound over NVLink; 2 ranks 89.2 us -- the
  //          fastest there -- 8 ranks 111.9);
  //   "rs"   reduce-scatter + all-gather over peer memory: TWO hops of 16-B remote accesses (loses everywhere: 130.7 us at 8).
  static const int comm_mode = [] { const char* e = getenv("D4PG_COMM_MODE");
                                    return !e ? 0 : (e[0] == 'p' ? 1 : (e[0] == 'r' ? 2 : (e[0] == 'm' && e[1] == 'c' && e[2] == '2' ? 4 : 3))); }();
  static const int mc_from = [] { const char* e = getenv("D4PG_COMM_MC_FROM"); return e ? atoi(e) : 3; }();
  static const int mc2_from = [] { const char* e = getenv("D4PG_COMM_MC2_FROM"); return e ? atoi(e) : 1000; }();
  const bool mc_avail = peer_mode && peers.mc != nullptr && inline_sync_possible;
  const bool peer_mc2 = mc_avail && (comm_mode == 4 || (comm_mode == 0 && peers.world >= mc2_from));
  const bool peer_mc = mc_avail && !peer_mc2 && (comm_mode == 3 || (comm_mode == 0 && peers.world >= mc_from));
  const bool peer_rs = peer_mode && !peer_mc && !peer_mc2 && comm_mode == 2;
  const bool use_mc_buf = peer_mc || peer_mc2;
  // this step's gradients go into this rank's half of the exchange buffer: the multicast-bound one when the in-switch
  // reduction is set up, else the IPC-mapped one the peers read directly
  if (peer_mode) { Ga = (use_mc_buf ? peers.mc_uc : peers.x[peers.rank]) + int64_t(gpar) * peers.n; Gc = Ga + da.total; }
  if (B >= 1024)                // dW levels run split-K with fp32 atomics: the gradient buffer must start at zero
    D4PG_CUDA_OK(cudaMemsetAsync(Ga, 0, size_t(da.total + dc.total) * sizeof(float), st));
  if (tcc) {
    // 5''. both dX chains on the tensor cores (transposed weight images; masks applied by the epilogue)
    const TccImage* U = L->tcc_img;
    D4PG_CUDA_OK(cudaStreamWaitEvent(st, L->ev_join2, 0));       // transposed weight images are packed
    TccArgs& ba = L->tcc_bwd_args;
    tcc_args_begin(ba, B, reinterpret_cast<uint8_t*>(w.xchg), c.precision == 1 ? 3 : 1); ba.step_slot = 5;
    TccCtx cx{L, &w, &da, &dc, Wa, Wat, Wc, Wct, B, S, A, N, Sp, Ap, Np};
    tcc_build_bwd_C(ba, 0, cx);                                  // C: critic loss
    if (!h7) tcc_build_bwd_P(ba, 1, cx);                         // P: policy loss (PRE-update critic weights, SURVEY.md H7)
    RUN(launch_mlp_tc_chain(ba, st));
  }
  if (chain) {
    // 5'. both dX chains as ONE cluster launch, then every dW of the step as ONE grouped launch
    //   C: critic loss  dlogits_q  -> fc3 -> fc2_2 -> fc2[:, :H]                         ddpg.py:230
    //   P: policy loss  dlogits_pi -> fc3 -> fc2_2 -> fc2[:, H:] (d action, tanh') ->
    //                   actor fc3 -> fc2_2 -> fc2   (PRE-update critic weights, SURVEY.md H7)  ddpg.py:242
    ChainArgs& cb = L->chain_bwd_args;
    chain_args_begin(cb, B, w.xchg, c.precision); cb.trace_base = 6 * CHAIN_MAX_SLOTS;
    ChainSlot sl; int t;
    sl = chain_dx(Wc + dc.w_off[3], lc[3], H, N, EPI_RELU_MASK, w.h3[2], H, w.c_dz22, H, 1); chain_src_global(sl, w.dlogits_q, Np); t = chain_add(cb, 0, sl);
    sl = chain_dx(Wc + dc.w_off[2], lc[2], H, H, EPI_RELU_MASK, w.h2[2], H, w.c_dz2, H, 1); chain_src_plane(sl, t); t = chain_add(cb, 0, sl);
    sl = chain_dx(Wc + dc.w_off[1], lc[1], H, H, EPI_RELU_MASK, w.h1[2], H, w.c_dz1, H, 0); chain_src_plane(sl, t); chain_add(cb, 0, sl);

    sl = chain_dx(Wc + dc.w_off[3], lc[3], H, N, EPI_RELU_MASK, w.h3[4], H, w.p_dz22, H, 1); chain_src_global(sl, w.dlogits_pi, Np); t = chain_add(cb, 1, sl);
    sl = chain_dx(Wc + dc.w_off[2], lc[2], H, H, EPI_RELU_MASK, w.h2[4], H, w.p_dz2, H, 1); chain_src_plane(sl, t); t = chain_add(cb, 1, sl);
    if (pre_ok) {      // d action (6 wide) as a pre-layer of the step through actor fc3
      sl = chain_dx(Wa + da.w_off[3], la[3], H, A, EPI_RELU_MASK, w.h3[3], H, w.a_dz22, H, 1);
      chain_pre_layer(sl, Wc + dc.w_off[1] + H, lc[1], nullptr, w.out[3], Ap, A, H, EPI_TANH_MASK, w.a_dz3, Ap, t, H, true);
      t = chain_add(cb, 1, sl);
    } else {
    sl = chain_dx(Wc + dc.w_off[1] + H, lc[1], A, H, EPI_TANH_MASK, w.out[3], Ap, w.a_dz3, Ap, 1); chain_src_plane(sl, t); t = chain_add(cb, 1, sl);
    sl = chain_dx(Wa + da.w_off[3], la[3], H, A, EPI_RELU_MASK, w.h3[3], H, w.a_dz22, H, 1); chain_src_plane(sl, t); t = chain_add(cb, 1, sl);
    }
    sl = chain_dx(Wa + da.w_off[2], la[2], H, H, EPI_NONE, nullptr, 0, w.a_dh2, H, 1); chain_src_plane(sl, t); t = chain_add(cb, 1, sl);
    sl = chain_dx(Wa + da.w_off[1], la[1], H, H, EPI_RELU_MASK, w.h1[3], H, w.a_dz1, H, 0); chain_src_plane(sl, t); chain_add(cb, 1, sl);
    RUN(launch_mlp_chain(cb, st));
  }
  if (chain || tcc) {                     // every dW of the step as ONE grouped launch
    GemmWideBatch& gw = L->dw_batch;
    PeerSignal sig1{};
    if (peer_mode) sig1 = comm_peer_signal(peers, 0);
    gemm_wide_begin(gw, peer_mode ? &sig1 : nullptr);              // its last CTA signals the peers
    gemm_wide_add(gw, gemm_dw(w.c_dz22, H, w.h2[2], H, Gc + dc.w_off[2], lc[2], Gc + dc.b_off[2], H, H, B));
    gemm_wide_add(gw, gemm_dw(w.c_dz2, H, w.h1[2], H, Gc + dc.w_off[1], lc[1], Gc + dc.b_off[1], H, H, B));
    if (!h7) gemm_wide_add(gw, gemm_dw(w.a_dz22, H, w.h2[3], H, Ga + da.w_off[2], la[2], Ga + da.b_off[2], H, H, B));
    if (!h7) gemm_wide_add(gw, gemm_dw(w.a_dh2, H, w.h1[3], H, Ga + da.w_off[1], la[1], Ga + da.b_off[1], H, H, B));
    gemm_wide_add(gw, gemm_dw(w.dlogits_q, Np, w.h3[2], H, Gc + dc.w_off[3], lc[3], Gc + dc.b_off[3], N, H, B));
    gemm_wide_add(gw, gemm_dw(w.c_dz2, H, w.a, Ap, Gc + dc.w_off[1] + H, lc[1], nullptr, H, A, B));
    gemm_wide_add(gw, gemm_dw(w.c_dz1, H, w.s, Sp, Gc + dc.w_off[0], lc[0], Gc + dc.b_off[0], H, S, B));
    if (!h7) gemm_wide_add(gw, gemm_dw(w.a_dz3, Ap, w.h3[3], H, Ga + da.w_off[3], la[3], Ga + da.b_off[3], A, H, B));
    if (!h7) gemm_wide_add(gw, gemm_dw(w.a_dz1, H, w.s, Sp, Ga + da.w_off[0], la[0], Ga + da.b_off[0], H, S, B));
    RUN(gemm_wide_launch(gw, st));
  } else {
  // 5. backward.  "c_" = critic-loss pass, "p_" = policy pass through the critic, "a_" = actor.
  // level B1: through critic.fc3
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_dx(w.dlogits_q, Np, Wc + dc.w_off[3], lc[3], w.c_dz22, H, B, H, N, EPI_RELU_MASK, w.h3[2], H));
  gemm_batch_add(g, gemm_dx(w.dlogits_pi, Np, Wc + dc.w_off[3], lc[3], w.p_dz22, H, B, H, N, EPI_RELU_MASK, w.h3[4], H));
  gemm_batch_add(g, gemm_dw(w.dlogits_q, Np, w.h3[2], H, Gc + dc.w_off[3], lc[3], Gc + dc.b_off[3], N, H, B));
  LEVEL(g);
  // level B2: through critic.fc2_2
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_dx(w.c_dz22, H, Wc + dc.w_off[2], lc[2], w.c_dz2, H, B, H, H, EPI_RELU_MASK, w.h2[2], H));
  gemm_batch_add(g, gemm_dx(w.p_dz22, H, Wc + dc.w_off[2], lc[2], w.p_dz2, H, B, H, H, EPI_RELU_MASK, w.h2[4], H));
  gemm_batch_add(g, gemm_dw(w.c_dz22, H, w.h2[2], H, Gc + dc.w_off[2], lc[2], Gc + dc.b_off[2], H, H, B));
  LEVEL(g);
  // level B3: through critic.fc2: dh1 (critic loss), d action (policy, tanh' folded in), dW2 = [dz2^T h1 | dz2^T a]
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_dx(w.c_dz2, H, Wc + dc.w_off[1], lc[1], w.c_dz1, H, B, H, H, EPI_RELU_MASK, w.h1[2], H));
  gemm_batch_add(g, gemm_dx(w.p_dz2, H, Wc + dc.w_off[1] + H, lc[1], w.a_dz3, Ap, B, A, H, EPI_TANH_MASK, w.out[3], Ap));
  gemm_batch_add(g, gemm_dw(w.c_dz2, H, w.h1[2], H, Gc + dc.w_off[1], lc[1], Gc + dc.b_off[1], H, H, B));
  gemm_batch_add(g, gemm_dw(w.c_dz2, H, w.a, Ap, Gc + dc.w_off[1] + H, lc[1], nullptr, H, A, B));
  LEVEL(g);
  // level B4: critic.fc1 weights; actor.fc3
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_dw(w.c_dz1, H, w.s, Sp, Gc + dc.w_off[0], lc[0], Gc + dc.b_off[0], H, S, B));
  gemm_batch_add(g, gemm_dx(w.a_dz3, Ap, Wa + da.w_off[3], la[3], w.a_dz22, H, B, H, A, EPI_RELU_MASK, w.h3[3], H));
  gemm_batch_add(g, gemm_dw(w.a_dz3, Ap, w.h3[3], H, Ga + da.w_off[3], la[3], Ga + da.b_off[3], A, H, B));
  LEVEL(g);
  // level B5: actor.fc2_2 (its input h2 has no activation -> plain dX)
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_dx(w.a_dz22, H, Wa + da.w_off[2], la[2], w.a_dh2, H, B, H, H, EPI_NONE, nullptr, 0));
  gemm_batch_add(g, gemm_dw(w.a_dz22, H, w.h2[3], H, Ga + da.w_off[2], la[2], Ga + da.b_off[2], H, H, B));
  LEVEL(g);
  // level B6: actor.fc2
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_dx(w.a_dh2, H, Wa + da.w_off[1], la[1], w.a_dz1, H, B, H, H, EPI_RELU_MASK, w.h1[3], H));
  gemm_batch_add(g, gemm_dw(w.a_dh2, H, w.h1[3], H, Ga + da.w_off[1], la[1], Ga + da.b_off[1], H, H, B));
  LEVEL(g);
  // level B7: actor.fc1
  gemm_batch_begin(g);
  gemm_batch_add(g, gemm_dw(w.a_dz1, H, w.s, Sp, Ga + da.w_off[0], la[0], Ga + da.b_off[0], H, S, B));
  LEVEL(g);

  }

  // 6. data-parallel gradient exchange: ONE all-reduce over the flat [P_a + P_c] buffer
  // every rank's half of this step must be complete before Adam sums them: the chain plans signal from the dW
  // kernel and wait inside the Adam kernel; the level plan (several dW launches) uses a small barrier launch
  const bool inline_sync = peer_mode && (chain || tcc);
  if (peer_mode && !inline_sync) RUN(comm_peer_barrier(L->comm, st));
  // reduce-scatter + all-gather over peer memory: each rank reduces its 1/N slice and pushes it to everyone
  if (peer_mc2) RUN(comm_mc_reduce_bcast(L->comm, gpar, st));
  else if (peer_rs) RUN(comm_peer_reduce_scatter(L->comm, gpar, st));
  else if (!peer_mode && c.world_size > 1) RUN(comm_allreduce(L->comm, Ga, da.total + dc.total, st));

  // 7. Adam (actor + critic), sync (identity), Polyak -- one launch, two segments
  AdamArgs aa{};
  aa.seg[0] = AdamSeg{b.actor, Ga, b.adam_m_actor, b.adam_v_actor, b.actor_target, da.total, nullptr, 0, 0.f, 0};
  aa.seg[1] = AdamSeg{b.critic, Gc, b.adam_m_critic, b.adam_v_critic, b.critic_target, dc.total, nullptr, 0, 0.f, 1};
  if (peer_mode) {                                              // sum of the ranks' halves, also stored in the caller's buffer
    aa.npeers = peers.world;
    for (int r = 0; r < peers.world; ++r) aa.peer_g[r] = peers.x[r] + int64_t(gpar) * peers.n;
    aa.seg[0].g_out = b.grad_actor; aa.seg[0].g_off = 0;
    aa.seg[1].g_out = b.grad_critic; aa.seg[1].g_off = da.total;
    aa.my_flags = inline_sync ? peers.flag[peers.rank] : nullptr; aa.rank = peers.rank;
    if (peer_mc) aa.mc_g = peers.mc + int64_t(gpar) * peers.n;    // NVSwitch reduces; signal 0 (every rank's dW done) is awaited in-kernel
    if (peer_mc2) {                                             // the reduced gradient was broadcast into the local multicast-bound buffer
      aa.peer_reduced = 1;
      aa.seg[0].g = peers.mc_uc + 2 * peers.n; aa.seg[1].g = peers.mc_uc + 2 * peers.n + da.total;
      aa.my_flags = peers.flag2[peers.rank];
    }
    if (peer_rs) {                                              // the reduced gradient is local: wait for every rank's "slice pushed", then stream it
      aa.peer_reduced = 1;
      aa.seg[0].g = peers.red[peers.rank]; aa.seg[1].g = peers.red[peers.rank] + da.total;
      aa.my_flags = peers.flag2[peers.rank];
    }
  }
  aa.nseg = 2;
  if (tcc) {                                                    // keep the forward weight images of the tcgen05 chains current
    const TccImage* U = L->tcc_img;
    const NetDims* nd[2] = {&da, &dc};
    const int base[2] = {U_A_F1, U_C_F1}, tbase[2] = {U_AT_F1, U_CT_F1};
    for (int sg = 0; sg < 2; ++sg) {
      aa.seg[sg].nimg = 4;
      for (int ly = 0; ly < 4; ++ly) {
        AdamImgLayer& I = aa.seg[sg].imgl[ly];
        I.w_off = nd[sg]->w_off[ly]; I.w_end = I.w_off + int64_t(nd[sg]->out[ly]) * nd[sg]->ld[ly];
        I.ld = nd[sg]->ld[ly]; I.nchunks = U[base[sg] + ly].kchunks;
        I.img = const_cast<uint8_t*>(U[base[sg] + ly].ptr); I.img_t = const_cast<uint8_t*>(U[tbase[sg] + ly].ptr);
      }
    }
  }
  aa.w1 = float(1.0 - c.beta1); aa.w2 = float(1.0 - c.beta2); aa.beta2 = float(c.beta2); aa.eps = float(c.adam_eps);
  aa.tau = float(c.tau); aa.one_minus_tau = float(1.0 - c.tau); aa.grad_scale = 1.0f; aa.clock = w.clock;
  aa.pipe_slot = pf ? par : -1;
  // tail slice of the same launch: reported batch-mean losses + advance the device clock
  aa.loss_rows = w.loss_rows; aa.pi_rows = w.pi_rows; aa.B = B; aa.inv_count = 1.0f / float(B); aa.loss_out = b.losses;
  if (h7) {
    // ---- post-update-critic plan, second half ---------------------------------------------------------------------
    AdamArgs ac = aa;                                            // critic update alone (writes the critic's forward images too)
    ac.seg[0] = aa.seg[1]; ac.nseg = 1; ac.skip_tail = 1;
    RUN(launch_adam(ac, st));
    RUN(launch_tcc_pack(L->tcc_pack_dx, st));                    // transposed images of the UPDATED critic for the policy backward
    TccCtx cx{L, &w, &da, &dc, Wa, Wat, Wc, Wct, B, S, A, N, Sp, Ap, Np};
    TccArgs& fb = L->tcc_fwd_args;
    tcc_args_begin(fb, B, reinterpret_cast<uint8_t*>(w.xchg), c.precision == 1 ? 3 : 1); fb.step_slot = 1;
    tcc_build_Q(fb, 0, cx, w.out[3], nullptr, w.h2[4], w.h3[4], w.out[4]);      // critic(s, actor(s)) with the new critic weights
    RUN(launch_mlp_tc_chain(fb, st));
    HeadsArgs hp = ha;
    hp.pi_logits = w.out[4]; hp.only_policy = 1; hp.sampler_clock = nullptr;
    RUN(launch_heads(hp, c.proj_mode, st));
    TccArgs& bb = L->tcc_bwd_args;
    tcc_args_begin(bb, B, reinterpret_cast<uint8_t*>(w.xchg), c.precision == 1 ? 3 : 1); bb.step_slot = 5;
    tcc_build_bwd_P(bb, 0, cx);
    RUN(launch_mlp_tc_chain(bb, st));
    GemmWideBatch& gw = L->dw_batch;
    gemm_wide_begin(gw, nullptr);
    gemm_wide_add(gw, gemm_dw(w.a_dz22, H, w.h2[3], H, Ga + da.w_off[2], la[2], Ga + da.b_off[2], H, H, B));
    gemm_wide_add(gw, gemm_dw(w.a_dh2, H, w.h1[3], H, Ga + da.w_off[1], la[1], Ga + da.b_off[1], H, H, B));
    gemm_wide_add(gw, gemm_dw(w.a_dz3, Ap, w.h3[3], H, Ga + da.w_off[3], la[3], Ga + da.b_off[3], A, H, B));
    gemm_wide_add(gw, gemm_dw(w.a_dz1, H, w.s, Sp, Ga + da.w_off[0], la[0], Ga + da.b_off[0], H, S, B));
    RUN(gemm_wide_launch(gw, st));
    AdamArgs ab = aa;                                            // actor update + the step's tail (loss means, clock)
    ab.nseg = 1;
    RUN(launch_adam(ab, st));
  } else RUN(launch_adam(aa, st));
  if (c.prioritized || pf) D4PG_CUDA_OK(cudaStreamWaitEvent(st, L->ev_join, 0));
#undef LEVEL
#undef RUN
  L->kernels_per_step = nk;
  return D4PG_OK;
}

extern "C" int64_t d4pg_learner_workspace_floats(const d4pg_learner_config_t* cfg) {
  if (!cfg) return -1;
  return carve(nullptr, cfg->batch, cfg->obs_dim, cfg->act_dim, cfg->n_atoms, step_plan(*cfg) == 1, piped(*cfg)).total;
}

extern "C" int32_t d4pg_learner_create(const d4pg_learner_config_t* cfg, const d4pg_learner_buffers_t* buf,
                                       d4pg_replay_t* replay, d4pg_comm_t* comm, d4pg_learner_t** out) {
  D4PG_REQUIRE(cfg && buf && replay && out, D4PG_EINVAL, "d4pg_learner_create: null argument");
  D4PG_REQUIRE(cfg->batch > 0 && cfg->obs_dim > 0 && cfg->act_dim > 0, D4PG_EINVAL, "d4pg_learner_create: bad dims");
  D4PG_REQUIRE(cfg->n_atoms >= 2 && cfg->n_atoms <= D4PG_MAX_ATOMS, D4PG_EINVAL, "d4pg_learner_create: n_atoms must be in [2,%d]", D4PG_MAX_ATOMS);
  D4PG_REQUIRE(cfg->v_max > cfg->v_min, D4PG_EINVAL, "d4pg_learner_create: v_max <= v_min");
  D4PG_REQUIRE(cfg->proj_mode == 0 || cfg->proj_mode == 1, D4PG_EINVAL, "d4pg_learner_create: proj_mode must be 0/1");
  D4PG_REQUIRE(cfg->precision >= 0 && cfg->precision <= 2, D4PG_ENOTSUP,
               "d4pg_learner_create: precision %d unknown (0 fp32 FFMA, 1 3xTF32 tcgen05, 2 TF32 tcgen05)", cfg->precision);
  D4PG_REQUIRE(cfg->world_size <= 1 || comm, D4PG_EINVAL, "d4pg_learner_create: world_size>1 needs a communicator");
  D4PG_REQUIRE(cfg->chain == 0 || cfg->chain == 1, D4PG_EINVAL, "d4pg_learner_create: chain must be 0 or 1");
  D4PG_REQUIRE(!(cfg->loss_flags & 4) || (tcc_shapes_ok(*cfg) && cfg->world_size <= 1), D4PG_ENOTSUP,
               "d4pg_learner_create: loss_flags & 4 (post-update-critic actor gradient) needs the tcgen05 chain plan: precision 1/2, chain 1, "
               "batch <= 512, obs_dim <= 32, act_dim <= 32, on one GPU");
  D4PG_REQUIRE(buf->actor && buf->actor_target && buf->critic && buf->critic_target && buf->grad_actor && buf->grad_critic &&
               buf->adam_m_actor && buf->adam_v_actor && buf->adam_m_critic && buf->adam_v_critic &&
               buf->idx && buf->prio && buf->td && buf->losses && buf->workspace, D4PG_EINVAL,
               "d4pg_learner_create: null device buffer");
  d4pg_learner* L = new (std::nothrow) d4pg_learner();
  D4PG_REQUIRE(L, D4PG_EINVAL, "d4pg_learner_create: out of host memory");
  L->cfg = *cfg; L->buf = *buf; L->replay = replay; L->comm = comm;
  L->da = actor_dims(cfg->obs_dim, cfg->act_dim);
  L->dc = critic_dims(cfg->obs_dim, cfg->act_dim, cfg->n_atoms);
  if (buf->grad_critic != buf->grad_actor + L->da.total) {
    set_error("d4pg_learner_create: grad_critic must equal grad_actor + P_a (one flat gradient buffer)");
    delete L; return D4PG_EINVAL;
  }
  L->ws = carve(buf->workspace, cfg->batch, cfg->obs_dim, cfg->act_dim, cfg->n_atoms, step_plan(*cfg) == 1, piped(*cfg));
  for (int i = 0; i < 4; ++i) { L->graph_exec[i] = nullptr; L->graph_ready[i] = false; }
  for (int i = 0; i < 2; ++i) { L->multi_exec[i] = nullptr; L->multi_ready[i] = false; }
  L->pipe_par = 0; L->last_par = 0; L->prefetch_valid = false; L->seen_gen = -1;
  L->steps_done = 0; L->kernels_per_step = 0;
  L->profiling = false;
  (void)debug_trace_buffer();          // allocate outside of any stream capture
  if (int rc = tcc_setup(L)) { delete L; return rc; }
  L->host_steps = 0; L->host_losses = nullptr; L->ev_in = nullptr; L->ev_out = nullptr;
  for (int i = 0; i < 4; ++i) { L->host_u[i] = nullptr; L->host_pos[i] = nullptr; L->ev_h2d[i] = nullptr; }
  for (int i = 0; i < 2; ++i) { L->loss_ring[i] = nullptr; L->ev_loss[i] = nullptr; }
  L->loss_steps = 0;
  L->ing = nullptr; L->ev_ing = nullptr; L->gate_flag = nullptr; L->images_dirty = true;
  if (host_pipe(*cfg)) {
    L->gate_flag = replay_gate_flag(replay);
    const bool ok = L->gate_flag && cudaStreamCreateWithFlags(&L->ing, cudaStreamNonBlocking) == cudaSuccess &&
                    cudaEventCreateWithFlags(&L->ev_ing, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
      set_error("d4pg_learner_create: ingest stream setup failed"); delete L; return D4PG_ECUDA;
    }
  }
  {
    const size_t nb = size_t(cfg->batch);
    bool ok = cudaEventCreateWithFlags(&L->ev_in, cudaEventDisableTiming) == cudaSuccess &&
              cudaEventCreateWithFlags(&L->ev_out, cudaEventDisableTiming) == cudaSuccess &&
              cudaHostAlloc(reinterpret_cast<void**>(&L->host_losses), 4 * sizeof(float), cudaHostAllocDefault) == cudaSuccess;
    for (int i = 0; i < 2 && ok; ++i)
      ok = cudaEventCreateWithFlags(&L->ev_loss[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaHostAlloc(reinterpret_cast<void**>(&L->loss_ring[i]), 4 * sizeof(float), cudaHostAllocDefault) == cudaSuccess;
    for (int i = 0; i < 4 && ok; ++i)
      ok = cudaEventCreateWithFlags(&L->ev_h2d[i], cudaEventDisableTiming) == cudaSuccess &&
           cudaHostAlloc(reinterpret_cast<void**>(&L->host_u[i]), nb * sizeof(double), cudaHostAllocMapped) == cudaSuccess &&
           cudaHostAlloc(reinterpret_cast<void**>(&L->host_pos[i]), nb * sizeof(int32_t), cudaHostAllocMapped) == cudaSuccess;
    if (!ok) { set_error("d4pg_learner_create: pinned staging allocation failed"); delete L; return D4PG_ECUDA; }
  }
  if (cudaStreamCreateWithFlags(&L->side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&L->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&L->ev_join, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&L->ev_fork2, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&L->ev_join2, cudaEventDisableTiming) != cudaSuccess) {
    set_error("d4pg_learner_create: stream/event creation failed"); delete L; return D4PG_ECUDA;
  }
  trace_set_side_stream(L->side);
  cudaError_t e = cudaMemset(L->ws.clock, 0, sizeof(LearnerClock));
  if (e == cudaSuccess) e = cudaMemset(L->ws.pipe_epoch, 0, sizeof(unsigned long long) * size_t(cdiv(cfg->batch, SAMPLE_ROWS)));
  if (e != cudaSuccess) { set_error("d4pg_learner_create: %s", cudaGetErrorString(e)); delete L; return D4PG_ECUDA; }
  *out = L;
  return D4PG_OK;
}

extern "C" int32_t d4pg_learner_destroy(d4pg_learner_t* L) {
  if (!L) return D4PG_OK;
  for (int i = 0; i < 4; ++i) if (L->graph_exec[i]) cudaGraphExecDestroy(L->graph_exec[i]);
  for (int i = 0; i < 2; ++i) if (L->multi_exec[i]) cudaGraphExecDestroy(L->multi_exec[i]);
  cudaEventDestroy(L->ev_fork); cudaEventDestroy(L->ev_join); cudaEventDestroy(L->ev_fork2); cudaEventDestroy(L->ev_join2);
  cudaStreamDestroy(L->side);
  if (L->tcc_images) cudaFree(L->tcc_images);
  if (L->ing) { cudaStreamSynchronize(L->ing); cudaStreamDestroy(L->ing); }
  if (L->ev_ing) cudaEventDestroy(L->ev_ing);
  if (L->ev_in) cudaEventDestroy(L->ev_in);
  if (L->ev_out) cudaEventDestroy(L->ev_out);
  if (L->host_losses) cudaFreeHost(L->host_losses);
  for (int i = 0; i < 2; ++i) {
    if (L->ev_loss[i]) cudaEventDestroy(L->ev_loss[i]);
    if (L->loss_ring[i]) cudaFreeHost(L->loss_ring[i]);
  }
  for (int i = 0; i < 4; ++i) {
    if (L->ev_h2d[i]) cudaEventDestroy(L->ev_h2d[i]);
    if (L->host_u[i]) cudaFreeHost(L->host_u[i]);
    if (L->host_pos[i]) cudaFreeHost(L->host_pos[i]);
  }
  delete L;
  return D4PG_OK;
}

// which half of the batch buffers the next step uses, and whether it has to sample it first
static void next_variant(d4pg_learner* L, int* par, bool* cold) {
  if (!piped(L->cfg)) { *par = 0; *cold = true; return; }
  *par = L->pipe_par;
  // host pipeline: a direct d4pg_learner_step samples in the graph; d4pg_learner_step_host presamples on the ingest stream
  *cold = host_pipe(L->cfg) || !L->prefetch_valid || replay_generation(L->replay) != L->seen_gen;
}
static void commit_variant(d4pg_learner* L, int par) {
  ++L->steps_done;
  if (!piped(L->cfg)) return;
  L->last_par = par; L->pipe_par = par ^ 1; L->prefetch_valid = true; L->seen_gen = replay_generation(L->replay);
}

static int launch_variant(d4pg_learner* L, cudaStream_t st, int par, bool cold);

extern "C" int32_t d4pg_learner_step(d4pg_learner_t* L, d4pg_stream_t stream) {
  D4PG_REQUIRE(L, D4PG_EINVAL, "d4pg_learner_step: null handle");
  cudaStream_t st = as_stream(stream);
  int par; bool cold;
  next_variant(L, &par, &cold);
  if (L->ing) {                                      // adds issued on the ingest stream come first
    D4PG_CUDA_OK(cudaEventRecord(L->ev_ing, L->ing));
    D4PG_CUDA_OK(cudaStreamWaitEvent(st, L->ev_ing, 0));
  }
  return launch_variant(L, st, par, cold);
}

// the step graph of variant (par, cold) on `st` (captured on first use); arms the ingest gate of the next step
static int launch_variant(d4pg_learner* L, cudaStream_t st, int par, bool cold) {
  auto arm_gate = [&] { if (L->ing) replay_arm_gate(L->replay); };
  if (!L->cfg.use_graph) {
    int rc = enqueue_step(L, st, par, cold, !(host_pipe(L->cfg) && !cold));
    if (rc == D4PG_OK) { commit_variant(L, par); arm_gate(); }
    return rc;
  }
  // without the prefetch pipeline the only per-step variation is the gradient half of the peer exchange
  const int v = piped(L->cfg) ? par * 2 + (cold ? 1 : 0) : int(L->steps_done & 1);
  if (!L->graph_ready[v]) {
    D4PG_REQUIRE(st != nullptr, D4PG_EINVAL, "d4pg_learner_step: graph capture needs a non-default stream");
    cudaGraph_t graph = nullptr;
    D4PG_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
    // warm host-pipeline variants start from a sampled batch AND packed forward images (d4pg_learner_step_host packs
    // eagerly on the learner stream while the ingest stream still samples)
    int rc = enqueue_step(L, st, par, cold, !(host_pipe(L->cfg) && !cold));
    cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (rc != D4PG_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
    if (e != cudaSuccess) { set_error("d4pg_learner_step: end capture: %s", cudaGetErrorString(e)); return D4PG_ECUDA; }
    e = cudaGraphInstantiate(&L->graph_exec[v], graph, 0);
    cudaGraphDestroy(graph);
    if (e != cudaSuccess) { set_error("d4pg_learner_step: instantiate: %s", cudaGetErrorString(e)); return D4PG_ECUDA; }
    L->graph_ready[v] = true;
  }
  D4PG_CUDA_OK(cudaGraphLaunch(L->graph_exec[v], st));
  commit_variant(L, par);
  arm_gate();
  return D4PG_OK;
}

static bool inline_wait(const d4pg_learner* L) {
  return step_plan(L->cfg) == 1 && L->cfg.precision >= 1 && L->tcc_ok && cdiv(L->cfg.batch, SAMPLE_ROWS) <= TCC_THREADS;
}

// host pipeline: sample + gather batch `par` from the device copy of this step's uniforms / positions (the launch the
// cold graph variant starts with, issued on the ingest stream instead)
static int presample(d4pg_learner* L, int par, const double* uniforms, const int32_t* positions, cudaStream_t st) {
  const d4pg_learner_config_t& c = L->cfg; const d4pg_learner_buffers_t& b = L->buf; const Workspace& o = L->ws;
  const ClockParams cp{c.lr_actor, c.lr_critic, c.beta1, c.beta2, c.per_beta0, c.per_beta_final,
                       c.per_beta_iters > 0 ? c.per_beta_iters : 1};
  (void)b;
  return learner_sample(L->replay, c.batch, c.prioritized, uniforms, !c.prioritized ? positions : nullptr, c.philox_seed,
                        o.clock, cp, o.idx2[par], o.wts2[par], par ? o.s_b : o.s, par ? o.a_b : o.a, par ? o.r_b : o.r,
                        par ? o.s2_b : o.s2, par ? o.done_b : o.done, pitch4(c.obs_dim), pitch4(c.act_dim), par, st,
                        true, o.pipe_epoch);
}

// The host-facing step: stage this step's host inputs in pinned memory, H2D, the step, order the caller after it.
static int step_host_common(d4pg_learner_t* L, const double* uniforms, const uint32_t* mt_words, const int32_t* positions,
                            d4pg_stream_t caller_stream, d4pg_stream_t learner_stream) {
  cudaStream_t cs = as_stream(caller_stream), ls = as_stream(learner_stream);
  const int B = L->cfg.batch;
  D4PG_CUDA_OK(cudaEventRecord(L->ev_in, cs));                 // adds / weight loads issued by the caller
  D4PG_CUDA_OK(cudaStreamWaitEvent(ls, L->ev_in, 0));
  const bool pipe = L->ing != nullptr && (uniforms || mt_words || positions);
  // piped: the sample kernel reads this step's uniforms / positions (2 KB) straight out of the pinned staging slot over
  // PCIe -- no copy node between the caller's add and the sample on the ingest stream -- so the slots form a ring of 4.
  // (The caller's replay operations on caller_stream are NOT waited for before sampling: the host mirror orders them
  // explicitly with d4pg_replay_order_after, see d4pg_learner_ingest_stream in the header.)
  const int par = int(L->host_steps & (pipe ? 3 : 1));
  double* du = L->buf.uniforms;
  int32_t* dpos = L->buf.positions;
  if (uniforms || mt_words || positions) {
    if (L->host_steps >= (pipe ? 4 : 2)) D4PG_CUDA_OK(cudaEventSynchronize(L->ev_h2d[par]));   // the last reader of this slot
    if (uniforms || mt_words) {
      D4PG_REQUIRE(du, D4PG_ESTATE, "d4pg_learner_step_host: no device uniforms buffer");
      double* u = L->host_u[par];
      if (uniforms) memcpy(u, uniforms, size_t(B) * sizeof(double));
      else                                                     // CPython random.random(): (a >> 5, b >> 6) -> (a * 2^26 + b) / 2^53
        for (int i = 0; i < B; ++i)
          u[i] = (double(mt_words[2 * i] >> 5) * 67108864.0 + double(mt_words[2 * i + 1] >> 6)) * (1.0 / 9007199254740992.0);
      if (pipe) D4PG_CUDA_OK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&du), u, 0));
      else D4PG_CUDA_OK(cudaMemcpyAsync(du, u, size_t(B) * sizeof(double), cudaMemcpyHostToDevice, ls));
    }
    if (positions) {
      D4PG_REQUIRE(dpos, D4PG_ESTATE, "d4pg_learner_step_host: no device positions buffer");
      memcpy(L->host_pos[par], positions, size_t(B) * sizeof(int32_t));
      if (pipe) D4PG_CUDA_OK(cudaHostGetDevicePointer(reinterpret_cast<void**>(&dpos), L->host_pos[par], 0));
      else D4PG_CUDA_OK(cudaMemcpyAsync(dpos, L->host_pos[par], size_t(B) * sizeof(int32_t), cudaMemcpyHostToDevice, ls));
    }
    if (!pipe) D4PG_CUDA_OK(cudaEventRecord(L->ev_h2d[par], ls));
    ++L->host_steps;
  }
  int rc;
  if (pipe) {
    // batch k on the ingest stream: behind the caller's add(k) (same stream) and the gate of step k-1, while step k-1's
    // backward pass / dW / Adam still run on the learner stream; the step graph starts from the sampled batch
    int bpar; bool cold_unused;
    next_variant(L, &bpar, &cold_unused);
    rc = replay_gate_consume(L->replay, L->ing);
    if (rc) return rc;
    rc = presample(L, bpar, du, dpos, L->ing);
    if (rc) return rc;
    D4PG_CUDA_OK(cudaEventRecord(L->ev_h2d[par], L->ing));      // the staging slot has been read
    D4PG_CUDA_OK(cudaEventRecord(L->ev_ing, L->ing));
    // forward weight images: the Adam kernel keeps them current, so they are re-packed only after the caller reported a
    // parameter write of its own (d4pg_learner_weights_changed) -- behind Adam(k-1), beside the ingest stream's tail
    if (L->images_dirty && step_plan(L->cfg) == 1 && L->cfg.precision >= 1 && L->tcc_ok) {
      rc = launch_tcc_pack(L->tcc_pack_fwd, ls);
      if (rc) return rc;
    }
    L->images_dirty = false;
    if (!inline_wait(L)) D4PG_CUDA_OK(cudaStreamWaitEvent(ls, L->ev_ing, 0));
    rc = launch_variant(L, ls, bpar, false);
  } else {
    rc = d4pg_learner_step(L, learner_stream);
  }
  if (rc) return rc;
  {                                                            // this step's result, queued for d4pg_learner_fetch_losses
    const int slot = int(L->loss_steps & 1);
    D4PG_CUDA_OK(cudaMemcpyAsync(L->loss_ring[slot], L->buf.losses, 4 * sizeof(float), cudaMemcpyDeviceToHost, ls));
    D4PG_CUDA_OK(cudaEventRecord(L->ev_loss[slot], ls));
    ++L->loss_steps;
  }
  D4PG_CUDA_OK(cudaEventRecord(L->ev_out, ls));
  D4PG_CUDA_OK(cudaStreamWaitEvent(cs, L->ev_out, 0));
  return D4PG_OK;
}

extern "C" int32_t d4pg_learner_fetch_losses(d4pg_learner_t* L, int32_t lag, float* out4) {
  D4PG_REQUIRE(L && out4 && (lag == 0 || lag == 1), D4PG_EINVAL, "d4pg_learner_fetch_losses: lag must be 0 or 1");
  D4PG_REQUIRE(L->loss_steps > lag, D4PG_ESTATE, "d4pg_learner_fetch_losses: no such step yet");
  const int slot = int((L->loss_steps - 1 - lag) & 1);
  D4PG_CUDA_OK(cudaEventSynchronize(L->ev_loss[slot]));
  for (int i = 0; i < 4; ++i) out4[i] = L->loss_ring[slot][i];
  return D4PG_OK;
}

extern "C" int32_t d4pg_learner_step_host(d4pg_learner_t* L, const double* uniforms, const int32_t* positions,
                                          d4pg_stream_t caller_stream, d4pg_stream_t learner_stream) {
  D4PG_REQUIRE(L, D4PG_EINVAL, "d4pg_learner_step_host: null handle");
  return step_host_common(L, uniforms, nullptr, positions, caller_stream, learner_stream);
}

extern "C" int32_t d4pg_learner_step_host_mt(d4pg_learner_t* L, const uint32_t* mt_words,
                                             d4pg_stream_t caller_stream, d4pg_stream_t learner_stream) {
  D4PG_REQUIRE(L && mt_words, D4PG_EINVAL, "d4pg_learner_step_host_mt: null argument");
  return step_host_common(L, nullptr, mt_words, nullptr, caller_stream, learner_stream);
}

extern "C" int32_t d4pg_learner_read_losses(d4pg_learner_t* L, float* out4, d4pg_stream_t learner_stream) {
  D4PG_REQUIRE(L && out4, D4PG_EINVAL, "d4pg_learner_read_losses: null argument");
  cudaStream_t ls = as_stream(learner_stream);
  D4PG_CUDA_OK(cudaMemcpyAsync(L->host_losses, L->buf.losses, 4 * sizeof(float), cudaMemcpyDeviceToHost, ls));
  D4PG_CUDA_OK(cudaStreamSynchronize(ls));
  for (int i = 0; i < 4; ++i) out4[i] = L->host_losses[i];
  return D4PG_OK;
}

// Back-to-back steps with nothing in between: warm prefetch steps are replayed RUN_UNROLL at a time from one graph
// (a graph launch boundary costs ~5 us of idle GPU; inside a graph consecutive steps are ordinary dependent nodes).
constexpr int RUN_UNROLL = 8;
extern "C" int32_t d4pg_learner_run(d4pg_learner_t* L, int32_t n_steps, d4pg_stream_t stream) {
  D4PG_REQUIRE(L && n_steps > 0, D4PG_EINVAL, "d4pg_learner_run: bad arguments");
  cudaStream_t st = as_stream(stream);
  int n = n_steps;
  while (n > 0) {
    int par; bool cold;
    next_variant(L, &par, &cold);
    if (L->cfg.use_graph && prefetching(L->cfg) && !cold && n >= RUN_UNROLL && st != nullptr) {
      if (!L->multi_ready[par]) {
        cudaGraph_t graph = nullptr;
        D4PG_CUDA_OK(cudaStreamBeginCapture(st, cudaStreamCaptureModeThreadLocal));
        int rc = D4PG_OK;
        for (int i = 0; i < RUN_UNROLL && rc == D4PG_OK; ++i) rc = enqueue_step(L, st, par ^ (i & 1), false, i == 0);
        cudaError_t e = cudaStreamEndCapture(st, &graph);
        if (rc != D4PG_OK) { if (graph) cudaGraphDestroy(graph); return rc; }
        if (e != cudaSuccess) { set_error("d4pg_learner_run: end capture: %s", cudaGetErrorString(e)); return D4PG_ECUDA; }
        e = cudaGraphInstantiate(&L->multi_exec[par], graph, 0);
        cudaGraphDestroy(graph);
        if (e != cudaSuccess) { set_error("d4pg_learner_run: instantiate: %s", cudaGetErrorString(e)); return D4PG_ECUDA; }
        L->multi_ready[par] = true;
      }
      D4PG_CUDA_OK(cudaGraphLaunch(L->multi_exec[par], st));
      for (int i = 0; i < RUN_UNROLL; ++i) commit_variant(L, par ^ (i & 1));
      n -= RUN_UNROLL;
      continue;
    }
    int rc = d4pg_learner_step(L, stream);
    if (rc) return rc;
    --n;
  }
  return D4PG_OK;
}

extern "C" int32_t d4pg_learner_profile_step(d4pg_learner_t* L, d4pg_stream_t stream, int32_t max_launches,
                                             float* ms_out, char* names_out, int32_t name_stride, int32_t* n_out) {
  D4PG_REQUIRE(L && ms_out && n_out && max_launches > 0, D4PG_EINVAL, "d4pg_learner_profile_step: bad arguments");
  cudaStream_t st = as_stream(stream);
  L->profiling = true; L->ev.clear(); L->ev_name.clear(); L->ev_reps.clear();
  int par; bool cold;
  next_variant(L, &par, &cold);
  if (L->ing) { D4PG_CUDA_OK(cudaEventRecord(L->ev_ing, L->ing)); D4PG_CUDA_OK(cudaStreamWaitEvent(st, L->ev_ing, 0)); }
  int rc = enqueue_step(L, st, par, cold);
  L->profiling = false;
  if (rc == D4PG_OK) { commit_variant(L, par); if (L->ing) replay_arm_gate(L->replay); }
  cudaError_t e = cudaStreamSynchronize(st);
  const int n = int(L->ev_name.size());
  *n_out = n < max_launches ? n : max_launches;
  for (int i = 0; i < n; ++i) {
    float ms = 0.f;
    if (e == cudaSuccess) cudaEventElapsedTime(&ms, L->ev[2 * i], L->ev[2 * i + 1]);
    ms /= float(L->ev_reps[i]);
    if (i < max_launches) {
      ms_out[i] = ms;
      if (names_out && name_stride > 1) {
        strncpy(names_out + size_t(i) * name_stride, L->ev_name[i].c_str(), name_stride - 1);
        names_out[size_t(i) * name_stride + name_stride - 1] = 0;
      }
    }
    cudaEventDestroy(L->ev[2 * i]); cudaEventDestroy(L->ev[2 * i + 1]);
  }
  L->ev.clear(); L->ev_name.clear(); L->ev_reps.clear();
  if (e != cudaSuccess) { set_error("d4pg_learner_profile_step: %s", cudaGetErrorString(e)); return D4PG_ECUDA; }
  return rc;
}

extern "C" int32_t d4pg_learner_weights_changed(d4pg_learner_t* L) {
  D4PG_REQUIRE(L, D4PG_EINVAL, "d4pg_learner_weights_changed: null handle");
  L->images_dirty = true;
  return D4PG_OK;
}
extern "C" void* d4pg_learner_ingest_stream(const d4pg_learner_t* L) { return L ? static_cast<void*>(L->ing) : nullptr; }
extern "C" int64_t d4pg_learner_steps_done(const d4pg_learner_t* L) { return L ? L->steps_done : -1; }
extern "C" int32_t d4pg_learner_kernels_per_step(const d4pg_learner_t* L) { return L ? L->kernels_per_step : -1; }

extern "C" int32_t d4pg_learner_set_counters(d4pg_learner_t* L, int64_t adam_step, int64_t beta_t, d4pg_stream_t stream) {
  D4PG_REQUIRE(L && adam_step >= 0 && beta_t >= 0, D4PG_EINVAL, "d4pg_learner_set_counters: bad arguments");
  LearnerClock c{};
  c.adam_step = adam_step; c.beta_t = beta_t; c.steps_done = adam_step;
  c.s_adam_step = adam_step; c.s_beta_t = beta_t; c.s_steps_done = adam_step;
  L->prefetch_valid = false;                          // a prefetched batch was drawn with the old counters
  D4PG_CUDA_OK(cudaMemsetAsync(L->ws.pipe_epoch, 0, sizeof(unsigned long long) * size_t(cdiv(L->cfg.batch, SAMPLE_ROWS)), as_stream(stream)));
  D4PG_CUDA_OK(cudaMemcpyAsync(L->ws.clock, &c, sizeof(c), cudaMemcpyHostToDevice, as_stream(stream)));
  D4PG_CUDA_OK(cudaStreamSynchronize(as_stream(stream)));
  return D4PG_OK;
}

extern "C" int32_t d4pg_learner_tensor(d4pg_learner_t* L, const char* name, void** ptr, int64_t* count, int32_t* ld) {
  D4PG_REQUIRE(L && name && ptr && count && ld, D4PG_EINVAL, "d4pg_learner_tensor: null argument");
  Workspace w = L->ws;
  if (piped(L->cfg) && L->last_par) { w.s = w.s_b; w.a = w.a_b; w.s2 = w.s2_b; w.r = w.r_b; w.done = w.done_b; }
  const int64_t B = L->cfg.batch;
  const int Sp = pitch4(L->cfg.obs_dim), Ap = pitch4(L->cfg.act_dim), Np = pitch4(L->cfg.n_atoms);
  struct E { const char* n; void* p; int64_t c; int ld; };
  const E table[] = {
      {"s", w.s, B * Sp, Sp}, {"a", w.a, B * Ap, Ap}, {"r", w.r, B, 1}, {"s2", w.s2, B * Sp, Sp}, {"done", w.done, B, 1},
      {"target_logits", w.out[1], B * Np, Np}, {"q_logits", w.out[2], B * Np, Np}, {"pi_logits", w.out[4], B * Np, Np},
      {"m", w.m, B * Np, Np}, {"q_probs", w.q_probs, B * Np, Np}, {"target_probs", w.target_probs, B * Np, Np},
      {"dlogits_q", w.dlogits_q, B * Np, Np}, {"dlogits_pi", w.dlogits_pi, B * Np, Np},
      {"actor_out", w.out[3], B * Ap, Ap}, {"actor_target_out", w.out[0], B * Ap, Ap},
      {"loss_rows", w.loss_rows, B, 1}, {"pi_rows", w.pi_rows, B, 1},
      {"h1_c", w.h1[2], B * 256, 256}, {"h2_c", w.h2[2], B * 256, 256}, {"h3_c", w.h3[2], B * 256, 256},
      {"h1_a", w.h1[3], B * 256, 256}, {"h2_a", w.h2[3], B * 256, 256}, {"h3_a", w.h3[3], B * 256, 256},
      {"h2_p", w.h2[4], B * 256, 256}, {"h3_p", w.h3[4], B * 256, 256},
      {"c_dz22", w.c_dz22, B * 256, 256}, {"c_dz2", w.c_dz2, B * 256, 256}, {"c_dz1", w.c_dz1, B * 256, 256},
      {"a_dz3", w.a_dz3, B * Ap, Ap}, {"a_dz22", w.a_dz22, B * 256, 256}, {"a_dh2", w.a_dh2, B * 256, 256},
      {"a_dz1", w.a_dz1, B * 256, 256}};
  for (const E& e : table)
    if (strcmp(e.n, name) == 0) { *ptr = e.p; *count = e.c; *ld = e.ld; return D4PG_OK; }
  set_error("d4pg_learner_tensor: unknown tensor '%s'", name);
  return D4PG_EINVAL;
}
