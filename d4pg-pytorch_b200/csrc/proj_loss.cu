// Fused categorical projection + critic CE loss + TD proxy / priority + logit gradients
// (+ the policy-loss head).  One warp per batch row; the atom support is staged in shared
// memory and every row reduction is a warp shuffle.
//
// Replaces (reference, relative to /root/reference):
//   ddpg.py:142-185  DDPG.reproject2              (proj_mode 0, the live projection)
//   ddpg.py:122-140  DDPG.reproj_categorical_dist (proj_mode 1, gamma**n, config 5)
//   ddpg.py:217      qdist_loss = -(m*log(q+1e-10)).sum(1).mean()
//   ddpg.py:220-222  td_errors  = -(m*q).sum(1);  ddpg.py:253 priorities = |td| + eps
//   ddpg.py:236-238  policy_loss = -critic(s,actor(s)).matmul(bin_centers).mean()
//   models.py:83     F.softmax(fc3(out), dim=1) for the three critic heads
//
// Bit-exactness plan (SURVEY.md section 7 "hard parts"): the bin index path is fp64 with explicit
// round-to-nearest intrinsics (no FMA contraction of r + c_j); the projected mass of mode 0 is
// accumulated per bin in atom order j=0..N-1, each add done in fp64 and rounded to fp32, which
// is exactly what NumPy does for `proj_distr[rows, l] += p * (u - b)` on an fp32 array.
#include "heads_dev.cuh"

namespace d4pg {

int launch_heads(const HeadsArgs& a_in, int mode, cudaStream_t st) {
  HeadsArgs a = a_in;
  a.trace = (a.sampler_clock && debug_trace_buffer()) ? debug_trace_buffer() + STEP_TRACE_BASE : nullptr;
  dim3 grid(cdiv(((a.pi_logits && !a.only_policy) ? 2 : 1) * a.B, HEAD_WARPS)), block(HEAD_WARPS * 32);   // policy heads on warps of their own
  D4PG_MAX_CARVEOUT((heads_kernel<0, 2>)); D4PG_MAX_CARVEOUT((heads_kernel<1, 2>));
  D4PG_MAX_CARVEOUT((heads_kernel<0, 4>)); D4PG_MAX_CARVEOUT((heads_kernel<1, 4>));
  // NT = atom slots per lane: 2 covers N<=64 (51 atoms), 4 covers N<=128 (101 atoms)
  if (a.N <= 64) {
    if (mode == 0) heads_kernel<0, 2><<<grid, block, 0, st>>>(a);
    else heads_kernel<1, 2><<<grid, block, 0, st>>>(a);
  } else {
    if (mode == 0) heads_kernel<0, 4><<<grid, block, 0, st>>>(a);
    else heads_kernel<1, 4><<<grid, block, 0, st>>>(a);
  }
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

}  // namespace d4pg

extern "C" int32_t d4pg_proj_loss(const float* target_logits, const float* q_logits, const float* pi_logits,
                                  const double* rewards, const uint8_t* dones,
                                  int32_t B, int32_t N, double v_min, double v_max, double discount,
                                  int32_t proj_mode, int32_t flags, double prio_eps, float grad_scale,
                                  float* m, int32_t* bins_l, int32_t* bins_u,
                                  float* target_probs, float* q_probs,
                                  float* loss_rows, float* td, float* prio, float* dlogits_q,
                                  float* pi_rows, float* dlogits_pi, d4pg_stream_t stream) {
  using namespace d4pg;
  D4PG_REQUIRE(target_logits && q_logits && rewards && dones, D4PG_EINVAL, "d4pg_proj_loss: null input");
  D4PG_REQUIRE(B > 0 && N >= 2 && N <= D4PG_MAX_ATOMS, D4PG_EINVAL, "d4pg_proj_loss: need B>0, 2<=N<=%d (got B=%d N=%d)", D4PG_MAX_ATOMS, B, N);
  D4PG_REQUIRE(proj_mode == 0 || proj_mode == 1, D4PG_EINVAL, "d4pg_proj_loss: proj_mode must be 0 or 1");
  D4PG_REQUIRE((bins_l == nullptr) == (bins_u == nullptr), D4PG_EINVAL, "d4pg_proj_loss: bins_l/bins_u must both be set or both NULL");
  D4PG_REQUIRE(v_max > v_min, D4PG_EINVAL, "d4pg_proj_loss: v_max <= v_min");
  HeadsArgs a{};
  a.target_logits = target_logits; a.q_logits = q_logits; a.pi_logits = pi_logits;
  a.rewards = rewards; a.dones = dones; a.B = B; a.N = N; a.flags = flags; a.ld = N;
  a.v_min = v_min; a.v_max = v_max;
  a.delta = (v_max - v_min) / double(N - 1);        // ddpg.py:46
  a.discount = discount; a.prio_eps = prio_eps; a.grad_scale = grad_scale;
  a.m = m; a.bins_l = bins_l; a.bins_u = bins_u; a.target_probs = target_probs; a.q_probs = q_probs;
  a.loss_rows = loss_rows; a.td = td; a.prio = prio; a.dlogits_q = dlogits_q;
  a.pi_rows = pi_rows; a.dlogits_pi = dlogits_pi;
  a.is_weights = nullptr; a.ce_priority = 0; a.only_policy = 0;
  return launch_heads(a, proj_mode, as_stream(stream));
}
