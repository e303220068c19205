// Device code of the fused projection / loss / priority / logit-gradient row kernel
// (included by proj_loss.cu).
#pragma once
#include "internal.cuh"

namespace d4pg {

constexpr int HEAD_WARPS = 4;

// softmax of one row held as 4 values per lane (atom k = lane + 32*t); fp32, max-subtracted,
// exp then divide (models.py:83 -> torch softmax).
template <int NT>
__device__ __forceinline__ void row_softmax(const float* __restrict__ logits, int N, int lane, float (&p)[NT],
                                            bool already_probs = false) {
  if (already_probs) {
#pragma unroll
    for (int t = 0; t < NT; ++t) { int k = lane + 32 * t; p[t] = (k < N) ? __ldg(logits + k) : 0.f; }
    return;
  }
  float x[NT];
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    int k = lane + 32 * t;
    x[t] = (k < N) ? __ldg(logits + k) : -INFINITY;
    mx = fmaxf(mx, x[t]);
  }
  mx = warp_max(mx);
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    int k = lane + 32 * t;
    p[t] = (k < N) ? expf(x[t] - mx) : 0.f;
    s += p[t];
  }
  s = warp_sum(s);
#pragma unroll
  for (int t = 0; t < NT; ++t) p[t] = p[t] / s;
}

// the same softmax on logits already in registers (rows whose loads were issued early)
template <int NT>
__device__ __forceinline__ void row_load(const float* __restrict__ logits, int N, int lane, float (&x)[NT], bool probs) {
#pragma unroll
  for (int t = 0; t < NT; ++t) { const int k = lane + 32 * t; x[t] = (k < N) ? __ldg(logits + k) : (probs ? 0.f : -INFINITY); }
}
template <int NT>
__device__ __forceinline__ void row_softmax_x(const float (&x)[NT], int N, int lane, float (&p)[NT], bool already_probs) {
  if (already_probs) {
#pragma unroll
    for (int t = 0; t < NT; ++t) p[t] = x[t];
    return;
  }
  float mx = -INFINITY;
#pragma unroll
  for (int t = 0; t < NT; ++t) mx = fmaxf(mx, x[t]);
  mx = warp_max(mx);
  float s = 0.f;
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    const int k = lane + 32 * t;
    p[t] = (k < N) ? expf(x[t] - mx) : 0.f;
    s += p[t];
  }
  s = warp_sum(s);
#pragma unroll
  for (int t = 0; t < NT; ++t) p[t] = p[t] / s;
}

// per-warp shared tables of one row (3.5 KB per warp)
struct HeadsWarpSmem {
  double wl[D4PG_MAX_ATOMS];
  double wu[D4PG_MAX_ATOMS];
  float p[D4PG_MAX_ATOMS];
  int l[D4PG_MAX_ATOMS];
  int u[D4PG_MAX_ATOMS];
};

// one batch row, executed by one warp.  parts: 1 = critic part (projection, CE loss, td, priority, d/d q-logits),
// 2 = policy head, 3 = both.  The two parts are independent, so the standalone kernel gives them to different warps;
// all global loads of a part are issued up front (three dependent round trips became one).
template <int MODE, int NT>
__device__ __forceinline__ void heads_row(const HeadsArgs& a, int row, int lane, HeadsWarpSmem& ws, int parts = 3) {
  const int N = a.N;
  const size_t ro = size_t(row) * a.ld;
  if (parts & 1) {

  // ---- target distribution ------------------------------------------------------------
  float p[NT], xt[NT], xq[NT];
  const bool t_probs = (a.flags & D4PG_PROJ_TARGET_IS_PROBS) != 0, q_probs = (a.flags & D4PG_PROJ_Q_IS_PROBS) != 0;
  row_load(a.target_logits + ro, N, lane, xt, t_probs);
  row_load(a.q_logits + ro, N, lane, xq, q_probs);
  const double r = a.rewards[row];
  const bool done = a.dones[row] != 0;
  const float isw = a.is_weights ? __ldg(a.is_weights + row) : 1.f;
  row_softmax_x(xt, N, lane, p, t_probs);

  float mk[NT];
#pragma unroll
  for (int t = 0; t < NT; ++t) mk[t] = 0.f;

  if (MODE == 0 && done) {
    // ddpg.py:165-181: zero the row, Dirac at clip(r); weights cast f64 -> f32
    double tz = fmin(a.v_max, fmax(a.v_min, r));
    double b = __ddiv_rn(__dsub_rn(tz, a.v_min), a.delta);
    double lf = floor(b), uf = ceil(b);
    int l = int(lf), u = int(uf);
    float wl = (l == u) ? 1.0f : __double2float_rn(__dsub_rn(uf, b));
    float wu = __double2float_rn(__dsub_rn(b, lf));
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      int k = lane + 32 * t;
      if (k < N) {
        if (k == l) mk[t] = wl;
        else if (k == u) mk[t] = wu;
        if (a.bins_l) { a.bins_l[ro + k] = l; a.bins_u[ro + k] = u; }
      }
    }
  } else {
    // per-atom bins and weights in fp64 (ddpg.py:155-158 / ddpg.py:129-134)
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      int j = lane + 32 * t;
      if (j < N) {
        double zj = __dadd_rn(a.v_min, __dmul_rn(double(j), a.delta));
        double c;
        if (MODE == 0) c = __dmul_rn(zj, a.discount);                        // (v_min+j*delta)*gamma
        else c = __dmul_rn(__dmul_rn(a.discount, done ? 0.0 : 1.0), zj);      // gamma^n*(1-d)*z_j
        double tz = fmin(a.v_max, fmax(a.v_min, __dadd_rn(r, c)));
        double b = __ddiv_rn(__dsub_rn(tz, a.v_min), a.delta);
        double lf = floor(b), uf = ceil(b);
        int l = int(lf), u = int(uf);
        double wl, wu;
        if (MODE == 0) {
          if (l == u) { wl = 1.0; wu = 0.0; }
          else { wl = __dsub_rn(uf, b); wu = __dsub_rn(b, lf); }
        } else {
          if (l == u && u > 0) l -= 1;                                        // ddpg.py:133
          if (l == u && l < N - 1) u += 1;                                    // ddpg.py:134
          wl = __dsub_rn(double(u), b);
          wu = __dsub_rn(b, double(l));
        }
        ws.p[j] = p[t];
        ws.l[j] = l; ws.u[j] = u;
        ws.wl[j] = wl; ws.wu[j] = wu;
        if (a.bins_l) { a.bins_l[ro + j] = l; a.bins_u[ro + j] = u; }
      }
    }
    __syncwarp();
    // ordered per-bin accumulation (gather form: lane owns output bins, visits atoms in order).
    // b_j is non-decreasing in j, so the atoms that touch bin k (l_j == k or u_j == k) form one
    // contiguous run [j0, j1): two binary searches over the shared tables bound the loop to the few
    // atoms that matter (gamma < 1 => ~2-3 per bin; clamped atoms pile up only on the edge bins).
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      const int k = lane + 32 * t;
      if (k >= N) continue;
      int lo = 0, hi = N;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (ws.u[mid] >= k) hi = mid; else lo = mid + 1; }
      const int j0 = lo;
      hi = N;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (ws.l[mid] > k) hi = mid; else lo = mid + 1; }
      const int j1 = lo;
      if (MODE == 0) {
        float acc = 0.f;
        for (int j = j0; j < j1; ++j) {
          const int l = ws.l[j], u = ws.u[j];
          const double pj = double(ws.p[j]);
          if (k == l) {
            // eq: f32+f32 add; ne: f32 + (f64 product) in f64, rounded to f32
            const double term = (l == u) ? pj : __dmul_rn(pj, ws.wl[j]);
            acc = __double2float_rn(__dadd_rn(double(acc), term));
          } else if (k == u) {
            acc = __double2float_rn(__dadd_rn(double(acc), __dmul_rn(pj, ws.wu[j])));
          }
        }
        mk[t] = acc;
      } else {
        double acc = 0.;
        for (int j = j0; j < j1; ++j) {
          const int l = ws.l[j], u = ws.u[j];
          const double pj = double(ws.p[j]);
          if (k == l) acc = __dadd_rn(acc, __dmul_rn(pj, ws.wl[j]));
          if (k == u) acc = __dadd_rn(acc, __dmul_rn(pj, ws.wu[j]));
        }
        mk[t] = __double2float_rn(acc);
      }
    }
  }

  // ---- online critic: CE loss, TD proxy, priority, d loss / d logits -------------------
  float q[NT];
  row_softmax_x(xq, N, lane, q, q_probs);
  float ce = 0.f, mq = 0.f, sq = 0.f;
  float gq[NT];
  const float gscale = a.grad_scale * isw;
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    int k = lane + 32 * t;
    gq[t] = 0.f;
    if (k < N) {
      float qe = q[t] + 1e-10f;
      ce += mk[t] * logf(qe);
      mq += mk[t] * q[t];
      gq[t] = -(mk[t] / qe) * gscale;                // d mean-loss / d q_k
      sq += q[t] * gq[t];
    }
  }
  ce = warp_sum(ce); mq = warp_sum(mq); sq = warp_sum(sq);
#pragma unroll
  for (int t = 0; t < NT; ++t) {
    int k = lane + 32 * t;
    if (k < N) {
      if (a.m) a.m[ro + k] = mk[t];
      if (a.target_probs) a.target_probs[ro + k] = p[t];
      if (a.q_probs) a.q_probs[ro + k] = q[t];
      if (a.dlogits_q) a.dlogits_q[ro + k] = q[t] * (gq[t] - sq);   // softmax backward
    }
  }
  if (lane == 0) {
    float tdv = -mq;
    if (a.loss_rows) a.loss_rows[row] = -ce * isw;
    if (a.td) a.td[row] = tdv;
    if (a.prio) a.prio[row] = (a.ce_priority ? -ce : fabsf(tdv)) + float(a.prio_eps);   // np.abs(f32) + 1e-6 (f32)
  }

  }   // parts & 1

  // ---- policy head: -E_q[z] and its logit gradient --------------------------------------
  if ((parts & 2) && a.pi_logits) {
    float qp[NT];
    row_softmax(a.pi_logits + ro, N, lane, qp);
    float ez = 0.f;
    float z[NT];
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      int k = lane + 32 * t;
      z[t] = (k < N) ? float(__dadd_rn(a.v_min, __dmul_rn(double(k), a.delta))) : 0.f;  // ddpg.py:47,238
      ez += qp[t] * z[t];
    }
    ez = warp_sum(ez);
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      int k = lane + 32 * t;
      if (k < N && a.dlogits_pi) a.dlogits_pi[ro + k] = -a.grad_scale * qp[t] * (z[t] - ez);
    }
    if (lane == 0 && a.pi_rows) a.pi_rows[row] = -ez;
  }
}


template <int MODE, int NT>
__global__ void __launch_bounds__(HEAD_WARPS * 32) heads_kernel(const HeadsArgs a) {
  __shared__ HeadsWarpSmem ws[HEAD_WARPS];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x * HEAD_WARPS + warp;            // warps [0, B): critic part of row g; [B, 2B): policy head of row g - B
  step_stamp(a.trace, 2);
  if (a.only_policy) { if (g < a.B) heads_row<MODE, NT>(a, g, lane, ws[warp], 2); }
  else if (g < a.B) heads_row<MODE, NT>(a, g, lane, ws[warp], 1);
  else if (g < 2 * a.B) heads_row<MODE, NT>(a, g - a.B, lane, ws[warp], 2);
  step_stamp(a.trace, 2 + 16);
  if (a.sampler_clock && blockIdx.x == 0 && threadIdx.x == 0) {
    a.sampler_clock->s_adam_step += 1; a.sampler_clock->s_beta_t += 1; a.sampler_clock->s_steps_done += 1;
  }
}

}  // namespace d4pg
