// C-ABI plumbing: error channel, version, network layouts, standalone actor/critic forward.
#include "common.cuh"
#include "gemm_ffma.cuh"
#include <string.h>

namespace d4pg {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static NetDims make_dims(const int* in, const int* out) {
  NetDims d{};
  int64_t off = 0;
  for (int l = 0; l < 4; ++l) {
    d.in[l] = in[l]; d.out[l] = out[l]; d.ld[l] = pitch4(in[l]);
    d.w_off[l] = off; off = align4(off + int64_t(d.ld[l]) * out[l]);
    d.b_off[l] = off; off = align4(off + out[l]);
  }
  d.total = off;
  return d;
}
// models.py:18-23
NetDims actor_dims(int obs_dim, int act_dim) {
  const int in[4] = {obs_dim, D4PG_HIDDEN, D4PG_HIDDEN, D4PG_HIDDEN};
  const int out[4] = {D4PG_HIDDEN, D4PG_HIDDEN, D4PG_HIDDEN, act_dim};
  return make_dims(in, out);
}
// models.py:56-62
NetDims critic_dims(int obs_dim, int act_dim, int n_atoms) {
  const int in[4] = {obs_dim, D4PG_HIDDEN + act_dim, D4PG_HIDDEN, D4PG_HIDDEN};
  const int out[4] = {D4PG_HIDDEN, D4PG_HIDDEN, D4PG_HIDDEN, n_atoms};
  return make_dims(in, out);
}

static void fill_layout(const NetDims& d, d4pg_net_layout_t* out) {
  for (int l = 0; l < 4; ++l) {
    out->offsets[2 * l] = d.w_off[l]; out->sizes[2 * l] = int64_t(d.ld[l]) * d.out[l]; out->pitch[l] = d.ld[l];
    out->offsets[2 * l + 1] = d.b_off[l]; out->sizes[2 * l + 1] = d.out[l];
  }
  out->total = d.total;
}

__global__ void softmax_rows_kernel(const float* logits, float* probs, int B, int N) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= B) return;
  const float* x = logits + size_t(warp) * N;
  float mx = -INFINITY;
  for (int k = lane; k < N; k += 32) mx = fmaxf(mx, x[k]);
  mx = warp_max(mx);
  float s = 0.f;
  for (int k = lane; k < N; k += 32) s += expf(x[k] - mx);
  s = warp_sum(s);
  for (int k = lane; k < N; k += 32) probs[size_t(warp) * N + k] = expf(x[k] - mx) / s;
}

}  // namespace d4pg

using namespace d4pg;

extern "C" const char* d4pg_last_error(void) { return g_err; }
extern "C" int32_t d4pg_version(void) { return 100; }   /* 0.1.0 */
/* sizeof of the structs that cross the ABI by pointer: a binding whose mirror has another size is out of date */
extern "C" int32_t d4pg_struct_size(int32_t which) {
  switch (which) {
    case 0: return int32_t(sizeof(d4pg_learner_config_t));
    case 1: return int32_t(sizeof(d4pg_learner_buffers_t));
    case 2: return int32_t(sizeof(d4pg_net_layout_t));
    default: return -1;
  }
}

extern "C" int32_t d4pg_device_sm(void) {
  int dev = 0, major = 0, minor = 0;
  D4PG_CUDA_OK(cudaGetDevice(&dev));
  D4PG_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
  D4PG_CUDA_OK(cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, dev));
  return major * 10 + minor;
}

extern "C" int32_t d4pg_actor_layout(int32_t obs_dim, int32_t act_dim, d4pg_net_layout_t* out) {
  D4PG_REQUIRE(out && obs_dim > 0 && act_dim > 0, D4PG_EINVAL, "d4pg_actor_layout: bad arguments");
  fill_layout(actor_dims(obs_dim, act_dim), out);
  return D4PG_OK;
}
extern "C" int32_t d4pg_critic_layout(int32_t obs_dim, int32_t act_dim, int32_t n_atoms, d4pg_net_layout_t* out) {
  D4PG_REQUIRE(out && obs_dim > 0 && act_dim > 0 && n_atoms >= 2 && n_atoms <= D4PG_MAX_ATOMS, D4PG_EINVAL,
               "d4pg_critic_layout: bad arguments");
  fill_layout(critic_dims(obs_dim, act_dim, n_atoms), out);
  return D4PG_OK;
}

// actor.forward, models.py:32-41: fc1 -> relu -> fc2 -> fc2_2 -> relu -> fc3 -> tanh  (no relu after fc2, H9)
extern "C" int32_t d4pg_actor_forward(const float* params, int32_t obs_dim, int32_t act_dim,
                                      const float* s, int32_t B, float* action, float* workspace,
                                      int32_t precision, d4pg_stream_t stream) {
  D4PG_REQUIRE(params && s && action && workspace && B > 0, D4PG_EINVAL, "d4pg_actor_forward: null/empty argument");
  D4PG_REQUIRE(precision >= 0 && precision <= 2, D4PG_ENOTSUP, "d4pg_actor_forward: unknown precision %d", precision);
  const NetDims d = actor_dims(obs_dim, act_dim);
  const int H = D4PG_HIDDEN;
  float* h1 = workspace; float* h2 = h1 + size_t(B) * H; float* h3 = h2 + size_t(B) * H;
  cudaStream_t st = as_stream(stream);
  const float* X[4] = {s, h1, h2, h3};
  float* Y[4] = {h1, h2, h3, action};
  const int epi[4] = {EPI_BIAS_RELU, EPI_BIAS, EPI_BIAS_RELU, EPI_BIAS_TANH};
  for (int l = 0; l < 4; ++l) {
    GemmBatch b; gemm_batch_begin(b);
    gemm_batch_add(b, gemm_fwd(X[l], d.in[l], nullptr, 0, 0, params + d.w_off[l], d.ld[l], params + d.b_off[l],
                               Y[l], d.out[l], B, d.out[l], d.in[l], epi[l]));
    int rc = gemm_launch(b, precision, st);
    if (rc) return rc;
  }
  return D4PG_OK;
}

// critic.forward, models.py:76-88: fc1 -> relu -> cat(.,a) -> fc2 -> relu -> fc2_2 -> relu -> fc3 -> softmax
extern "C" int32_t d4pg_critic_forward(const float* params, int32_t obs_dim, int32_t act_dim, int32_t n_atoms,
                                       const float* s, const float* a, int32_t B, float* probs, float* logits,
                                       float* workspace, int32_t precision, d4pg_stream_t stream) {
  D4PG_REQUIRE(params && s && a && workspace && B > 0 && (probs || logits), D4PG_EINVAL, "d4pg_critic_forward: null/empty argument");
  D4PG_REQUIRE(precision >= 0 && precision <= 2, D4PG_ENOTSUP, "d4pg_critic_forward: unknown precision %d", precision);
  D4PG_REQUIRE(n_atoms >= 2 && n_atoms <= D4PG_MAX_ATOMS, D4PG_EINVAL, "d4pg_critic_forward: n_atoms out of range");
  const NetDims d = critic_dims(obs_dim, act_dim, n_atoms);
  const int H = D4PG_HIDDEN;
  float* h1 = workspace; float* h2 = h1 + size_t(B) * H; float* h3 = h2 + size_t(B) * H;
  // logits scratch lives behind h3 when the caller only wants probabilities
  float* z = logits ? logits : h1;   // h1 is dead after fc2
  cudaStream_t st = as_stream(stream);
  int rc;
  GemmBatch b;
  gemm_batch_begin(b);
  gemm_batch_add(b, gemm_fwd(s, obs_dim, nullptr, 0, 0, params + d.w_off[0], d.ld[0], params + d.b_off[0], h1, H, B, H, obs_dim, EPI_BIAS_RELU));
  if ((rc = gemm_launch(b, precision, st))) return rc;
  gemm_batch_begin(b);
  gemm_batch_add(b, gemm_fwd(h1, H, a, act_dim, H, params + d.w_off[1], d.ld[1], params + d.b_off[1], h2, H, B, H, H + act_dim, EPI_BIAS_RELU));
  if ((rc = gemm_launch(b, precision, st))) return rc;
  gemm_batch_begin(b);
  gemm_batch_add(b, gemm_fwd(h2, H, nullptr, 0, 0, params + d.w_off[2], H, params + d.b_off[2], h3, H, B, H, H, EPI_BIAS_RELU));
  if ((rc = gemm_launch(b, precision, st))) return rc;
  gemm_batch_begin(b);
  gemm_batch_add(b, gemm_fwd(h3, H, nullptr, 0, 0, params + d.w_off[3], H, params + d.b_off[3], z, n_atoms, B, n_atoms, H, EPI_BIAS));
  if ((rc = gemm_launch(b, precision, st))) return rc;
  if (probs) {
    softmax_rows_kernel<<<cdiv(B * 32, 256), 256, 0, st>>>(z, probs, B, n_atoms);
    D4PG_LAUNCH_OK();
  }
  return D4PG_OK;
}
