// Fused Adam (beta=(0.9,0.9) by default) + Polyak soft target update over flat fp32 buffers.
//
// Replaces (reference, relative to /root/reference):
//   shared_adam.py:3-17 + torch.optim.Adam.step as called at ddpg.py:232,244.  Arithmetic follows
//     torch 2.11 `_single_tensor_adam` (the form the reference executes in this image):
//       m <- lerp(m, g, 1-b1); v <- v*b2 + (1-b2)*g*g;
//       p <- p - (lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps),  bc = 1 - b^step
//   ddpg.py:118-120 sync_local_global: identity (local and global share storage)
//   ddpg.py:110-116 update_target_parameters: t <- (1-tau)*t + tau*p   (p = post-step value)
// Pure streaming kernel: 4 reads + 4 writes of P floats -> HBM/L2 bound, float4 vectorised.
#include "adam_dev.cuh"
#include <math.h>
#include <algorithm>

namespace d4pg {

__global__ void __launch_bounds__(256) adam_polyak_kernel(const AdamArgs a) {
  __shared__ float red[2][8];
  if (int(blockIdx.y) == a.nseg) {
    if (blockIdx.x == 0) adam_tail(a, red);
    return;
  }
  step_stamp(a.trace, 7);
  adam_segment(a, blockIdx.y, blockIdx.x, gridDim.x);
  step_stamp(a.trace, 7 + 16);
}


int launch_adam(const AdamArgs& a_in, cudaStream_t st) {
  AdamArgs a = a_in;
  a.trace = (a.clock && debug_trace_buffer()) ? debug_trace_buffer() + STEP_TRACE_BASE : nullptr;
  int64_t nmax = 0;
  for (int i = 0; i < a.nseg; ++i) nmax = a.seg[i].n > nmax ? a.seg[i].n : nmax;
  int blocks = int((nmax / 4 + 255) / 256);
  if (blocks > 148 * 4) blocks = 148 * 4;
  if (blocks < 1) blocks = 1;
  D4PG_MAX_CARVEOUT(adam_polyak_kernel);
  const int tail = ((a.clock || a.loss_out) && !a.skip_tail) ? 1 : 0;
  adam_polyak_kernel<<<dim3(blocks, a.nseg + tail), 256, 0, st>>>(a);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

}  // namespace d4pg

using namespace d4pg;

extern "C" int32_t d4pg_adam_polyak(float* p, const float* g, float* m, float* v, float* target, int64_t n,
                                    double lr, double beta1, double beta2, double eps, int64_t step,
                                    double tau, float grad_scale, d4pg_stream_t stream) {
  D4PG_REQUIRE(p && g && m && v, D4PG_EINVAL, "d4pg_adam_polyak: null buffer");
  D4PG_REQUIRE(n > 0 && n % 4 == 0, D4PG_EINVAL, "d4pg_adam_polyak: n must be a positive multiple of 4 (flat layout is 4-aligned)");
  D4PG_REQUIRE(step >= 1, D4PG_EINVAL, "d4pg_adam_polyak: step is the post-increment count (>= 1)");
  AdamArgs a{};
  const double bc1 = 1.0 - pow(beta1, double(step));
  const double bc2 = 1.0 - pow(beta2, double(step));
  a.seg[0] = AdamSeg{p, g, m, v, target, n, nullptr, 0, float(-(lr / bc1)), -1};
  a.seg[0].nimg = 0;
  a.nseg = 1;
  a.w1 = float(1.0 - beta1); a.w2 = float(1.0 - beta2); a.beta2 = float(beta2); a.eps = float(eps);
  a.bc2_sqrt = float(sqrt(bc2)); a.tau = float(tau); a.one_minus_tau = float(1.0 - tau);
  a.grad_scale = grad_scale; a.clock = nullptr; a.loss_out = nullptr; a.pipe_slot = -1; a.trace = nullptr; a.npeers = 0; a.my_flags = nullptr;
  return launch_adam(a, as_stream(stream));
}

namespace d4pg {
__global__ void polyak_kernel(float* t, const float* s, int64_t n, float tau, float omt) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x)
    t[i] = __fadd_rn(__fmul_rn(omt, t[i]), __fmul_rn(tau, s[i]));
}
}  // namespace d4pg

extern "C" int32_t d4pg_polyak(float* target, const float* src, int64_t n, double tau, d4pg_stream_t stream) {
  D4PG_REQUIRE(target && src && n > 0, D4PG_EINVAL, "d4pg_polyak: bad arguments");
  int blocks = int(std::min<int64_t>(592, (n + 255) / 256));
  polyak_kernel<<<blocks, 256, 0, as_stream(stream)>>>(target, src, n, float(tau), float(1.0 - tau));
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

extern "C" int32_t d4pg_copy_f32(float* dst, const float* src, int64_t n, d4pg_stream_t stream) {
  D4PG_REQUIRE(dst && src && n >= 0, D4PG_EINVAL, "d4pg_copy_f32: bad arguments");
  D4PG_CUDA_OK(cudaMemcpyAsync(dst, src, size_t(n) * sizeof(float), cudaMemcpyDeviceToDevice, as_stream(stream)));
  return D4PG_OK;
}
