// Shared host/device helpers for libd4pg_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/d4pg_b200.h"

namespace d4pg {

void set_error(const char* fmt, ...);

#define D4PG_CUDA_OK(expr)                                                              \
  do {                                                                                  \
    cudaError_t _e = (expr);                                                            \
    if (_e != cudaSuccess) {                                                            \
      ::d4pg::set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return D4PG_ECUDA;                                                                \
    }                                                                                   \
  } while (0)

#define D4PG_REQUIRE(cond, code, ...)                                                   \
  do {                                                                                  \
    if (!(cond)) { ::d4pg::set_error(__VA_ARGS__); return (code); }                     \
  } while (0)

#define D4PG_LAUNCH_OK()                                                                \
  do {                                                                                  \
    cudaError_t _e = cudaGetLastError();                                                \
    if (_e != cudaSuccess) {                                                            \
      ::d4pg::set_error("%s:%d: kernel launch -> %s", __FILE__, __LINE__, cudaGetErrorString(_e)); \
      return D4PG_ECUDA;                                                                \
    }                                                                                   \
  } while (0)

// All kernels of a step ask for the same (maximum) shared-memory carve-out: a step mixes kernels
// with 0 KB, 14 KB, 32 KB and 197 KB of shared memory, and letting the driver pick a per-kernel
// L1/shared split makes every kernel boundary an SM reconfiguration (ncu: ~17 us of a 20 us
// gemm_tc2 launch had no active SM cycles).
#define D4PG_MAX_CARVEOUT(kernel)                                                                     \
  do {                                                                                                \
    static bool _carved = false;                                                                      \
    if (!_carved) {                                                                                   \
      cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout,                    \
                           int(cudaSharedmemCarveoutMaxShared));                                      \
      _carved = true;                                                                                 \
    }                                                                                                 \
  } while (0)

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------
// Only the host pipeline's sample kernel is launched with the programmatic-stream-serialization attribute
// (replay.cu: launch_sample): the tree add before it triggers early, the sample kernel waits for its writes.
__device__ __forceinline__ void pdl_trigger_raw() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// step timeline (D4PG_TC_TRACE): thread 0 of CTA 0 of every step kernel stamps %globaltimer at entry / exit
__device__ __forceinline__ void step_stamp(unsigned long long* tr, int slot) {
  if (tr && blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0) {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    tr[slot] = t;
  }
}
unsigned long long* debug_trace_buffer();
constexpr int STEP_TRACE_BASE = 96;      // stamps [96, 128) of the debug buffer: entry of kernel k at 96+k, exit at 112+k

static inline cudaStream_t as_stream(d4pg_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

__host__ __device__ static inline int64_t align4(int64_t x) { return (x + 3) & ~int64_t(3); }
__host__ __device__ static inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// ---- warp helpers --------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- Philox4x32-10 (counter-based RNG for device-side sampling) -----------------------
struct Philox {
  __device__ static inline void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
    uint32_t hi0 = __umulhi(M0, c[0]), lo0 = M0 * c[0];
    uint32_t hi1 = __umulhi(M1, c[2]), lo1 = M1 * c[2];
    uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
  }
  // 53-bit uniform in [0,1), same construction as CPython's random.random():
  // (a>>5, b>>6) -> (a*2^26 + b) / 2^53.
  __device__ static inline double uniform53(uint64_t seed, uint64_t counter, uint32_t lane) {
    uint32_t c[4] = {uint32_t(counter), uint32_t(counter >> 32), lane, 0x9E3779B9u};
    uint32_t k0 = uint32_t(seed), k1 = uint32_t(seed >> 32);
#pragma unroll
    for (int i = 0; i < 10; ++i) {
      round(c, k0, k1);
      k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    uint32_t a = c[0] >> 5, b = c[1] >> 6;
    return (double(a) * 67108864.0 + double(b)) * (1.0 / 9007199254740992.0);
  }
};

// ---- network layout ------------------------------------------------------------------
struct NetDims {
  int in[4], out[4];        // per layer fc1, fc2, fc2_2, fc3
  int ld[4];                // row pitch of each weight matrix in floats: in[] rounded up to 4 (16-B rows,
                            // so every operand is TMA- and float4-addressable); pad columns stay zero
  int64_t w_off[4], b_off[4];
  int64_t total;
};
__host__ __device__ static inline int pitch4(int x) { return (x + 3) & ~3; }
NetDims actor_dims(int obs_dim, int act_dim);
NetDims critic_dims(int obs_dim, int act_dim, int n_atoms);

}  // namespace d4pg
