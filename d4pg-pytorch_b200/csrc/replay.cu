// GPU-resident prioritized replay: fp32 sum/min segment trees + SoA transition storage.
//
// Replaces (reference, relative to /root/reference):
//   prioritized_replay_memory.py:33-113   SegmentTree (__setitem__, reduce, _reduce_helper)
//   prioritized_replay_memory.py:114-162  SumSegmentTree.sum/find_prefixsum_idx, MinSegmentTree.min
//   prioritized_replay_memory.py:164-222  ReplayBuffer.add/_encode_sample
//   prioritized_replay_memory.py:224-335  PrioritizedReplayBuffer.add/_sample_proportional/sample/
//                                         update_priorities
//   replay_memory.py:14-19,61-80          Replay.add / Replay.sample (gather only)
//
// Tree layout is the reference's: root at 1, leaves at [cap, 2cap), V[i] = op(V[2i], V[2i+1]).
// Node dtype is fp32 -- what the reference's Python evaluates to under NumPy 2 (SURVEY.md H11).
// Everything is HBM/L2 pointer chasing + row gathers: no tensor-core work here.
#include "replay_dev.cuh"
#include <new>
#include <string.h>
#include <algorithm>

struct d4pg_replay {
  int64_t size, cap; int log2cap;
  int obs_dim, act_dim;
  double alpha; float alpha_f32;
  float* sum; float* mn;
  float* obs; float* act; double* rew; float* obs2; uint8_t* done;
  int32_t* scratch; float* state;
  int64_t len, next_idx;
  int pristine;
  int64_t gen;            // bumped by every external mutation (add / set / update): a learner's prefetched batch is stale
  // host ingest staging (caller-owned buffers registered by d4pg_replay_set_staging)
  // two slots (halves of the registered buffers) so the host can stage add k+1 while add k still waits on the device
  uint8_t* stage_host; uint8_t* stage_dev; int64_t stage_bytes; cudaEvent_t stage_ev[2]; bool stage_busy[2]; int stage_slot;
  // ingest gate (learner host pipeline): the next kernel that touches the store / trees on the ingest stream first waits
  // until *gate_flag >= gate_target (the priority write-back of the last launched learner step)
  // The flag lives with the buffer (learners come and go); every gated step bumps it once and arms target = #armed.
  unsigned long long* gate_flag; unsigned long long gate_target; bool gate_pending;
  cudaEvent_t order_ev;
};

namespace d4pg {
// step timeline (D4PG_TC_TRACE, tools/e2e_timeline.py): ingest kernels stamp slots 10 (gate), 11 (ring write), 12 (tree add)
static unsigned long long* step_trace() { unsigned long long* p = debug_trace_buffer(); return p ? p + STEP_TRACE_BASE : nullptr; }


__global__ void __launch_bounds__(SAMPLE_THREADS) sample_gather_kernel(const SampleArgs a) {
  __shared__ SampleSmem sm;
  pdl_wait();
  step_stamp(a.trace, a.trace_slot);
  sample_body(a, blockIdx.x, sm);
  if (a.done_epoch) {                          // the forward chains of the step poll these instead of a stream event
    __syncthreads();
    if (threadIdx.x == 0) {
      __threadfence();
      const unsigned long long e = (unsigned long long)(a.clock->s_steps_done + 1);
      asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(a.done_epoch + blockIdx.x), "l"(e) : "memory");
    }
  }
  step_stamp(a.trace, a.trace_slot + 16);
}

template <int MODE>
__global__ void __launch_bounds__(TREE_THREADS) tree_write_kernel(const TreeArgs a) {
  __shared__ float red[32];
  step_stamp(a.trace, 3);
  tree_write_body<MODE, TREE_THREADS>(a, red);
  step_stamp(a.trace, 3 + 16);
}


__global__ void __launch_bounds__(TREE_FAST_MAX) tree_update_fast_kernel(const TreeArgs a, int hs, int D) {
  extern __shared__ __align__(16) unsigned char tree_smem[];
  __shared__ float red[32];
  step_stamp(a.trace, 3);
  tree_update_fast_body(a, tree_smem, hs, red, blockIdx.x, D);
  step_stamp(a.trace, 3 + 16);
}

// add(): the new leaves are one contiguous ring range [start, start+n) (no wrap: the host splits a
// wrapping add), so level l only has the nodes (cap+start)>>l .. (cap+start+n-1)>>l to recompute:
// ~2n node updates in total instead of n*log2(cap), and the narrow top of the tree is finished by
// one warp without block-wide barriers.
__global__ void __launch_bounds__(TREE_THREADS) tree_add_range_kernel(float* sum, float* mn, int64_t cap, int log2cap,
                                                                      int64_t start, int64_t n, const ReplayState* state,
                                                                      float alpha_f32) {
  const int t = threadIdx.x;
  const float leaf = pow_alpha(state->max_priority, alpha_f32);      // :255-256
  for (int64_t i = t; i < n; i += TREE_THREADS) { sum[cap + start + i] = leaf; mn[cap + start + i] = leaf; }
  int lvl = 1;
  for (; lvl <= log2cap; ++lvl) {
    const int64_t lo = (cap + start) >> lvl, hi = (cap + start + n - 1) >> lvl;
    if (hi - lo + 1 <= 32) break;                                     // narrow: hand over to warp 0
    __syncthreads();
    for (int64_t node = lo + t; node <= hi; node += TREE_THREADS) {
      sum[node] = __fadd_rn(__ldcg(sum + 2 * node), __ldcg(sum + 2 * node + 1));
      mn[node] = fminf(__ldcg(mn + 2 * node), __ldcg(mn + 2 * node + 1));
    }
  }
  __syncthreads();
  if (t < 32) {
    for (; lvl <= log2cap; ++lvl) {
      const int64_t lo = (cap + start) >> lvl, hi = (cap + start + n - 1) >> lvl;
      const int64_t node = lo + t;
      if (node <= hi) {
        sum[node] = __fadd_rn(__ldcg(sum + 2 * node), __ldcg(sum + 2 * node + 1));
        mn[node] = fminf(__ldcg(mn + 2 * node), __ldcg(mn + 2 * node + 1));
      }
      __threadfence_block();
      __syncwarp();
    }
  }
}

// The same update with ONE round trip to L2 (n <= TREE_ADD_FAST_MAX): a parent inside the recomputed range has both
// children inside the range of the level below, except at the two edges, where the outside child is an OLD node.
// Those <= 2 old nodes per level (and tree) are fetched up front, in flight together; the levels are then computed
// from shared memory.  Identical arithmetic (fp32 left + right, fminf), so the resulting tree is bit-identical.
constexpr int TREE_ADD_FAST_MAX = 2048;
__global__ void __launch_bounds__(TREE_THREADS) tree_add_range_fast_kernel(float* sum, float* mn, int64_t cap, int log2cap,
                                                                           int64_t start, int64_t n, const ReplayState* state,
                                                                           float alpha_f32, unsigned long long* trace,
                                                                           const unsigned long long* gate_flag,
                                                                           unsigned long long gate_target) {
  __shared__ float vs[2][TREE_ADD_FAST_MAX], vm[2][TREE_ADD_FAST_MAX];
  __shared__ float old_s[2][32], old_m[2][32];                         // [left / right edge][level]
  const int t = threadIdx.x;
  step_stamp(trace, 10);
  if (gate_flag) {                                                     // ingest gate, fused: saves a kernel boundary
    if (t == 0) {
      unsigned long long v;
      do { asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(gate_flag) : "memory"); } while (v < gate_target);
    }
    __syncthreads();
  }
  pdl_trigger_raw();      // a programmatically dependent sample kernel (host pipeline) may become resident now; it still waits for this grid's end
  step_stamp(trace, 12);
  const float leaf = pow_alpha(state->max_priority, alpha_f32);       // :255-256
  if (t < 2 * log2cap) {
    const int lvl = (t >> 1) + 1, side = t & 1;                        // the outside child needed by level `lvl`
    const int64_t plo = (cap + start) >> (lvl - 1), phi = (cap + start + n - 1) >> (lvl - 1);
    float a = 0.f, b = INFINITY;
    if (side == 0 && (plo & 1)) { a = __ldcg(sum + plo - 1); b = __ldcg(mn + plo - 1); }
    if (side == 1 && !(phi & 1)) { a = __ldcg(sum + phi + 1); b = __ldcg(mn + phi + 1); }
    old_s[side][lvl] = a; old_m[side][lvl] = b;
  }
  for (int64_t i = t; i < n; i += TREE_THREADS) {
    sum[cap + start + i] = leaf; mn[cap + start + i] = leaf;
    vs[0][i] = leaf; vm[0][i] = leaf;
  }
  __syncthreads();
  for (int lvl = 1; lvl <= log2cap; ++lvl) {
    const int cur = lvl & 1, prev = cur ^ 1;
    const int64_t lo = (cap + start) >> lvl, hi = (cap + start + n - 1) >> lvl;
    const int64_t plo = (cap + start) >> (lvl - 1), phi = (cap + start + n - 1) >> (lvl - 1);
    for (int64_t j = t; j <= hi - lo; j += TREE_THREADS) {
      const int64_t node = lo + j, l = 2 * node, r = 2 * node + 1;
      const float ls = l >= plo ? vs[prev][l - plo] : old_s[0][lvl], lm = l >= plo ? vm[prev][l - plo] : old_m[0][lvl];
      const float rs = r <= phi ? vs[prev][r - plo] : old_s[1][lvl], rm = r <= phi ? vm[prev][r - plo] : old_m[1][lvl];
      const float s2 = __fadd_rn(ls, rs), m2 = fminf(lm, rm);
      vs[cur][j] = s2; vm[cur][j] = m2;
      sum[node] = s2; mn[node] = m2;
    }
    __syncthreads();
  }
  step_stamp(trace, 12 + 16);
}

// bulk path for large adds: grid-wide leaf fill, then one launch per level
__global__ void leaf_fill_kernel(float* sum, float* mn, int64_t cap, int64_t size, int64_t ring_start,
                                 int64_t n, const ReplayState* state, float alpha_f32) {
  const float leaf = pow_alpha(state->max_priority, alpha_f32);
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t p = (ring_start + i) % size;
    sum[cap + p] = leaf; mn[cap + p] = leaf;
  }
}
__global__ void level_rebuild_kernel(float* sum, float* mn, int64_t first, int64_t count) {
  for (int64_t i = blockIdx.x * int64_t(blockDim.x) + threadIdx.x; i < count; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t node = first + i;
    sum[node] = __fadd_rn(sum[2 * node], sum[2 * node + 1]);
    mn[node] = fminf(mn[2 * node], mn[2 * node + 1]);
  }
}

// ring insert of n rows from device staging buffers (ReplayBuffer.add, :180-187)
__global__ void ring_write_kernel(float* obs, float* act, double* rew, float* obs2, uint8_t* done,
                                  const float* s, const float* a, const double* r, const float* s2,
                                  const uint8_t* d, int64_t n, int obs_dim, int act_dim,
                                  int64_t size, int64_t ring_start, ReplayState* state,
                                  int64_t new_len, int64_t new_next, unsigned long long* trace) {
  const int64_t stride = int64_t(gridDim.x) * blockDim.x, t0 = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  step_stamp(trace, 11);
  if (t0 == 0) { state->len = new_len; state->next_idx = new_next; }
  for (int64_t e = t0; e < n * obs_dim; e += stride) {
    const int64_t i = e / obs_dim, c = e - i * obs_dim, p = (ring_start + i) % size;
    obs[p * obs_dim + c] = s[e];
    obs2[p * obs_dim + c] = s2[e];
  }
  for (int64_t e = t0; e < n * act_dim; e += stride) {
    const int64_t i = e / act_dim, c = e - i * act_dim, p = (ring_start + i) % size;
    act[p * act_dim + c] = a[e];
  }
  for (int64_t i = t0; i < n; i += stride) {
    const int64_t p = (ring_start + i) % size;
    rew[p] = r[i]; done[p] = d[i];
  }
  step_stamp(trace, 11 + 16);
}

__global__ void tree_init_kernel(float* sum, float* mn, int32_t* scratch, ReplayState* state, int64_t cap) {
  const int64_t stride = int64_t(gridDim.x) * blockDim.x;
  const int64_t t0 = blockIdx.x * int64_t(blockDim.x) + threadIdx.x;
  for (int64_t i = t0; i < 2 * cap; i += stride) {
    sum[i] = 0.f; mn[i] = INFINITY;                                  // neutral elements, :116-120,152-156
    if (i < cap) scratch[i] = -1;
  }
  if (t0 == 0) {
    state->max_priority = 1.0f;                                      // :249
    state->pristine = 1; state->len = 0; state->next_idx = 0; state->reserved = 0;
  }
}

__global__ void state_set_kernel(ReplayState* state, int64_t len, int64_t next_idx, int pristine) {
  state->len = len; state->next_idx = next_idx; state->pristine = pristine;
}

// SegmentTree.reduce(start, end+1) for an arbitrary range with _reduce_helper's association
// (:61-96): after the first split the left part is a suffix query (left-nested from the deepest
// node up) and the right part a prefix query (right-nested); IS_SUM selects + or min.
template <bool IS_SUM>
__device__ float range_reduce_ref(const float* __restrict__ V, int64_t cap, int64_t s, int64_t e) {
  auto op = [](float a, float b) { return IS_SUM ? __fadd_rn(a, b) : fminf(a, b); };
  int64_t node = 1, lo = 0, hi = cap - 1;
  while (true) {                                   // descend while the range sits in one child
    if (s == lo && e == hi) return __ldcg(V + node);
    const int64_t mid = (lo + hi) >> 1;
    if (e <= mid) { node = 2 * node; hi = mid; }
    else if (s > mid) { node = 2 * node + 1; lo = mid + 1; }
    else break;
  }
  const int64_t mid = (lo + hi) >> 1;
  // left: suffix [s, mid] of node 2*node
  float terms[40]; int n = 0;
  int64_t nd = 2 * node, l2 = lo, h2 = mid;
  while (s != l2) {
    const int64_t m2 = (l2 + h2) >> 1;
    if (s > m2) { nd = 2 * nd + 1; l2 = m2 + 1; }
    else { terms[n++] = __ldcg(V + 2 * nd + 1); nd = 2 * nd; h2 = m2; }
  }
  float left = __ldcg(V + nd);
  for (int i = n - 1; i >= 0; --i) left = op(left, terms[i]);
  // right: prefix [mid+1, e] of node 2*node+1
  n = 0; nd = 2 * node + 1; l2 = mid + 1; h2 = hi;
  while (e != h2) {
    const int64_t m2 = (l2 + h2) >> 1;
    if (e <= m2) { nd = 2 * nd; h2 = m2; }
    else { terms[n++] = __ldcg(V + 2 * nd); nd = 2 * nd + 1; l2 = m2 + 1; }
  }
  float right = __ldcg(V + nd);
  for (int i = n - 1; i >= 0; --i) right = op(terms[i], right);
  return op(left, right);
}

__global__ void reduce_kernel(const float* sum, const float* mn, int64_t cap, int64_t s, int64_t e, float* out) {
  if (threadIdx.x == 0) { out[0] = range_reduce_ref<true>(sum, cap, s, e); out[1] = range_reduce_ref<false>(mn, cap, s, e); }
}

// SumSegmentTree.find_prefixsum_idx (:126-149) for caller-supplied masses (fp32 descent)
__global__ void find_prefix_kernel(const float* sum, int64_t cap, int n, const double* masses, int32_t* idx) {
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  float mass = __double2float_rn(masses[t]);
  int64_t i = 1;
  while (i < cap) {
    const float left = __ldcg(sum + 2 * i);
    if (left > mass) i = 2 * i;
    else { mass = __fsub_rn(mass, left); i = 2 * i + 1; }
  }
  idx[t] = int32_t(i - cap);
}

static cudaStream_t g_side_stream = nullptr;          // trace only: which launches are the prefetching sampler's
void trace_set_side_stream(cudaStream_t s) { g_side_stream = s; }
static bool st_is_side(cudaStream_t st) { return g_side_stream != nullptr && st == g_side_stream; }
int launch_sample(const d4pg_replay* h, SampleArgs& a, cudaStream_t st, bool dependent = false) {
  a.sum = h->sum; a.mn = h->mn; a.cap = h->cap; a.state = reinterpret_cast<const ReplayState*>(h->state);
  a.obs = h->obs; a.act = h->act; a.rew = h->rew; a.obs2 = h->obs2; a.done = h->done;
  a.obs_dim = h->obs_dim; a.act_dim = h->act_dim;
  a.trace = (a.clock && debug_trace_buffer()) ? debug_trace_buffer() + STEP_TRACE_BASE : nullptr;
  a.trace_slot = a.pipe_slot >= 0 && a.uniforms == nullptr && st_is_side(st) ? 4 : 0;
  D4PG_MAX_CARVEOUT(sample_gather_kernel);
  // dependent: programmatic dependent launch behind the previous kernel of the stream (the host pipeline's tree add): the
  // grid is resident when that kernel ends, pdl_wait() at the top of the kernel holds it until its writes are visible
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(cdiv(a.B, SAMPLE_ROWS)); cfg.blockDim = dim3(SAMPLE_THREADS); cfg.dynamicSmemBytes = 0; cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = dependent ? 1 : 0;
  D4PG_CUDA_OK(cudaLaunchKernelEx(&cfg, sample_gather_kernel, a));
  return D4PG_OK;
}

int learner_sample(d4pg_replay* h, int B, int prioritized, const double* uniforms, const int32_t* positions,
                   uint64_t seed, LearnerClock* clock, const ClockParams& cp,
                   int32_t* idx, float* weights, float* s, float* a, double* r, float* s2, uint8_t* d,
                   int ld_obs, int ld_act, int pipe_slot, cudaStream_t st, bool dependent, unsigned long long* done_epoch) {
  SampleArgs sa{};
  sa.done_epoch = done_epoch;
  sa.ld_obs = ld_obs; sa.ld_act = ld_act; sa.pipe_slot = pipe_slot;
  sa.uniforms = uniforms; sa.seed = seed; sa.counter = 0; sa.clock = clock; sa.clock_params = cp;
  sa.beta = 1.f; sa.B = B; sa.idx = idx; sa.weights = prioritized ? weights : nullptr;
  sa.s = s; sa.a = a; sa.r = r; sa.s2 = s2; sa.d = d;
  if (!prioritized) { sa.idx_in = positions; sa.uniform_mode = positions ? 0 : 1; }
  return launch_sample(h, sa, st, dependent);
}

void learner_sample_args(d4pg_replay* h, int B, int prioritized, const double* uniforms, const int32_t* positions,
                         uint64_t seed, LearnerClock* clock, const ClockParams& cp,
                         int32_t* idx, float* weights, float* s, float* a, double* r, float* s2, uint8_t* d,
                         int ld_obs, int ld_act, SampleArgs& sa) {
  sa = SampleArgs{};
  sa.ld_obs = ld_obs; sa.ld_act = ld_act; sa.pipe_slot = -1;
  sa.uniforms = uniforms; sa.seed = seed; sa.counter = 0; sa.clock = clock; sa.clock_params = cp;
  sa.beta = 1.f; sa.B = B; sa.idx = idx; sa.weights = prioritized ? weights : nullptr;
  sa.s = s; sa.a = a; sa.r = r; sa.s2 = s2; sa.d = d;
  if (!prioritized) { sa.idx_in = positions; sa.uniform_mode = positions ? 0 : 1; }
  sa.sum = h->sum; sa.mn = h->mn; sa.cap = h->cap; sa.state = reinterpret_cast<const ReplayState*>(h->state);
  sa.obs = h->obs; sa.act = h->act; sa.rew = h->rew; sa.obs2 = h->obs2; sa.done = h->done;
  sa.obs_dim = h->obs_dim; sa.act_dim = h->act_dim;
}
void tree_update_args(d4pg_replay* h, int B, const int32_t* idx, const float* prio, TreeArgs& a) {
  a = TreeArgs{};
  a.sum = h->sum; a.mn = h->mn; a.cap = h->cap; a.log2cap = h->log2cap; a.size = h->size;
  a.n = B; a.idx = idx; a.v0 = prio; a.alpha_f32 = h->alpha_f32; a.scratch = h->scratch;
  a.state = reinterpret_cast<ReplayState*>(h->state);
  h->pristine = 0;
}

int64_t replay_generation(const d4pg_replay* h) { return h->gen; }

int launch_gate_signal(unsigned long long* flag, cudaStream_t st);
int launch_tree_update(d4pg_replay* h, int B, const int32_t* idx, const float* prio, cudaStream_t st, unsigned long long* gate) {
  TreeArgs a{};
  a.sum = h->sum; a.mn = h->mn; a.cap = h->cap; a.log2cap = h->log2cap; a.size = h->size;
  a.n = B; a.idx = idx; a.v0 = prio; a.alpha_f32 = h->alpha_f32; a.scratch = h->scratch; a.state = reinterpret_cast<ReplayState*>(h->state);
  a.trace = (st_is_side(st) && debug_trace_buffer()) ? debug_trace_buffer() + STEP_TRACE_BASE : nullptr;
  if (B <= TREE_FAST_MAX && h->log2cap < TREE_FAST_LEVELS) {
    int hs = 64;
    while (hs < 2 * B) hs *= 2;
    const int threads = ((B + 31) / 32) * 32;
    const size_t smem = size_t(hs) * 2 * (sizeof(int) + sizeof(float2));     // 12 KB at B = 512
    D4PG_MAX_CARVEOUT(tree_update_fast_kernel);
    const int D = std::min(4, h->log2cap);                     // 2^D CTAs, one per top-level subtree
    if (D > 0) { a.gate = gate; gate = nullptr; }   // the last CTA opens the gate itself
    tree_update_fast_kernel<<<1 << D, threads, smem, st>>>(a, hs, D);
  } else {
    D4PG_MAX_CARVEOUT(tree_write_kernel<TREE_UPDATE>);
    tree_write_kernel<TREE_UPDATE><<<1, TREE_THREADS, 0, st>>>(a);
  }
  D4PG_LAUNCH_OK();
  if (gate) { int rc = launch_gate_signal(gate, st); if (rc) return rc; }
  h->pristine = 0;
  return D4PG_OK;
}

}  // namespace d4pg

using namespace d4pg;

extern "C" int32_t d4pg_replay_capacity(int64_t size, int64_t* cap_out) {
  D4PG_REQUIRE(size > 0 && cap_out, D4PG_EINVAL, "d4pg_replay_capacity: bad arguments");
  int64_t cap = 1;
  while (cap < size) cap *= 2;                                       // :243-245
  *cap_out = cap;
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_create(int64_t size, int32_t obs_dim, int32_t act_dim, double alpha,
                                      float* sum_tree, float* min_tree,
                                      float* obs, float* act, double* rew, float* obs2, uint8_t* done,
                                      int32_t* scratch, float* state, d4pg_stream_t stream, d4pg_replay_t** out) {
  D4PG_REQUIRE(out && size > 0 && size < (int64_t(1) << 30), D4PG_EINVAL, "d4pg_replay_create: size out of range");
  D4PG_REQUIRE(obs_dim > 0 && act_dim > 0, D4PG_EINVAL, "d4pg_replay_create: dims must be positive");
  D4PG_REQUIRE(alpha >= 0, D4PG_EINVAL, "d4pg_replay_create: alpha must be >= 0");                      // :240
  D4PG_REQUIRE(sum_tree && min_tree && obs && act && rew && obs2 && done && scratch && state, D4PG_EINVAL,
               "d4pg_replay_create: null buffer");
  d4pg_replay* h = new (std::nothrow) d4pg_replay();
  D4PG_REQUIRE(h, D4PG_EINVAL, "d4pg_replay_create: out of host memory");
  h->size = size; d4pg_replay_capacity(size, &h->cap);
  h->log2cap = 0; while ((int64_t(1) << h->log2cap) < h->cap) ++h->log2cap;
  h->obs_dim = obs_dim; h->act_dim = act_dim; h->alpha = alpha; h->alpha_f32 = float(alpha);
  h->sum = sum_tree; h->mn = min_tree; h->obs = obs; h->act = act; h->rew = rew; h->obs2 = obs2; h->done = done;
  h->scratch = scratch; h->state = state; h->len = 0; h->next_idx = 0; h->pristine = 1;
  h->stage_host = nullptr; h->stage_dev = nullptr; h->stage_bytes = 0; h->stage_slot = 0;
  for (int i = 0; i < 2; ++i) { h->stage_ev[i] = nullptr; h->stage_busy[i] = false; }
  h->gate_flag = nullptr; h->gate_target = 0; h->gate_pending = false; h->order_ev = nullptr;
  tree_init_kernel<<<296, 256, 0, as_stream(stream)>>>(h->sum, h->mn, h->scratch,
                                                        reinterpret_cast<ReplayState*>(h->state), h->cap);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) { set_error("d4pg_replay_create: %s", cudaGetErrorString(e)); delete h; return D4PG_ECUDA; }
  *out = h;
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_destroy(d4pg_replay_t* h) {
  if (h) {
    for (int i = 0; i < 2; ++i) if (h->stage_ev[i]) cudaEventDestroy(h->stage_ev[i]);
    if (h->order_ev) cudaEventDestroy(h->order_ev);
    if (h->gate_flag) { cudaDeviceSynchronize(); cudaFree(h->gate_flag); }
  }
  delete h;
  return D4PG_OK;
}

namespace {
struct PackLayout { int64_t obs, obs2, act, rew, done, total; };
PackLayout pack_layout(const d4pg_replay* h, int64_t n) {
  PackLayout p;
  const int64_t S = int64_t(h->obs_dim) * 4, A = int64_t(h->act_dim) * 4;
  p.obs = 0; p.obs2 = p.obs + n * S; p.act = p.obs2 + n * S;
  p.rew = (p.act + n * A + 15) & ~int64_t(15);
  p.done = p.rew + n * 8;
  p.total = (p.done + n + 15) & ~int64_t(15);
  return p;
}
}  // namespace

extern "C" int64_t d4pg_replay_staging_bytes(const d4pg_replay_t* h, int64_t rows) {
  return (h && rows > 0) ? 2 * pack_layout(h, rows).total : -1;      // two staging slots
}

extern "C" int32_t d4pg_replay_set_staging(d4pg_replay_t* h, void* pinned_host, void* device, int64_t bytes) {
  D4PG_REQUIRE(h && pinned_host && device && bytes > 0, D4PG_EINVAL, "d4pg_replay_set_staging: bad arguments");
  h->stage_host = static_cast<uint8_t*>(pinned_host); h->stage_dev = static_cast<uint8_t*>(device);
  h->stage_bytes = (bytes / 2) & ~int64_t(15);                        // per slot
  for (int i = 0; i < 2; ++i) {
    if (!h->stage_ev[i]) D4PG_CUDA_OK(cudaEventCreateWithFlags(&h->stage_ev[i], cudaEventDisableTiming));
    h->stage_busy[i] = false;
  }
  h->stage_slot = 0;
  return D4PG_OK;
}

// ---- device-side ingest: n-step return accumulation at insert (replay_memory.py:38-45) ------------------------
// Transition i of an episode of T steps: (s_i, a_i, sum_{k<n} gamma^k r_{i+k}, s'_{i+n-1}, done_{i+n-1}).  Only the
// reward needs arithmetic -- s'/done are the same arrays shifted by n-1 rows -- and it is the reference's own
// left-to-right f64 loop (`cum += exp_gamma * r; exp_gamma *= gamma`) with explicit _rn ops (no FMA contraction).
__global__ void nstep_returns_kernel(const double* __restrict__ rew, int64_t T, int n, double gamma, double* __restrict__ out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i + n > T) return;
  double cum = 0.0, eg = 1.0;
  for (int k = 0; k < n; ++k) {
    cum = __dadd_rn(cum, __dmul_rn(eg, rew[i + k]));
    eg = __dmul_rn(eg, gamma);
  }
  out[i] = cum;
}

extern "C" int32_t d4pg_nstep_returns(const double* rew, int64_t T, int32_t n_steps, double gamma, double* out,
                                      d4pg_stream_t stream) {
  D4PG_REQUIRE(rew && out && T > 0 && n_steps >= 1, D4PG_EINVAL, "d4pg_nstep_returns: bad arguments");
  if (T < n_steps) return D4PG_OK;                        // the reference adds nothing before step n-1 (:38)
  const int64_t m = T - n_steps + 1;
  nstep_returns_kernel<<<unsigned((m + 255) / 256), 256, 0, as_stream(stream)>>>(rew, T, n_steps, gamma, out);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_add_nstep(d4pg_replay_t* h, int64_t T, const float* obs, const float* act, const double* rew,
                                         const float* obs2, const uint8_t* done, int32_t n_steps, double gamma,
                                         double* rew_scratch, int32_t prioritized, d4pg_stream_t stream) {
  D4PG_REQUIRE(h && obs && act && rew && obs2 && done && rew_scratch && T > 0 && n_steps >= 1, D4PG_EINVAL,
               "d4pg_replay_add_nstep: bad arguments");
  if (T < n_steps) return D4PG_OK;
  int rc = d4pg_nstep_returns(rew, T, n_steps, gamma, rew_scratch, stream);
  if (rc) return rc;
  const int64_t shift = n_steps - 1;
  return d4pg_replay_add(h, T - shift, obs, act, rew_scratch, obs2 + shift * h->obs_dim, done + shift, prioritized, stream);
}

// ---- device-side ingest: hindsight relabelling (main.py:154-184, "future" strategy) ------------------------------
// Episode of T goal-conditioned steps: obs/obs_next [T, So] f32, goal [T, G] f64 (the desired goal of every step),
// ag_next [T, G] f64 (achieved goal of the NEXT state), act [T, A], rew [T] f64, done [T].  Output rows, in the
// reference's order: for every t the original transition (s = obs_t || goal_t, s' = obs_next_t || goal_t), directly
// followed -- where select[t] != 0 -- by its relabelled copy with the achieved goal of step future[t] >= t as the goal,
// reward = -(||ag_next_t - goal'||_2 > threshold) (the sparse gym-robotics compute_reward, f64, sqrt of the
// left-to-right sum of squares like np.linalg.norm(axis=-1)) and done = (reward == 0).  select / future are the
// caller's random draws (np.random.uniform() < her_ratio, np.random.randint(t, T): main.py:166,170), `dst_row[t]` the
// exclusive prefix count of output rows.  The reference stores the relabelled copy with the LAST action of the rollout
// (`action`, main.py:184, not the step's own `a`): her_action_mode 0 reproduces that, 1 uses a_t.
struct HerArgs {
  const float* obs; const float* obs_next; const double* goal; const double* ag_next; const float* act;
  const double* rew; const uint8_t* done; const uint8_t* select; const int32_t* future; const int32_t* dst_row;
  int T, So, G, A, action_mode; double threshold;
  float* o_s; float* o_a; double* o_r; float* o_s2; uint8_t* o_d;
};
__global__ void her_relabel_kernel(const HerArgs a) {
  const int t = blockIdx.x;
  if (t >= a.T) return;
  const int S = a.So + a.G, row = a.dst_row[t];
  const bool sel = a.select[t] != 0;
  const int f = sel ? a.future[t] : t;
  for (int j = threadIdx.x; j < S; j += blockDim.x) {
    const bool is_obs = j < a.So;
    const float so = is_obs ? a.obs[size_t(t) * a.So + j] : float(a.goal[size_t(t) * a.G + (j - a.So)]);
    const float sn = is_obs ? a.obs_next[size_t(t) * a.So + j] : so;
    a.o_s[size_t(row) * S + j] = so;
    a.o_s2[size_t(row) * S + j] = sn;
    if (sel) {
      const float g2 = is_obs ? 0.f : float(a.ag_next[size_t(f) * a.G + (j - a.So)]);
      a.o_s[size_t(row + 1) * S + j] = is_obs ? so : g2;
      a.o_s2[size_t(row + 1) * S + j] = is_obs ? sn : g2;
    }
  }
  for (int j = threadIdx.x; j < a.A; j += blockDim.x) {
    a.o_a[size_t(row) * a.A + j] = a.act[size_t(t) * a.A + j];
    if (sel) a.o_a[size_t(row + 1) * a.A + j] = a.act[size_t(a.action_mode ? t : a.T - 1) * a.A + j];
  }
  if (threadIdx.x == 0) {
    a.o_r[row] = a.rew[t];
    a.o_d[row] = a.done[t];
    if (sel) {
      double ss = 0.0;
      for (int j = 0; j < a.G; ++j) {
        const double d = __dsub_rn(a.ag_next[size_t(t) * a.G + j], a.ag_next[size_t(f) * a.G + j]);
        ss = __dadd_rn(ss, __dmul_rn(d, d));
      }
      const double r = (__dsqrt_rn(ss) > a.threshold) ? -1.0 : -0.0;     // -(d > threshold), as gym-robotics returns it
      a.o_r[row + 1] = r;
      a.o_d[row + 1] = (r == 0.0) ? 1 : 0;
    }
  }
}

extern "C" int32_t d4pg_her_relabel(int32_t T, int32_t obs_dim, int32_t goal_dim, int32_t act_dim,
                                    const float* obs, const float* obs_next, const double* goal, const double* ag_next,
                                    const float* act, const double* rew, const uint8_t* done,
                                    const uint8_t* select, const int32_t* future, const int32_t* dst_row,
                                    double threshold, int32_t her_action_mode,
                                    float* out_s, float* out_a, double* out_r, float* out_s2, uint8_t* out_d,
                                    d4pg_stream_t stream) {
  D4PG_REQUIRE(T > 0 && obs_dim > 0 && goal_dim > 0 && act_dim > 0 && obs && obs_next && goal && ag_next && act && rew && done &&
               select && future && dst_row && out_s && out_a && out_r && out_s2 && out_d, D4PG_EINVAL, "d4pg_her_relabel: bad arguments");
  HerArgs a{obs, obs_next, goal, ag_next, act, rew, done, select, future, dst_row, T, obs_dim, goal_dim, act_dim,
            her_action_mode ? 1 : 0, threshold, out_s, out_a, out_r, out_s2, out_d};
  her_relabel_kernel<<<T, 64, 0, as_stream(stream)>>>(a);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_add_host(d4pg_replay_t* h, int64_t n, const float* obs, const float* act, const double* rew,
                                        const float* obs2, const uint8_t* done, int32_t prioritized, d4pg_stream_t stream) {
  if (h) ++h->gen;
  D4PG_REQUIRE(h && obs && act && rew && obs2 && done && n > 0, D4PG_EINVAL, "d4pg_replay_add_host: null/empty argument");
  D4PG_REQUIRE(h->stage_host, D4PG_ESTATE, "d4pg_replay_add_host: call d4pg_replay_set_staging first");
  const PackLayout p = pack_layout(h, n);
  D4PG_REQUIRE(p.total <= h->stage_bytes, D4PG_EINVAL, "d4pg_replay_add_host: %lld rows do not fit the staging buffer", (long long)n);
  const int slot = h->stage_slot; h->stage_slot ^= 1;
  if (h->stage_busy[slot]) D4PG_CUDA_OK(cudaEventSynchronize(h->stage_ev[slot]));   // the add that used this slot has consumed it
  uint8_t* hp = h->stage_host + size_t(slot) * h->stage_bytes;
  uint8_t* d = h->stage_dev + size_t(slot) * h->stage_bytes;
  memcpy(hp + p.obs, obs, size_t(n) * h->obs_dim * 4);
  memcpy(hp + p.obs2, obs2, size_t(n) * h->obs_dim * 4);
  memcpy(hp + p.act, act, size_t(n) * h->act_dim * 4);
  memcpy(hp + p.rew, rew, size_t(n) * 8);
  memcpy(hp + p.done, done, size_t(n));
  cudaStream_t st = as_stream(stream);
  D4PG_CUDA_OK(cudaMemcpyAsync(d, hp, size_t(p.total), cudaMemcpyHostToDevice, st));   // ahead of the ingest gate
  int rc = d4pg_replay_add(h, n, reinterpret_cast<const float*>(d + p.obs), reinterpret_cast<const float*>(d + p.act),
                           reinterpret_cast<const double*>(d + p.rew), reinterpret_cast<const float*>(d + p.obs2),
                           d + p.done, prioritized, stream);
  D4PG_CUDA_OK(cudaEventRecord(h->stage_ev[slot], st));               // device slot read by the ring write
  h->stage_busy[slot] = true;
  return rc;
}

// ---- ingest gate + stream ordering (learner host pipeline, learner.cu) ------------------------------------------
namespace d4pg {
__global__ void gate_wait_kernel(const unsigned long long* flag, unsigned long long target, unsigned long long* trace) {
  unsigned long long v;
  step_stamp(trace, 10);
  do { asm volatile("ld.acquire.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory"); } while (v < target);
  step_stamp(trace, 10 + 16);
}
__global__ void gate_signal_kernel(unsigned long long* flag) {
  unsigned long long v;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(flag) : "memory");
  asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(flag), "l"(v + 1) : "memory");
}
unsigned long long* replay_gate_flag(d4pg_replay* h) {
  if (!h->gate_flag) {
    if (cudaMalloc(reinterpret_cast<void**>(&h->gate_flag), 16) != cudaSuccess || cudaMemset(h->gate_flag, 0, 16) != cudaSuccess) return nullptr;
  }
  return h->gate_flag;
}
void replay_arm_gate(d4pg_replay* h) { ++h->gate_target; h->gate_pending = true; }
int replay_gate_consume(d4pg_replay* h, cudaStream_t st) {
  if (!h->gate_pending) return D4PG_OK;
  gate_wait_kernel<<<1, 1, 0, st>>>(h->gate_flag, h->gate_target, step_trace());
  D4PG_LAUNCH_OK();
  h->gate_pending = false;
  return D4PG_OK;
}
int launch_gate_signal(unsigned long long* flag, cudaStream_t st) {
  gate_signal_kernel<<<1, 1, 0, st>>>(flag);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}
}  // namespace d4pg

extern "C" int32_t d4pg_replay_order_after(d4pg_replay_t* h, d4pg_stream_t first, d4pg_stream_t then) {
  D4PG_REQUIRE(h, D4PG_EINVAL, "d4pg_replay_order_after: null handle");
  if (as_stream(first) == as_stream(then)) return D4PG_OK;
  if (!h->order_ev) D4PG_CUDA_OK(cudaEventCreateWithFlags(&h->order_ev, cudaEventDisableTiming));
  D4PG_CUDA_OK(cudaEventRecord(h->order_ev, as_stream(first)));
  D4PG_CUDA_OK(cudaStreamWaitEvent(as_stream(then), h->order_ev, 0));
  return D4PG_OK;
}
extern "C" int64_t d4pg_replay_len(const d4pg_replay_t* h) { return h ? h->len : -1; }
extern "C" int64_t d4pg_replay_next_idx(const d4pg_replay_t* h) { return h ? h->next_idx : -1; }

extern "C" int32_t d4pg_replay_set_len(d4pg_replay_t* h, int64_t len, int64_t next_idx, int32_t pristine, d4pg_stream_t stream) {
  if (h) ++h->gen;
  D4PG_REQUIRE(h && len >= 0 && len <= h->size && next_idx >= 0 && next_idx < h->size, D4PG_EINVAL,
               "d4pg_replay_set_len: out of range");
  h->len = len; h->next_idx = next_idx; h->pristine = pristine ? 1 : 0;
  state_set_kernel<<<1, 1, 0, as_stream(stream)>>>(reinterpret_cast<ReplayState*>(h->state), len, next_idx, h->pristine);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_add(d4pg_replay_t* h, int64_t n, const float* obs, const float* act,
                                   const double* rew, const float* obs2, const uint8_t* done,
                                   int32_t prioritized, d4pg_stream_t stream) {
  if (h) ++h->gen;
  D4PG_REQUIRE(h && obs && act && rew && obs2 && done, D4PG_EINVAL, "d4pg_replay_add: null argument");
  D4PG_REQUIRE(n > 0 && n <= h->size, D4PG_EINVAL, "d4pg_replay_add: need 0 < n <= size (n=%lld)", (long long)n);
  cudaStream_t st = as_stream(stream);
  const int64_t start = h->next_idx;
  const int64_t new_len = std::min<int64_t>(h->size, std::max<int64_t>(h->len, start + n));
  const int64_t new_next = (start + n) % h->size;
  const int blocks = int(std::min<int64_t>(148 * 4, (n * h->obs_dim + 255) / 256));
  ring_write_kernel<<<blocks, 256, 0, st>>>(h->obs, h->act, h->rew, h->obs2, h->done, obs, act, rew, obs2, done,
                                             n, h->obs_dim, h->act_dim, h->size, start,
                                             reinterpret_cast<ReplayState*>(h->state), new_len, new_next, step_trace());
  D4PG_LAUNCH_OK();
  if (prioritized) {
    // ingest gate (host pipeline): the rows above only had to follow the previous gather (stream order); the trees wait for
    // the last launched learner step's priority write-back -- inside the first tree kernel when that is the 1-CTA fast one
    const int64_t n1g = std::min<int64_t>(n, h->size - start);
    const unsigned long long* gflag = nullptr; unsigned long long gtarget = 0;
    if (h->gate_pending && n <= 65536 && n1g <= TREE_ADD_FAST_MAX && h->log2cap < 32) {
      gflag = h->gate_flag; gtarget = h->gate_target; h->gate_pending = false;
    } else {
      int grc = replay_gate_consume(h, st); if (grc) return grc;
    }
    if (n <= 65536) {
      // split a wrapping add into its two contiguous pieces
      const int64_t n1 = std::min<int64_t>(n, h->size - start);
      auto add_range = [&](int64_t s0, int64_t cnt) {
        if (cnt <= TREE_ADD_FAST_MAX && h->log2cap < 32) {
          tree_add_range_fast_kernel<<<1, TREE_THREADS, 0, st>>>(h->sum, h->mn, h->cap, h->log2cap, s0, cnt,
                                                                 reinterpret_cast<const ReplayState*>(h->state), h->alpha_f32, step_trace(),
                                                                 gflag, gtarget);
          gflag = nullptr;
        }
        else
          tree_add_range_kernel<<<1, TREE_THREADS, 0, st>>>(h->sum, h->mn, h->cap, h->log2cap, s0, cnt,
                                                            reinterpret_cast<const ReplayState*>(h->state), h->alpha_f32);
      };
      add_range(start, n1);
      D4PG_LAUNCH_OK();
      if (n1 < n) {
        add_range(0, n - n1);
        D4PG_LAUNCH_OK();
      }
    } else {
      leaf_fill_kernel<<<296, 256, 0, st>>>(h->sum, h->mn, h->cap, h->size, start, n,
                                            reinterpret_cast<const ReplayState*>(h->state), h->alpha_f32);
      D4PG_LAUNCH_OK();
      for (int64_t c = h->cap / 2; c >= 1; c /= 2) {
        const int b = int(std::min<int64_t>(296, (c + 255) / 256));
        level_rebuild_kernel<<<b, 256, 0, st>>>(h->sum, h->mn, c, c);
        D4PG_LAUNCH_OK();
      }
    }
  }
  h->len = new_len;
  h->next_idx = new_next;
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_sample(d4pg_replay_t* h, int32_t B, const double* uniforms,
                                      uint64_t philox_seed, uint64_t philox_counter, double beta,
                                      int32_t* idx, float* weights,
                                      float* s, float* a, double* r, float* s2, uint8_t* done,
                                      d4pg_stream_t stream) {
  D4PG_REQUIRE(h && B > 0 && idx && s && a && r && s2 && done, D4PG_EINVAL, "d4pg_replay_sample: null/empty argument");
  D4PG_REQUIRE(h->len >= 2, D4PG_ESTATE, "d4pg_replay_sample: needs at least 2 stored transitions (sum(0,len-1))");
  D4PG_REQUIRE(beta > 0, D4PG_EINVAL, "d4pg_replay_sample: beta must be > 0");                           // :299
  SampleArgs sa{};
  sa.uniforms = uniforms; sa.seed = philox_seed; sa.counter = philox_counter; sa.beta = float(beta);
  sa.B = B; sa.idx = idx; sa.weights = weights; sa.s = s; sa.a = a; sa.r = r; sa.s2 = s2; sa.d = done;
  return launch_sample(h, sa, as_stream(stream));
}

extern "C" int32_t d4pg_replay_gather(d4pg_replay_t* h, int32_t B, const int32_t* idx,
                                      float* s, float* a, double* r, float* s2, uint8_t* done, d4pg_stream_t stream) {
  D4PG_REQUIRE(h && B > 0 && idx && s && a && r && s2 && done, D4PG_EINVAL, "d4pg_replay_gather: null/empty argument");
  SampleArgs sa{};
  sa.B = B; sa.idx_in = idx; sa.s = s; sa.a = a; sa.r = r; sa.s2 = s2; sa.d = done;
  return launch_sample(h, sa, as_stream(stream));
}

extern "C" int32_t d4pg_replay_update_priorities(d4pg_replay_t* h, int32_t B, const int32_t* idx,
                                                 const float* prio, d4pg_stream_t stream) {
  if (h) ++h->gen;
  D4PG_REQUIRE(h && B > 0 && idx && prio, D4PG_EINVAL, "d4pg_replay_update_priorities: null/empty argument");
  return launch_tree_update(h, B, idx, prio, as_stream(stream));
}

extern "C" int32_t d4pg_replay_set_leaves(d4pg_replay_t* h, int32_t n, const int32_t* idx, const float* sum_vals,
                                          const float* min_vals, d4pg_stream_t stream) {
  if (h) ++h->gen;
  D4PG_REQUIRE(h && n > 0 && idx && sum_vals && min_vals, D4PG_EINVAL, "d4pg_replay_set_leaves: null/empty argument");
  TreeArgs a{};
  a.sum = h->sum; a.mn = h->mn; a.cap = h->cap; a.log2cap = h->log2cap; a.size = h->size;
  a.n = n; a.idx = idx; a.v0 = sum_vals; a.v1 = min_vals; a.scratch = h->scratch; a.state = reinterpret_cast<ReplayState*>(h->state);
  tree_write_kernel<TREE_SET><<<1, TREE_THREADS, 0, as_stream(stream)>>>(a);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_reduce(d4pg_replay_t* h, int64_t start, int64_t end, float* out, d4pg_stream_t stream) {
  D4PG_REQUIRE(h && out, D4PG_EINVAL, "d4pg_replay_reduce: null argument");
  if (end <= 0) end += h->cap;                                        // :91-94 (None / negative end)
  D4PG_REQUIRE(start >= 0 && start < end && end <= h->cap, D4PG_EINVAL, "d4pg_replay_reduce: bad range [%lld,%lld)",
               (long long)start, (long long)end);
  reduce_kernel<<<1, 32, 0, as_stream(stream)>>>(h->sum, h->mn, h->cap, start, end - 1, out);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}

extern "C" int32_t d4pg_replay_find_prefixsum(d4pg_replay_t* h, int32_t n, const double* masses, int32_t* idx,
                                              d4pg_stream_t stream) {
  D4PG_REQUIRE(h && n > 0 && masses && idx, D4PG_EINVAL, "d4pg_replay_find_prefixsum: null/empty argument");
  find_prefix_kernel<<<cdiv(n, 128), 128, 0, as_stream(stream)>>>(h->sum, h->cap, n, masses, idx);
  D4PG_LAUNCH_OK();
  return D4PG_OK;
}
