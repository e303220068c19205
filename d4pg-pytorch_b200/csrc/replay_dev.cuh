// Device code of the GPU-resident prioritized replay.
#pragma once
#include "internal.cuh"
#include "adam.cuh"

namespace d4pg {

// Device-resident bookkeeping (lives in the caller's `state` buffer, 32 bytes).  Kernels read
// len / pristine from here so a captured CUDA graph stays valid while add() keeps filling.
struct ReplayState {
  float max_priority;      // PrioritizedReplayBuffer._max_priority, :249,335
  int32_t pristine;        // 1 until the first update_priorities (tree still "all Python floats")
  int64_t len;             // len(self._storage)
  int64_t next_idx;        // self._next_idx
  int64_t reserved;
};
static_assert(sizeof(ReplayState) == 32, "ReplayState must fit the 8-float state buffer");

// leaf = priority ** alpha with np.float32 ** float semantics: powf(p, (float)alpha).  glibc's
// powf is correctly rounded in all but vanishing cases, so we evaluate in fp64 and round once.
__device__ __forceinline__ float pow_alpha(float p, float alpha_f32) {
  if (p == 1.0f) return 1.0f;
  return __double2float_rn(pow(double(p), double(alpha_f32)));
}

// SumSegmentTree.sum(0, end+1): reduce over leaves [0, end] with _reduce_helper's association
// (prioritized_replay_memory.py:61-96): V[left] + (V[left'] + (... + V[last])), fp32.
static __device__ float prefix_sum_ref(const float* __restrict__ V, int64_t cap, int64_t e) {
  // the node cover depends only on (cap, e): collect the addresses first so the loads are
  // independent and overlap (one L2 round trip instead of log2(cap) dependent ones)
  int64_t nodes[40];
  int n = 0;
  int64_t node = 1, lo = 0, hi = cap - 1;
  while (true) {
    if (e == hi) { nodes[n++] = node; break; }
    int64_t mid = (lo + hi) >> 1;
    if (e <= mid) { node = 2 * node; hi = mid; }
    else { nodes[n++] = 2 * node; node = 2 * node + 1; lo = mid + 1; }
  }
  float terms[40];
#pragma unroll 8
  for (int i = 0; i < n; ++i) terms[i] = __ldcg(V + nodes[i]);
  float acc = terms[n - 1];
  for (int i = n - 2; i >= 0; --i) acc = __fadd_rn(terms[i], acc);
  return acc;
}
static __device__ float prefix_min_ref(const float* __restrict__ V, int64_t cap, int64_t e) {
  float acc = INFINITY;
  int64_t node = 1, lo = 0, hi = cap - 1;
  while (true) {
    if (e == hi) { acc = fminf(acc, __ldcg(V + node)); break; }
    int64_t mid = (lo + hi) >> 1;
    if (e <= mid) { node = 2 * node; hi = mid; }
    else { acc = fminf(acc, __ldcg(V + 2 * node)); node = 2 * node + 1; lo = mid + 1; }
  }
  return acc;
}

struct SampleArgs {
  const float* sum; const float* mn; int64_t cap; const ReplayState* state;
  const double* uniforms; uint64_t seed, counter; float beta;
  LearnerClock* clock;              // optional (learner): Philox counter / beta from the device clock;
  ClockParams clock_params;         //   block 0 also derives this step's Adam scalars into it
  const float* obs; const float* act; const double* rew; const float* obs2; const uint8_t* done;
  int obs_dim, act_dim; int B;
  int ld_obs, ld_act;               // row pitch of the gathered s/s2 and a batches (0 = dense)
  const int32_t* idx_in;            // gather-only mode when non-null
  int uniform_mode;                 // 1: idx = floor(u*len) (device-side uniform replay, with replacement)
  int32_t* idx; float* weights;
  float* s; float* a; double* r; float* s2; uint8_t* d;
  int pipe_slot;                    // >= 0 (prefetch pipeline): use the sampler's own counters, derive into this slot
  unsigned long long* trace; int trace_slot;
  unsigned long long* done_epoch;   // host pipeline: CTA b publishes (release) s_steps_done + 1 in [b] when its rows are gathered
};

constexpr int SAMPLE_THREADS = 256;
constexpr int TOP_LEVELS = 11;       // tree levels 0..10 (nodes 1..2047) are staged in shared memory

// sum(0, len-1) by one warp: the prefix [0,x) (x = len-1) is covered by one node per set bit of x;
// _reduce_helper (:61-96) adds them right-nested, i.e. lowest bit first: acc = t_b + acc going up.
// Each lane fetches the node of "its" bit (all loads in flight together), lane 0 folds them in order.
__device__ __forceinline__ float warp_prefix_sum(const float* __restrict__ V, int64_t cap, int64_t x, int lane) {
  float term = 0.f;
  const bool has = ((x >> lane) & 1) != 0;
  if (has) {
    const int64_t start = x & ~((int64_t(2) << lane) - 1);
    term = __ldcg(V + (cap >> lane) + (start >> lane));
  }
  const unsigned mask = __ballot_sync(0xffffffffu, has);
  float acc = 0.f;
  bool first = true;
  for (int b = 0; b < 32; ++b) {
    const float t = __shfl_sync(0xffffffffu, term, b);
    if ((mask >> b) & 1) { acc = first ? t : __fadd_rn(t, acc); first = false; }
  }
  return acc;
}

// _sample_proportional (:258-265) + IS weights (:303-311) + _encode_sample (:189-199), fused.
struct SampleSmem {
  float top[1 << TOP_LEVELS];
  int32_t idx[SAMPLE_ROWS];
  float total;
};
// rows [bid*32, bid*32+32) of the batch, executed by one 256-thread CTA
__device__ __forceinline__ void sample_body(const SampleArgs& a, int bid, SampleSmem& sm) {
  int32_t* idx_s = sm.idx;
  float* top_s = sm.top;
  float& total_s = sm.total;
  const int row0 = bid * SAMPLE_ROWS;
  const int nrows = min(SAMPLE_ROWS, a.B - row0);
  const int t = threadIdx.x;
  const bool piped = a.clock && a.pipe_slot >= 0;
  if (a.clock && bid == 0 && t == SAMPLE_THREADS - 1) {
    if (piped) clock_derive_pipelined(a.clock, a.clock_params, a.pipe_slot);
    else { clock_derive(a.clock, a.clock_params); a.clock->beta = clock_beta(a.clock, a.clock_params); }
  }
  const bool descend = (a.idx_in == nullptr) && !a.uniform_mode;
  const int64_t len = a.state->len;
  int top_levels = 0;
  if (descend) {
    // stage the top of the sum tree (one L2 round trip for the whole CTA) and the prefix total
    while ((int64_t(1) << top_levels) < a.cap && top_levels < TOP_LEVELS) ++top_levels;
    for (int i = t; i < (1 << top_levels); i += SAMPLE_THREADS) top_s[i] = (i >= 1) ? __ldcg(a.sum + i) : 0.f;
    if (t < 32) {
      const float tot = warp_prefix_sum(a.sum, a.cap, len - 1, t);       // sum(0, len-1): leaves [0, len-2]
      if (t == 0) total_s = tot;
    }
    __syncthreads();
  }
  if (t < nrows) {
    const int row = row0 + t;
    int32_t leaf_idx;
    if (a.idx_in) {
      leaf_idx = a.idx_in[row];
    } else {
      const uint64_t ctr = a.counter + (a.clock ? uint64_t(piped ? a.clock->s_steps_done : a.clock->steps_done) : 0ull);
      const double u = a.uniforms ? a.uniforms[row] : Philox::uniform53(a.seed, ctr, uint32_t(row));
      int64_t i = 1;
      const int64_t top_end = int64_t(1) << (top_levels - 1);              // nodes < 2*top_end have children in top_s
      if (a.uniform_mode) {
        int64_t pick = int64_t(u * double(len));
        i = a.cap + (pick < len ? pick : len - 1);
      } else if (a.state->pristine) {
        // tree of Python floats: mass and the descent are fp64 (all node values are integers)
        double mass = __dmul_rn(u, double(total_s));
        while (i < a.cap && 2 * i < 2 * top_end) {                    // levels staged in shared memory
          const double left = double(top_s[2 * i]);
          if (left > mass) i = 2 * i;                                 // strict, :144
          else { mass = __dsub_rn(mass, left); i = 2 * i + 1; }
        }
        // below: THREE levels per L2 round trip -- the 7 left children the next three decisions can ask for are
        // fetched together; the comparisons and subtractions are the same ones, in the same order
        while (4 * i < a.cap) {
          const float* V = a.sum;
          const float l1 = __ldcg(V + 2 * i), l20 = __ldcg(V + 4 * i), l21 = __ldcg(V + 4 * i + 2);
          const float l30 = __ldcg(V + 8 * i), l31 = __ldcg(V + 8 * i + 2), l32 = __ldcg(V + 8 * i + 4), l33 = __ldcg(V + 8 * i + 6);
          const bool r1 = !(double(l1) > mass); if (r1) mass = __dsub_rn(mass, double(l1));
          const float l2 = r1 ? l21 : l20;
          const bool r2 = !(double(l2) > mass); if (r2) mass = __dsub_rn(mass, double(l2));
          const float l3 = r1 ? (r2 ? l33 : l32) : (r2 ? l31 : l30);
          const bool r3 = !(double(l3) > mass); if (r3) mass = __dsub_rn(mass, double(l3));
          i = 8 * i + 4 * int(r1) + 2 * int(r2) + int(r3);
        }
        while (i < a.cap) {
          const double left = double(__ldcg(a.sum + 2 * i));
          if (left > mass) i = 2 * i;
          else { mass = __dsub_rn(mass, left); i = 2 * i + 1; }
        }
      } else {
        float mass = __fmul_rn(__double2float_rn(u), total_s);         // weak float * np.float32
        while (i < a.cap && 2 * i < 2 * top_end) {
          const float left = top_s[2 * i];
          if (left > mass) i = 2 * i;
          else { mass = __fsub_rn(mass, left); i = 2 * i + 1; }
        }
        while (4 * i < a.cap) {
          const float* V = a.sum;
          const float l1 = __ldcg(V + 2 * i), l20 = __ldcg(V + 4 * i), l21 = __ldcg(V + 4 * i + 2);
          const float l30 = __ldcg(V + 8 * i), l31 = __ldcg(V + 8 * i + 2), l32 = __ldcg(V + 8 * i + 4), l33 = __ldcg(V + 8 * i + 6);
          const bool r1 = !(l1 > mass); if (r1) mass = __fsub_rn(mass, l1);
          const float l2 = r1 ? l21 : l20;
          const bool r2 = !(l2 > mass); if (r2) mass = __fsub_rn(mass, l2);
          const float l3 = r1 ? (r2 ? l33 : l32) : (r2 ? l31 : l30);
          const bool r3 = !(l3 > mass); if (r3) mass = __fsub_rn(mass, l3);
          i = 8 * i + 4 * int(r1) + 2 * int(r2) + int(r3);
        }
        while (i < a.cap) {
          const float left = __ldcg(a.sum + 2 * i);
          if (left > mass) i = 2 * i;
          else { mass = __fsub_rn(mass, left); i = 2 * i + 1; }
        }
      }
      leaf_idx = int32_t(i - a.cap);
      if (a.weights && !a.uniform_mode) {
        const float tot = __ldcg(a.sum + 1);
        const float pmin = __fdiv_rn(__ldcg(a.mn + 1), tot);
        const float n = float(len);
        const float beta = a.clock ? clock_beta(a.clock, a.clock_params, piped) : a.beta;
        const float maxw = __double2float_rn(pow(double(__fmul_rn(pmin, n)), double(-beta)));
        const float ps = __fdiv_rn(__ldcg(a.sum + a.cap + leaf_idx), tot);
        const float w = __double2float_rn(pow(double(__fmul_rn(ps, n)), double(-beta)));
        a.weights[row] = __fdiv_rn(w, maxw);
      }
    }
    idx_s[t] = leaf_idx;
    if (a.idx) a.idx[row] = leaf_idx;
    if (a.r) a.r[row] = a.rew[leaf_idx];
    if (a.d) a.d[row] = a.done[leaf_idx];
  }
  __syncthreads();
  // coalesced row gathers: consecutive threads walk consecutive features of one transition
  const int od = a.obs_dim, ad = a.act_dim;
  const int lo = a.ld_obs ? a.ld_obs : od, la = a.ld_act ? a.ld_act : ad;
  for (int e = t; e < nrows * od; e += SAMPLE_THREADS) {
    const int rr = e / od, c = e - rr * od;
    const size_t src = size_t(idx_s[rr]) * od + c, dst = size_t(row0 + rr) * lo + c;
    a.s[dst] = __ldg(a.obs + src);
    a.s2[dst] = __ldg(a.obs2 + src);
  }
  for (int e = t; e < nrows * ad; e += SAMPLE_THREADS) {
    const int rr = e / ad, c = e - rr * ad;
    a.a[size_t(row0 + rr) * la + c] = __ldg(a.act + size_t(idx_s[rr]) * ad + c);
  }
}

// ---- leaf writes + level-synchronous parent recompute, one CTA ---------------------------
// update_priorities (:315-335) is a sequential Python loop; its final state equals "write all
// leaves (last writer wins on duplicates), then recompute every touched ancestor bottom-up",
// because each node's last recompute sees its children's final values.
enum { TREE_UPDATE = 0, TREE_SET = 1, TREE_ADD = 2 };
struct TreeArgs {
  float* sum; float* mn; int64_t cap; int log2cap; int64_t size;
  int n; const int32_t* idx; const float* v0; const float* v1;   // UPDATE: v0=prio; SET: v0=sum vals, v1=min vals
  int64_t ring_start;                                              // ADD: positions (ring_start+i) % size
  float alpha_f32; int32_t* scratch; ReplayState* state;
  unsigned long long* trace;
  unsigned long long* gate;     // non-null (host pipeline): bumped once, with release order, when every node is written
};
constexpr int TREE_THREADS = 1024;

// executed by ONE CTA of NT threads
template <int MODE, int NT>
__device__ __forceinline__ void tree_write_body(const TreeArgs& a, float* red) {
  const int t = threadIdx.x;
  auto pos = [&](int i) -> int64_t {
    return MODE == TREE_ADD ? (a.ring_start + i) % a.size : int64_t(a.idx[i]);
  };
  if (MODE != TREE_ADD) {
    for (int i = t; i < a.n; i += NT) atomicMax(a.scratch + pos(i), i);
    __syncthreads();
  }
  float local_max = 0.f;
  const float add_leaf = (MODE == TREE_ADD) ? pow_alpha(a.state->max_priority, a.alpha_f32) : 0.f;  // :255-256
  for (int i = t; i < a.n; i += NT) {
    const int64_t p = pos(i);
    if (MODE == TREE_ADD || a.scratch[p] == i) {
      float ls, lm;
      if (MODE == TREE_UPDATE) { ls = lm = pow_alpha(a.v0[i], a.alpha_f32); }
      else if (MODE == TREE_SET) { ls = a.v0[i]; lm = a.v1[i]; }
      else { ls = lm = add_leaf; }
      a.sum[a.cap + p] = ls;
      a.mn[a.cap + p] = lm;
    }
    if (MODE == TREE_UPDATE) local_max = fmaxf(local_max, a.v0[i]);
  }
  if (MODE == TREE_UPDATE) {                                       // _max_priority, :335
    local_max = warp_max(local_max);
    if ((t & 31) == 0) red[t >> 5] = local_max;
    __syncthreads();
    if (t < 32) {
      float v = warp_max(t < NT / 32 ? red[t] : 0.f);
      if (t == 0) {
        if (v > a.state->max_priority) a.state->max_priority = v;
        a.state->pristine = 0;
      }
    }
  }
  __syncthreads();
  if (MODE != TREE_ADD)
    for (int i = t; i < a.n; i += NT) a.scratch[pos(i)] = -1;
  for (int lvl = 1; lvl <= a.log2cap; ++lvl) {
    __syncthreads();
    for (int i = t; i < a.n; i += NT) {
      const int64_t node = (a.cap + pos(i)) >> lvl;
      const float l = __ldcg(a.sum + 2 * node), r = __ldcg(a.sum + 2 * node + 1);
      a.sum[node] = __fadd_rn(l, r);
      a.mn[node] = fminf(__ldcg(a.mn + 2 * node), __ldcg(a.mn + 2 * node + 1));
    }
  }
}

// ---- update_priorities for up to 512 leaves with ONE round trip to L2 -------------------------------------
// tree_write_body pays an L2 round trip per level (20 at capacity 2^20: 30-50 us, and the next step's sampler
// waits for it).  Here every thread owns one updated leaf and first fetches the OLD value of the sibling of every
// node on its leaf-to-root path (2 x log2(cap) independent loads, in flight together, kept in registers).  The
// walk up is then done entirely in shared memory: at each level the new values of the touched nodes go into a
// small hash table (key = node id), a thread finds its sibling there if another updated leaf shares it and falls
// back to the prefetched old value if not, and the parent's value moves up in registers.  fp32 `left + right` is
// commutative and every thread that shares a node computes the same value from the same inputs, so the final
// tree is exactly "write all leaves (last writer wins), recompute every touched ancestor" like tree_write_body.
constexpr int TREE_FAST_MAX = 512;        // leaves per call (one thread each; 2 x 24 prefetched siblings live in registers)
constexpr int TREE_FAST_LEVELS = 24;      // capacity up to 2^23
struct TreeHashSmem { int* keys[2]; float2* vals[2]; int mask; };

__device__ __forceinline__ void tree_hash_put(int* keys, float2* vals, int mask, int node, float s, float m) {
  unsigned h = (unsigned(node) * 2654435761u) >> 7;
  while (true) {
    h &= unsigned(mask);
    const int old = atomicCAS(&keys[h], 0, node);
    if (old == 0 || old == node) { vals[h] = make_float2(s, m); return; }     // same node -> same value from every writer
    ++h;
  }
}
__device__ __forceinline__ bool tree_hash_get(const int* keys, const float2* vals, int mask, int node, float& s, float& m) {
  unsigned h = (unsigned(node) * 2654435761u) >> 7;
  while (true) {
    h &= unsigned(mask);
    const int k = keys[h];
    if (k == node) { const float2 v = vals[h]; s = v.x; m = v.y; return true; }
    if (k == 0) return false;
    ++h;
  }
}

// CTA `c` of 2^D owns the leaves (and all their ancestors below depth D) of top-level subtree c: subtrees never
// share a node, so the CTAs are independent; the last one to finish recomputes the 2^D - 1 nodes above.
// `hash` = 2 tables of `hs` entries (int key + float2 value), hs = pow2 >= 2 n.
__device__ __forceinline__ void tree_update_fast_body(const TreeArgs& a, unsigned char* smem_raw, int hs, float* red, int c, int D) {
  const int t = threadIdx.x, n = a.n;
  int* keys0 = reinterpret_cast<int*>(smem_raw);
  int* keys1 = keys0 + hs;
  float2* vals0 = reinterpret_cast<float2*>(keys1 + hs);
  float2* vals1 = vals0 + hs;
  const int mask = hs - 1;
  const int L = a.log2cap - D;                               // levels walked inside the subtree (its root is level L)
  for (int i = t; i < 2 * hs; i += blockDim.x) keys0[i] = 0;
  const int64_t p = t < n ? int64_t(a.idx[t]) : 0;
  const bool act = t < n && int(p >> L) == c;
  if (act) atomicMax(a.scratch + p, t);                      // duplicates: the last writer (largest i) wins, :329-333
  // old sibling values along the path (the loads overlap each other and the barrier)
  float so[TREE_FAST_LEVELS], mo[TREE_FAST_LEVELS];
#pragma unroll
  for (int lvl = 0; lvl < TREE_FAST_LEVELS; ++lvl) {
    so[lvl] = 0.f; mo[lvl] = 0.f;
    if (act && lvl < L) {
      const int64_t sib = ((a.cap + p) >> lvl) ^ 1;
      so[lvl] = __ldcg(a.sum + sib); mo[lvl] = __ldcg(a.mn + sib);
    }
  }
  __syncthreads();
  float vs = 0.f, vm = 0.f;
  if (act) {
    const int w = a.scratch[p];                               // winning writer of this leaf
    vs = vm = pow_alpha(a.v0[w], a.alpha_f32);
  }
  if (c == 0) {                                               // _max_priority (:335) over the whole call
    float local_max = warp_max(t < n ? a.v0[t] : 0.f);
    if ((t & 31) == 0) red[t >> 5] = local_max;
    __syncthreads();
    if (t < 32) {
      const float v = warp_max(t < int(blockDim.x) / 32 ? red[t] : 0.f);
      if (t == 0) {
        if (v > a.state->max_priority) a.state->max_priority = v;
        a.state->pristine = 0;
      }
    }
  }
  __syncthreads();                                            // every sharer of a duplicated leaf has read its winner
  if (act) a.scratch[p] = -1;
#pragma unroll 1
  for (int lvl = 0; lvl <= L; ++lvl) {
    int* keys = (lvl & 1) ? keys1 : keys0;
    float2* vals = (lvl & 1) ? vals1 : vals0;
    const int node = int((a.cap + p) >> lvl);
    // threads of a warp that share the node elect one writer
    const unsigned peers = __match_any_sync(0xffffffffu, act ? node : -1 - (t & 31));
    const bool leader = act && (__ffs(peers) - 1) == (t & 31);
    if (leader) {
      a.sum[node] = vs; a.mn[node] = vm;                      // every sharer holds the same value
      if (lvl < L) tree_hash_put(keys, vals, mask, node, vs, vm);
    }
    if (lvl == L) break;
    __syncthreads();                                          // this level's table is complete
    if (act) {
      float ss, sm;
      if (!tree_hash_get(keys, vals, mask, node ^ 1, ss, sm)) {
        ss = 0.f; sm = 0.f;                                   // static register indexing: the prefetched sibling of this level
#pragma unroll
        for (int q = 0; q < TREE_FAST_LEVELS; ++q) if (q == lvl) { ss = so[q]; sm = mo[q]; }
      }
      vs = __fadd_rn(vs, ss);
      vm = fminf(vm, sm);
    }
    int* nk = (lvl & 1) ? keys0 : keys1;                      // clear the other table for the next level
    for (int i = t; i < hs; i += blockDim.x) nk[i] = 0;
    __syncthreads();
  }
  if (D == 0) return;
  // ---- the 2^D - 1 nodes above the subtree roots: by the last CTA to get here -------------------------------
  __shared__ int is_last;
  __syncthreads();
  if (t == 0) {
    __threadfence();
    unsigned long long* ticket = reinterpret_cast<unsigned long long*>(&a.state->reserved);
    const unsigned long long k = atomicAdd(ticket, 1ull);
    is_last = (k == (1ull << D) - 1ull);
    if (is_last) { *ticket = 0ull; __threadfence(); }
  }
  __syncthreads();
  if (is_last && t < 32) {
    for (int d = D - 1; d >= 0; --d) {
      if (t < (1 << d)) {
        const int node = (1 << d) + t;
        a.sum[node] = __fadd_rn(__ldcg(a.sum + 2 * node), __ldcg(a.sum + 2 * node + 1));
        a.mn[node] = fminf(__ldcg(a.mn + 2 * node), __ldcg(a.mn + 2 * node + 1));
      }
      __threadfence_block();
      __syncwarp();
    }
    if (a.gate) {                                             // the ingest gate opens: the trees are complete
      __threadfence();
      __syncwarp();
      if (t == 0) {
        unsigned long long v;
        asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(a.gate) : "memory");
        asm volatile("st.release.gpu.global.u64 [%0], %1;" :: "l"(a.gate), "l"(v + 1) : "memory");
      }
    }
  }
}

}  // namespace d4pg
